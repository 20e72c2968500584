"""The two-tile schedule of mpc_rollout_tc_kernel (two tiles per CTA, offset by half a step) against the one-tile
schedule: same operands, same K order, same conversions, so every output must be bit-identical.  SS_TC_PAIR=0
forces the one-tile schedule; ss_mpc_last_tc_schedule reports which one ran."""
import os

import numpy as np
import pytest

from smartstartcontinuous_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

TILE = 128


def _model(rng, d, da, h):
    if d == 3:
        obs, act = syn.pendulum_rollouts(rng, 8, 200)
    else:
        obs = [rng.normal(size=(200, d)) for _ in range(8)]
        act = [rng.uniform(-1, 1, size=(199, da)) for _ in range(8)]
    norm = syn.normalisation_stats(np.concatenate(list(obs)),
                                   np.concatenate([np.concatenate([a, a[-1:]]) for a in act]))
    w, b = syn.xavier_mlp(rng, d, da, 2, h, scale=0.5)
    from smartstartcontinuous_b200.nnd_mb_agent import plan_from_path
    plan = plan_from_path(list(obs[0][:60]), mean_per_stepsize=1, std_per_stepsize=1,
                          stepsizes_in_waypoint_radii=1, path_shortcutting=True, theta=1, steps_per_waypoint=1)
    return w, b, norm, plan, obs[0][0]


def _run(engine, force_one_tile, fn):
    old = os.environ.get("SS_TC_PAIR")
    os.environ["SS_TC_PAIR"] = "0" if force_one_tile else "1"
    try:
        out = fn()
        return out, engine.last_tc_schedule()
    finally:
        if old is None:
            del os.environ["SS_TC_PAIR"]
        else:
            os.environ["SS_TC_PAIR"] = old


def _sms(engine):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count // 2 * 2


# tile iterations per CTA: 2 (even), 3 (odd: the third tile runs alone), 4, a K whose last wave leaves some
# CTAs a lone padding tile, and grid + 5 tiles (the second tile of most CTAs' pair is padding); K is never a
# multiple of the tile.  d = 3, da = 1 runs <4,3,16>; d = 2, da = 2 runs <4,2,16>.
@pytest.mark.parametrize("iters,extra_tiles", [(2, 0), (3, 0), (4, 0), (3, -40), (1, 5)])
@pytest.mark.parametrize("mode", ["reference", "per_sample"])
@pytest.mark.parametrize("d,da", [(3, 1), (2, 2)])
def test_two_tile_schedule_is_bit_identical(engine, iters, extra_tiles, mode, d, da):
    rng = np.random.default_rng(100 + iters + 10 * d)
    w, b, norm, plan, start = _model(rng, d, da, 500)
    engine.set_model(w, b, norm)
    engine.set_plan(plan["desired_states"], plan["distances_left"], plan["radii"])
    grid = _sms(engine)
    K = (iters * grid + extra_tiles) * TILE - 37
    kw = dict(K=K, H=5, seed=4, act_low=[-2.0] * da, act_high=[2.0] * da, penalty_mode=mode, precision="bf16_tc",
              want_scores=True)
    one, s1 = _run(engine, True, lambda: engine.plan(start, 0, **kw))
    two, s2 = _run(engine, False, lambda: engine.plan(start, 0, **kw))
    assert engine.last_rollout_kernel() == "mpc_rollout_tc_kernel"
    assert (s1, s2) == ("one_tile", "two_tile")
    np.testing.assert_array_equal(two["scores"], one["scores"])
    assert two["best_k"] == one["best_k"]
    np.testing.assert_array_equal(two["best_sequence"], one["best_sequence"])
    np.testing.assert_array_equal(two["best_path"], one["best_path"])


@pytest.mark.parametrize("d,da", [(3, 1), (2, 2)])
def test_two_tile_forward_sim_rows_is_bit_identical(engine, d, da):
    """Per-sequence start states (the ROWS variant) on both schedules."""
    rng = np.random.default_rng(7 + d)
    w, b, norm, plan, start = _model(rng, d, da, 500)
    engine.set_model(w, b, norm)
    K = (2 * _sms(engine) + 5) * TILE - 3
    starts = start + 0.1 * rng.normal(size=(K, d))
    acts = rng.uniform(-2, 2, size=(K, 4, da))
    one, s1 = _run(engine, True, lambda: engine.forward_sim(starts, acts, precision="bf16_tc"))
    two, s2 = _run(engine, False, lambda: engine.forward_sim(starts, acts, precision="bf16_tc"))
    np.testing.assert_array_equal(two, one)
    assert (s1, s2) == ("one_tile", "two_tile")


@pytest.mark.parametrize("d,da,h", [(2, 3, 500), (3, 1, 200)])
def test_layouts_without_two_tile_schedule(engine, d, da, h):
    """K1 = 32 layouts (no room for both H1 images) and hidden widths padded to 256 keep the one-tile schedule."""
    rng = np.random.default_rng(d * 10 + da)
    w, b, norm, plan, start = _model(rng, d, da, h)
    engine.set_model(w, b, norm)
    engine.set_plan(plan["desired_states"], plan["distances_left"], plan["radii"])
    K = 3 * _sms(engine) * TILE - 11
    kw = dict(K=K, H=3, seed=5, act_low=[-1.0] * da, act_high=[1.0] * da, penalty_mode="reference",
              precision="bf16_tc", want_scores=True)
    res, s = _run(engine, False, lambda: engine.plan(start, 0, **kw))
    assert s == "one_tile"
    assert np.isfinite(res["scores"]).all()
