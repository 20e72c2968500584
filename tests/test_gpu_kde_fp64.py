"""The float64 selection (ss_kde_set_precision(SS_PRECISION_FP64), csrc/kde_fp64.cu) against scipy.stats.gaussian_kde
itself and numpy's UCB expression with float32 values: densities to 1e-12 relative and scipy's choice wherever the
top-two gap is larger than that."""
import random

import numpy as np
import pytest

from conftest import load_golden
from oracle import kde_oracle
from smartstartcontinuous_b200 import synthetic as syn
from smartstartcontinuous_b200.distributed import argmax_pick, shard_bounds

pytestmark = pytest.mark.gpu

RTOL = 1e-12


@pytest.fixture(scope="module")
def eng64():
    """A context of its own, set to FP64: the session's `engine` stays in the default precision that the other
    files' tests assume."""
    from smartstartcontinuous_b200.engine import Engine
    eng = Engine(0)
    eng.kde_set_precision("fp64")
    yield eng
    eng.close()


def numpy_ucb(dens, values, n, volume, alpha, beta):
    """smartexplorationcontinuous.py:275-279 as numpy evaluates it: `values` is float32, so alpha * values is a
    float32 product."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return alpha * np.asarray(values, dtype=np.float32) + np.sqrt((beta * np.log(n)) / (n * (dens * volume)))


def ucb_bound(want, values, alpha):
    """RTOL * (|alpha V| + bonus): each term is good to RTOL, not their difference when they cancel."""
    av = (alpha * np.asarray(values, dtype=np.float32)).astype(np.float64)
    with np.errstate(invalid="ignore"):
        return RTOL * (np.abs(av) + np.abs(want - av))


def assert_ucb_close(ucb, want, values, alpha):
    finite = np.isfinite(want)
    assert np.all(np.abs(ucb[finite] - want[finite]) <= ucb_bound(want, values, alpha)[finite])
    assert np.array_equal(ucb[~finite], want[~finite], equal_nan=True)


def top_two_gap(ucb):
    o = np.sort(ucb[np.isfinite(ucb)])[::-1]
    return (o[0] - o[1]) / abs(o[0])


def select(eng, data, q, vals, n, volume=1.0, alpha=1.0, beta=2.0):
    return eng.select_start(data, q, vals, n, volume, alpha, beta, want_density=True, want_ucb=True)


def random_case(d, n, m, seed):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(d, d)) / np.sqrt(d) + 2 * np.eye(d)
    data = rng.normal(size=(n, d)) @ A + rng.normal(size=d) * 5
    q = data[rng.choice(n, m, replace=False)] + 0.05 * rng.normal(size=(m, d))
    vals = rng.normal(size=m).astype(np.float32)
    return data, q, vals


@pytest.mark.parametrize("name", ["kde_pendulum.npz", "kde_mountaincar.npz"])
def test_goldens(eng64, name):
    g = load_golden(name)
    best, best_ucb, dens, ucb = select(eng64, g["in_all_states"], g["in_queries"], g["in_values"],
                                       int(g["in_n_transitions"]), float(g["in_volume"]), float(g["in_alpha"]),
                                       float(g["in_beta"]))
    np.testing.assert_allclose(dens, g["out_density"], rtol=RTOL, atol=0)
    np.testing.assert_allclose(ucb, g["out_ucb"], rtol=RTOL, atol=0)
    assert best == int(g["out_best_j"]) and best_ucb == ucb[best]


# seeds fixed so that scipy's top-two relative UCB gap exceeds 1e-11 in every case (asserted)
@pytest.mark.parametrize("d,n,m", [(1, 700, 33), (2, 5000, 1000), (3, 20001, 2049), (4, 3000, 257), (6, 4000, 100),
                                   (9, 2500, 64), (17, 2000, 40), (24, 3000, 200), (32, 2500, 150)])
def test_random_shapes_vs_scipy(eng64, d, n, m):
    data, q, vals = random_case(d, n, m, d * 1000 + n)
    best, best_ucb, dens, ucb = select(eng64, data, q, vals, n - 1, 0.37)
    odens = kde_oracle.scipy_density(data, q)
    oucb = numpy_ucb(odens, vals, n - 1, 0.37, 1.0, 2.0)
    assert top_two_gap(oucb) > 1e-11
    np.testing.assert_allclose(dens, odens, rtol=RTOL, atol=0)
    assert_ucb_close(ucb, oucb, vals, 1.0)
    assert best == int(np.argmax(oucb)) and best_ucb == ucb[best]


def test_alpha_times_values_is_a_float32_product(eng64):
    """alpha = 0.7 with float32 values: numpy rounds 0.7 * v to float32 before adding the bonus.  The same product
    in double differs from it by ~1e-8 relative, far outside the bound."""
    data, q, _ = random_case(3, 6000, 700, 12)
    rng = np.random.default_rng(13)
    vals = (rng.normal(size=len(q)) * 10.0 ** rng.uniform(-3, 3, len(q))).astype(np.float32)
    _, _, dens, ucb = select(eng64, data, q, vals, 5999, 1.0, 0.7, 2.0)
    want = numpy_ucb(kde_oracle.scipy_density(data, q), vals, 5999, 1.0, 0.7, 2.0)
    assert_ucb_close(ucb, want, vals, 0.7)
    in_double = 0.7 * vals.astype(np.float64) + (want - (0.7 * vals).astype(np.float64))
    assert np.any(np.abs(in_double - want) > ucb_bound(want, vals, 0.7))


def test_near_tie_and_exact_tie(eng64):
    """alpha = 0: the top UCB is the lowest density.  Two candidates in a sparse region, 1e-9 apart in density, the
    later one lower: scipy picks the later one, and so must FP64.  Duplicated rows with equal values: the first."""
    rng = np.random.default_rng(21)
    data = rng.normal(size=(5000, 2))
    a = np.array([3.0, 1.0])
    da, dd = kde_oracle.scipy_density(data, np.stack([a, a * (1 + 1e-4)]))
    t = 1e-4 * 1e-9 / ((da - dd) / da)                  # density falls linearly with the step this close
    core = data[np.linalg.norm(data, axis=1) < 1.5][:200]          # dense: low bonus
    cands = np.concatenate([core, [a, a * (1 + t)]])
    vals = np.zeros(len(cands), dtype=np.float32)
    odens = kde_oracle.scipy_density(data, cands)
    oucb = numpy_ucb(odens, vals, 4999, 1.0, 0.0, 2.0)
    assert 1e-10 < (odens[200] - odens[201]) / odens[200] < 1e-8
    assert int(np.argmax(oucb)) == 201
    best, _, dens, _ = select(eng64, data, cands, vals, 4999, 1.0, 0.0, 2.0)
    np.testing.assert_allclose(dens, odens, rtol=RTOL, atol=0)
    assert best == 201

    dup = np.concatenate([data[:50], [1.3 * a] * 3, data[50:60], [1.3 * a]])
    vals = np.zeros(len(dup), dtype=np.float32)
    best, best_ucb, _, ucb = select(eng64, data, dup, vals, 4999, 1.0, 1.0, 2.0)
    assert best == 50 and ucb[50] == ucb[51] == ucb[52] == ucb[-1] == best_ucb


def test_underflow_gives_zero_density_and_infinite_ucb(eng64):
    """Queries so far away that scipy's density is exactly 0: density 0, ucb +inf, the first inf wins; the finite
    ones (kept >= 1e-290, away from the subnormal edge) stay within the bound."""
    rng = np.random.default_rng(5)
    data = rng.normal(size=(4000, 3))
    far = np.array([[40.0, 0, 0], [0, 45.0, 0], [30.0, 30.0, 0.0]])
    mid = np.array([[4.0, 0, 0], [0, 4.5, 0], [3.0, 3.0, 0.0]])
    q = np.concatenate([data[:30], mid, far[:1], data[30:40], far[1:]])
    vals = rng.normal(size=len(q)).astype(np.float32)
    odens = kde_oracle.scipy_density(data, q)
    zero = odens == 0
    assert zero.sum() == 3 and np.all(odens[~zero] >= 1e-290)
    oucb = numpy_ucb(odens, vals, 3999, 1.0, 1.0, 2.0)
    best, best_ucb, dens, ucb = select(eng64, data, q, vals, 3999)
    assert np.all(dens[zero] == 0) and np.all(ucb[zero] == np.inf)
    np.testing.assert_allclose(dens[~zero], odens[~zero], rtol=RTOL, atol=0)
    assert_ucb_close(ucb, oucb, vals, 1.0)
    assert best == 33 == int(np.argmax(oucb)) and best_ucb == np.inf


def test_first_nan_wins(eng64):
    rng = np.random.default_rng(6)
    data = rng.normal(size=(1000, 2))
    q = data[rng.choice(1000, 300, replace=False)]
    vals = rng.normal(size=300).astype(np.float32)
    vals[137] = np.nan
    vals[250] = np.nan
    best, best_ucb, _, _ = select(eng64, data, q, vals, 999)
    assert best == 137 and np.isnan(best_ucb)


def test_errors(eng64):
    rng = np.random.default_rng(7)
    data = rng.normal(size=(100, 3))
    flat = data.copy()
    flat[:, 2] = flat[:, 0]
    with pytest.raises(np.linalg.LinAlgError):
        eng64.select_start(flat, flat[:5], np.zeros(5, np.float32), 99)
    with pytest.raises(ValueError):
        eng64.select_start(data[:3], data[:2], np.zeros(2, np.float32), 2)          # n <= d
    with pytest.raises(ValueError):
        eng64.kde_set_precision("fp16")
    with pytest.raises(ValueError):
        eng64.kde_set_precision("bf16_tc")
    best, _, dens, _ = select(eng64, data, data[:20], np.zeros(20, np.float32), 99)       # still usable, still FP64
    np.testing.assert_allclose(dens, kde_oracle.scipy_density(data, data[:20]), rtol=RTOL, atol=0)


def test_a_querys_density_does_not_depend_on_its_batch(eng64):
    """The point slices are cut from N alone: a query's density is the same bits in a repeated call, in another
    batch, at another position, and on either half of a two-way query shard; the merged shard picks equal the
    full call's pick."""
    all_states, s2, _ = syn.pendulum_buffer(200_000, seed=4)
    rng = np.random.default_rng(4)
    q = s2[rng.choice(200_000, 3000, replace=False)]
    vals = syn.critic_like_values(q)
    full = select(eng64, all_states, q, vals, 200_000)
    again = select(eng64, all_states, q, vals, 200_000)
    assert full[:2] == again[:2]
    np.testing.assert_array_equal(again[2], full[2])
    np.testing.assert_array_equal(again[3], full[3])
    head = select(eng64, all_states, q[:1234], vals[:1234], 200_000)
    tail = select(eng64, all_states, q[1234:], vals[1234:], 200_000)
    np.testing.assert_array_equal(np.concatenate([head[2], tail[2]]), full[2])
    perm = rng.permutation(len(q))
    shuffled = select(eng64, all_states, q[perm], vals[perm], 200_000)
    np.testing.assert_array_equal(shuffled[2], full[2][perm])
    picks, ucbs = [], []
    for r in range(2):
        off, cnt = shard_bounds(len(q), 2, r)
        part = select(eng64, all_states, q[off:off + cnt], vals[off:off + cnt], 200_000)
        np.testing.assert_array_equal(part[2], full[2][off:off + cnt])
        picks.append(off + part[0])
        ucbs.append(part[1])
    w = argmax_pick(ucbs, picks)
    assert picks[w] == full[0] and ucbs[w] == full[1]


def test_mirror_matches_host_path_and_scipy(eng64):
    """select_start_mirror in FP64 fits from the mirror's rows: it equals select_start on the same data to 1e-13
    with the same pick, while the buffer grows, after it wraps, and after a rebuild -- and scipy to 1e-12."""
    from smartstartcontinuous_b200.replay_buffer import ReplayBuffer
    rng = np.random.default_rng(31)
    agent = object()
    rb = ReplayBuffer(agent, 3000)
    obs, _ = syn.pendulum_rollouts(rng, 30, 200)
    vals_all = rng.normal(size=4096).astype(np.float32)
    added = 0
    for ep, traj in enumerate(obs):
        rb.start_new_episode(agent)
        for t in range(len(traj) - 1):
            rb.add(agent, traj[t], np.zeros(1), 0.0, False, traj[t + 1])
            added += 1
        if ep in (3, 14, 22, 29):                          # grows, fills, wraps, wraps again
            ring = rb.state_ring()
            idx = rb.get_possible_smart_start_indices(500)
            vals = vals_all[:len(idx)]
            data, q = rb.get_all_states(), rb.states_s2(idx)
            want = select(eng64, data, q, vals, len(rb), 0.5)
            got = eng64.select_start_mirror(ring, idx, vals, len(rb), 0.5, 1.0, 2.0, want_density=True, want_ucb=True)
            np.testing.assert_allclose(got[2], want[2], rtol=1e-13, atol=0)
            assert got[0] == want[0]
            odens = kde_oracle.scipy_density(data, q)
            np.testing.assert_allclose(got[2], odens, rtol=RTOL, atol=0)
            assert_ucb_close(got[3], numpy_ucb(odens, vals, len(rb), 0.5, 1.0, 2.0), vals, 1.0)
    assert added > 3000
    rb._rebuild_mirror()
    idx = rb.get_possible_smart_start_indices(200)
    want = select(eng64, rb.get_all_states(), rb.states_s2(idx), vals_all[:len(idx)], len(rb), 0.5)
    got = eng64.select_start_mirror(rb.state_ring(), idx, vals_all[:len(idx)], len(rb), 0.5, 1.0, 2.0,
                                    want_density=True)
    np.testing.assert_allclose(got[2], want[2], rtol=1e-13, atol=0)
    assert got[0] == want[0]


def test_config2_seed0_is_the_float64_choice(eng64):
    """Config-2 size (100 001 points, 16 384 candidates), seed 0: the top two UCBs are 1.4e-5 apart relative, inside
    the default path's tolerance.  The FP64 pick is the float64 oracle's argmax over all candidates; densities
    match scipy on a 512-query subset."""
    all_states, s2, _ = syn.pendulum_buffer(100_000, seed=0)
    rng = np.random.default_rng(0)
    q = s2[rng.choice(100_000, 16_384, replace=False)]
    vals = syn.critic_like_values(q)
    best, best_ucb, dens, ucb = select(eng64, all_states, q, vals, 100_000)
    oucb = numpy_ucb(kde_oracle.kde_density(all_states, q), vals, 100_000, 1.0, 1.0, 2.0)
    assert top_two_gap(oucb) < 1e-4
    assert best == int(np.argmax(oucb)) and best_ucb == ucb[best]
    sub = np.sort(rng.choice(16_384, 512, replace=False))
    odens = kde_oracle.scipy_density(all_states, q[sub])
    np.testing.assert_allclose(dens[sub], odens, rtol=RTOL, atol=0)
    assert_ucb_close(ucb[sub], numpy_ucb(odens, vals[sub], 100_000, 1.0, 1.0, 2.0), vals[sub], 1.0)


@pytest.mark.parametrize("name,env,n,n_ss,seed", [("kde_pendulum.npz", "pendulum", 3000, 300, 0),
                                                  ("kde_mountaincar.npz", "mountaincar", 2000, 5000, 1)])
def test_smart_start_fp64_path_equals_the_references_from_the_seed(eng64, name, env, n, n_ss, seed):
    """SmartStartContinuous(kde_precision="fp64") from random.seed(seed) chooses the golden's buffer index, with
    the golden's UCB to 1e-12, and returns its path.  The agent sets the precision before every selection, so an
    engine left in FP32 by someone else does not matter."""
    from smartstartcontinuous_b200.smart_start import SmartStartContinuous
    from test_replay_buffer import _golden_buffer

    g = load_golden(name)
    rb, episodes = _golden_buffer(name, env, n, seed)
    d = episodes[0][0].shape[1]

    class Box:
        low, high, shape = np.array([-2.0]), np.array([2.0]), (1,)

    class Env:
        action_space = Box()

    class Base:
        replay_buffer = rb

        def set_replay_buffer_main_agent(self, main): pass
        def get_action(self, s): return np.zeros(1)
        def observe(self, *a): pass
        def start_new_episode(self, s): pass
        def end_episode(self): pass
        def get_param_dict(self): return {}
        def get_state_value(self, states): return syn.critic_like_values(np.asarray(states), seed + 7).reshape(-1, 1)

    rng = np.random.default_rng(0)
    td = dict(dataX=rng.normal(size=(64, d)), dataY=rng.normal(size=(64, 1)), dataZ=rng.normal(size=(64, d)))
    ss = SmartStartContinuous(Base(), Env(), None, n_ss=n_ss, print_ss_stuff=False, nnd_mb_num_fc_layers=1,
                              nnd_mb_depth_fc_layers=8, nnd_mb_verbose=False, engine=eng64,
                              nnd_mb_extra=dict(training_data=td), kde_precision="fp64")
    ss.nnd_mb_agent.radii = g["in_radii"] if len(g["in_radii"]) else None
    eng64.kde_set_precision("fp32")
    random.seed(seed)
    path = ss.get_smart_start_path()
    chosen, ucb = ss.last_selection
    assert chosen == int(g["out_chosen_buffer_index"])
    assert ucb == pytest.approx(float(g["out_ucb"][int(g["out_best_j"])]), rel=RTOL, abs=0)
    np.testing.assert_array_equal(np.asarray(path), g["out_path"])
    with pytest.raises(ValueError):
        SmartStartContinuous(Base(), Env(), None, engine=eng64, nnd_mb_verbose=False,
                             nnd_mb_extra=dict(training_data=td), kde_precision="fp16")


def test_switching_back_to_fp32_equals_a_fresh_context(eng64):
    from smartstartcontinuous_b200.engine import Engine
    data, q, vals = random_case(3, 20001, 2049, 3 * 1000 + 20001)
    fresh = Engine(0)
    try:
        want = select(fresh, data, q, vals, 20000, 0.37)
        eng64.kde_set_precision("fp32")
        got = select(eng64, data, q, vals, 20000, 0.37)
    finally:
        eng64.kde_set_precision("fp64")
        fresh.close()
    assert got[:2] == want[:2]
    np.testing.assert_array_equal(got[2], want[2])
    np.testing.assert_array_equal(got[3], want[3])
