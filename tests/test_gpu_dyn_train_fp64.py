"""The float64 device trainer (ss_dyn_set_precision(SS_PRECISION_FP64), csrc/dyn_train.cu) against the float64
numpy oracle of Dyn_Model.train's optimisation step: identical initial parameters and batches, so the two differ
only in the summation order of the GEMMs and of the batch reductions."""
import numpy as np
import numpy.random as npr
import pytest

from oracle import dyn_train_oracle as dto
from oracle import mpc_oracle
from smartstartcontinuous_b200 import _lib
from smartstartcontinuous_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

# Bounds against the oracle, relative to how far Adam moved each tensor (Frobenius, and per element against the
# largest element's movement); the FP32 trainer needs 3e-3 and 10 % here (tests/test_gpu_dyn_train.py).  Measured
# on a B200 over the four oracle cases: losses 9e-16, parameters 1.4e-15 (Frobenius) and 3.6e-14 (element), eval
# loss 2.3e-16 (scripts/dev/dyn_fp64_errors.py -> profiles/r04_dyn_fp64_errors.json).
PARAM_FROB = 1e-13
PARAM_ELEM = 1e-12
LOSS_RTOL = 1e-13


@pytest.fixture(autouse=True)
def _fp32_afterwards(engine):
    """The engine is shared by the whole session: leave its trainer in the default precision."""
    yield
    engine.dyn_set_precision("fp32")


def param_errors(got_list, want_list, init_list):
    """(worst Frobenius error / Frobenius movement, worst max element error / max element movement)."""
    frob = elem = 0.0
    for got, want, init in zip(got_list, want_list, init_list):
        moved = np.abs(want - init).max()
        assert moved > 0
        frob = max(frob, np.linalg.norm(got - want) / np.linalg.norm(want - init))
        elem = max(elem, np.abs(got - want).max() / moved)
    return frob, elem


def assert_params_close(got_list, want_list, init_list):
    frob, elem = param_errors(got_list, want_list, init_list)
    assert frob <= PARAM_FROB and elem <= PARAM_ELEM, (frob, elem)


def setup_fp64(engine, seed, d, da, L, h, n_old, n_new):
    rng = np.random.default_rng(seed)
    w, b = syn.xavier_mlp(rng, d, da, L, h)
    norm = dict(mean_x=np.zeros(d), std_x=np.ones(d), mean_y=np.zeros(da), std_y=np.ones(da), mean_z=np.zeros(d),
                std_z=np.ones(d))
    X = rng.normal(size=(n_old + n_new, d + da))
    Z = np.tanh(X[:, :d] * 0.7 + 0.3 * X[:, d:d + 1]) + 0.05 * rng.normal(size=(n_old + n_new, d))
    engine.set_model(w, b, norm)
    engine.dyn_set_precision("fp64")
    engine.dyn_reset_optimizer()
    engine.dyn_set_data(0, X[:n_old], Z[:n_old])
    engine.dyn_set_data(1, X[n_old:], Z[n_old:])
    return w, b, norm, X, Z


# the four cases of test_gpu_dyn_train.py::test_device_training_matches_float64_oracle:
# (d, da, L, h, batch, fraction of new rows, Adam steps)
ORACLE_CASES = [(3, 1, 2, 500, 512, 0.9, 40), (2, 1, 1, 32, 512, 0.9, 120), (3, 1, 3, 64, 200, 0.5, 60),
                (2, 1, 2, 500, 512, 1.0, 12)]


def oracle_case(engine, cfg):
    """Train one case on the device in float64 and with the oracle; returns the measured errors."""
    d, da, L, h, batch, frac, steps = cfg
    n_old, n_new = 3000, 1500
    w, b, norm, X, Z = setup_fp64(engine, 5, d, da, L, h, n_old, n_new)
    ow, ob = [a.copy() for a in w], [a.copy() for a in b]
    state = dto.AdamState(ow, ob)
    npr.seed(11)
    if frac < 1.0:
        io, inw = dto.epoch_batches(n_old, n_new, batch, frac)
    else:
        nb = n_new // batch
        io, inw = np.empty((nb, 0), dtype=np.int64), np.arange(nb * batch).reshape(nb, batch)
    io, inw = io[:steps], inw[:steps]
    want_losses = dto.train_batches(ow, ob, state, X[:n_old], Z[:n_old], X[n_old:], Z[n_old:], io, inw, 1e-3)
    got_losses = engine.dyn_train_batches(io, inw, 1e-3)
    gw, gb = engine.dyn_get_params()
    loss_dev, nb = engine.dyn_eval_loss(0, batch)
    assert nb == n_old // batch
    want_eval = np.mean([dto.loss_and_grads(X[i * batch:(i + 1) * batch], Z[i * batch:(i + 1) * batch], ow, ob)[0]
                         for i in range(nb)])
    frob, elem = param_errors(gw + gb, ow + ob, w + b)
    return dict(loss_rel=float(np.max(np.abs(got_losses - want_losses) / np.abs(want_losses))), param_frob=frob,
                param_elem=elem, eval_loss_rel=abs(loss_dev - want_eval) / want_eval)


@pytest.mark.parametrize("cfg", ORACLE_CASES)
def test_fp64_training_matches_float64_oracle(engine, cfg):
    """The BASELINE network (2x500, batch 512), the example's default (1x32), a 3-layer case with a ragged batch
    and the new-data-only branch, trained in float64."""
    e = oracle_case(engine, cfg)
    assert e["loss_rel"] <= LOSS_RTOL, e
    assert e["param_frob"] <= PARAM_FROB and e["param_elem"] <= PARAM_ELEM, e
    assert e["eval_loss_rel"] <= LOSS_RTOL, e


def _plan_problem(engine):
    from smartstartcontinuous_b200.nnd_mb_agent import plan_from_path
    obs, _ = syn.pendulum_rollouts(np.random.default_rng(0), 1, 80)
    plan = plan_from_path(list(obs[0][:60]), mean_per_stepsize=1, std_per_stepsize=1, stepsizes_in_waypoint_radii=1,
                          path_shortcutting=True, theta=1, steps_per_waypoint=1)
    engine.set_plan(plan["desired_states"], plan["distances_left"], plan["radii"])
    return obs[0][0], plan, np.random.RandomState(3).uniform(-2, 2, (700, 6, 1))


def test_fp64_continuity_commit_and_export(engine):
    """Two training calls continue one optimisation; after ss_dyn_commit the fp64 rollout gives the oracle-trained
    model's scores and decision, and set_model with the exported parameters reproduces the committed fp64, fp32 and
    bf16_tc decisions bit for bit (commit and export hand over the same float64 masters)."""
    w, b, norm, X, Z = setup_fp64(engine, 7, 3, 1, 2, 500, 2000, 1000)
    ow, ob = [a.copy() for a in w], [a.copy() for a in b]
    state = dto.AdamState(ow, ob)
    npr.seed(2)
    io, inw = dto.epoch_batches(2000, 1000, 512, 0.9)
    dto.train_batches(ow, ob, state, X[:2000], Z[:2000], X[2000:], Z[2000:], io[:20], inw[:20], 1e-3)
    engine.dyn_train_batches(io[:8], inw[:8], 1e-3, want_losses=False)
    engine.dyn_train_batches(io[8:20], inw[8:20], 1e-3, want_losses=False)
    gw, gb = engine.dyn_get_params()
    assert_params_close(gw + gb, ow + ob, w + b)
    engine.dyn_commit()
    s0, plan, acts = _plan_problem(engine)
    o = mpc_oracle.plan(s0, acts, ow, ob, norm, plan["desired_states"], plan["distances_left"], plan["radii"], 0, .75, .5)
    o_init = mpc_oracle.plan(s0, acts, w, b, norm, plan["desired_states"], plan["distances_left"], plan["radii"], 0,
                             .75, .5)
    assert np.abs(o["scores"] - o_init["scores"]).max() > 1e-2          # training changed the predictions
    kw = dict(actions=acts, want_scores=True)
    committed = {p: engine.plan(s0, 0, precision=p, **kw) for p in ("fp64", "fp32", "bf16_tc")}
    res = committed["fp64"]
    assert (np.abs(res["scores"] - o["scores"]) / np.maximum(np.abs(o["scores"]), 1.0)).max() <= 1e-9
    assert res["best_k"] == int(np.argmax(o["scores"]))
    engine.set_model(gw, gb, norm)
    for p, want in committed.items():
        got = engine.plan(s0, 0, precision=p, **kw)
        np.testing.assert_array_equal(got["scores"], want["scores"], err_msg=p)
        assert got["best_k"] == want["best_k"], p


def _pendulum_data():
    rng = np.random.default_rng(3)
    obs, act = syn.pendulum_rollouts(rng, 12, 200)
    xs = np.concatenate([o[:-1] for o in obs]); ys = np.concatenate(list(act)); zs = np.concatenate([o[1:] - o[:-1] for o in obs])
    st = {k: v for k, v in zip(("mean_x", "mean_y", "mean_z"), (xs.mean(0), ys.mean(0), zs.mean(0)))}
    sd = {k: v for k, v in zip(("std_x", "std_y", "std_z"), (xs.std(0), ys.std(0), zs.std(0)))}
    inputs = np.concatenate([(xs - st["mean_x"]) / sd["std_x"], (ys - st["mean_y"]) / sd["std_y"]], axis=1)
    outputs = (zs - st["mean_z"]) / sd["std_z"]
    return rng, obs, st, sd, inputs, outputs


def _oracle_dyn_model_train(ow, ob, X_old, Z_old, X_new, Z_new, n_epochs, batch, frac, lr):
    """Dyn_Model.train's epochs with the oracle: the same npr draws in the same order, both branches."""
    state = dto.AdamState(ow, ob)
    n_old, n_new = len(X_old), len(X_new)
    n_n = n_new if n_new < batch * frac else int(batch * frac)
    new_order = np.arange(n_new)
    for _ in range(n_epochs):
        if batch - n_n <= 0:                                                    # new data only
            npr.choice(np.arange(n_old), size=(n_old,), replace=False)
            nb = n_new // n_n
            io, inw = np.empty((nb, 0), dtype=np.int64), new_order[:nb * n_n].reshape(nb, n_n)
            dto.train_batches(ow, ob, state, X_old, Z_old, X_new, Z_new, io, inw, lr)
            new_order = new_order[npr.permutation(n_new)]
        else:
            io, inw = dto.epoch_batches(n_old, n_new, batch, frac)
            dto.train_batches(ow, ob, state, X_old, Z_old, X_new, Z_new, io, inw, lr)


@pytest.mark.parametrize("frac, epochs", [(0.9, 4), (1.0, 6)])
def test_dyn_model_fp64_train_matches_oracle(engine, frac, epochs):
    """Dyn_Model(precision="fp64").train end to end, in the mixed and the new-data-only branch: the weights are the
    oracle's, run_validation gives the oracle's loss, and do_forward_sim rolls out the trained model."""
    from smartstartcontinuous_b200.dynamics_model import Dyn_Model
    rng, obs, st, sd, inputs, outputs = _pendulum_data()
    m = Dyn_Model(4, 3, None, 1e-3, 512, 2, 64, st["mean_x"], st["mean_y"], st["mean_z"], sd["std_x"], sd["std_y"],
                  sd["std_z"], "float64", False, engine=engine, seed=0, precision="fp64")
    engine.dyn_reset_optimizer()
    w0, b0 = m.export()
    ow, ob = [a.copy() for a in w0], [a.copy() for a in b0]
    npr.seed(0)
    _oracle_dyn_model_train(ow, ob, inputs[:1800], outputs[:1800], inputs[1800:], outputs[1800:], epochs, 512, frac,
                            1e-3)
    npr.seed(0)
    m.train(inputs[:1800], outputs[:1800], inputs[1800:], outputs[1800:], epochs, None, frac, save_results=False)
    w, b = m.export()
    assert_params_close(w + b, ow + ob, w0 + b0)
    val = m.run_validation(inputs[:1024], outputs[:1024], quiet=True)
    want = np.mean([dto.loss_and_grads(inputs[i:i + 512], outputs[i:i + 512], ow, ob)[0] for i in (0, 512)])
    assert val == pytest.approx(want, rel=LOSS_RTOL, abs=0)
    acts = rng.uniform(-2, 2, (5, 7, 1))
    want_states = mpc_oracle.forward_sim(obs[0][0], acts, ow, ob, m.norm())
    states = np.stack(m.do_forward_sim([obs[0][0], 0], acts, True))             # the FP32 rollout
    np.testing.assert_allclose(states, want_states, rtol=1e-4, atol=1e-5)
    states64 = engine.forward_sim(obs[0][0], acts, precision="fp64")
    np.testing.assert_allclose(states64, want_states, rtol=1e-9, atol=1e-12)


def test_switching_precision(engine):
    """A change of precision discards the trainer state: an FP32 run repeats bit for bit after an FP64 round,
    training without re-uploaded data fails cleanly, setting the current precision keeps the state, and values
    other than fp32 / fp64 are rejected."""
    w, b, norm, X, Z = setup_fp64(engine, 9, 2, 1, 2, 64, 1200, 600)
    npr.seed(4)
    io, inw = dto.epoch_batches(1200, 600, 256, 0.75)

    def fp32_run():
        engine.dyn_set_precision("fp32")
        engine.dyn_set_data(0, X[:1200], Z[:1200])
        engine.dyn_set_data(1, X[1200:], Z[1200:])
        losses = engine.dyn_train_batches(io[:10], inw[:10], 1e-3)
        return losses, engine.dyn_get_params()

    l1, (w1, b1) = fp32_run()
    engine.dyn_set_precision("fp64")
    with pytest.raises(ValueError, match="out of range"):                # the FP32 data sets are gone
        engine.dyn_train_batches(io[:1], inw[:1], 1e-3)
    engine.dyn_set_data(0, X[:1200], Z[:1200])
    engine.dyn_set_data(1, X[1200:], Z[1200:])
    straight = engine.dyn_train_batches(io[:6], inw[:6], 1e-3)
    ws, bs = engine.dyn_get_params()
    engine.dyn_reset_optimizer()
    first = engine.dyn_train_batches(io[:3], inw[:3], 1e-3)
    engine.dyn_set_precision("fp64")                                     # the current value: state kept
    second = engine.dyn_train_batches(io[3:6], inw[3:6], 1e-3)
    np.testing.assert_array_equal(np.concatenate([first, second]), straight)
    wk, bk = engine.dyn_get_params()
    for got, want in zip(wk + bk, ws + bs):
        np.testing.assert_array_equal(got, want)
    l2, (w2, b2) = fp32_run()
    np.testing.assert_array_equal(l2, l1)
    for got, want in zip(w2 + b2, w1 + b1):
        np.testing.assert_array_equal(got, want)
    for bad in ("bf16_tc", "auto", "fp16", 3):
        with pytest.raises(ValueError):
            engine.dyn_set_precision(bad)
    for code in (_lib.PRECISION_BF16_TC, _lib.PRECISION_AUTO, 7, -1):
        assert engine._lib.ss_dyn_set_precision(engine._h, code) == _lib.SS_EINVAL
    from smartstartcontinuous_b200.dynamics_model import Dyn_Model
    with pytest.raises(ValueError):
        Dyn_Model(3, 2, None, 1e-3, 256, 2, 64, np.zeros(2), np.zeros(1), np.zeros(2), np.ones(2), np.ones(1),
                  np.ones(2), "float64", False, engine=engine, seed=0, precision="fp16")
