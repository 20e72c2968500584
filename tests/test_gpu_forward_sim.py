"""ss_mpc_forward_sim / Engine.forward_sim / Dyn_Model.do_forward_sim from per-sequence start states, on the GPU.

Every rollout kernel family takes a per-row start (load_start in csrc/mpc_kernels.cuh, the kernels' ROWS flag).
Each case below names the kernel and instantiation it runs (the dispatch table of test_gpu_mpc_dims.py) and asserts
last_rollout_kernel().  The float64 reference is forward_sim_rows (test_forward_sim_host.py): the oracle's loop with
a [K, d] start.  Tolerances are those of the existing tests for the kernel: tcgen05 5e-4, FP32 1e-4 of the
per-dimension state scale (test_gpu_mpc_dims.py), float64 1e-10 (test_gpu_mpc_fp64.py); tcgen05 on a Dyn_Model
network over Pendulum data 2e-3 (test_gpu_mpc.py)."""
import os
from collections import namedtuple

import numpy as np
import pytest

from smartstartcontinuous_b200 import _lib
from smartstartcontinuous_b200 import synthetic as syn
from test_forward_sim_host import forward_sim_rows

pytestmark = pytest.mark.gpu

TC, QUAD = "mpc_rollout_tc_kernel", "mpc_rollout_tc_quad_kernel"
SIMT, THREAD, FP64 = "mpc_rollout_simt_kernel", "mpc_rollout_thread_kernel", "mpc_rollout_fp64_kernel"
TOL = {TC: 5e-4, QUAD: 5e-4, SIMT: 1e-4, THREAD: 1e-4, FP64: 1e-10}
TC_STATE_RTOL_DYN = 2e-3     # tcgen05 on Dyn_Model-initialised Pendulum networks (test_gpu_mpc.py TC_STATE_RTOL)

Row = namedtuple("Row", "d da L h kernel inst precision")
ROWS = [
    Row(1, 2, 2, 64, TC, "<4,2,16>", "bf16_tc"),
    Row(3, 1, 2, 128, TC, "<4,3,16>", "bf16_tc"),
    Row(3, 2, 2, 500, TC, "<4,3,32>", "bf16_tc"),
    Row(4, 1, 2, 256, TC, "<4,4,32>", "bf16_tc"),
    Row(5, 2, 2, 128, TC, "<8,8,32>", "bf16_tc"),
    Row(2, 3, 2, 500, QUAD, "<4,2,32>", "bf16_tc"),
    Row(3, 2, 2, 500, QUAD, "<4,3,32>", "bf16_tc"),
    Row(4, 6, 2, 500, QUAD, "<4,4,32>", "bf16_tc"),
    Row(3, 3, 2, 100, SIMT, "<4>", "fp32"),
    Row(6, 2, 3, 64, SIMT, "<8>", "fp32"),
    Row(32, 8, 1, 96, SIMT, "<32>", "fp32"),
    Row(2, 1, 1, 32, THREAD, "<4,32>", "fp32"),
    Row(7, 3, 1, 64, THREAD, "<8,64>", "fp32"),
    Row(3, 2, 2, 64, FP64, "<4>", "fp64"),
]
K_ROWS, H_ROWS = 1003, 10        # 8 tiles of 128 rows, the last one ragged; the last warp of 32 partial


def _row_id(r):
    return "%s%s-d%d-da%d-L%d-h%d" % (r.kernel.split("_")[2], r.inst, r.d, r.da, r.L, r.h)


Problem = namedtuple("Problem", "w b norm starts acts")


def _problem(r, K=K_ROWS, H=H_ROWS, seed=0):
    """A random model of the row's shape; start states spread over 2.5 standard deviations of mean_x."""
    rng = np.random.default_rng(7919 * r.d + 101 * r.da + 13 * r.L + r.h + seed)
    w, b = syn.xavier_mlp(rng, r.d, r.da, r.L, r.h, scale=0.5)
    norm = dict(mean_x=rng.normal(size=r.d), std_x=rng.uniform(0.5, 2.0, r.d), mean_y=np.zeros(r.da),
                std_y=np.full(r.da, 1 / np.sqrt(3.0)), mean_z=0.05 * rng.normal(size=r.d),
                std_z=rng.uniform(0.05, 0.2, r.d))
    starts = norm["mean_x"] + 2.5 * norm["std_x"] * rng.normal(size=(K, r.d))
    return Problem(w, b, norm, starts, rng.uniform(-1, 1, (K, H, r.da)))


def _run(engine, r, fn):
    """fn() with the pair / quad choice forced for the tcgen05 rows; asserts the row's kernel ran."""
    quad = {TC: "0", QUAD: "1"}.get(r.kernel)
    old = os.environ.get("SS_TC_QUAD")
    if quad is not None:
        os.environ["SS_TC_QUAD"] = quad
    try:
        out = fn()
    finally:
        if quad is not None:
            if old is None:
                os.environ.pop("SS_TC_QUAD", None)
            else:
                os.environ["SS_TC_QUAD"] = old
    assert engine.last_rollout_kernel() == r.kernel
    return out


def _fsim(engine, r, starts, acts, **kw):
    return _run(engine, r, lambda: engine.forward_sim(starts, acts, r.precision, **kw))


def _rel_err(got, want, norm):
    scale = np.maximum(np.abs(want).max(axis=(0, 1)), np.asarray(norm["std_x"], dtype=np.float64))
    return (np.abs(got - want).max(axis=(0, 1)) / scale).max()


def _check_start_rows(r, got, starts):
    """t = 0 is each row's own start: exactly for float64, rounded to float otherwise."""
    want = starts if r.kernel == FP64 else starts.astype(np.float32).astype(np.float64)
    np.testing.assert_array_equal(got[0], want)


def _plan_of(p):
    return np.stack([p.norm["mean_x"], p.norm["mean_x"] + p.norm["std_x"]]), np.array([1.0, 0.0]), p.norm["std_x"]


@pytest.mark.parametrize("r", ROWS, ids=_row_id)
def test_per_row_starts_against_float64_oracle(engine, r):
    p = _problem(r)
    engine.set_model(p.w, p.b, p.norm)
    got = _fsim(engine, r, p.starts, p.acts)
    assert got.shape == (H_ROWS + 1, K_ROWS, r.d)
    want = forward_sim_rows(p.starts, p.acts, p.w, p.b, p.norm)
    assert _rel_err(got, want, p.norm) <= TOL[r.kernel]
    _check_start_rows(r, got, p.starts)
    # negative control: a kernel that ignored the per-row starts would compute this, far outside the tolerance
    wrong = forward_sim_rows(np.tile(p.starts[0], (K_ROWS, 1)), p.acts, p.w, p.b, p.norm)
    assert _rel_err(got, wrong, p.norm) > 10 * TOL[r.kernel]


@pytest.mark.parametrize("r", ROWS, ids=_row_id)
def test_per_row_starts_are_bitwise_consistent(engine, r):
    """K equal rows, one shared start and the decision rollout's trajectories are the same bits; permuting starts
    and actions together permutes the output rows bit for bit."""
    p = _problem(r, seed=1)
    engine.set_model(p.w, p.b, p.norm)
    s = p.starts[3]
    rows = _fsim(engine, r, np.tile(s, (K_ROWS, 1)), p.acts)
    shared = _fsim(engine, r, s, p.acts)
    engine.set_plan(*_plan_of(p))
    _run(engine, r, lambda: engine.rollout(s, 0, actions=p.acts, penalty_mode="reference", precision=r.precision))
    decision = engine.get_states()
    np.testing.assert_array_equal(rows, shared)
    np.testing.assert_array_equal(rows, decision)
    full = _fsim(engine, r, p.starts, p.acts)
    perm = np.random.default_rng(5).permutation(K_ROWS)
    np.testing.assert_array_equal(_fsim(engine, r, p.starts[perm], p.acts[perm]), full[:, perm])


def test_chunked_host_upload(engine):
    """bf16_tc with host actions and many waves of tiles: the actions are uploaded in chunks and every chunk is
    launched with its tile offset; the start rows are indexed by the batch-local sequence number."""
    r = Row(3, 1, 2, 500, TC, "<4,3,16>", "bf16_tc")
    K, H = 131072, 20
    p = _problem(r, K=K, H=H)
    engine.set_model(p.w, p.b, p.norm)
    got = _fsim(engine, r, p.starts, p.acts)
    _check_start_rows(r, got, p.starts)
    idx = np.union1d(np.random.default_rng(2).choice(K, 4096, replace=False), [0, K - 1])
    want = forward_sim_rows(p.starts[idx], p.acts[idx], p.w, p.b, p.norm)
    assert _rel_err(got[:, idx], want, p.norm) <= TOL[TC]


@pytest.mark.parametrize("r", [ROWS[2], ROWS[8], ROWS[-1]], ids=_row_id)
def test_device_actions(engine, r):
    """numpy's MT19937 draw made on the device (mt19937_uniform) gives the bits of the same draw from the host."""
    p = _problem(r)
    engine.set_model(p.w, p.b, p.norm)
    lo, hi = -np.ones(r.da), np.ones(r.da)
    rs = np.random.RandomState(11)
    st = rs.get_state()
    host = rs.uniform(lo, hi, (K_ROWS, H_ROWS, r.da))
    ptr = engine.mt19937_uniform(st, K_ROWS * H_ROWS * r.da, lo, hi)
    dev = _fsim(engine, r, p.starts, None, actions_dev=ptr, K=K_ROWS, H=H_ROWS)
    np.testing.assert_array_equal(dev, _fsim(engine, r, p.starts, host))


def test_fresh_engine_needs_only_a_model():
    from smartstartcontinuous_b200.engine import Engine
    r = ROWS[2]
    p = _problem(r)
    eng = Engine(0)
    try:
        eng.set_model(p.w, p.b, p.norm)
        got = _fsim(eng, r, p.starts, p.acts)
        assert _rel_err(got, forward_sim_rows(p.starts, p.acts, p.w, p.b, p.norm), p.norm) <= TOL[TC]
        np.testing.assert_array_equal(eng.get_states(), got)
    finally:
        eng.close()


@pytest.mark.parametrize("r", [ROWS[2], ROWS[6], ROWS[8], ROWS[-1]], ids=_row_id)
def test_decision_unchanged_by_forward_sim(engine, r):
    """A decision after a forward simulation is the bits of the same decision before it; in between the context
    holds the forward simulation: its kernel, its states, and no decision to finish, replay or all-reduce."""
    p = _problem(r)
    engine.set_model(p.w, p.b, p.norm)
    engine.set_plan(*_plan_of(p))
    plan = lambda: _run(engine, r, lambda: engine.plan(p.starts[0], 0, actions=p.acts, precision=r.precision,
                                                       want_scores=True))
    before = plan()
    fs = _fsim(engine, r, p.starts, p.acts)
    np.testing.assert_array_equal(engine.get_states(), fs)
    lib, h = engine._lib, engine._h
    assert lib.ss_mpc_finish(h, None, None, None) == _lib.SS_ESTATE
    assert lib.ss_mpc_finish_package(h, 0, None, None) == _lib.SS_ESTATE
    assert lib.ss_mpc_replay(h, 0, None, None) == _lib.SS_ESTATE
    assert lib.ss_mpc_projection_sums(h, None, None) == _lib.SS_ESTATE
    assert engine.last_rollout_kernel() == r.kernel
    after = plan()
    assert after["best_k"] == before["best_k"] and after["best_score"] == before["best_score"]
    for key in ("scores", "best_sequence", "best_path"):
        np.testing.assert_array_equal(after[key], before[key])
    engine.finish_package()          # the decision state is back


# ---- Dyn_Model.do_forward_sim ------------------------------------------------------------------------------------
def _pendulum_stats(rng, episodes=12, steps=200):
    obs, act = syn.pendulum_rollouts(rng, episodes, steps)
    xs = np.concatenate([o[:-1] for o in obs]); ys = np.concatenate(list(act)); zs = np.concatenate([o[1:] - o[:-1] for o in obs])
    mean = dict(mean_x=xs.mean(0), mean_y=ys.mean(0), mean_z=zs.mean(0))
    std = dict(std_x=xs.std(0), std_y=ys.std(0), std_z=zs.std(0))
    inputs = np.concatenate([(xs - mean["mean_x"]) / std["std_x"], (ys - mean["mean_y"]) / std["std_y"]], axis=1)
    outputs = (zs - mean["mean_z"]) / std["std_z"]
    return obs, act, mean, std, inputs, outputs


def _dyn_model(engine, mean, std, precision="fp32", seed=0):
    from smartstartcontinuous_b200.dynamics_model import Dyn_Model
    return Dyn_Model(4, 3, None, 1e-3, 512, 2, 64, mean["mean_x"], mean["mean_y"], mean["mean_z"], std["std_x"],
                     std["std_y"], std["std_z"], "float64", False, engine=engine, seed=seed, precision=precision)


def test_dyn_model_call_forms(engine):
    rng = np.random.default_rng(4)
    obs, _, mean, std, _, _ = _pendulum_stats(rng)
    m = _dyn_model(engine, mean, std)
    N, H = 257, 9
    starts = obs[:, :, :].reshape(-1, 3)[rng.choice(obs.shape[0] * obs.shape[1], N, replace=False)]
    y = rng.uniform(-2, 2, (N, H, 1))
    w, b = m.export()

    tiled = np.stack(m.do_forward_sim([starts[0], 0], y, True))
    np.testing.assert_array_equal(tiled, engine.forward_sim(starts[0], y))
    assert _rel_err(tiled, forward_sim_rows(np.tile(starts[0], (N, 1)), y, w, b, m.norm()), m.norm()) <= TOL[SIMT]

    rows = np.stack(m.do_forward_sim(starts, y, True))
    np.testing.assert_array_equal(rows, engine.forward_sim(starts, y))
    assert _rel_err(rows, forward_sim_rows(starts, y, w, b, m.norm()), m.norm()) <= TOL[SIMT]
    np.testing.assert_array_equal(np.stack(m.do_forward_sim([s for s in starts], y, True)), rows)

    # a [2, d] array is the reference's [state, 0] test too: row 0 starts every sequence
    np.testing.assert_array_equal(np.stack(m.do_forward_sim(starts[:2], y, True)), tiled)

    for bad in (starts[:N - 1], np.concatenate([starts, starts[:, :1]], axis=1)):
        with pytest.raises(ValueError):
            m.do_forward_sim(bad, y, True)

    single = np.stack(m.do_forward_sim([starts[0], 0], y[0], False))
    np.testing.assert_array_equal(single, engine.forward_sim(starts[0], y[:1])[:, 0])

    f64 = np.stack(m.do_forward_sim(starts, y, True, precision="fp64"))
    assert engine.last_rollout_kernel() == FP64
    np.testing.assert_array_equal(f64[0], starts)
    assert _rel_err(f64, forward_sim_rows(starts, y, w, b, m.norm()), m.norm()) <= TOL[FP64]


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_dyn_model_after_device_training(engine, precision):
    """Per-sequence forward simulation of a model trained on the device, against the oracle on its exported
    weights: FP32 training rolls out in FP32, FP64 training with precision="fp64" in float64."""
    rng = np.random.default_rng(3)
    obs, _, mean, std, inputs, outputs = _pendulum_stats(rng)
    try:
        m = _dyn_model(engine, mean, std, precision=precision)
        engine.dyn_reset_optimizer()
        m.train(inputs[:1800], outputs[:1800], inputs[1800:], outputs[1800:], 2, None, 0.9, save_results=False)
        w, b = m.export()
        N, H = 300, 7
        starts = obs[:, 5:-1:8].reshape(-1, 3)[:N]
        y = rng.uniform(-2, 2, (N, H, 1))
        got = np.stack(m.do_forward_sim(starts, y, True, precision=precision))
        assert engine.last_rollout_kernel() == (FP64 if precision == "fp64" else SIMT)
        assert _rel_err(got, forward_sim_rows(starts, y, w, b, m.norm()), m.norm()) <= TOL[FP64 if precision == "fp64" else SIMT]
    finally:
        engine.dyn_set_precision("fp32")


@pytest.mark.parametrize("precision", ["fp32", "auto", "fp64"])
def test_k_step_validation_workload(engine, precision):
    """Multi-step prediction from every window of validation rollouts (the states_val / controls_val of
    NND_MB_agent): 20 Pendulum rollouts of 333 steps, every start t < 333 - H a sequence of H = 10 steps."""
    rng = np.random.default_rng(8)
    _, _, mean, std, _, _ = _pendulum_stats(rng)
    states_val, controls_val = syn.pendulum_rollouts(rng, 20, 333)
    H = 10
    starts = states_val[:, :333 - H].reshape(-1, 3)
    y = np.stack([controls_val[e, t:t + H] for e in range(20) for t in range(333 - H)])
    m = _dyn_model(engine, mean, std, seed=2)
    w, b = m.export()
    got = np.stack(m.do_forward_sim(starts, y, True, precision=precision))
    kernel = {"fp32": SIMT, "fp64": FP64, "auto": TC if engine.tc_supported() else SIMT}[precision]
    assert engine.last_rollout_kernel() == kernel
    assert got.shape == (H + 1, 20 * (333 - H), 3)
    # tcgen05: the bound tests/test_gpu_mpc.py sets for Pendulum-type networks (TC_STATE_RTOL); Dyn_Model's Xavier
    # weights and biases and angular velocities up to ~10 give bf16 errors above the small-weight problems of
    # test_gpu_mpc_dims.py (1.3e-3 of the scale measured on an NVIDIA B200, power limit 1000 W)
    tol = TC_STATE_RTOL_DYN if kernel == TC else TOL[kernel]
    assert _rel_err(got, forward_sim_rows(starts, y, w, b, m.norm()), m.norm()) <= tol
    wrong = forward_sim_rows(np.tile(starts[0], (len(starts), 1)), y, w, b, m.norm())
    assert _rel_err(got, wrong, m.norm()) > 10 * tol


def test_errors(engine):
    from smartstartcontinuous_b200.engine import Engine
    r = ROWS[8]
    p = _problem(r)
    engine.set_model(p.w, p.b, p.norm)
    with pytest.raises(ValueError):                    # n_starts = 3, K = 1003
        engine.forward_sim(p.starts[:3], p.acts)
    with pytest.raises(ValueError):
        engine.forward_sim(p.starts[0, :2], p.acts)     # [d - 1]
    bad = p.starts.copy()
    bad[17, 1] = np.nan
    with pytest.raises(ValueError):
        engine.forward_sim(bad, p.acts)
    lib, h = engine._lib, engine._h
    K, H = p.acts.shape[:2]
    out = np.empty((H + 1, K, r.d))
    st, acts = np.ascontiguousarray(p.starts), np.ascontiguousarray(p.acts)
    call = lambda s, n, k, hh, a, o: lib.ss_mpc_forward_sim(h, s, n, k, hh, a, 0, o)
    assert call(None, K, K, H, acts.ctypes.data, out.ctypes.data) == _lib.SS_EINVAL
    assert call(st.ctypes.data, K, K, H, None, out.ctypes.data) == _lib.SS_EINVAL
    assert call(st.ctypes.data, K, K, H, acts.ctypes.data, None) == _lib.SS_EINVAL
    assert call(st.ctypes.data, 2, K, H, acts.ctypes.data, out.ctypes.data) == _lib.SS_EINVAL
    assert call(st.ctypes.data, 1, 0, H, acts.ctypes.data, out.ctypes.data) == _lib.SS_EINVAL
    assert call(st.ctypes.data, 1, K, 0, acts.ctypes.data, out.ctypes.data) == _lib.SS_EINVAL
    assert call(st.ctypes.data, K, K, H, acts.ctypes.data, out.ctypes.data) == _lib.SS_OK
    fresh = Engine(0)
    try:
        assert fresh._lib.ss_mpc_forward_sim(fresh._h, st.ctypes.data, K, K, H, acts.ctypes.data, 0,
                                             out.ctypes.data) == _lib.SS_ESTATE
        with pytest.raises(RuntimeError):
            fresh.forward_sim(p.starts, p.acts)
    finally:
        fresh.close()
