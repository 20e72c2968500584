"""The MPC rollout kernels at every state and action dimension they accept, against the float64 oracle.

ss_mpc_set_model accepts 1 <= d <= 32 and 1 <= da <= 8.  Which kernel and which template instantiation rolls a
model out is decided by its shape (csrc/mpc_tc.cu, mpc_tc_quad.cu, mpc_simt.cu):

  tcgen05 (precision "bf16_tc", and "auto" whenever mpc_tc_shape_supported holds:
  L = 2, 64 <= h <= 510, d <= 8, dz + da <= 10).  Layer-1 layout: dz = 2 (d <= 2), 3 (d = 3), 4 (d = 4),
  8 (5 <= d <= 8) state inputs, action j in input dz + j; k1 = 16 K slots if 3 (dz + da) + 2 <= 16, else 32.

    shape rule                 (dz, k1)   pair kernel mpc_rollout_tc_kernel   quad kernel mpc_rollout_tc_quad_kernel
    d <= 2, da <= 2            (2, 16)    <4,2,16>                           <4,2,16>
    d <= 2, 3 <= da <= 8       (2, 32)    <4,2,32>                           <4,2,32>
    d = 3,  da = 1             (3, 16)    <4,3,16>                           <4,3,16>
    d = 3,  2 <= da <= 7       (3, 32)    <4,3,32>                           <4,3,32>
    d = 4,  da <= 6            (4, 32)    <4,4,32>                           <4,4,32>
    5 <= d <= 8, da <= 2       (8, 32)    <8,8,32>                           -

  The quad kernel serves d <= 4 when h + 2 pads to 512 (255 <= h <= 510) and the global batch fits its
  co-resident clusters; SS_TC_QUAD = 0 / 1 forces the pair / quad kernel.

  FP32 (precision "fp32", and "auto" for every other shape):
    L = 1, h <= 64, d <= 8     mpc_rollout_thread_kernel<4 if d <= 4 else 8, 32 if h <= 32 else 64>
    otherwise                  mpc_rollout_simt_kernel<4 if d <= 4, 8 if d <= 8, else 32>

Each row below names the instantiation it runs and why it is there.  The tcgen05 rows with da >= 2 also get a
host-only negative control: the oracle recomputed with the actions moved by one input slot (what a kernel
instantiated for another layer-1 layout computes) must miss the tolerance by at least 10x, so these rows can
see a layout mismatch."""
import os
from collections import namedtuple

import numpy as np
import numpy.random as npr
import pytest

from oracle import dyn_train_oracle as dto
from oracle import mpc_oracle, philox
from smartstartcontinuous_b200 import synthetic as syn

TC, QUAD = "mpc_rollout_tc_kernel", "mpc_rollout_tc_quad_kernel"
SIMT, THREAD = "mpc_rollout_simt_kernel", "mpc_rollout_thread_kernel"

Row = namedtuple("Row", "d da L h kernel inst why")

TC_ROWS = [
    Row(1, 2, 2, 64, TC, "<4,2,16>", "d = 1 and da = 2"),
    Row(2, 3, 2, 500, TC, "<4,2,32>", "d <= 2 with da >= 3: packed with dz = 2"),
    Row(1, 8, 2, 128, TC, "<4,2,32>", "all 10 layer-1 inputs used"),
    Row(3, 2, 2, 500, TC, "<4,3,32>", "d = 3 with da >= 2: packed with dz = 3"),
    Row(3, 7, 2, 100, TC, "<4,3,32>", "all 10 layer-1 inputs used"),
    Row(4, 1, 2, 256, TC, "<4,4,32>", "d = 4"),
    Row(4, 6, 2, 500, TC, "<4,4,32>", "d = 4 at its largest da"),
    Row(5, 2, 2, 128, TC, "<8,8,32>", "smallest d of the instantiation"),
    Row(8, 2, 2, 500, TC, "<8,8,32>", "largest d of the tcgen05 kernels"),
]
QUAD_ROWS = [r._replace(kernel=QUAD) for r in TC_ROWS if r.h == 500 and r.d <= 4]
FP32_ROWS = [
    Row(3, 3, 2, 100, SIMT, "<4>", "da > 1 on the CTA kernel (a tcgen05 shape, run with precision fp32)"),
    Row(6, 2, 3, 64, SIMT, "<8>", "4 < d <= 8"),
    Row(17, 3, 2, 48, SIMT, "<32>", "d > 8"),
    Row(32, 8, 1, 96, SIMT, "<32>", "largest d and da"),
    Row(1, 8, 1, 32, THREAD, "<4,32>", "largest da on the thread kernel"),
    Row(5, 2, 1, 20, THREAD, "<8,32>", "d > 4 on the thread kernel"),
    Row(7, 3, 1, 64, THREAD, "<8,64>", "d > 4, h = 64"),
]
# tcgen05 shapes mpc_tc_shape_supported turns down: "auto" runs the FP32 CTA kernel
UNSUPPORTED_ROWS = [
    Row(9, 1, 2, 128, SIMT, "<32>", "d > 8"),
    Row(5, 3, 2, 128, SIMT, "<8>", "dz = 8: 8 + 3 inputs > 10"),
    Row(4, 7, 2, 128, SIMT, "<4>", "dz = 4: 4 + 7 inputs > 10"),
    Row(3, 8, 2, 128, SIMT, "<4>", "dz = 3: 3 + 8 inputs > 10"),
]
MODES = ["reference", "per_sample"]

# Tolerances.  FP32 rows: those of tests/test_gpu_mpc.py (relative, <= 1 % waypoint-switch outliers).
STATE_RTOL = 1e-4
SCORE_TOL = 1e-4
# tcgen05 rows (the H1 / W2 operands are bf16): about 3x the largest errors measured on these problems on a B200
# by scripts/dev/tc_dims_errors.py, profiles/r06_tc_dims_errors.json, over both kernels, both penalty modes and
# every case of a shape.  Scores: an absolute bound per shape (d, da, h), 3x the largest 99th percentile of the
# score error (<= 1 % of the samples may exceed it: waypoint-switch flips), and a median bound; states: 3x the
# largest error over the per-dimension scale.
# Measured on an NVIDIA B200 (power limit 1000 W): the largest score error of any case is 1.9e-3 (d = 3, da = 7,
# h = 100), all below the 5e-2 of tests/test_gpu_mpc.py, and every arg-best equals the oracle's.
TC_SCORE_ATOL = {            # (d, da, h): bound     measured largest p99
    (1, 2, 64): 1.5e-3,      # 4.8e-4
    (2, 3, 500): 7.5e-4,     # 2.4e-4
    (1, 8, 128): 1.5e-3,     # 5.0e-4
    (3, 2, 500): 1.6e-3,     # 5.3e-4 (after device training; 2.5e-4 on the initial weights)
    (3, 7, 100): 5e-3,       # 1.6e-3
    (4, 1, 256): 6e-4,       # 2.0e-4
    (4, 6, 500): 1.7e-3,     # 5.5e-4
    (5, 2, 128): 1.9e-3,     # 6.2e-4
    (8, 2, 500): 1.2e-3,     # 3.8e-4
}
TC_SCORE_MEDIAN = 3e-3       # largest median 9.4e-4
TC_STATE_RTOL = 5e-4         # largest state or path error 1.6e-4 of the scale

ACT_LOW = np.array([-1.0, 0.0, -2.0, -0.5, -3.0, 1.0, -1.5, 0.25])
ACT_HIGH = np.array([1.0, 3.0, 0.5, 0.5, -1.0, 2.0, 1.5, 0.75])
K_HOST, H_HOST = 1003, 10          # 8 tiles of 128 rows, the last one ragged


def _row_id(r):
    return "%s%s-d%d-da%d-L%d-h%d" % ("quad" if r.kernel == QUAD else r.kernel.split("_")[2], r.inst, r.d, r.da, r.L, r.h)


# ---- the dispatch, restated --------------------------------------------------------------------------------------
def _dz(d):
    return 2 if d <= 2 else 3 if d == 3 else 4 if d == 4 else 8


def _k1(d, da):
    return 16 if 3 * (_dz(d) + da) + 2 <= 16 else 32


def _tc_supported(r):
    return r.L == 2 and 64 <= r.h <= 510 and r.d <= 8 and _dz(r.d) + r.da <= 10


def _instantiation(r):
    if r.kernel in (TC, QUAD):
        return "<%d,%d,%d>" % (8 if _dz(r.d) == 8 else 4, _dz(r.d), _k1(r.d, r.da))
    h_pad = (r.h + 15) // 16 * 16
    if r.kernel == THREAD:
        return "<%d,%d>" % (4 if r.d <= 4 else 8, 32 if h_pad <= 32 else 64)
    return "<%d>" % (4 if r.d <= 4 else 8 if r.d <= 8 else 32)


def _parent_dz(r):
    """DZ of the kernel the launcher ran before it dispatched on the packed layout: <4,2,16> / <4,3,16> only for
    k1 = 16, otherwise <4,4,32> for every dz <= 4."""
    dz = _dz(r.d)
    return dz if _k1(r.d, r.da) == 16 or dz == 8 else 4


def test_dispatch_table_rows_run_their_instantiation():
    """Every row sits where the table says: its shape is (or is not) a tcgen05 shape, and the restated dispatch
    gives the instantiation the row names.  Together the rows cover every tcgen05 and FP32 instantiation."""
    for r in TC_ROWS + QUAD_ROWS:
        assert _tc_supported(r) and _instantiation(r) == r.inst, r
    for r in QUAD_ROWS:
        assert r.d <= 4 and 255 <= r.h <= 510
    for r in FP32_ROWS:
        assert _instantiation(r) == r.inst, r
        assert r.kernel == SIMT or (r.L == 1 and r.h <= 64 and r.d <= 8)
    for r in UNSUPPORTED_ROWS:
        assert not _tc_supported(r) and _instantiation(r) == r.inst, r
    assert {r.inst for r in TC_ROWS} == {"<4,2,16>", "<4,2,32>", "<4,3,32>", "<4,4,32>", "<8,8,32>"}
    assert {r.inst for r in QUAD_ROWS} == {"<4,2,32>", "<4,3,32>", "<4,4,32>"}
    assert {r.inst for r in FP32_ROWS if r.kernel == SIMT} == {"<4>", "<8>", "<32>"}
    assert {r.inst for r in FP32_ROWS if r.kernel == THREAD} == {"<4,32>", "<8,32>", "<8,64>"}
    # the rows the launcher used to send to a kernel of another layout
    assert [r for r in TC_ROWS if _parent_dz(r) != _dz(r.d)] == [r for r in TC_ROWS if r.inst in ("<4,2,32>", "<4,3,32>")]


# ---- problems ----------------------------------------------------------------------------------------------------
def _problem(r, seed=0):
    """A random model and plan of the row's shape.  Every action has its own bounds, and its normalisation
    statistics match them, so each action moves the first layer as much as a state input does."""
    rng = np.random.default_rng(1000 * r.d + 100 * r.da + 10 * r.L + r.h + seed)
    w, b = syn.xavier_mlp(rng, r.d, r.da, r.L, r.h, scale=0.5)
    lo, hi = ACT_LOW[:r.da], ACT_HIGH[:r.da]
    norm = dict(mean_x=rng.normal(size=r.d), std_x=rng.uniform(0.5, 2.0, r.d), mean_y=(lo + hi) / 2,
                std_y=(hi - lo) / np.sqrt(12.0), mean_z=0.05 * rng.normal(size=r.d), std_z=rng.uniform(0.05, 0.2, r.d))
    W = 12
    ds = np.cumsum(rng.uniform(0.05, 0.3, (W, r.d)), axis=0)
    radii = rng.uniform(0.1, 0.4, r.d)
    hops = np.append(np.sqrt((((ds[1:] - ds[:-1]) / radii) ** 2).sum(-1)), 0.0)
    dl = np.asarray([sum(hops[i:].tolist()) for i in range(W)])
    start = ds[1] + 0.05 * rng.normal(size=r.d)
    acts = lo + (hi - lo) * rng.random((K_HOST, H_HOST, r.da))
    return dict(w=w, b=b, norm=norm, ds=ds, dl=dl, radii=radii, start=start, lo=lo, hi=hi, acts=acts)


def _oracle(p, acts, mode, w=None):
    return mpc_oracle.plan(p["start"], acts, p["w"] if w is None else w, p["b"], p["norm"], p["ds"], p["dl"], p["radii"],
                           1, .75, .5, penalty_mode=0 if mode == "reference" else 1)


def _shifted_actions(w, d, da, shift):
    """First-layer weights under which the oracle computes what a kernel that reads action j from input
    dz + shift + j computes on images packed with action j in input dz + j: action j meets the weights of
    action j + shift, the last `shift` actions meet zero weights, and the first `shift` action weights meet 0."""
    w0 = w[0].copy()
    w0[d:d + da - shift] = w[0][d + shift:d + da]
    w0[d + da - shift:d + da] = 0.0
    return [w0] + list(w[1:])


def _with_env(name, value, fn):
    old = os.environ.get(name)
    if value is None:
        os.environ.pop(name, None)
    else:
        os.environ[name] = value
    try:
        return fn()
    finally:
        if old is None:
            os.environ.pop(name, None)
        else:
            os.environ[name] = old


def _quad_env(r):
    return "1" if r.kernel == QUAD else "0"


def _setup(engine, p):
    engine.set_model(p["w"], p["b"], p["norm"])
    engine.set_plan(p["ds"], p["dl"], p["radii"])


# ---- checks ------------------------------------------------------------------------------------------------------
def _state_scale(states, norm):
    return np.maximum(np.abs(states).max(axis=(0, 1)), np.asarray(norm["std_x"], dtype=np.float64))


def _check_best(best_k, want, tol_of):
    """The kernel's pick equals the oracle's when the oracle's top-2 gap exceeds twice the score tolerance;
    otherwise the picked sample's oracle score is within that of the top."""
    order = np.argsort(-want, kind="stable")
    top, second = want[order[0]], want[order[1]]
    tol = tol_of(top)
    if top - second > 2 * tol:
        assert best_k == int(order[0]), "arg-best %d, oracle %d (gap %.3g)" % (best_k, order[0], top - second)
    else:
        assert want[best_k] >= top - 2 * tol, "chosen score %.6g, oracle top %.6g" % (want[best_k], top)


def _plan(engine, row, p, mode, precision, quad=None, **kw):
    """One decision; returns (result, kernel name, reference-mode trajectories [H+1, K, d] or None)."""
    res = _with_env("SS_TC_QUAD", quad, lambda: engine.plan(p["start"], 1, penalty_mode=mode, precision=precision,
                                                            want_scores=True, **kw))
    kernel = engine.last_rollout_kernel()
    return res, kernel, engine.get_states() if mode == "reference" else None


def _errors(row, p, res, states, acts, o):
    """The quantities the checks bound (also what scripts/dev/tc_dims_errors.py records)."""
    scale = _state_scale(o["states"], p["norm"])
    err = np.abs(res["scores"] - o["scores"])
    order = np.argsort(-o["scores"], kind="stable")
    return dict(
        score_err=err, score_rel_err=err / np.maximum(np.abs(o["scores"]), 1.0),
        state_err=None if states is None else np.abs(states - o["states"]).max(axis=(0, 1)) / scale,
        path_err=np.abs(res["best_path"] - o["states"][:, res["best_k"]]).max(axis=0) / scale,
        top2_gap=float(o["scores"][order[0]] - o["scores"][order[1]]), oracle_best_k=int(order[0]))


def _assert_matches_oracle(row, p, res, states, acts, o):
    """Scores, arg-best, returned sequence (bit for bit) and path against the oracle; in reference mode every
    trajectory of the batch as well."""
    e = _errors(row, p, res, states, acts, o)
    tc = row.kernel in (TC, QUAD)
    state_tol = TC_STATE_RTOL if tc else STATE_RTOL
    if states is not None:
        assert e["state_err"].max() <= state_tol, e["state_err"].max()
    if tc:
        atol = TC_SCORE_ATOL[row.d, row.da, row.h]
        bad = e["score_err"] > atol
        assert np.median(e["score_err"]) < TC_SCORE_MEDIAN, np.median(e["score_err"])
        _check_best(res["best_k"], o["scores"], lambda top: atol)
    else:
        bad = e["score_rel_err"] > SCORE_TOL
        _check_best(res["best_k"], o["scores"], lambda top: SCORE_TOL * max(abs(top), 1.0))
    assert bad.mean() <= 0.01, "%.2f%% of scores off (max %.3g)" % (100 * bad.mean(), e["score_err"].max())
    assert res["best_k"] == int(np.argmax(res["scores"]))
    np.testing.assert_array_equal(res["best_sequence"], acts[res["best_k"]])
    assert e["path_err"].max() <= state_tol, e["path_err"].max()


# ---- the cases (scripts/dev/tc_dims_errors.py runs the tcgen05 ones to measure the bounds above) ----------------
def run_host_case(engine, row, mode):
    """Host samples of the row's shape on the row's kernel: precision "auto" for the tcgen05 rows (the default
    path), "fp32" for the FP32 rows."""
    p = _problem(row)
    _setup(engine, p)
    tc = row.kernel in (TC, QUAD)
    assert engine.tc_supported() == _tc_supported(row)
    res, kernel, states = _plan(engine, row, p, mode, "auto" if tc else "fp32", _quad_env(row) if tc else None,
                                actions=p["acts"])
    assert kernel == row.kernel
    return p, res, states, p["acts"], _oracle(p, p["acts"], mode)


SAMPLED_ROWS = [TC_ROWS[1], FP32_ROWS[0], FP32_ROWS[6]]
K_DEV, H_DEV, SEED_DEV = 1003, 8, 4242


def run_philox_case(engine, row, mode):
    """Philox samples drawn inside the kernel, each action with its own bounds."""
    p = _problem(row)
    _setup(engine, p)
    tc = row.kernel in (TC, QUAD)
    res, kernel, states = _plan(engine, row, p, mode, "auto" if tc else "fp32", _quad_env(row) if tc else None,
                                K=K_DEV, H=H_DEV, seed=SEED_DEV, act_low=p["lo"], act_high=p["hi"])
    assert kernel == row.kernel
    acts = philox.sample_actions(K_DEV, H_DEV, row.da, SEED_DEV, p["lo"], p["hi"])
    return p, res, states, acts, _oracle(p, acts, mode)


def run_mt19937_case(engine, mode="reference"):
    """numpy's npr.uniform(low, high, (K, H, 3)) drawn on the device from np.random.get_state(); returns the case
    and (the generator state the engine reports afterwards, numpy's)."""
    row = TC_ROWS[1]
    p = _problem(row)
    _setup(engine, p)
    npr.seed(2024)
    before = npr.get_state()
    acts = npr.uniform(p["lo"], p["hi"], (K_DEV, H_DEV, row.da))
    after = npr.get_state()
    res, kernel, states = _plan(engine, row, p, mode, "auto", "0", K=K_DEV, H=H_DEV, act_low=p["lo"],
                                act_high=p["hi"], rng_state=before)
    assert kernel == TC
    return (p, res, states, acts, _oracle(p, acts, mode)), (res["rng_state"], after)


COMMIT_ROW = Row(3, 2, 2, 500, TC, "<4,3,32>", "ss_dyn_commit re-packs the images at da = 2")


def train_and_commit(engine, train_precision):
    """d = 3, da = 2, 2 x 500: five device Adam steps, ss_dyn_commit.  Returns (the problem with the initial
    weights, the problem with dyn_get_params()).  Leaves the trainer in train_precision."""
    row = COMMIT_ROW
    p = _problem(row, seed=7)
    rng = np.random.default_rng(7)
    n_old, n_new, d = 2000, 1000, row.d
    X = rng.normal(size=(n_old + n_new, d + row.da))
    Z = np.tanh(0.7 * X[:, :d] + 0.4 * X[:, d:d + 1] - 0.6 * X[:, d + 1:d + 2]) + 0.05 * rng.normal(size=(n_old + n_new, d))
    engine.dyn_set_precision(train_precision)
    _setup(engine, p)
    engine.dyn_reset_optimizer()
    engine.dyn_set_data(0, X[:n_old], Z[:n_old])
    engine.dyn_set_data(1, X[n_old:], Z[n_old:])
    npr.seed(3)
    io, inw = dto.epoch_batches(n_old, n_new, 512, 0.9)
    engine.dyn_train_batches(io[:5], inw[:5], 1e-3, want_losses=False)
    engine.dyn_commit()
    gw, gb = engine.dyn_get_params()
    return p, dict(p, w=gw, b=gb)


COMMIT_KERNELS = ((TC, "bf16_tc", "0"), (QUAD, "bf16_tc", "1"), (SIMT, "fp32", None))


def run_commit_cases(engine, p, trained, mode):
    """The trained model planned by the pair, quad and FP32 kernels: [(row, case)]."""
    o = _oracle(trained, p["acts"], mode)
    out = []
    for kernel, prec, quad in COMMIT_KERNELS:
        row = COMMIT_ROW._replace(kernel=kernel)
        res, got, states = _plan(engine, row, trained, mode, prec, quad, actions=p["acts"])
        assert got == kernel
        out.append((row, (trained, res, states, p["acts"], o)))
    return out


# ---- host samples: every row of the table ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("row", TC_ROWS + QUAD_ROWS, ids=_row_id)
def test_tc_rows_vs_float64_oracle(engine, row, mode):
    """The default precision ("auto") on a tcgen05 shape: the row's kernel runs and matches the oracle."""
    _assert_matches_oracle(row, *run_host_case(engine, row, mode))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("row", FP32_ROWS, ids=_row_id)
def test_fp32_rows_vs_float64_oracle(engine, row, mode):
    _assert_matches_oracle(row, *run_host_case(engine, row, mode))


@pytest.mark.gpu
@pytest.mark.parametrize("row", UNSUPPORTED_ROWS, ids=_row_id)
def test_shapes_without_tc_kernel_run_fp32(engine, row):
    """A two-layer shape outside mpc_tc_shape_supported: no tcgen05 images, "bf16_tc" is refused, and "auto" runs
    the FP32 CTA kernel, which matches the oracle."""
    p = _problem(row)
    _setup(engine, p)
    assert not engine.tc_supported()
    with pytest.raises(ValueError):
        engine.plan(p["start"], 1, actions=p["acts"], precision="bf16_tc")
    for mode in MODES:
        res, kernel, states = _plan(engine, row, p, mode, "auto", actions=p["acts"])
        assert kernel == SIMT
        _assert_matches_oracle(row, p, res, states, p["acts"], _oracle(p, p["acts"], mode))


@pytest.mark.parametrize("row", [r for r in TC_ROWS if r.da >= 2], ids=_row_id)
def test_negative_control_layout_mismatch_misses_the_tolerance(row):
    """Host only.  The oracle with the actions moved by one input slot (the first action's weights meet 0, the
    last action meets zero weights: what <4,4,32> computes on images packed for d = 3) -- and, for d <= 2, by the
    two slots that kernel moved them there -- is at least 10x outside the row's tcgen05 tolerance: the median
    score error and the largest trajectory error.  Reference penalty mode, the default: with d = 1 the per-sample
    penalty is 0 (a one-dimensional trajectory never leaves the line between two waypoints), so per-sample scores
    of the d = 1 rows keep only the progress term and the same mismatch moves their median by 4-6x the bound."""
    p = _problem(row)
    shifts = sorted({1, _parent_dz(row) - _dz(row.d)} - {0})
    for mode in ["reference"]:
        want = _oracle(p, p["acts"], mode)
        scale = _state_scale(want["states"], p["norm"])
        for s in shifts:
            got = _oracle(p, p["acts"], mode, w=_shifted_actions(p["w"], row.d, row.da, s))
            med = np.median(np.abs(got["scores"] - want["scores"]))
            assert med >= 10 * TC_SCORE_ATOL[row.d, row.da, row.h], (s, mode, med)
            assert (np.abs(got["states"] - want["states"]).max(axis=(0, 1)) / scale).max() >= 10 * TC_STATE_RTOL


# ---- device samples with several actions -------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("row", SAMPLED_ROWS, ids=_row_id)
def test_philox_samples_with_per_action_bounds(engine, row, mode):
    """The returned sequence is philox.sample_actions' bit for bit, the scores are the oracle's on those samples,
    and two k_offset shards give the whole batch's per-sample scores bit for bit."""
    p, res, states, acts, o = run_philox_case(engine, row, mode)
    assert np.all((acts >= p["lo"]) & (acts <= p["hi"]))
    _assert_matches_oracle(row, p, res, states, acts, o)
    if mode == "per_sample":
        tc = row.kernel in (TC, QUAD)
        parts = []
        for off, n in ((0, 389), (389, K_DEV - 389)):
            r, kernel, _ = _plan(engine, row, p, mode, "auto" if tc else "fp32", _quad_env(row) if tc else None, K=n,
                                 k_offset=off, K_global=K_DEV, H=H_DEV, seed=SEED_DEV, act_low=p["lo"], act_high=p["hi"])
            assert kernel == row.kernel
            parts.append(r["scores"])
        np.testing.assert_array_equal(np.concatenate(parts), res["scores"])


@pytest.mark.gpu
def test_mt19937_samples_with_per_action_bounds(engine):
    """numpy's npr.uniform(low, high, (K, H, 3)) drawn on the device from np.random.get_state() and rolled in place:
    the samples are numpy's (the returned sequence bit for bit, the scores the oracle's on numpy's draw) and the
    generator state afterwards is numpy's."""
    case, (got, want) = run_mt19937_case(engine)
    assert got[0] == "MT19937" and got[2] == want[2] and np.array_equal(got[1], want[1])
    _assert_matches_oracle(TC_ROWS[1], *case)


# ---- ss_dyn_commit re-packs the tcgen05 images at da = 2 ---------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("train_precision", ["fp32", "fp64"])
def test_commit_feeds_the_tc_planner_at_two_actions(engine, train_precision):
    """A few device Adam steps (FP32 or FP64 trainer), ss_dyn_commit, then the pair, quad and FP32 kernels plan
    with the trained weights -- compared with the oracle on dyn_get_params()."""
    try:
        p, trained = train_and_commit(engine, train_precision)
        for mode in MODES:
            moved = np.abs(_oracle(trained, p["acts"], mode)["scores"] - _oracle(p, p["acts"], mode)["scores"])
            assert np.median(moved) > 10 * TC_SCORE_ATOL[COMMIT_ROW.d, COMMIT_ROW.da, COMMIT_ROW.h]   # training moved the model
            for row, case in run_commit_cases(engine, p, trained, mode):
                _assert_matches_oracle(row, *case)
    finally:
        engine.dyn_set_precision("fp32")
