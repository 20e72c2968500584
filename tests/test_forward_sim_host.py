"""Forward simulation from per-sequence start states, host side (no GPU).

Dyn_Model.do_forward_sim(many_in_parallel=True) (dynamics_model.py:199-270) has two call forms in the reference:
[state, 0], whose first entry is tiled over the N sequences, and N start states, one per sequence.  The goldens
(oracle/make_golden.py) only cover the tiled form, and the reference's sources are not in the tree, so no golden can
be made for the per-sequence form.  forward_sim_rows() below is the oracle's loop (oracle/mpc_oracle.forward_sim)
with a [K, d] start instead of the tiled [d] one; it is pinned by the reading of dynamics_model.py:204-240 and by
the two tests here, which tie it to the oracle itself.  The GPU tests (test_gpu_forward_sim.py) compare the kernels
with it.

The rest of the file checks which Engine.forward_sim call each form of Dyn_Model.do_forward_sim makes, with a stub
engine in place of the GPU."""
import numpy as np
import pytest

from oracle import mpc_oracle


def forward_sim_rows(starts, actions, weights, biases, norm):
    """dynamics_model.py:204-240 with one start state per sequence: starts [K, d], actions [K, H, da] -> states
    [H+1, K, d] (float64).  Same operations as mpc_oracle.forward_sim, row for row."""
    actions = np.asarray(actions, dtype=np.float64)
    K, H, _ = actions.shape
    s = np.array(starts, dtype=np.float64).reshape(K, -1)
    out = [s.copy()]
    with np.errstate(divide="ignore", invalid="ignore"):
        for t in range(H):
            xs = np.nan_to_num((s - norm["mean_x"]) / norm["std_x"])
            ys = np.nan_to_num((actions[:, t, :] - norm["mean_y"]) / norm["std_y"])
            z = mpc_oracle.mlp_forward(np.concatenate([xs, ys], axis=1), weights, biases)
            s = s + (z * norm["std_z"] + norm["mean_z"])
            out.append(s.copy())
    return np.stack(out)


def _problem(seed=0, d=3, da=2, K=37, H=6, h=24):
    rng = np.random.default_rng(seed)
    sizes = [d + da, h, h, d]
    w = [rng.normal(0, 1 / np.sqrt(i), (i, o)) for i, o in zip(sizes[:-1], sizes[1:])]
    b = [rng.normal(0, 0.1, o) for o in sizes[1:]]
    norm = dict(mean_x=rng.normal(size=d), std_x=rng.uniform(0.5, 2, d), mean_y=np.zeros(da), std_y=np.ones(da),
                mean_z=0.05 * rng.normal(size=d), std_z=rng.uniform(0.05, 0.2, d))
    starts = norm["mean_x"] + 3 * norm["std_x"] * rng.normal(size=(K, d))
    acts = rng.uniform(-1, 1, (K, H, da))
    return w, b, norm, starts, acts


def test_equal_rows_are_the_tiled_form_bit_for_bit():
    w, b, norm, starts, acts = _problem()
    rows = np.tile(starts[5], (acts.shape[0], 1))
    np.testing.assert_array_equal(forward_sim_rows(rows, acts, w, b, norm),
                                  mpc_oracle.forward_sim(starts[5], acts, w, b, norm))


def test_rows_agree_with_one_oracle_call_per_start():
    w, b, norm, starts, acts = _problem(seed=1)
    got = forward_sim_rows(starts, acts, w, b, norm)
    assert np.array_equal(got[0], starts)
    for k in range(acts.shape[0]):
        want = mpc_oracle.forward_sim(starts[k], acts[k:k + 1], w, b, norm)[:, 0]
        np.testing.assert_allclose(got[:, k], want, rtol=1e-12, atol=1e-12)


# ---- Dyn_Model.do_forward_sim call forms against a stub engine ---------------------------------------------------
class _StubEngine:
    """Records Engine.forward_sim calls; returns states whose t = 0 row is the start it was given."""

    def __init__(self):
        self.calls = []

    def dyn_set_precision(self, precision):
        pass

    def set_model(self, weights, biases, norm):
        pass

    def forward_sim(self, state, actions, precision="fp32"):
        self.calls.append((np.array(state, dtype=np.float64), np.array(actions), precision))
        K, H = actions.shape[0], actions.shape[1]
        st = np.asarray(state, dtype=np.float64)
        return np.broadcast_to(st if st.ndim == 2 else st[None], (H + 1, K, st.shape[-1])).copy()


D, DA, N, H = 3, 1, 5, 4


def _model():
    from smartstartcontinuous_b200.dynamics_model import Dyn_Model
    z = np.zeros(D)
    eng = _StubEngine()
    m = Dyn_Model(D + DA, D, None, 1e-3, 16, 2, 8, z, np.zeros(DA), z, np.ones(D), np.ones(DA), np.ones(D),
                  "float64", False, engine=eng, seed=0)
    return m, eng


def test_state_zero_form_tiles_the_first_entry():
    m, eng = _model()
    s = np.array([0.1, 0.2, 0.3])
    y = np.zeros((N, H, DA))
    out = m.do_forward_sim([s, 0], y, True)
    (state, acts, prec), = eng.calls
    assert state.shape == (D,) and np.array_equal(state, s) and acts.shape == (N, H, DA) and prec == "fp32"
    assert len(out) == H + 1 and out[0].shape == (N, D)


@pytest.mark.parametrize("as_list", [False, True])
def test_per_sequence_starts(as_list):
    m, eng = _model()
    starts = np.arange(N * D, dtype=np.float64).reshape(N, D)
    x = [row.copy() for row in starts] if as_list else starts
    out = m.do_forward_sim(x, np.zeros((N, H, DA)), True, precision="fp64")
    (state, _, prec), = eng.calls
    assert np.array_equal(state, starts) and prec == "fp64"
    assert np.array_equal(out[0], starts)


def test_two_by_d_array_takes_the_tiled_branch_like_the_reference():
    """len(forwardsim_x_true) == 2 is the reference's test for the [state, 0] form, so two start states in a [2, d]
    array also take it: the first row starts every sequence."""
    m, eng = _model()
    two = np.array([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]])
    m.do_forward_sim(two, np.zeros((2, H, DA)), True)
    (state, _, _), = eng.calls
    assert np.array_equal(state, two[0])


@pytest.mark.parametrize("x", [np.zeros((N + 1, D)), np.zeros((N, D + 1)), np.zeros((N, D, 1)), np.zeros(7)],
                         ids=["wrong-N", "wrong-d", "3-D", "1-D"])
def test_malformed_starts_raise_value_error(x):
    m, eng = _model()
    with pytest.raises(ValueError):
        m.do_forward_sim(x, np.zeros((N, H, DA)), True)
    assert eng.calls == []


def test_single_sequence_form_is_unchanged():
    m, eng = _model()
    s = np.array([0.1, 0.2, 0.3])
    out = m.do_forward_sim([s, 0], np.zeros((H, DA)), False)
    (state, acts, prec), = eng.calls
    assert np.array_equal(state, s) and acts.shape == (1, H, DA) and prec == "fp32"
    assert len(out) == H + 1 and out[0].shape == (D,)
