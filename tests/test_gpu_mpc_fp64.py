"""precision="fp64": the float64 rollout and tail against the reference's goldens and the float64 oracle.
Decisions are compared without a gap condition: fp64 must pick the oracle's index."""
import numpy as np
import numpy.random as npr
import pytest

from conftest import golden_model, load_golden
from oracle import mpc_oracle, philox
from smartstartcontinuous_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

MPC_CASES = ["mpc_mountaincar_L2.npz", "mpc_pendulum_L1.npz", "mpc_mountaincar_L3_xavier.npz",
             "mpc_pendulum_2x500.npz"]
STATE_RTOL = 1e-10    # of the per-dimension state scale
SCORE_RTOL = 1e-9     # of max(|score|, 1)


def _setup(engine, g):
    w, b, norm = golden_model(g)
    engine.set_model(w, b, norm)
    engine.set_plan(g["out_desired_states"], g["out_distances_left"], g["out_radii"])
    return w, b, norm


def _assert_scores(got, want):
    err = np.abs(got - want) / np.maximum(np.abs(want), 1.0)
    assert err.max() <= SCORE_RTOL, err.max()


def _assert_path(got, want):
    scale = np.abs(want).max(axis=0)
    assert (np.abs(got - want) <= STATE_RTOL * np.maximum(scale, 1e-300)).all()


@pytest.mark.parametrize("name", MPC_CASES)
def test_golden_forward_sim_and_decision(engine, name):
    g = load_golden(name)
    _setup(engine, g)
    states = engine.forward_sim(g["in_start_state"], g["in_actions"], precision="fp64")
    assert engine.last_rollout_kernel() == "mpc_rollout_fp64_kernel"
    scale = np.abs(g["out_states"]).max(axis=(0, 1))
    assert (np.abs(states - g["out_states"]).max(axis=(0, 1)) <= STATE_RTOL * scale).all()
    res = engine.plan(g["in_start_state"], int(g["in_wp_index"]), actions=g["in_actions"],
                      gamma=float(g["in_gamma"]), horizontal_penalty_factor=float(g["in_hpf"]),
                      penalty_mode="reference", precision="fp64", want_scores=True)
    _assert_scores(res["scores"], g["out_scores"])
    assert res["best_k"] == int(g["out_best_k"])
    assert res["best_score"] == res["scores"][res["best_k"]]
    np.testing.assert_array_equal(res["best_sequence"], g["in_actions"][res["best_k"]])
    np.testing.assert_array_equal(res["best_sequence"][0], g["out_best_action"])
    _assert_path(res["best_path"], g["out_best_path"])
    seq, path = engine.replay(res["best_k"])
    np.testing.assert_array_equal(seq, res["best_sequence"])
    np.testing.assert_array_equal(path, res["best_path"])


def _random_problem(rng, L, h, d, da):
    w, b = syn.xavier_mlp(rng, d, da, L, h, scale=0.5)
    norm = dict(mean_x=rng.normal(size=d), std_x=rng.uniform(0.5, 2.0, d), mean_y=rng.normal(size=da),
                std_y=rng.uniform(0.5, 2.0, da), mean_z=0.05 * rng.normal(size=d), std_z=rng.uniform(0.05, 0.2, d))
    W = 12
    ds = np.cumsum(rng.uniform(0.05, 0.3, (W, d)), axis=0)
    radii = rng.uniform(0.1, 0.4, d)
    hops = np.append(np.sqrt((((ds[1:] - ds[:-1]) / radii) ** 2).sum(-1)), 0.0)
    dl = np.asarray([sum(hops[i:].tolist()) for i in range(W)])
    start = ds[1] + 0.05 * rng.normal(size=d)
    return w, b, norm, ds, dl, radii, start


@pytest.mark.parametrize("L,h,d,da", [(1, 32, 1, 1), (2, 100, 2, 2), (3, 32, 3, 3), (2, 500, 5, 1), (1, 100, 8, 2),
                                      (3, 100, 17, 1), (1, 500, 17, 3), (2, 32, 8, 1)])
@pytest.mark.parametrize("mode", ["reference", "per_sample"])
def test_random_shapes_vs_float64_oracle(engine, L, h, d, da, mode):
    rng = np.random.default_rng(1000 * L + 10 * d + da + h)
    w, b, norm, ds, dl, radii, start = _random_problem(rng, L, h, d, da)
    engine.set_model(w, b, norm)
    engine.set_plan(ds, dl, radii)
    K, H = 203 + 8 * d, 6
    acts = rng.uniform(-1, 1, (K, H, da))
    res = engine.plan(start, 1, actions=acts, penalty_mode=mode, precision="fp64", want_scores=True)
    o = mpc_oracle.plan(start, acts, w, b, norm, ds, dl, radii, 1, .75, .5,
                        penalty_mode=0 if mode == "reference" else 1)
    _assert_scores(res["scores"], o["scores"])
    assert res["best_k"] == int(np.argmax(o["scores"]))
    np.testing.assert_array_equal(res["best_sequence"], acts[res["best_k"]])
    _assert_path(res["best_path"], o["best_path"])


@pytest.mark.parametrize("mode", ["reference", "per_sample"])
def test_near_tie_and_exact_tie(engine, mode):
    """A duplicate of the best sequence with its last action nudged so that the oracle's best two scores
    differ by ~1e-9 relative: fp64 picks the oracle's index; the fp32 path's score error is larger than the
    gap, so its pick between the two is not determined by the scores.  An exact duplicate gives the first index."""
    g = load_golden("mpc_mountaincar_L2.npz")
    w, b, norm = _setup(engine, g)
    args = (g["out_desired_states"], g["out_distances_left"], g["out_radii"], int(g["in_wp_index"]),
            float(g["in_gamma"]), float(g["in_hpf"]))
    pm = 0 if mode == "reference" else 1
    acts = g["in_actions"]
    best = int(np.argmax(mpc_oracle.plan(g["in_start_state"], acts, w, b, norm, *args, penalty_mode=pm)["scores"]))

    def with_dup(eps):
        a = np.concatenate([acts, acts[best:best + 1]])
        a[-1, -1, 0] += eps
        return a, mpc_oracle.plan(g["in_start_state"], a, w, b, norm, *args, penalty_mode=pm)["scores"]

    _, s1 = with_dup(1e-6)
    slope = (s1[-1] - s1[best]) / 1e-6
    assert slope != 0.0
    eps = 1e-9 * abs(s1[best]) / abs(slope)
    a, want = with_dup(eps)
    gap = abs(want[-1] - want[best]) / abs(want[best])
    assert 1e-10 < gap < 1e-8 and sorted(np.argsort(-want)[:2]) == [best, len(a) - 1]
    kw = dict(actions=a, gamma=args[4], horizontal_penalty_factor=args[5], penalty_mode=mode, want_scores=True)
    res = engine.plan(g["in_start_state"], args[3], precision="fp64", **kw)
    assert res["best_k"] == int(np.argmax(want))
    _assert_scores(res["scores"], want)
    r32 = engine.plan(g["in_start_state"], args[3], precision="fp32", **kw)
    pair = [best, len(a) - 1]
    assert np.abs(r32["scores"][pair] - want[pair]).max() > abs(want[-1] - want[best])
    a[-1] = acts[best]
    want = mpc_oracle.plan(g["in_start_state"], a, w, b, norm, *args, penalty_mode=pm)["scores"]
    res = engine.plan(g["in_start_state"], args[3], precision="fp64", **dict(kw, actions=a))
    assert res["scores"][-1] == res["scores"][best] and res["best_k"] == best == int(np.argmax(want))


@pytest.mark.parametrize("name,seed", [("mpc_pendulum_2x500.npz", 4), ("mpc_mountaincar_L2.npz", 1)])
def test_seeded_agent_reproduces_the_reference_decision(engine, name, seed):
    """From np.random.seed(seed) the drop-in agent with precision="fp64" in its default sampling draws the
    golden's samples and makes the reference's decision, whatever the gap between the best two scores."""
    from smartstartcontinuous_b200.nnd_mb_agent import NND_MB_agent

    g = load_golden(name)
    w, b, norm = golden_model(g)
    K, H, _ = g["in_actions"].shape
    d = w[-1].shape[1]

    class Box:
        low, high, shape = g["in_act_low"], g["in_act_high"], (1,)

    class Env:
        action_space = Box()

    rng = np.random.default_rng(0)
    td = dict(dataX=rng.normal(size=(64, d)), dataY=rng.normal(size=(64, 1)), dataZ=rng.normal(size=(64, d)))
    ag = NND_MB_agent(Env(), None, horizon=H, num_control_samples=K, num_fc_layers=len(w) - 1,
                      depth_fc_layers=w[0].shape[1], gamma=float(g["in_gamma"]),
                      horizontal_penalty_factor=float(g["in_hpf"]), verbose=False, training_data=td, engine=engine,
                      precision="fp64")
    for k in ("mean_x", "std_x", "mean_y", "std_y", "mean_z", "std_z"):
        setattr(ag, k, np.asarray(g["in_" + k], dtype=np.float64))
        setattr(ag.dyn_model, k, getattr(ag, k))
    ag.dyn_model.set_weights(w, b)
    engine.set_plan(g["out_desired_states"], g["out_distances_left"], g["out_radii"])
    ag.desired_states, ag.distances_left, ag.radii = g["out_desired_states"], g["out_distances_left"], g["out_radii"]
    ag.current_desired_state_index = int(g["in_wp_index"])

    np.random.seed(seed)
    best_action, best_k, best_seq, best_path = ag.get_best_sim_actions(g["in_start_state"])
    after = np.random.get_state()
    np.random.seed(seed)
    np.random.uniform(g["in_act_low"], g["in_act_high"], (K, H, 1))
    want_after = np.random.get_state()
    assert after[2] == want_after[2] and np.array_equal(after[1], want_after[1])
    assert best_k == int(g["out_best_k"])
    np.testing.assert_array_equal(best_seq, g["in_actions"][best_k])
    np.testing.assert_array_equal(best_action, g["out_best_action"])
    _assert_path(best_path, g["out_best_path"])


@pytest.mark.parametrize("mode", ["reference", "per_sample"])
def test_device_philox_sampling(engine, mode):
    g = load_golden("mpc_mountaincar_L2.npz")
    w, b, norm = _setup(engine, g)
    K, H, seed = 1000, 12, 77
    res = engine.plan(g["in_start_state"], 0, K=K, H=H, seed=seed, act_low=[-1.0], act_high=[1.0],
                      penalty_mode=mode, precision="fp64", want_scores=True)
    acts = philox.sample_actions(K, H, 1, seed, [-1.0], [1.0])
    o = mpc_oracle.plan(g["in_start_state"], acts, w, b, norm, g["out_desired_states"], g["out_distances_left"],
                        g["out_radii"], 0, .75, .5, penalty_mode=0 if mode == "reference" else 1)
    _assert_scores(res["scores"], o["scores"])
    assert res["best_k"] == int(np.argmax(o["scores"]))
    np.testing.assert_array_equal(res["best_sequence"], acts[res["best_k"]])
    _assert_path(res["best_path"], o["best_path"])


def test_shards_on_one_gpu(engine):
    """Per-sample: two k_offset shards give the whole batch's scores bit for bit.  Reference: rollout of each
    shard, projection sums added over the shards, finish_package per shard, pick of the winner = the unsharded
    decision."""
    rng = np.random.default_rng(12)
    w, b, norm, ds, dl, radii, start = _random_problem(rng, 2, 100, 3, 1)
    engine.set_model(w, b, norm)
    engine.set_plan(ds, dl, radii)
    K, H = 700, 7
    kw = dict(H=H, seed=3, act_low=[-1.0], act_high=[1.0], precision="fp64")
    full = engine.plan(start, 1, K=K, penalty_mode="per_sample", want_scores=True, **kw)
    parts = [engine.plan(start, 1, K=n, k_offset=off, K_global=K, penalty_mode="per_sample", want_scores=True, **kw)
             for off, n in ((0, 300), (300, 400))]
    np.testing.assert_array_equal(np.concatenate([p["scores"] for p in parts]), full["scores"])
    assert max(parts, key=lambda p: (p["best_score"], -p["best_k"]))["best_k"] == full["best_k"]

    full = engine.plan(start, 1, K=K, penalty_mode="reference", want_scores=True, **kw)
    shards = ((0, 300), (300, 400))
    sums = 0.0
    for off, n in shards:
        engine.rollout(start, 1, K=n, k_offset=off, K_global=K, penalty_mode="reference", **kw)
        ptr, cnt = engine.projection_sums_ptr()
        sums = sums + engine.read_device_doubles(ptr, cnt)
    pkgs = []
    for off, n in shards:
        engine.rollout(start, 1, K=n, k_offset=off, K_global=K, penalty_mode="reference", **kw)
        ptr, cnt = engine.projection_sums_ptr()
        engine._check(engine._lib.ss_memcpy_h2d(engine._h, ptr, sums.ctypes.data, cnt * 8))
        _, n_pkg = engine.finish_package(True)
        pkgs.append(engine.read_package(n_pkg))
    win = max(pkgs, key=lambda p: (p[0], -p[1]))
    assert int(win[1]) == full["best_k"]
    assert win[0] == pytest.approx(full["best_score"], rel=1e-13)
    np.testing.assert_array_equal(win[2:2 + H], full["best_sequence"].reshape(-1))
    np.testing.assert_array_equal(win[2 + H:], full["best_path"].reshape(-1))


def test_after_device_training(engine):
    """After Dyn_Model.train (device Adam, then commit), fp64 rolls out exactly the exported model."""
    from smartstartcontinuous_b200.dynamics_model import Dyn_Model
    from smartstartcontinuous_b200.nnd_mb_agent import plan_from_path
    rng = np.random.default_rng(3)
    obs, act = syn.pendulum_rollouts(rng, 12, 200)
    xs = np.concatenate([o[:-1] for o in obs]); ys = np.concatenate(list(act)); zs = np.concatenate([o[1:] - o[:-1] for o in obs])
    st = {k: v for k, v in zip(("mean_x", "mean_y", "mean_z"), (xs.mean(0), ys.mean(0), zs.mean(0)))}
    sd = {k: v for k, v in zip(("std_x", "std_y", "std_z"), (xs.std(0), ys.std(0), zs.std(0)))}
    inputs = np.concatenate([(xs - st["mean_x"]) / sd["std_x"], (ys - st["mean_y"]) / sd["std_y"]], axis=1)
    outputs = (zs - st["mean_z"]) / sd["std_z"]
    m = Dyn_Model(4, 3, None, 1e-3, 512, 2, 64, st["mean_x"], st["mean_y"], st["mean_z"], sd["std_x"], sd["std_y"],
                  sd["std_z"], "float64", False, engine=engine, seed=0)
    engine.dyn_reset_optimizer()
    npr.seed(0)
    m.train(inputs[:1800], outputs[:1800], inputs[1800:], outputs[1800:], 3, None, 0.9, save_results=False)
    w, b = m.export()
    plan = plan_from_path(list(obs[0][:60]), mean_per_stepsize=1, std_per_stepsize=1, stepsizes_in_waypoint_radii=1,
                          path_shortcutting=True, theta=1, steps_per_waypoint=1)
    engine.set_plan(plan["desired_states"], plan["distances_left"], plan["radii"])
    acts = rng.uniform(-2, 2, (517, 6, 1))
    res = engine.plan(obs[0][0], 0, actions=acts, precision="fp64", want_scores=True)
    o = mpc_oracle.plan(obs[0][0], acts, w, b, m.norm(), plan["desired_states"], plan["distances_left"],
                        plan["radii"], 0, .75, .5)
    _assert_scores(res["scores"], o["scores"])
    assert res["best_k"] == int(np.argmax(o["scores"]))
    _assert_path(res["best_path"], o["best_path"])


def test_switching_precision_leaves_no_state(engine):
    g = load_golden("mpc_pendulum_2x500.npz")
    _setup(engine, g)
    kw = dict(actions=g["in_actions"], gamma=float(g["in_gamma"]), horizontal_penalty_factor=float(g["in_hpf"]),
              want_scores=True)
    for mode in ("reference", "per_sample"):
        runs = []
        for prec in ("fp32", "fp64", "fp32", "bf16_tc", "fp64"):
            runs.append(engine.plan(g["in_start_state"], int(g["in_wp_index"]), precision=prec, penalty_mode=mode, **kw))
            runs[-1]["kernel"] = engine.last_rollout_kernel()
            runs[-1]["states"] = engine.get_states()
        for i, j in ((0, 2), (1, 4)):
            for key in ("scores", "best_sequence", "best_path", "states"):
                np.testing.assert_array_equal(runs[i][key], runs[j][key])
            assert runs[i]["best_k"] == runs[j]["best_k"] and runs[i]["kernel"] == runs[j]["kernel"]
        assert runs[0]["kernel"] == "mpc_rollout_simt_kernel" and runs[1]["kernel"] == "mpc_rollout_fp64_kernel"
        assert runs[3]["kernel"].startswith("mpc_rollout_tc")
    with pytest.raises(KeyError):
        engine.plan(g["in_start_state"], 0, precision="fp16", **kw)
    st = np.ascontiguousarray(g["in_start_state"], dtype=np.float64)
    a = np.ascontiguousarray(g["in_actions"])
    rc = engine._lib.ss_mpc_rollout(engine._h, st.ctypes.data, 0, a.shape[0], 0, a.shape[0], a.shape[1], a.ctypes.data,
                                    0, None, None, .75, .5, 0, 4)
    assert rc == -1            # SS_EINVAL
