#!/usr/bin/env python
"""bench.py -- headline benchmark of the SmartStart hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  Headline metric: NND-MPC rollout-steps/s; the second half of
BASELINE.json's metric, KDE kernel-evals/s, is reported in the same line under "kde".

  step      one MPC decision (NND_MB_agent.get_best_sim_actions): K action sequences rolled H steps
            through the 2x500 dynamics MLP, scored against the waypoint plan, arg-best
            (reference-exact penalty mode).  Workload per GPU: Pendulum d=3, da=1, K=131072
            (= BASELINE config 4's K=1M / 8), H=50 -- at N=8 this is exactly config 4.
  value     K_total * H / device time, inputs resident (actions sampled on the device, Philox)
  e2e       the same decision through the drop-in plugin call NND_MB_agent.get_best_sim_actions
            (NND_MB_agent.py:498-520) in its DEFAULT configuration: the K*H*da float64 samples of
            npr.uniform (:500-501) come from numpy's global MT19937 stream, generated on the GPU from
            np.random.get_state() bit for bit (csrc/mt19937.cu) and the advanced state set back; inputs
            per call = the state + the generator key, outputs = winner package + key.  e2e_host_rng is
            the same call with host_rng=True (samples drawn on the host inside the timer, uploaded),
            e2e_device_sampling the call with device_sampling=True (Philox on the GPU), e2e_host_samples
            the C-ABI call on pre-drawn pinned samples (52 MB H2D per step, no host RNG in the timer).
  kde       BASELINE config 2: 100 001 Pendulum states x 16 384 candidate queries per GPU; its e2e
            goes through SmartStartContinuous.get_smart_start_path (smartexplorationcontinuous.py:223-305)
  small_k   BASELINE configs 3 (MountainCar, K=4096, H=20, 2x500) and 1 (the example's shapes:
            K=5000, H=4, MLP 1x32; KDE n_ss=2000): ms per decision resident and through the agent
  roofline  tensor pipe for the rollout kernel: achieved = 507 000 FLOP x K*H / kernel time against the
            measured BURST bf16 peak (the timed region is ~50 ms at the maximum SM clock; the ratio
            to the sustained figure is kept as frac_of_sustained_peak); SFU pipe (16 MUFU.EX2 / clk /
            SM) for the KDE pair kernel
  --impl reference: the reference's own CPU code for the path (NND_MB_agent.get_best_sim_actions
            executed from the staged copy oracle/_ref through oracle/ref_harness.py; TensorFlow's
            sess.run evaluated in float64 numpy/BLAS on all host cores) -- or the oracle port when the
            staged copy is absent -- and scipy gaussian_kde with the queries chunked over a
            multiprocessing.Pool, timed on bounded samples of the same workload plus one full-size
            step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

FLOP_PER_STEP = {2: 505_000, 3: 507_000}      # SURVEY 8(d): 2*[(d+da)h + h^2 + h d], h=500
K_PER_GPU = 131_072
HORIZON = 50
KDE_N = 100_000
KDE_M = 16_384
C3_K, C3_H = 4096, 20                          # BASELINE config 3
C1_K, C1_H, C1_NSS = 5000, 4, 2000             # BASELINE config 1 (the example's hyper-parameters)
SFU_PER_CLK_PER_SM = 16                        # MUFU.EX2 lanes per SM per clock (sm_100)
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full
# captures of exactly these workloads (profiles/r02k_ncu_summary.md); not measurable live
NCU_TRAFFIC = {"mpc_rollout_tc_kernel": 623_872 + 53_846_784, "kde_pairs_tc_kernel": 7_491_584}
NCU_TRAFFIC_SOURCE = "profiles/r02k_ncu_summary.md (ncu --set full, same workload)"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_sustained=p["bf16_tflops_sustained"], bf16_burst=p["bf16_tflops"],
                    sm_max_mhz=p.get("sm_max_mhz", 1965.0), source="MEASURED_PEAKS.json")
    return dict(hbm_gbs=6650.0, bf16_sustained=1400.0, bf16_burst=1590.0, sm_max_mhz=1965.0,
                source="fallback (B200_PROFILING.md)")


# --------------------------------------------------------------------------- workloads
def _plan(path):
    from smartstartcontinuous_b200.nnd_mb_agent import plan_from_path
    return plan_from_path(path, mean_per_stepsize=1, std_per_stepsize=1, stepsizes_in_waypoint_radii=1,
                          path_shortcutting=True, theta=1, steps_per_waypoint=1)


def make_workload(seed=0):
    """BASELINE config 4 / 5 shapes: Pendulum d=3, da=1, MLP 2x500 (seeded synthetic, SURVEY 8d)."""
    from smartstartcontinuous_b200 import synthetic as syn
    rng = np.random.default_rng(seed)
    obs, act = syn.pendulum_rollouts(rng, 25, 333)          # 25 x 333 random-policy transitions
    norm = syn.normalisation_stats(np.concatenate(list(obs)),
                                   np.concatenate([np.concatenate([a, a[-1:]]) for a in act]))
    w, b = syn.xavier_mlp(rng, 3, 1, 2, 500, scale=0.5)
    path = list(obs[0][:80])
    return dict(w=w, b=b, norm=norm, plan=_plan(path), path=path, state=obs[0][0].copy(), low=[-2.0], high=[2.0],
                d=3, da=1, L=2, h=500)


def make_workload_mountaincar(L, h, seed=3):
    """BASELINE configs 3 (L=2, h=500) and 1 (L=1, h=32): MountainCar d=2, da=1."""
    from smartstartcontinuous_b200 import synthetic as syn
    rng = np.random.default_rng(seed)
    roll = [syn.mountaincar_rollout(rng, 200) for _ in range(8)]
    norm = syn.normalisation_stats(np.concatenate([r[0] for r in roll]),
                                   np.concatenate([np.concatenate([r[1], r[1][-1:]]) for r in roll]))
    w, b = syn.xavier_mlp(rng, 2, 1, L, h, scale=0.5)
    path = list(roll[0][0][:60])
    return dict(w=w, b=b, norm=norm, plan=_plan(path), path=path, state=roll[0][0][0].copy(), low=[-1.0], high=[1.0],
                d=2, da=1, L=L, h=h)


def kde_workload(seed=0, n=KDE_N, m=KDE_M):
    from smartstartcontinuous_b200 import synthetic as syn
    all_states, s2, _ = syn.pendulum_buffer(n, seed=seed)
    rng = np.random.default_rng(seed)
    q = np.ascontiguousarray(s2[rng.choice(n, m, replace=False)])
    return dict(all_states=all_states, queries=q, values=syn.critic_like_values(q), n=n, volume=1e-3)


def workload_name():
    return ("NND_MB random-shooting MPC, Pendulum-v0 d=3 da=1, K=%d per GPU (BASELINE config 4 = K=1M over 8 GPUs), "
            "H=%d, MLP 2x500, reference-exact penalty" % (K_PER_GPU, HORIZON))


def shared_config(world):
    """`config` of the JSON line: identical keys and values in both arms (ours / --impl reference)."""
    return {"workload": workload_name(), "K_per_gpu": K_PER_GPU, "K_total": K_PER_GPU * world, "H": HORIZON,
            "mlp": "2x500", "d": 3, "da": 1, "penalty_mode": "reference", "gamma": .75, "horizontal_penalty_factor": .5}


def dump_decision(out_dir, res):
    """--dump-outputs: the arrays an MPC decision hands its caller, one float64 .npy each (scalars as shape (1,))."""
    os.makedirs(out_dir, exist_ok=True)
    for name in ("best_k", "best_score", "best_sequence", "best_path"):
        np.save(os.path.join(out_dir, name + ".npy"), np.array(res[name], dtype=np.float64, ndmin=1))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except OSError:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        busy = [v for v in sm if v > 0]
        return dict(sm_mhz=float(np.median(busy)) if busy else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# --------------------------------------------------------------------------- CPU (reference) arm
class CpuPlanner:
    """The reference's CPU planner for one workload.  With the reference staged (oracle/_ref, or
    /root/reference in the build container) this is its OWN NND_MB_agent: start_new_episode_plan +
    get_best_sim_actions (npr.uniform sampling, do_forward_sim, generate_scores_add_delta, argmax),
    the TF session replaced by a float64 numpy evaluation of the same MLP (oracle/ref_harness.py).
    Otherwise the oracle port of the same functions."""

    def __init__(self, wl, K, H):
        from oracle import ref_harness as rh
        self.wl, self.K, self.H = wl, K, H
        self.kind = "port"
        self.agent = None
        if rh.available():
            ref = rh.load_reference()
            self.agent = rh.make_nnd_agent(ref, wl["w"], wl["b"], wl["norm"], wl["low"], wl["high"], horizon=H,
                                           num_control_samples=K)
            self.agent.start_new_episode_plan(wl["state"], [np.asarray(p) for p in wl["path"]])
            self.kind = "reference"

    def set_K(self, K):
        self.K = K
        if self.agent is not None:
            self.agent.N = K

    def decide(self, seed):
        """One decision; returns seconds (sampling included, as in the reference)."""
        wl = self.wl
        np.random.seed(seed)
        t0 = time.perf_counter()
        if self.agent is not None:
            self.agent.get_best_sim_actions(wl["state"])
        else:
            from oracle import mpc_oracle
            acts = np.random.uniform(wl["low"], wl["high"], (self.K, self.H, wl["da"]))
            mpc_oracle.plan(wl["state"], acts, wl["w"], wl["b"], wl["norm"], wl["plan"]["desired_states"],
                            wl["plan"]["distances_left"], wl["plan"]["radii"], 0, .75, .5)
        return time.perf_counter() - t0


def cpu_reference_kde(kw, m):
    """scipy.stats.gaussian_kde fit + evaluate + UCB + argmax on one core (the reference as written,
    smartexplorationcontinuous.py:260-280).  Returns seconds."""
    from oracle import kde_oracle
    t0 = time.perf_counter()
    kde_oracle.select_start(kw["all_states"], kw["queries"][:m], kw["values"][:m], kw["n"], kw["volume"], 1.0, 2.0,
                            density_fn=kde_oracle.scipy_density)
    return time.perf_counter() - t0


_POOL_KDE = {}


def _pool_kde_chunk(span):
    lo, hi = span
    return _POOL_KDE["kernel"](_POOL_KDE["queries"][lo:hi].T)


def cpu_reference_kde_pool(kw, m, procs, reps):
    """The same numeric core with the queries chunked over a multiprocessing.Pool (the reference's
    own parallel idiom, smartstart/utilities/experimenter.py:84-92): fit once in the parent
    (timed), evaluate in `procs` forked workers, UCB + argmax in the parent.  Returns the mean
    seconds of `reps` repetitions (pool start-up excluded)."""
    import multiprocessing as mp
    from scipy.stats import gaussian_kde
    q = np.ascontiguousarray(kw["queries"][:m])
    _POOL_KDE["queries"] = q
    _POOL_KDE["kernel"] = gaussian_kde(kw["all_states"].T, bw_method="scott")
    spans = [(int(a[0]), int(a[-1]) + 1) for a in np.array_split(np.arange(m), procs) if len(a)]
    times = []
    with mp.get_context("fork").Pool(procs) as pool:
        pool.map(_pool_kde_chunk, [(0, 8)] * procs)                      # warm the workers
        for _ in range(reps):
            t0 = time.perf_counter()
            kernel = gaussian_kde(kw["all_states"].T, bw_method="scott")   # the fit is part of the path
            _ = kernel.factor
            dens = np.concatenate(pool.map(_pool_kde_chunk, spans))
            c_hat = kw["n"] * dens * kw["volume"]
            ucb = 1.0 * np.asarray(kw["values"][:m], dtype=np.float64) + np.sqrt(2.0 * np.log(kw["n"]) / c_hat)
            int(np.argmax(ucb))
            times.append(time.perf_counter() - t0)
    return float(np.mean(times))


def dyn_train_workload(seed=0):
    """Row f1: the training call of NND_MB_agent.train_dynamics_model at the BASELINE shapes --
    25 x 333 random-policy Pendulum transitions as the initial data (NND_MB_agent.py:75-76), 3000
    aggregated transitions, MLP 2x500, batch 512 (90 % new), lr 1e-3."""
    from smartstartcontinuous_b200 import synthetic as syn
    rng = np.random.default_rng(seed)
    obs, act = syn.pendulum_rollouts(rng, 34, 333)
    xs = np.concatenate([o[:-1] for o in obs]); ys = np.concatenate(list(act))
    zs = np.concatenate([o[1:] - o[:-1] for o in obs])
    st = dict(mean_x=xs.mean(0), std_x=xs.std(0), mean_y=ys.mean(0), std_y=ys.std(0), mean_z=zs.mean(0), std_z=zs.std(0))
    X = np.concatenate([(xs - st["mean_x"]) / st["std_x"], (ys - st["mean_y"]) / st["std_y"]], axis=1)
    Z = (zs - st["mean_z"]) / st["std_z"]
    n_old = 25 * 333
    w, b = syn.xavier_mlp(rng, 3, 1, 2, 500)
    return dict(X_old=X[:n_old], Z_old=Z[:n_old], X_new=X[n_old:n_old + 2997], Z_new=Z[n_old:n_old + 2997], w=w, b=b,
                norm=st, batch=512, frac=0.9, lr=1e-3, epochs=30)


DYN_FLOP_PER_STEP = 2 * 512 * (4 * 500 + 500 * 500 + 500 * 3) * 3      # forward + two backward products per layer


def cpu_dyn_train(cores):
    """One Adam step of Dyn_Model.train on the CPU: float64 numpy restatement (oracle/dyn_train_oracle.py;
    TensorFlow cannot run here), BLAS on all cores.  Returns ms per step over 20 steps."""
    from oracle import dyn_train_oracle as dto
    tw = dyn_train_workload()
    w, b = [a.copy() for a in tw["w"]], [a.copy() for a in tw["b"]]
    state = dto.AdamState(w, b)
    np.random.seed(0)
    io, inw = dto.epoch_batches(len(tw["X_old"]), len(tw["X_new"]), tw["batch"], tw["frac"])
    dto.train_batches(w, b, state, tw["X_old"], tw["Z_old"], tw["X_new"], tw["Z_new"], io[:3], inw[:3], tw["lr"])
    t0 = time.perf_counter()
    dto.train_batches(w, b, state, tw["X_old"], tw["Z_old"], tw["X_new"], tw["Z_new"], io[3:23], inw[3:23], tw["lr"])
    ms = 1e3 * (time.perf_counter() - t0) / 20
    steps_per_training = tw["epochs"] * len(io)
    return {"ms_per_adam_step": ms, "steps_per_training": steps_per_training, "training_s_scaled": ms * steps_per_training / 1e3,
            "kind": "port (float64 numpy restatement of the TF graph + AdamOptimizer)", "cores": cores,
            "sample": "20 Adam steps of batch 512 on the 2x500 network"}


def pin_blas_threads():
    """All host cores for the BLAS behind numpy, whatever OMP_NUM_THREADS says (torch.distributed.run
    exports OMP_NUM_THREADS=1 to its workers).  Returns (controller to keep alive, threads in use)."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        ctl = threadpool_limits(limits=n)
        used = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
        return ctl, used
    except Exception:
        return None, 1


REF_K_SAMPLE = 4096          # sequences per timed MPC step of the CPU arm


def run_reference(args, guard):
    """--impl reference: the reference's CPU path on rank 0 only, all host threads, bounded samples of
    the same workload (+ one full-size step unless --no-full-step)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ctl, cores = pin_blas_threads()
    wl = make_workload()
    kw = kde_workload()
    K_s = REF_K_SAMPLE
    cpu = CpuPlanner(wl, K_s, HORIZON)
    for _ in range(args.warmup):
        cpu.set_K(512)
        cpu.decide(0)
    cpu.set_K(K_s)
    t_mpc = [cpu.decide(i) for i in range(args.steps)]
    v = K_s * HORIZON / float(np.mean(t_mpc))
    full = None
    if not args.no_full_step:
        cpu.set_K(K_PER_GPU)
        t_full = cpu.decide(99)
        full = {"K": K_PER_GPU, "H": HORIZON, "seconds": t_full, "value": K_PER_GPU * HORIZON / t_full,
                "unit": "rollout-steps/s"}
    # BASELINE configs 3 and 1 on the CPU (whole decisions, these are small)
    small = {}
    for name, (L, h, K, H) in (("config3", (2, 500, C3_K, C3_H)), ("config1", (1, 32, C1_K, C1_H))):
        wls = make_workload_mountaincar(L, h)
        cp = CpuPlanner(wls, K, H)
        cp.decide(0)
        ts = [cp.decide(i) for i in range(3)]
        small[name] = {"ms_per_decision": 1e3 * float(np.mean(ts)), "rollout_steps_per_s": K * H / float(np.mean(ts)),
                       "K": K, "H": H, "mlp": "%dx%d" % (L, h), "kind": cp.kind, "cores": cores}
    small["dyn_train"] = cpu_dyn_train(cores)
    procs = os.cpu_count() or 1
    m_pool = min(KDE_M, 256 * procs)
    reps = max(1, min(args.steps, 5))
    t_pool = cpu_reference_kde_pool(kw, m_pool, procs, reps)
    kv = m_pool * (kw["n"] + 1) / t_pool
    t_one = [cpu_reference_kde(kw, 256) for _ in range(2)]
    kv_one = 256 * (kw["n"] + 1) / float(np.mean(t_one))
    kw1 = kde_workload(seed=2, n=KDE_N, m=C1_NSS)
    t_c1 = [cpu_reference_kde(kw1, 256) for _ in range(2)]
    small["config1"]["kde_n_ss_2000_ms_one_core_scaled"] = 1e3 * float(np.mean(t_c1)) * C1_NSS / 256
    sample = "%d steps of K=%d (of %d) sequences, H=%d (rate is K-independent: GEMM-bound)%s" % (
        args.steps, K_s, K_PER_GPU, HORIZON,
        "; one full K=%d step: %.1f s = %.3g rollout-steps/s" % (K_PER_GPU, full["seconds"], full["value"]) if full else "")
    note = ("the reference's own NND_MB_agent.get_best_sim_actions (staged copy, oracle/ref_harness.py) with sess.run "
            "evaluated in float64 numpy/BLAS" if cpu.kind == "reference" else
            "oracle port of the reference's numpy/TF-CPU path (no staged reference copy found)")
    guard.emit(json.dumps({
        "impl": "reference", "metric": "mpc_rollout_steps_per_s", "value": v, "unit": "rollout-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean(t_mpc)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": shared_config(max(1, args.gpus)),
        "reference_note": note + "; TensorFlow 1.5 is not installable here; BLAS threads pinned to all %d cores "
                                 "(OMP_NUM_THREADS ignored)" % cores,
        "cpu_baseline": {"value": v, "unit": "rollout-steps/s", "cores": cores, "kind": cpu.kind, "sample": sample},
        "full_step": full,
        "e2e": {"value": v, "unit": "rollout-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "small_k": small,
        "kde": {"metric": "kde_kernel_evals_per_s", "value": kv, "unit": "kernel-evals/s", "cores": procs,
                "kind": "reference-library (scipy.stats.gaussian_kde; queries chunked over a "
                        "multiprocessing.Pool, the reference's parallel idiom)",
                "sample": "%d x %d (of %d) queries x %d points" % (reps, m_pool, KDE_M, kw["n"] + 1),
                "single_core": {"value": kv_one, "cores": 1, "sample": "2 x 256 queries x %d points" % (kw["n"] + 1)}},
    }))
    del ctl


class _StdoutGuard:
    """Everything libraries print to fd 1 (e.g. NCCL's version banner) goes to stderr; only the
    final JSON line reaches the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


# --------------------------------------------------------------------------- drop-in agents for the e2e legs
class _Box:
    def __init__(self, low, high):
        self.low, self.high = np.asarray(low, dtype=np.float64), np.asarray(high, dtype=np.float64)
        self.shape = self.low.shape


class _Env:
    def __init__(self, low, high):
        self.action_space = _Box(low, high)


def make_nav_agent(eng, wl, K, H, device_sampling, planner=None, host_rng=None):
    """The drop-in NND_MB_agent carrying the benchmark's network and plan (no environment: the
    constructor gets a tiny synthetic training set, the weights are set afterwards)."""
    from smartstartcontinuous_b200.nnd_mb_agent import NND_MB_agent
    rng = np.random.default_rng(0)
    d, da = wl["d"], wl["da"]
    td = dict(dataX=rng.normal(size=(64, d)), dataY=rng.normal(size=(64, da)), dataZ=rng.normal(size=(64, d)))
    ag = NND_MB_agent(_Env(wl["low"], wl["high"]), None, horizon=H, num_control_samples=K, num_fc_layers=wl["L"],
                      depth_fc_layers=wl["h"], verbose=False, engine=eng, training_data=td,
                      device_sampling=device_sampling, host_rng=host_rng, precision="auto", penalty_mode="reference",
                      planner=planner)
    for k in ("mean_x", "std_x", "mean_y", "std_y", "mean_z", "std_z"):
        setattr(ag, k, np.asarray(wl["norm"][k], dtype=np.float64))
        setattr(ag.dyn_model, k, getattr(ag, k))
    ag.dyn_model.set_weights(wl["w"], wl["b"])          # -> Engine.set_model
    ag.num_episodes_finished = 1                        # no training at this plan
    ag.num_episodes_for_aggregation = 10 ** 9
    ag.start_new_episode_plan(wl["state"], [np.asarray(p) for p in wl["path"]])   # -> Engine.set_plan
    return ag


def ddpg_like_nets(d, seed=11):
    """Actor / critic of the example's DDPG agent (models_editted.py:22-100: dense-relu 64, dense-relu 32,
    dense; the action enters the critic's second layer), random weights, in Engine.set_value_net's format."""
    rng = np.random.default_rng(seed)

    def lin(i, o, scale=None):
        sc = scale if scale is not None else 1.0 / np.sqrt(i)
        return rng.uniform(-sc, sc, (i, o)).astype(np.float32), rng.uniform(-sc, sc, o).astype(np.float32)
    return dict(actor=[lin(d, 64), lin(64, 32), lin(32, 1, 3e-3)], critic=[lin(d, 64), lin(64 + 1, 32), lin(32, 1, 3e-3)],
                last_layer_tanh=True, obs_clip=(-5.0, 5.0))


class _ValueBase:
    """Base agent of the selection e2e: get_state_value like DDPG_Baselines_agent.py:197-204, i.e.
    critic(obs, actor(obs)) of `net`, evaluated on the host in float32 numpy (the stand-in for the
    user's TensorFlow session; its time is reported as host_value_fn_ms)."""

    def __init__(self, net):
        self.net = net
        self.seconds = 0.0

    def get_action(self, s): return np.zeros(1)
    def observe(self, *a): pass
    def start_new_episode(self, s): pass
    def end_episode(self): pass
    def get_param_dict(self): return {}

    def get_state_value(self, states):
        t0 = time.perf_counter()
        x = np.clip(np.asarray(states, dtype=np.float32), *self.net["obs_clip"])
        (aw1, ab1), (aw2, ab2), (aw3, ab3) = self.net["actor"]
        (cw1, cb1), (cw2, cb2), (cw3, cb3) = self.net["critic"]
        a = np.tanh(np.maximum(np.maximum(x @ aw1 + ab1, 0) @ aw2 + ab2, 0) @ aw3 + ab3)
        h = np.maximum(x @ cw1 + cb1, 0)
        v = np.maximum(np.concatenate([h, a], axis=1) @ cw2 + cb2, 0) @ cw3 + cb3
        self.seconds += time.perf_counter() - t0
        return v.reshape(-1, 1)


def make_smart_start(eng, kw, n_ss, device_values=False):
    """SmartStartContinuous over a replay buffer filled (through its own add / start_new_episode API)
    with the KDE workload's transitions.  device_values: the base agent's nets are handed over as
    value_net (row f4), so the candidates' values are computed on the device."""
    from smartstartcontinuous_b200.smart_start import SmartStartContinuous
    d = kw["all_states"].shape[1]
    rng = np.random.default_rng(0)
    td = dict(dataX=rng.normal(size=(64, d)), dataY=rng.normal(size=(64, 1)), dataZ=rng.normal(size=(64, d)))
    n = kw["n"]
    net = ddpg_like_nets(d)
    ss = SmartStartContinuous(_ValueBase(net), _Env([-2.0], [2.0]), None, buffer_size=n, n_ss=n_ss, print_ss_stuff=False,
                              nnd_mb_num_fc_layers=1, nnd_mb_depth_fc_layers=32, nnd_mb_verbose=False, engine=eng,
                              nnd_mb_extra=dict(training_data=td), value_net=net if device_values else None)
    rb = ss.replay_buffer
    s_all = kw["all_states"]
    a0 = np.zeros(1)
    for i in range(n):
        if i % 200 == 0:
            rb.start_new_episode(ss)
        rb.add(ss, s_all[i], a0, 0.0, (i % 200) == 199, s_all[i + 1])
    return ss


def main():
    guard = _StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-step", action="store_true", help="reference arm: skip the full K=131072 step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed MPC decision returned (best_k, best_score, "
                         "best_sequence, best_path) as DIR/<name>.npy in float64; the inputs depend only on the "
                         "arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args, guard)
        return

    import random

    import torch
    import torch.distributed as dist
    from smartstartcontinuous_b200.distributed import ShardedPlanner, ShardedSelector
    from smartstartcontinuous_b200.engine import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    eng = Engine(local_rank)
    stream = torch.cuda.current_stream()
    wl = make_workload()
    eng.set_model(wl["w"], wl["b"], wl["norm"])
    eng.set_plan(wl["plan"]["desired_states"], wl["plan"]["distances_left"], wl["plan"]["radii"])
    planner = ShardedPlanner(eng, device=dev)         # binds the Engine to torch's current stream
    selector = ShardedSelector(eng, device=dev)
    if world > 1 and os.environ.get("SS_PEER", "1") != "0":
        eng.peer_setup()         # projection sums + winner packages over NVLink peer memory, inside the kernels
    K_total = K_PER_GPU * world
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        """Per-step CUDA-event times on the launching stream; L2 flushed between steps (outside
        the events).  Returns (sum of per-step ms, max over ranks)."""
        for _ in range(warmup):
            fn(0)
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for i in range(steps):
            flush.zero_()
            ev[i][0].record(stream)
            fn(i + 1)
            ev[i][1].record(stream)
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in ev)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    half = max(3, args.steps // 2)
    precision = "bf16_tc" if eng.tc_supported() else "fp32"
    rollout_ms = []
    last_decision = {}

    def mpc_step(i):
        last_decision["res"] = planner.plan(wl["state"], 0, K=K_total, H=HORIZON, seed=1000 + i, act_low=wl["low"],
                                            act_high=wl["high"], penalty_mode="reference", precision=precision,
                                            want_path=True)
        if i > 0:
            rollout_ms.append(dict(eng.last_timings()).get("mpc_rollout", 0.0))

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = eng.launch_count()
    eng.set_timing(True)        # per-phase events inside the timed region: the rollout kernel's own time (roofline)
    ms_total = timed(mpc_step, args.steps, args.warmup)
    eng.set_timing(False)       # the library's default; the end-to-end legs below run as a user's calls do
    launches = eng.launch_count() - launches0
    ms_per_step = ms_total / args.steps
    value = K_total * HORIZON / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:         # every rank returns the same decision
        dump_decision(args.dump_outputs, last_decision["res"])

    # ---- e2e through the plugin call: NND_MB_agent.get_best_sim_actions -------------------------
    np.random.seed(1234)                      # identical on every rank (lock-step agents)
    nav_default = make_nav_agent(eng, wl, K_total, HORIZON, device_sampling=False, planner=planner if world > 1 else None)
    nav_host = make_nav_agent(eng, wl, K_total, HORIZON, device_sampling=False, host_rng=True,
                              planner=planner if world > 1 else None)
    nav_dev = make_nav_agent(eng, wl, K_total, HORIZON, device_sampling=True, planner=planner if world > 1 else None)

    def e2e_agent_step(i):
        nav_default.get_best_sim_actions(wl["state"])

    def e2e_agent_host_rng_step(i):
        nav_host.get_best_sim_actions(wl["state"])

    def e2e_agent_dev_step(i):
        nav_dev.get_best_sim_actions(wl["state"])

    # the default call and the host_rng=True call make the same decision from the same generator state
    st_check = np.random.get_state()
    r_default = nav_default.get_best_sim_actions(wl["state"])
    st_after = np.random.get_state()
    np.random.set_state(st_check)
    r_host = nav_host.get_best_sim_actions(wl["state"])
    st_after_host = np.random.get_state()
    mt_same = bool(r_default[1] == r_host[1] and np.array_equal(r_default[2], r_host[2]) and
                   st_after[2] == st_after_host[2] and np.array_equal(st_after[1], st_after_host[1]))
    if world > 1:
        mt_same = None          # with host_rng a rank draws only its own K/world sequences: a different draw

    e2e_ms = timed(e2e_agent_step, half, 3) / half
    e2e_value = K_total * HORIZON / (e2e_ms * 1e-3)
    e2e_steps = max(3, min(half, 6))
    e2e_host_rng_ms = timed(e2e_agent_host_rng_step, e2e_steps, 2) / e2e_steps
    t0 = time.perf_counter()
    for _ in range(3):
        np.random.random_sample((K_PER_GPU, HORIZON, 1))
    rng_ms = 1e3 * (time.perf_counter() - t0) / 3
    e2e_dev_ms = timed(e2e_agent_dev_step, half, 2) / half

    # the C-ABI call on pre-drawn host samples in pinned memory (no host RNG inside the timer)
    n_act = K_PER_GPU * HORIZON
    pinned = torch.empty(n_act, dtype=torch.float64).pin_memory()
    host_actions = pinned.numpy().reshape(K_PER_GPU, HORIZON, 1)
    host_actions[:] = np.random.RandomState(rank).uniform(wl["low"], wl["high"], (K_PER_GPU, HORIZON, 1))

    def e2e_samples_step(i):
        planner.plan(wl["state"], 0, K=K_total, H=HORIZON, local_actions=host_actions, penalty_mode="reference",
                     precision=precision, want_path=True)

    e2e_samples_ms = timed(e2e_samples_step, half, 2) / half

    # ---- the same decision with the per-sample projection (penalty_mode=1: the evidently intended
    # maths, SURVEY 8a Q1; fully fused, no second pass) -------------------------------------------
    def mpc_per_sample_step(i):
        planner.plan(wl["state"], 0, K=K_total, H=HORIZON, seed=3000 + i, act_low=wl["low"], act_high=wl["high"],
                     penalty_mode="per_sample", precision=precision, want_path=True)

    per_sample_ms = timed(mpc_per_sample_step, half, 2) / half

    # ---- KDE (BASELINE config 2 per GPU) -----------------------------------------------------
    kw = kde_workload()
    d_data = torch.as_tensor(kw["all_states"], device=dev)
    d_q = torch.as_tensor(kw["queries"], device=dev)
    d_v = torch.as_tensor(kw["values"], device=dev)
    pairs_ms = []

    def kde_step(i):
        eng.select_start_dev(d_data.data_ptr(), d_data.shape[0], 3, d_q.data_ptr(), d_q.shape[0], d_v.data_ptr(),
                             kw["n"], kw["volume"], 1.0, 2.0)
        if i > 0:
            pairs_ms.append(dict(eng.last_timings()).get("kde_pairs", 0.0))

    # the call is timed without the per-phase CUDA events (ss_set_timing(0): what a caller gets); a second short
    # pass with them gives the pair kernel's own time for the roofline
    eng.set_timing(False)
    kde_ms = timed(lambda i: kde_step(0), args.steps, args.warmup) / args.steps
    eng.set_timing(True)
    timed(kde_step, max(4, half // 2), 1)
    eng.set_timing(False)
    evals = KDE_M * (KDE_N + 1) * world
    kde_value = evals / (kde_ms * 1e-3)

    def kde_e2e_step(i):
        eng.select_start(kw["all_states"], kw["queries"], kw["values"], kw["n"], kw["volume"], 1.0, 2.0)

    kde_e2e_ms = timed(kde_e2e_step, half, 2) / half

    # through the plugin call SmartStartContinuous.get_smart_start_path: candidate sampling
    # (random.sample), candidate gather, host value function, selection from the device mirror of
    # the replay buffer's state ring, episodic path extraction -- everything the reference call does
    random.seed(7)
    ss = make_smart_start(eng, kw, KDE_M)

    def kde_agent_step(i):
        ss.get_smart_start_path()

    kde_agent_ms = timed(kde_agent_step, half, 2) / half
    ss.agent.seconds = 0.0
    for _ in range(3):
        ss.get_smart_start_path()
    kde_value_fn_ms = 1e3 * ss.agent.seconds / 3
    ss_dev = make_smart_start(eng, kw, KDE_M, device_values=True)
    kde_agent_dev_ms = timed(lambda i: ss_dev.get_smart_start_path(), half, 2) / half
    eng.set_value_net(None)
    del ss_dev
    ss2k = make_smart_start(eng, kde_workload(seed=2, n=KDE_N, m=C1_NSS), C1_NSS)
    d2k = kde_workload(seed=2, n=KDE_N, m=C1_NSS)
    t_data = torch.as_tensor(d2k["all_states"], device=dev)
    t_q = torch.as_tensor(d2k["queries"], device=dev)
    t_v = torch.as_tensor(d2k["values"], device=dev)
    pairs2k_ms = []

    def kde2k_step(i):
        eng.select_start_dev(t_data.data_ptr(), t_data.shape[0], 3, t_q.data_ptr(), t_q.shape[0], t_v.data_ptr(),
                             d2k["n"], d2k["volume"], 1.0, 2.0)
        if i > 0:
            pairs2k_ms.append(dict(eng.last_timings()).get("kde_pairs", 0.0))

    eng.set_timing(False)
    kde2k_ms = timed(lambda i: kde2k_step(0), args.steps, args.warmup) / args.steps
    eng.set_timing(True)
    timed(kde2k_step, max(4, half // 2), 1)
    eng.set_timing(False)
    kde2k_agent_ms = timed(lambda i: ss2k.get_smart_start_path(), half, 2) / half
    del ss, ss2k

    # ---- BASELINE config 5 (strong scaling): 1 000 001-state buffer KDE with the 16 384 candidates
    # sharded over the ranks + MPC with K = 262 144 sequences in total, both device-resident ----------
    eng.set_model(wl["w"], wl["b"], wl["norm"])
    eng.set_plan(wl["plan"]["desired_states"], wl["plan"]["distances_left"], wl["plan"]["radii"])
    C5_K = 262_144
    kw5 = kde_workload(seed=1, n=1_000_000)
    d5_data = torch.as_tensor(kw5["all_states"], device=dev)
    d5_q = torch.as_tensor(kw5["queries"], device=dev)
    d5_v = torch.as_tensor(kw5["values"], device=dev)

    def c5_kde_step(i):
        selector.select_start_dev(d5_data.data_ptr(), d5_data.shape[0], 3, d5_q.data_ptr(), d5_q.shape[0],
                                  d5_v.data_ptr(), kw5["n"], kw5["volume"], 1.0, 2.0)

    def c5_mpc_step(i):
        planner.plan(wl["state"], 0, K=C5_K, H=HORIZON, seed=2000 + i, act_low=wl["low"], act_high=wl["high"],
                     penalty_mode="reference", precision=precision, want_path=True)

    c5_kde_ms = timed(c5_kde_step, 5, 3) / 5        # (no per-phase events inside these calls: ~30 us per decision)
    c5_mpc_ms = timed(c5_mpc_step, 5, 3) / 5
    del d5_data, d5_q, d5_v

    # ---- BASELINE configs 3 and 1: the small-K decisions a drop-in user of the example gets -------
    small = {}
    for name, (L, h, K, H) in (("config3", (2, 500, C3_K, C3_H)), ("config1", (1, 32, C1_K, C1_H))):
        wls = make_workload_mountaincar(L, h)
        np.random.seed(4321)
        ag_host = make_nav_agent(eng, wls, K, H, device_sampling=False, planner=planner if world > 1 else None)
        ag_hrng = make_nav_agent(eng, wls, K, H, device_sampling=False, host_rng=True,
                                 planner=planner if world > 1 else None)
        ag_dev = make_nav_agent(eng, wls, K, H, device_sampling=True, planner=planner if world > 1 else None)
        prec_s = "bf16_tc" if eng.tc_supported() else "fp32"
        k_ms = []

        def resident(i):
            planner.plan(wls["state"], 0, K=K, H=H, seed=500 + i, act_low=wls["low"], act_high=wls["high"],
                         penalty_mode="reference", precision=prec_s, want_path=True)
            if i > 0:
                k_ms.append(dict(eng.last_timings()).get("mpc_rollout", 0.0))

        n_s = max(10, args.steps)
        eng.set_timing(True)
        res_ms = timed(resident, n_s, 3) / n_s                 # per-phase events on: gives the rollout kernel's time
        kern_ms = list(k_ms)
        eng.set_timing(False)                                  # the library's default
        fast_ms = timed(resident, n_s, 3) / n_s
        host_ms = timed(lambda i: ag_host.get_best_sim_actions(wls["state"]), n_s, 3) / n_s
        hrng_ms = timed(lambda i: ag_hrng.get_best_sim_actions(wls["state"]), n_s, 3) / n_s
        devs_ms = timed(lambda i: ag_dev.get_best_sim_actions(wls["state"]), n_s, 3) / n_s
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(n_s):
            ag_dev.get_best_sim_actions(wls["state"])
        wall_ms = 1e3 * (time.perf_counter() - t0) / n_s
        resident(0)
        kernel_name = eng.last_rollout_kernel()
        k_ms = kern_ms
        kern = float(np.mean(k_ms)) if k_ms else None
        small[name] = {
            "workload": "MountainCar d=2 da=1, K=%d (strong-scaled over %d GPU(s)), H=%d, MLP %dx%d, reference penalty"
                        % (K, world, H, L, h),
            "kernel": kernel_name,
            "ms_per_decision_resident": fast_ms, "ms_per_decision_resident_with_phase_events": res_ms,
            "rollout_kernel_ms": kern,
            "decision_over_rollout_kernel": (fast_ms / kern) if kern else None,
            "rollout_steps_per_s_resident": K * H / (fast_ms * 1e-3),
            "ms_per_decision_agent_default": host_ms, "rollout_steps_per_s_agent_default": K * H / (host_ms * 1e-3),
            "ms_per_decision_agent_host_rng": hrng_ms,
            "ms_per_decision_agent_device_sampling": devs_ms, "wall_ms_agent_device_sampling": wall_ms,
            "tensor_frac_of_burst_peak": (FLOP_PER_STEP[2] * K * H / (kern * 1e-3) / 1e12 / measured_peaks()["bf16_burst"])
            if (kern and prec_s == "bf16_tc") else None}
    eng.set_model(wl["w"], wl["b"], wl["norm"])
    eng.set_plan(wl["plan"]["desired_states"], wl["plan"]["distances_left"], wl["plan"]["radii"])

    # ---- row f1: dynamics-model training on the device (Dyn_Model.train, 30 epochs) -----------------
    dyn = None
    if rank == 0:
        from smartstartcontinuous_b200.dynamics_model import Dyn_Model
        tw = dyn_train_workload()
        nm = tw["norm"]
        model = Dyn_Model(4, 3, None, tw["lr"], tw["batch"], 2, 500, nm["mean_x"], nm["mean_y"], nm["mean_z"], nm["std_x"],
                          nm["std_y"], nm["std_z"], "float64", False, engine=eng, seed=0)
        model.set_weights(tw["w"], tw["b"])
        eng.dyn_reset_optimizer()
        np.random.seed(0)
        model.train(tw["X_old"], tw["Z_old"], tw["X_new"], tw["Z_new"], 1, None, tw["frac"], save_results=False)   # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tr_loss, old_loss, new_loss = model.train(tw["X_old"], tw["Z_old"], tw["X_new"], tw["Z_new"], tw["epochs"], None,
                                                  tw["frac"], save_results=False)
        torch.cuda.synchronize()
        train_s = time.perf_counter() - t0
        from oracle import dyn_train_oracle as dto_
        io, inw = dto_.epoch_batches(len(tw["X_old"]), len(tw["X_new"]), tw["batch"], tw["frac"])
        eng.dyn_train_batches(io, inw, tw["lr"], want_losses=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        eng.dyn_train_batches(io, inw, tw["lr"], want_losses=False)
        e1.record(stream)
        torch.cuda.synchronize()
        step_ms = e0.elapsed_time(e1) / len(io)
        fp32_peak = 148 * 128 * 2 * measured_peaks()["sm_max_mhz"] * 1e6 / 1e12
        dyn = {"workload": "Dyn_Model.train: %d old + %d new rows, MLP 2x500, batch 512 (52 old + 460 new), %d epochs x %d "
                           "Adam steps" % (len(tw["X_old"]), len(tw["X_new"]), tw["epochs"], len(io)),
               "training_s": train_s, "adam_steps": tw["epochs"] * len(io), "ms_per_adam_step_wall": 1e3 * train_s / (tw["epochs"] * len(io)),
               "ms_per_adam_step_device": step_ms, "final_training_loss": tr_loss, "old_loss": old_loss, "new_loss": new_loss,
               "roofline": {"bound": "fp32 (FFMA)", "achieved": DYN_FLOP_PER_STEP / (step_ms * 1e-3) / 1e12,
                            "peak": fp32_peak, "unit": "TFLOP/s", "frac": DYN_FLOP_PER_STEP / (step_ms * 1e-3) / 1e12 / fp32_peak,
                            "note": "0.77 GFLOP per step in 9 launches: latency-bound, not throughput-bound"}}
        eng.set_model(wl["w"], wl["b"], wl["norm"])
        eng.set_plan(wl["plan"]["desired_states"], wl["plan"]["distances_left"], wl["plan"]["radii"])

    # ---- multi-GPU self-check: the sharded decision equals the unsharded one ----------------------
    multi = None
    if world > 1:
        barrier()          # rank 0 comes from the training leg: nobody may spin in an exchange kernel waiting for it

        def same_decision(route):
            ok = True
            for mode in ("reference", "per_sample"):
                kwp = dict(K=20000, H=12, seed=7, act_low=wl["low"], act_high=wl["high"], penalty_mode=mode,
                           precision=precision)
                sh = planner.plan(wl["state"], 0, **kwp)
                torch.cuda.synchronize()
                one = eng.plan(wl["state"], 0, **kwp)
                ok &= sh["best_k"] == one["best_k"]
                ok &= abs(sh["best_score"] - one["best_score"]) <= 1e-5 * max(1.0, abs(one["best_score"]))
                ok &= bool(np.array_equal(sh["best_sequence"], one["best_sequence"]))
                ok &= bool(np.allclose(sh["best_path"], one["best_path"], rtol=1e-5, atol=1e-6))
            # numpy's MT19937 stream: every rank generates its slice of the one global draw on its GPU
            rs = np.random.RandomState(99)
            rs.random_sample(321)
            st0 = rs.get_state()
            kwm = dict(K=20000, H=12, act_low=wl["low"], act_high=wl["high"], penalty_mode="reference",
                       precision=precision, rng_state=st0)
            sh = planner.plan(wl["state"], 0, **kwm)
            torch.cuda.synchronize()
            one = eng.plan(wl["state"], 0, **kwm)
            rs.uniform(wl["low"], wl["high"], (20000, 12, 1))
            ok &= sh["best_k"] == one["best_k"] and bool(np.array_equal(sh["best_sequence"], one["best_sequence"]))
            for res in (sh, one):
                ok &= res["rng_state"][2] == rs.get_state()[2] and bool(np.array_equal(res["rng_state"][1], rs.get_state()[1]))
            return ok

        peer_was = eng.peer_ready
        ok_peer = same_decision("peer") if peer_was else None
        if peer_was:
            eng.peer_close()
        ok_nccl = same_decision("nccl")
        if peer_was:
            eng.peer_setup()                   # re-opening the exchange must work (fresh flags and epochs)
            ok_peer = bool(ok_peer) and same_decision("peer again")
        kws = kde_workload(n=20000, m=4096)
        sel = selector.select_start(kws["all_states"], kws["queries"], kws["values"], kws["n"], kws["volume"])
        one = eng.select_start(kws["all_states"], kws["queries"], kws["values"], kws["n"], kws["volume"])
        ok_kde = sel[0] == one[0] and abs(sel[1] - one[1]) <= 1e-9 * abs(one[1])
        flags = torch.tensor([1.0 if (ok_peer is None or ok_peer) else 0.0, 1.0 if ok_nccl else 0.0,
                              1.0 if ok_kde else 0.0], device=dev)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        multi = {"sharded_equals_single": bool(flags[0].item() == 1.0 and flags[1].item() == 1.0),
                 "sharded_equals_single_peer_memory": bool(flags[0].item() == 1.0) if peer_was else None,
                 "sharded_equals_single_nccl": bool(flags[1].item() == 1.0),
                 "kde_sharded_equals_single": bool(flags[2].item() == 1.0),
                 "check": "K=20000, H=12, reference and per-sample penalty (Philox) and numpy's MT19937 stream with every "
                          "rank generating its slice, %s: best_k and sequence identical, score "
                          "within 1e-5 relative, path within 1e-5, generator state after the draw = numpy's; KDE n=20000, m=4096: same index, ucb within 1e-9"
                          % precision}
    clocks = sampler.stop() if rank == 0 else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    info = eng.device_info()
    k_ms = float(np.mean(rollout_ms)) if rollout_ms else ms_per_step
    achieved_tf = FLOP_PER_STEP[3] * K_PER_GPU * HORIZON / (k_ms * 1e-3) / 1e12
    p_ms = float(np.mean(pairs_ms)) if pairs_ms else kde_ms
    sfu_peak = SFU_PER_CLK_PER_SM * info["sm_count"] * peaks["sm_max_mhz"] * 1e6
    kde_achieved = KDE_M * (KDE_N + 1) / (p_ms * 1e-3)
    kde_bytes = 4 * 3 * (KDE_N + 1 + KDE_M) + 4 * KDE_M + 8
    pkg_bytes = int(16 + HORIZON * 8 + (HORIZON + 1) * 3 * 8)
    cfg = shared_config(world)
    out = {
        "metric": "mpc_rollout_steps_per_s", "value": value, "unit": "rollout-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 (tcgen05, fp32 accumulate; first/last layer, state, scoring fp32)" if precision == "bf16_tc" else "f32",
        "data": "synthetic",
        "config": cfg,
        "run": {"actions": "device Philox4x32-10 for `value`; numpy's MT19937 stream generated on the device for `e2e`",
                "l2": "flushed between timed steps (256 MiB memset, outside the event-timed region)",
                "collective": ("peer-memory" if eng.peer_ready else ("nccl" if world > 1 else "none")),
                "parallelism": "K sharded over %d GPU(s); all-reduce of %d float64 + all-gather of the winner packages, %s"
                               % (world, 2 * (HORIZON + 1),
                                  "fused into the kernels over NVLink peer memory (csrc/peer.cu)" if eng.peer_ready
                                  else ("NCCL" if world > 1 else "none at N=1"))},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "rollout-steps/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(3 * 8 + 624 * 4 + 8), "d2h_bytes_per_step": int(pkg_bytes + 624 * 4 + 8),
                "same_decision_and_rng_state_as_host_draw": mt_same,
                "path": "NND_MB_agent.get_best_sim_actions in its default configuration: the K*H*da samples of "
                        "npr.uniform(low, high, (K, H, da)) (NND_MB_agent.py:500-501) are generated ON THE GPU from "
                        "np.random.get_state() -- numpy's MT19937 stream bit for bit, polynomial jump-ahead over the SMs "
                        "(csrc/mt19937.cu) -- and the advanced generator state is handed back with np.random.set_state; "
                        "inputs per decision: the state and the 2.5 KB generator key; outputs: winner package + key"},
        "e2e_host_rng": {"value": K_total * HORIZON / (e2e_host_rng_ms * 1e-3), "unit": "rollout-steps/s",
                         "ms_per_step": e2e_host_rng_ms, "h2d_bytes_per_step": int(n_act * 8 + 3 * 8),
                         "d2h_bytes_per_step": pkg_bytes, "host_rng_ms": rng_ms,
                         "path": "the same call with host_rng=True: the samples drawn on the host from the same stream "
                                 "(host_rng_ms of the step, inside the timer), uploaded inside the call"},
        "e2e_device_sampling": {"value": K_total * HORIZON / (e2e_dev_ms * 1e-3), "unit": "rollout-steps/s",
                                "ms_per_step": e2e_dev_ms, "h2d_bytes_per_step": 24, "d2h_bytes_per_step": pkg_bytes,
                                "path": "NND_MB_agent(device_sampling=True).get_best_sim_actions: state in, Philox on the "
                                        "GPU, winner package out"},
        "e2e_host_samples": {"value": K_total * HORIZON / (e2e_samples_ms * 1e-3), "unit": "rollout-steps/s",
                             "ms_per_step": e2e_samples_ms, "h2d_bytes_per_step": int(n_act * 8 + 3 * 8),
                             "d2h_bytes_per_step": pkg_bytes,
                             "path": "ShardedPlanner.plan -> ss_mpc_rollout / ss_mpc_finish_package on PRE-DRAWN float64 "
                                     "samples in pinned host memory (uploaded in chunks that overlap the rollout)"},
        "gpu_launches": int(launches),
        "per_sample_penalty": {"value": K_total * HORIZON / (per_sample_ms * 1e-3), "unit": "rollout-steps/s",
                               "ms_per_step": per_sample_ms,
                               "note": "penalty_mode=per_sample (fully fused scoring, no penalty passes)"},
        "roofline": {"bound": "tensor", "achieved": achieved_tf, "peak": peaks["bf16_burst"], "unit": "TFLOP/s",
                     "frac": achieved_tf / peaks["bf16_burst"],
                     "traffic": NCU_TRAFFIC["mpc_rollout_tc_kernel"] if precision == "bf16_tc" else None,
                     "traffic_source": NCU_TRAFFIC_SOURCE,
                     "frac_of_sustained_peak": achieved_tf / peaks["bf16_sustained"],
                     "kernel": "mpc_rollout_tc_kernel" if precision == "bf16_tc" else "mpc_rollout_simt_kernel",
                     "kernel_ms": k_ms,
                     "peak_source": peaks["source"] + " (bf16_tflops, the burst figure: the timed region is a few tens of ms "
                                                      "at the maximum SM clock)",
                     "algorithmic_flop_per_rollout_step": FLOP_PER_STEP[3]},
        "kde": {"metric": "kde_kernel_evals_per_s", "value": kde_value, "unit": "kernel-evals/s", "ms_per_step": kde_ms,
                "config": {"workload": "KDE+UCB+argmax, %d Pendulum states (d=3) x %d queries per GPU (BASELINE config 2)"
                                       % (KDE_N + 1, KDE_M)},
                "e2e": {"value": evals / (kde_agent_ms * 1e-3), "unit": "kernel-evals/s", "ms_per_step": kde_agent_ms,
                        "h2d_bytes_per_step": int(12 * KDE_M), "d2h_bytes_per_step": 16,
                        "host_value_fn_ms": kde_value_fn_ms,
                        "path": "SmartStartContinuous.get_smart_start_path (smartexplorationcontinuous.py:223-305): "
                                "random.sample of the candidates (the interpreter's stream, drawn in C++: "
                                "csrc/py_random.cu), the base agent's get_state_value on the host (host_value_fn_ms, a "
                                "numpy stand-in for the user's TF critic), selection from the device mirror "
                                "of the replay buffer (row indices + values uploaded), episodic path extraction"},
                "e2e_device_values": {"value": evals / (kde_agent_dev_ms * 1e-3), "unit": "kernel-evals/s",
                                      "ms_per_step": kde_agent_dev_ms, "h2d_bytes_per_step": int(8 * KDE_M),
                                      "d2h_bytes_per_step": 16,
                                      "path": "the same call with value_net= the agent's actor / critic parameters: "
                                              "V = critic(q, actor(q)) evaluated on the device in front of the UCB "
                                              "(row f4), only the candidate row indices are uploaded"},
                "e2e_full_upload": {"value": evals / (kde_e2e_ms * 1e-3), "unit": "kernel-evals/s", "ms_per_step": kde_e2e_ms,
                                    "h2d_bytes_per_step": int(8 * 3 * (KDE_N + 1 + KDE_M) + 4 * KDE_M), "d2h_bytes_per_step": 16,
                                    "path": "ss_kde_ucb_argmax with host float64 buffers (whole data set uploaded)"},
                "n_ss_2000": {"workload": "%d states x %d queries (the example's n_ss)" % (KDE_N + 1, C1_NSS),
                              "ms_per_step": kde2k_ms, "value": C1_NSS * (KDE_N + 1) / (kde2k_ms * 1e-3),
                              "pairs_kernel_ms": float(np.mean(pairs2k_ms)) if pairs2k_ms else None,
                              "frac_of_sfu_peak": (C1_NSS * (KDE_N + 1) / (float(np.mean(pairs2k_ms)) * 1e-3) / sfu_peak)
                              if pairs2k_ms else None,
                              "ms_per_step_agent": kde2k_agent_ms},
                "roofline": {"bound": "sfu", "achieved": kde_achieved, "peak": sfu_peak, "unit": "kernel-evals/s",
                             "frac": kde_achieved / sfu_peak, "kernel": "kde_pairs_tc_kernel", "kernel_ms": p_ms,
                             "peak_source": "16 MUFU.EX2/clk/SM x %d SMs x %.0f MHz (max SM clock); the kernel takes 3/8 of "
                                            "its exp2 evaluations on the FMA pipe (polynomial) and the exponents from the "
                                            "tensor pipe, so frac > 1 is possible" % (info["sm_count"], peaks["sm_max_mhz"]),
                             "hbm_achieved_gbs": kde_bytes / (p_ms * 1e-3) / 1e9, "hbm_peak_gbs": peaks["hbm_gbs"],
                             "traffic": NCU_TRAFFIC["kde_pairs_tc_kernel"],
                             "traffic_source": NCU_TRAFFIC_SOURCE}},
        "small_k": small,
        "dyn_train": dyn,
    }
    if multi is not None:
        out["multi_gpu_check"] = multi
        out["sharded_equals_single"] = multi["sharded_equals_single"]
        out["collective"] = out["run"]["collective"]
    out["config5"] = {"workload": "BASELINE config 5, strong scaling over %d GPU(s): KDE 1 000 001 states x %d queries "
                                  "(queries sharded) + MPC K=%d total, H=%d (sequences sharded), device-resident"
                                  % (world, KDE_M, C5_K, HORIZON),
                      "kde_ms": c5_kde_ms, "kde_evals_per_s": KDE_M * 1_000_001 / (c5_kde_ms * 1e-3),
                      "mpc_ms": c5_mpc_ms, "mpc_rollout_steps_per_s": C5_K * HORIZON / (c5_mpc_ms * 1e-3),
                      "episode_ms": c5_kde_ms + c5_mpc_ms}
    # ---- row f3 (plan set-up): pair extraction of path_shortcutter, P = 1000 path states ----------
    try:
        from smartstartcontinuous_b200 import numerical as num
        from smartstartcontinuous_b200 import synthetic as syn
        obs, _ = syn.pendulum_rollouts(np.random.default_rng(7), 1, 1000)
        path = np.asarray(obs[0][:1000])
        stds, means = num.path_deltas_stds_and_means_per_dim(path)
        radii = num.radii_calc(means, stds, 1, 1, 1)
        dist_fn = num.elliptical_euclidean_distance_function_generator(radii)
        eng.path_shortcut(path, radii, 1.0)
        t0 = time.perf_counter()
        for _ in range(10):
            keep = eng.path_shortcut(path, radii, 1.0)
        t_full_dev = (time.perf_counter() - t0) / 10
        t0 = time.perf_counter()
        host_path = num.path_shortcutter(path, dist_fn, 1.0)
        t_full_host = time.perf_counter() - t0
        out["plan_setup"] = {"what": "path_shortcutter (numerical.py:226-246), P=1000, d=3, host buffers in and out",
                             "shortcut_gpu_ms": 1e3 * t_full_dev, "shortcut_host_ms": 1e3 * t_full_host,
                             "shortcut_identical": bool(np.array_equal(path[keep], host_path)),
                             "kept_states": int(len(keep))}
    except Exception as exc:
        out["plan_setup"] = {"error": repr(exc)}
    if world == 1 and not args.no_cpu_baseline:
        # the CPU leg runs in a fresh process (fork-based pool, no CUDA context): the same code as
        # `--impl reference`, ~20-30 s of CPU work on bounded samples of the workload
        try:
            ref = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "6",
                                  "--warmup", "1", "--no-full-step"], capture_output=True, text=True, timeout=900)
            r = json.loads(ref.stdout.strip().splitlines()[-1])
            out["cpu_baseline"] = r["cpu_baseline"]
            out["kde"]["cpu_baseline"] = {k: r["kde"][k] for k in ("value", "unit", "cores", "kind", "sample", "single_core")}
            for name in small:
                small[name]["cpu_baseline"] = r["small_k"].get(name)
            if dyn is not None:
                dyn["cpu_baseline"] = r["small_k"].get("dyn_train")
        except Exception as exc:                                     # never lose the GPU line
            out["cpu_baseline"] = {"value": None, "unit": "rollout-steps/s", "cores": 0, "kind": "port",
                                   "sample": "failed: %r" % (exc,)}
    guard.emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
