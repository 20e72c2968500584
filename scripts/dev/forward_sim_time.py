"""Development helper: Engine.forward_sim (ss_mpc_forward_sim) time from per-sequence start states next to one shared
start, for precisions "fp32", "bf16_tc" and "fp64", at BASELINE config 3 (MountainCar, K = 4096, H = 20, 2 x 500),
the config-4 shard (Pendulum, K = 131 072, H = 50, 2 x 500) and a k-step validation workload (20 Pendulum rollouts of
333 steps, every window start a sequence: K = 20 x 323 = 6460, H = 10, 2 x 500).  Writes one JSON document to the
path given (default: stdout), with the card's name and power limit read in the same run.

Times (best of N after warm-up): call = wall clock around forward_sim (it returns after the states are on the host);
kernel = the library's "mpc_rollout" phase event (ss_set_timing(1), a separate pass); copy = wall clock around
get_states(), the device -> host copy and widening of the [H+1, K, d] states that forward_sim ends with."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import bench  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402

CONFIGS = [("c3", "mountaincar", 4096, 20, 10), ("c4_shard", "pendulum", 131072, 50, 3),
           ("validation", "pendulum", 20 * (333 - 10), 10, 10)]
PRECISIONS = ["fp32", "bf16_tc", "fp64"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def best(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts)


def main(out_path=None):
    eng = Engine(0)
    result = dict(card=card(), configs=[])
    for name, env, K, H, reps in CONFIGS:
        wl = bench.make_workload() if env == "pendulum" else bench.make_workload_mountaincar(2, 500)
        eng.set_model(wl["w"], wl["b"], wl["norm"])
        rng = np.random.default_rng(0)
        d, da = wl["d"], wl["da"]
        std = np.asarray(wl["norm"]["std_x"], dtype=np.float64)
        rows = np.asarray(wl["state"], dtype=np.float64) + 0.5 * std * rng.normal(size=(K, d))
        acts = rng.uniform(wl["low"], wl["high"], (K, H, da))
        for prec in PRECISIONS:
            if prec == "bf16_tc" and not eng.tc_supported():
                continue
            for starts_kind, starts in (("per_row", rows), ("shared", rows[0])):
                call = lambda: eng.forward_sim(starts, acts, prec)
                for _ in range(2):
                    call()
                call_s = best(call, reps)
                copy_s = best(eng.get_states, reps)
                eng.set_timing(True)
                kern = []
                for _ in range(reps):
                    call()
                    kern.append(dict(eng.last_timings()).get("mpc_rollout", float("nan")) * 1e-3)
                eng.set_timing(False)
                row = dict(config=name, env=env, K=K, H=H, d=d, da=da, precision=prec, starts=starts_kind,
                           kernel=eng.last_rollout_kernel(), call_s=call_s, kernel_s=min(kern), copy_s=copy_s)
                result["configs"].append(row)
                print(json.dumps(row), flush=True)
    eng.close()
    text = json.dumps(result, indent=1)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
