"""Development helper: decision time of precision="fp64" next to "fp32" and "bf16_tc" at BASELINE configs 1, 3 and
the config-4 shard, the fp64 rollout kernel's FP64 rate, and the FP64 peak of the card (scripts/dev/micro/fp64_peak.cu,
DFMA and DMMA) as its denominator.  Writes one JSON document to the path given (default: stdout).

Times: device = CUDA events around one decision on the engine's stream (torch's current stream); host = wall clock
from the call to the returned result; rollout kernel = the library's "mpc_rollout" phase event (ss_set_timing(1),
taken in a separate pass so that its events do not count in the decision times).  Best of N after warm-up.
FLOP per rollout-step = 2 [(d + da) h + (L - 1) h^2 + h d]."""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402

CONFIGS = [("c1", "mountaincar", 1, 32, 5000, 4, 20), ("c3", "mountaincar", 2, 500, 4096, 20, 10),
           ("c4_shard", "pendulum", 2, 500, 131072, 50, 3)]
PRECISIONS = ["fp64", "fp32", "bf16_tc"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def fp64_peak():
    src = os.path.join(ROOT, "scripts", "dev", "micro", "fp64_peak.cu")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "fp64_peak")
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe, src])
        return json.loads(subprocess.check_output([exe]).decode().strip().splitlines()[-1])


def main(out_path=None):
    eng = Engine(0)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    result = dict(card=card(), peak=fp64_peak(), configs=[])
    for name, env, L, h, K, H, reps in CONFIGS:
        wl = bench.make_workload() if env == "pendulum" else bench.make_workload_mountaincar(L, h)
        eng.set_model(wl["w"], wl["b"], wl["norm"])
        eng.set_plan(wl["plan"]["desired_states"], wl["plan"]["distances_left"], wl["plan"]["radii"])
        d, da = wl["d"], wl["da"]
        flop = 2.0 * ((d + da) * h + (L - 1) * h * h + h * d) * K * H
        for prec in PRECISIONS:
            if prec == "bf16_tc" and not eng.tc_supported():
                continue

            def decide(i):
                return eng.plan(wl["state"], 0, K=K, H=H, seed=100 + i, act_low=wl["low"], act_high=wl["high"],
                                penalty_mode="reference", precision=prec)

            for i in range(2):
                decide(i)
            dev, host = [], []
            for i in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                e0.record()
                decide(i)
                e1.record()
                host.append(time.perf_counter() - t0)
                e1.synchronize()
                dev.append(e0.elapsed_time(e1) * 1e-3)
            eng.set_timing(True)
            kern = []
            for i in range(reps):
                decide(i)
                kern.append(dict(eng.last_timings()).get("mpc_rollout", float("nan")) * 1e-3)
            eng.set_timing(False)
            row = dict(config=name, env=env, L=L, h=h, K=K, H=H, precision=prec, kernel=eng.last_rollout_kernel(),
                       decision_device_s=min(dev), decision_host_s=min(host), rollout_kernel_s=min(kern),
                       flop=flop, rollout_tflops=flop / min(kern) / 1e12)
            if prec == "fp64":
                row["share_of_dfma_peak"] = row["rollout_tflops"] / result["peak"]["dfma_tflops"]
                row["share_of_dmma_peak"] = row["rollout_tflops"] / result["peak"]["dmma_tflops"]
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
