"""Development helper: cost of the float64 device trainer (ss_dyn_set_precision(SS_PRECISION_FP64)) next to the FP32
trainer on the 2x500 training workload of bench.dyn_train_workload() (52 old + 460 new rows per batch, 160 Adam
steps per epoch).  Per precision: device time per Adam step (CUDA events around one epoch, best of 3 after a warm-up
epoch), wall time of the 30-epoch training (batches drawn per epoch with the reference's numpy calls, as
Dyn_Model.train does), and the GEMM kernels' time from torch.profiler over one epoch with their FP64 rate against
the card's DFMA peak (scripts/dev/micro/fp64_peak.cu, measured in the same command).  Writes one JSON document to
the path given (default: stdout)."""
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from fp64_time import card, fp64_peak  # noqa: E402
from oracle import dyn_train_oracle as dto  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402


def main(out_path=None):
    eng = Engine(0)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    tw = bench.dyn_train_workload()
    n_old, n_new = len(tw["X_old"]), len(tw["X_new"])
    B, h = tw["batch"], 500
    gemm_flop_per_step = 3 * 2.0 * B * h * h            # hidden forward, dH and dW of the one h x h layer
    result = dict(card=card(), peak=fp64_peak(), workload="bench.dyn_train_workload(): %d old + %d new rows, MLP 2x500, "
                  "batch %d, %d epochs" % (n_old, n_new, B, tw["epochs"]), gemm_flop_per_step=gemm_flop_per_step,
                  rows=[])
    for prec in ("fp32", "fp64"):
        eng.set_model(tw["w"], tw["b"], tw["norm"])
        eng.dyn_set_precision(prec)
        eng.dyn_reset_optimizer()
        eng.dyn_set_data(0, tw["X_old"], tw["Z_old"])
        eng.dyn_set_data(1, tw["X_new"], tw["Z_new"])
        np.random.seed(0)
        io, inw = dto.epoch_batches(n_old, n_new, B, tw["frac"])
        eng.dyn_train_batches(io, inw, tw["lr"], want_losses=False)
        torch.cuda.synchronize()
        step = []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.dyn_train_batches(io, inw, tw["lr"], want_losses=False)
            e1.record()
            e1.synchronize()
            step.append(e0.elapsed_time(e1) * 1e-3 / len(io))
        # 30 epochs from the initial weights, as Dyn_Model.train runs them
        eng.set_model(tw["w"], tw["b"], tw["norm"])
        eng.dyn_reset_optimizer()
        np.random.seed(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(tw["epochs"]):
            e_io, e_inw = dto.epoch_batches(n_old, n_new, B, tw["frac"])
            eng.dyn_train_batches(e_io, e_inw, tw["lr"])              # the per-epoch loss read-back synchronises
        train_s = time.perf_counter() - t0
        # kernel times of one epoch
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            eng.dyn_train_batches(io, inw, tw["lr"], want_losses=False)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if "dyn_" in ev.key and ev.self_device_time_total > 0:
                name = ev.key[ev.key.index("dyn_"):].split("(")[0]
                kern[name] = kern.get(name, 0.0) + ev.self_device_time_total * 1e-6
        gemm_s = sum(v for k, v in kern.items() if "dyn_gemm_kernel" in k) / len(io)
        row = dict(precision=prec, adam_step_s=min(step), train_30_epochs_s=train_s, steps_per_epoch=len(io),
                   kernel_s_per_step={k: v / len(io) for k, v in sorted(kern.items())}, gemm_s_per_step=gemm_s,
                   gemm_tflops=gemm_flop_per_step / gemm_s / 1e12)
        if prec == "fp64":
            row["gemm_share_of_dfma_peak"] = row["gemm_tflops"] / result["peak"]["dfma_tflops"]
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
    result["fp64_over_fp32_step"] = result["rows"][1]["adam_step_s"] / result["rows"][0]["adam_step_s"]
    eng.dyn_set_precision("fp32")
    eng.close()
    text = json.dumps(result, indent=1)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
