"""Development helper: cost of the float64 selection (ss_kde_set_precision(SS_PRECISION_FP64)) next to the default
FP32 path, with data, candidates and values resident on the device (select_start_dev).  Workloads: config 2
(100 001 points x 16 384 candidates), the example's n_ss = 2000 on the same buffer, and the config-5 shard
(1 000 001 x 16 384), all d = 3.  Per workload and precision: ms per call (host clock around calls that end with
the result in host memory, median of 10 after a warm-up), the pair kernel's time (the "kde_pairs" phase of
ss_last_timings, CUDA events, median of 10), evaluations per second, and for FP64 the pair kernel's FP64
instruction rate against the card's DFMA rate (scripts/dev/micro/fp64_peak.cu, measured in the same command).
Writes one JSON document to the path given (default: stdout)."""
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

from fp64_time import card, fp64_peak  # noqa: E402
from smartstartcontinuous_b200 import synthetic as syn  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402

# FP64-pipe instructions (DFMA, DADD, DMUL, DSETP) per (query, point) pair on the fast path of
# kde_pairs_fp64_kernel<3, 4>: 224 in the unrolled loop body (2 points x 4 queries), outside the blocks exp() only
# enters for arguments near its overflow / underflow limits -- counted from cuobjdump -sass of the sm_100a build.
FP64_INSTR_PER_PAIR_D3 = 28


def workloads():
    buf2, s2_2, _ = syn.pendulum_buffer(100_000, seed=0)
    rng = np.random.default_rng(0)
    q2 = s2_2[rng.choice(100_000, 16_384, replace=False)]
    yield "config2 100001 x 16384", buf2, q2, 100_000
    yield "n_ss 2000, 100001 x 2000", buf2, q2[:2000], 100_000
    buf5, s2_5, _ = syn.pendulum_buffer(1_000_000, seed=1)
    rng = np.random.default_rng(1)
    yield "config5 shard 1000001 x 16384", buf5, s2_5[rng.choice(1_000_000, 16_384, replace=False)], 1_000_000


def main(out_path=None):
    eng = Engine(0)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    peak = fp64_peak()
    result = dict(card=card(), peak=peak, fp64_instr_per_pair_d3=FP64_INSTR_PER_PAIR_D3, rows=[])
    dfma_instr_per_s = peak["dfma_tflops"] * 1e12 / 2
    for name, data, q, n_tr in workloads():
        dev = torch.device("cuda", 0)
        X = torch.from_numpy(np.ascontiguousarray(data)).to(dev)
        Q = torch.from_numpy(np.ascontiguousarray(q)).to(dev)
        V = torch.from_numpy(syn.critic_like_values(q)).to(dev)
        pairs = float(len(data)) * len(q)

        def call():
            return eng.select_start_dev(X.data_ptr(), len(data), data.shape[1], Q.data_ptr(), len(q), V.data_ptr(),
                                        n_tr, 1.0, 1.0, 2.0)
        for prec in ("fp32", "fp64"):
            eng.kde_set_precision(prec)
            call()
            torch.cuda.synchronize()
            wall = []
            for _ in range(10):
                t0 = time.perf_counter()
                call()
                wall.append(time.perf_counter() - t0)
            eng.set_timing(True)
            pair = []
            for _ in range(10):
                call()
                pair.append(dict(eng.last_timings())["kde_pairs"] * 1e-3)
            eng.set_timing(False)
            row = dict(workload=name, precision=prec, n_points=len(data), m=len(q), call_ms=float(np.median(wall)) * 1e3,
                       pair_kernel_ms=float(np.median(pair)) * 1e3, evals_per_s=pairs / float(np.median(pair)))
            if prec == "fp64":
                rate = row["evals_per_s"] * FP64_INSTR_PER_PAIR_D3
                row.update(fp64_instr_per_s=rate, share_of_dfma_instr_rate=rate / dfma_instr_per_s)
            result["rows"].append(row)
            print(json.dumps(row), flush=True)
    eng.kde_set_precision("fp32")
    eng.close()
    text = json.dumps(result, indent=1)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
