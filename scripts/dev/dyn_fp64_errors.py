"""Development helper: what the float64 trainer changes for the planner.

The full 30-epoch training of bench.dyn_train_workload() (2x500, 160 Adam steps per epoch) runs on the same batches
with the float64 oracle (oracle/dyn_train_oracle.py, numpy on the CPU), with the FP32 device trainer and with the
float64 device trainer.  A fourth run is the oracle again with the rows of every batch permuted (old rows reversed,
new rows reversed): the same mathematics, a different summation order in the gradient reductions -- how far two
float64 implementations that differ only in summation order drift apart on this training trajectory.

Per epoch: parameter error of each run against the oracle (worst Frobenius error over the Frobenius movement, and
worst element error over the largest element movement).  After epochs 1, 5 and 30: 50 decisions of the config-3
size (K = 4096, H = 20, Philox samples, start states along the Pendulum plan of bench.make_workload()) with
precision="fp64" from each set of weights; recorded: how many differ from the decisions with the oracle's weights,
the largest score difference, and the oracle-weight top-2 score gaps.  Also the measured errors of the four oracle
cases of tests/test_gpu_dyn_train_fp64.py.  Writes JSON to the path given (default: stdout)."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import bench  # noqa: E402
from oracle import dyn_train_oracle as dto  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402
from test_gpu_dyn_train_fp64 import ORACLE_CASES, oracle_case, param_errors  # noqa: E402

N_DECISIONS, K, H = 50, 4096, 20
CHECKPOINTS = (1, 5, 30)


def snapshot(w, b):
    return [a.copy() for a in w], [a.copy() for a in b]


def oracle_run(tw, batches, permute):
    w, b = snapshot(tw["w"], tw["b"])
    state = dto.AdamState(w, b)
    snaps = []
    for io, inw in batches:
        if permute:
            io, inw = io[:, ::-1], inw[:, ::-1]
        dto.train_batches(w, b, state, tw["X_old"], tw["Z_old"], tw["X_new"], tw["Z_new"], io, inw, tw["lr"])
        snaps.append(snapshot(w, b))
    return snaps


def device_run(eng, tw, batches, prec):
    eng.set_model(tw["w"], tw["b"], tw["norm"])
    eng.dyn_set_precision(prec)
    eng.dyn_reset_optimizer()
    eng.dyn_set_data(0, tw["X_old"], tw["Z_old"])
    eng.dyn_set_data(1, tw["X_new"], tw["Z_new"])
    snaps = []
    for io, inw in batches:
        eng.dyn_train_batches(io, inw, tw["lr"], want_losses=False)
        snaps.append(eng.dyn_get_params())
    eng.dyn_set_precision("fp32")
    return snaps


def main(out_path=None):
    eng = Engine(0)
    out = dict(oracle_cases=[])
    for cfg in ORACLE_CASES:
        out["oracle_cases"].append(dict(cfg=dict(zip(("d", "da", "L", "h", "batch", "frac", "steps"), cfg)),
                                        **oracle_case(eng, cfg)))
        print(json.dumps(out["oracle_cases"][-1]), flush=True)
    eng.dyn_set_precision("fp32")
    tw = bench.dyn_train_workload()
    n_old, n_new = len(tw["X_old"]), len(tw["X_new"])
    np.random.seed(0)
    batches = [dto.epoch_batches(n_old, n_new, tw["batch"], tw["frac"]) for _ in range(tw["epochs"])]
    t0 = time.perf_counter()
    runs = {"oracle": oracle_run(tw, batches, False)}
    oracle_s = time.perf_counter() - t0
    runs["oracle_permuted_rows"] = oracle_run(tw, batches, True)
    runs["fp32_trainer"] = device_run(eng, tw, batches, "fp32")
    runs["fp64_trainer"] = device_run(eng, tw, batches, "fp64")
    init = tw["w"] + tw["b"]
    out["training"] = dict(epochs=tw["epochs"], adam_steps=sum(len(io) for io, _ in batches), oracle_cpu_s=oracle_s,
                           per_epoch={})
    for name in ("oracle_permuted_rows", "fp32_trainer", "fp64_trainer"):
        errs = [param_errors(w + b, ow + ob, init) for (w, b), (ow, ob) in zip(runs[name], runs["oracle"])]
        out["training"]["per_epoch"][name] = dict(param_frob_over_movement=[e[0] for e in errs],
                                                  param_elem_over_max_movement=[e[1] for e in errs])
        print(name, "after epochs 1, 5, 30:", [errs[c - 1] for c in CHECKPOINTS], flush=True)
    wl = bench.make_workload()
    p = wl["plan"]
    starts = wl["path"][:N_DECISIONS]
    out["decisions"] = dict(count=N_DECISIONS, K=K, H=H, precision="fp64", after_epoch={})
    for c in CHECKPOINTS:
        scores = {}
        for name, snaps in runs.items():
            w, b = snaps[c - 1]
            eng.set_model(w, b, tw["norm"])
            eng.set_plan(p["desired_states"], p["distances_left"], p["radii"])
            scores[name] = [eng.plan(starts[i], 0, K=K, H=H, seed=1000 + i, act_low=wl["low"], act_high=wl["high"],
                                     precision="fp64", want_scores=True)["scores"] for i in range(N_DECISIONS)]
        gaps = [float(np.diff(np.sort(s)[-2:])[0]) for s in scores["oracle"]]
        best = {name: [int(np.argmax(s)) for s in v] for name, v in scores.items()}
        row = dict(oracle_top2_gap_min=min(gaps), oracle_top2_gap_median=float(np.median(gaps)), oracle_top2_gaps=gaps)
        for name in ("oracle_permuted_rows", "fp32_trainer", "fp64_trainer"):
            err = max(float(np.max(np.abs(a - o) / np.maximum(np.abs(o), 1.0)))
                      for a, o in zip(scores[name], scores["oracle"]))
            row[name] = dict(differing_decisions=sum(x != y for x, y in zip(best[name], best["oracle"])),
                             max_score_err_rel=err)
        out["decisions"]["after_epoch"][c] = row
        print("epoch", c, json.dumps({k: v for k, v in row.items() if k != "oracle_top2_gaps"}), flush=True)
    eng.close()
    text = json.dumps(out, indent=1)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
