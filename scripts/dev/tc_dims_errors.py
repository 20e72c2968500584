"""Development helper: errors of the tcgen05 rollout kernels against the float64 oracle at every state / action
dimension of tests/test_gpu_mpc_dims.py, on exactly the problems that file checks (its host-sample rows on the pair
and quad kernels, the Philox and MT19937 rows, the model after device training with both trainers), in both penalty
modes.  Per case: score error max / p99.9 / p99 / median, state and path error over the per-dimension scale, the
oracle's top-2 gap and whether the arg-best equals the oracle's.  Per shape (d, da, h): the largest of each over its
cases, and the bounds 3x those maxima suggest.  Writes JSON (with the card's name and power limit) to the path given.

  python scripts/dev/tc_dims_errors.py OUT.json
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import test_gpu_mpc_dims as t  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power = [x.strip() for x in q.split(",")]
    return dict(name=name, power_limit=power)


def record(case_name, row, mode, case):
    p, res, states, acts, o = case
    e = t._errors(row, p, res, states, acts, o)
    se = e["score_err"]
    return dict(case=case_name, row=t._row_id(row), shape=[row.d, row.da, row.h], kernel=row.kernel, mode=mode,
                K=int(acts.shape[0]), H=int(acts.shape[1]),
                score_err_max=float(se.max()), score_err_p999=float(np.percentile(se, 99.9)),
                score_err_p99=float(np.percentile(se, 99)), score_err_median=float(np.median(se)),
                state_err_over_scale=None if e["state_err"] is None else float(e["state_err"].max()),
                path_err_over_scale=float(e["path_err"].max()), top2_gap=e["top2_gap"],
                best_k=int(res["best_k"]), oracle_best_k=e["oracle_best_k"],
                same_best=bool(res["best_k"] == e["oracle_best_k"]))


def main(out_path):
    info = card()
    print(json.dumps(info), flush=True)
    eng = Engine(0)
    cases = []

    def add(name, row, mode, case):
        cases.append(record(name, row, mode, case))
        print(json.dumps(cases[-1]), flush=True)

    for mode in t.MODES:
        for row in t.TC_ROWS + t.QUAD_ROWS:
            add("host samples", row, mode, t.run_host_case(eng, row, mode))
        row = t.SAMPLED_ROWS[0]
        add("philox samples", row, mode, t.run_philox_case(eng, row, mode))
    add("mt19937 samples", t.TC_ROWS[1], "reference", t.run_mt19937_case(eng)[0])
    for train_precision in ("fp32", "fp64"):
        p, trained = t.train_and_commit(eng, train_precision)
        for mode in t.MODES:
            for row, case in t.run_commit_cases(eng, p, trained, mode):
                if row.kernel != t.SIMT:
                    add("after %s training + commit" % train_precision, row, mode, case)
    eng.dyn_set_precision("fp32")
    eng.close()

    shapes = {}
    for c in cases:
        s = shapes.setdefault("%d,%d,%d" % tuple(c["shape"]), dict(score_err_p99=0.0, score_err_median=0.0,
                                                                   score_err_max=0.0, state_err_over_scale=0.0,
                                                                   path_err_over_scale=0.0))
        for k in s:
            if c[k] is not None:
                s[k] = max(s[k], c[k])
    for s in shapes.values():
        s["score_atol_3x_p99"] = 3 * s["score_err_p99"]
    overall = dict(score_err_median=max(s["score_err_median"] for s in shapes.values()),
                   state_or_path_err_over_scale=max(max(s["state_err_over_scale"], s["path_err_over_scale"])
                                                    for s in shapes.values()),
                   all_same_best=all(c["same_best"] for c in cases))
    out = dict(card=info, overall=overall, shapes=shapes, cases=cases)
    print(json.dumps(dict(overall=overall, shapes=shapes), indent=1), flush=True)
    with open(out_path, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
