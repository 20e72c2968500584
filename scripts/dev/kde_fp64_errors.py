"""Development helper: how often each selection precision makes the float64 choice at config-2 size.  For each seed:
synthetic.pendulum_buffer(100 000, seed) (100 001 points), 16 384 candidates drawn from its s2 rows,
critic_like_values, alpha = 1, beta = 2, volume = 1.  The float64 choice is the argmax of numpy's UCB expression
(float32 values) over the densities of scipy's fitted estimator (its cho_cov, weights and normalisation) summed in
float64 on the GPU with torch from direct differences -- a float64 evaluation independent of the library.  Records
the top-two relative UCB gap, the largest relative density error of each precision against scipy itself on a
256-candidate subset, and whether each precision's pick equals the float64 choice.  Writes one JSON document to the
path given (default: stdout)."""
import json
import math
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import numpy as np  # noqa: E402
import scipy.linalg  # noqa: E402
import scipy.stats  # noqa: E402
import torch  # noqa: E402

from fp64_time import card  # noqa: E402
from smartstartcontinuous_b200 import synthetic as syn  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402

SEEDS = range(24)


def float64_density(kde, q, chunk=256):
    """scipy's estimator summed in float64 with torch: sum_i w * exp(-|P_i - Z_j|^2 / 2) * norm."""
    L = kde.cho_cov
    P = torch.from_numpy(scipy.linalg.solve_triangular(L, kde.dataset, lower=True).T.copy()).cuda()
    Z = torch.from_numpy(scipy.linalg.solve_triangular(L, q.T, lower=True).T.copy()).cuda()
    norm = math.pow(2 * math.pi, -kde.d / 2.0) / float(np.prod(np.diag(L)))
    w = float(kde.weights[0])
    out = []
    for s in range(0, len(Z), chunk):
        r = P[None, :, :] - Z[s:s + chunk, None, :]
        out.append((w * (torch.exp(-(r * r).sum(-1) / 2) * norm)).sum(1))
    return torch.cat(out).cpu().numpy()


def main(out_path=None):
    eng = Engine(0)
    result = dict(card=card(), workload="pendulum_buffer(100000, seed): 100001 points x 16384 candidates, d = 3, "
                  "alpha 1, beta 2, volume 1", seeds=[])
    agree = {"fp32": 0, "fp64": 0}
    for seed in SEEDS:
        data, s2, _ = syn.pendulum_buffer(100_000, seed=seed)
        rng = np.random.default_rng(seed)
        q = s2[rng.choice(100_000, 16_384, replace=False)]
        vals = syn.critic_like_values(q)
        kde = scipy.stats.gaussian_kde(data.T, bw_method="scott")
        with np.errstate(divide="ignore"):
            oucb = vals + np.sqrt((2.0 * np.log(100_000)) / (100_000 * float64_density(kde, q)))
        top = np.sort(oucb)[::-1]
        sub = np.sort(rng.choice(16_384, 256, replace=False))
        sdens = kde(q[sub].T)
        row = dict(seed=seed, top_two_gap=float((top[0] - top[1]) / abs(top[0])), float64_pick=int(np.argmax(oucb)))
        for prec in ("fp32", "fp64"):
            eng.kde_set_precision(prec)
            best, _, dens, _ = eng.select_start(data, q, vals, 100_000, 1.0, 1.0, 2.0, want_density=True)
            row[prec + "_pick"] = best
            row[prec + "_max_rel_density_error_vs_scipy"] = float(np.max(np.abs(dens[sub] - sdens) / sdens))
            agree[prec] += int(best == row["float64_pick"])
        result["seeds"].append(row)
        print(json.dumps(row), flush=True)
    result["picks_equal_to_float64_choice"] = dict(agree, of=len(SEEDS))
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
