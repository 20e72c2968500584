"""Development helper: errors of precision="fp64" against the reference's goldens and the float64 oracle (the fp64 row
of DESIGN.md 3.4).  Per case: max state error / per-dimension scale, max score error / max(|score|, 1), max path
error / scale, the oracle's top-2 gap, and whether the arg-best equals the oracle's.  Writes JSON to the path given."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import bench  # noqa: E402
from conftest import golden_model, load_golden  # noqa: E402
from oracle import mpc_oracle, philox  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402


def report(name, res, states, o):
    scale = np.maximum(np.abs(o["states"]).max(axis=(0, 1)), 1e-300)
    top2 = np.sort(o["scores"])[-2:]
    return dict(case=name, K=int(o["scores"].shape[0]), H=int(o["states"].shape[0] - 1),
                state_err_over_scale=float((np.abs(states - o["states"]).max(axis=(0, 1)) / scale).max()),
                score_err_rel=float((np.abs(res["scores"] - o["scores"]) / np.maximum(np.abs(o["scores"]), 1.0)).max()),
                path_err_over_scale=float((np.abs(res["best_path"] - o["best_path"]).max(axis=0) / scale).max()),
                top2_gap=float(top2[1] - top2[0]), best_k=res["best_k"], oracle_best_k=int(np.argmax(o["scores"])),
                same_best=bool(res["best_k"] == int(np.argmax(o["scores"]))))


def main(out_path=None):
    eng = Engine(0)
    rows = []
    for name in ("mpc_mountaincar_L2.npz", "mpc_pendulum_L1.npz", "mpc_mountaincar_L3_xavier.npz", "mpc_pendulum_2x500.npz"):
        g = load_golden(name)
        w, b, norm = golden_model(g)
        eng.set_model(w, b, norm)
        eng.set_plan(g["out_desired_states"], g["out_distances_left"], g["out_radii"])
        res = eng.plan(g["in_start_state"], int(g["in_wp_index"]), actions=g["in_actions"], gamma=float(g["in_gamma"]),
                       horizontal_penalty_factor=float(g["in_hpf"]), precision="fp64", want_scores=True)
        states = eng.get_states()
        o = dict(states=g["out_states"], scores=g["out_scores"], best_path=g["out_best_path"])
        rows.append(report("golden " + name, res, states, o))
        print(json.dumps(rows[-1]), flush=True)
    for name, wl, K, H in (("config 3", bench.make_workload_mountaincar(2, 500), 4096, 20),
                           ("config 4 shard", bench.make_workload(), 16384, 50)):
        eng.set_model(wl["w"], wl["b"], wl["norm"])
        p = wl["plan"]
        eng.set_plan(p["desired_states"], p["distances_left"], p["radii"])
        res = eng.plan(wl["state"], 0, K=K, H=H, seed=11, act_low=wl["low"], act_high=wl["high"], precision="fp64",
                       want_scores=True)
        states = eng.get_states()
        acts = philox.sample_actions(K, H, wl["da"], 11, wl["low"], wl["high"])
        o = mpc_oracle.plan(wl["state"], acts, wl["w"], wl["b"], wl["norm"], p["desired_states"], p["distances_left"],
                            p["radii"], 0, .75, .5)
        rows.append(report(name, res, states, o))
        print(json.dumps(rows[-1]), flush=True)
    eng.close()
    if out_path:
        with open(out_path, "w") as f:
            json.dump(rows, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
