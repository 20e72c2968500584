"""Development helper: SM clock and board power while the config-4 shard (bench.make_workload: Pendulum, 2 x 500,
K = 131 072, H = 50, reference penalty, device-sampled actions) rolls back to back for about 2 s on
mpc_rollout_tc_kernel.  nvidia-smi --query-gpu is polled (read only) every 50 ms from a second thread.

  python scripts/dev/tc_power.py [label] [seconds]

Prints one JSON line: label, the schedule that ran (two-tile / one-tile), decisions, ms per decision, the
median / max of clocks.sm and power.draw over the window and how often each clock-limit reason mask was active
(0x4 = software power cap, 0x20 / 0x40 = software / hardware thermal slowdown), with the card's name and power
limit."""
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import bench  # noqa: E402
from smartstartcontinuous_b200.engine import Engine  # noqa: E402


def query_cmd():
    """clocks.sm, power.draw and the active clock-limit reasons (bit mask; the field was renamed across drivers)."""
    for reasons in ("clocks_event_reasons.active", "clocks_throttle_reasons.active"):
        cmd = ["nvidia-smi", "--query-gpu=clocks.sm,power.draw," + reasons, "--format=csv,noheader,nounits", "-i", "0"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode == 0 and len(r.stdout.strip().split(",")) == 3:
            return cmd
    return ["nvidia-smi", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader,nounits", "-i", "0"]


def main():
    label = sys.argv[1] if len(sys.argv) > 1 else "tree"
    seconds = float(sys.argv[2]) if len(sys.argv) > 2 else 2.0
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                           "-i", "0"], capture_output=True, text=True).stdout.strip()
    wl = bench.make_workload()
    eng = Engine(0)
    eng.set_model(wl["w"], wl["b"], wl["norm"])
    eng.set_plan(wl["plan"]["desired_states"], wl["plan"]["distances_left"], wl["plan"]["radii"])
    kw = dict(K=bench.K_PER_GPU, H=bench.HORIZON, seed=1, act_low=wl["low"], act_high=wl["high"],
              penalty_mode="reference", precision="bf16_tc")
    for _ in range(3):
        eng.plan(wl["state"], 0, **kw)
    schedule = getattr(eng, "last_tc_schedule", lambda: None)()
    query = query_cmd()
    samples, reasons, stop = [], {}, threading.Event()

    def poll():
        while not stop.is_set():
            out = subprocess.run(query, capture_output=True, text=True).stdout.strip().split(",")
            try:
                samples.append((float(out[0]), float(out[1])))
                if len(out) > 2:
                    reasons[out[2].strip()] = reasons.get(out[2].strip(), 0) + 1
            except (ValueError, IndexError):
                pass
            time.sleep(0.05)

    th = threading.Thread(target=poll)
    th.start()
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        eng.plan(wl["state"], 0, **kw)
        n += 1
    dt = time.perf_counter() - t0
    stop.set()
    th.join()
    clk = np.array([s[0] for s in samples]) if samples else np.zeros(1)
    pw = np.array([s[1] for s in samples]) if samples else np.zeros(1)
    print(json.dumps(dict(label=label, card=card, schedule=schedule, decisions=n, ms_per_decision=1e3 * dt / n,
                          samples=len(samples), sm_clock_mhz_median=float(np.median(clk)),
                          sm_clock_mhz_min=float(clk.min()), power_w_median=float(np.median(pw)),
                          power_w_max=float(pw.max()), clock_limit_reasons=reasons)))


if __name__ == "__main__":
    main()
