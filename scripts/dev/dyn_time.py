"""Development helper: device time per Adam step of the trainer (row f1)."""
import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import bench
from oracle import dyn_train_oracle as dto
from smartstartcontinuous_b200.engine import Engine
eng = Engine(0)
tw = bench.dyn_train_workload()
eng.set_model(tw["w"], tw["b"], tw["norm"])
eng.dyn_set_data(0, tw["X_old"], tw["Z_old"]); eng.dyn_set_data(1, tw["X_new"], tw["Z_new"])
np.random.seed(0)
io, inw = dto.epoch_batches(len(tw["X_old"]), len(tw["X_new"]), tw["batch"], tw["frac"])
eng.dyn_train_batches(io, inw, tw["lr"], want_losses=False)
for _ in range(3):
    t0 = time.perf_counter()
    l = eng.dyn_train_batches(io, inw, tw["lr"])
    dt = time.perf_counter() - t0
    print("epoch of %d steps: %.2f ms wall = %.1f us/step; device %s; loss %.5f -> %.5f" % (len(io), 1e3 * dt, 1e6 * dt / len(io), eng.last_timings(), l[0], l[-1]))
