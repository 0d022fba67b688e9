"""Developer diagnostic: config #5 (65 536 closed-loop scenarios, N = 50) tick by tick: solve and read-back time, iterations, QP size."""
import os, sys, time, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "bilevel-gait-gen_b200"))
import common
from common import wl
c = wl.CONFIGS["a1_config_distr_rejection"]
B = 65536
st, t0, ee = wl.disturbance_sweep_inputs(c, B, seed=7)
m = common.make_gpu("a1_config_distr_rejection", B, st)
z = torch.zeros((B, 12 * 51 + 160), dtype=torch.float64).pin_memory().numpy()
m.upload(st, t0, ee); m.solve_resident(); m.download(z_out=z)
for tick in range(int(__import__('os').environ.get('TICKS', 40))):
    t = time.perf_counter(); m.advance_plant(c["integrator_dt"]); m.solve_resident(); m.synchronize(); t1 = time.perf_counter()
    r = m.download(z_out=z); t2 = time.perf_counter()
    print(tick, "solve ms", round(1e3 * (t1 - t), 1), "download ms", round(1e3 * (t2 - t1), 1), "iters mean", r["iters"].mean(), "solved", (r["status"] == 0).mean(), "nu", m.sizes(0)["nu"], "samples", m.sizes(0)["n_samples"])
