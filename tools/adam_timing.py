#!/usr/bin/env python
"""GPU box: cost of the sampling-fraction replay (adam_seq_kernel, the "adam" kernel class of PPG_KERNEL_TIMING) on SPACESHIP, same seed and a
sample budget (so every run does the same work), median over runs.  usage: adam_timing.py [W H spp runs]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "practical-path-guiding_b200")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
from common import load_fixture_scene
from ppg_b200.integrator import GuidedPathTracer
W, H, spp, runs = (int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], int(sys.argv[4])) if len(sys.argv) > 4 else (640, 360, "60", 5)
os.environ["PPG_KERNEL_TIMING"] = "1"
sc = load_fixture_scene("spaceship-improved").with_film(W, H)
adam, other, total = [], [], []
for r in range(runs):
    g = GuidedPathTracer(dict(sc.integrator, budgetType="spp", budget=spp, seed="1234")); g.set_scene(sc)
    ptr, st = g.render_device()
    adam.append(st["kernel_ms"]["adam"]); other.append(st["kernel_ms"]["other"]); total.append(st["render_device_ms"])
    print(f"run {r}: adam {adam[-1]:.2f} ms  other {other[-1]:.2f} ms  render {total[-1]:.1f} ms  vertices {st['total_vertices']}", flush=True)
    del g
print(f"median adam {np.median(adam):.2f} ms  other {np.median(other):.2f} ms  render {np.median(total):.1f} ms  ({W}x{H}, {spp} spp, {runs} runs)")
