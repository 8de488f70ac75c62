#!/usr/bin/env python3
"""Minimal driver for ncu: set up one synthetic config, run reset+carve a few times (no torch)."""
import argparse
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import ar_voxel_project_b200 as A
from ar_voxel_project_b200.synth import Workload, CONFIGS

ap = argparse.ArgumentParser()
ap.add_argument("--config", default="C4")
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--mode", type=int, default=0)
ap.add_argument("--slab", default=None, help="z0,z1: carve only this z-slab (what one rank of an N-GPU run does)")
ap.add_argument("--lib", default=None, help="experiment variant of libvoxcarve.so (see build.build(out=...))")
a = ap.parse_args()
if a.lib:
    import ar_voxel_project_b200._lib as L
    L.LIB_PATH = os.path.abspath(a.lib)
w = Workload(**CONFIGS[a.config])
z0, z1 = [int(x) for x in a.slab.split(",")] if a.slab else (0, w.Z)
with A.VoxelEngine(w.X, w.Y, w.Z, w.s, z_begin=z0, z_end=z1) as e:
    e.set_views(w.P, w.W, w.H, w.M)
    e.set_masks_bits(w.mask_bits)
    e.set_profiling(True)   # plain launches: ncu sees every kernel, stats() splits classification from the per-voxel kernel
    for _ in range(a.reps):
        e.reset()
        e.carve(a.mode)
        e.synchronize()
        st = e.stats()
        print("carve ms", st["last_carve_ms"], "of which classify+fill", st["last_classify_ms"])
    e.reset()
    e.carve(a.mode, count_executed=True)
    st = e.stats()
    print("executed", st["executed_voxel_views"], "of which brick corners", st["brick_corner_views"], "nominal", st["nominal_voxel_views"], "occupied", e.count_occupied())
    print("filter rows", st["filter_rows"], "slow rows", st["filter_slow_rows"], "mismatches", st["filter_mismatches"])
