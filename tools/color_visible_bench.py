"""Cost of occlusion-aware colouring (vc_color_visible) against the reference colouring (vc_color) on the synthetic C4 / C5
captures, and the share of observations it keeps.

  python tools/color_visible_bench.py [--configs C4 C5] [--reps 10] [--out color_visible.json]

Per config, after one carve: vc_color(2) and vc_color_visible(2, 2.0) alternately, each timed with CUDA events on the engine's
stream (both calls end in their own stream synchronise: the surface count is read back).  The split by stage comes from a
separate torch.profiler run (kernel durations by name): surface records (count pass, scan, emit pass), splat, observe, colour.
Bytes are those of the observation bits and the depth-buffer chunk.  Kept fractions: observations of vc_color_visible(mode 2,
tolerance) over those of vc_color, for tolerance 0, 1, 2, 4, inf, on each config and on human_dataset at 100^3.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TOLERANCES = (0.0, 1.0, 2.0, 4.0, float("inf"))
BUDGET = 256 << 20  # VC_VIS_ZBUF_BUDGET in voxcarve.cu


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def kept(e, tolerances, mode=2):
    e.color(mode)
    ref = int(e.download_colors()[1][:, 3].astype(np.int64).sum())
    out = {}
    for t in tolerances:
        e.color_visible(mode, t)
        out[str(t)] = int(e.download_colors()[1][:, 3].astype(np.int64).sum()) / max(ref, 1)
    return ref, out


def stage_split(e, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    names = {"vc_surface_pass_kernel": "records", "vc_scan_sums_kernel": "records", "vc_vis_splat_kernel": "splat",
             "vc_vis_observe_kernel": "observe", "vc_surface_color_kernel": "colour", "Memset": "zbuf memset"}
    res = {}
    for label, call in (("vc_color", lambda: e.color(2)), ("vc_color_visible", lambda: e.color_visible(2, 2.0))):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                call()
            torch.cuda.synchronize()
        split = {}
        for ev in prof.key_averages():
            for k, v in names.items():
                if k in ev.key:
                    split[v] = split.get(v, 0.0) + ev.device_time_total / 1e3 / reps  # us -> ms per call
        res[label] = {k: round(v, 4) for k, v in split.items()}
    return res


def run_config(A, name, reps):
    import torch
    from ar_voxel_project_b200.synth import CONFIGS, Workload
    w = Workload(**CONFIGS[name])
    N = CONFIGS[name]["N"]
    img = w.images_bgr()
    out = {"config": name, "grid": N, "views": w.P.shape[0], "image": [w.W, w.H]}
    with A.VoxelEngine(N, N, N, w.s) as e:
        stream = torch.cuda.Stream()
        e.set_stream(stream.cuda_stream)
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(img)
        e.carve()
        e.color(2)
        n = e.surface_count()
        V = w.P.shape[0]
        chunk = max(1, min(V, BUDGET // (w.W * w.H * 4)))
        out["surface_voxels"] = n
        out["observation_bit_bytes"] = ((n + 31) // 32) * 4 * V
        out["depth_buffer_bytes"] = chunk * w.W * w.H * 4
        out["views_per_chunk"] = chunk
        for _ in range(2):  # warm-up of both paths
            e.color(2)
            e.color_visible(2, 2.0)
        t = {"vc_color": [], "vc_color_visible": []}
        for _ in range(reps):
            for label, call in (("vc_color", lambda: e.color(2)), ("vc_color_visible", lambda: e.color_visible(2, 2.0))):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                call()
                b.record(stream)
                b.synchronize()
                t[label].append(a.elapsed_time(b))
        out["ms"] = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "n": len(v)} for k, v in t.items()}
        out["stage_ms_per_call"] = stage_split(e, max(3, reps // 2))
        out["observations_vc_color"], out["kept_fraction"] = kept(e, TOLERANCES)
    return out


def run_human(A):
    vs = A.ViewSet.from_npz(os.path.join(ROOT, "tests", "golden", "human_views.npz"))
    s = np.float32(0.28) / np.float32(100)
    with A.VoxelEngine(100, 100, 100, s) as e:
        e.set_views(vs.P, vs.W, vs.H, vs.M)
        e.set_masks_bits(vs.mask_bits)
        e.set_images(vs.images_bgr)
        e.carve()
        ref, fr = kept(e, TOLERANCES)
        return {"config": "human_dataset 100^3", "views": len(vs.P), "surface_voxels": e.surface_count(),
                "observations_vc_color": ref, "kept_fraction": fr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["C4", "C5"])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import ar_voxel_project_b200 as A
    res = {"card": card(), "tolerance_of_the_times": 2.0, "mode": 2, "runs": [run_config(A, c, a.reps) for c in a.configs] + [run_human(A)]}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
