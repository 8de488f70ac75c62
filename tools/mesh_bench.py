"""Time the mesh of main.cpp:291-303 on the synthetic configs: colour (average) -> vc_mesh_from_volumes(1, 1, 3, 0.5), from the
bit volumes, with and without the download of the triangles; at C4 also the dense chain (vc_dense_from_volumes + vc_dense_closure(3)
+ vc_mc_mesh), alternated with it in the same process.  (At C5 the dense Model needs 256 GiB and cannot run on one GPU.)

  python tools/mesh_bench.py [--configs C4,C5] [--reps 5] [--out profiles/mesh_bench_C4_C5_1gpu.json]

Times are host clocks around work that ends in a device synchronisation, median of --reps after one warm-up of every chain.
The peak device memory is the largest used amount (cudaMemGetInfo) seen right after each chain, which includes the CUDA context."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else ""
    return dict(zip(q.split(","), [x.strip() for x in line.split(",")])) if line else {"nvidia-smi": "unavailable"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C4,C5")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import ar_voxel_project_b200 as A
    from ar_voxel_project_b200.synth import CONFIGS, Workload
    if not torch.cuda.is_available():
        sys.exit("mesh_bench needs a CUDA device")
    peak = [0]

    def used():
        free, total = torch.cuda.mem_get_info()
        peak[0] = max(peak[0], total - free)

    def timed(fn):
        t0 = time.perf_counter()
        out = fn()
        used()
        return (time.perf_counter() - t0) * 1e3, out

    result = {"gpu": gpu_info(), "torch": torch.__version__, "configs": {}}
    for name in a.configs.split(","):
        w = Workload(**CONFIGS[name])
        peak[0] = 0
        with A.VoxelEngine(w.X, w.Y, w.Z, w.s) as e:
            e.set_views(w.P, w.W, w.H, w.M)
            e.set_masks_bits(w.mask_bits)
            e.set_images(w.images_bgr())
            e.carve()
            e.synchronize()

            def sparse(download):
                def run():
                    e.color(2)
                    r = e.mesh_from_volumes(True, True, 3, 0.5, download=download)
                    e.synchronize()
                    return r
                return run

            def dense():
                e.color(2)
                e.dense_from_volumes(True, True)
                e.dense_closure(3)
                n = e.mc_mesh(0.5)
                e.synchronize()
                return n

            chains = {"sparse_ms": sparse(False), "sparse_with_download_ms": sparse(True)}
            if name == "C4":
                chains["dense_with_download_ms"] = dense
            times = {k: [] for k in chains}
            outs = {}
            peak_sparse = None
            for k, fn in chains.items():  # warm-up; the dense chain's 2 x 16 B per voxel stay allocated once it has run
                if k.startswith("dense"):
                    peak_sparse = peak[0]
                outs[k] = fn()
                used()
            for _ in range(a.reps):
                for k, fn in chains.items():  # alternated
                    t, outs[k] = timed(fn)
                    times[k].append(t)
            n_tris = outs["sparse_ms"]
            entry = {"workload": w.name, "triangles": n_tris, "surface_records": e.surface_count(), "reps": a.reps,
                     "peak_device_bytes_used": peak[0], "peak_device_bytes_used_sparse_only": peak_sparse or peak[0]}
            for k, v in times.items():
                entry[k] = float(np.median(v))
                entry[k.replace("_ms", "_all_ms")] = [round(x, 3) for x in v]
            if "dense_with_download_ms" in outs:
                dv, dc = outs["dense_with_download_ms"]
                sv, sc = outs["sparse_with_download_ms"]
                entry["dense_equals_sparse"] = bool(np.array_equal(dv.view(np.uint32), sv.view(np.uint32)) and np.array_equal(dc, sc))
        result["configs"][name] = entry
        print(json.dumps({name: entry}), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
