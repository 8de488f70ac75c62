"""Time the mesh of main.cpp:291-303 on the synthetic configs: colour (average) -> vc_mesh_from_volumes(1, 1, 3, 0.5), from the
bit volumes, with and without the download of the triangles; at C4 also the dense chain (vc_dense_from_volumes + vc_dense_closure(3)
+ vc_mc_mesh), alternated with it in the same process.  (At C5 the dense Model needs 256 GiB and cannot run on one GPU.)

  python tools/mesh_bench.py [--configs C4,C5] [--reps 5] [--out profiles/mesh_bench_C4_C5_1gpu.json]

Times are host clocks around work that ends in a device synchronisation, median of --reps after one warm-up of every chain.
The peak device memory is the largest used amount (cudaMemGetInfo) seen right after each chain, which includes the CUDA context.

  python tools/mesh_bench.py --off --baseline-include DIR [--configs C4,C5] [--reps 5] [--cpp-reps 2] [--out ...]

The .off writer of that mesh: vc_mesh_format_off (format_ms), the download of the whole text in 64 MiB chunks into one pageable
buffer (download_ms), the file write of that text (write_ms) and VoxelEngine.write_mesh_off, download and write interleaved
(write_mesh_off_ms).  Then the whole of vc::carveToMesh (tools/carve_to_mesh_bench.cpp) built against include/ and against the
voxcarve_host.hpp in DIR (an older version, e.g. the parent commit's), the two programs alternated --cpp-reps times, with the
SHA-256 of every file they write.  Files go to a temporary directory and are deleted after hashing."""
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


def sha256(path):
    import hashlib
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for b in iter(lambda: f.read(64 << 20), b""):
            h.update(b)
    return h.hexdigest()


def off_main(a):
    import shutil
    import tempfile
    import torch
    import ar_voxel_project_b200 as A
    from ar_voxel_project_b200 import build
    from ar_voxel_project_b200.synth import CONFIGS, Workload
    if not torch.cuda.is_available():
        sys.exit("mesh_bench needs a CUDA device")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tmp = tempfile.mkdtemp()
    libdir = os.path.dirname(build.build())
    exes = {}
    for name, inc in (("new", os.path.join(root, "include")), ("baseline", a.baseline_include)):
        exes[name] = os.path.join(tmp, "carve_to_mesh_" + name)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-pthread", "-I", inc, os.path.join(root, "tools", "carve_to_mesh_bench.cpp"),
                               "-o", exes[name], "-L", libdir, "-lvoxcarve", f"-Wl,-rpath,{libdir}"])
    result = {"gpu": gpu_info(), "torch": torch.__version__, "host_cpus": os.cpu_count(), "configs": {}}
    try:
        for name in a.configs.split(","):
            w = Workload(**CONFIGS[name])
            case = os.path.join(tmp, "case.bin")
            with open(case, "wb") as f:
                np.array([w.X, w.Y, w.Z, w.V, w.W, w.H], np.int32).tofile(f)
                np.array([w.s], np.float32).tofile(f)
                w.P.astype(np.float32).tofile(f)
                w.M.astype(np.float32).tofile(f)
                w.mask_bits.astype(np.uint32).tofile(f)
                w.images_bgr().astype(np.uint8).tofile(f)
            sc, t = float(np.float32(1.5) * w.s), (0.5, -0.25, 2.0)
            times = {k: [] for k in ("format_ms", "download_ms", "write_ms", "write_mesh_off_ms")}
            path = os.path.join(tmp, "py.off")
            with A.VoxelEngine(w.X, w.Y, w.Z, w.s) as e:
                e.set_views(w.P, w.W, w.H, w.M)
                e.set_masks_bits(w.mask_bits)
                e.set_images(w.images_bgr())
                e.carve()
                e.color(2)
                n_tris = e.mesh_from_volumes(True, True, 3, 0.5, download=False)
                n = e.format_off(sc, t)  # warm-up (allocates the text buffer)
                buf = np.empty(n, np.uint8)
                chunk = 64 << 20
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    n = e.format_off(sc, t)
                    t1 = time.perf_counter()
                    for o in range(0, n, chunk):
                        k = min(chunk, n - o)
                        e._check(e._lib.vc_download_mesh_off(e._h, o, buf[o:o + k].ctypes.data, k))
                    t2 = time.perf_counter()
                    with open(path, "wb") as f:
                        f.write(memoryview(buf)[:n])
                    t3 = time.perf_counter()
                    e.write_mesh_off(path, sc, t)
                    t4 = time.perf_counter()
                    for k, v in zip(times, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                        times[k].append(v * 1e3)
            py_hash = sha256(path)
            os.remove(path)
            entry = {"workload": w.name, "triangles": n_tris, "text_bytes": n, "reps": a.reps}
            for k, v in times.items():
                entry[k] = float(np.median(v))
                entry[k.replace("_ms", "_all_ms")] = [round(x, 3) for x in v]
            cpp = {k: [] for k in exes}
            hashes = {k: set() for k in exes}
            for r in range(a.cpp_reps):
                for k in (("baseline", "new") if r % 2 == 0 else ("new", "baseline")):  # alternated
                    out = os.path.join(tmp, k + ".off")
                    p = subprocess.run([exes[k], case, out], capture_output=True, text=True)
                    if p.returncode != 0:
                        sys.exit(f"{k} carveToMesh failed: {p.stderr[-2000:]}")
                    cpp[k].append(float(p.stdout.strip().splitlines()[-1]))
                    hashes[k].add(sha256(out))
                    os.remove(out)
            for k in exes:
                entry[f"carve_to_mesh_{k}_ms"] = float(np.median(cpp[k]))
                entry[f"carve_to_mesh_{k}_all_ms"] = [round(x, 1) for x in cpp[k]]
                entry[f"carve_to_mesh_{k}_sha256"] = sorted(hashes[k])
            entry["same_file"] = len(hashes["new"]) == 1 and hashes["new"] == hashes["baseline"] == {py_hash}
            result["configs"][name] = entry
            print(json.dumps({name: entry}), flush=True)
            os.remove(case)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C4,C5")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--off", action="store_true", help="time the .off writer and carveToMesh against --baseline-include")
    ap.add_argument("--baseline-include", default=None)
    ap.add_argument("--cpp-reps", type=int, default=2)
    a = ap.parse_args()
    if a.off:
        if not a.baseline_include:
            sys.exit("--off needs --baseline-include DIR (a voxcarve_host.hpp to compare with)")
        return off_main(a)
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
