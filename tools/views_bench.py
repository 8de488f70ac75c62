"""Time captures of more than 256 views at C4 geometry (1024^3 grid, 1920x1080 images, synth.cameras / silhouettes with V views).

  python tools/views_bench.py [--views 72,256,257,512,1024] [--reps 5] [--out profiles/views_bench_C4_1gpu.json]

For every V: the engine gets the first min(V, 256) views with vc_set_views and the rest with vc_append_views in chunks of 72
views.  Recorded:
  carve_ms       a fresh VC_EXACT carve of all views (vc_reset + vc_carve): host clock around the call and a stream
                 synchronisation, a 256 MiB buffer written before every pass so that the 126 MB L2 holds nothing of the previous one
  carve_event_ms the same carve as the engine's CUDA events time it (vc_stats.last_carve_ms)
  color_avg_ms   vc_color(VC_COLOR_AVG) on the carved volumes, host clock around the call and a stream synchronisation
  first_append_ms, first_append_views
                 host clock around the first vc_append_views (it ends in a stream synchronisation) and the views it added: 72,
                 or fewer when V - 256 is smaller; append_ms_all / append_views_all: every chunk
  plain_carve_ms, plain_carve_event_ms (V <= 256 only)
                 the same carve as plain launches (VOXCARVE_NO_GRAPH=1) instead of the one cached CUDA graph that a capture of at
                 most 256 views uses: what one graph saves per group of 256 views.  A capture of more views carves group by group
                 with plain launches
  volumes_sha256 of the occupied + seen words after the carve, and the same hash from a second engine that starts with 8 views
                 and appends 8 at a time, carving only the new views onto the volumes on the device; the two must agree
The colour images are 72 synthetic images, view v using image v % 72.  The card's name and power limit are read by the same
process (nvidia-smi).

  --bench-parent DIR [--bench-configs C4,C5] [--bench-rounds 2]

then runs `bench.py --gpus 1 --steps 5 --warmup 2 --config C --no-cpu-baseline` of this tree and of the tree in DIR (an older
version, e.g. the parent commit's, built in place), alternated, and stores their result lines: the path of at most 256 views
is the one bench.py measures."""
import argparse
import hashlib
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
    ap.add_argument("--views", default="72,256,257,512,1024")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--bench-parent", default=None)
    ap.add_argument("--bench-configs", default="C4,C5")
    ap.add_argument("--bench-rounds", type=int, default=2)
    a = ap.parse_args()
    import torch
    import ar_voxel_project_b200 as A
    from ar_voxel_project_b200.synth import CONFIGS, cameras, images, scene, silhouettes
    if not torch.cuda.is_available():
        sys.exit("views_bench needs a CUDA device")
    cfg = CONFIGS["C4"]
    N, W, H = cfg["N"], cfg["W"], cfg["H"]
    s = np.float32(0.28) / np.float32(N)
    base_images = images(72, W, H, 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out = {"gpu": gpu_info(), "config": dict(N=N, W=W, H=H, voxel_size=float(s)), "l2": "256 MiB written between timed carves",
           "reps": a.reps, "results": []}

    def build(V, P, M, bits, first, chunk, with_images, carve_new=False):
        e = A.VoxelEngine(N, N, N, s)
        k = min(first, V)
        e.set_views(P[:k], W, H, M[:k])
        e.set_masks_bits(bits[:k])
        if with_images:
            e.set_images(np.ascontiguousarray(base_images[np.arange(k) % 72]))
        if carve_new:
            e.reset()
            e.carve()
        append_ms, append_views = [], []
        for v in range(k, V, chunk):
            n = min(chunk, V - v)
            append_views.append(n)
            img = np.ascontiguousarray(base_images[np.arange(v, v + n) % 72]) if with_images else None
            t0 = time.perf_counter()
            e.append_views(P[v:v + n], M[v:v + n], mask_bits=bits[v:v + n], images_bgr=img)
            append_ms.append((time.perf_counter() - t0) * 1e3)
            if carve_new:
                e.carve(0, v, -1)
        return e, append_ms, append_views

    def volumes_hash(e):
        e.synchronize()
        h = hashlib.sha256()
        h.update(e.download_occupied().tobytes())
        h.update(e.download_seen().tobytes())
        return h.hexdigest()

    def timed(e, fn, reps, flush_l2):
        """host clock around fn() and the engine's stream synchronisation, after the GPU is idle"""
        times = []
        for _ in range(reps):
            if flush_l2:
                flush.fill_(1)
            torch.cuda.synchronize()
            e.synchronize()
            t0 = time.perf_counter()
            fn()
            e.synchronize()
            times.append((time.perf_counter() - t0) * 1e3)
        return times

    for V in [int(x) for x in a.views.split(",")]:
        t0 = time.perf_counter()
        K32, M, P = cameras(V, W, H)
        bits = silhouettes(M, K32, W, H, scene(0))
        gen_s = time.perf_counter() - t0
        e, append_ms, append_views = build(V, P, M, bits, 256, 72, True)

        def carve():
            e.reset()
            e.carve()
        carve()
        color = lambda: e.color(2)  # noqa: E731
        carve_ms = timed(e, carve, a.reps, True)
        carve()
        e.color(2)
        color_ms = timed(e, color, a.reps, False)
        carve()
        ev_ms = []  # the engine's own CUDA-event time of the last carve (vc_stats.last_carve_ms)
        for _ in range(a.reps):
            flush.fill_(1)
            torch.cuda.synchronize()
            carve()
            ev_ms.append(e.stats()["last_carve_ms"])
        h_set = volumes_hash(e)
        e.close()
        e2, _, _ = build(V, P, M, bits, 8, 8, False, carve_new=True)
        h_stream = volumes_hash(e2)
        e2.close()
        plain = {}
        if V <= 256:  # the engine reads the switch at its first carve
            os.environ["VOXCARVE_NO_GRAPH"] = "1"
            e3, _, _ = build(V, P, M, bits, 256, 72, False)
            del os.environ["VOXCARVE_NO_GRAPH"]

            def carve3():
                e3.reset()
                e3.carve()
            carve3()
            plain["plain_carve_ms"] = timed(e3, carve3, a.reps, True)
            plain["plain_carve_event_ms"] = []
            for _ in range(a.reps):
                flush.fill_(1)
                torch.cuda.synchronize()
                carve3()
                plain["plain_carve_event_ms"].append(e3.stats()["last_carve_ms"])
            plain["plain_carve_ms_median"] = float(np.median(plain["plain_carve_ms"]))
            plain["plain_carve_event_ms_median"] = float(np.median(plain["plain_carve_event_ms"]))
            plain["plain_sha256_equal"] = volumes_hash(e3) == h_set
            e3.close()
        r = dict(V=V, carve_ms_median=float(np.median(carve_ms)), carve_ms=carve_ms, carve_event_ms_median=float(np.median(ev_ms)),
                 carve_event_ms=ev_ms, color_avg_ms_median=float(np.median(color_ms)), color_avg_ms=color_ms,
                 first_append_ms=append_ms[0] if append_ms else None, first_append_views=append_views[0] if append_views else None,
                 append_ms_all=append_ms, append_views_all=append_views, volumes_sha256=h_set, volumes_sha256_streamed=h_stream,
                 hashes_equal=h_set == h_stream, input_generation_s=gen_s, **plain)
        print(json.dumps({k: v for k, v in r.items() if not isinstance(v, list)}), flush=True)
        out["results"].append(r)
    if a.bench_parent:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        subprocess.check_call([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=a.bench_parent, stdout=subprocess.DEVNULL)
        out["bench_py"] = []
        for cfg in a.bench_configs.split(","):
            for rnd in range(a.bench_rounds):
                for name, tree in (("this", root), ("parent", a.bench_parent)):
                    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "5", "--warmup", "2", "--config", cfg,
                                        "--no-cpu-baseline"], cwd=tree, capture_output=True, text=True)
                    line = json.loads(r.stdout.strip().splitlines()[-1])
                    row = dict(config=cfg, round=rnd, tree=name, ms_per_step=line.get("ms_per_step"),
                               cold_ms_per_step=line.get("cold_ms_per_step"), result=line)
                    print(json.dumps({k: v for k, v in row.items() if k != "result"}), flush=True)
                    out["bench_py"].append(row)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    if not all(r["hashes_equal"] and r.get("plain_sha256_equal", True) for r in out["results"]):
        sys.exit("volumes of set_views + appends and of the streamed engine differ")


if __name__ == "__main__":
    main()
