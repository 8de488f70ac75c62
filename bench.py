#!/usr/bin/env python3
"""bench.py — voxel-view projections/s of the carve hot path on N B200s (z-slab sharded), next to the
reference's CPU carve (the oracle restatement) timed on the same box.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C4|C3|C5|C4-noisy|C1|C2|ref6] [--impl ours|reference]
                  [--dump-outputs DIR]

Step = one full carve (Model ctor state -> occupied + seen volumes complete) of the synthetic workload
BASELINE.json quotes the metric on (default C4: 1024^3 x 72 views, 1920x1080 silhouettes; SURVEY §8d).
`value`  = X*Y*Z*V (nominal voxel-view projections of the job) / device time, masks + their summed-area tables resident in HBM.
`value_cold` = the same with the summed-area tables built inside the timed region (bit masks resident, vc_set_masks + carve).
`value_with_consumer` = carve + (N > 1: one-plane halo exchange over NCCL) + cube-index classification of the slab, per step.
`e2e`    = same metric through the C ABI with HOST buffers: per step H2D of P/M + the masks from pinned memory, summed-area
           tables, reset, carve, D2H of the result in sparse form (a flag byte per 32x8x8 brick + the words of the bricks that
           were evaluated per voxel: the complete result, 1/25 of the bytes) into pinned memory; wall clock, max over ranks.
           `e2e_dense` = the same with both bit volumes downloaded as plain words (PCIe-bound).
`roofline` = projections executed by the dominant kernel (vc_carve_bricks: the corner projections of its 8x8x8 sub-brick
           classification + the per-voxel projections left after three levels of classification and the early exits)
           * 23 FLOP / that kernel's time against the measured FFMA peak of this GPU (CUDA-core bound, SURVEY §8d);
           `roofline_hbm` = grid-write bound of the whole carve against the copy bandwidth of MEASURED_PEAKS.json.
`cpu_baseline` / --impl reference = oracle/ (C restatement of VoxelCarving.cpp:60-72) on a bounded z-slab sample.
C4-noisy = C4 with hostile silhouettes (1 % salt-and-pepper + a ragged 2-px grey fringe, through the 8UC3 path): bounds how much
           of the speed depends on clean masks.  C1 / C2 / ref6 = the datasets at the reference's own sizes, every phase of
           main.cpp:350-436 (carve V1 / V2, colouring, closure, marching cubes) timed beside the CPU port and BASELINE.md's table.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

# stdout carries exactly ONE line, the JSON result: library chatter written to file descriptor 1 (NCCL prints its version banner
# there) is sent to stderr instead, and emit() writes the result to the real stdout
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _RESULT_OUT.write(json.dumps(obj) + "\n")
    _RESULT_OUT.flush()


import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "voxel_view_projections_per_s"
UNIT = "voxel-views/s"
F_ALG = 23.0  # FLOP per voxel-view as the reference evaluates it (SURVEY §8d): 12 mul + 9 add + 2 div
SMALL = ("C1", "C2", "ref6")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C4", choices=["C1", "C2", "ref6", "C3", "C4", "C4-noisy", "C5"])
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="target seconds of CPU work per reference step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-color", action="store_true", help="skip the colour-reconstruction timing (uploads V x H x W x 3 image bytes)")
    ap.add_argument("--uniform-slabs", action="store_true", help="equal-height z-slabs instead of the planner's balanced ones")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.config in SMALL):
        ap.error("--dump-outputs needs --impl ours and a synthetic config (C3, C4, C4-noisy, C5)")
    return a


def config_dict(w, n_gpus, name):
    """identical in both arms (ours / reference) for the same command line"""
    return {"workload": w.name, "config": name, "grid": [w.X, w.Y, w.Z], "views": w.V, "image": [w.W, w.H],
            "voxel_size": float(w.s), "partition": f"z-slabs x{n_gpus}", "arithmetic": "exact (bit-identical to reference)"}


def make_workload(name):
    from ar_voxel_project_b200.synth import Workload, CONFIGS, noisy_masks
    if name == "C4-noisy":
        w = Workload(**CONFIGS["C4"])
        w.noisy_bgr, w.mask_bits = noisy_masks(w)   # the 8UC3 masks the engine is given, and their exact bit image for the CPU arm
        w.label = "C4-noisy"
        return w
    return Workload(**CONFIGS[name])


def workload_name(w):
    return w.name + (" + 1% salt-and-pepper + ragged 2-px grey fringe (8UC3)" if getattr(w, "label", "") == "C4-noisy" else "")


def grid_hash(words):
    return hashlib.blake2b(np.ascontiguousarray(words).view(np.uint8), digest_size=8).hexdigest()


DUMP_SAMPLE_WORDS = 1 << 20


def dump_outputs(out_dir, occ, seen):
    """--dump-outputs: the occupied and seen volumes a caller of the timed step receives (uint32 words [Z][Y][ceil(X/32)]), cut to
    a size that can be kept and compared between builds (C4: 32 MiB, C5: 56 MiB):
      word_index.npy          flat word positions of a fixed sample (seed 0; every word when there are at most 2^20)
      <volume>_words.npy      the words at those positions, float64 (exact for uint32)
      <volume>_row_counts.npy set bits of every row [Z][Y], float32 (exact up to 2^24): every voxel counts somewhere"""
    os.makedirs(out_dir, exist_ok=True)
    n = occ.size
    idx = np.arange(n) if n <= DUMP_SAMPLE_WORDS else np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE_WORDS, replace=False))
    np.save(os.path.join(out_dir, "word_index.npy"), idx.astype(np.float64))
    for name, vol in (("occupied", occ), ("seen", seen)):
        np.save(os.path.join(out_dir, f"{name}_words.npy"), vol.reshape(-1)[idx].astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}_row_counts.npy"), np.bitwise_count(vol).sum(axis=-1, dtype=np.uint32).astype(np.float32))


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------- CPU reference
def cpu_reference(w, seconds, steps, warmup):
    """oracle.carve on a contiguous z-slab of the same workload, all host threads. -> (vv/s, cores, sample text, ms/step)"""
    from oracle import oracle as O
    nthr = O.max_threads()
    z_mid = w.Z // 2

    def run(n):
        z0 = max(0, min(w.Z - n, z_mid - n // 2))
        t = time.perf_counter()
        O.carve(w.X, w.Y, w.Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=z0, z1=z0 + n, nthreads=nthr)
        return time.perf_counter() - t, z0

    n = min(w.Z, nthr)
    t1, _ = run(n)  # calibration (also warms the page cache / threads)
    n = int(max(n, min(w.Z, round(n * seconds / max(t1, 1e-3)))))
    n = max(nthr, (n // nthr) * nthr) if n >= nthr else n
    n = min(n, w.Z)
    for _ in range(max(0, warmup - 1)):
        run(n)
    ts = [run(n) for _ in range(steps)]
    t = float(np.mean([a for a, _ in ts]))
    vv = w.X * w.Y * n * w.V
    sample = (f"{n} contiguous z-planes [{ts[0][1]},{ts[0][1] + n}) of {w.Z} ({vv / 1e9:.2f} G of {w.X * w.Y * w.Z * w.V / 1e9:.1f} G voxel-views), "
              f"{nthr} pthreads, gcc -O2 -ffp-contract=off, bit-packed masks; CPU cost per voxel-view is position-independent")
    return vv / t, nthr, sample, t * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if args.config in SMALL:
        return run_small(args, reference_only=True)
    w = make_workload(args.config)
    v, cores, sample, ms = cpu_reference(w, args.cpu_seconds, args.steps, args.warmup)
    cfg = config_dict(w, args.gpus, args.config)
    cfg["workload"] = workload_name(w)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference C++ cannot be built here (needs OpenCV C++ + Eigen); this is oracle/, its pinned C restatement"}
    emit(line)
    return 0


# ------------------------------------------------------- the datasets at the reference's own sizes
PUBLISHED_FIG4 = {  # BASELINE.md §1 / Report.pdf p.5 Fig. 4 (i7 @ 4.5 GHz, 1 thread; carve and colouring INCLUDE ~60 / ~69 ms of pose estimation + undistortion)
    ("small", 1): dict(carve=60.0509, color=69.7923, closure=0.0572, mc=0.1263, overall=137.076),
    ("medium", 1): dict(carve=757.221, color=86.1754, closure=6.4862, mc=2.0385, overall=931.708),
    ("large", 1): dict(carve=5681.31, color=140.681, closure=65.6279, mc=15.0167, overall=6197.77),
    ("small", 2): dict(carve=70.8081, color=69.1268, closure=0.0572, mc=0.0608, overall=147.935),
    ("medium", 2): dict(carve=181.486, color=83.7593, closure=7.4642, mc=2.0345, overall=355.334),
    ("large", 2): dict(carve=895.371, color=133.797, closure=64.0341, mc=15.1265, overall=1399.95),
}


def small_cases(name):
    """(label, dataset, (X, Y, Z), voxel size, carve method) — main.cpp:26-29 defaults and the -c=6 chain main.cpp:350-436"""
    f32 = np.float32
    if name == "C1":
        return [("box_dataset 100^3 V1", "box", (100, 100, 100), f32(0.0028), 1)]
    if name == "C2":
        return [("human_dataset 100^3 V1 + colouring", "human", (100, 100, 100), f32(0.0028), 1)]
    rows = []
    for method in (1, 2):
        for size, dims, s in (("small", (10, 10, 5), 0.028), ("medium", (50, 50, 25), 0.0056), ("large", (100, 100, 50), 0.0028)):
            rows.append((f"{size} V{method}", "box", dims, f32(s), method, size))
    return rows


def run_small(args, reference_only=False):
    """every phase of main.cpp:350-436 on the cached dataset views: GPU engine (through the Python mirror of the C ABI, wall clock
    incl. every host round trip a caller sees, result downloads excluded) beside the oracle on 1 thread and on all threads"""
    from ar_voxel_project_b200.api import ViewSet
    from oracle import oracle as O
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    gpu = not reference_only
    if gpu:
        import torch
        import ar_voxel_project_b200 as A
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    nthr = O.max_threads()
    rows = []
    views = {}

    def wall(fn, reps):
        ts = []
        for _ in range(reps):
            t = time.perf_counter()
            fn()
            ts.append((time.perf_counter() - t) * 1e3)
        return float(np.median(ts))

    first = None
    for case in small_cases(args.config):
        label, ds, (X, Y, Z), s, method = case[:5]
        if ds not in views:
            views[ds] = ViewSet.from_npz(os.path.join(ROOT, "tests", "golden", f"{ds}_views.npz"))
        vs = views[ds]
        nominal = X * Y * Z * vs.V
        row = {"case": label, "grid": [X, Y, Z], "voxel_size": float(s), "views": vs.V, "nominal_voxel_views": nominal}
        # ---- CPU port (oracle): the reference's algorithm without cv::Mat overhead, poses / undistortion cached for both sides
        cpu = {}
        if method == 1:
            cpu["carve_1thread"] = wall(lambda: O.carve(X, Y, Z, s, vs.P, vs.W, vs.H, mask_bits=vs.mask_bits, nthreads=1), 1)
            cpu[f"carve_{nthr}threads"] = wall(lambda: O.carve(X, Y, Z, s, vs.P, vs.W, vs.H, mask_bits=vs.mask_bits, nthreads=nthr), 3)
            ro, rs = O.carve(X, Y, Z, s, vs.P, vs.W, vs.H, mask_bits=vs.mask_bits, nthreads=nthr)
        else:
            cpu["carve_1thread"] = wall(lambda: O.fast_carve(X, Y, Z, s, vs.P, vs.W, vs.H, mask_bits=vs.mask_bits), 1)
            ro, rs = O.fast_carve(X, Y, Z, s, vs.P, vs.W, vs.H, mask_bits=vs.mask_bits)
        cpu["color_avg_1thread"] = wall(lambda: O.color(X, Y, Z, s, vs.P, vs.M, vs.W, vs.H, vs.images_bgr, ro, 2), 1)
        ci, cc = O.color(X, Y, Z, s, vs.P, vs.M, vs.W, vs.H, vs.images_bgr, ro, 2)
        dense = O.dense_model(X, Y, Z, ro, rs, ci, cc)
        cpu["closure_1thread"] = wall(lambda: O.closure(X, Y, Z, dense, 3), 1)
        closed = O.closure(X, Y, Z, dense, 3)
        cpu["mc_1thread"] = wall(lambda: O.marching_cubes(X, Y, Z, closed, 0.5), 1)
        rv, _ = O.marching_cubes(X, Y, Z, closed, 0.5)
        row["cpu_port_ms"] = cpu
        row["triangles"] = int(len(rv))
        row["occupied_voxels"] = int(O.unpack(ro, X).sum())
        if len(case) > 5:
            row["published_reference_ms"] = PUBLISHED_FIG4[(case[5], method)]
        if gpu:
            g = {}
            with A.VoxelEngine(X, Y, Z, s) as e:
                e.set_views(vs.P, vs.W, vs.H, vs.M)
                e.set_masks_bits(vs.mask_bits)
                e.set_images(vs.images_bgr)

                def do_carve():
                    if method == 1:
                        e.reset(), e.carve()
                    else:
                        e.fast_carve()
                    e.synchronize()
                for _ in range(args.warmup):
                    do_carve()
                g["carve"] = wall(do_carve, args.steps)
                g["carve_device_only"] = e.stats()["last_carve_ms"] if method == 1 else None

                def do_color():
                    e.color(2), e.synchronize()
                do_color()
                g["color_avg"] = wall(do_color, args.steps)
                e.dense_from_volumes(apply_colors=True, handle_unseen=True), e.synchronize()
                g["model_on_device"] = wall(lambda: (e.dense_from_volumes(apply_colors=True, handle_unseen=True), e.synchronize()), 5)

                ts = []
                for _ in range(4):   # applied ONCE to a freshly built Model, like main.cpp:297-299 (a second pass would dilate again); first round = warm-up
                    e.dense_from_volumes(apply_colors=True, handle_unseen=True), e.synchronize()
                    t = time.perf_counter()
                    e.dense_closure(3), e.synchronize()
                    ts.append((time.perf_counter() - t) * 1e3)
                g["closure"] = float(np.median(ts[1:]))
                def do_mc():
                    e.mc_mesh(0.5)
                do_mc()
                g["mc_mesh_incl_download"] = wall(do_mc, 5)
                verts, _ = e.mc_mesh(0.5)
                occ, seen = None, None
                # parity of what was timed: the carve against the oracle, the final mesh triangle count
                if method == 1:
                    e.reset(), e.carve()
                else:
                    e.fast_carve()
                occ, seen = e.download_occupied(), e.download_seen()
            row["gpu_ms"] = g
            row["bit_exact_vs_cpu_port"] = bool(np.array_equal(occ, ro) and np.array_equal(seen, rs) and len(verts) == len(rv))
            row["value"] = nominal / (g["carve"] * 1e-3)
        rows.append(row)
        if first is None:
            first = row
    key = rows[-1] if args.config != "ref6" else [r for r in rows if r["case"] == "large V1"][0]
    ms = key["gpu_ms"]["carve"] if gpu else key["cpu_port_ms"]["carve_1thread"]
    cfg = {"workload": f"{args.config}: " + "; ".join(r["case"] for r in rows), "config": args.config, "grid": key["grid"], "views": key["views"],
           "image": [640, 480], "voxel_size": key["voxel_size"], "partition": f"z-slabs x{args.gpus}", "arithmetic": "exact (bit-identical to reference)"}
    line = {"metric": METRIC, "value": key["nominal_voxel_views"] / (ms * 1e-3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "reference datasets (Data/box_dataset, Data/human_dataset) through the cached poses + undistorted masks of tests/golden/*_views.npz (cv2 4.13)",
            "config": cfg, "rows": rows,
            "timing": "wall clock around the public call incl. its host round trips, median; the published column is the literal reference on an "
                      "i7 @ 4.5 GHz incl. ~60 ms (carve) / ~69 ms (colouring) of per-call pose estimation + undistortion that both arms here take cached",
            "cpu_baseline": {"value": key["nominal_voxel_views"] / (key["cpu_port_ms"]["carve_1thread"] * 1e-3), "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": "the whole job of the key row, 1 thread (the reference is single-threaded)"}}
    if reference_only:
        line["impl"] = "reference"
        line["e2e"] = {"value": line["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        line["gpu_launches"] = 0
    else:
        line["gpu_launches"] = 3 * args.steps
    emit(line)
    return 0


# --------------------------------------------------------------------------------- ours
def run_ours(args):
    if args.config in SMALL:
        return run_small(args)
    import torch
    import torch.distributed as dist
    import ar_voxel_project_b200 as A
    from ar_voxel_project_b200.engine import measure_peaks

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs writes the whole grid of a single-process run; each rank here holds only its slab")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # a non-default stream: its handle is what the engine launches on, so torch events bracket our kernels
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def allgather(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world == 1:
            return [float(x)]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def timed(fn, n, flush_l2=True):
        """device time of fn() per call: n calls, each bracketed by events on the launching stream, L2 flushed before each"""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        barrier()
        for a, b in ev:
            if flush_l2:
                flush.fill_(1)
            a.record()
            fn()
            b.record()
        barrier()
        return allmax(float(np.mean([a.elapsed_time(b) for a, b in ev])))

    w = make_workload(args.config)
    noisy = getattr(w, "label", "") == "C4-noisy"
    X, Y, Z, V = w.X, w.Y, w.Z, w.V
    Wx = (X + 31) // 32
    nominal_total = X * Y * Z * V

    # whole-grid device buffers owned by the engine (vc_alloc_full_volumes: compressible memory when the GPU grants it): slabs are
    # carved in place, gathered in place
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    # every rank holds all views; z-slab boundaries come from the engine's planner (super-brick classification of the
    # whole grid, identical on every rank) so that the per-voxel work, not the plane count, is balanced
    eng = A.VoxelEngine(X, Y, Z, w.s, device=local)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.set_views(w.P, w.W, w.H, w.M)
    if noisy:
        eng.set_masks_bgr(w.noisy_bgr)   # the 8UC3 path: packed on the device
        assert np.array_equal(eng.download_masks(), w.mask_bits), "device packing of the noisy 8UC3 masks differs from the CPU arm's bits"
    else:
        eng.set_masks_bits(w.mask_bits)
    bounds = eng.plan_slabs(world) if (world > 1 and not args.uniform_slabs) else [(r * Z) // world for r in range(world)] + [Z]
    # single-GPU result of the same job, hashed: what the gathered grid of an N > 1 run must equal (rank 0, before the slabs)
    ref_hash = None
    if rank == 0:
        eng.alloc_full_volumes()
        eng.reset(), eng.carve(A._lib.VC_EXACT)
        ref_hash = {"occupied": grid_hash(eng.download_occupied()), "seen": grid_hash(eng.download_seen())}
    z0, z1 = bounds[rank], bounds[rank + 1]
    if world > 1:
        eng.set_slab(z0, z1)
        from ar_voxel_project_b200.dist import init_engine_comm
        init_engine_comm(eng)   # NCCL communicator inside libvoxcarve.so; torch only carried its 128-byte id
    eng.alloc_full_volumes()

    def step():
        eng.reset()
        eng.carve(A._lib.VC_EXACT)

    def step_with_consumer():   # what a device-side consumer of the grid costs on top: one-plane halos instead of an all-gather
        eng.reset()
        eng.carve(A._lib.VC_EXACT)
        if world > 1:
            eng.exchange_halos()
        eng.mc_classify()

    clocks = ClockSampler(local)  # spans warm-up, the timed steps and an identical untimed tail (nvidia-smi period: 100 ms)
    t_clk = time.perf_counter()
    for _ in range(args.warmup):
        flush.fill_(1)
        step()
    ms_per_step = timed(step, args.steps)
    dumped = (eng.download_occupied(), eng.download_seen()) if args.dump_outputs else None   # the last timed step's result
    n_tail = 0
    while time.perf_counter() - t_clk < 2.0:  # keep the same load up until the sampler has ~20 samples
        flush.fill_(1)
        step()
        n_tail += 1
    torch.cuda.synchronize()
    clk = clocks.stop()
    clk["sampled_over"] = f"{args.warmup} warm-up + {args.steps} timed + {n_tail} identical untimed steps"
    launches = 4 * args.steps  # vc_blind_fill_kernel (absorbs the reset), vc_brick_classify_kernel<1>, <0>, vc_carve_bricks (its first blocks patch the words the blind fill got wrong), per step

    for _ in range(2):
        step_with_consumer()
    with_consumer_ms = timed(step_with_consumer, args.steps)
    mc_hist = eng.allreduce_u64(eng.download_mc()[0])
    mc_tris = int((mc_hist * np.array(TRI_COUNTS(), np.uint64)).sum())

    # cold start: bit masks resident on the device, their summed-area tables built inside the timed region
    d_bits = torch.from_numpy(w.mask_bits.view(np.int32)).to(dev)

    def step_cold():
        eng.set_masks_bits_device(d_bits.data_ptr())
        eng.reset()
        eng.carve(A._lib.VC_EXACT)
    step_cold()
    cold_ms = timed(step_cold, args.steps)

    # carve-kernel-only time (events inside vc_carve) and executed voxel-views (separate, untimed counting pass)
    kt, ct = [], []
    eng.set_profiling(True)   # plain launches with an event between classification and per-voxel kernel (the timed steps above ran the cached CUDA graph)
    for _ in range(5):
        flush.fill_(1)
        torch.cuda.synchronize()  # plain launches onto an idle GPU; the blind fill runs in front of the classification here (DESIGN.md s.9)
        step()
        st = eng.stats()
        kt.append(st["last_carve_ms"]), ct.append(st["last_classify_ms"])
    eng.set_profiling(False)
    kernel_ms = float(np.mean(kt))
    classify_ms = float(np.mean(ct))
    eng.reset()
    eng.carve(A._lib.VC_EXACT, count_executed=True)
    st = eng.stats()
    volumes_compressible = int(st["volumes_compressible"])
    executed_total = allsum(float(st["executed_voxel_views"]))
    corner_total = allsum(float(st["brick_corner_views"]))
    sub_corner_total = allsum(float(st["subbrick_corner_views"]))
    filter_rows, filter_slow, filter_bad = (allsum(float(st[k])) for k in ("filter_rows", "filter_slow_rows", "filter_mismatches"))
    bricks_listed = allsum(float(st["bricks_listed"]))
    bricks_total = allsum(float(st["bricks_total"]))
    # the same job without brick classification (VC_EXACT_FLAT), for reference
    flat = []
    for _ in range(2):
        flush.fill_(1)
        eng.reset()
        eng.carve(A._lib.VC_EXACT_FLAT)
        flat.append(eng.stats()["last_carve_ms"])
    flat_ms = allmax(float(flat[-1]))
    step()
    n_occ, n_seen = eng.count_occupied()
    occupied_total = allsum(float(n_occ))
    kernel_ms_max = allmax(kernel_ms)
    fine_ms_max = allmax(kernel_ms - classify_ms)
    classify_ms_max = allmax(classify_ms)
    per_rank = {"carve_ms": allgather(kernel_ms), "classify_ms": allgather(classify_ms),
                "per_voxel_projections": allgather(float(st["executed_voxel_views"]) - float(st["brick_corner_views"])),
                "bricks_listed": allgather(float(st["bricks_listed"]))}

    # the cube-index pass alone (N > 1: on the slab, with the halos exchanged above)
    if world > 1:
        eng.exchange_halos()
    eng.mc_classify()
    mc_ms = timed(eng.mc_classify, 3, flush_l2=False)
    halo_ms = None
    if world > 1:   # 20 exchanges inside one pair of events: a single one mostly measures how far apart the ranks arrive
        def halos20():
            for _ in range(20):
                eng.exchange_halos()
        halos20()
        halo_ms = timed(halos20, 2, flush_l2=False) / 20.0

    # per-surface-voxel colouring of the carved grid (ColorReconstruction.cpp:22-70) on the same device-resident volume;
    # the 8UC3 images (V x H x W x 3, hash-coloured) are uploaded outside the timed region
    color_ms = None
    if not args.no_color:
        eng.set_images(w.images_bgr())
        color_ms = {}
        for name, mode in (("average", A._lib.VC_COLOR_AVG), ("closest", A._lib.VC_COLOR_CLOSEST)):
            eng.color(mode)
            torch.cuda.synchronize()
            color_ms[name] = timed(lambda: eng.color(mode), 2, flush_l2=False)
        color_ms["surface_voxels"] = allsum(float(eng.surface_count()))

    # on-demand assembly of the bit-packed grid (NCCL over NVLink, inside the library), timed separately; only a consumer that
    # needs every voxel (the host Model, fastCarve's flood) pays for it
    gather = None
    hashes = dict(ref_hash) if ref_hash else None
    if world > 1:
        step()
        torch.cuda.synchronize()
        eng.gather(bounds, occupied=True, seen=True)   # first use: NCCL sets up its peer connections (seconds at 8 ranks), untimed
        torch.cuda.synchronize()
        g_occ = timed(lambda: eng.gather(bounds, occupied=True, seen=False), 3, flush_l2=False)
        g_both = timed(lambda: eng.gather(bounds, occupied=True, seen=True), 3, flush_l2=False)
        got = {"occupied": grid_hash(eng.download_full(0)), "seen": grid_hash(eng.download_full(1))}
        box = [ref_hash]
        dist.broadcast_object_list(box, src=0)
        same = got == box[0]
        all_same = allsum(1.0 if same else 0.0) == world
        recv = (Z - (z1 - z0)) * Y * Wx * 4
        gather = {"occupied_ms": g_occ, "occupied_and_seen_ms": g_both, "received_bytes_per_rank_per_volume": recv,
                  "occupied_GBps_received_per_rank": recv / (g_occ * 1e-3) / 1e9,
                  "how": "vc_gather inside libvoxcarve.so: in-place ncclAllGather for equal slabs, one group of ncclSend/ncclRecv for balanced (ragged) slabs",
                  "gathered_grid_equals_single_gpu_carve": bool(all_same), "hash_gathered": got, "hash_single_gpu": box[0]}
        hashes = got
        if not all_same:
            raise SystemExit(f"bench.py: rank {rank}: gathered grid {got} differs from the single-GPU carve {box[0]}")
        eng.set_gathered(False)

    # end to end through the C ABI with host buffers: (a) the cached bit-packed silhouettes (SURVEY §7-1 cache format,
    # what the CPU arm consumes too) and (b) the 8UC3 undistorted masks as the reference holds them in memory
    e2e = None
    e2e_bgr = None
    e2e_dense = None
    noncarved_bricks_total = None
    if not args.no_e2e:
        out_occ = torch.empty((z1 - z0, Y, Wx), dtype=torch.int32).pin_memory()
        out_seen = torch.empty_like(out_occ).pin_memory()
        d2h = 2 * out_occ.numel() * 4
        bits_pinned = torch.from_numpy(w.mask_bits.view(np.int32)).pin_memory()
        bgr = torch.from_numpy(w.noisy_bgr if noisy else w.mask_bgr()).pin_memory()

        def e2e_run(use_bits):
            def one():
                eng.set_views(w.P, w.W, w.H, w.M)
                if use_bits:
                    eng.set_masks_bits_async(bits_pinned)
                else:
                    eng.set_masks_bgr(bgr, sync=False)
                eng.reset()
                eng.carve_download(out_occ, out_seen)   # carve + D2H of both volumes, z-chunks overlapped
            for _ in range(2):
                one()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                one()
            barrier()
            return allmax((time.perf_counter() - t0) / args.steps)

        s_bits = e2e_run(True)
        s_bgr = e2e_run(False)
        # sparse result: one flag byte per 32x8x8 brick + the words of the bricks that were evaluated per voxel
        nbz_, nby_, nbx_ = ((z1 - z0) + 7) // 8, (Y + 7) // 8, Wx
        flags_p = torch.empty(nbz_ * nby_ * nbx_, dtype=torch.uint8).pin_memory()
        cap = max(1024, flags_p.numel() // 4)
        listed_p = torch.empty(cap, dtype=torch.int32).pin_memory()
        words_p = torch.empty(cap * 128, dtype=torch.int32).pin_memory()
        sparse_n = [0]

        def one_sparse(use_bits=True):
            eng.set_views(w.P, w.W, w.H, w.M)
            if use_bits:
                eng.set_masks_bits_async(bits_pinned)
            else:
                eng.set_masks_bgr(bgr, sync=False)
            f_, l_, w_ = eng.carve_download_sparse(flags_p, listed_p, words_p)   # reset + carve + D2H of flags and listed words
            sparse_n[0] = len(l_)
            return f_, l_, w_

        def sparse_run(use_bits):
            for _ in range(2):
                one_sparse(use_bits)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                one_sparse(use_bits)
            barrier()
            return allmax((time.perf_counter() - t0) / args.steps)
        s_sparse = sparse_run(True)
        s_sparse_bgr = sparse_run(False)
        f_, l_, w_ = one_sparse()
        t0 = time.perf_counter()
        xo, xs = eng.expand_sparse(f_, l_, w_)
        expand_ms = (time.perf_counter() - t0) * 1e3
        eng.reset(), eng.carve()
        sparse_ok = bool(np.array_equal(xo, eng.download_occupied()) and np.array_equal(xs, eng.download_seen()))
        if not sparse_ok:
            raise SystemExit("bench.py: the expanded sparse result differs from the dense volumes")
        sparse_d2h = int(flags_p.numel() + sparse_n[0] * (4 + 512))
        noncarved_bricks_total = allsum(float(((np.asarray(f_) & 1) == 0).sum()))  # bricks whose words vc_carve_bricks writes (patch pass + work items)
        h2d_bits = int(bits_pinned.numel() * 4 + w.P.nbytes + w.M.nbytes)
        h2d_bgr = int(bgr.numel() + w.P.nbytes + w.M.nbytes)
        # kernels per e2e step: [pack_bgr] + 3 SAT passes + 2 classify + carve_bricks + flag resolve + pack  (dense: 4 z-chunks x (2 classify + fill + carve_bricks))
        e2e = {"value": nominal_total / s_sparse, "unit": UNIT, "h2d_bytes_per_step": h2d_bits, "d2h_bytes_per_step": sparse_d2h, "ms_per_step": s_sparse * 1e3,
               "input": "cached bit-packed undistorted silhouettes (VC_MASK_BITS) + P/M, pinned host memory",
               "result": f"sparse: one flag byte per 32x8x8-voxel brick + occupied/seen words of the {sparse_n[0]} listed bricks (vc_carve_download_sparse); "
                         "expands to exactly the dense volumes (checked after the timed region), which include/voxcarve_host.hpp applies to the Model brick by brick",
               "call": "vc_set_views + vc_set_masks + vc_reset + vc_carve_download_sparse", "gpu_launches": 9 * args.steps,
               "result_identical_to_dense": sparse_ok, "host_expand_numpy_ms_untimed": expand_ms}
        e2e_bgr = {"value": nominal_total / s_sparse_bgr, "unit": UNIT, "h2d_bytes_per_step": h2d_bgr, "d2h_bytes_per_step": sparse_d2h, "ms_per_step": s_sparse_bgr * 1e3,
                   "input": "8UC3 undistorted masks (VC_MASK_BGR8), packed on device", "result": "sparse", "gpu_launches": 10 * args.steps}
        e2e_dense = {"bits": {"value": nominal_total / s_bits, "ms_per_step": s_bits * 1e3, "h2d_bytes_per_step": h2d_bits, "d2h_bytes_per_step": int(d2h),
                              "call": "vc_set_views + vc_set_masks + vc_reset + vc_carve_download (both volumes as plain words, z-chunks overlapped with PCIe)", "gpu_launches": 19 * args.steps},
                     "bgr8": {"value": nominal_total / s_bgr, "ms_per_step": s_bgr * 1e3, "h2d_bytes_per_step": h2d_bgr, "d2h_bytes_per_step": int(d2h), "gpu_launches": 20 * args.steps}}
        if noisy:   # the hostile masks only exist as 8UC3: that path is the headline e2e of this config
            e2e, e2e_bgr = e2e_bgr, e2e
        eng.set_masks_bits(w.mask_bits)

    out = None
    if rank == 0:
        ffma, dfma = measure_peaks(local)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            key = f"{args.config}_x{world}"
            if key in tr:
                traffic = tr[key]["vc_carve_bricks_dram_bytes"]
        except Exception:
            pass
        kt_s = kernel_ms_max * 1e-3
        fine_s = fine_ms_max * 1e-3
        # projections of one vc_carve_bricks launch (rank average): per-voxel ones + the corners of its sub-brick classification
        exec_rank = (executed_total - corner_total + sub_corner_total) / world
        ach = exec_rank * F_ALG / fine_s / 1e12
        vol_bytes = 2.0 * (Z / world) * Y * Wx * 4
        alg_bytes = vol_bytes + w.mask_bits.nbytes
        # what vc_carve_bricks itself has to move: vc_blind_fill_kernel has written "carved and seen" everywhere, so the kernel writes
        # the words of the bricks that are not carved as a whole (patch pass of its first blocks + the work items' listed bricks: 64
        # words per brick and volume), reads each silhouette bit it tests at least once (<= the mask set) and four summed-area-table
        # corners per sub-brick test
        sat_bytes = sub_corner_total / world / 8.0 * 16.0
        if noncarved_bricks_total is None:  # --no-e2e: no flag bytes at hand; every occupied voxel lies in such a brick (2048 voxels each)
            noncarved_bricks_total = max(bricks_listed, occupied_total / 2048.0)
        brick_bytes = noncarved_bricks_total / world * 64 * 4 * 2
        cfg = config_dict(w, world, args.config)
        cfg["workload"] = workload_name(w)
        out = {
            "metric": METRIC, "value": nominal_total / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg, "l2": "flushed between timed iterations (256 MiB fill)", "slab_bounds": bounds,
            "value_cold": nominal_total / (cold_ms * 1e-3), "cold_ms_per_step": cold_ms,
            "value_with_consumer": nominal_total / (with_consumer_ms * 1e-3), "with_consumer_ms_per_step": with_consumer_ms,
            "with_consumer": "vc_reset + vc_carve" + (" + vc_exchange_halos (one plane of occupied per neighbour, NCCL send/recv)" if world > 1 else "")
                             + " + vc_mc_classify on the slab, per step, device time, max over ranks",
            "halo_exchange_ms": halo_ms,
            "executed_voxel_views": executed_total, "executed_fraction": executed_total / nominal_total,
            "executed_value": executed_total / (ms_per_step * 1e-3),
            "occupied_voxels": occupied_total, "carve_kernel_ms": kernel_ms_max, "grid_hash": hashes,
            "kernels_ms": {"vc_blind_fill_kernel + vc_brick_classify_kernel<1> + <0> (plain launches, in stream order; the graph of the timed steps runs the fill beside the other two)": classify_ms_max,
                           "vc_carve_bricks (incl. its patch pass)": fine_ms_max,
                           "flat_vc_carve_rows_same_job": flat_ms},
            "bricks": {"total": bricks_total, "needing_per_voxel_work": bricks_listed, "corner_projections": corner_total,
                       "of_which_sub_brick_level": sub_corner_total},
            "filter": {"evaluations_x32": filter_rows, "exact_reevaluations_x32": filter_slow, "mismatches_vs_exact": filter_bad,
                       "note": "per-voxel f32 filter with rigorous radius; every decision cross-checked against the exact path in the counting run"},
            "roofline": {"bound": "fp32", "achieved": ach, "peak": ffma, "unit": "TFLOP/s", "frac": ach / ffma if ffma else None,
                         "traffic": traffic, "algorithmic_bytes": brick_bytes + w.mask_bits.nbytes + sat_bytes,
                         "algorithmic_bytes_parts": {"words_of_bricks_not_carved_as_a_whole": brick_bytes, "silhouette_bits_read_once": w.mask_bits.nbytes, "sat_corners_of_sub_brick_tests": sat_bytes},
                         "blind_fill": {"kernel": "vc_blind_fill_kernel", "bytes": vol_bytes, "note": "both volumes written once with the 'carved and seen' pattern next to the classification; in compressible memory its DRAM traffic is a fraction of that (profiles/traffic.json)", "volumes_compressible": volumes_compressible},
                         "kernel": "vc_carve_bricks",
                         "peak_source": "FFMA microbenchmark on this GPU (vc_measure_peaks); MEASURED_PEAKS.json carries no FP32 CUDA-core entry",
                         "how": f"projections of one vc_carve_bricks launch ({exec_rank:.4g}: per-voxel + sub-brick corners) x {F_ALG:.0f} FLOP / its time "
                                f"({fine_ms_max:.3f} ms, CUDA events inside vc_carve: from the end of the classification to the end of the carve, i.e. the kernel with its patch pass); peak = FFMA microbenchmark on this GPU "
                                f"(vc_measure_peaks); DFMA peak {dfma:.1f} TFLOP/s. The kernel is issue-bound, see profiles/"},
            "roofline_hbm": {"bound": "hbm", "achieved": alg_bytes / kt_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes / kt_s / 1e9 / hbm_peak, "traffic": None, "write_only_floor_ms": vol_bytes / 6.4e12 * 1e3,
                             "how": f"grid-write bound: occupied+seen slab written once + masks read once = {alg_bytes / 1e6:.1f} MB / kernel time; peak = {hbm_src}; "
                                    "write_only_floor_ms = the two volumes at the 6.4 TB/s a store-only kernel reaches on this GPU (tools/experiments/fill_pattern_probe.cu, "
                                    "profiles/r2B_fill_probes.txt); vc_blind_fill_kernel runs at that rate"},
            "gather": gather, "mc_classify_ms": mc_ms, "mc_triangles": mc_tris, "color_ms": color_ms, "per_rank": per_rank,
            "e2e": e2e, "e2e_bgr8": e2e_bgr, "e2e_dense": e2e_dense, "gpu_launches": launches, "clocks": clk,
        }
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample, _ = cpu_reference(w, args.cpu_seconds, 1, 1)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if dumped:
            dump_outputs(args.dump_outputs, *dumped)
        emit(out)
    return 0


def TRI_COUNTS():
    """triangles per cube index from the packed table the library ships (csrc/mc_tables.inc): row length / 3"""
    txt = open(os.path.join(ROOT, "ar_voxel_project_b200", "csrc", "mc_tables.inc")).read()
    hexs = "".join(part for part in txt.split('"')[1::2])
    return [sum(c != "f" for c in hexs[i * 16:(i + 1) * 16]) // 3 for i in range(256)]


if __name__ == "__main__":
    a = parse()
    sys.exit(run_reference(a) if a.impl == "reference" else run_ours(a))
