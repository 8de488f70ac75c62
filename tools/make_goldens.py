#!/usr/bin/env python3
"""Generate the golden fixtures under tests/golden/ (run ONLY in the build container).

Needs /root/reference (datasets) and Python cv2 4.13.0 — neither exists on the GPU
box, so everything this script produces is committed. Nothing under tests/, bench.py
or the product imports this file.

What it writes
  gemm_kat.npz          known-answer vectors for the projection arithmetic: outputs of
                        cv2.gemm (the function behind `intr * pose * world`,
                        VoxelCarving.cpp:19) on random, dataset-derived and adversarial
                        near-tie inputs.
  box_views.npz         the per-dataset pose/mask/image cache (SURVEY §7-1): K32, M, P,
  human_views.npz       bit-packed undistorted masks, PNG-encoded undistorted images.
  box_literal.npz       the reference algorithm run LITERALLY (one cv2.gemm pair per
  human_literal.npz     voxel-view, VoxelCarving.cpp:39-55; colour pass
                        ColorReconstruction.h:34-74 + .cpp:22-70) on small grids.
  soft_box_1off.json    header numbers of Data/box_dataset/generated_models/1.off.
  undistort_kat.npz     cv2.undistort known answers on dataset images and a few calibrations.
  undistort_hostile_kat.npz  cv2.undistort on seeded noise images over hostile calibrations and
                        sizes (`python tools/make_goldens.py undistort_hostile` writes only this
                        file; it needs cv2 4.13.0 and undistort_kat.npz, not the datasets).

Pose recipe follows PoseEstimation.h:18-76 using the cv2>=4.7 aruco API (the legacy
free functions are gone from 4.13): detectMarkers -> interpolateCornersCharuco ->
estimatePoseCharucoBoard -> Rodrigues -> [R^T | -R^T t] as CV_32F.
"""
import glob
import hashlib
import json
import math
import os
import sys

import cv2
import numpy as np

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")
f32 = np.float32


# ----------------------------------------------------------------------------- poses
def read_calibration(path):
    fs = cv2.FileStorage(path, cv2.FILE_STORAGE_READ)
    K = fs.getNode("camera_matrix").mat()
    dist = fs.getNode("distortion_coefficients").mat()
    fs.release()
    return K, dist


def estimate_pose(K, dist, image):
    """PoseEstimation.h:18-76 -> 4x4 CV_32F camera->world, identity on failure (:34)."""
    dictionary = cv2.aruco.getPredefinedDictionary(cv2.aruco.DICT_6X6_250)
    board = cv2.aruco.CharucoBoard((5, 7), 0.04, 0.02, dictionary)
    cp = cv2.aruco.CharucoParameters()
    cp.cameraMatrix = K
    cp.distCoeffs = dist
    det = cv2.aruco.CharucoDetector(board, cp, cv2.aruco.DetectorParameters())
    ch_corners, ch_ids, m_corners, m_ids = det.detectBoard(image)
    T = np.eye(4, dtype=f32)
    n_ch = 0 if ch_ids is None else len(ch_ids)
    if m_ids is None or len(m_ids) == 0 or n_ch == 0:
        return T, n_ch, False
    rvec = np.zeros((3, 1))
    tvec = np.zeros((3, 1))
    valid = False
    if n_ch >= 4:  # estimatePoseCharucoBoard needs >= 4 corners
        obj, img = board.matchImagePoints(ch_corners, ch_ids)
        valid, rvec, tvec = cv2.solvePnP(obj, img, K, dist)
    # the `if (valid)` at PoseEstimation.h:48 guards only drawFrameAxes: the matrix is
    # built from rvec/tvec (zeros when invalid) either way (:50-67)
    R, _ = cv2.Rodrigues(rvec)
    Rt = R.T
    t = -Rt @ tvec
    T[:3, :3] = Rt.astype(f32)
    T[:3, 3] = t.ravel().astype(f32)
    return T, n_ch, bool(valid)


def pack_bits(bg):
    """bg: (H, W) bool, True = background (carve). -> (H, ceil(W/32)) uint32, bit x&31."""
    H, W = bg.shape
    Ww = (W + 31) // 32
    pad = np.zeros((H, Ww * 32), dtype=np.uint8)
    pad[:, :W] = bg
    b = np.packbits(pad.reshape(H, Ww, 32), axis=2, bitorder="little")  # (H, Ww, 4) bytes
    return b.reshape(H, Ww, 4).view("<u4").reshape(H, Ww).copy()


def build_cache(name):
    d = os.path.join(REF, "Data", name)
    K, dist = read_calibration(os.path.join(d, "cameracalibration.yml"))
    # cv::glob sorts lexicographically (main.cpp:203-208)
    img_files = sorted(glob.glob(os.path.join(d, "images", "*")))
    msk_files = sorted(glob.glob(os.path.join(d, "masks", "*")))
    assert len(img_files) == len(msk_files) and img_files
    K32 = K.astype(f32)  # VoxelCarving.cpp:29-30
    Ms, Ps, Ts, bits, pngs, info = [], [], [], [], [], []
    for fi, fm in zip(img_files, msk_files):
        image = cv2.imread(fi, 1)
        mask = cv2.imread(fm, 1)
        T, n_ch, valid = estimate_pose(K, dist, image)
        inv = cv2.invert(T)[1]  # pose.inv(), 4x4 f32 LU (VoxelCarving.cpp:26)
        M = np.ascontiguousarray(inv[:3, :])  # pose(Rect(0,0,4,3)) (:41)
        P = cv2.gemm(K32, M, 1.0, None, 0.0)  # first product of `intr * pose * world` (:19)
        und_mask = cv2.undistort(mask, K, dist)  # (:36)
        und_img = cv2.undistort(image, K, dist)  # ColorReconstruction.h:23
        bg = (und_mask[:, :, 0] == 0) & (und_mask[:, :, 1] == 0) & (und_mask[:, :, 2] == 0)  # (:50)
        ok, png = cv2.imencode(".png", und_img, [cv2.IMWRITE_PNG_COMPRESSION, 9])
        assert ok
        Ms.append(M), Ps.append(P), Ts.append(T), bits.append(pack_bits(bg)), pngs.append(png.ravel())
        info.append((os.path.basename(fi), n_ch, valid, float(bg.mean())))
    H, W = image.shape[:2]
    offs = np.cumsum([0] + [len(p) for p in pngs]).astype(np.int64)
    np.savez_compressed(
        os.path.join(OUT, f"{name.split('_')[0]}_views.npz"),
        V=len(Ms), W=W, H=H, K32=K32, M=np.stack(Ms), P=np.stack(Ps), T_c2w=np.stack(Ts),
        mask_bits=np.stack(bits), png_blob=np.concatenate(pngs), png_offsets=offs,
        files=np.array([i[0] for i in info]),
    )
    for i in info:
        print(f"  {name}: {i[0]:>14s} charuco={i[1]:2d} valid={i[2]} bg_frac={i[3]:.3f}")
    return dict(K=K, dist=dist, K32=K32, M=np.stack(Ms), P=np.stack(Ps), bits=np.stack(bits),
                W=W, H=H, images=[cv2.imdecode(p, 1) for p in pngs])


# ----------------------------------------------------------------------- literal run
def c_round(x):
    """(int)std::round(float): half away from zero; NaN/inf/overflow -> INT_MIN (x86)."""
    x = float(x)
    if not math.isfinite(x):
        return -(2 ** 31)
    r = math.floor(abs(x) + 0.5)
    r = -r if x < 0 else r
    if r >= 2 ** 31 or r < -(2 ** 31):
        return -(2 ** 31)
    return int(r)


def literal_run(cache, X, Y, Z, s, out_name):
    """Reference semantics with the reference's own arithmetic calls (cv2.gemm per voxel-view)."""
    s = f32(s)
    K32, Ms, bits, W, H = cache["K32"], cache["M"], cache["bits"], cache["W"], cache["H"]
    V = len(Ms)
    occ = np.ones((Z, Y, X), dtype=bool)  # Model ctor: alpha = 1 (Model.cpp:9-14)
    seen = np.zeros((Z, Y, X), dtype=bool)
    px_all = np.zeros((V, Z, Y, X, 2), dtype=np.int64)
    for v in range(V):
        for x in range(X):
            for y in range(Y):
                for z in range(Z):
                    w = np.array([[f32(y) * s], [f32(x) * s], [f32(-1 * z) * s], [f32(1)]], dtype=f32)  # Model.h:134-136
                    proj = cv2.gemm(cv2.gemm(K32, Ms[v], 1.0, None, 0.0), w, 1.0, None, 0.0).ravel()  # :19
                    with np.errstate(all="ignore"):
                        u, vv = proj[0] / proj[2], proj[1] / proj[2]  # :20, f32 divides
                    px, py = c_round(u), c_round(vv)  # :44
                    px_all[v, z, y, x] = (px, py)
                    if not (0 <= px < W and 0 <= py < H):  # :45
                        continue
                    if (bits[v, py, px >> 5] >> np.uint32(px & 31)) & np.uint32(1):  # :50
                        occ[z, y, x] = False
                    seen[z, y, x] = True  # :54
    # colour pass (ColorReconstruction.h:34-74) on the carved model, both bodies
    def get(x, y, z):
        if x < 0 or x >= X or y < 0 or y >= Y or z < 0 or z >= Z:
            return False
        return bool(occ[z, y, x])
    cams = [np.array([M[0, 3], M[1, 3], M[2, 3], 1], dtype=f32) for M in Ms]  # ColorReconstruction.h:21
    surf, avg, closest, nobs = [], [], [], []
    norm_diff = 0
    for x in range(X):
        for y in range(Y):
            for z in range(Z):
                inner = (get(x - 1, y, z) and get(x + 1, y, z) and get(x, y - 1, z)
                         and get(x, y + 1, z) and get(x, y, z - 1) and get(x, y, z + 1))
                if not occ[z, y, x] or inner:
                    continue
                w = np.array([f32(y) * s, f32(x) * s, f32(-1 * z) * s, f32(1)], dtype=f32)
                obs = []
                for v in range(V):
                    px, py = px_all[v, z, y, x]
                    if not (0 <= px < W and 0 <= py < H):
                        continue
                    b, g, r = cache["images"][v][py, px]
                    d = (cams[v] - w).astype(f32)  # Vec4f - Vec4f
                    dd = d.astype(np.float64)
                    # cv::norm(Vec4f): sqrt of f64-accumulated squares (recalled from matx.hpp), -> float depth
                    depth = f32(math.sqrt(((dd[0] * dd[0] + dd[1] * dd[1]) + dd[2] * dd[2]) + dd[3] * dd[3]))
                    if f32(cv2.norm(d.reshape(4, 1))) != depth:
                        norm_diff += 1
                    obs.append((int(r), int(g), int(b), depth))
                surf.append((x, y, z)), nobs.append(len(obs))
                if not obs:
                    avg.append((50, 168, 141)), closest.append((50, 168, 141))  # MODEL_COLOR untouched
                    continue
                sm = [f32(0), f32(0), f32(0)]
                for o in obs:
                    sm = [f32(sm[i] + f32(o[i])) for i in range(3)]
                a = [c_round(f32(sm[i] / f32(len(obs)))) for i in range(3)]  # .cpp:60-66
                avg.append(tuple(a))
                best = obs[0]
                for o in obs[1:]:
                    if o[3] < best[3]:  # .cpp:34-40 first strict minimum
                        best = o
                closest.append(best[:3])
    np.savez_compressed(os.path.join(OUT, out_name), X=X, Y=Y, Z=Z, s=s, occ=occ, seen=seen,
                        surf=np.array(surf, dtype=np.int32), nobs=np.array(nobs, dtype=np.int32),
                        avg=np.array(avg, dtype=np.uint8), closest=np.array(closest, dtype=np.uint8))
    print(f"  {out_name}: occupied={int(occ.sum())}/{occ.size} seen={int(seen.sum())} surface={len(surf)} "
          f"cv2.norm-vs-model depth mismatches={norm_diff}")


# ---------------------------------------------------------------------------- gemm KAT
def gemm_kat(caches):
    rng = np.random.default_rng(20261018)
    Ps, ws = [], []
    # (1) dataset matrices x lattice points at several voxel sizes
    for c in caches:
        for P in c["P"]:
            for _ in range(400):
                s = f32(rng.choice([0.0028, 0.0056, 0.028, 0.28 / 1024, 0.28 / 2048]))
                x, y, z = rng.integers(0, 2048, 3)
                Ps.append(P), ws.append([f32(y) * s, f32(x) * s, f32(-z) * s, f32(1)])
    # (2) random matrices incl. behind-camera / near-zero depth
    for _ in range(20000):
        P = (rng.standard_normal((3, 4)) * rng.choice([1, 100, 500, 4000])).astype(f32)
        Ps.append(P), ws.append([f32(rng.uniform(0, .3)), f32(rng.uniform(0, .3)), f32(-rng.uniform(0, .3)), f32(1)])
    # (3) adversarial near-tie rows: discriminate the f64 association order (see DESIGN.md)
    for _ in range(20000):
        m = f32(1 + rng.integers(0, 2 ** 23) / 2 ** 23)
        tie = f32(2.0 ** -24) * rng.choice([1, -1, 3, -3])
        tiny = [f32(rng.integers(1, 8) * 2.0 ** -int(rng.integers(53, 57))) * rng.choice([1, -1]) for _ in range(2)]
        sv = [m, tie] + tiny
        sv = [sv[i] for i in rng.permutation(4)]
        sc = [f32(2.0 ** int(rng.integers(-3, 4))) for _ in range(3)] + [f32(1)]
        P = np.array([[sv[k] / sc[k] for k in range(4)]] * 3, dtype=f32)
        P[1] *= f32(2)
        P[2] *= f32(-0.5)
        Ps.append(P), ws.append(sc)
    Ps = np.array(Ps, dtype=f32)
    ws = np.array(ws, dtype=f32)
    out = np.stack([cv2.gemm(P, w.reshape(4, 1), 1.0, None, 0.0).ravel() for P, w in zip(Ps, ws)])
    # K32 * M (3x3 . 3x4) vectors
    Ks = (rng.standard_normal((4000, 3, 3)) * 400).astype(f32)
    Mm = rng.standard_normal((4000, 3, 4)).astype(f32)
    KM = np.stack([cv2.gemm(a, b, 1.0, None, 0.0) for a, b in zip(Ks, Mm)])
    np.savez_compressed(os.path.join(OUT, "gemm_kat.npz"), P=Ps, w=ws, proj=out, K=Ks, M=Mm, KM=KM)
    print(f"  gemm_kat.npz: {len(Ps)} 3x4.4x1 vectors, {len(Ks)} 3x3.3x4 vectors (cv2 {cv2.__version__})")


def soft_golden():
    p = os.path.join(REF, "Data/box_dataset/generated_models/1.off")
    with open(p) as f:
        assert f.readline().strip() == "OFF"
        nv, nf, _ = map(int, f.readline().split())
        verts = np.array([[float(t) for t in f.readline().split()] for _ in range(nv)])
        faces = [f.readline().split() for _ in range(nf)]
    # vertices are voxel indices * 0.0028 (scale 1, no translation): keep them as the multiset of integer index triplets
    idx = np.rint(verts / 0.0028).astype(np.int16)
    assert np.abs(verts / 0.0028 - idx).max() < 1e-2
    uniq, counts = np.unique(idx, axis=0, return_counts=True)
    colors = sorted({tuple(int(c) for c in fc[4:7]) for fc in faces})
    np.savez_compressed(os.path.join(OUT, "soft_box_1off_vertices.npz"), uniq=uniq, counts=counts.astype(np.int32),
                        first_lines=np.array(open(p).read().splitlines()[:12]), face_colors=np.array(colors, np.int32))
    json.dump({"source": "Data/box_dataset/generated_models/1.off", "vertices": nv, "faces": nf,
               "command": "-c=5 -z=50 (x=y=100, size=0.0028, carve=1, color=0, postprocessing=true)"},
              open(os.path.join(OUT, "soft_box_1off.json"), "w"), indent=1)
    print(f"  soft_box_1off.json: {nv} vertices / {nf} faces")


def undistort_kat():
    """cv2.undistort (VoxelCarving.cpp:36, ColorReconstruction.h:23) known answers: raw inputs + outputs, PNG-compressed."""
    rng = np.random.default_rng(7)
    K, dist = read_calibration(os.path.join(REF, "Data/box_dataset/cameracalibration.yml"))
    cases = []
    cases.append(("box_mask0000", cv2.imread(os.path.join(REF, "Data/box_dataset/masks/mask0000.jpg"), 1), K, dist))
    cases.append(("box_image0003", cv2.imread(os.path.join(REF, "Data/box_dataset/images/image0003.jpg"), 1), K, dist))
    cases.append(("human_mask_5", cv2.imread(os.path.join(REF, "Data/human_dataset/masks/5.jpg"), 1), K, dist))
    K2 = np.array([[150.3, 0, 99.7], [0, 149.1, 60.2], [0, 0, 1]])
    cases.append(("random_strong5", rng.integers(0, 256, (123, 201, 3), dtype=np.uint8), K2, np.array([[0.4, -0.9, 0.01, -0.02, 0.3]])))
    cases.append(("random_k8", rng.integers(0, 256, (97, 130, 3), dtype=np.uint8), np.array([[90.5, 0.3, 64.2], [0, 91.5, 48.9], [0, 0, 1]]),
                  np.array([[0.2, -0.1, 0.003, 0.004, 0.05, 0.1, -0.05, 0.02]])))
    cases.append(("random_4coef_tall", rng.integers(0, 256, (301, 33, 3), dtype=np.uint8), np.array([[40.0, 0, 16.0], [0, 42.0, 150.0], [0, 0, 1]]),
                  np.array([[-0.3, 0.1, 0.0, 0.0]])))
    out = {}
    for name, img, Kc, dc in cases:
        ref = cv2.undistort(img, Kc, dc)
        ok1, a = cv2.imencode(".png", img, [cv2.IMWRITE_PNG_COMPRESSION, 9])
        ok2, b = cv2.imencode(".png", ref, [cv2.IMWRITE_PNG_COMPRESSION, 9])
        out[name + "_src"], out[name + "_dst"], out[name + "_K"], out[name + "_dist"] = a.ravel(), b.ravel(), Kc, dc
    np.savez_compressed(os.path.join(OUT, "undistort_kat.npz"), names=np.array([c[0] for c in cases]), **out)
    print(f"  undistort_kat.npz: {len(cases)} cases (cv2 {cv2.__version__})")


def undistort_hostile_cases():
    """(name, W, H, K, dist, seed) of the undistort sweep: the dataset calibration at three sizes, random calibrations, round-number
    K that put many map coordinates on rounding ties, distortion strong enough to leave int16 and int32, a rational denominator
    that reaches 0 inside the image, and widths for every column count of the scalar tail (W % 8) and for the 4096 / W stripes."""
    z = np.load(os.path.join(OUT, "undistort_kat.npz"))
    K0, d0 = z["box_mask0000_K"], z["box_mask0000_dist"].ravel()  # Data/box_dataset/cameracalibration.yml
    Km = lambda fx, fy, cx, cy, skew=0.0: np.array([[fx, skew, cx], [0, fy, cy], [0, 0, 1.0]])
    cases = [("dataset_640x480", 640, 480, K0, d0)]
    for f, (W, H) in [(3, (1920, 1080)), (6, (3840, 2160))]:
        cases.append((f"dataset_{W}x{H}", W, H, K0 * [[f], [f], [1]], d0))
    rng = np.random.default_rng(2026)
    for t, n in enumerate([4, 5, 8, 4, 5, 8]):
        W, H = int(rng.integers(60, 700)), int(rng.integers(30, 500))
        f = rng.uniform(0.5, 2) * W
        K = Km(f, f * rng.uniform(0.9, 1.1), W / 2 + rng.normal() * W / 10, H / 2 + rng.normal() * H / 10, rng.normal() * 2)
        cases.append((f"random{t}_n{n}", W, H, K, rng.normal(size=n) * np.array([0.3, 0.5, 0.01, 0.01, 0.5, 0.3, 0.3, 0.3])[:n]))
    ties = [("tie_500_k1", 640, 480, Km(500, 500, 320, 240), [0.25, 0, 0, 0]),
            ("tie_512_k1k2", 643, 480, Km(512, 512, 320, 240), [0.25, -0.125, 0, 0]),
            ("tie_512_tangential", 645, 481, Km(512, 512, 320, 240), [0, 0, 1 / 64, -1 / 32]),
            ("tie_512_rational", 647, 479, Km(512, 512, 320, 240), [0, 0, 0, 0, 0, 0.125, -0.0625, 0.03125]),
            ("tie_500_zero", 641, 477, Km(500, 500, 320, 240), [0, 0, 0, 0, 0])]
    strong = [("int16_k3", 100, 40, Km(100, 100, 50, 20), [5, 500, 0, 0, 1e5]),      # |u| past 2^15
              ("int16_tail", 1001, 77, Km(100, 100, 500, 38), [5, 50, 0.1, 0.1, 500]),
              ("int32_k3", 103, 40, Km(100, 100, 50, 20), [5, 500, 0, 0, 1e9]),      # u * 32 past 2^31
              ("int32_tail", 1001, 61, Km(100, 100, 0, 30), [5, 50, 0.1, 0.1, 500]),
              ("den0_tail", 101, 41, Km(100, 100, 50, 20), [0, 0, 0, 0, 0, -4, 0, 0]),  # 1 + k4 r2 = 0 at column 100
              ("den0_body", 104, 41, Km(100, 100, 4, 20), [0, 0, 0, 0, 0, -4, 0, 0]),   # ... at column 54
              ("den0_wide", 333, 211, Km(120, 121, 166, 105), [0.1, 0, 0, 0, 0, -3, 0.5, 0.1])]
    cases += [(n, W, H, K, np.array(d, np.float64)) for n, W, H, K, d in ties + strong]
    for r in range(8):  # every W % 8, twice, with a strong random calibration
        for W in (8 * int(rng.integers(1, 6)) + r, 8 * int(rng.integers(20, 90)) + r):
            W = max(W, 1)
            H = int(rng.integers(1, 90))
            f = rng.uniform(0.3, 1.5) * W
            n = int(rng.choice([4, 5, 8]))
            d = rng.normal(size=n) * np.array([0.5, 0.5, 0.05, 0.05, 1, 0.5, 0.5, 0.5])[:n] * float(rng.choice([1, 10]))
            cases.append((f"w{W}_h{H}", W, H, Km(f, f * rng.uniform(0.95, 1.05), rng.uniform(0, W), rng.uniform(0, H), rng.normal()), d))
    cases += [("w1", 1, 300, Km(100, 100, 0, 150), np.array([0.3, 0.1, 0, 0])),
              ("h1", 300, 1, Km(100, 100, 150, 0), np.array([0.3, 0.1, 0.01, 0])),
              ("w1_h1", 1, 1, Km(2, 2, 0.5, 0.5), np.array([0.3, 0.1, 0, 0])),
              ("stripe40_h77", 100, 77, Km(80, 80, 50, 38), np.array([-0.2, 0.05, 0.001, 0.002, 0.01])),   # stripe 40
              ("stripe13_h50", 300, 50, Km(250, 250, 150, 25), np.array([0.2, -0.1, 0, 0])),              # stripe 13
              ("stripe1_w5000", 5000, 3, Km(2500, 2500, 2500, 1.5), np.array([0.1, -0.05, 0.001, 0, 0.02])),
              ("w32766", 32766, 2, Km(16000, 16000, 16383, 1), np.array([0.3, 0.1, 0, 0]))]
    return [(n, W, H, np.asarray(K, np.float64), np.asarray(d, np.float64), 1000 + i) for i, (n, W, H, K, d) in enumerate(cases)]


def undistort_hostile_kat():
    """cv2.undistort over undistort_hostile_cases() on noise images from the seeds: the SHA-256 of every input and output, the
    output itself for the cases of at most 20000 pixels, and the cv2 version and CPU path the answers came from."""
    cases = undistort_hostile_cases()
    out = {"names": np.array([c[0] for c in cases]), "cv2_version": np.array(cv2.__version__),
           "dispatch": np.array("AVX2" if cv2.checkHardwareSupport(11) else "baseline")}
    for name, W, H, K, d, seed in cases:
        img = np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)
        ref = cv2.undistort(img, K, d)
        out[f"{name}_WHseed"] = np.array([W, H, seed], np.int64)
        out[f"{name}_K"], out[f"{name}_dist"] = K, d
        out[f"{name}_src_sha256"] = np.array(hashlib.sha256(img.tobytes()).hexdigest())
        out[f"{name}_sha256"] = np.array(hashlib.sha256(ref.tobytes()).hexdigest())
        if W * H <= 20000:
            out[f"{name}_dst"] = ref
    np.savez_compressed(os.path.join(OUT, "undistort_hostile_kat.npz"), **out)
    print(f"  undistort_hostile_kat.npz: {len(cases)} cases (cv2 {cv2.__version__}, {out['dispatch']})")


def main():
    os.makedirs(OUT, exist_ok=True)
    if sys.argv[1:] == ["undistort_hostile"]:
        undistort_hostile_kat()
        return
    print("cv2", cv2.__version__)
    box = build_cache("box_dataset")
    human = build_cache("human_dataset")
    gemm_kat([box, human])
    literal_run(box, 24, 20, 12, 0.012, "box_literal.npz")
    literal_run(human, 20, 24, 28, 0.011, "human_literal.npz")
    soft_golden()
    undistort_kat()
    undistort_hostile_kat()
    for f in sorted(os.listdir(OUT)):
        p = os.path.join(OUT, f)
        print(f"  {f:24s} {os.path.getsize(p):9d} B sha256={hashlib.sha256(open(p,'rb').read()).hexdigest()[:16]}")


if __name__ == "__main__":
    sys.exit(main())
