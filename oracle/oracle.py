"""ctypes front-end of the CPU oracle (oracle/voxcarve_oracle.c).

TEST INFRASTRUCTURE, NOT PRODUCT: importable only from tests/, __graft_entry__.smoke()
and bench.py's cpu_baseline / --impl reference legs. Nothing under ar_voxel_project_b200/
imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libvoxcarve_oracle.so")
_lib = None

u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")


def build(force=False):
    src = os.path.join(_HERE, "voxcarve_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.vo_gemm3x3_3x4.argtypes = [f32p, f32p, f32p]
        L.vo_project.argtypes = [f32p, f32p, f32p]
        L.vo_round_to_int.argtypes = [C.c_float]
        L.vo_round_to_int.restype = C.c_int32
        L.vo_carve.argtypes = [C.c_int] * 3 + [C.c_float] + [C.c_int] * 5 + [f32p, C.c_void_p, C.c_void_p, u32p, u32p, C.c_int]
        L.vo_fast_carve.argtypes = [C.c_int] * 3 + [C.c_float] + [C.c_int] * 3 + [f32p, C.c_void_p, C.c_void_p, u32p, u32p]
        L.vo_color.argtypes = [C.c_int] * 3 + [C.c_float] + [C.c_int] * 3 + [f32p, f32p, u8p, u32p, C.c_int, u64p, u8p, C.c_uint64]
        L.vo_color.restype = C.c_uint64
        L.vo_mc_classify.argtypes = [C.c_int] * 3 + [u32p, u8p, u64p, u64p, u64p]
        L.vo_pixel_of.argtypes = [f32p] + [C.c_int] * 3 + [C.c_float, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), f32p]
        L.vo_max_threads.restype = C.c_int
        L.vo_box_pixel_bounds.argtypes = [f32p, C.c_float] + [C.c_int] * 9 + [np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")]
        L.vo_undistort.argtypes = [C.c_int, C.c_int, u8p, np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS"),
                                   np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS"), C.c_int, u8p]
        L.vo_undistort_map.argtypes = [C.c_int, C.c_int, np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS"),
                                       np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS"), C.c_int, C.c_void_p, C.c_void_p]
        L.vo_closure.argtypes = [C.c_int] * 4 + [f32p, f32p]
        L.vo_marching_cubes.argtypes = [C.c_int] * 3 + [f32p, C.c_float, np.ctypeslib.ndpointer(np.int8, flags="C_CONTIGUOUS"), f32p, u32p, C.c_uint64]
        L.vo_marching_cubes.restype = C.c_uint64
        L.vo_write_off.argtypes = [C.c_char_p, C.c_uint64, f32p, u32p] + [C.c_float] * 4
        _lib = L
    return _lib


def words_per_row(X):
    return (X + 31) // 32


def gemm3x3_3x4(K, M):
    P = np.empty((3, 4), np.float32)
    lib().vo_gemm3x3_3x4(np.ascontiguousarray(K, np.float32), np.ascontiguousarray(M, np.float32), P)
    return P


def project(P, w):
    out = np.empty(3, np.float32)
    lib().vo_project(np.ascontiguousarray(P, np.float32), np.ascontiguousarray(w, np.float32), out)
    return out


def round_to_int(v):
    return lib().vo_round_to_int(float(np.float32(v)))


def pixel_of(P, x, y, z, s, W, H):
    px, py = C.c_int(), C.c_int()
    uv = np.empty(2, np.float32)
    ins = lib().vo_pixel_of(np.ascontiguousarray(P, np.float32), x, y, z, float(np.float32(s)), W, H, C.byref(px), C.byref(py), uv)
    return bool(ins), px.value, py.value, uv


def box_pixel_bounds(P, lo, hi, s, W, H, nthreads=0):
    """the reference's pixels over EVERY voxel of the box [lo, hi] (inclusive x, y, z) -> (all_inside, none_inside, px_min,
    px_max, py_min, py_max, bad_depth): bad_depth = some voxel's proj_2 is <= 0 or not finite; NaN or out-of-range coordinates
    count as INT32_MIN.  nthreads < 1: every core"""
    out = np.empty(7, np.int32)
    rc = lib().vo_box_pixel_bounds(np.ascontiguousarray(P, np.float32).reshape(12), float(np.float32(s)), int(W), int(H),
                                   *(int(c) for c in lo), *(int(c) for c in hi), int(nthreads), out)
    if rc != 0:
        raise ValueError(f"empty box {lo} {hi}")
    return bool(out[0]), bool(out[1]), int(out[2]), int(out[3]), int(out[4]), int(out[5]), bool(out[6])


def _mask_args(mask_bits, mask_bgr):
    if mask_bits is not None:
        mb = np.ascontiguousarray(mask_bits, np.uint32)
        return mb, mb.ctypes.data, None
    mg = np.ascontiguousarray(mask_bgr, np.uint8)
    return mg, None, mg.ctypes.data


def carve(X, Y, Z, s, P, W, H, mask_bits=None, mask_bgr=None, z0=0, z1=None, nthreads=1):
    """-> (occupied, seen) uint32[(z1-z0), Y, ceil(X/32)]"""
    z1 = Z if z1 is None else z1
    P = np.ascontiguousarray(P, np.float32).reshape(-1, 12)
    keep, pb, pg = _mask_args(mask_bits, mask_bgr)
    occ = np.empty((z1 - z0, Y, words_per_row(X)), np.uint32)
    seen = np.empty_like(occ)
    rc = lib().vo_carve(X, Y, Z, float(np.float32(s)), z0, z1, len(P), W, H, P, pb, pg, occ, seen, nthreads)
    if rc != 0:
        raise RuntimeError(f"vo_carve failed: {rc}")
    return occ, seen


def fast_carve(X, Y, Z, s, P, W, H, mask_bits=None, mask_bgr=None):
    P = np.ascontiguousarray(P, np.float32).reshape(-1, 12)
    keep, pb, pg = _mask_args(mask_bits, mask_bgr)
    occ = np.empty((Z, Y, words_per_row(X)), np.uint32)
    seen = np.empty_like(occ)
    rc = lib().vo_fast_carve(X, Y, Z, float(np.float32(s)), len(P), W, H, P, pb, pg, occ, seen)
    if rc != 0:
        raise RuntimeError(f"vo_fast_carve failed: {rc}")
    return occ, seen


def color(X, Y, Z, s, P, M, W, H, images_bgr, occ, mode):
    """mode 1 = closest, 2 = average (the reference's -color flag). -> (idx uint64[n], rgbn uint8[n,4])"""
    P = np.ascontiguousarray(P, np.float32).reshape(-1, 12)
    M = np.ascontiguousarray(M, np.float32).reshape(-1, 12)
    img = np.ascontiguousarray(images_bgr, np.uint8)
    occ = np.ascontiguousarray(occ, np.uint32)
    cap = int(np.unpackbits(occ.view(np.uint8)).sum())
    idx = np.empty(max(cap, 1), np.uint64)
    rgbn = np.empty((max(cap, 1), 4), np.uint8)
    n = lib().vo_color(X, Y, Z, float(np.float32(s)), len(P), W, H, P, M, img, occ, mode, idx, rgbn, cap)
    return idx[:n].copy(), rgbn[:n].copy()


def tri_counts():
    """triangles per cube index, parsed from the packed table the product also ships."""
    txt = open(os.path.join(_HERE, "..", "ar_voxel_project_b200", "csrc", "mc_tables.inc")).read()
    hexs = "".join(part for part in txt.split('"')[1::2])
    assert len(hexs) == 4096
    return np.array([sum(c != "f" for c in hexs[i * 16:(i + 1) * 16]) // 3 for i in range(256)], np.uint8)


def mc_classify(X, Y, Z, occ):
    hist = np.zeros(256, np.uint64)
    na = np.zeros(1, np.uint64)
    nt = np.zeros(1, np.uint64)
    lib().vo_mc_classify(X, Y, Z, np.ascontiguousarray(occ, np.uint32), tri_counts(), hist, na, nt)
    return hist, int(na[0]), int(nt[0])


def max_threads():
    return lib().vo_max_threads()


def unpack(words, X):
    """uint32[..., Wx] -> bool[..., X]"""
    b = np.unpackbits(np.ascontiguousarray(words).view(np.uint8), bitorder="little").reshape(*words.shape[:-1], -1)
    return b[..., :X].astype(bool)


def tri_table():
    """triTable as int8[256,16] (-1 terminated), parsed from the packed table the product also ships"""
    txt = open(os.path.join(_HERE, "..", "ar_voxel_project_b200", "csrc", "mc_tables.inc")).read()
    hexs = "".join(part for part in txt.split('"')[1::2])
    return np.array([[-1 if c == "f" else int(c, 16) for c in hexs[i * 16:(i + 1) * 16]] for i in range(256)], np.int8)


def closure(X, Y, Z, rgba, kernel_size=3):
    """applyClosure on a dense RGBA model float32[X*Y*Z, 4] (flatten order). -> new array"""
    a = np.ascontiguousarray(rgba, np.float32).reshape(-1)
    out = np.empty_like(a)
    rc = lib().vo_closure(X, Y, Z, kernel_size, a, out)
    if rc != 0:
        raise ValueError("Invalid kernel size for post processing")
    return out.reshape(-1, 4)


def marching_cubes(X, Y, Z, rgba, threshold=0.5):
    """-> (verts float32[T,3,3], rgb uint32[T,3])"""
    a = np.ascontiguousarray(rgba, np.float32).reshape(-1)
    tt = np.ascontiguousarray(tri_table())
    n = lib().vo_marching_cubes(X, Y, Z, a, threshold, tt, np.empty(9, np.float32), np.empty(3, np.uint32), 0)
    verts = np.empty(max(n, 1) * 9, np.float32)
    rgb = np.empty(max(n, 1) * 3, np.uint32)
    n2 = lib().vo_marching_cubes(X, Y, Z, a, threshold, tt, verts, rgb, n)
    assert n2 == n
    return verts[:n * 9].reshape(n, 3, 3), rgb[:n * 3].reshape(n, 3)


def write_off(path, verts, rgb, scale=1.0, translation=(0.0, 0.0, 0.0)):
    v = np.ascontiguousarray(verts, np.float32).reshape(-1)
    c = np.ascontiguousarray(rgb, np.uint32).reshape(-1)
    rc = lib().vo_write_off(path.encode(), len(c) // 3, v, c, float(np.float32(scale)), *[float(np.float32(t)) for t in translation])
    if rc != 0:
        raise OSError(f"cannot write {path}")


def dense_model(X, Y, Z, occ_words, seen_words=None, color_idx=None, color_rgbn=None):
    """the reference Model's voxels after carve [+ colour pass] [+ handleUnseen] (Model.cpp:9-14,36-47): float32[X*Y*Z,4]"""
    occ = unpack(occ_words, X).reshape(-1)
    rgba = np.tile(np.array([50, 168, 141, 1], np.float32), (X * Y * Z, 1))
    rgba[~occ] = 0
    if color_idx is not None:
        m = color_rgbn[:, 3] > 0
        rgba[color_idx[m].astype(np.int64), :3] = color_rgbn[m, :3]
    if seen_words is not None:
        rgba[~unpack(seen_words, X).reshape(-1)] = (204, 0, 0, 1)
    return rgba


def undistort(img_bgr, K, dist):
    """cv::undistort of an 8UC3 image (VoxelCarving.cpp:36) -> uint8[H,W,3]"""
    img = np.ascontiguousarray(img_bgr, np.uint8)
    H, W = img.shape[:2]
    d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())
    out = np.empty_like(img)
    rc = lib().vo_undistort(W, H, img, np.ascontiguousarray(K, np.float64).reshape(9), d, len(d), out)
    if rc != 0:
        raise ValueError("distortion vector must have 4, 5 or 8 coefficients, and W and H must be below 32767")
    return out


def undistort_map(K, dist, W, H):
    """the int16 map cv::undistort remaps with, stripe by stripe: (int16[H,W,2] sx/sy, uint16[H,W] (iv & 31) * 32 + (iu & 31)),
    the layout of cv2.initUndistortRectifyMap(..., cv2.CV_16SC2)"""
    d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())
    sxy, frac = np.empty((H, W, 2), np.int16), np.empty((H, W), np.uint16)
    rc = lib().vo_undistort_map(int(W), int(H), np.ascontiguousarray(K, np.float64).reshape(9), d, len(d),
                                sxy.ctypes.data_as(C.c_void_p), frac.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise ValueError("distortion vector must have 4, 5 or 8 coefficients, and W and H must be below 32767")
    return sxy, frac
