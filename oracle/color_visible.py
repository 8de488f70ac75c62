"""ctypes front-end of oracle/color_visible_oracle.c: the CPU restatement of occlusion-aware colouring (vc_color_visible).

TEST INFRASTRUCTURE, NOT PRODUCT, like oracle/oracle.py.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "color_visible_oracle.c")
_SO = os.path.join(_HERE, "libcolor_visible_oracle.so")
_lib = None

f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")


def build(force=False):
    """gcc with the flags of oracle/Makefile: -ffp-contract=off, the reference arithmetic has no FMA contraction"""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility=hidden", "-Wall", "-Wextra",
                               "-std=c11", "-o", _SO, _SRC, "-lm"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.vo_color_visible.argtypes = ([C.c_int] * 3 + [C.c_float] + [C.c_int] * 3 + [f32p, f32p, u8p, u32p, C.c_int, C.c_float,
                                       u64p, u8p, C.c_void_p, C.c_uint64])
        L.vo_color_visible.restype = C.c_uint64
        _lib = L
    return _lib


def color_visible(X, Y, Z, s, P, M, W, H, images_bgr, occ, mode, tolerance, observations=False):
    """-> (idx uint64[n], rgbn uint8[n,4]) [, obs bool[n, V]: which views each record observes]"""
    P = np.ascontiguousarray(P, np.float32).reshape(-1, 12)
    M = np.ascontiguousarray(M, np.float32).reshape(-1, 12)
    V = len(P)
    img = np.ascontiguousarray(images_bgr, np.uint8)
    occ = np.ascontiguousarray(occ, np.uint32)
    cap = int(np.unpackbits(occ.view(np.uint8)).sum())
    idx = np.empty(max(cap, 1), np.uint64)
    rgbn = np.empty((max(cap, 1), 4), np.uint8)
    obs = np.zeros((max(cap, 1), V), np.uint8)
    n = lib().vo_color_visible(X, Y, Z, float(np.float32(s)), V, W, H, P, M, img, occ, mode, float(np.float32(tolerance)),
                               idx, rgbn, obs.ctypes.data if observations else None, cap)
    if n == 2**64 - 1:
        raise MemoryError("vo_color_visible: out of memory")
    out = idx[:n].copy(), rgbn[:n].copy()
    return out + (obs[:n].astype(bool),) if observations else out
