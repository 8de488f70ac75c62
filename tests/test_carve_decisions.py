"""The carve's two approximations, checked in the compiled code against the reference pixel of every voxel.

vc_probe_boxes runs the brick classifier of vc_brick_classify_kernel / vc_carve_bricks, vc_probe_voxels the per-voxel f32 filter
of vc_carve_bricks and the exact evaluation, on boxes and voxel-views chosen here, with an engine's own views, tables and
constants.  The reference is the C oracle (vo_box_pixel_bounds: every voxel of a box) and the numpy restatement of the reference
arithmetic in test_classifier_math.py, which that file checks against the oracle voxel by voxel.  (test_classifier_math.py checks
the derivation behind the radii on a numpy restatement of the kernels; this file checks the kernels.)

A classifier answer is sound when code 1 has no voxel inside the image, codes 2-4 have every voxel inside and every voxel's
pixel in the rectangle, and codes 2 / 3 agree with the background count of the rectangle.  A filter answer is sound when a decided
voxel-view has the reference's pixel and inside test.  The cases come in named families; the constructed near-ties put a
voxel's (or a box corner's) u_ref at a chosen distance from a pixel edge k + 1/2 by stepping P[0][3] or P[1][3] one f32 at a time.
The CPU test at the end shows that the sampling reaches the cases where the radii matter: the numpy restatement with its radii
set to 0 fails the same checks on the same cases.  VC_PROBE_SEEDS=n runs n seeds of the GPU sampling (default 1).
"""
import os
from collections import Counter, defaultdict

import numpy as np
import pytest

from test_classifier_math import WIDE_TALL, filter_constants, filter_pixels, random_camera, rect_of_box, tie_camera

F = np.float32
LEVELS = {"super": (128, 32, 32), "brick": (32, 8, 8), "sub": (8, 8, 8)}


# ---- reference arithmetic for many (view, voxel) pairs ------------------------------------------------------------------------
def reference(P, xs, ys, zs, s, W, H):
    """(px, py, inside, u, v, p2) of voxel-views with per-voxel-view matrices P[n, 3, 4]: the restatement of
    test_classifier_math.reference_pixels (DESIGN.md section 2), with the quotients and the depth handed back too"""
    w = [(ys.astype(F) * F(s)).astype(np.float64), (xs.astype(F) * F(s)).astype(np.float64), ((-zs).astype(F) * F(s)).astype(np.float64)]
    Pd = P.astype(np.float64)
    with np.errstate(all="ignore"):
        proj = [((((Pd[:, i, 0] * w[0]) + (Pd[:, i, 1] * w[1])) + (Pd[:, i, 2] * w[2])) + Pd[:, i, 3]).astype(F) for i in range(3)]
        u = (proj[0] / proj[2]).astype(F)
        v = (proj[1] / proj[2]).astype(F)
        ud, vd = u.astype(np.float64), v.astype(np.float64)
        px = np.where(ud >= 0, np.floor(ud + 0.5), -np.floor(-ud + 0.5))
        py = np.where(vd >= 0, np.floor(vd + 0.5), -np.floor(-vd + 0.5))
    inside = np.isfinite(px) & np.isfinite(py) & (px >= 0) & (px < W) & (py >= 0) & (py < H)
    return px, py, inside, u, v, proj[2]


def bg_count(bits, px0, px1, py0, py1):
    """background pixels of the rectangle [px0, px1] x [py0, py1] of one view's mask words uint32[H, Ww]"""
    j0, j1 = px0 >> 5, (px1 >> 5) + 1
    sub = np.ascontiguousarray(bits[py0:py1 + 1, j0:j1])
    b = np.unpackbits(sub.view(np.uint8), axis=-1, bitorder="little")
    return int(b[:, px0 - 32 * j0:px1 - 32 * j0 + 1].sum())


# ---- scenes: one engine's grid, slab, views, masks, and the boxes and voxel-views probed on it -----------------------------
class Scene:
    def __init__(self, family, name, dims, s, W, H, P, z0=0, z1=None):
        self.family, self.name = family, name
        self.X, self.Y, self.Z = dims
        self.s, self.W, self.H = F(s), int(W), int(H)
        self.P = np.ascontiguousarray(P, F).reshape(-1, 3, 4)
        self.z0, self.z1 = z0, (self.Z if z1 is None else z1)
        self.Ww = (self.W + 31) // 32
        self.boxes = np.zeros((0, 7), np.int32)
        self.vox = np.zeros((0, 4), np.int32)
        self.near = np.zeros(0, bool)     # voxel-views that are constructed near-ties
        self.masks = None                 # uint32[V, H, Ww], 1 = background: the set the engine holds last
        self.first_masks = None           # a different set handed to vc_set_masks before (the tables must forget it)
        self.expect = set()               # classifier codes this family must produce

    @property
    def V(self):
        return len(self.P)

    def add_boxes(self, b):
        self.boxes = np.concatenate([self.boxes, np.asarray(b, np.int32).reshape(-1, 7)])

    def add_vox(self, v, near=False):
        v = np.asarray(v, np.int32).reshape(-1, 4)
        self.vox = np.concatenate([self.vox, v])
        self.near = np.concatenate([self.near, np.full(len(v), near)])


def lattice_boxes(rng, sc, n, level, views=None):
    """n boxes of one level of the carve's hierarchy, on its lattice (x, y from 0, z from the slab's first plane) and clipped at
    the grid and slab edges as the kernels clip them; random views"""
    bx, by, bz = LEVELS[level]
    nz = sc.z1 - sc.z0
    x0 = rng.integers(0, -(-sc.X // bx), n) * bx
    y0 = rng.integers(0, -(-sc.Y // by), n) * by
    z0 = rng.integers(0, -(-nz // bz), n) * bz
    v = rng.integers(0, sc.V, n) if views is None else np.asarray(views)[rng.integers(0, len(views), n)]
    return np.stack([v, x0, y0, sc.z0 + z0, np.minimum(x0 + bx, sc.X) - 1, np.minimum(y0 + by, sc.Y) - 1,
                     sc.z0 + np.minimum(z0 + bz, nz) - 1], 1)


def random_vox(rng, sc, n, views=None):
    v = rng.integers(0, sc.V, n) if views is None else np.asarray(views)[rng.integers(0, len(views), n)]
    return np.stack([v, rng.integers(0, sc.X, n), rng.integers(0, sc.Y, n), rng.integers(sc.z0, sc.z1, n)], 1)


def blob_masks(rng, V, W, H):
    """1 = background; each view: a few foreground ellipses and rectangles over a background, large uniform regions of both"""
    from ar_voxel_project_b200.synth import pack_bits
    out = np.empty((V, H, (W + 31) // 32), np.uint32)
    yy, xx = np.ogrid[0:H, 0:W]
    for v in range(V):
        fg = np.zeros((H, W), bool)
        for _ in range(int(rng.integers(1, 4))):
            cx, cy = rng.uniform(0, W), rng.uniform(0, H)
            rx, ry = W * rng.uniform(0.05, 0.35), H * rng.uniform(0.05, 0.35)
            if rng.random() < 0.5:
                fg |= ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 <= 1.0
            else:
                fg |= (np.abs(xx - cx) <= rx) & (np.abs(yy - cy) <= ry)
        if rng.random() < 0.1:
            fg[:] = rng.random() < 0.5   # a view that is all foreground or all background
        out[v] = pack_bits(~fg)
    return out


def band_masks(rng, V, W, H):
    """1 = background in a checkerboard of word bands: cheap masks for very large images"""
    Ww = (W + 31) // 32
    out = np.empty((V, H, Ww), np.uint32)
    for v in range(V):
        a, b = int(rng.integers(1, 64)), int(rng.integers(8, 512))
        i, j = np.ogrid[0:H, 0:Ww]
        out[v] = np.where(((j // a) + (i // b)) % 2 == 0, np.uint32(0xFFFFFFFF), np.uint32(0))
    if W % 32:
        out[..., -1] &= np.uint32((1 << (W % 32)) - 1)
    return out


# ---- constructed near-ties -------------------------------------------------------------------------------------------------
def step_f32(x, k):
    """x stepped k floats up (k < 0: down) through the f32 values"""
    x = np.full(np.shape(k), F(x)) if np.ndim(k) else F(x)
    k = np.asarray(k)
    out = x.copy()
    for sgn, d in ((1, np.inf), (-1, -np.inf)):
        m = np.sign(k) == sgn
        for _ in range(int(np.abs(k).max(initial=0))):
            out = np.where(m & (np.abs(k) > 0), np.nextafter(out, F(d)), out).astype(F)
            k = np.where(m, k - sgn, k)
    return out


def place_tie(P, row, vox, s, half, d):
    """P with P[row][3] moved to the f32 that puts the voxel's u_ref (row 0) or v_ref (row 1) closest to half + d, on the side
    of the half-integer `half` that d is on -> (P, achieved distance from `half`), or None"""
    target = half + d
    x, y, z = vox
    one = lambda Q: reference(Q[None], np.array([x]), np.array([y]), np.array([z]), s, 1, 1)
    _, _, _, u, v, p2 = one(P)
    c = (u if row == 0 else v)[0]
    if not (np.isfinite(c) and p2[0] > 0):
        return None
    Q = P.copy()
    Q[row, 3] = F(np.float64(P[row, 3]) + (target - np.float64(c)) * np.float64(p2[0]))
    ks = np.arange(-48, 49)
    cands = np.tile(Q, (len(ks), 1, 1))
    cands[:, row, 3] = step_f32(Q[row, 3], ks)
    _, _, _, uu, vv, _ = reference(cands, np.full(len(ks), x), np.full(len(ks), y), np.full(len(ks), z), s, 1, 1)
    got = (uu if row == 0 else vv).astype(np.float64)
    ok = np.sign(got - half) == np.sign(d) if d != 0 else np.ones(len(ks), bool)
    if not ok.any():
        return None
    err = np.where(ok, np.abs(got - target), np.inf)
    best = int(np.argmin(err))
    return cands[best], got[best] - half


def tie_distances(rng, c, delta):
    """distances from a half-integer: an exact tie, +-1..8 ulps of it, fractions of the view's radius up to 2 delta"""
    ulp = float(np.spacing(F(abs(c) + 1.0)))
    ds = 2 * ([0.0] + [sg * j * ulp for sg in (1, -1) for j in (1, 2, 3, 5, 8)])   # two in three within 8 ulps
    ds += [sg * f * delta for sg in (1, -1) for f in (0.3, 0.7, 0.95, 1.05, 1.5, 2.0)]
    return [ds[int(i)] for i in rng.permutation(len(ds))]


def near_tie_scene(rng, family, n_general, n_plane, N=192, W=640, H=480, far=False):
    """n_general random cameras (half of them close to the grid) with one chosen voxel near a tie, and n_plane cameras whose
    u depends on x alone (depth too), so that a whole x-plane of voxels shares one u_ref near a tie.  far: ties in u only, at
    u >= W / 4, with cameras whose projections reach across a wide image (there an ulp of u exceeds the classifier's 2^-10 pixel
    of slack, so a radius without its error terms misses a voxel's pixel)"""
    s = F(0.28 / N)
    sc = Scene(family, f"{family}-N{N}-{W}x{H}", (N, N, N), s, W, H, np.zeros((0, 3, 4), F))
    Ps, general, planes, corners = [], [], [], []
    dims = (N, N, N)
    while len(Ps) < n_general + n_plane:
        plane = len(Ps) >= n_general
        row = 0 if far else int(rng.integers(0, 2))
        n_side = W if row == 0 else H
        half = [-0.5, n_side - 0.5, float(rng.integers(1, n_side - 1)) + 0.5][int(rng.integers(0, 3))]
        if far:
            half = [W - 0.5, float(rng.integers(W // 4, W - 1)) + 0.5][int(rng.integers(0, 2))]
        vox = (int(rng.integers(0, N)), int(rng.integers(0, N)), int(rng.integers(0, N)))
        if plane:
            row = 0
            half = [-0.5, W - 0.5, float(rng.integers(1, W - 1)) + 0.5][int(rng.integers(0, 3))]
            a, g = rng.uniform(0.5, 4.0) * W / 0.28, rng.uniform(-2.0, 2.0)
            h = rng.uniform(0.02, 1.5) if rng.random() < 0.5 else rng.uniform(1.5, 6.0)
            b, c = rng.uniform(-0.5, 0.5, 2) * H / 0.28
            P = np.array([[0, a, 0, W / 2], [b, g * H / 2, c, h * H / 2], [0, g, 0, h]], F)
        else:
            P = random_camera(rng, 0.28, W, H, fit=far)
            if len(Ps) % 2 and not far:   # close to the grid: the depth term Cu |r| dominates the radius
                P = close_camera(rng, 0.28, W, H)
            P = centre_other(P, 1 - row, vox, s, (H if row == 0 else W) * rng.uniform(0.3, 0.7) + 0.25)
        Cu, Cv, hDu, hDv = filter_constants(P, dims, s, W, H)
        _, _, _, _, _, p2 = reference(P[None], np.array([vox[0]]), np.array([vox[1]]), np.array([vox[2]]), s, W, H)
        if not (p2[0] > 0) or not np.isfinite(Cu):
            continue
        delta = float((Cu if row == 0 else Cv) / p2[0] + (0.5 - (hDu if row == 0 else hDv)))
        d = tie_distances(rng, half, delta)[0]
        if far:   # exact ties and 1 - 3 ulps: where the corner projections' own rounding decides
            d = float(np.spacing(F(half))) * float(rng.choice([0, 1, -1, 2, -2, 3, -3]))
        r = place_tie(P, row, vox, s, half, d)
        if r is None:
            continue
        Ps.append(r[0])
        if plane:
            planes.append((len(Ps) - 1, vox))
        else:
            general.append((len(Ps) - 1, row, r[1], vox))
    sc.P = np.stack(Ps)
    for v, row, d, (x, y, z) in general:   # the chosen voxel, and boxes of each level with it as their extreme corner in u (v)
        sc.add_vox([v, x, y, z], near=True)
        for lv, (bx, by, bz) in LEVELS.items():
            if lv == "super" and rng.random() < 0.7:
                continue
            box = tie_box(sc, v, row, d, (x, y, z), (bx, by, bz))
            if box is not None:
                sc.add_boxes([v, *box])
    for v, (x, y, z) in planes:    # every voxel-view of the x-plane is a near-tie in u
        yy, zz = np.meshgrid(np.arange(0, N, 3), np.arange(0, N, 3))
        sc.add_vox(np.stack([np.full(yy.size, v), np.full(yy.size, x), yy.ravel(), zz.ravel()], 1), near=True)
        for lv in ("sub", "brick"):
            bx, by, bz = LEVELS[lv]
            for _ in range(2):
                y0, z0 = int(rng.integers(0, N - by)), int(rng.integers(0, N - bz))
                x0 = x if rng.random() < 0.5 else max(x - bx + 1, 0)
                sc.add_boxes([v, x0, y0, z0, min(x0 + bx, N) - 1, y0 + by - 1, z0 + bz - 1])
    sc.masks = blob_masks(rng, sc.V, W, H) if W * H < 1e6 else band_masks(rng, sc.V, W, H)
    sc.expect = {0, 1, 2, 3, 4}
    return sc


def centre_other(P, row, vox, s, c):
    """P with P[row][3] moved so that the voxel's coordinate of that row (u for 0, v for 1) lies near c: the other coordinate of
    a near-tie voxel inside the image, so that boxes around it can be decided"""
    _, _, _, u, v, p2 = reference(P[None], *(np.array([t]) for t in vox), s, 1, 1)
    cur = (u if row == 0 else v)[0]
    if not (np.isfinite(cur) and p2[0] > 0):
        return P
    Q = P.copy()
    Q[row, 3] = F(np.float64(P[row, 3]) + (c - np.float64(cur)) * np.float64(p2[0]))
    return Q


def tie_box(sc, v, row, d, vox, size):
    """a box of the given size with the voxel at one of its corners, oriented so that the voxel's coordinate (u for row 0, v for
    row 1) is the box's largest when the reference rounds it up (d >= 0, u_ref >= k + 1/2 with u > 0) and its smallest otherwise:
    the corner on which a rectangle too narrow by a rounding would miss the voxel's pixel -> (x0, y0, z0, x1, y1, z1) or None"""
    best = None
    for o in range(8):
        lo = [vox[k] if (o >> k) & 1 else vox[k] - size[k] + 1 for k in range(3)]
        dims = (sc.X, sc.Y, sc.Z)
        lo = [max(min(lo[k], dims[k] - size[k]), 0) for k in range(3)]
        hi = [min(lo[k] + size[k], dims[k]) - 1 for k in range(3)]
        c = np.array([[cx, cy, cz] for cx in (lo[0], hi[0]) for cy in (lo[1], hi[1]) for cz in (lo[2], hi[2])])
        _, _, _, u, w, _ = reference(np.broadcast_to(sc.P[v], (8, 3, 4)), c[:, 0], c[:, 1], c[:, 2], sc.s, sc.W, sc.H)
        cu = (u if row == 0 else w).astype(np.float64)
        _, _, _, u0, w0, _ = reference(sc.P[v][None], *(np.array([t]) for t in vox), sc.s, sc.W, sc.H)
        mine = float((u0 if row == 0 else w0)[0])
        if not np.all(np.isfinite(cu)):
            continue
        if (d >= 0 and mine >= cu.max()) or (d < 0 and mine <= cu.min()):
            return (*lo, *hi)
        best = best or (*lo, *hi)
    return best


def close_camera(rng, extent, W, H):
    """a camera 0.05 to 0.3 extents from the grid's centre, looking at it"""
    c = np.array([0.5, 0.5, -0.5]) * extent
    d = rng.normal(size=3); d /= np.linalg.norm(d)
    eye = c + d * extent * rng.uniform(0.6, 1.0)
    f = c - eye; f /= np.linalg.norm(f)
    upv = rng.normal(size=3); r = np.cross(f, upv); r /= np.linalg.norm(r); u = np.cross(f, r)
    R = np.stack([r, u, f]); t = -R @ eye
    fl = W * 10 ** rng.uniform(-0.5, 0.3)
    K = np.array([[fl, 0, W * rng.uniform(0.3, 0.7)], [0, fl, H * rng.uniform(0.3, 0.7)], [0, 0, 1]])
    M = np.concatenate([R, t[:, None]], 1)[:, [1, 0, 2, 3]]
    return (K.astype(F) @ M.astype(F)).astype(F)


# ---- the families ------------------------------------------------------------------------------------------------------------
def ordinary(rng, sc, n_boxes, n_vox, levels=("super", "brick", "sub"), weights=(0.12, 0.44, 0.44)):
    for lv, wgt in zip(levels, weights):
        sc.add_boxes(lattice_boxes(rng, sc, max(int(n_boxes * wgt), 1), lv))
    sc.add_vox(random_vox(rng, sc, n_vox))


def scenes(seed, scale=1.0):
    """every family's scenes for one seed; scale multiplies the numbers of boxes and voxel-views"""
    rng = np.random.default_rng(1000 + seed)
    nb = lambda n: max(int(n * scale), 8)
    out = []
    # random cameras from inside the grid to 20 extents away, grids of 100 to 2048 voxels; the first set of masks is replaced
    for k, (N, (W, H)) in enumerate([(100, (640, 480)), (512, (640, 480)), (1024, (3840, 2160)), (2048, (640, 480)), (300, (1920, 1080))]):
        V = 48 if W * H < 1e6 else 12
        sc = Scene("random", f"random-N{N}-{W}x{H}", (N, N, N), 0.28 / N, W, H, np.stack([random_camera(rng, 0.28, W, H) for _ in range(V)]))
        ordinary(rng, sc, nb(3000), nb(3_000_000))
        sc.masks = blob_masks(rng, V, W, H)
        if k % 2 == 0:
            sc.first_masks = blob_masks(rng, V, W, H)
        sc.expect = {0, 1, 2, 3, 4}
        out.append(sc)
    # anisotropic grids with cameras that stretch the long axis: an x / y swap shows only here
    for dims, col in (((2048, 16, 16), 1), ((16, 2048, 16), 0)):
        Ps = []
        for _ in range(32):
            P = random_camera(rng, 0.28, 640, 480).astype(np.float64)
            P[:, col] *= 24.0
            P[:, 1 - col] /= 24.0
            Ps.append(P.astype(F))
        sc = Scene("anisotropic", f"anisotropic-{dims[0]}x{dims[1]}x{dims[2]}", dims, 0.28 / 2048, 640, 480, np.stack(Ps))
        ordinary(rng, sc, nb(1500), nb(1_500_000), levels=("brick", "sub", "super"), weights=(0.45, 0.45, 0.1))
        sc.masks = blob_masks(rng, sc.V, 640, 480)
        sc.expect = {0, 1, 2, 3, 4}
        out.append(sc)
    # a z-slab that starts inside the grid
    sc = Scene("slab", "slab-256-z[100,200)", (256, 256, 256), 0.28 / 256, 640, 480,
               np.stack([random_camera(rng, 0.28, 640, 480) for _ in range(40)]), z0=100, z1=200)
    ordinary(rng, sc, nb(1500), nb(1_500_000))
    sc.masks = blob_masks(rng, sc.V, 640, 480)
    sc.expect = {0, 1, 2, 3, 4}
    out.append(sc)
    # ragged grid edges: every level clipped in x, y and z
    sc = Scene("ragged", "ragged-157x45x37-z[3,37)", (157, 45, 37), 0.28 / 157, 640, 480,
               np.stack([random_camera(rng, 0.28, 640, 480) for _ in range(40)]), z0=3, z1=37)
    ordinary(rng, sc, nb(1500), nb(1_000_000))
    sc.masks = blob_masks(rng, sc.V, 640, 480)
    sc.expect = {0, 1, 2, 3, 4}
    out.append(sc)
    # very wide and very tall images: random cameras whose projections reach across them, and dyadic tie cameras (every voxel
    # exactly on a pixel edge)
    for W, H in WIDE_TALL:
        n, big = max(W, H), W * H > 1e8   # 2^20 x 2046: 1 GB of mask words and 4 GB of table per view
        n_rand = 2 if big else 6
        Ps = [random_camera(rng, 24.0, W, H, fit=True) for _ in range(n_rand)]   # grid extent 96 x 0.25
        offs = (float(n // 2) + 0.5, float(n) - 100.5, -0.5 - 2 * 20, 0.5 + 1.0)
        Ps += [tie_camera(W, H, off) for off in (offs[:2] if big else offs)]
        sc = Scene("wide_tall", f"wide_tall-{W}x{H}", (96, 96, 96), 0.25, W, H, np.stack(Ps))
        ordinary(rng, sc, nb(600), nb(400_000), levels=("brick", "sub"), weights=(0.5, 0.5))
        tie_views = list(range(n_rand, len(Ps)))
        sc.add_boxes(lattice_boxes(rng, sc, nb(400), "sub", views=tie_views))
        sc.add_vox(random_vox(rng, sc, nb(200_000), views=tie_views))
        sc.masks = band_masks(rng, sc.V, W, H)
        sc.expect = {0, 1, 4} if n >= 1 << 20 else {0, 1, 2, 3, 4}
        out.append(sc)
    # constructed near-ties, in the image's interior and at both edges, for random, close and x-plane cameras
    out.append(near_tie_scene(rng, "near_tie", 1200, 40))
    out.append(near_tie_scene(rng, "near_tie", 600, 30, N=64, W=96, H=4000))
    out.append(near_tie_scene(rng, "near_tie", 1500, 0, N=64, W=65537, H=48, far=True))
    # depths near the classifier's 64 e2 cut-off and near 0
    out.append(depth_scene(rng, nb))
    # NaN, inf, 1e38 and denormal matrices
    out.append(hostile_scene(rng, nb))
    # rectangles of area 65 535, 65 536 and more, and one with exactly 65 536 background pixels in a larger one
    out.append(large_rect_scene())
    # more than 256 views: the views past 256 come from vc_append_views
    sc = Scene("many_views", "many_views-300", (200, 200, 200), 0.28 / 200, 320, 240,
               np.stack([random_camera(rng, 0.28, 320, 240) for _ in range(300)]))
    sc.add_boxes(lattice_boxes(rng, sc, nb(1200), "brick", views=range(250, 300)))
    sc.add_boxes(lattice_boxes(rng, sc, nb(600), "sub", views=range(256, 300)))
    sc.add_vox(random_vox(rng, sc, nb(1_000_000), views=range(240, 300)))
    sc.masks = blob_masks(rng, sc.V, 320, 240)
    sc.expect = {0, 1, 2, 3, 4}
    out.append(sc)
    return out


def depth_scene(rng, nb):
    """each view moves P[2][3] so that the smallest corner depth of one box is f * 64 e2 (f near 1), or a voxel's depth ~ 0"""
    N, W, H = 256, 640, 480
    s = F(0.28 / N)
    sc = Scene("depth", "depth-N256", (N, N, N), s, W, H, np.zeros((0, 3, 4), F))
    Ps, boxes = [], []
    for i in range(160):
        P = random_camera(rng, 0.28, W, H)
        lv = ("sub", "brick", "super")[i % 3]
        bx, by, bz = LEVELS[lv]
        lo = np.array([rng.integers(0, N - bx), rng.integers(0, N - by), rng.integers(0, N - bz)])
        hi = lo + np.array([bx, by, bz]) - 1
        cw = [np.array([F(lo[k]) * s, F(hi[k]) * s], F) for k in range(2)] + [np.array([F(-lo[2]) * s, F(-hi[2]) * s], F)]
        ax, ay, az = (float(np.max(np.abs(c))) for c in cw)
        aP = np.abs(P[2].astype(np.float64))
        if i % 4 == 3:   # depth through zero inside the box
            P[2, 3] = F(-(P[2, 0] * cw[1][0] + P[2, 1] * cw[0][0] + P[2, 2] * cw[2][0]) + rng.normal() * 1e-7)
        else:
            for _ in range(3):
                e2 = 2.6822092e-07 * (aP[3] + aP[2] * az + aP[0] * ay + aP[1] * ax)
                depths = [P[2, 0] * wy + P[2, 1] * wx + P[2, 2] * wz for wy in cw[1] for wx in cw[0] for wz in cw[2]]
                f = [0.98, 0.999, 1.0, 1.001, 1.02, 1.2][int(rng.integers(0, 6))]
                P[2, 3] = F(64.0 * e2 * f - min(depths))
                aP = np.abs(P[2].astype(np.float64))
        Ps.append(P)
        boxes.append([i, *lo, *hi])
    sc.P = np.stack(Ps)
    sc.add_boxes(boxes)
    sc.add_boxes(lattice_boxes(rng, sc, nb(600), "sub"))
    sc.add_vox(random_vox(rng, sc, nb(600_000)))
    for i, (_, x0, y0, z0, x1, y1, z1) in enumerate(boxes):   # the corners of each view's box
        sc.add_vox([[i, x, y, z] for x in (x0, x1) for y in (y0, y1) for z in (z0, z1)])
    sc.masks = blob_masks(rng, sc.V, W, H)
    sc.expect = {0, 1, 2, 3, 4}
    return sc


def hostile_scene(rng, nb):
    N, W, H = 128, 640, 480
    Ps = []
    specials = [np.nan, np.inf, -np.inf, 1e38, -1e38, 1e-40, -1e-42, 1e-45, 0.0]
    for i in range(64):
        P = random_camera(rng, 0.28, W, H)
        k = int(rng.integers(1, 4))
        for _ in range(k):
            P[rng.integers(0, 3), rng.integers(0, 4)] = F(specials[int(rng.integers(0, len(specials)))])
        if i % 8 == 0:
            P = (rng.normal(size=(3, 4)) * 1e-40).astype(F)   # every entry denormal
        if i % 8 == 1:
            P = np.full((3, 4), np.nan, F)
        Ps.append(P)
    sc = Scene("hostile", "hostile-N128", (N, N, N), 0.28 / N, W, H, np.stack(Ps))
    ordinary(rng, sc, nb(600), nb(300_000))
    sc.masks = blob_masks(rng, sc.V, W, H)
    sc.expect = {0}
    return sc


def large_rect_scene():
    """u = x + 0.25, v = y + 0.25 (dyadic voxel size 1/64, depth 1): a box of nx by ny voxels gets a rectangle of exactly nx ny
    pixels.  Views: all background, all foreground, and exactly 65 536 background pixels inside the 300 x 256 rectangle"""
    W, H = 640, 480
    P = np.array([[0, 64, 0, 0.25], [64, 0, 0, 0.25], [0, 0, 0, 1]], F)
    sc = Scene("large_rect", "large_rect-320x320x4", (320, 320, 4), 1.0 / 64, W, H, np.stack([P, P, P]))
    Ww = sc.Ww
    bg, fg = np.full((H, Ww), 0xFFFFFFFF, np.uint32), np.zeros((H, Ww), np.uint32)
    bg[:, -1] &= np.uint32((1 << (W % 32)) - 1) if W % 32 else np.uint32(0xFFFFFFFF)
    part = fg.copy()
    part[8:8 + 256, 0:8] = 0xFFFFFFFF                          # columns 0..255 of rows 8..263: 65 536 pixels
    sc.masks = np.stack([bg, fg, part])
    for v in range(3):
        for nx, ny in ((255, 257), (256, 256), (257, 256), (300, 256), (8, 8), (256, 255), (300, 300)):
            sc.add_boxes([v, 0, 8, 0, nx - 1, 8 + ny - 1, 3])
    sc.expect = {2, 3, 4}
    return sc


# ---- the checks ----------------------------------------------------------------------------------------------------------
def check_boxes(sc, res, oracle, log, fails):
    """res int32[n, 5] from the classifier (or its restatement) for sc.boxes"""
    codes = Counter()
    for b, r in zip(sc.boxes, res):
        v, x0, y0, z0, x1, y1, z1 = (int(t) for t in b)
        code, px0, px1, py0, py1 = (int(t) for t in r)
        codes[code] += 1
        if code == 0:
            continue
        all_in, none_in, qx0, qx1, qy0, qy1, _ = oracle.box_pixel_bounds(sc.P[v], (x0, y0, z0), (x1, y1, z1), sc.s, sc.W, sc.H,
                                                                          nthreads=0 if (x1 - x0 + 1) * (y1 - y0 + 1) * (z1 - z0 + 1) > 20000 else 1)
        what = f"{sc.name}: box {b.tolist()} code {code} rect {(px0, px1, py0, py1)}"
        if code == 1:
            if not none_in:
                fails.append(f"{what}: some voxel is inside the image")
            continue
        if not all_in:
            fails.append(f"{what}: some voxel is outside the image")
            continue
        if not (px0 <= qx0 and qx1 <= px1 and py0 <= qy0 and qy1 <= py1):
            fails.append(f"{what}: the voxels' pixels span {(qx0, qx1, qy0, qy1)}")
        if not (px0 >= qx0 - 1 and px1 <= qx1 + 1 and py0 >= qy0 - 1 and py1 <= qy1 + 1):
            fails.append(f"{what}: more than a pixel wider than the voxels' pixels {(qx0, qx1, qy0, qy1)}")
        area = (px1 - px0 + 1) * (py1 - py0 + 1)
        if area >= 1 << 16:
            if code != 4:
                fails.append(f"{what}: area {area} >= 2^16 but code {code}")
            continue
        bg = bg_count(sc.masks[v], px0, px1, py0, py1)
        want = 3 if bg == area else 2 if bg == 0 else 4
        if code != want:
            fails.append(f"{what}: {bg} background pixels of {area}, want code {want}")
    log[sc.family]["codes"].update(codes)
    return codes


def check_voxels(sc, res, log, fails, oracle=None, rng=None):
    """res int32[n, 11] from the filter (or its restatement) for sc.vox; -> the decided mask"""
    v, x, y, z = (sc.vox[:, k] for k in range(4))
    px, py, ins, u, w, p2 = reference(sc.P[v], x, y, z, sc.s, sc.W, sc.H)
    dec, fin, fpx, fpy, ein, epx, epy = (res[:, k] for k in range(7))
    dec, fin, ein = dec.astype(bool), fin.astype(bool), ein.astype(bool)
    name = sc.name

    def report(bad, what):
        if bad.any():
            i = np.flatnonzero(bad)[:5]
            fails.append(f"{name}: {int(bad.sum())} voxel-views {what}, e.g. (view, x, y, z) {sc.vox[i].tolist()}")

    # the exact path is the reference
    report(ein != ins, "with the exact path's inside test wrong")
    report(ins & ((epx != px) | (epy != py)), "with the exact path's pixel wrong")
    # decided => the reference's answer
    report(dec & (fin != ins), "decided with the wrong inside test")
    report(dec & ins & ((fpx != px) | (fpy != py)), "decided with the wrong pixel")
    # undecided, finite and well conditioned => within twice the radius of a pixel edge
    Cu, Cv, hDu, hDv = (res[:, k].view(F) for k in range(7, 11))
    with np.errstate(all="ignore"):
        # |1/q2| of the filter, bounded through |q2 - p2| <= eta_2 <= Cu / (W + 3) (vc_filter_constants); depths within that
        # bound of 0 are not well conditioned
        eta2 = np.minimum(Cu.astype(np.float64) / (sc.W + 3.0), Cv.astype(np.float64) / (sc.H + 3.0))
        ar = 1.0 / (np.abs(p2.astype(np.float64)) - eta2)
        du = 2 * (Cu.astype(np.float64) * ar + (0.5 - hDu.astype(np.float64)))
        dv = 2 * (Cv.astype(np.float64) * ar + (0.5 - hDv.astype(np.float64)))
        eu = np.abs(u.astype(np.float64) - (np.floor(u.astype(np.float64)) + 0.5))
        ev = np.abs(w.astype(np.float64) - (np.floor(w.astype(np.float64)) + 0.5))
        # (the radius Cu |r| + D bounds |u~ - u_ref| for |u| <= W + 2 only; further out the filter need not decide)
        good = np.isfinite(u) & np.isfinite(w) & (np.abs(u) <= sc.W + 2) & (np.abs(w) <= sc.H + 2) & np.isfinite(Cu) & np.isfinite(Cv) \
            & np.isfinite(p2) & (ar > 0)
        report(~dec & good & ~((eu <= du) | (ev <= dv)), "undecided although u_ref and v_ref are further than 2 delta from a pixel edge")
    if oracle is not None:   # spot checks of the numpy reference against the C oracle
        for i in rng.choice(len(v), min(len(v), 40), replace=False):
            ok, opx, opy, _ = oracle.pixel_of(sc.P[v[i]], int(x[i]), int(y[i]), int(z[i]), sc.s, sc.W, sc.H)
            if bool(ok) != bool(ins[i]) or (ok and (opx, opy) != (int(px[i]), int(py[i]))):
                fails.append(f"{name}: numpy reference and oracle disagree at {sc.vox[i].tolist()}")
    L = log[sc.family]
    L["voxel_views"] += len(v); L["decided"] += int(dec.sum()); L["near"] += int(sc.near.sum())
    L["near_decided"] += int((dec & sc.near).sum())
    return dec


def check_constants(sc, res, fails):
    """Cu, Cv of every view and hDu, hDv bitwise equal to the numpy restatement of vc_filter_constants"""
    seen = {}
    for r, vw in zip(res, sc.vox[:, 0]):
        seen.setdefault(int(vw), r[7:11])
    for vw, r in seen.items():
        want = np.array(filter_constants(sc.P[vw], (sc.X, sc.Y, sc.Z), sc.s, sc.W, sc.H), F).view(np.int32)
        if not np.array_equal(r, want):
            fails.append(f"{sc.name}: view {vw} filter constants {r.view(F).tolist()}, want {want.view(F).tolist()}")


# ---- the numpy restatement as a probe (CPU) ------------------------------------------------------------------------------
class Restatement:
    """probe_boxes / probe_voxels of test_classifier_math's restatement; zero_radius: Eu = Ev = 0, Cu = Cv = 0, hD = 0.5"""
    def __init__(self, sc, zero_radius):
        self.sc, self.zero = sc, zero_radius

    def probe_boxes(self, boxes):
        sc, out = self.sc, np.zeros((len(boxes), 5), np.int32)
        for i, (v, x0, y0, z0, x1, y1, z1) in enumerate(boxes):
            r = rect_of_box(sc.P[v], np.array([x0, y0, z0]), np.array([x1, y1, z1]), sc.s, sc.W, sc.H, zero_radius=self.zero)
            if r[0] == 4:
                _, a, b, c, d = r
                area = (b - a + 1) * (d - c + 1)
                bg = bg_count(sc.masks[v], a, b, c, d) if area < 1 << 16 else -1
                out[i] = (3 if bg == area else 2 if bg == 0 else 4, a, b, c, d)
            else:
                out[i, 0] = r[0]
        return out

    def probe_voxels(self, vox):
        sc, out = self.sc, np.zeros((len(vox), 11), np.int32)
        for vw in np.unique(vox[:, 0]):
            m = vox[:, 0] == vw
            c = filter_constants(sc.P[vw], (sc.X, sc.Y, sc.Z), sc.s, sc.W, sc.H) if not self.zero else (F(0), F(0), F(0.5), F(0.5))
            dec, px, py, ins = filter_pixels(sc.P[vw], vox[m, 1], vox[m, 2], vox[m, 3], sc.s, sc.W, sc.H, c)
            epx, epy, ein, _, _, _ = reference(np.broadcast_to(sc.P[vw], (int(m.sum()), 3, 4)), vox[m, 1], vox[m, 2], vox[m, 3], sc.s, sc.W, sc.H)
            out[m, 0], out[m, 1], out[m, 2], out[m, 3] = dec, ins, px, py
            out[m, 4], out[m, 5], out[m, 6] = ein, np.where(ein, epx, 0), np.where(ein, epy, 0)
            out[m, 7:11] = np.array(c, F).view(np.int32)
        return out


# ---- tests -----------------------------------------------------------------------------------------------------------------
def test_box_pixel_bounds_equal_pixel_of(oracle):
    rng = np.random.default_rng(5)
    for trial in range(40):
        N = int(rng.choice([16, 100, 512])); s = F(0.28 / N); W, H = (640, 480) if trial % 2 else (96, 4000)
        P = random_camera(rng, 0.28, W, H) if trial % 5 else close_camera(rng, 0.28, W, H)
        if trial % 7 == 0:
            P[2, 3] = F(np.nan)
        lo = rng.integers(0, N - 6, 3); hi = lo + rng.integers(0, 6, 3)
        got = oracle.box_pixel_bounds(P, lo, hi, s, W, H, nthreads=1 + trial % 3)
        g = [a.ravel() for a in np.meshgrid(*(np.arange(lo[k], hi[k] + 1) for k in range(3)), indexing="ij")]
        ins, pxs, pys, bad = [], [], [], False
        for x, y, z in zip(*g):
            ok, px, py, _ = oracle.pixel_of(P, int(x), int(y), int(z), s, W, H)
            ins.append(ok); pxs.append(px); pys.append(py)
            p = oracle.project(P, np.array([F(y) * s, F(x) * s, F(-int(z)) * s, 1], F))
            bad |= not (p[2] > 0 and np.isfinite(p[2]))
        assert got == (all(ins), not any(ins), min(pxs), max(pxs), min(pys), max(pys), bad), (trial, got)


def _power_cases():
    """the CPU-sized subset of the sampled families: near-ties, depth cut-offs, ragged edges"""
    rng = np.random.default_rng(77)
    out = [near_tie_scene(rng, "near_tie", 400, 6, N=64)]
    rng2 = np.random.default_rng(78)
    out.append(depth_scene(rng2, lambda n: max(int(n * 0.005), 8)))
    return out


def test_sampling_reaches_the_radius(oracle):
    """the numpy restatement with zero radii fails the soundness checks on the sampled cases, and with its radii passes them"""
    n_fail = Counter()
    for sc in _power_cases():
        for zero in (True, False):
            log, fails = defaultdict(lambda: defaultdict(int)), []
            log[sc.family]["codes"] = Counter()
            probe = Restatement(sc, zero)
            check_boxes(sc, probe.probe_boxes(sc.boxes), oracle, log, fails)
            box_fails = len(fails)
            check_voxels(sc, probe.probe_voxels(sc.vox), log, fails)
            if zero:
                n_fail["boxes"] += box_fails
                n_fail["voxel check"] += len(fails) - box_fails
            else:
                # the restatement with its radii is sound (its pixel arithmetic stands in for the kernel's; the exact-path
                # entries are the reference itself)
                assert not fails, (sc.name, fails[:6])
    assert n_fail["boxes"] >= 3 and n_fail["voxel check"] >= 1, n_fail


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


def _engine(A, sc):
    e = A.VoxelEngine(sc.X, sc.Y, sc.Z, sc.s, z_begin=sc.z0, z_end=sc.z1)
    k = min(sc.V, 256)
    e.set_views(sc.P[:k].reshape(-1, 12), sc.W, sc.H)
    if sc.first_masks is not None:
        e.set_masks_bits(sc.first_masks[:k])
    e.set_masks_bits(sc.masks[:k])
    if sc.V > k:
        e.append_views(sc.P[k:].reshape(-1, 12), mask_bits=sc.masks[k:])
    return e


def _table(log):
    lines = [f"{'family':12s} {'code0':>7s} {'code1':>7s} {'code2':>7s} {'code3':>7s} {'code4':>7s} {'voxel-views':>12s} {'decided':>10s} "
             f"{'undecided':>10s} {'near-ties':>10s} {'near dec.':>10s}"]
    for fam, L in log.items():
        c = L["codes"]
        lines.append(f"{fam:12s} " + " ".join(f"{c.get(k, 0):7d}" for k in range(5)) +
                     f" {L['voxel_views']:12d} {L['decided']:10d} {L['voxel_views'] - L['decided']:10d} {L['near']:10d} {L['near_decided']:10d}")
    return "\n".join(lines)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(int(os.environ.get("VC_PROBE_SEEDS", "1"))))
def test_classifier_and_filter_against_the_reference(A, oracle, seed):
    rng = np.random.default_rng(seed)
    log, fails = defaultdict(lambda: defaultdict(int)), []
    n_boxes = n_super = 0
    for sc in scenes(seed):
        log[sc.family].setdefault("codes", Counter())
        with _engine(A, sc) as e:
            codes = check_boxes(sc, e.probe_boxes(sc.boxes), oracle, log, fails)
            res = e.probe_voxels(sc.vox)
        n_boxes += len(sc.boxes)
        n_super += int(((sc.boxes[:, 4] - sc.boxes[:, 1]) >= 64).sum())
        dec = check_voxels(sc, res, log, fails, oracle, rng)
        check_constants(sc, res, fails)
        log[sc.family]["expect"] = log[sc.family].get("expect", set()) | sc.expect
        if sc.family in ("random", "anisotropic", "slab", "ragged", "many_views"):
            if not dec.mean() > 0.5:
                fails.append(f"{sc.name}: the filter decides only {dec.mean():.3f} of the voxel-views")
    for fam, L in log.items():
        missing = L["expect"] - set(L["codes"])
        if missing:
            fails.append(f"{fam}: classifier codes {sorted(missing)} never occurred")
    tot = sum(L["voxel_views"] for L in log.values())
    near = sum(L["near"] for L in log.values())
    print(f"\nseed {seed}: {n_boxes} (box, view) cases, {n_super} of them super-bricks; {tot} voxel-views, {near} constructed near-ties")
    print(_table(log))
    assert n_boxes >= 20000 and n_super >= 2000 and tot >= 20_000_000 and near >= 100_000, (n_boxes, n_super, tot, near)
    assert not fails, f"{len(fails)} failures:\n" + "\n".join(fails[:40])


@pytest.mark.gpu
def test_probe_refusals(A):
    from ar_voxel_project_b200 import _lib as L
    with A.VoxelEngine(40, 30, 20, 0.01, z_begin=5, z_end=15) as e:
        box = np.array([[0, 0, 0, 5, 7, 7, 12]], np.int32)
        vox = np.array([[0, 1, 2, 5]], np.int32)
        for f, a in ((e.probe_boxes, box), (e.probe_voxels, vox)):
            with pytest.raises(A.VoxCarveError) as ei:
                f(a)
            assert ei.value.code == L.VC_ERR_STATE
        P = random_camera(np.random.default_rng(0), 0.4, 64, 48)
        e.set_views(np.stack([P, P]).reshape(-1, 12), 64, 48)
        for f, a in ((e.probe_boxes, box), (e.probe_voxels, vox)):   # views but no masks
            with pytest.raises(A.VoxCarveError) as ei:
                f(a)
            assert ei.value.code == L.VC_ERR_STATE
        e.set_masks_bits(np.zeros((2, 48, 2), np.uint32))
        assert e.probe_boxes(box).shape == (1, 5) and e.probe_voxels(vox).shape == (1, 11)
        bad_boxes = [[2, 0, 0, 5, 7, 7, 12], [-1, 0, 0, 5, 7, 7, 12], [0, -1, 0, 5, 7, 7, 12], [0, 0, 0, 5, 40, 7, 12],
                     [0, 0, 0, 4, 7, 7, 12], [0, 0, 0, 5, 7, 7, 15], [0, 5, 0, 5, 4, 7, 12], [0, 0, 3, 5, 7, 2, 12],
                     [0, 0, 0, 9, 7, 7, 8], [0, 0, 0, 5, 7, 30, 12]]
        bad_vox = [[2, 1, 2, 5], [-1, 1, 2, 5], [0, 40, 2, 5], [0, -1, 2, 5], [0, 1, 30, 5], [0, 1, 2, 4], [0, 1, 2, 15]]
        out5, out11 = np.full((2, 5), 7, np.int32), np.full((2, 11), 7, np.int32)
        for b in bad_boxes:   # a refused record anywhere in the list: nothing written
            two = np.array([box[0], b], np.int32)
            assert e._lib.vc_probe_boxes(e._h, 2, two.ctypes.data, out5.ctypes.data) == L.VC_ERR_ARG, b
            assert (out5 == 7).all()
        for b in bad_vox:
            two = np.array([vox[0], b], np.int32)
            assert e._lib.vc_probe_voxels(e._h, 2, two.ctypes.data, out11.ctypes.data) == L.VC_ERR_ARG, b
            assert (out11 == 7).all()
        assert e._lib.vc_probe_boxes(e._h, 1, None, out5.ctypes.data) == L.VC_ERR_ARG
        assert e._lib.vc_probe_voxels(e._h, 1, vox.ctypes.data, None) == L.VC_ERR_ARG
        assert e._lib.vc_probe_boxes(e._h, (1 << 26) + 1, box.ctypes.data, out5.ctypes.data) == L.VC_ERR_ARG
        assert e._lib.vc_probe_boxes(e._h, 0, None, None) == L.VC_OK
