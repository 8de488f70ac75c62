"""The error-radius argument behind the conservative (brick, view) classifier, checked on the CPU under far more hostile sampling
than the GPU parity tests can afford.

`rect_of_box` restates `vc_classify_brick_view` (ar_voxel_project_b200/csrc/vc_kernels.cuh: f32 corner projections with an
approximate reciprocal, error radii in f32, the widened rectangle) in numpy float32; `reference_pixels` restates the reference
arithmetic (DESIGN.md section 2; checked below against the C oracle voxel by voxel).  Property: whenever the classifier does
not answer "undecided", the reference pixel of EVERY voxel of the box lies inside the rectangle it hands to the SAT
(codes 2/3/4), respectively outside the image (code 1).  The restatement is test infrastructure, like oracle/."""
import numpy as np
import pytest

F = np.float32


def fma32(a, b, c):
    """f32 FMA emulated through f64 (the product of two f32 is exact in f64; the sum is rounded twice: at most 1 ulp instead of 1/2,
    far inside the slack of the radius under test)"""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F)


def reference_pixels(P, xs, ys, zs, s, W, H):
    """(px, py, inside) of voxels as VoxelCarving.cpp:18-21,44-45 computes them: f32 world coordinates, f64 sequential accumulation,
    one rounding to f32, IEEE f32 divides, round half away from zero"""
    w = [(ys.astype(F) * s).astype(np.float64), (xs.astype(F) * s).astype(np.float64), ((-zs).astype(F) * s).astype(np.float64)]
    Pd = P.astype(np.float64)
    proj = [((((Pd[i, 0] * w[0]) + (Pd[i, 1] * w[1])) + (Pd[i, 2] * w[2])) + Pd[i, 3]).astype(F) for i in range(3)]
    with np.errstate(all="ignore"):
        u = (proj[0] / proj[2]).astype(np.float64)
        v = (proj[1] / proj[2]).astype(np.float64)
        px = np.where(u >= 0, np.floor(u + 0.5), -np.floor(-u + 0.5))
        py = np.where(v >= 0, np.floor(v + 0.5), -np.floor(-v + 0.5))
    ok = np.isfinite(px) & np.isfinite(py)
    inside = ok & (px >= 0) & (px < W) & (py >= 0) & (py < H)
    return px, py, inside


def rect_of_box(P, lo, hi, s, W, H):
    """-> (code, px0, px1, py0, py1): code 0 = undecided, 1 = all outside, 4 = all inside with the pixel rectangle"""
    Pf = P.astype(F)
    cw = [np.array([F(lo[k]) * s, F(hi[k]) * s], F) for k in range(3)]         # voxel index -> f32 world (x, y, z); z negated below
    cw[2] = np.array([F(-lo[2]) * s, F(-hi[2]) * s], F)
    wx, wy, wz = cw
    ax, ay, az = (F(np.max(np.abs(c))) for c in (wx, wy, wz))
    us, vs, ds = [], [], []
    for cy in range(2):
        for cx in range(2):
            X = [fma32(Pf[i, 1:2], wx[cx:cx + 1], Pf[i, 3:4]) for i in range(3)]
            Y = [fma32(Pf[i, 0:1], wy[cy:cy + 1], X[i]) for i in range(3)]
            for cz in range(2):
                q = [fma32(Pf[i, 2:3], wz[cz:cz + 1], Y[i])[0] for i in range(3)]
                with np.errstate(all="ignore"):
                    r = F(1.0) / q[2]                                             # rcp.approx: <= 1 ulp, inside the slack
                    us.append(F(q[0] * r)); vs.append(F(q[1] * r)); ds.append(q[2])
    us, vs, ds = np.array(us, F), np.array(vs, F), np.array(ds, F)
    if not (np.all(np.abs(us) < 3.0e38) and np.all(np.abs(vs) < 3.0e38)):
        return (0,)
    npos = int(np.sum(ds > 0))
    if npos not in (0, 8):
        return (0,)
    k = F(2.6822092e-07)
    aP = np.abs(Pf)
    e = [F(k * F(F(F(aP[i, 0] * ay) + F(aP[i, 1] * ax)) + F(aP[i, 2] * az) + aP[i, 3])) for i in range(3)]
    dmin = F(np.min(np.abs(ds)))
    if not (dmin > F(64.0) * e[2]) or not (dmin < F(1.0e30)):
        return (0,)
    U = F(max(abs(us.min()), abs(us.max())) + F(1.0)); V = F(max(abs(vs.min()), abs(vs.max())) + F(1.0))
    rd = F(F(1.12) / dmin)
    Eu = F(F(3.0) * F(F(F(e[0] + F(U * e[2])) * rd) + F(U * F(2.3841858e-07))) + F(9.765625e-04))
    Ev = F(F(3.0) * F(F(F(e[1] + F(V * e[2])) * rd) + F(V * F(2.3841858e-07))) + F(9.765625e-04))
    if not (Eu < F(0.25) and Ev < F(0.25)):
        return (0,)
    down = lambda a: np.nextafter(F(a), F(-np.inf)); up = lambda a: np.nextafter(F(a), F(np.inf))   # at least as wide as __fadd_rd / _ru
    lo_u, hi_u, lo_v, hi_v = down(us.min() - Eu), up(us.max() + Eu), down(vs.min() - Ev), up(vs.max() + Ev)
    Wm, Hm = F(W) - F(0.5), F(H) - F(0.5)
    if hi_u < F(-0.5) or lo_u >= Wm or hi_v < F(-0.5) or lo_v >= Hm:
        return (1,)
    if not (lo_u > F(-0.5) and hi_u < Wm and lo_v > F(-0.5) and hi_v < Hm):
        return (0,)
    fl = lambda c: int(np.floor(np.float64(c) + 0.5))
    return (4, fl(lo_u), fl(hi_u), fl(lo_v), fl(hi_v))


def random_camera(rng, extent, W, H, fit=False):
    """P = K [R | t] in f32 looking roughly at the grid from a random place - from inside the grid to twenty extents away.
    fit: the vertical focal length scales with H instead of W, so that projections reach across very wide or very tall images"""
    c = np.array([0.5, 0.5, -0.5]) * extent
    d = rng.normal(size=3); d /= np.linalg.norm(d)
    dist = extent * 10 ** rng.uniform(-1.0, 1.3)
    eye = c + d * dist + rng.normal(size=3) * extent * 0.2
    f = c + rng.normal(size=3) * extent * 0.3 - eye; f /= np.linalg.norm(f)
    upv = rng.normal(size=3); r = np.cross(f, upv); r /= np.linalg.norm(r); u = np.cross(f, r)
    R = np.stack([r, u, f]); t = -R @ eye
    fl = W * 10 ** rng.uniform(-0.5, 1.0)
    K = np.array([[fl, 0, W * rng.uniform(0.2, 0.8)], [0, fl * rng.uniform(0.8, 1.25) * (H / W if fit else 1.0), H * rng.uniform(0.2, 0.8)], [0, 0, 1]])
    M = np.concatenate([R, t[:, None]], 1)[:, [1, 0, 2, 3]]   # world = (y s, x s, -z s): columns 0 and 1 act on (wy, wx) like the product's P
    return (K.astype(F) @ M.astype(F)).astype(F)


# images at the ends of the accepted sizes: a long side of 2^16 + 1 and of 2^20 (where f32 pixel coordinates have an ulp of 1/8)
WIDE_TALL = [(65537, 48), (1 << 20, 2046), (48, 1 << 20)]


def tie_camera(W, H, offset):
    """dyadic camera for voxel size 0.25: along the long side the coordinate is 2i + offset (i = x for a wide image, y for a tall
    one), the other one 24.5 - 2z; with offset = k + 0.5 every voxel lies exactly on a pixel edge"""
    if W >= H:
        return np.array([[0, 8, 0, offset], [0, 0, 8, 24.5], [0, 0, 0, 1]], F)
    return np.array([[0, 0, 8, 24.5], [8, 0, 0, offset], [0, 0, 0, 1]], F)


def tie_offsets(W, H):
    n = max(W, H)
    return [float(n // 2) + 0.5, float(n) - 100.5]   # |c| > 2^19 for a side of 2^20; the far edge c = n - 0.5 (rounds to n: outside)


def test_reference_pixels_equal_the_oracle(oracle):
    rng = np.random.default_rng(3)
    for _ in range(6):
        N = int(rng.choice([64, 300, 1024])); s = F(0.28 / N); W, H = 640, 480
        P = random_camera(rng, 0.28, W, H)
        xs, ys, zs = (rng.integers(0, N, 200) for _ in range(3))
        px, py, inside = reference_pixels(P, xs, ys, zs, s, W, H)
        for i in range(len(xs)):
            ok, opx, opy, _ = oracle.pixel_of(P, int(xs[i]), int(ys[i]), int(zs[i]), s, W, H)
            assert bool(ok) == bool(inside[i])
            if ok:
                assert (opx, opy) == (int(px[i]), int(py[i]))
    for W, H in WIDE_TALL:   # exact ties far from the origin round half away from zero, in the restatement and the oracle alike
        for off in tie_offsets(W, H):
            P = tie_camera(W, H, off)
            i = np.arange(0, 96)
            z = np.arange(0, 30)
            ii, zz = (a.ravel() for a in np.meshgrid(i, z))
            xs, ys = (ii, np.zeros_like(ii)) if W >= H else (np.zeros_like(ii), ii)
            px, py, inside = reference_pixels(P, xs, ys, zz, F(0.25), W, H)
            along = px if W >= H else py
            assert np.array_equal(along, 2 * ii + off + 0.5)
            for k in range(0, len(ii), 7):
                ok, opx, opy, _ = oracle.pixel_of(P, int(xs[k]), int(ys[k]), int(zz[k]), F(0.25), W, H)
                assert bool(ok) == bool(inside[k])
                if ok:
                    assert (opx, opy) == (int(px[k]), int(py[k]))


def check_rectangle(P, lo, hi, s, W, H):
    """rect_of_box's answer for the box [lo, hi] holds for every voxel in it; -> its code"""
    res = rect_of_box(P, lo, hi, s, W, H)
    if res[0] == 0:
        return 0
    g = np.meshgrid(np.arange(lo[0], hi[0] + 1), np.arange(lo[1], hi[1] + 1), np.arange(lo[2], hi[2] + 1), indexing="ij")
    px, py, inside = reference_pixels(P, g[0].ravel(), g[1].ravel(), g[2].ravel(), s, W, H)
    if res[0] == 1:
        assert not inside.any()
    else:
        _, x0, x1, y0, y1 = res
        assert inside.all()
        assert px.min() >= x0 and px.max() <= x1 and py.min() >= y0 and py.max() <= y1
    return res[0]


@pytest.mark.parametrize("box", [(128, 32, 32), (32, 8, 8), (8, 8, 8), (8, 4, 4)])
def test_rectangle_contains_every_voxel_pixel(box):
    rng = np.random.default_rng(sum(box))
    decided = outside = 0
    for trial in range(700):
        N = int(rng.choice([100, 512, 1024, 2048])); s = F(0.28 / N)
        W, H = (640, 480) if trial % 3 else (3840, 2160)
        P = random_camera(rng, 0.28, W, H)
        lo = np.array([rng.integers(0, max(N - box[k], 1)) for k in range(3)])
        hi = np.minimum(lo + np.array(box) - 1, N - 1)
        code = check_rectangle(P, lo, hi, s, W, H)
        outside += code == 1
        decided += code == 4
    assert decided > 50 and outside > 20   # the sampling exercises both answers
    # very wide and very tall images, with cameras whose projections reach across them
    for W, H in WIDE_TALL:
        codes = []
        for trial in range(150):
            N = int(rng.choice([100, 512, 1024, 2048])); s = F(0.28 / N)
            P = random_camera(rng, 0.28, W, H, fit=True)
            lo = np.array([rng.integers(0, max(N - box[k], 1)) for k in range(3)])
            codes.append(check_rectangle(P, lo, np.minimum(lo + np.array(box) - 1, N - 1), s, W, H))
        # at a side of 2^20 the corner-projection radius exceeds its 1/4 pixel cap and every box stays undecided today (the
        # check still guards a finer radius); at 2^16 + 1 both answers occur
        if max(W, H) < 1 << 20:
            assert codes.count(4) >= 5 and codes.count(1) >= 5, (W, H, codes.count(4), codes.count(1))
        for off in tie_offsets(W, H):   # boxes whose voxels all lie on pixel edges, in the middle and across the far edge
            P = tie_camera(W, H, off)
            for i0 in (0, 40, 47, 50, 60):
                lo = np.array([i0, 0, 3]) if W >= H else np.array([0, i0, 3])
                check_rectangle(P, lo, lo + (np.array(box) - 1) // 4, F(0.25), W, H)


def filter_constants(P, dims, s, W, H):
    """vc_filter_constants (voxcarve.cu): radius coefficients Cu, Cv of a view and the thresholds 0.5 - D, all rounded outwards"""
    up = 1.0 + 2.0 ** -22
    ax, ay, az = ((d - 1) * float(s) * up for d in dims)
    eta = []
    for i in range(3):
        T = abs(float(P[i, 0])) * ay + abs(float(P[i, 1])) * ax + abs(float(P[i, 2])) * az + abs(float(P[i, 3]))
        eta.append(4.0 * 2.0 ** -24 * T * (1.0 + 2.0 ** -19) + 2.0 ** -100)
    W3, H3 = W + 3.0, H + 3.0
    Cu = np.nextafter(F((eta[0] + W3 * eta[2]) * (1.0 + 2.0 ** -19)), F(np.inf))
    Cv = np.nextafter(F((eta[1] + H3 * eta[2]) * (1.0 + 2.0 ** -19)), F(np.inf))
    hDu = np.nextafter(F(0.5 - (W3 * 2.0 ** -22 * (1.0 + 2.0 ** -10) + 2.0 ** -20)), F(-np.inf))
    hDv = np.nextafter(F(0.5 - (H3 * 2.0 ** -22 * (1.0 + 2.0 ** -10) + 2.0 ** -20)), F(-np.inf))
    return Cu, Cv, hDu, hDv


def filter_pixels(P, xs, ys, zs, s, W, H, consts):
    """vc_filter_pixel (vc_kernels.cuh) for arrays of voxels: (decided, px, py, inside) from three f32 FMAs per coordinate, an
    approximate reciprocal and the 1.5 * 2^23 rounding trick"""
    Cu, Cv, hDu, hDv = consts
    Pf = P.astype(F)
    wx, wy, wz = (xs.astype(F) * s).astype(F), (ys.astype(F) * s).astype(F), ((-zs).astype(F) * s).astype(F)
    q = [fma32(np.broadcast_to(Pf[i, 2], wz.shape), wz, fma32(np.broadcast_to(Pf[i, 0], wy.shape), wy,
         fma32(np.broadcast_to(Pf[i, 1], wx.shape), wx, np.broadcast_to(Pf[i, 3], wx.shape)))) for i in range(3)]
    magic = F(12582912.0)
    with np.errstate(all="ignore"):
        r = (F(1.0) / q[2]).astype(F)
        ar = np.abs(r)
        out = []
        for qi, C, hD, n in ((q[0], Cu, hDu, W), (q[1], Cv, hDv, H)):
            h = fma32(np.broadcast_to(-C, ar.shape), ar, np.broadcast_to(hD, ar.shape))
            m = fma32(qi, r, np.broadcast_to(magic, r.shape))
            d = fma32(qi, r, -(m - magic).astype(F))
            idx = m.view(np.int32).astype(np.int64) - 0x4B400000
            out.append((np.abs(d) < h, idx, (idx >= 0) & (idx < n)))
    return out[0][0] & out[1][0], out[0][1], out[1][1], out[0][2] & out[1][2]


def test_filter_decisions_are_the_reference_pixels():
    """decided => (pixel, inside) equal the reference's: 3 M voxel-views over random cameras (a zero radius fails this test)"""
    rng = np.random.default_rng(11)
    n_decided = n_total = 0
    for trial in range(150):
        N = int(rng.choice([100, 512, 1024, 2048])); s = F(0.28 / N)
        W, H = (640, 480) if trial % 3 else (3840, 2160)
        P = random_camera(rng, 0.28, W, H)
        xs, ys, zs = (rng.integers(0, N, 20000) for _ in range(3))
        dec = check_filter(P, xs, ys, zs, (N, N, N), s, W, H)
        n_total += dec.size; n_decided += int(dec.sum())
    assert n_decided > 0.5 * n_total   # the filter decides most voxel-views (it is switched off only for degenerate views)
    # very wide and very tall images.  The radius grows with the image size: at a side of 2^20 the threshold 0.5 - D is about
    # 1/4 and the view's term Cu |r| at least as large, so nothing is decided there today; the check guards a finer radius.
    for W, H in WIDE_TALL:
        n_decided = n_total = 0
        for trial in range(50):
            N = int(rng.choice([100, 512, 1024, 2048])); s = F(0.28 / N)
            P = random_camera(rng, 0.28, W, H, fit=True)
            xs, ys, zs = (rng.integers(0, N, 20000) for _ in range(3))
            dec = check_filter(P, xs, ys, zs, (N, N, N), s, W, H)
            n_total += dec.size; n_decided += int(dec.sum())
        if max(W, H) < 1 << 20:
            assert n_decided > 0.3 * n_total, (W, H, n_decided, n_total)
        for off in tie_offsets(W, H):   # every voxel exactly on a pixel edge
            i, z = (a.ravel() for a in np.meshgrid(np.arange(96), np.arange(30)))
            xs, ys = (i, np.zeros_like(i)) if W >= H else (np.zeros_like(i), i)
            check_filter(tie_camera(W, H, off), xs, ys, z, (96, 96, 30), F(0.25), W, H)


def check_filter(P, xs, ys, zs, dims, s, W, H):
    """every voxel-view the filter decides has the reference's pixel and inside test; -> the decided mask"""
    consts = filter_constants(P, dims, s, W, H)
    dec, px, py, ins = filter_pixels(P, xs, ys, zs, s, W, H, consts)
    rpx, rpy, rin = reference_pixels(P, xs, ys, zs, s, W, H)
    assert np.array_equal(ins[dec], rin[dec])
    both = dec & rin
    assert np.array_equal(px[both], rpx[both].astype(np.int64)) and np.array_equal(py[both], rpy[both].astype(np.int64))
    return dec
