"""Captures of more than 256 views: vc_append_views, the view groups of 256 consecutive views that carve, plan and sparse
download loop over, and the colour pass over every view.  Every result is compared bit for bit with the CPU oracle, which takes
any number of views.  Views are jittered copies of a few base cameras (all copies of a base see the same silhouette edge, so
listed bricks carry many undecided views in every group), plus per-view background specks so that every view carves voxels
of its own."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
DIMS = (64, 48, 40)
S = F(0.01)


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


# ---- capture helpers (camera ring and masks as in test_input_limits.py) ----------------------------------------------------
def _grid_centre(X, Y, Z, s):
    return np.array([(Y - 1) * float(s) / 2, (X - 1) * float(s) / 2, -(Z - 1) * float(s) / 2])


def _look_at(eye, target, fx, fy, cx, cy):
    from ar_voxel_project_b200.synth import gemm_k_m_f32
    zc = target - eye
    zc = zc / np.linalg.norm(zc)
    up = np.array([0.0, 0.0, -1.0]) if abs(zc[2]) < 0.9 else np.array([1.0, 0.0, 0.0])
    xc = np.cross(zc, up)
    xc /= np.linalg.norm(xc)
    yc = np.cross(zc, xc)
    R = np.stack([xc, yc, zc])
    M = np.concatenate([R, (-R @ eye)[:, None]], axis=1).astype(F)
    K = np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], F)
    return gemm_k_m_f32(K, M), M


def _ring(X, Y, Z, s, V, W, H, n_base, span=0.6, seed=0):
    """V cameras on a ring looking at the grid's centre; view v is a copy of base camera v % n_base, jittered below a pixel"""
    rng = np.random.default_rng(seed)
    c = _grid_centre(X, Y, Z, s)
    ext = float(s) * max(X, Y, Z) * 1.5
    dist = 3.0 * ext
    P, M = [], []
    for v in range(V):
        b = v % n_base
        az, el = 2 * np.pi * (b + 0.3) / n_base, np.deg2rad(25.0 if b % 2 else 55.0)
        eye = c + dist * np.array([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), -np.sin(el)])
        eye = eye + rng.uniform(-1, 1, 3) * dist * 1e-4
        jx, jy = rng.uniform(-0.5, 0.5, 2)
        p, m = _look_at(eye, c, span * W * dist / ext, span * H * dist / ext, W / 2 + jx, H / 2 + jy)
        P.append(p), M.append(m)
    return np.stack(P), np.stack(M)


def _ellipse_bits(W, H, cx, cy, rx, ry, rng, n_specks):
    """uint32[H][ceil(W/32)] (1 = background): a foreground ellipse plus n_specks random background pixels"""
    from ar_voxel_project_b200.synth import pack_bits
    yy, xx = np.mgrid[0:H, 0:W]
    bg = ((xx - cx) / rx) ** 2 + ((yy - cy) / ry) ** 2 > 1.0
    bg[rng.integers(0, H, n_specks), rng.integers(0, W, n_specks)] = True
    return pack_bits(bg)


def _capture(V, W=160, H=120, n_base=8, seed=0, dup=0, specks=0.002, radius=1.0, dims=DIMS):
    """-> dict(P, M, bits, images); with dup, views 256 .. 256+dup-1 are exact copies (P, M, mask) of views 0 .. dup-1 with images
    of their own, so equal depths meet across the group boundary in the closest-colour pass"""
    X, Y, Z = dims
    P, M = _ring(X, Y, Z, S, V, W, H, n_base, seed=seed)
    rng = np.random.default_rng(seed + 1)
    r = min(W, H) * radius
    bits = np.stack([_ellipse_bits(W, H, W / 2, H / 2, r * (0.16 + 0.02 * (v % n_base)), r * (0.18 + 0.015 * (v % n_base)), rng,
                                   int(specks * W * H)) for v in range(V)])
    if dup:
        P[256:256 + dup], M[256:256 + dup], bits[256:256 + dup] = P[:dup], M[:dup], bits[:dup]
    images = rng.integers(0, 256, (V, H, W, 3), dtype=np.uint8)
    return dict(P=P, M=M, bits=bits, images=images, W=W, H=H, V=V, dims=dims)


def _engine(A, c, z0=0, z1=None, images=False, first=256):
    """an engine holding all views of the capture: vc_set_views takes the first `first`, vc_append_views the rest"""
    X, Y, Z = c["dims"]
    e = A.VoxelEngine(X, Y, Z, S, z_begin=z0, z_end=z1)
    k = min(first, c["V"])
    e.set_views(c["P"][:k], c["W"], c["H"], c["M"][:k])
    e.set_masks_bits(c["bits"][:k])
    if images:
        e.set_images(c["images"][:k])
    if c["V"] > k:
        e.append_views(c["P"][k:], c["M"][k:], mask_bits=c["bits"][k:], images_bgr=c["images"][k:] if images else None)
    assert e.V == c["V"]
    return e


def _oracle_carve(oracle, c, v1=None, z0=0, z1=None, mask_bgr=None):
    X, Y, Z = c["dims"]
    v1 = c["V"] if v1 is None else v1
    if mask_bgr is not None:
        return oracle.carve(X, Y, Z, S, c["P"][:v1], c["W"], c["H"], mask_bgr=mask_bgr[:v1], z0=z0, z1=z1, nthreads=0)
    return oracle.carve(X, Y, Z, S, c["P"][:v1], c["W"], c["H"], mask_bits=c["bits"][:v1], z0=z0, z1=z1, nthreads=0)


def _volumes(e):
    return e.download_occupied(), e.download_seen()


def _same(a, b, what):
    assert np.array_equal(a[0], b[0]), f"occupied differs: {what}"
    assert np.array_equal(a[1], b[1]), f"seen differs: {what}"


_CAPTURES = {}


def _cap(V, **kw):
    key = (V, tuple(sorted(kw.items())))
    if key not in _CAPTURES:
        _CAPTURES[key] = _capture(V, **kw)
    return _CAPTURES[key]


# ---- 1. carve -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [257, 300, 511, 512, 513, 1000])
@pytest.mark.parametrize("slab", [None, (8, 32)], ids=["grid", "slab"])
def test_carve_many_views(A, oracle, V, slab):
    c = _cap(V)
    z0, z1 = slab or (0, None)
    ref = _oracle_carve(oracle, c, z0=z0, z1=z1)
    assert 0 < int(oracle.unpack(ref[0], DIMS[0]).sum()) < DIMS[0] * DIMS[1] * ((z1 or DIMS[2]) - z0)
    with _engine(A, c, z0, z1) as e:
        e.reset()
        e.carve(0, 0, 256, count_executed=True)
        listed_group0 = e.stats()["bricks_listed"]
        e.reset()
        e.carve(0, count_executed=True)
        st = e.stats()
        assert st["filter_mismatches"] == 0
        assert st["bricks_listed"] > listed_group0 > 0  # summed over the groups
        _same(_volumes(e), ref, f"VC_EXACT counting run, V={V}")
        e.reset()
        e.carve(0)
        _same(_volumes(e), ref, f"VC_EXACT, V={V}")
        e.reset()
        e.carve(2)
        _same(_volumes(e), ref, f"VC_EXACT_FLAT, V={V}")
        e.reset()
        e.carve(1)  # the diagnostic f32 pipeline runs over every group (not bit-exact by design)
        occ, _ = _volumes(e)
        assert occ.shape == ref[0].shape


# ---- 2. one carving view among 1000 ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 255, 256, 257, 511, 512, 767, 999])
def test_one_carving_view_among_1000(A, oracle, k):
    c = dict(_cap(1000))
    bits = np.zeros_like(c["bits"])
    bits[k] = c["bits"][k]
    c["bits"] = bits
    ref = _oracle_carve(oracle, c)
    assert int(oracle.unpack(ref[0], DIMS[0]).sum()) < DIMS[0] * DIMS[1] * DIMS[2]  # view k carves
    with _engine(A, c) as e:
        for mode in (0, 2):
            e.reset()
            e.carve(mode)
            _same(_volumes(e), ref, f"view {k}, mode {mode}")


# ---- 3. view ranges across group boundaries ---------------------------------------------------------------------------------
@pytest.mark.parametrize("ranges", [[(200, 300), (300, 1000), (0, 200)], [(0, 256), (256, 512), (512, 1000)],
                                    [(255, 257), (0, 255), (257, 1000)], [(600, 1000), (0, 600)], [(0, 1), (999, 1000), (1, 999)],
                                    [(300, 300), (0, 1000)]])
def test_ranges_across_group_boundaries(A, oracle, ranges):
    c = _cap(1000)
    ref = _oracle_carve(oracle, c)
    with _engine(A, c) as e:
        for mode in (0, 2):
            e.reset()
            for v0, v1 in ranges:
                e.carve(mode, v0, v1)
            _same(_volumes(e), ref, f"{ranges} mode {mode}")


# ---- 4. streaming: a capture that grows while the volumes stay on the device -------------------------------------------------
def _bgr_of_bits(bits, W, rng):
    """8UC3 masks whose (0,0,0) pixels are the background bits"""
    bg = np.unpackbits(bits.view(np.uint8), bitorder="little").reshape(*bits.shape[:-1], -1)[..., :W].astype(bool)
    img = rng.integers(1, 256, bg.shape + (3,), dtype=np.uint8)
    img[bg] = 0
    return img


@pytest.mark.parametrize("fmt", ["bits", "bgr", "raw"])
def test_streaming_appends(A, oracle, golden, fmt):
    X, Y, Z = DIMS
    c = _cap(600)
    W, H = c["W"], c["H"]
    rng = np.random.default_rng(5)
    masks = c["bits"] if fmt == "bits" else _bgr_of_bits(c["bits"], W, rng)
    images = c["images"]
    und_masks, und_images = None, images
    if fmt == "raw":
        z = golden("undistort_kat.npz")
        K = z["box_mask0000_K"].astype(np.float64).copy()
        K[:2] /= 4.0  # the 640x480 calibration scaled to 160x120
        dist = z["box_mask0000_dist"]
        und_masks = np.stack([oracle.undistort(m, K, dist) for m in masks])
        und_images = np.stack([oracle.undistort(m, K, dist) for m in images])
    elif fmt == "bgr":
        und_masks = masks
    checks = {8, 256, 264, 512, 520, 600}
    with A.VoxelEngine(X, Y, Z, S) as e:
        e.set_views(c["P"][:8], W, H, c["M"][:8])
        if fmt == "raw":
            e.set_calibration(K, dist)
            e.set_masks_raw(masks[:8])
            e.set_images_raw(images[:8])
        elif fmt == "bgr":
            e.set_masks_bgr(masks[:8])
            e.set_images(images[:8])
        else:
            e.set_masks_bits(masks[:8])
            e.set_images(images[:8])
        e.reset()
        e.carve(0)
        for v in range(8, 600, 8):
            if v in checks:
                _same(_volumes(e), _oracle_carve(oracle, c, v, mask_bgr=und_masks), f"{fmt}: prefix of {v} views")
            if fmt == "bits":
                e.append_views(c["P"][v:v + 8], c["M"][v:v + 8], mask_bits=masks[v:v + 8], images_bgr=images[v:v + 8])
            else:
                e.append_views(c["P"][v:v + 8], c["M"][v:v + 8], mask_bgr=masks[v:v + 8], raw=fmt == "raw", images_bgr=images[v:v + 8])
            e.carve(0 if v % 16 else 2, v, -1)  # only the new views, onto the volumes on the device
        ro, rs = _oracle_carve(oracle, c, 600, mask_bgr=und_masks)
        _same(_volumes(e), (ro, rs), f"{fmt}: 600 views")
        assert np.array_equal(e.download_images(), und_images)
        if fmt != "bits":
            from ar_voxel_project_b200.synth import pack_bits
            assert np.array_equal(e.download_masks(), pack_bits((und_masks == 0).all(-1)))
        else:
            assert np.array_equal(e.download_masks(), masks)
        e.color(2)
        idx, rgbn = e.download_colors()
    ridx, rrgbn = oracle.color(X, Y, Z, S, c["P"], c["M"], W, H, und_images, ro, 2)
    assert np.array_equal(idx, ridx) and np.array_equal(rgbn, rrgbn)


# ---- 5. colour over every view ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [300, 1000])
@pytest.mark.parametrize("mode", [1, 2], ids=["closest", "avg"])
def test_color_many_views(A, oracle, V, mode):
    X, Y, Z = DIMS
    c = _cap(V, dup=40)
    ro, _ = _oracle_carve(oracle, c)
    ridx, rrgbn = oracle.color(X, Y, Z, S, c["P"], c["M"], c["W"], c["H"], c["images"], ro, mode)
    assert (rrgbn[:, 3] == 255).sum() > 0  # voxels seen by more than 255 views: the stored count saturates
    with _engine(A, c, images=True) as e:
        e.carve()
        e.color(mode)
        idx, rgbn = e.download_colors()
    assert np.array_equal(idx, ridx)
    assert np.array_equal(rgbn, rrgbn)


def test_closest_colour_ties_across_the_group_boundary(A, oracle):
    """views 256.. are exact copies of views 0..: every depth of group 1 ties one of group 0, and the first strict minimum keeps
    group 0's colour; a capture whose group-0 copy is removed must pick the group-1 colour instead"""
    X, Y, Z = DIMS
    c = _cap(300, dup=40)
    ro, _ = _oracle_carve(oracle, c)
    with _engine(A, c, images=True) as e:
        e.carve()
        e.color(1)
        idx, rgbn = e.download_colors()
    c2 = dict(c)
    c2["images"] = c["images"].copy()
    c2["images"][256:296] = c["images"][:40]
    with _engine(A, c2, images=True) as e:
        e.carve()
        e.color(1)
        idx2, rgbn2 = e.download_colors()
    assert np.array_equal(idx, idx2)
    assert np.array_equal(rgbn, rgbn2)  # the copies' own images never win a tie
    ridx, rrgbn = oracle.color(X, Y, Z, S, c["P"], c["M"], c["W"], c["H"], c["images"], ro, 1)
    assert np.array_equal(rgbn, rrgbn)


# ---- 6. fastCarve ------------------------------------------------------------------------------------------------------------
def test_fast_carve_300(A, oracle):
    X, Y, Z = DIMS
    c = _cap(300)
    ref = oracle.fast_carve(X, Y, Z, S, c["P"], c["W"], c["H"], mask_bits=c["bits"])
    with _engine(A, c) as e:
        e.fast_carve()
        _same(_volumes(e), ref, "fast_carve, 300 views")


# ---- 7. sparse download ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dims,slab", [(DIMS, None), (DIMS, (8, 32)), ((70, 45, 37), None), ((70, 45, 37), (3, 30))],
                         ids=["grid", "slab", "ragged_grid", "ragged_slab"])
def test_sparse_download_300(A, oracle, dims, slab):
    """the ragged cases have bricks cut by the grid's x end (a partial last word), its y end and the slab's z end"""
    c = _cap(300, specks=0.0, radius=0.4, dims=dims)  # a small object and no specks: bricks carved whole next to the listed ones
    z0, z1 = slab or (0, None)
    ref = _oracle_carve(oracle, c, z0=z0, z1=z1)
    with _engine(A, c, z0, z1) as e:
        flags, listed, words = e.carve_download_sparse()
        assert 0 < len(listed) < flags.size
        assert set(np.unique(flags)) <= {0, 2, 3, 8} and (flags == 3).any()
        if dims != DIMS:  # the tail bricks in x, y and z include bricks carved whole
            assert (flags[:, :, -1] == 3).any() and (flags[:, -1, :] == 3).any() and (flags[-1] == 3).any()
        assert np.array_equal(np.sort(listed), np.flatnonzero(flags.reshape(-1) == 8))
        _same(e.expand_sparse(flags, listed, words), ref, "expanded sparse download")
        _same(_volumes(e), ref, "volumes after the sparse download")


def test_carve_download_chunks_300(A, oracle):
    """vc_carve_download into page-locked buffers carves in z-chunks (every chunk over every group) while the finished ones travel"""
    import torch
    c = _cap(300, dims=(64, 48, 72))
    ref = _oracle_carve(oracle, c)
    with _engine(A, c) as e:
        occ = torch.empty(ref[0].shape, dtype=torch.int32).pin_memory()
        seen = torch.empty(ref[0].shape, dtype=torch.int32).pin_memory()
        for _ in range(2):
            e.reset()
            e.carve_download(occ, seen)
            _same((occ.numpy().view(np.uint32), seen.numpy().view(np.uint32)), ref, "chunked carve_download")
            _same(e.carve_download(), ref, "carve_download into pageable buffers")


# ---- 8. plan_slabs -----------------------------------------------------------------------------------------------------------
def test_plan_slabs_600(A, oracle):
    X, Y, Z = DIMS
    c = _cap(600)
    ref = _oracle_carve(oracle, c)
    with _engine(A, c) as e:
        for n in (2, 3, 5):
            b = e.plan_slabs(n)
            assert b[0] == 0 and b[-1] == Z and all(b[i] < b[i + 1] for i in range(n))
            assert all(x % 8 == 0 for x in b[1:-1])
            for i in range(n):
                with _engine(A, c, b[i], b[i + 1]) as es:
                    es.carve()
                    _same(_volumes(es), (ref[0][b[i]:b[i + 1]], ref[1][b[i]:b[i + 1]]), f"slab {i} of {b}")


# ---- 9. the mesh ---------------------------------------------------------------------------------------------------------------
def test_mesh_off_300(A, oracle, tmp_path):
    X, Y, Z = DIMS
    c = _cap(300, dup=40)
    ro, rs = _oracle_carve(oracle, c)
    ridx, rrgbn = oracle.color(X, Y, Z, S, c["P"], c["M"], c["W"], c["H"], c["images"], ro, 2)
    rgba = oracle.closure(X, Y, Z, oracle.dense_model(X, Y, Z, ro, rs, ridx, rrgbn), 3)
    rv, rc = oracle.marching_cubes(X, Y, Z, rgba, 0.5)
    t = (0.5, -0.25, 2.0)
    p = str(tmp_path / "ref.off")
    oracle.write_off(p, rv, rc, F(1.5) * S, t)
    with _engine(A, c, images=True) as e:
        e.carve()
        e.color(2)
        n = e.mesh_from_volumes(True, True, 3, 0.5, download=False)
        assert n == len(rv) > 0
        text = e.mesh_off(F(1.5) * S, t)
    assert text == open(p, "rb").read()


# ---- 10. two engines on one device -----------------------------------------------------------------------------------------------
def test_two_engines_interleaved(A, oracle):
    X, Y, Z = DIMS
    big, small = _cap(600, dup=40), _cap(8, seed=3)
    rb, rs_ = _oracle_carve(oracle, big), _oracle_carve(oracle, small)
    cb = {m: oracle.color(X, Y, Z, S, big["P"], big["M"], big["W"], big["H"], big["images"], rb[0], m) for m in (1, 2)}
    cs = {m: oracle.color(X, Y, Z, S, small["P"], small["M"], small["W"], small["H"], small["images"], rs_[0], m) for m in (1, 2)}
    with _engine(A, big, images=True) as eb, _engine(A, small, images=True) as es:
        for rnd in range(2):
            eb.reset()
            es.reset()
            eb.carve(0, 0, 300)
            es.carve(0)
            eb.carve(2 if rnd else 0, 300, -1)
            _same(_volumes(eb), rb, f"big engine, round {rnd}")
            _same(_volumes(es), rs_, f"small engine, round {rnd}")
            for m in (1, 2):
                eb.color(m)
                es.color(m)
                for e, ref in ((eb, cb[m]), (es, cs[m])):
                    idx, rgbn = e.download_colors()
                    assert np.array_equal(idx, ref[0]) and np.array_equal(rgbn, ref[1]), (rnd, m, e.V)


# ---- 11. refusals ------------------------------------------------------------------------------------------------------------------
def test_refused_appends_leave_the_engine_as_it_was(A, oracle):
    import ctypes as C
    from ar_voxel_project_b200 import _lib as L
    X, Y, Z = DIMS
    c = _cap(300)
    W, H = c["W"], c["H"]
    with A.VoxelEngine(X, Y, Z, S) as e:
        with pytest.raises(A.VoxCarveError) as ex:  # before vc_set_views
            e.append_views(c["P"][:1], c["M"][:1], mask_bits=c["bits"][:1])
        assert ex.value.code == L.VC_ERR_STATE
        e.set_views(c["P"][:256], W, H, c["M"][:256])
        with pytest.raises(A.VoxCarveError) as ex:  # before vc_set_masks
            e.append_views(c["P"][256:], c["M"][256:], mask_bits=c["bits"][256:])
        assert ex.value.code == L.VC_ERR_STATE
    with _engine(A, c, images=True) as e:
        e.reset()
        e.carve()
        state = (e.V, e.download_masks(), e.download_images(), _volumes(e))
        n = 8
        P, M, bits, img = c["P"][:n], c["M"][:n], c["bits"][:n], c["images"][:n]
        bgr = _bgr_of_bits(bits, W, np.random.default_rng(0))
        lib, h = e._lib, e._h
        refusals = [
            (L.VC_ERR_ARG, lambda: lib.vc_append_views(h, 0, P.ctypes.data, M.ctypes.data, C.c_void_p(bits.ctypes.data), L.VC_MASK_BITS, C.c_void_p(img.ctypes.data))),
            (L.VC_ERR_ARG, lambda: lib.vc_append_views(h, -3, P.ctypes.data, M.ctypes.data, C.c_void_p(bits.ctypes.data), L.VC_MASK_BITS, C.c_void_p(img.ctypes.data))),
            (L.VC_ERR_ARG, lambda: lib.vc_append_views(h, L.VC_MAX_TOTAL_VIEWS - 300 + 1, P.ctypes.data, M.ctypes.data, C.c_void_p(bits.ctypes.data), L.VC_MASK_BITS, C.c_void_p(img.ctypes.data))),
            (L.VC_ERR_ARG, lambda: lib.vc_append_views(h, n, P.ctypes.data, None, C.c_void_p(bits.ctypes.data), L.VC_MASK_BITS, C.c_void_p(img.ctypes.data))),   # M missing
            (L.VC_ERR_ARG, lambda: lib.vc_append_views(h, n, P.ctypes.data, M.ctypes.data, C.c_void_p(bits.ctypes.data), L.VC_MASK_BITS, None)),  # images missing
            (L.VC_ERR_ARG, lambda: lib.vc_append_views(h, n, P.ctypes.data, M.ctypes.data, C.c_void_p(bits.ctypes.data), 7, C.c_void_p(img.ctypes.data))),
            (L.VC_ERR_ARG, lambda: lib.vc_append_views(h, n, None, M.ctypes.data, C.c_void_p(bits.ctypes.data), L.VC_MASK_BITS, C.c_void_p(img.ctypes.data))),
            (L.VC_ERR_STATE, lambda: lib.vc_append_views(h, n, P.ctypes.data, M.ctypes.data, C.c_void_p(bgr.ctypes.data), L.VC_MASK_BGR8_RAW, C.c_void_p(img.ctypes.data))),  # no calibration
        ]
        for code, call in refusals:
            assert call() == code, lib.vc_last_error(h).decode()
            assert e.V == state[0]
            assert np.array_equal(e.download_masks(), state[1]) and np.array_equal(e.download_images(), state[2])
            _same(_volumes(e), state[3], "volumes after a refused append")
            e.reset()
            e.carve()
            _same(_volumes(e), state[3], "carve after a refused append")
    with _engine(A, c) as e:  # no M, no images on the engine: giving them is refused
        e.set_views(c["P"][:256], W, H)
        e.set_masks_bits(c["bits"][:256])
        with pytest.raises(A.VoxCarveError):
            e.append_views(c["P"][256:], c["M"][256:], mask_bits=c["bits"][256:])
        with pytest.raises(A.VoxCarveError):
            e.append_views(c["P"][256:], mask_bits=c["bits"][256:], images_bgr=c["images"][256:])
        e.append_views(c["P"][256:], mask_bits=c["bits"][256:])
        e.reset()
        e.carve()
        _same(_volumes(e), _oracle_carve(oracle, c), "appended without M")
        # vc_set_views after appends: back to a set of at most 256 views
        e.set_views(c["P"][40:140], W, H, c["M"][40:140])
        e.set_masks_bits(c["bits"][40:140])
        assert e.download_masks().shape[0] == 100
        e.reset()
        e.carve()
        X, Y, Z = DIMS
        _same(_volumes(e), oracle.carve(X, Y, Z, S, c["P"][40:140], W, H, mask_bits=c["bits"][40:140], nthreads=0), "set_views after appends")


@pytest.mark.parametrize("V2", [200, 256])
def test_set_views_after_a_small_append(A, oracle, V2):
    """set_views(8) + append 8 leaves 16 views; a following set_views of up to 256 views must have room for all of them"""
    X, Y, Z = DIMS
    c = _cap(300)
    W, H = c["W"], c["H"]
    with A.VoxelEngine(X, Y, Z, S) as e:
        e.set_views(c["P"][:8], W, H, c["M"][:8])
        e.set_masks_bits(c["bits"][:8])
        e.append_views(c["P"][8:16], c["M"][8:16], mask_bits=c["bits"][8:16])
        e.reset()
        e.carve()
        _same(_volumes(e), _oracle_carve(oracle, c, 16), "16 views")
        e.set_views(c["P"][:V2], W, H, c["M"][:V2])
        e.set_masks_bits(c["bits"][:V2])
        ref = _oracle_carve(oracle, c, V2)
        e.reset()
        e.carve(0, count_executed=True)
        assert e.stats()["filter_mismatches"] == 0
        _same(_volumes(e), ref, f"set_views({V2}) after the append, counting run")
        e.reset()
        e.carve()
        _same(_volumes(e), ref, f"set_views({V2}) after the append")
        e.append_views(c["P"][V2:300], c["M"][V2:300], mask_bits=c["bits"][V2:300])
        e.reset()
        e.carve()
        _same(_volumes(e), _oracle_carve(oracle, c), "grown again to 300 views")


def test_refused_append_past_2p31_mask_words(A):
    """mask words (V+n) * H * ceil(W/32) >= 2^31 are refused before anything is read or allocated"""
    import ctypes as C
    from ar_voxel_project_b200 import _lib as L
    W, H = 1 << 20, 1024  # 2^25 mask words per view: 64 views reach 2^31
    P, _ = _ring(8, 8, 8, S, 1, W, H, 1)
    with A.VoxelEngine(8, 8, 8, S) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(np.zeros((1, H, W // 32), np.uint32))
        e.reset()
        e.carve()
        before = _volumes(e)
        one = np.zeros(64, np.uint32)
        Pn = np.repeat(P, 63, axis=0)
        assert e._lib.vc_append_views(e._h, 63, Pn.ctypes.data, None, C.c_void_p(one.ctypes.data), L.VC_MASK_BITS, None) == L.VC_ERR_ARG
        assert e.V == 1 and e.download_masks().shape[0] == 1
        e.reset()
        e.carve()
        _same(_volumes(e), before, "after a refused append")


# ---- the C++ host layer ------------------------------------------------------------------------------------------------------------
def test_cpp_host_layer_300_views(A, oracle, tmp_path, lib_built):
    """vc::carve into a stand-in Model and vc::carveToMesh from a 300-view ViewCache (setViews appends past 256)"""
    X, Y, Z = DIMS
    c = _cap(300, dup=40)
    case = tmp_path / "case.bin"
    with open(case, "wb") as f:
        np.array([X, Y, Z, c["V"], c["W"], c["H"]], np.int32).tofile(f)
        np.array([S], np.float32).tofile(f)
        c["P"].astype(np.float32).tofile(f)
        c["M"].astype(np.float32).tofile(f)
        c["bits"].astype(np.uint32).tofile(f)
        c["images"].astype(np.uint8).tofile(f)
    exe = str(tmp_path / "many_views")
    libdir = os.path.dirname(lib_built)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "many_views.cpp"), "-o", exe,
                           "-L", libdir, "-lvoxcarve", f"-Wl,-rpath,{libdir}"])
    model, off = tmp_path / "model.bin", tmp_path / "mesh.off"
    subprocess.check_call([exe, str(case), str(model), str(off)], stdout=subprocess.DEVNULL)
    raw = np.fromfile(model, np.uint8)
    n = X * Y * Z
    ro, rs = _oracle_carve(oracle, c)
    assert np.array_equal(raw[:n].astype(bool), oracle.unpack(ro, X).reshape(-1))
    assert np.array_equal(raw[n:].astype(bool), oracle.unpack(rs, X).reshape(-1))
    ridx, rrgbn = oracle.color(X, Y, Z, S, c["P"], c["M"], c["W"], c["H"], c["images"], ro, 2)
    rv, rc = oracle.marching_cubes(X, Y, Z, oracle.closure(X, Y, Z, oracle.dense_model(X, Y, Z, ro, rs, ridx, rrgbn), 3), 0.5)
    ref = tmp_path / "ref.off"
    oracle.write_off(str(ref), rv, rc, F(1.5) * S, (0.5, -0.25, 2.0))
    assert open(off, "rb").read() == open(ref, "rb").read()


def test_api_view_set_above_256(A, oracle):
    """api.carve / reconstructAvgColor take a ViewSet of more than 256 views"""
    from ar_voxel_project_b200 import api
    X, Y, Z = DIMS
    c = _cap(300)
    vs = api.ViewSet(c["P"], c["M"], c["W"], c["H"], mask_bits=c["bits"], images_bgr=c["images"])
    with api._engine_for(A.Model(X, Y, Z, S), vs, need_images=True) as e:
        assert e.V == 300
        e.carve()
        _same(_volumes(e), _oracle_carve(oracle, c), "api engine")
