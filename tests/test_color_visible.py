"""vc_color_visible (occlusion-aware colouring): the CPU restatement (oracle/color_visible_oracle.c) on scenes whose answer is
known, its properties on the goldens, and the device records bit for bit against it (idx and all four bytes of rgbn)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN

F = np.float32
INF = float("inf")


@pytest.fixture(scope="module")
def CV():
    from oracle import color_visible as CV
    CV.build()
    return CV


# ---- scenes -------------------------------------------------------------------------------------------------------------------
def _look_at(eye, target, f, W, H, cx=None, cy=None):
    """P = K [R|t] (K's last row (0, 0, 1)) and M = [R|t] of a camera at world point `eye` looking at `target`"""
    from ar_voxel_project_b200.synth import gemm_k_m_f32
    zc = np.asarray(target, float) - np.asarray(eye, float)
    zc = zc / np.linalg.norm(zc)
    up = np.array([0.0, 0.0, -1.0]) if abs(zc[2]) < 0.9 else np.array([1.0, 0.0, 0.0])
    xc = np.cross(zc, up)
    xc /= np.linalg.norm(xc)
    yc = np.cross(zc, xc)
    R = np.stack([xc, yc, zc])
    M = np.concatenate([R, (-R @ np.asarray(eye, float))[:, None]], axis=1).astype(F)
    K = np.array([[f, 0, W / 2 if cx is None else cx], [0, f, H / 2 if cy is None else cy], [0, 0, 1]], F)
    return gemm_k_m_f32(K, M), M


def _world(x, y, z, s):
    """world point of voxel index (x, y, z) (Model.h:134-136: (y s, x s, -z s))"""
    return np.array([y * float(s), x * float(s), -z * float(s)])


def _words(vol):
    """bool[Z, Y, X] -> uint32[Z, Y, ceil(X/32)]"""
    from ar_voxel_project_b200.synth import pack_bits
    return np.stack([pack_bits(vol[z]) for z in range(vol.shape[0])])


def _blocks(dims, boxes):
    X, Y, Z = dims
    vol = np.zeros((Z, Y, X), bool)
    for (x0, x1), (y0, y1), (z0, z1) in boxes:
        vol[z0:z1, y0:y1, x0:x1] = True
    return _words(vol)


def _flat_images(V, W, H):
    """view v is one flat colour that encodes v: BGR (3v + 1, 3v + 2, 3v + 3)"""
    img = np.empty((V, H, W, 3), np.uint8)
    for v in range(V):
        img[v] = (3 * v + 1, 3 * v + 2, 3 * v + 3)
    return img


def _p2_all_corners(P, x, y, z, s):
    """p2 of the centre and the 8 corners of voxel (x, y, z) (f64 sequential accumulation, one f32 rounding)"""
    out = []
    for dx, dy, dz in [(0, 0, 0)] + [(a, b, c) for c in (-.5, .5) for b in (-.5, .5) for a in (-.5, .5)]:
        w = (F(F(y + dy) * F(s)), F(F(x + dx) * F(s)), F(-F(z + dz) * F(s)))
        acc = float(P[2, 0]) * float(w[0])
        acc = acc + float(P[2, 1]) * float(w[1])
        acc = acc + float(P[2, 2]) * float(w[2])
        acc = acc + float(P[2, 3])
        out.append(F(acc))
    return np.array(out)


# two solid blocks 8^3 along x, 12 voxels apart; cameras far out on +x, -x, +y, -y, all looking at the grid centre
BLOCK_DIMS = (40, 16, 16)
BLOCK_S = F(0.01)
BLOCKS = [((4, 12), (4, 12), (4, 12)), ((24, 32), (4, 12), (4, 12))]


def _block_scene():
    X, Y, Z = BLOCK_DIMS
    c = _world((X - 1) / 2, (Y - 1) / 2, (Z - 1) / 2, BLOCK_S)
    d = 2.0
    eyes = [c + [0, d, 0], c - [0, d, 0], c + [d, 0, 0], c - [d, 0, 0]]  # world axis 1 = x, axis 0 = y
    PM = [_look_at(e, c, 400.0, 320, 320) for e in eyes]
    P, M = np.stack([p for p, _ in PM]), np.stack([m for _, m in PM])
    return P, M, 320, 320, _flat_images(4, 320, 320), _blocks(BLOCK_DIMS, BLOCKS)


def _colour_of(v):
    return (3 * v + 3, 3 * v + 2, 3 * v + 1)  # RGB of view v's flat BGR image


# ---- CPU: the oracle on a known scene ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [1, 2], ids=["closest", "avg"])
def test_oracle_two_blocks_known_answer(CV, mode):
    X, Y, Z = BLOCK_DIMS
    P, M, W, H, img, occ = _block_scene()
    idx, rgbn, obs = CV.color_visible(X, Y, Z, BLOCK_S, P, M, W, H, img, occ, mode, 2.0, observations=True)
    where = {int(f): k for k, f in enumerate(idx)}

    def rec(x, y, z):
        return where[x + X * (y + Y * z)]

    expect = {  # face centre -> the views that observe it (0: +x camera, 1: -x, 2: +y, 3: -y)
        (31, 8, 8): {0},      # far block's outer face, towards +x
        (4, 8, 8): {1},       # near block's outer face, towards -x
        (11, 8, 8): set(),    # near block's face towards +x: hidden from the +x camera by the far block
        (24, 8, 8): set(),    # far block's face towards -x: hidden from the -x camera by the near block
        (8, 11, 8): {2}, (28, 11, 8): {2},  # the +y camera reaches both blocks
        (8, 4, 8): {3}, (28, 4, 8): {3},    # the -y camera too
    }
    for (x, y, z), views in expect.items():
        k = rec(x, y, z)
        assert set(np.flatnonzero(obs[k])) == views, (x, y, z)
        assert rgbn[k, 3] == len(views)
        if views:
            assert tuple(rgbn[k, :3]) == _colour_of(next(iter(views))), (x, y, z)
        else:
            assert tuple(rgbn[k, :3]) == (50, 168, 141)  # MODEL_COLOR
    # the reference colouring counts the hidden faces as observed by the cameras they face
    from oracle import oracle as O
    ridx, rrgbn = O.color(X, Y, Z, BLOCK_S, P, M, W, H, img, occ, mode)
    assert np.array_equal(ridx, idx)
    assert rrgbn[rec(11, 8, 8), 3] >= 1 and rrgbn[rec(24, 8, 8), 3] >= 1


@pytest.mark.parametrize("ds", ["box", "human"])
def test_oracle_properties_on_goldens(CV, oracle, ds):
    import ar_voxel_project_b200 as A
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, f"{ds}_views.npz"))
    X = Y = Z = 100
    s = F(0.28) / F(X)
    occ, _ = oracle.carve(X, Y, Z, s, vs.P, vs.W, vs.H, mask_bits=vs.mask_bits, nthreads=0)
    for mode in (1, 2):
        ridx, rrgbn = oracle.color(X, Y, Z, s, vs.P, vs.M, vs.W, vs.H, vs.images_bgr, occ, mode)
        idx, rgbn = CV.color_visible(X, Y, Z, s, vs.P, vs.M, vs.W, vs.H, vs.images_bgr, occ, mode, INF)
        assert np.array_equal(idx, ridx) and np.array_equal(rgbn, rrgbn), "tolerance = inf must equal vo_color here"
    prev_obs, prev_n = None, None
    for tol in (INF, 4.0, 2.0, 1.0, 0.0):  # observations shrink as the tolerance falls
        idx, rgbn, obs = CV.color_visible(X, Y, Z, s, vs.P, vs.M, vs.W, vs.H, vs.images_bgr, occ, 2, tol, observations=True)
        assert np.array_equal(rgbn[:, 3], np.minimum(obs.sum(1), 255))
        if prev_obs is not None:
            assert not (obs & ~prev_obs).any(), tol
            assert (rgbn[:, 3] <= prev_n).all() and obs.sum() < prev_obs.sum(), tol
        prev_obs, prev_n = obs, rgbn[:, 3]
    assert prev_obs.sum() > 0  # tolerance 0: a voxel never hides itself


def test_oracle_camera_inside_the_grid(CV, oracle):
    """a camera inside the grid has voxels behind it: their pairs (some p2 <= 0) neither occlude nor observe, while the
    reference point-reflects them into the image"""
    X, Y, Z = 32, 24, 20
    s = F(0.01)
    vol = np.zeros((Z, Y, X), bool)
    vol[2:18, 2:22, 2:30] = True
    vol[6:14, 8:16, 12:20] = False  # a hollow around the camera
    occ = _words(vol)
    P0, M0 = _look_at(_world(15.5, 11.5, 9.5, s), _world(31, 11.5, 9.5, s), 60.0, 64, 48)
    P1, M1 = _look_at(_world(16, 12, 10, s) + [0, 0, 3.0], _world(16, 12, 10, s), 300.0, 64, 48)
    P, M = np.stack([P0, P1]), np.stack([M0, M1])
    img = _flat_images(2, 64, 48)
    idx, rgbn, obs = CV.color_visible(X, Y, Z, s, P, M, 64, 48, img, occ, 2, INF, observations=True)
    _, rrgbn = oracle.color(X, Y, Z, s, P, M, 64, 48, img, occ, 2)
    behind = reflected = 0
    for k, f in enumerate(idx):
        x, y, z = int(f) % X, int(f) // X % Y, int(f) // (X * Y)
        p2 = _p2_all_corners(P[0], x, y, z, s)
        if not (p2 > 0).all():
            behind += 1
            assert not obs[k, 0], (x, y, z)
            ok, *_ = oracle.pixel_of(P[0], x, y, z, s, 64, 48)
            reflected += ok
    assert behind > 0 and reflected > 0  # the reference counts some of them (point-reflected into the image)
    assert obs[:, 0].any() and obs[:, 1].any()
    assert (rgbn[:, 3] < rrgbn[:, 3]).any()


# ---- GPU: bit for bit against the oracle ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


def _engine(A, dims, s, P, M, W, H, img, occ):
    X, Y, Z = dims
    e = A.VoxelEngine(X, Y, Z, s)
    k = min(256, len(P))
    e.set_views(P[:k], W, H, M[:k])
    e.set_masks_bits(np.zeros((k, H, (W + 31) // 32), np.uint32))
    e.set_images(img[:k])
    if len(P) > k:
        e.append_views(P[k:], M[k:], mask_bits=np.zeros((len(P) - k, H, (W + 31) // 32), np.uint32), images_bgr=img[k:])
    e.upload_volumes(occ, np.full_like(occ, 0xffffffff))
    return e


def _check(e, CV, dims, s, P, M, W, H, img, occ, modes=(1, 2), tols=(0.0, 1.0, 2.0, INF)):
    X, Y, Z = dims
    for mode in modes:
        for tol in tols:
            e.color_visible(mode, tol)
            idx, rgbn = e.download_colors()
            ridx, rrgbn = CV.color_visible(X, Y, Z, s, P, M, W, H, img, occ, mode, tol)
            assert np.array_equal(idx, ridx), (mode, tol)
            assert np.array_equal(rgbn, rrgbn), (mode, tol, int((rgbn != rrgbn).any(1).sum()))
    return idx, rgbn


@pytest.mark.gpu
@pytest.mark.parametrize("ds", ["box", "human"])
def test_goldens_vs_oracle(A, CV, ds):
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, f"{ds}_views.npz"))
    X = Y = Z = 100
    s = F(0.28) / F(X)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(vs.P, vs.W, vs.H, vs.M)
        e.set_masks_bits(vs.mask_bits)
        e.set_images(vs.images_bgr)
        e.carve()
        occ = e.download_occupied()
        _check(e, CV, (X, Y, Z), s, vs.P, vs.M, vs.W, vs.H, vs.images_bgr, occ)
        for mode in (1, 2):  # tolerance = inf is vc_color on these captures
            e.color_visible(mode, INF)
            got = e.download_colors()
            e.color(mode)
            ref = e.download_colors()
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(70, 45, 3), (33, 20, 5), (100, 37, 1)], ids=["70x45x3", "33x20x5", "100x37x1"])
def test_ragged_synthetic(A, CV, dims):
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = dims
    w = Workload(64, 12, 320, 240, seed=3, dims=dims)
    img = w.images_bgr()
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(img)
        e.carve()
        occ = e.download_occupied()
        _check(e, CV, dims, w.s, w.P.reshape(-1, 3, 4), w.M.reshape(-1, 3, 4), w.W, w.H, img, occ)


@pytest.mark.gpu
def test_c3_whole(A, CV):
    from ar_voxel_project_b200.synth import CONFIGS, Workload
    w = Workload(**CONFIGS["C3"])
    img = w.images_bgr()
    with A.VoxelEngine(512, 512, 512, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(img)
        e.carve()
        occ = e.download_occupied()
        _check(e, CV, (512, 512, 512), w.s, w.P.reshape(-1, 3, 4), w.M.reshape(-1, 3, 4), w.W, w.H, img, occ, modes=(2,), tols=(2.0,))


@pytest.mark.gpu
def test_two_blocks_on_the_device(A, CV):
    P, M, W, H, img, occ = _block_scene()
    with _engine(A, BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ) as e:
        _check(e, CV, BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ)


@pytest.mark.gpu
def test_camera_inside_and_close_cameras(A, CV):
    """a camera inside the grid (pairs behind it are ineligible), and cameras so close that rectangles exceed 10^4 pixels
    (the warp-cooperative splat)"""
    X, Y, Z = 48, 40, 36
    s = F(0.01)
    vol = np.zeros((Z, Y, X), bool)
    vol[2:34, 2:38, 2:46] = True
    vol[10:26, 12:28, 14:34] = False
    occ = _words(vol)
    W, H = 640, 480
    c = _world(23.5, 19.5, 17.5, s)
    cams = [_look_at(c, _world(47, 19.5, 17.5, s), 100.0, W, H),             # inside the hollow
            _look_at(c, _world(23.5, 0, 17.5, s), 100.0, W, H),
            _look_at(_world(23.5, 19.5, -1.5, s), c, 5000.0, W, H),          # just outside the grid, long focal length
            _look_at(_world(-0.8, 19.5, 17.5, s), c, 4000.0, W, H)]
    P, M = np.stack([p for p, _ in cams]), np.stack([m for _, m in cams])
    img = np.random.default_rng(5).integers(0, 256, (len(P), H, W, 3), dtype=np.uint8)
    # the third camera is 3.5 voxel sizes from the nearest occupied plane: 5000 / 3.5 pixels per voxel size, so the rectangles
    # there (clipped to the 640 x 480 image) exceed 10^4 pixels
    assert (5000.0 / 3.5) ** 2 > 1e4
    with _engine(A, (X, Y, Z), s, P, M, W, H, img, occ) as e:
        _check(e, CV, (X, Y, Z), s, P, M, W, H, img, occ)


@pytest.mark.gpu
@pytest.mark.parametrize("WH,V", [((1, 1), 6), ((1 << 20, 1), 80)], ids=["1x1", "2^20x1"])
def test_image_shapes(A, CV, WH, V):
    """1x1 images, and 2^20 x 1 images: 4 MiB depth buffers, 80 views take two chunks of the 256 MiB budget"""
    W, H = WH
    X, Y, Z = 40, 30, 20
    s = F(0.01)
    vol = np.zeros((Z, Y, X), bool)
    vol[3:17, 4:26, 5:35] = True
    vol[6:14, 8:22, 20:28] = False
    occ = _words(vol)
    c = _world(19.5, 14.5, 9.5, s)
    rng = np.random.default_rng(7)
    cams = []
    for v in range(V):
        a = 2 * np.pi * v / V
        eye = c + 1.2 * np.array([np.cos(a), np.sin(a), -0.3 + 0.1 * (v % 3)])
        f = 0.3 * W if W > 1 else 1.0
        cams.append(_look_at(eye, c + rng.uniform(-0.02, 0.02, 3), f, W, H, cx=(W - 1) / 2, cy=(H - 1) / 2))
    P, M = np.stack([p for p, _ in cams]), np.stack([m for _, m in cams])
    img = rng.integers(0, 256, (V, H, W, 3), dtype=np.uint8)
    with _engine(A, (X, Y, Z), s, P, M, W, H, img, occ) as e:
        _check(e, CV, (X, Y, Z), s, P, M, W, H, img, occ, tols=(0.0, 2.0, INF))


def _ring_300(V=300):
    """V views around two blocks; view 256 + k repeats the position of view k, so an occluder's views lie on both sides of the
    256-view group boundary"""
    X, Y, Z = BLOCK_DIMS
    c = _world((X - 1) / 2, (Y - 1) / 2, (Z - 1) / 2, BLOCK_S)
    W, H = 96, 80
    cams = []
    for v in range(V):
        k = v % 256
        a = 2 * np.pi * k / 256
        cams.append(_look_at(c + 1.5 * np.array([np.cos(a), np.sin(a), -0.4 + 0.2 * np.sin(5 * a)]), c, 120.0, W, H))
    P, M = np.stack([p for p, _ in cams]), np.stack([m for _, m in cams])
    img = np.random.default_rng(11).integers(0, 256, (V, H, W, 3), dtype=np.uint8)
    return P, M, W, H, img, _blocks(BLOCK_DIMS, BLOCKS + [((15, 21), (0, 16), (6, 10))])


@pytest.mark.gpu
def test_300_views(A, CV):
    P, M, W, H, img, occ = _ring_300()
    with _engine(A, BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ) as e:
        idx, rgbn = _check(e, CV, BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ)
    _, _, obs = CV.color_visible(*BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ, 2, INF, observations=True)
    _, _, vis = CV.color_visible(*BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ, 2, 2.0, observations=True)
    hidden = obs & ~vis
    assert hidden[:, :256].any() and hidden[:, 256:].any()  # occluded pairs in both view groups


@pytest.mark.gpu
def test_records_feed_the_mesh(A, CV, oracle, tmp_path):
    P, M, W, H, img, occ = _ring_300(40)
    X, Y, Z = BLOCK_DIMS
    seen = np.full_like(occ, 0xffffffff)
    ridx, rrgbn = CV.color_visible(X, Y, Z, BLOCK_S, P, M, W, H, img, occ, 2, 2.0)
    rv, rc = oracle.marching_cubes(X, Y, Z, oracle.closure(X, Y, Z, oracle.dense_model(X, Y, Z, occ, seen, ridx, rrgbn), 3), 0.5)
    p = str(tmp_path / "ref.off")
    oracle.write_off(p, rv, rc, F(1.5) * BLOCK_S, (0.5, -0.25, 2.0))
    with _engine(A, BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ) as e:
        e.color_visible(2, 2.0)
        verts, rgb = e.mesh_from_volumes(True, True, 3, 0.5)
        assert np.array_equal(verts.view(np.uint32), rv.view(np.uint32)) and np.array_equal(rgb, rc)
        assert e.mesh_off(F(1.5) * BLOCK_S, (0.5, -0.25, 2.0)) == open(p, "rb").read()


@pytest.mark.gpu
def test_refusals_and_vc_color_after(A, CV):
    P, M, W, H, img, occ = _block_scene()
    with _engine(A, BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ) as e:
        e.color_visible(1, 2.0)
        before = e.download_colors()
        for mode, tol in ((2, float("nan")), (2, -1.0), (2, -1e-30), (3, 2.0), (0, 2.0)):
            with pytest.raises(A.VoxCarveError) as ei:
                e.color_visible(mode, tol)
            assert ei.value.code == 1
            after = e.download_colors()
            assert np.array_equal(after[0], before[0]) and np.array_equal(after[1], before[1])
        e.color(2)
        ref = e.download_colors()
        from oracle import oracle as O
        ridx, rrgbn = O.color(*BLOCK_DIMS, BLOCK_S, P, M, W, H, img, occ, 2)
        assert np.array_equal(ref[0], ridx) and np.array_equal(ref[1], rrgbn)
    import torch
    X, Y, Z = BLOCK_DIMS
    with A.VoxelEngine(X, Y, Z, BLOCK_S, z_begin=0, z_end=8) as e:  # a slab engine: refused, its vc_color records stay
        e.set_views(P, W, H, M)
        e.set_masks_bits(np.zeros((4, H, (W + 31) // 32), np.uint32))
        e.set_images(img)
        e.upload_volumes(occ[:8], np.full_like(occ[:8], 0xffffffff))
        halo = torch.from_numpy(occ[8].view(np.int32).copy()).cuda()
        e.import_halo(1, halo.data_ptr())
        e.color(1)
        before = e.download_colors()
        with pytest.raises(A.VoxCarveError) as ei:
            e.color_visible(2, 2.0)
        assert ei.value.code == 3
        after = e.download_colors()
        assert len(before[0]) > 0 and np.array_equal(after[0], before[0]) and np.array_equal(after[1], before[1])
    with A.VoxelEngine(X, Y, Z, BLOCK_S) as e:
        e.set_views(P, W, H, None)
        e.set_masks_bits(np.zeros((4, H, (W + 31) // 32), np.uint32))
        e.set_images(img)
        with pytest.raises(A.VoxCarveError) as ei:
            e.color_visible(2, 2.0)
        assert ei.value.code == 3
