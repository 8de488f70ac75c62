"""vc_mesh_from_volumes: the mesh of main.cpp:291-303 (handleUnseen -> applyClosure -> marchingCubes) straight from the bit
volumes and colour records.  Bit-exact, in emission order, against the dense chain on the device (vc_dense_from_volumes ->
vc_dense_closure -> vc_mc_mesh) and against the CPU oracle's restatement of the reference."""
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu

THRESHOLDS = (0.5, 1.0, 1e-30, 0.0, 1.5, float("nan"))


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


def _dense(e, ac, hu, k, thr):
    e.dense_from_volumes(apply_colors=ac, handle_unseen=hu)
    if k:
        e.dense_closure(k)
    return e.mc_mesh(thr)


def _oracle(oracle, X, Y, Z, occ, seen, idx, rgbn, ac, hu, k, thr):
    m = oracle.dense_model(X, Y, Z, occ, seen if hu else None, idx if ac else None, rgbn if ac else None)
    if k:
        m = oracle.closure(X, Y, Z, m, k)
    return oracle.marching_cubes(X, Y, Z, m, thr)


def _same(a, b, what=""):
    (va, ca), (vb, cb) = a, b
    assert va.shape == vb.shape, (what, va.shape, vb.shape)
    assert np.array_equal(va.view(np.uint32), vb.view(np.uint32)), what
    assert np.array_equal(ca, cb), what


def _all_against_dense(e, X, Y, Z, cases, oracle=None, vols=None):
    """every (colour mode, handle_unseen, closure_k, threshold) of `cases` on the engine's current volumes"""
    idx = rgbn = None
    for cm in sorted({c[0] for c in cases}):
        if cm:
            e.color(cm)
            idx, rgbn = e.download_colors()
        models = {}
        for c, hu, k, thr in cases:
            if c != cm:
                continue
            what = (cm, hu, k, thr)
            got = e.mesh_from_volumes(bool(cm), bool(hu), k, thr)
            _same(got, _dense(e, bool(cm), bool(hu), k, thr), what)
            if oracle is not None:
                if (hu, k) not in models:
                    m = oracle.dense_model(X, Y, Z, vols[0], vols[1] if hu else None, idx if cm else None, rgbn if cm else None)
                    models[(hu, k)] = oracle.closure(X, Y, Z, m, k) if k else m
                _same(got, oracle.marching_cubes(X, Y, Z, models[(hu, k)], thr), what)


@pytest.mark.parametrize("ds,dims", [("box", (50, 50, 25)), ("human", (50, 50, 25)), ("box", (100, 100, 100)), ("human", (100, 100, 100))])
def test_goldens_full_matrix_vs_oracle_and_dense(A, oracle, tmp_path, ds, dims):
    from ar_voxel_project_b200.mesh import write_off
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, f"{ds}_views.npz"))
    X, Y, Z = dims
    s = np.float32(0.28) / np.float32(X)
    cases = [(c, hu, k, t) for c in (0, 1, 2) for hu in (0, 1) for k in (0, 1, 3, 5) for t in THRESHOLDS]
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(vs.P, vs.W, vs.H, vs.M)
        e.set_masks_bits(vs.mask_bits)
        e.set_images(vs.images_bgr)
        e.carve()
        vols = e.download_occupied(), e.download_seen()
        _all_against_dense(e, X, Y, Z, cases, oracle, vols)
        e.color(2)
        verts, rgb = e.mesh_from_volumes(True, True, 3, 0.5)
        assert len(verts) > 0
        idx, rgbn = e.download_colors()
    # the package's .off writer on the device mesh against the oracle's C writer on the oracle mesh
    rv, rc = _oracle(oracle, X, Y, Z, vols[0], vols[1], idx, rgbn, True, True, 3, 0.5)
    a, b = str(tmp_path / "a.off"), str(tmp_path / "b.off")
    write_off(a, verts, rgb, np.float32(1.0) * s)
    oracle.write_off(b, rv, rc, np.float32(1.0) * s)
    assert open(a).read() == open(b).read()


def _views_for(A, X, Y, Z):
    from ar_voxel_project_b200.synth import Workload
    return Workload(max(X, Y, Z, 8), 4, 96, 64, seed=3, dims=(X, Y, Z))


@pytest.mark.parametrize("dims", [(1, 1, 1), (1, 7, 5), (31, 6, 5), (32, 5, 1), (33, 1, 6), (65, 9, 7), (64, 3, 4)])
def test_ragged_uploaded_volumes_vs_oracle_and_dense(A, oracle, dims):
    """ragged X (padding bits, words carried across in the x-dilation), Y or Z = 1, and uploaded states with carved-but-unseen
    voxels, for which handleUnseen sets alpha 1 (they join the mesh), next to all-carved and nothing-carved grids"""
    from ar_voxel_project_b200.synth import pack_bits
    X, Y, Z = dims
    w = _views_for(A, X, Y, Z)
    rng = np.random.default_rng(X * 7 + Y * 131 + Z)
    cases = [(c, hu, k, 0.5) for c in (0, 2) for hu in (0, 1) for k in (0, 3, 5)]
    states = [(rng.random((Z, Y, X)) < 0.5, rng.random((Z, Y, X)) < 0.7),      # random occupancy, random seen
              (rng.random((Z, Y, X)) < 0.05, rng.random((Z, Y, X)) < 0.9),     # sparse
              (np.zeros((Z, Y, X), bool), np.ones((Z, Y, X), bool)),            # all carved
              (np.ones((Z, Y, X), bool), np.zeros((Z, Y, X), bool)),            # nothing carved
              (np.zeros((Z, Y, X), bool), rng.random((Z, Y, X)) < 0.8)]        # carved but partly unseen
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_images(w.images_bgr())
        for occ, seen in states:
            vols = pack_bits(occ), pack_bits(seen)
            e.upload_volumes(*vols)
            _all_against_dense(e, X, Y, Z, cases, oracle, vols)


def test_object_touching_every_face_and_fast_carve(A, oracle):
    """an object cut by all six grid faces (vertices on original voxels whose empty corner lies outside the grid), then the state
    fastCarve leaves"""
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 70, 45, 38
    w = Workload(24, 6, 160, 120, seed=2, dims=(X, Y, Z))
    cases = [(c, hu, k, 0.5) for c in (0, 1, 2) for hu in (0, 1) for k in (0, 1, 3, 7)]
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(w.images_bgr())
        e.carve()
        occ = e.download_occupied()
        u = oracle.unpack(occ, X)
        assert u[0].any() and u[-1].any() and u[:, 0].any() and u[:, -1].any() and u[..., 0].any() and u[..., -1].any()
        _all_against_dense(e, X, Y, Z, cases, oracle, (occ, e.download_seen()))
        e.fast_carve()
        _all_against_dense(e, X, Y, Z, cases)


def test_noisy_silhouettes_256(A):
    from ar_voxel_project_b200.synth import Workload, noisy_masks
    w = Workload(256, 12, 320, 240, seed=5)
    bgr, _ = noisy_masks(w, seed=1)
    cases = [(2, 1, 3, 0.5), (2, 0, 5, 0.5), (1, 1, 0, 1.0), (0, 1, 1, 0.5), (0, 0, 15, 0.5)]
    with A.VoxelEngine(256, 256, 256, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bgr(bgr)
        e.set_images(w.images_bgr())
        e.carve()
        _all_against_dense(e, 256, 256, 256, cases)


def test_refusals_keep_the_previous_mesh(A):
    from ar_voxel_project_b200.synth import Workload
    w = Workload(40, 4, 96, 64, seed=1)
    with A.VoxelEngine(40, 40, 40, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(w.images_bgr())
        e.carve()
        e.color(2)
        ref = e.mesh_from_volumes(True, True, 3, 0.5)
        assert len(ref[0]) > 0
        for k in (2, -1, 17, 4):
            with pytest.raises(A.VoxCarveError) as ei:
                e.mesh_from_volumes(True, True, k, 0.5)
            assert ei.value.code == 1
            _same(e.download_mesh(len(ref[0])), ref, k)
        for k in (1, 3, 5, 15):
            e.mesh_from_volumes(False, True, k, 0.5, download=False)
        e.mesh_from_volumes(True, True, 3, 0.5, download=False)
        e.carve()                       # re-carve: the colour records are stale
        with pytest.raises(A.VoxCarveError) as ei:
            e.mesh_from_volumes(True, True, 3, 0.5)
        assert ei.value.code == 3
        _same(e.download_mesh(len(ref[0])), ref, "stale colours")
        e.reset()                       # no colours at all
        with pytest.raises(A.VoxCarveError) as ei:
            e.mesh_from_volumes(True, False, 0, 0.5)
        assert ei.value.code == 3
        _same(e.download_mesh(len(ref[0])), ref, "no colours")
    with A.VoxelEngine(40, 40, 40, w.s, z_begin=0, z_end=20) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.carve()
        with pytest.raises(A.VoxCarveError) as ei:
            e.mesh_from_volumes(False, True, 3, 0.5)
        assert ei.value.code == 3


def test_cpp_chain_writes_the_dense_chains_off(tmp_path, lib_built):
    from ar_voxel_project_b200.api import ViewSet
    vs = ViewSet.from_npz(os.path.join(GOLDEN, "box_views.npz"))
    X, Y, Z, s = 37, 30, 21, np.float32(0.008)
    case = tmp_path / "case.bin"
    with open(case, "wb") as f:
        np.array([X, Y, Z, vs.V, vs.W, vs.H], np.int32).tofile(f)
        np.array([s], np.float32).tofile(f)
        vs.P.astype(np.float32).tofile(f)
        vs.M.astype(np.float32).tofile(f)
        vs.mask_bits.astype(np.uint32).tofile(f)
        vs.images_bgr.astype(np.uint8).tofile(f)
    exe = str(tmp_path / "mesh_from_volumes")
    libdir = os.path.dirname(lib_built)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-pthread", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "mesh_from_volumes.cpp"), "-o", exe,
                           "-L", libdir, "-lvoxcarve", f"-Wl,-rpath,{libdir}"])
    a, b = tmp_path / "sparse.off", tmp_path / "dense.off"
    subprocess.check_call([exe, str(case), str(a), str(b)], stdout=subprocess.DEVNULL)
    ta = open(a).read()
    assert ta == open(b).read() and len(ta.splitlines()) > 100


def _carved(A, name, colour=True):
    from ar_voxel_project_b200.synth import CONFIGS, Workload
    w = Workload(**CONFIGS[name])
    e = A.VoxelEngine(w.X, w.Y, w.Z, w.s)
    e.set_views(w.P, w.W, w.H, w.M)
    e.set_masks_bits(w.mask_bits)
    if colour:
        e.set_images(w.images_bgr())
    e.carve()
    if colour:
        e.color(2)
    return w, e


def test_c4_full_size_vs_dense(A):
    _, e = _carved(A, "C4")
    with e:
        for ac, hu, k in ((True, True, 3), (False, False, 0)):
            got = e.mesh_from_volumes(ac, hu, k, 0.5)
            assert len(got[0]) > 0
            _same(got, _dense(e, ac, hu, k, 0.5), (ac, hu, k))


def _dilate_words(words, X, s):
    """E dilated by the (2s+1)^3 box, on packed words [Z][Y][Wx] with numpy shifts (independent of the kernel)"""
    w = words
    lo = np.zeros_like(w)
    hi = np.zeros_like(w)
    lo[..., 1:] = w[..., :-1]
    hi[..., :-1] = w[..., 1:]
    d = w.copy()
    for k in range(1, s + 1):
        d |= (w << np.uint32(k)) | (lo >> np.uint32(32 - k)) | (w >> np.uint32(k)) | (hi << np.uint32(32 - k))
    del lo, hi
    rem = X - 32 * (w.shape[-1] - 1)
    if rem < 32:
        d[..., -1] &= np.uint32((1 << rem) - 1)
    out = d.copy()
    for k in range(1, s + 1):
        out[:, k:] |= d[:, :-k]
        out[:, :-k] |= d[:, k:]
    d[...] = out
    for k in range(1, s + 1):
        out[k:] |= d[:-k]
        out[:-k] |= d[k:]
    return out


@pytest.fixture(scope="module")
def c5(A):
    """2048^3 x 72 views, carved and coloured (average): the dense Model (128 GiB, 256 GiB with the closure's second buffer) cannot
    be built on one B200, so here the mesh is checked against the cube-index classifier and against the oracle on crops"""
    w, e = _carved(A, "C5")
    with e:
        idx, rgbn = e.download_colors()
        yield w, e, e.download_occupied(), e.download_seen(), idx, rgbn


def test_c5_full_size_counts(A, c5):
    """triangle totals: without a closure against vc_mc_classify, with closure 3 against vc_mc_classify of an independently
    dilated occupancy uploaded into a second engine"""
    w, e, occ, seen, _, _ = c5
    n0 = e.mesh_from_volumes(False, False, 0, 0.5, download=False)
    e.mc_classify()
    assert n0 == e.download_mc()[2] > 0
    n3 = e.mesh_from_volumes(False, True, 3, 0.5, download=False)
    eff = occ | ~seen
    rem = w.X - 32 * (eff.shape[-1] - 1)
    if rem < 32:
        eff[..., -1] &= np.uint32((1 << rem) - 1)
    dil = _dilate_words(eff, w.X, 1)
    del eff
    with A.VoxelEngine(w.X, w.Y, w.Z, w.s) as e2:
        e2.upload_volumes(dil, dil)
        e2.mc_classify()
        assert n3 == e2.download_mc()[2] > n0 * 0.5


def _crop_bits(words, x0, y0, cw, ch, oracle):
    """bool[Z][ch][cw] of the voxels x0 .. x0+cw-1, y0 .. y0+ch-1 of packed words [Z][Y][Wx]"""
    j0, j1 = x0 // 32, (x0 + cw - 1) // 32 + 1
    b = oracle.unpack(np.ascontiguousarray(words[:, y0:y0 + ch, j0:j1]), (j1 - j0) * 32)
    return b[..., x0 - 32 * j0:x0 - 32 * j0 + cw]


def _inner(verts, lo_x, hi_x, lo_y, hi_y):
    """triangles whose vertices all lie on x in [lo_x+1, hi_x], y in [lo_y+1, hi_y]: their cell column (x, y) is certainly one of
    [lo_x, hi_x] x [lo_y, hi_y] (a cell's vertices sit on its corners x, x+1 and y, y+1)"""
    vx, vy = verts[:, :, 0], verts[:, :, 1]
    return (vx.min(1) >= lo_x + 1) & (vx.max(1) <= hi_x) & (vy.min(1) >= lo_y + 1) & (vy.max(1) <= hi_y)


@pytest.mark.parametrize("hu,k", [(True, 3), (False, 5)])
def test_c5_crops_vs_oracle(A, oracle, c5, hu, k):
    """full-Z crops of 24 x 24 columns across the object's silhouette edges, at grid corners and on grid faces: every triangle of
    the columns at least s+2 inside the crop (or on the grid's own border) equals, in order, vertex and colour, the oracle chain
    (dense Model + handleUnseen + applyClosure + marchingCubes) run on the crop with the GPU's colour records.  Flatten indices
    pass 2^32 here, so the records are found through 64-bit keys and a row table of 4 M + 1 rows."""
    from ar_voxel_project_b200.synth import pack_bits
    w, e, occ, seen, idx, rgbn = c5
    X, Y, Z = w.X, w.Y, w.Z
    s, C = (k - 1) // 2, 24
    verts, rgb = e.mesh_from_volumes(True, hu, k, 0.5)
    assert len(verts) > 0
    rx, ry, rz = (idx % X).astype(np.int64), ((idx // X) % Y).astype(np.int64), (idx // (X * Y)).astype(np.int64)
    seen_rec = np.flatnonzero(rgbn[:, 3] > 0)
    starts = [(0, 0), (X - C, Y - C), (0, Y - C), (X - C, 0), (X // 2 - C // 2, 0), (0, Y // 2 - C // 2)]
    for f in (0.1, 0.3, 0.5, 0.7, 0.9):   # centred on coloured surface voxels: the object's silhouette edges
        r = seen_rec[int(f * (len(seen_rec) - 1))]
        starts.append((int(min(max(rx[r] - C // 2, 0), X - C)), int(min(max(ry[r] - C // 2, 0), Y - C))))
    compared = 0
    for x0, y0 in starts:
        o = _crop_bits(occ, x0, y0, C, C, oracle)
        sn = _crop_bits(seen, x0, y0, C, C, oracle)
        m = (rx >= x0) & (rx < x0 + C) & (ry >= y0) & (ry < y0 + C)
        cidx = ((rx[m] - x0) + C * ((ry[m] - y0) + C * rz[m])).astype(np.uint64)
        rv, rc = _oracle(oracle, C, C, Z, pack_bits(o), pack_bits(sn), cidx, rgbn[m], True, hu, k, 0.5)
        rv = rv + np.array([x0, y0, 0], np.float32)
        lo_x = -1 if x0 == 0 else x0 + s + 2
        hi_x = X - 1 if x0 + C == X else x0 + C - s - 3
        lo_y = -1 if y0 == 0 else y0 + s + 2
        hi_y = Y - 1 if y0 + C == Y else y0 + C - s - 3
        sel_g, sel_o = _inner(verts, lo_x, hi_x, lo_y, hi_y), _inner(rv, lo_x, hi_x, lo_y, hi_y)
        _same((verts[sel_g], rgb[sel_g]), (rv[sel_o], rc[sel_o]), (x0, y0))
        compared += int(sel_g.sum())
        if (x0, y0) in starts[6:]:
            assert sel_g.sum() > 0, (x0, y0)
    assert compared > 1000
