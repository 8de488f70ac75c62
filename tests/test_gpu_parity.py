"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the golden fixtures.
Bit-exact: occupancy / seen volumes, colour records, cube-index histograms."""
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


def _carve(A, X, Y, Z, s, P, W, H, bits=None, bgr=None, M=None, z0=0, z1=None, mode=0, count=False):
    """carve with VC_EXACT (brick-classified) and check VC_EXACT_FLAT (every voxel-view) gives the same bits"""
    with A.VoxelEngine(X, Y, Z, s, z_begin=z0, z_end=z1) as e:
        e.set_views(P, W, H, M)
        if bits is not None:
            e.set_masks_bits(bits)
        else:
            e.set_masks_bgr(bgr)
        e.carve(mode, count_executed=count)
        out = e.download_occupied(), e.download_seen(), e.stats()
        if mode == 0 and count:  # a counting run cross-checks every decision of the per-voxel f32 filter against the exact evaluation
            assert out[2]["filter_mismatches"] == 0, f"f32 filter accepted {out[2]['filter_mismatches']} pixels the exact path rejects"
            assert out[2]["filter_slow_rows"] <= out[2]["filter_rows"]
        if mode == 0:
            e.reset()
            e.carve(2)
            assert np.array_equal(e.download_occupied(), out[0]), "VC_EXACT and VC_EXACT_FLAT disagree (occupied)"
            assert np.array_equal(e.download_seen(), out[1]), "VC_EXACT and VC_EXACT_FLAT disagree (seen)"
        return out


@pytest.mark.parametrize("ds", ["box", "human"])
def test_carve_matches_literal_cv2_golden(A, oracle, golden, ds):
    v, L = golden(f"{ds}_views.npz"), golden(f"{ds}_literal.npz")
    X, Y, Z, s = int(L["X"]), int(L["Y"]), int(L["Z"]), L["s"]
    occ, seen, _ = _carve(A, X, Y, Z, s, v["P"], int(v["W"]), int(v["H"]), bits=v["mask_bits"])
    assert np.array_equal(oracle.unpack(occ, X), L["occ"])
    assert np.array_equal(oracle.unpack(seen, X), L["seen"])


@pytest.mark.parametrize("ds,dims", [("box", (100, 100, 100)), ("human", (100, 100, 100)), ("box", (100, 100, 50))])
def test_carve_datasets_default_resolution(A, oracle, golden, ds, dims):
    """BASELINE configs[0], [1]: box / human at the default 100^3, s = 0.0028 (main.cpp:26-29)"""
    v = golden(f"{ds}_views.npz")
    X, Y, Z = dims
    s = np.float32(0.0028)
    ro, rs = oracle.carve(X, Y, Z, s, v["P"], int(v["W"]), int(v["H"]), mask_bits=v["mask_bits"], nthreads=0)
    occ, seen, st = _carve(A, X, Y, Z, s, v["P"], int(v["W"]), int(v["H"]), bits=v["mask_bits"], count=True)
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)
    assert 0 < st["executed_voxel_views"] <= st["nominal_voxel_views"] == X * Y * Z * int(v["V"])
    assert 0 < st["brick_corner_views"] < st["executed_voxel_views"]


@pytest.mark.parametrize("dims", [(1, 1, 1), (5, 3, 2), (31, 7, 3), (32, 4, 4), (33, 5, 2), (127, 9, 3), (129, 2, 5), (200, 3, 3), (64, 64, 64)])
def test_carve_ragged_grids_synthetic(A, oracle, dims):
    """X not a multiple of 32 / 128, single voxel, thin grids: padding bits stay 0"""
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = dims
    w = Workload(max(dims), 7, 320, 200, seed=5, dims=dims)
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits)
    occ, seen, _ = _carve(A, X, Y, Z, w.s, w.P, w.W, w.H, bits=w.mask_bits, count=True)
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)
    if X % 32:
        assert (occ[..., -1] >> np.uint32(X % 32)).max() == 0 and (seen[..., -1] >> np.uint32(X % 32)).max() == 0


def test_carve_bgr_masks_with_near_black_pixels(A, oracle, golden):
    from ar_voxel_project_b200.synth import unpack_bits
    v = golden("box_views.npz")
    W, H = int(v["W"]), int(v["H"])
    bg = unpack_bits(v["mask_bits"], W)
    rng = np.random.default_rng(11)
    bgr = rng.integers(0, 4, size=(*bg.shape, 3), dtype=np.uint8)
    bgr[..., 1] |= 1  # foreground: never all-zero, but nearly black
    bgr[bg] = 0
    s = np.float32(0.0056)
    ro, rs = oracle.carve(50, 50, 25, s, v["P"], W, H, mask_bgr=bgr)
    occ, seen, _ = _carve(A, 50, 50, 25, s, v["P"], W, H, bgr=bgr)
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)


def test_carve_adversarial_cameras(A, oracle):
    """behind-camera voxels still carve (no depth test, VoxelCarving.cpp:18-21); NaN/inf/zero-depth
    projections are out of bounds; pixel-edge ties follow round-half-away."""
    rng = np.random.default_rng(7)
    W, H, X, Y, Z = 64, 48, 40, 12, 9
    s = np.float32(0.25)
    P = []
    P.append(np.array([[0, 8, 0, 0.5], [0, 0, 8, 24.5], [0, 0, 0, 1]], np.float32))      # u = 8*x*s + .5 -> exact .5 ties
    P.append(np.array([[0, 4, 0, -0.5], [4, 0, 0, 1.5], [0, 0, 0, 1]], np.float32))      # ties at -0.5 / .5
    P.append(np.array([[30, 0, 0, 5], [0, 30, 0, 5], [0, 1, 0, -2.5]], np.float32))      # depth crosses zero inside the grid
    P.append(np.array([[30, 0, 0, 5], [0, 30, 0, 5], [0, 0, 0, 0]], np.float32))         # depth == 0 -> inf / NaN
    P.append(np.array([[np.nan, 0, 0, 5], [0, 30, 0, 5], [0, 0, 0, 1]], np.float32))     # NaN matrix
    P.append(np.array([[1e38, 1e38, 0, 0], [0, 30, 0, 5], [0, 0, 1e-38, 1e-38]], np.float32))  # overflow / denormal depth
    P.append(np.array([[-20, 3, 1, 30], [2, -25, 4, 40], [0.1, 0.2, -0.3, -1]], np.float32))   # camera behind: negative depth
    for _ in range(6):
        P.append((rng.standard_normal((3, 4)) * np.array([40, 40, 40, 20])).astype(np.float32))
    P = np.stack(P)
    bits = rng.integers(0, 2 ** 32, size=(len(P), H, (W + 31) // 32), dtype=np.uint64).astype(np.uint32)
    for v0 in range(len(P)):  # one view at a time, so a disagreement names its view
        ro, rs = oracle.carve(X, Y, Z, s, P[v0:v0 + 1], W, H, mask_bits=bits[v0:v0 + 1])
        occ, seen, _ = _carve(A, X, Y, Z, s, P[v0:v0 + 1], W, H, bits=bits[v0:v0 + 1], count=True)
        assert np.array_equal(occ, ro), f"occupied differs for adversarial view {v0}"
        assert np.array_equal(seen, rs), f"seen differs for adversarial view {v0}"
    ro, rs = oracle.carve(X, Y, Z, s, P, W, H, mask_bits=bits)
    occ, seen, _ = _carve(A, X, Y, Z, s, P, W, H, bits=bits)
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)


def test_view_ranges_accumulate_and_carve_is_idempotent(A, golden):
    """carving views one by one (the -intermediateMesh path, VoxelCarving.cpp:63-68) == one call; a
    second pass changes nothing"""
    v = golden("human_views.npz")
    W, H, V = int(v["W"]), int(v["H"]), int(v["V"])
    with A.VoxelEngine(100, 100, 60, 0.0028) as e:
        e.set_views(v["P"], W, H)
        e.set_masks_bits(v["mask_bits"])
        e.carve()
        occ, seen = e.download_occupied(), e.download_seen()
        e.carve()
        assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen)
        e.reset()
        for i in range(V):
            e.carve(0, i, i + 1)
        assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen)
        n_occ, n_seen = e.count_occupied()
        from ar_voxel_project_b200.synth import unpack_bits
        assert n_occ == unpack_bits(occ, 100).sum() and n_seen == unpack_bits(seen, 100).sum()


def test_z_slabs_tile_the_single_gpu_result(A, oracle):
    from ar_voxel_project_b200.synth import Workload
    w = Workload(96, 9, 320, 240, seed=2)
    full = _carve(A, 96, 96, 96, w.s, w.P, w.W, w.H, bits=w.mask_bits)
    for G in (2, 3, 8):
        edges = [round(i * 96 / G) for i in range(G + 1)]
        parts = [_carve(A, 96, 96, 96, w.s, w.P, w.W, w.H, bits=w.mask_bits, z0=a, z1=b) for a, b in zip(edges[:-1], edges[1:])]
        assert np.array_equal(np.concatenate([p[0] for p in parts]), full[0])
        assert np.array_equal(np.concatenate([p[1] for p in parts]), full[1])
    ro, rs = oracle.carve(96, 96, 96, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=40, z1=44)
    assert np.array_equal(full[0][40:44], ro) and np.array_equal(full[1][40:44], rs)


def test_config3_512cubed_properties_and_oracle_slab(A, oracle):
    """BASELINE configs[2] (512^3 x 36 views, 640x480) at full size: oracle on a 3-plane slab, plus
    size-independent properties (carved => seen, padding, monotone in views, slab == whole)."""
    from ar_voxel_project_b200.synth import Workload, CONFIGS, unpack_bits
    w = Workload(**CONFIGS["C3"])
    with A.VoxelEngine(512, 512, 512, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        e.carve(0, 0, 12)
        occ12 = e.download_occupied()
        e.carve(0, 12, -1)
        occ, seen = e.download_occupied(), e.download_seen()
        e.reset()
        e.carve(2)
        assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen)
    assert ((~occ) & (~seen)).max() == 0            # carved => seen
    assert (occ & ~occ12).max() == 0                # more views never un-carve
    frac = unpack_bits(occ[::8], 512).mean()
    assert 0.01 < frac < 0.25, frac
    for z0 in (0, 255, 509):
        ro, rs = oracle.carve(512, 512, 512, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=z0, z1=z0 + 3, nthreads=0)
        assert np.array_equal(occ[z0:z0 + 3], ro) and np.array_equal(seen[z0:z0 + 3], rs)


@pytest.mark.parametrize("ds", ["box", "human"])
def test_colour_and_mc_match_literal_golden_and_oracle(A, oracle, golden, ds):
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, f"{ds}_views.npz"))
    L = golden(f"{ds}_literal.npz")
    X, Y, Z, s = int(L["X"]), int(L["Y"]), int(L["Z"]), L["s"]
    sf = L["surf"].astype(np.int64)
    fl = sf[:, 0] + X * (sf[:, 1] + Y * sf[:, 2])
    order = np.argsort(fl)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(vs.P, vs.W, vs.H, vs.M)
        e.set_masks_bits(vs.mask_bits)
        e.set_images(vs.images_bgr)
        e.carve()
        for mode, key in ((1, "closest"), (2, "avg")):
            e.color(mode)
            idx, rgbn = e.download_colors()
            assert np.array_equal(idx, fl[order].astype(np.uint64))
            assert np.array_equal(rgbn[:, :3], L[key][order])          # tolerance: 0/255 (north_star allows 1/255)
            assert np.array_equal(rgbn[:, 3], np.minimum(L["nobs"][order], 255))
        e.mc_classify()
        hist, na, nt = e.download_mc()
        occ = e.download_occupied()
    rh, rna, rnt = oracle.mc_classify(X, Y, Z, occ)
    assert np.array_equal(hist, rh) and (na, nt) == (rna, rnt)


def test_config2_human_colour_default_resolution(A, oracle):
    """BASELINE configs[1]: human_dataset carve + ColorReconstruction at 100^3"""
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, "human_views.npz"))
    s = np.float32(0.0028)
    ro, _ = oracle.carve(100, 100, 100, s, vs.P, vs.W, vs.H, mask_bits=vs.mask_bits, nthreads=0)
    with A.VoxelEngine(100, 100, 100, s) as e:
        e.set_views(vs.P, vs.W, vs.H, vs.M)
        e.set_masks_bits(vs.mask_bits)
        e.set_images(vs.images_bgr)
        e.carve()
        assert np.array_equal(e.download_occupied(), ro)
        for mode in (1, 2):
            e.color(mode)
            idx, rgbn = e.download_colors()
            ridx, rrgbn = oracle.color(100, 100, 100, s, vs.P, vs.M, vs.W, vs.H, vs.images_bgr, ro, mode)
            assert np.array_equal(idx, ridx)
            assert np.abs(rgbn[:, :3].astype(int) - rrgbn[:, :3].astype(int)).max() <= 1   # north_star tolerance
            assert np.array_equal(rgbn, rrgbn)                                              # and in fact exact
        e.mc_classify()
        hist, na, nt = e.download_mc()
    rh, rna, rnt = oracle.mc_classify(100, 100, 100, ro)
    assert np.array_equal(hist, rh) and (na, nt) == (rna, rnt)


@pytest.mark.parametrize("dims", [(4, 4, 4), (31, 5, 7), (32, 6, 3), (33, 3, 3), (64, 9, 5), (95, 17, 11)])
def test_mc_classify_random_volumes(A, oracle, dims):
    """random occupancy incl. X = 31/32/33 (cell rows one longer than voxel rows)"""
    from ar_voxel_project_b200.synth import pack_bits
    X, Y, Z = dims
    rng = np.random.default_rng(X * 131 + Y)
    for p in (0.0, 0.5, 0.93, 1.0):
        occ = pack_bits(rng.random((Z, Y, X)) < p)
        with A.VoxelEngine(X, Y, Z, 1.0) as e:
            e.upload_volumes(occ, occ)
            e.mc_classify()
            hist, na, nt = e.download_mc()
        rh, rna, rnt = oracle.mc_classify(X, Y, Z, occ)
        assert np.array_equal(hist, rh) and (na, nt) == (rna, rnt)
        assert hist.sum() == (X + 1) * (Y + 1) * (Z + 1)


@pytest.mark.parametrize("dims", [(1088, 20, 3), (2100, 19, 2), (150, 300, 3), (160, 40, 33)])
def test_mc_and_surface_wide_and_ragged_volumes(A, oracle, dims):
    """shapes the warp-cooperative consumer kernels have to get right: more than 32 voxel-word columns (a warp's lane 0 then
    has a left neighbour word), X % 32 == 0 (cell c = X in a word of its own), rows that do not fill a thread's 4 words
    (Wx = 5), planes spanning several 1024-word blocks; random noise, solid boxes (faces parallel to x: 32 mixed cells per
    word) and an empty / a full grid.  Surface = occupied & !isInner is checked through vc_color's record indices."""
    from ar_voxel_project_b200.synth import Workload, pack_bits
    X, Y, Z = dims
    rng = np.random.default_rng(X + 7 * Y + 131 * Z)
    w = Workload(16, 2, 64, 48, seed=4)   # any two views: only the voxel set of the records is compared here
    vols = [rng.random((Z, Y, X)) < 0.5, rng.random((Z, Y, X)) < 0.97, np.zeros((Z, Y, X), bool), np.ones((Z, Y, X), bool)]
    box = np.zeros((Z, Y, X), bool)
    box[Z // 3:, Y // 4:Y - Y // 4, 5:X - 3] = True
    box[:, Y // 2, X // 2:X // 2 + 70] = False
    vols.append(box)
    for vol in vols:
        occ = pack_bits(vol)
        with A.VoxelEngine(X, Y, Z, 1e-3) as e:
            e.set_views(w.P, w.W, w.H, w.M)
            e.set_images(w.images_bgr())
            e.upload_volumes(occ, occ)
            e.mc_classify()
            hist, na, nt = e.download_mc()
            e.color(A._lib.VC_COLOR_AVG)
            idx, _ = e.download_colors()
        rh, rna, rnt = oracle.mc_classify(X, Y, Z, occ)
        assert np.array_equal(hist, rh) and (na, nt) == (rna, rnt)
        pad = np.pad(vol, 1)
        inner = pad[:-2, 1:-1, 1:-1] & pad[2:, 1:-1, 1:-1] & pad[1:-1, :-2, 1:-1] & pad[1:-1, 2:, 1:-1] & pad[1:-1, 1:-1, :-2] & pad[1:-1, 1:-1, 2:]
        ref_idx = np.flatnonzero((vol & ~inner).ravel()).astype(np.uint64)   # flatten = x + X*(y + Y*z) is the C order of [z][y][x]
        assert np.array_equal(idx, ref_idx)


def test_reference_named_api_on_model(A, oracle, golden):
    """carve / reconstructAvgColor / marchingCubesClassify on a host Model, as main.cpp:260-303 calls them"""
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, "box_views.npz"))
    L = golden("box_literal.npz")
    X, Y, Z, s = int(L["X"]), int(L["Y"]), int(L["Z"]), L["s"]
    m = A.Model(X, Y, Z, s)
    A.carve(vs, m)
    assert np.array_equal(m.occupied_grid(), L["occ"])
    assert np.array_equal(m.seen.reshape(Z, Y, X), L["seen"])
    A.reconstructAvgColor(vs, m)
    for (x, y, z), rgb, n in zip(L["surf"], L["avg"], L["nobs"]):
        exp = rgb if n > 0 else (50, 168, 141)
        assert tuple(m.get(x, y, z)[:3].astype(int)) == tuple(int(c) for c in exp)
    m.handleUnseen()
    hist, na, nt = A.marchingCubesClassify(m)
    rh, rna, rnt = oracle.mc_classify(X, Y, Z, __import__("ar_voxel_project_b200.synth", fromlist=["pack_bits"]).pack_bits(m.occupied_grid()))
    assert np.array_equal(hist, rh) and nt == rnt


def test_errors_are_loud(A):
    with pytest.raises(ValueError):
        A.Model(0, 1, 1, 0.1)
    with pytest.raises(A.VoxCarveError):
        A.VoxelEngine(4, 4, 4, -1.0)
    with A.VoxelEngine(4, 4, 4, 0.1) as e:
        with pytest.raises(A.VoxCarveError):
            e.carve()  # no views
        e.set_views(np.zeros((2, 12), np.float32), 8, 8)
        with pytest.raises(A.VoxCarveError):
            e.carve()  # no masks
        with pytest.raises(A.VoxCarveError):
            e.color(2)  # no images
    with A.VoxelEngine(4, 4, 8, 0.1, z_begin=2, z_end=4) as e:
        with pytest.raises(A.VoxCarveError):
            e.mc_classify()  # needs neighbour planes


def test_arithmetic_shortcuts_selftest(A):
    """shared-reciprocal divide == IEEE div.rn (bitwise) and the 5-instruction pixel index == (int)roundf + inside(),
    over 2 x 2^31 pseudo-random inputs incl. ties, edges, NaN/inf"""
    from ar_voxel_project_b200.engine import selftest
    for which in (0, 1):
        bad, checked = selftest(which, 1 << 31, seed=12345 + which)
        assert checked > (1 << 30) and bad == 0, (which, bad, checked)


def test_bound_whole_grid_buffer_slabs_in_place(A, oracle):
    """the multi-GPU data path on one GPU: two engines carve their z-slabs IN PLACE inside one caller-owned
    whole-grid buffer (vc_bind_volumes); after that the 'gathered' buffer serves neighbour planes to the
    colour and cube-index passes of both slabs, and the per-slab results add up to the whole-grid oracle."""
    import torch
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 90, 40, 33
    w = Workload(64, 6, 320, 240, seed=9, dims=(X, Y, Z))
    Wx = (X + 31) // 32
    occ_full = torch.zeros((Z, Y, Wx), dtype=torch.int32, device="cuda")
    seen_full = torch.zeros_like(occ_full)
    engines = []
    for z0, z1 in ((0, 16), (16, Z)):
        e = A.VoxelEngine(X, Y, Z, w.s, z_begin=z0, z_end=z1)
        e.bind_volumes(occ_full.data_ptr(), seen_full.data_ptr())
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(w.images_bgr())
        engines.append(e)
    for e in engines:
        e.carve()
        e.synchronize()
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits)
    assert np.array_equal(occ_full.cpu().numpy().view(np.uint32), ro)
    assert np.array_equal(seen_full.cpu().numpy().view(np.uint32), rs)
    with pytest.raises(A.VoxCarveError):
        engines[1].mc_classify()  # neighbour planes not declared valid yet
    hist = np.zeros(256, np.uint64)
    idx_all, rgbn_all = [], []
    for e in engines:
        e.set_gathered(True)
        e.mc_classify()
        h, _, _ = e.download_mc()
        hist += h
        e.color(2)
        i, c = e.download_colors()
        idx_all.append(i), rgbn_all.append(c)
    rh, rna, rnt = oracle.mc_classify(X, Y, Z, ro)
    assert np.array_equal(hist, rh)
    ridx, rrgbn = oracle.color(X, Y, Z, w.s, w.P, w.M, w.W, w.H, w.images_bgr(), ro, 2)
    assert np.array_equal(np.concatenate(idx_all), ridx) and np.array_equal(np.concatenate(rgbn_all), rrgbn)
    for e in engines:
        e.close()


@pytest.mark.parametrize("case", ["box24", "human28", "box100", "synth70", "origin_solid"])
def test_fast_carve_matches_oracle_bfs(A, oracle, golden, case):
    """fastCarve() (VoxelCarving.cpp:74-167): device flood fill == the oracle's literal BFS, occupied and seen"""
    from ar_voxel_project_b200.synth import Workload
    if case in ("box24", "human28", "box100"):
        ds = "human" if case.startswith("human") else "box"
        v = golden(f"{ds}_views.npz")
        P, W, H, bits = v["P"], int(v["W"]), int(v["H"]), v["mask_bits"]
        if case == "box100":
            X, Y, Z, s = 100, 100, 50, np.float32(0.0028)
        else:
            L = golden(f"{ds}_literal.npz")
            X, Y, Z, s = int(L["X"]), int(L["Y"]), int(L["Z"]), L["s"]
    else:
        X, Y, Z = (70, 33, 41)
        w = Workload(64, 9, 320, 240, seed=3, dims=(X, Y, Z))
        P, W, H, bits, s = w.P, w.W, w.H, w.mask_bits.copy(), w.s
        if case == "origin_solid":
            bits[:] = 0  # nothing is background: the origin is not carved, the BFS stops at once
    ro, rs = oracle.fast_carve(X, Y, Z, s, P, W, H, mask_bits=bits)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        e.fast_carve()
        occ, seen = e.download_occupied(), e.download_seen()
        assert e.stats()["flood_rounds"] >= 1
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)
    if case == "origin_solid":
        assert oracle.unpack(occ, X).all() and oracle.unpack(seen, X).sum() == 1
    with A.VoxelEngine(X, Y, 2 * Z, s, z_begin=0, z_end=Z) as e:
        with pytest.raises(A.VoxCarveError):
            e.fast_carve()  # a slab cannot flood from the origin


def test_planned_slabs_tile_the_grid_and_match(A, oracle):
    """vc_plan_slabs / vc_set_slab: balanced contiguous slabs (boundaries on 8-plane brick layers) carve to the same bits"""
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 96, 64, 160
    w = Workload(160, 8, 320, 240, seed=6, dims=(X, Y, Z))
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        e.carve()
        full = e.download_occupied(), e.download_seen()
        for n in (1, 2, 3, 5):
            b = e.plan_slabs(n)
            assert b[0] == 0 and b[-1] == Z and all(x < y for x, y in zip(b[:-1], b[1:])) and all(x % 8 == 0 for x in b[:-1])
        with pytest.raises(A.VoxCarveError):
            e.plan_slabs(Z + 1)
        b = e.plan_slabs(3)
        parts = []
        for z0, z1 in zip(b[:-1], b[1:]):
            e.set_slab(z0, z1)
            e.carve()
            parts.append((e.download_occupied(), e.download_seen()))
            assert parts[-1][0].shape[0] == z1 - z0
    assert np.array_equal(np.concatenate([p[0] for p in parts]), full[0])
    assert np.array_equal(np.concatenate([p[1] for p in parts]), full[1])
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=64, z1=70)
    assert np.array_equal(full[0][64:70], ro) and np.array_equal(full[1][64:70], rs)


def _off_text(tmp_path, name, verts, rgb, oracle, scale, t=(0.0, 0.0, 0.0)):
    p = str(tmp_path / name)
    oracle.write_off(p, verts, rgb, scale, t)
    return open(p).read()


@pytest.mark.parametrize("color_mode", [0, 1, 2])
def test_closure_and_marching_cubes_mesh_match_oracle(A, oracle, tmp_path, color_mode):
    """main.cpp:260-303 on the device: carve -> [colour] -> handleUnseen -> applyClosure(3) -> marchingCubes, compared
    with the oracle's restatement voxel by voxel (f32 RGBA, bit-exact) and triangle by triangle, and as .off text
    written by ar_voxel_project_b200.mesh.write_off (WriteMesh, MarchingCubes.h:59-87)."""
    from ar_voxel_project_b200.mesh import write_off
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, "box_views.npz"))
    X, Y, Z, s = 50, 50, 25, np.float32(0.0056)   # the benchmark's "medium" grid (main.cpp:362)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(vs.P, vs.W, vs.H, vs.M)
        e.set_masks_bits(vs.mask_bits)
        e.set_images(vs.images_bgr)
        e.carve()
        occ, seen = e.download_occupied(), e.download_seen()
        idx = rgbn = None
        if color_mode:
            e.color(color_mode)
            idx, rgbn = e.download_colors()
        e.dense_from_volumes(apply_colors=bool(color_mode), handle_unseen=True)
        ref = oracle.dense_model(X, Y, Z, occ, seen, idx, rgbn)
        assert np.array_equal(e.dense_download(), ref)
        with pytest.raises(A.VoxCarveError):
            e.dense_closure(2)            # even kernel size (Postprocessing3d.cpp:8-11)
        e.dense_closure(3)
        ref_c = oracle.closure(X, Y, Z, ref, 3)
        got_c = e.dense_download()
        assert np.array_equal(got_c.view(np.uint32), ref_c.view(np.uint32))
        verts, rgb = e.mc_mesh(0.5)
    rverts, rrgb = oracle.marching_cubes(X, Y, Z, ref_c, 0.5)
    assert verts.shape == rverts.shape and np.array_equal(verts, rverts) and np.array_equal(rgb, rrgb)
    out = str(tmp_path / "mesh.off")
    write_off(out, verts, rgb, scale=np.float32(1.0) * s)
    assert open(out).read() == _off_text(tmp_path, "ref.off", rverts, rrgb, oracle, np.float32(1.0) * s)


def test_mc_mesh_general_alpha_and_upload(A, oracle):
    """VertexInterp's interpolating branch (MarchingCubes.h:443-467): fractional alphas, default-colour rule, threshold != 0.5"""
    rng = np.random.default_rng(5)
    X, Y, Z = 13, 9, 7
    rgba = np.zeros((X * Y * Z, 4), np.float32)
    rgba[:, 3] = rng.choice([0.0, 0.25, 0.5, 0.75, 1.0], X * Y * Z)
    rgba[:, :3] = rng.integers(0, 256, (X * Y * Z, 3))
    rgba[rng.random(X * Y * Z) < 0.2, :3] = (50, 168, 141)
    rgba[rng.random(X * Y * Z) < 0.1, :3] = (204, 0, 0)
    for thr in (0.5, 0.3):
        with A.VoxelEngine(X, Y, Z, 1.0) as e:
            e.dense_upload(rgba)
            verts, rgb = e.mc_mesh(thr)
        rverts, rrgb = oracle.marching_cubes(X, Y, Z, rgba, thr)
        assert np.array_equal(verts, rverts) and np.array_equal(rgb, rrgb)


def test_soft_golden_box_mesh_on_device(A, oracle, golden):
    """Data/box_dataset/generated_models/1.off (-z=50, defaults): 49056 vertices / 16352 faces.  Poses come from a different
    OpenCV build, so this is a soft check: face count within 0.5 % and >= 97 % of the golden vertex lines present."""
    import json
    soft = json.load(open(os.path.join(GOLDEN, "soft_box_1off.json")))
    v = golden("box_views.npz")
    s = np.float32(0.0028)
    with A.VoxelEngine(100, 100, 50, s) as e:
        e.set_views(v["P"], int(v["W"]), int(v["H"]))
        e.set_masks_bits(v["mask_bits"])
        e.carve()
        e.dense_from_volumes(handle_unseen=True)
        e.dense_closure(3)
        verts, rgb = e.mc_mesh(0.5)
    assert abs(len(verts) - soft["faces"]) / soft["faces"] < 0.005
    assert (rgb == (50, 168, 141)).all()   # 1.off faces are all MODEL_COLOR


@pytest.mark.parametrize("dims", [(64, 40, 300), (96, 33, 70), (40, 20, 31)])
def test_carve_download_chunked_equals_plain(A, oracle, dims):
    """vc_carve_download (z-chunks, D2H overlapped with the next chunk) == vc_carve + downloads == oracle slab"""
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = dims
    w = Workload(max(dims), 7, 320, 240, seed=8, dims=dims)
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        e.carve()
        occ, seen = e.download_occupied(), e.download_seen()
        for _ in range(2):
            e.reset()
            o2, s2 = e.carve_download()
            assert np.array_equal(o2, occ) and np.array_equal(s2, seen)
        e.carve_download(o2, s2)  # accumulate on the carved state: nothing changes
        assert np.array_equal(o2, occ) and np.array_equal(s2, seen)
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=Z // 2, z1=Z // 2 + 3)
    assert np.array_equal(occ[Z // 2:Z // 2 + 3], ro) and np.array_equal(seen[Z // 2:Z // 2 + 3], rs)


def _oracle_planes(oracle, w, X, Y, Z, planes, occ, seen):
    """compare the given z-planes (grouped into contiguous runs) of occ / seen with the oracle; returns #planes compared"""
    planes = sorted({int(z) for z in planes if 0 <= z < Z})
    runs, a = [], 0
    while a < len(planes):
        b = a
        while b + 1 < len(planes) and planes[b + 1] == planes[b] + 1:
            b += 1
        runs.append((planes[a], planes[b] + 1))
        a = b + 1
    for z0, z1 in runs:
        ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=z0, z1=z1, nthreads=0)
        assert np.array_equal(occ[z0:z1], ro), f"occupied differs from the oracle in planes [{z0},{z1})"
        assert np.array_equal(seen[z0:z1], rs), f"seen differs from the oracle in planes [{z0},{z1})"
    return len(planes)


def _object_edge_planes(occ):
    """first / last z-plane that still holds an occupied voxel seen by some view: the silhouette-edge planes of the object"""
    nz = np.flatnonzero(occ.reshape(occ.shape[0], -1).any(axis=1))
    return (int(nz[0]), int(nz[-1])) if len(nz) else (0, 0)


def test_config4_1024cubed_full_size_properties(A, oracle):
    """BASELINE configs[3] at full size (1024^3 x 72 views x 1920x1080) on one GPU: VC_EXACT == VC_EXACT_FLAT bit for bit,
    carved => seen, every filter decision cross-checked, and >= 64 z-planes against the oracle: the grid's first / last planes,
    every boundary +-1 the slab planner picks for 2, 4 and 8 GPUs, the planes where the object starts / ends, and a regular
    stride through the volume."""
    from ar_voxel_project_b200.synth import Workload, CONFIGS
    w = Workload(**CONFIGS["C4"])
    with A.VoxelEngine(1024, 1024, 1024, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        bounds = sorted({b for n in (2, 4, 8) for b in e.plan_slabs(n)})
        occ, seen = e.carve_download()
        n_occ, n_seen = e.count_occupied()
        e.reset()
        e.carve(2)
        assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen)
        e.reset()
        e.carve(0, count_executed=True)  # every decision of the per-voxel f32 filter checked against the exact evaluation
        st = e.stats()
        assert st["filter_mismatches"] == 0 and st["filter_rows"] > 0
        assert st["filter_slow_rows"] < 0.5 * st["filter_rows"], (st["filter_slow_rows"], st["filter_rows"])
        assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen)
    assert ((~occ) & (~seen)).max() == 0
    assert 0.02 < n_occ / 1024 ** 3 < 0.25 and n_seen <= 1024 ** 3
    # planes that still hold voxels no view carved because no view sees them do not count as the object: use the seen ones
    lo, hi = _object_edge_planes(occ & seen)
    planes = {0, 1, 1022, 1023, 511, 512}
    planes |= {b + d for b in bounds for d in (-1, 0)}
    planes |= {z + d for z in (lo, hi) for d in (-2, -1, 0, 1, 2)}
    planes |= set(range(5, 1024, 24))
    n = _oracle_planes(oracle, w, 1024, 1024, 1024, planes, occ, seen)
    assert n >= 64, n


def test_config5_2048cubed_full_size_properties(A, oracle):
    """BASELINE configs[4] at full size (2048^3 x 72 views x 3840x2160; 1 GiB per bit volume, 2.4 GB of summed-area tables)
    on one GPU.  The reference cannot even index this grid (`int flatten`, Model.h:104-106), so the oracle slab check is the
    only possible pin: VC_EXACT == VC_EXACT_FLAT bit for bit over the whole volume, carved => seen, and two-plane oracle slabs
    at z = 0, the middle (1023/1024), the end (2046), the planner's 8-GPU boundaries and the object's first / last planes."""
    from ar_voxel_project_b200.synth import Workload, CONFIGS
    w = Workload(**CONFIGS["C5"])
    N = 2048
    with A.VoxelEngine(N, N, N, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        bounds = e.plan_slabs(8)
        e.carve()
        occ, seen = e.download_occupied(), e.download_seen()
        n_occ, n_seen = e.count_occupied()
        e.reset()
        e.carve(2)
        flat_occ = e.download_occupied()
        assert np.array_equal(flat_occ, occ)
        del flat_occ
        flat_seen = e.download_seen()
        assert np.array_equal(flat_seen, seen)
        del flat_seen
        e.reset()
        o2, s2 = e.carve_download()   # the chunked path crosses 2^31 bits per chunk too
        assert np.array_equal(o2, occ) and np.array_equal(s2, seen)
        del o2, s2
        e.mc_classify()
        hist, na, nt = e.download_mc()
    assert int(hist.sum()) == (N + 1) ** 3 and nt > 0
    assert ((~occ) & (~seen)).max() == 0
    assert 0.02 < n_occ / N ** 3 < 0.25 and n_seen <= N ** 3
    assert int(np.unpackbits(occ[1000:1002].view(np.uint8)).sum()) > 0
    lo, hi = _object_edge_planes(occ & seen)
    planes = set()
    for z0 in [0, 1023, 2046, lo - 1, hi] + [b - 1 for b in bounds[1:-1]]:
        planes |= {z0, z0 + 1}
    n = _oracle_planes(oracle, w, N, N, N, planes, occ, seen)
    assert n >= 16, n
    # the cube-index histogram of a two-plane slab against the oracle's (cells between planes 1023 and 1024 are interior to it)
    ro = occ[1022:1026]
    rh, _, _ = oracle.mc_classify(N, N, 4, np.ascontiguousarray(ro))
    with A.VoxelEngine(N, N, 4, w.s) as e2:
        e2.upload_volumes(np.ascontiguousarray(ro), np.zeros_like(ro))
        e2.mc_classify()
        h2, _, _ = e2.download_mc()
    assert np.array_equal(h2, rh)


def test_device_undistort_matches_cv2_kat_and_raw_mask_path(A, oracle, golden):
    """SURVEY §8f-4: cv::undistort on the device. (1) vc_undistort_bgr == cv2 4.13.0 outputs byte for byte on every KAT case;
    (2) raw (distorted) masks / images handed to the engine give the same bit masks / images as undistorting with the oracle."""
    import cv2  # PNG decode of the fixture only
    from ar_voxel_project_b200.engine import undistort_bgr
    from ar_voxel_project_b200.synth import pack_bits
    z = golden("undistort_kat.npz")
    for n in z["names"]:
        src, dst = cv2.imdecode(z[f"{n}_src"], 1), cv2.imdecode(z[f"{n}_dst"], 1)
        assert np.array_equal(undistort_bgr(src, z[f"{n}_K"], z[f"{n}_dist"]), dst), n
    raw = np.stack([cv2.imdecode(z["box_mask0000_src"], 1), cv2.imdecode(z["human_mask_5_src"], 1)])
    img = np.stack([cv2.imdecode(z["box_image0003_src"], 1)] * 2)
    K, dist = z["box_mask0000_K"], z["box_mask0000_dist"]
    und = np.stack([oracle.undistort(m, K, dist) for m in raw])
    v = golden("box_views.npz")
    with A.VoxelEngine(40, 40, 20, 0.007) as e:
        e.set_views(v["P"][:2], 640, 480, v["M"][:2])
        with pytest.raises(A.VoxCarveError):
            e.set_masks_raw(raw)  # no calibration yet
        e.set_calibration(K, dist)
        e.set_masks_raw(raw)
        assert np.array_equal(e.download_masks(), pack_bits((und == 0).all(-1)))
        e.set_images_raw(img)
        assert np.array_equal(e.download_images()[0], cv2.imdecode(z["box_image0003_dst"], 1))
        e.carve()
        occ = e.download_occupied()
    ro, _ = oracle.carve(40, 40, 20, np.float32(0.007), v["P"][:2], 640, 480, mask_bgr=und)
    assert np.array_equal(occ, ro)


@pytest.mark.parametrize("seed", range(int(os.environ.get("VC_STRESS_SEEDS", "10"))))
def test_hierarchical_carve_random_stress(A, oracle, seed):
    """random grids / slabs / view counts / image sizes / camera placements (incl. cameras inside or grazing the grid, so that
    depth changes sign inside bricks and whole bricks fall outside the image): VC_EXACT == VC_EXACT_FLAT == oracle"""
    rng = np.random.default_rng(1000 + seed)
    X, Y, Z = (int(rng.integers(1, 140)), int(rng.integers(1, 75)), int(rng.integers(1, 75)))
    V = int(rng.choice([1, 2, 7, 31, 32, 33, 40, 65, 70]))
    W, H = int(rng.integers(8, 300)), int(rng.integers(8, 200))
    s = np.float32(rng.uniform(0.002, 0.02))
    ext = np.array([Y * s, X * s, Z * s])  # world extents: (y*s, x*s, -z*s)
    centre = np.array([ext[0] / 2, ext[1] / 2, -ext[2] / 2])
    P = []
    for v in range(V):
        kind = rng.integers(0, 4)
        if kind == 0:    # outside, looking at the grid
            pos = centre + rng.normal(size=3) * ext.max() * rng.uniform(1.0, 3.0)
        elif kind == 1:  # inside the grid
            pos = centre + (rng.random(3) - 0.5) * ext * 0.8
        elif kind == 2:  # on a face
            pos = centre + (rng.random(3) - 0.5) * ext
            pos[rng.integers(0, 3)] = centre[0] + ext[0] / 2
        else:            # far away, narrow view: most bricks outside the image
            pos = centre + rng.normal(size=3) * ext.max() * 6
        target = centre + (rng.random(3) - 0.5) * ext * (0.2 if kind != 3 else 3.0)
        zc = target - pos
        zc /= np.linalg.norm(zc) + 1e-12
        up = rng.normal(size=3)
        xc = np.cross(zc, up)
        xc /= np.linalg.norm(xc) + 1e-12
        yc = np.cross(zc, xc)
        R = np.stack([xc, yc, zc])
        f = W * rng.uniform(0.4, 2.5)
        K = np.array([[f, 0, W / 2 + rng.normal() * 3], [0, f * rng.uniform(0.9, 1.1), H / 2 + rng.normal() * 3], [0, 0, 1]])
        M = np.concatenate([R, (-R @ pos)[:, None]], axis=1).astype(np.float32)
        P.append(oracle.gemm3x3_3x4(K.astype(np.float32), M))
    P = np.stack(P)
    # blobby random masks: large background / foreground regions plus noise, so that whole bricks are decided
    yy, xx = np.mgrid[0:H, 0:W]
    bg = np.zeros((V, H, W), bool)
    for v in range(V):
        cx, cy, r = rng.uniform(0, W), rng.uniform(0, H), rng.uniform(0.1, 0.8) * max(W, H)
        bg[v] = ((xx - cx) ** 2 + (yy - cy) ** 2) > r * r
        bg[v] ^= rng.random((H, W)) < rng.choice([0.0, 0.0, 0.02])
    from ar_voxel_project_b200.synth import pack_bits
    bits = pack_bits(bg)
    z0 = int(rng.integers(0, Z))
    z1 = int(rng.integers(z0 + 1, Z + 1))
    ro, rs = oracle.carve(X, Y, Z, s, P, W, H, mask_bits=bits, z0=z0, z1=z1)
    occ, seen, _ = _carve(A, X, Y, Z, s, P, W, H, bits=bits, z0=z0, z1=z1, count=True)   # runs VC_EXACT (filter cross-checked) and VC_EXACT_FLAT
    assert np.array_equal(occ, ro), f"occupied differs (X,Y,Z,V,W,H,z0,z1)={(X, Y, Z, V, W, H, z0, z1)}"
    assert np.array_equal(seen, rs), f"seen differs (X,Y,Z,V,W,H,z0,z1)={(X, Y, Z, V, W, H, z0, z1)}"
    # and in two view ranges that split a 32-view word
    if V > 2:
        with A.VoxelEngine(X, Y, Z, s, z_begin=z0, z_end=z1) as e:
            e.set_views(P, W, H)
            e.set_masks_bits(bits)
            cut = int(rng.integers(1, V))
            e.carve(0, 0, cut)
            e.carve(0, cut, -1)
            assert np.array_equal(e.download_occupied(), ro) and np.array_equal(e.download_seen(), rs)


@pytest.mark.parametrize("mode", [0, 2])
def test_carve_accumulates_onto_uploaded_state_like_the_reference(A, oracle, mode):
    """vc_upload_volumes + vc_carve = carve() called on a Model that already holds state.  The reference projects EVERY voxel,
    occupied or not, and marks it seen when its pixel is inside the image (VoxelCarving.cpp:45-54): a voxel that arrives carved but
    unseen must come out seen if any view has it inside, although every kernel skips already-carved voxels."""
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 70, 37, 29
    w = Workload(70, 9, 200, 150, seed=3, dims=(X, Y, Z))
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits)
    rng = np.random.default_rng(7)
    Wx = (X + 31) // 32
    valid = np.full(Wx, 0xffffffff, np.uint32)
    valid[-1] = (1 << (X - 32 * (Wx - 1))) - 1 if X % 32 else 0xffffffff
    occ0 = rng.integers(0, 2 ** 32, size=(Z, Y, Wx), dtype=np.uint64).astype(np.uint32) & valid
    seen0 = rng.integers(0, 2 ** 32, size=(Z, Y, Wx), dtype=np.uint64).astype(np.uint32) & valid
    occ0[: Z // 3] = 0          # a block that is carved and unseen as a whole (whole bricks of it)
    seen0[: Z // 3] = 0
    assert ((~occ0) & (~seen0) & valid).any()
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        e.upload_volumes(occ0, seen0)
        e.carve(mode)
        occ, seen = e.download_occupied(), e.download_seen()
        assert np.array_equal(occ, occ0 & ro), "occupied: uploaded state AND what the views carve"
        assert np.array_equal(seen, seen0 | rs), "seen: uploaded state OR every voxel some view has inside its image"
        e.upload_volumes(occ0, seen0)
        o2, s2 = e.carve_download(mode=mode)
        assert np.array_equal(o2, occ) and np.array_equal(s2, seen)


def test_engines_sharing_a_device_keep_their_own_views(A, oracle):
    """the view tables live in per-device __constant__ memory shared by every engine on the GPU: two engines with DIFFERENT
    views, driven alternately without synchronising in between, must each carve with their own"""
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 96, 64, 48
    wa = Workload(96, 12, 320, 240, seed=1, dims=(X, Y, Z))
    wb = Workload(96, 5, 256, 200, seed=2, dims=(X, Y, Z))
    ra = oracle.carve(X, Y, Z, wa.s, wa.P, wa.W, wa.H, mask_bits=wa.mask_bits)
    rb = oracle.carve(X, Y, Z, wb.s, wb.P, wb.W, wb.H, mask_bits=wb.mask_bits)
    with A.VoxelEngine(X, Y, Z, wa.s) as ea, A.VoxelEngine(X, Y, Z, wb.s) as eb:
        ea.set_views(wa.P, wa.W, wa.H, wa.M), ea.set_masks_bits(wa.mask_bits), ea.set_images(wa.images_bgr())
        eb.set_views(wb.P, wb.W, wb.H, wb.M), eb.set_masks_bits(wb.mask_bits), eb.set_images(wb.images_bgr())
        for _ in range(6):   # launches of one engine still in flight when the other uploads its tables
            ea.reset(), ea.carve(2)
            eb.reset(), eb.carve(2)
            ea.reset(), ea.carve(0), ea.color(2)
            eb.reset(), eb.carve(0), eb.color(1)
        for e, r, w, mode in ((ea, ra, wa, 2), (eb, rb, wb, 1)):
            assert np.array_equal(e.download_occupied(), r[0]) and np.array_equal(e.download_seen(), r[1])
            idx, rgbn = e.download_colors()
            ridx, rrgbn = oracle.color(X, Y, Z, w.s, w.P, w.M, w.W, w.H, w.images_bgr(), r[0], mode)
            assert np.array_equal(idx, ridx) and np.array_equal(rgbn, rrgbn)


def _whole_grid_reference(A, w, X, Y, Z, with_images=True):
    """single-engine results of the consumers on the whole grid: occupied, seen, cube-index histogram, colour records (avg, closest)"""
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.carve()
        occ, seen = e.download_occupied(), e.download_seen()
        e.mc_classify()
        hist, na, nt = e.download_mc()
        cols = {}
        if with_images:
            e.set_images(w.images_bgr())
            for mode in (2, 1):
                e.color(mode)
                cols[mode] = e.download_colors()
    return occ, seen, hist, nt, cols


@pytest.mark.parametrize("bounds", [[0, 13, 40], [0, 8, 9, 24, 40], [0, 1, 2, 40]])
def test_one_plane_halos_replace_the_gather_for_colour_and_cube_index(A, oracle, bounds):
    """SURVEY §8e: the consumers of a slab need ONE neighbour plane of `occupied` on each side, not the whole grid.  Engines on
    slabs (incl. one-plane slabs) of one device swap those planes (vc_exchange_halos_peer); their cube-index histograms then sum
    to the whole grid's and their colour records concatenate to it, bit for bit - with slab-sized AND with bound whole-grid volumes."""
    import torch
    from ar_voxel_project_b200.engine import exchange_halos_peer
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 70, 44, 40
    w = Workload(70, 6, 240, 180, seed=5, dims=(X, Y, Z))
    occ, seen, hist, nt, cols = _whole_grid_reference(A, w, X, Y, Z)
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits)
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)
    rh, _, rnt = oracle.mc_classify(X, Y, Z, ro)
    assert np.array_equal(hist, rh) and nt == rnt
    for bound_full in (False, True):
        engines, fulls = [], []
        try:
            for z0, z1 in zip(bounds[:-1], bounds[1:]):
                e = A.VoxelEngine(X, Y, Z, w.s, z_begin=z0, z_end=z1)
                engines.append(e)
                if bound_full:  # every engine its own whole-grid buffer, as separate GPUs would have; garbage outside the slab
                    f = [torch.randint(-2 ** 31, 2 ** 31 - 1, (Z, Y, (X + 31) // 32), dtype=torch.int32, device="cuda") for _ in range(2)]
                    fulls.append(f)
                    e.bind_volumes(f[0].data_ptr(), f[1].data_ptr())
                e.set_views(w.P, w.W, w.H, w.M)
                e.set_masks_bits(w.mask_bits)
                e.set_images(w.images_bgr())
                e.carve()
            if len(engines) > 1:
                with pytest.raises(A.VoxCarveError):   # no halos yet: a slab cannot classify its last cell plane
                    engines[0].mc_classify()
            exchange_halos_peer(engines[::-1])          # any order
            tot = np.zeros(256, np.uint64)
            for e in engines:
                e.mc_classify()
                tot += e.download_mc()[0]
            assert np.array_equal(tot, hist), f"cube-index histograms of the slabs do not sum to the grid's (bound_full={bound_full})"
            for mode in (2, 1):
                idx, rgbn = [], []
                for e in engines:
                    e.color(mode)
                    i, c = e.download_colors()
                    idx.append(i), rgbn.append(c)
                assert np.array_equal(np.concatenate(idx), cols[mode][0]) and np.array_equal(np.concatenate(rgbn), cols[mode][1])
            assert np.array_equal(np.concatenate([e.download_occupied() for e in engines]), occ)
            # a new carve invalidates the imported planes
            engines[0].reset(), engines[0].carve()
            if len(engines) > 1:
                with pytest.raises(A.VoxCarveError):
                    engines[0].mc_classify()
            # explicit export / import of single planes does the same job (here through device pointers of the same GPU)
            if len(engines) > 1:
                engines[0].synchronize(), engines[1].synchronize()
                engines[0].import_halo(1, engines[1].export_halo(0))
                engines[0].mc_classify()
                with pytest.raises(A.VoxCarveError):
                    engines[0].import_halo(0, engines[1].export_halo(0))  # plane -1 is outside the grid
        finally:
            for e in engines:
                e.close()


def test_nccl_two_ranks_halos_gather_bitwise(A, tmp_path):
    """VERDICT r1 #1c: two processes, one GPU each, NCCL inside libvoxcarve.so (vc_comm_init / vc_exchange_halos / vc_gather /
    vc_comm_allreduce_u64): planned (ragged) slabs are carved, halos exchanged, consumers run on the slabs, the grid gathered -
    and every word compared with the single-GPU result and oracle planes (tests/nccl_slab_worker.py writes the verdicts)."""
    import json
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (NCCL refuses two ranks on one device); a 2-GPU log is kept in profiles/")
    from conftest import ROOT
    port = 29500 + os.getpid() % 2000
    out = tmp_path / "nccl"
    out.mkdir()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "nccl_slab_worker.py"), str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for rank in range(2):
        v = json.load(open(out / f"rank{rank}.json"))
        assert v["ok"], v
        assert v["world"] == 2 and v["nccl_version"] > 0


@pytest.mark.parametrize("dims,slab", [((64, 64, 64), None), ((100, 37, 45), None), ((33, 9, 10), None), ((130, 70, 50), (13, 41)), ((5, 3, 2), None)])
def test_sparse_download_expands_to_the_dense_result(A, oracle, dims, slab):
    """vc_carve_download_sparse: flag byte per brick + words of the listed bricks only; expanded on the host it is the same
    pair of volumes carve + download delivers (and the oracle computes) - on ragged grids, slabs, grids smaller than a brick"""
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = dims
    z0, z1 = slab if slab else (0, Z)
    w = Workload(max(dims), 8, 256, 192, seed=11, dims=dims)
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=z0, z1=z1)
    with A.VoxelEngine(X, Y, Z, w.s, z_begin=z0, z_end=z1) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        flags, listed, words = e.carve_download_sparse()
        occ, seen = e.expand_sparse(flags, listed, words)
        assert np.array_equal(occ, ro) and np.array_equal(seen, rs)
        assert np.array_equal(e.download_occupied(), ro)          # the device volumes are complete too
        assert len(listed) == int(((flags & 8) != 0).sum())
        assert len(set(listed.tolist())) == len(listed)
        assert ((flags.reshape(-1)[listed] & 8) != 0).all()
        # sparse bytes vs dense bytes
        assert flags.nbytes + listed.nbytes + words.nbytes <= 2 * occ.nbytes + flags.nbytes + 4096
        # room for one listed brick too few: VC_ERR_CAPACITY, nothing half-written is reported as a result
        if len(listed) > 1:
            import ctypes as C
            n = C.c_uint64()
            small_l, small_w = np.empty(len(listed) - 1, np.uint32), np.empty((len(listed) - 1) * 128, np.uint32)
            e.reset()
            rc = e._lib.vc_carve_download_sparse(e._h, C.c_void_p(flags.ctypes.data), flags.size, C.c_void_p(small_l.ctypes.data), C.c_void_p(small_w.ctypes.data),
                                                 len(listed) - 1, C.byref(n))
            assert rc == A._lib.VC_ERR_CAPACITY and n.value == len(listed)
        # not a fresh carve: the sparse form cannot describe it
        import ctypes as C
        n = C.c_uint64()
        rc = e._lib.vc_carve_download_sparse(e._h, C.c_void_p(flags.ctypes.data), flags.size, C.c_void_p(listed.ctypes.data), C.c_void_p(words.ctypes.data), len(listed), C.byref(n))
        assert rc == A._lib.VC_ERR_STATE


def test_rectangles_beyond_the_16_bit_table_are_left_to_the_children(A, oracle):
    """the summed-area tables are kept modulo 2^16: a (super-)brick whose pixel rectangle holds 2^16 pixels or more cannot be
    counted and must stay undecided - close cameras on a large image make whole super-bricks project to > 256 x 256 pixels;
    the volumes still equal the oracle's and the flat kernel's"""
    from ar_voxel_project_b200.synth import pack_bits
    X, Y, Z, W, H = 256, 64, 64, 1024, 768
    s = np.float32(0.004)
    rng = np.random.default_rng(21)
    ext = np.array([Y * s, X * s, Z * s])
    centre = np.array([ext[0] / 2, ext[1] / 2, -ext[2] / 2])
    P = []
    for v in range(6):
        pos = centre + rng.normal(size=3) * ext.max() * (0.55 if v < 4 else 2.0)   # four cameras right at the grid, two further away
        zc = centre + (rng.random(3) - 0.5) * ext * 0.3 - pos
        zc /= np.linalg.norm(zc)
        xc = np.cross(zc, rng.normal(size=3))
        xc /= np.linalg.norm(xc)
        R = np.stack([xc, np.cross(zc, xc), zc])
        f = W * 1.4
        K = np.array([[f, 0, W / 2], [0, f, H / 2], [0, 0, 1]])
        M = np.concatenate([R, (-R @ pos)[:, None]], axis=1).astype(np.float32)
        P.append(oracle.gemm3x3_3x4(K.astype(np.float32), M))
    P = np.stack(P)
    yy, xx = np.mgrid[0:H, 0:W]
    bg = np.stack([((xx - W * (0.3 + 0.1 * v)) ** 2 + (yy - H / 2) ** 2) > (0.35 * H) ** 2 for v in range(6)])
    bg[1] = True      # one view that is background everywhere: carves whatever it sees, in rectangles of any size
    bg[2] = False     # and one that is foreground everywhere
    bits = pack_bits(bg)
    ro, rs = oracle.carve(X, Y, Z, s, P, W, H, mask_bits=bits, nthreads=0)
    occ, seen, st = _carve(A, X, Y, Z, s, P, W, H, bits=bits, count=True)
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)


def test_masks_from_page_locked_memory_without_a_sync(A, oracle):
    """page-locked host masks (bits or 8UC3) uploaded asynchronously with the carve enqueued right behind them (the end-to-end
    path of bench.py): same device masks, same carve as the synchronous path"""
    import torch
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 80, 50, 40
    w = Workload(80, 11, 300, 220, seed=13, dims=(X, Y, Z))   # 11 views: groups of 2, 3, 3, 3
    ro, rs = oracle.carve(X, Y, Z, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits)
    bits_p = torch.from_numpy(w.mask_bits.view(np.int32).copy()).pin_memory()
    bgr_p = torch.from_numpy(w.mask_bgr()).pin_memory()
    with A.VoxelEngine(X, Y, Z, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        for kind in ("bits", "bgr", "bits"):
            if kind == "bits":
                e.set_masks_bits_async(bits_p)
            else:
                e.set_masks_bgr(bgr_p, sync=False)
            e.reset()
            e.carve()          # enqueued right behind the uploads
            assert np.array_equal(e.download_occupied(), ro) and np.array_equal(e.download_seen(), rs), kind
            assert np.array_equal(e.download_masks(), w.mask_bits), kind


def test_peer_gather_assembles_the_grid_in_every_engine(A, oracle):
    """vc_gather_peer: engines of one process (here: three slabs on one device) pull each other's slabs into their whole-grid
    buffers; every engine then holds the single-engine volumes and runs its consumers on the gathered grid"""
    from ar_voxel_project_b200.engine import gather_peer
    from ar_voxel_project_b200.synth import Workload
    X, Y, Z = 70, 44, 40
    w = Workload(70, 6, 240, 180, seed=5, dims=(X, Y, Z))
    occ, seen, hist, nt, _ = _whole_grid_reference(A, w, X, Y, Z, with_images=False)
    bounds = [0, 9, 26, 40]
    engines = []
    try:
        for z0, z1 in zip(bounds[:-1], bounds[1:]):
            e = A.VoxelEngine(X, Y, Z, w.s, z_begin=z0, z_end=z1)
            e.alloc_full_volumes()
            e.set_views(w.P, w.W, w.H, w.M), e.set_masks_bits(w.mask_bits)
            e.carve()
            engines.append(e)
        with pytest.raises(A.VoxCarveError):
            engines[1].download_full(0)       # not gathered yet
        gather_peer(engines[::-1], occupied=True, seen=True)
        tot = np.zeros(256, np.uint64)
        for e in engines:
            assert np.array_equal(e.download_full(0), occ) and np.array_equal(e.download_full(1), seen)
            e.mc_classify()
            tot += e.download_mc()[0]
        assert np.array_equal(tot, hist)
        with pytest.raises(A.VoxCarveError):
            gather_peer(engines[:2])          # the slabs must tile the grid
    finally:
        for e in engines:
            e.close()


def test_fill_schemes_and_volume_memory_agree(A, oracle):
    """The fresh carve's fill (blind 'carved and seen' pass next to the classification + patch) with the volumes in compressible
    memory when the GPU grants it, against the same in plain cudaMalloc memory (VOXCARVE_COMPRESSIBLE=0: read once per process,
    hence the subprocesses) and against the oracle - whole grid, a ragged slab with a partial last word, a grid whose rows are
    not whole quads (no blind pass there), twice in a row (graph replay)."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    script = r'''
import hashlib, json, sys
import numpy as np
sys.path.insert(0, %r)
import ar_voxel_project_b200 as A
from ar_voxel_project_b200.synth import Workload
out = {}
for name, dims, slab in (("cube", (256, 256, 256), None), ("slab7", (200, 130, 150), (37, 120)), ("slabq", (250, 70, 90), (13, 77))):
    w = Workload(max(dims), 10, 320, 240, seed=5, dims=dims)
    z0, z1 = slab if slab else (0, dims[2])
    with A.VoxelEngine(*dims, w.s, z_begin=z0, z_end=z1) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        hs = []
        for rep in range(2):
            e.reset()
            e.carve(0)
            hs.append(hashlib.sha256(e.download_occupied().tobytes() + e.download_seen().tobytes()).hexdigest())
        assert hs[0] == hs[1]
        out[name] = hs[0]
        out[name + "_compressible"] = int(e.stats()["volumes_compressible"])
print(json.dumps(out))
''' % ROOT
    res = {}
    for tag, env in (("default", {}), ("blind_plain_memory", {"VOXCARVE_COMPRESSIBLE": "0"})):
        r = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600, env={**os.environ, **env})
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        res[tag] = json.loads(r.stdout.strip().splitlines()[-1])
    for name in ("cube", "slab7", "slabq"):
        assert res["default"][name] == res["blind_plain_memory"][name], (name, res)
    assert res["blind_plain_memory"]["cube_compressible"] == 0
    # ... and the default against the oracle (the other parity tests all run the default too)
    import hashlib
    from ar_voxel_project_b200.synth import Workload
    dims, (z0, z1) = (250, 70, 90), (13, 77)
    w = Workload(max(dims), 10, 320, 240, seed=5, dims=dims)
    ro, rs = oracle.carve(*dims, w.s, w.P, w.W, w.H, mask_bits=w.mask_bits, z0=z0, z1=z1)
    assert hashlib.sha256(ro.tobytes() + rs.tobytes()).hexdigest() == res["default"]["slabq"]
