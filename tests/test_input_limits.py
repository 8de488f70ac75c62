"""The ends of the C ABI's input range, bit for bit against the CPU oracle: up to 256 views per engine (every word of the 256-bit
undecided-view mask of a brick, view indices above 127 in the narrow fields of the classifier and the per-voxel queue), images
from 1x1 up to 2^20 pixels wide or tall (the f32 filter's radius grows with the image size, pixel coordinates near 2^20 have an
f32 ulp of 1/8), summed-area tables at the 2^31-element row-offset limit and views whose table starts past 2^31 elements, and
vc_set_views calls that are refused and must leave the engine as it was.

Every carve runs three ways: VC_EXACT with every per-voxel filter decision checked against the exact evaluation, VC_EXACT through
the cached CUDA graph, and VC_EXACT_FLAT (every voxel-view evaluated); all three must give the same bits."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F = np.float32


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


# ---- helpers -------------------------------------------------------------------------------------------------------------------
def _run_all_modes(e, v0=0, v1=-1):
    """carve the engine's views [v0, v1) from a fresh state in the three modes; -> (occupied, seen, stats of the counting run)"""
    e.reset()
    e.carve(0, v0, v1, count_executed=True)
    st = e.stats()
    assert st["filter_mismatches"] == 0, f"f32 filter accepted {st['filter_mismatches']} pixels the exact path rejects"
    occ, seen = e.download_occupied(), e.download_seen()
    e.reset()
    e.carve(0, v0, v1)   # through the cached graph
    assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen), "VC_EXACT: graph and counting run disagree"
    e.reset()
    e.carve(2, v0, v1)
    assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen), "VC_EXACT and VC_EXACT_FLAT disagree"
    return occ, seen, st


def _carve(A, X, Y, Z, s, P, W, H, bits, z0=0, z1=None):
    with A.VoxelEngine(X, Y, Z, s, z_begin=z0, z_end=z1) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        return _run_all_modes(e)


def _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen, z0=0, z1=None, what=""):
    ro, rs = oracle.carve(X, Y, Z, s, P, W, H, mask_bits=bits, z0=z0, z1=z1, nthreads=0)
    assert np.array_equal(occ, ro), f"occupied differs from the oracle {what}"
    assert np.array_equal(seen, rs), f"seen differs from the oracle {what}"
    return ro, rs


def _grid_centre(X, Y, Z, s):
    """world point of the grid's centre; world = (y s, x s, -z s)"""
    return np.array([(Y - 1) * float(s) / 2, (X - 1) * float(s) / 2, -(Z - 1) * float(s) / 2])


def _look_at(eye, target, fx, fy, cx, cy):
    """-> (P, M) float32 3x4, P = K M evaluated like cv::gemm (synth.gemm_k_m_f32)"""
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


def _ring(X, Y, Z, s, V, W, H, n_base=None, span=0.6, seed=0):
    """V cameras on a ring around the grid, looking at its centre; the grid's projection covers about `span` of the image
    (each axis on its own, so wide and tall images are spanned too).  With n_base, view v is a copy of base camera v % n_base
    whose principal point and position are jittered below a pixel: all copies of a base see the same silhouette edge."""
    rng = np.random.default_rng(seed)
    c = _grid_centre(X, Y, Z, s)
    ext = float(s) * max(X, Y, Z) * 1.5
    dist = 3.0 * ext
    nb = n_base or V
    P, M = [], []
    for v in range(V):
        b = v % nb
        az, el = 2 * np.pi * (b + 0.3) / nb, np.deg2rad(25.0 if b % 2 else 55.0)
        eye = c + dist * np.array([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), -np.sin(el)])
        fx, fy = span * W * dist / ext, span * H * dist / ext
        if n_base:
            eye = eye + rng.uniform(-1, 1, 3) * dist * 1e-4
            jx, jy = rng.uniform(-0.5, 0.5, 2)
        else:
            jx = jy = 0.0
        p, m = _look_at(eye, c, fx, fy, W / 2 + jx, H / 2 + jy)
        P.append(p), M.append(m)
    return np.stack(P), np.stack(M)


def _ellipse_bits(W, H, cx, cy, rx, ry, rng=None, n_specks=0):
    """uint32[H][ceil(W/32)] bit mask (1 = background) of a foreground ellipse, built from the rows' foreground intervals without
    a boolean image; plus n_specks random background pixels"""
    Ww = (W + 31) // 32
    out = np.empty((H, Ww), np.uint32)
    x0 = np.arange(Ww, dtype=np.int64) * 32
    one = np.uint64(1)
    valid = (one << np.clip(W - x0, 0, 32).astype(np.uint64)) - one
    step = max(1, (1 << 22) // Ww)
    for r0 in range(0, H, step):
        y = np.arange(r0, min(H, r0 + step), dtype=np.float64)
        t = 1.0 - ((y - cy) / ry) ** 2
        dx = np.where(t > 0, rx * np.sqrt(np.maximum(t, 0)), -1.0)
        lo = np.where(t > 0, np.ceil(cx - dx), 0).astype(np.int64)
        hi = np.where(t > 0, np.floor(cx + dx) + 1, 0).astype(np.int64)
        a = np.clip(lo[:, None] - x0, 0, 32).astype(np.uint64)
        b = np.clip(hi[:, None] - x0, 0, 32).astype(np.uint64)
        fg = ((one << b) - one) & ~((one << a) - one)
        out[r0:r0 + len(y)] = (~fg & valid).astype(np.uint32)
    if n_specks:
        xs, ys = rng.integers(0, W, n_specks), rng.integers(0, H, n_specks)
        np.bitwise_or.at(out, (ys, xs >> 5), (np.uint32(1) << (xs & 31).astype(np.uint32)))
    return out


def _view_masks(V, W, H, n_base, seed, specks=0.002):
    """per-view masks: one disc per base camera (radius differs by base), so all copies of a base are undecided on the same
    bricks, and per-view background specks, so that every view carves voxels of its own"""
    rng = np.random.default_rng(seed)
    r = min(W, H)
    return np.stack([_ellipse_bits(W, H, W / 2, H / 2, r * (0.16 + 0.02 * (v % n_base)), r * (0.18 + 0.015 * (v % n_base)),
                                   rng, int(specks * W * H)) for v in range(V)])


def _random_bits(rng, V, W, H):
    """uniformly random bit masks, padding bits of the last word clear"""
    bits = rng.integers(0, 2 ** 32, size=(V, H, (W + 31) // 32), dtype=np.uint64).astype(np.uint32)
    if W % 32:
        bits[..., -1] &= np.uint32((1 << (W % 32)) - 1)
    return bits


MANY_GRIDS = [((96, 64, 48), None), ((130, 70, 50), (7, 43))]


# ---- many views --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [96, 97, 128, 160, 255, 256])
@pytest.mark.parametrize("gi", [0, 1], ids=["96x64x48", "130x70x50_slab"])
def test_many_views_full_masks(A, oracle, V, gi):
    """jittered copies of a few base cameras: listed bricks carry up to 256 undecided views, every word of their mask set"""
    (X, Y, Z), slab = MANY_GRIDS[gi]
    z0, z1 = slab or (0, Z)
    s = F(0.28 / 96)
    W, H, nb = 320, 240, 6
    P, _ = _ring(X, Y, Z, s, V, W, H, n_base=nb, seed=V)
    bits = _view_masks(V, W, H, nb, seed=V + 1)
    occ, seen, st = _carve(A, X, Y, Z, s, P, W, H, bits, z0, z1)
    _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen, z0, z1)
    assert st["bricks_listed"] > 0
    n_occ = int(oracle.unpack(occ, X).sum())
    assert 0 < n_occ < X * Y * (z1 - z0)


@pytest.mark.parametrize("k", [0, 31, 32, 95, 96, 127, 128, 191, 192, 223, 224, 254, 255])
def test_one_carving_view_among_256(A, oracle, k):
    """every view but k sees all foreground: only view k can carve, so a dropped or shifted mask word at any level shows"""
    X, Y, Z = 96, 64, 48
    s = F(0.28 / 96)
    W, H, V, nb = 320, 240, 256, 6
    P, _ = _ring(X, Y, Z, s, V, W, H, n_base=nb, seed=3)
    bits = np.zeros((V, H, (W + 31) // 32), np.uint32)
    bits[k] = _ellipse_bits(W, H, W / 2 + 3, H / 2 - 2, 0.17 * H, 0.2 * H, np.random.default_rng(k), 150)
    occ, seen, _ = _carve(A, X, Y, Z, s, P, W, H, bits)
    ro, _ = _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen, what=f"(carving view {k})")
    assert not oracle.unpack(ro, X).all(), "view k must carve something"


def test_view_ranges_of_256_views(A, oracle):
    """ranges cut at 32-view words, at odd places, and starting at >= 128 (the v0 offset of the level-1 pass) == the single call"""
    X, Y, Z = 96, 64, 48
    s = F(0.28 / 96)
    W, H, V, nb = 320, 240, 256, 6
    P, _ = _ring(X, Y, Z, s, V, W, H, n_base=nb, seed=5)
    bits = _view_masks(V, W, H, nb, seed=6)
    cuts_list = [list(range(0, 257, 32)), [0, 200, 256], [0, 1, 97, 128, 129, 255, 256], [0, 160, 224, 256]]
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        occ, seen, _ = _run_all_modes(e)
        _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen)
        for cuts in cuts_list:
            for mode in (0, 2):
                e.reset()
                for a, b in zip(cuts[:-1], cuts[1:]):
                    e.carve(mode, a, b)
                assert np.array_equal(e.download_occupied(), occ) and np.array_equal(e.download_seen(), seen), (cuts, mode)
        for a, b in ((128, 256), (200, 256), (129, 193), (255, 256)):   # a range alone == the oracle on those views
            o, sn, _ = _run_all_modes(e, a, b)
            _check_oracle(oracle, X, Y, Z, s, P[a:b], W, H, bits[a:b], o, sn, what=f"views [{a},{b})")


def test_colour_mc_sparse_with_256_views(A, oracle):
    """colour records of voxels in front of all 256 cameras: the stored count saturates at 255, the average divides by 256"""
    from ar_voxel_project_b200.synth import images
    X, Y, Z = 64, 48, 40
    s = F(0.28 / 64)
    W, H, V, nb = 160, 120, 256, 8
    P, M = _ring(X, Y, Z, s, V, W, H, n_base=nb, seed=7)
    bits = _view_masks(V, W, H, nb, seed=8, specks=0.0005)
    img = images(V, W, H, seed=9)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(P, W, H, M)
        e.set_masks_bits(bits)
        e.set_images(img)
        occ, seen, _ = _run_all_modes(e)
        ro, _ = _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen)
        for mode in (2, 1):
            e.color(mode)
            idx, rgbn = e.download_colors()
            ridx, rrgbn = oracle.color(X, Y, Z, s, P, M, W, H, img, ro, mode)
            assert np.array_equal(idx, ridx) and np.array_equal(rgbn, rrgbn), f"colour mode {mode}"
            # a record whose voxel is inside all 256 images: its count is stored as 255, its average is over 256 samples
            full = np.flatnonzero(rgbn[:, 3] == 255)
            assert len(full) > 0
            i = int(idx[full[0]])
            x, y, z = i % X, (i // X) % Y, i // (X * Y)
            assert sum(oracle.pixel_of(P[v], x, y, z, s, W, H)[0] for v in range(V)) == V
        e.mc_classify()
        hist, na, nt = e.download_mc()
        rh, rna, rnt = oracle.mc_classify(X, Y, Z, ro)
        assert np.array_equal(hist, rh) and (na, nt) == (rna, rnt)
        flags, listed, words = e.carve_download_sparse()
        so, ss = e.expand_sparse(flags, listed, words)
        assert np.array_equal(so, occ) and np.array_equal(ss, seen)


def test_fast_carve_with_256_views(A, oracle):
    X, Y, Z = 80, 60, 44
    s = F(0.28 / 80)
    W, H, V, nb = 200, 150, 256, 5
    P, _ = _ring(X, Y, Z, s, V, W, H, n_base=nb, seed=11)
    bits = _view_masks(V, W, H, nb, seed=12)
    ro, rs = oracle.fast_carve(X, Y, Z, s, P, W, H, mask_bits=bits)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        e.fast_carve()
        assert np.array_equal(e.download_occupied(), ro) and np.array_equal(e.download_seen(), rs)


def test_two_engines_with_256_and_255_views_share_a_device(A, oracle):
    """each engine's launches take the whole constant bank over from the other one's, without a synchronisation in between"""
    from ar_voxel_project_b200.synth import images
    X, Y, Z = 96, 64, 48
    s = F(0.28 / 96)
    W, H = 160, 120
    cfg = []
    for V, seed in ((256, 21), (255, 22)):
        P, M = _ring(X, Y, Z, s, V, W, H, n_base=7, seed=seed)
        bits = _view_masks(V, W, H, 7, seed=seed + 100)
        img = images(V, W, H, seed=seed)
        r = oracle.carve(X, Y, Z, s, P, W, H, mask_bits=bits, nthreads=0)
        cfg.append((P, M, bits, img, r))
    with A.VoxelEngine(X, Y, Z, s) as ea, A.VoxelEngine(X, Y, Z, s) as eb:
        for e, (P, M, bits, img, _) in zip((ea, eb), cfg):
            e.set_views(P, W, H, M), e.set_masks_bits(bits), e.set_images(img)
        for _ in range(4):
            ea.reset(), ea.carve(2)
            eb.reset(), eb.carve(2)
            ea.reset(), ea.carve(0), ea.color(2)
            eb.reset(), eb.carve(0), eb.color(1)
        for e, (P, M, bits, img, r), mode in ((ea, cfg[0], 2), (eb, cfg[1], 1)):
            assert np.array_equal(e.download_occupied(), r[0]) and np.array_equal(e.download_seen(), r[1])
            idx, rgbn = e.download_colors()
            ridx, rrgbn = oracle.color(X, Y, Z, s, P, M, W, H, img, r[0], mode)
            assert np.array_equal(idx, ridx) and np.array_equal(rgbn, rrgbn)


def test_changing_view_count_on_one_engine(A, oracle):
    """256 -> 3 -> 256 views with new masks each time: the cached graph is re-keyed and the tables reallocated"""
    X, Y, Z = 96, 64, 48
    s = F(0.28 / 96)
    W, H = 240, 180
    with A.VoxelEngine(X, Y, Z, s) as e:
        for V, seed in ((256, 31), (3, 32), (256, 33)):
            P, _ = _ring(X, Y, Z, s, V, W, H, n_base=min(V, 6), seed=seed)
            bits = _view_masks(V, W, H, min(V, 6), seed=seed + 50)
            e.set_views(P, W, H)
            e.set_masks_bits(bits)
            occ, seen, _ = _run_all_modes(e)
            _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen, what=f"with {V} views")


# ---- image shapes ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("WH", [(1, 1), (1, 37), (37, 1), (2, 2), (31, 5), (32, 7), (33, 3)])
def test_tiny_images(A, oracle, WH):
    """fewer rows than the SAT builder's warps, a single word column, the direct-row path; the grid's projection is larger than
    the image, so every view cuts through it"""
    W, H = WH
    X, Y, Z = 40, 30, 24
    s = F(0.28 / 40)
    V = 6
    P, _ = _ring(X, Y, Z, s, V, W, H, span=2.5)
    bits = _random_bits(np.random.default_rng(W * 100 + H), V, W, H)
    bits[0] = 0                     # one view foreground only: seen, never carves
    occ, seen, _ = _carve(A, X, Y, Z, s, P, W, H, bits)
    ro, rs = _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen)
    n_seen = int(oracle.unpack(rs, X).sum())
    assert 0 < n_seen < X * Y * Z, "the image must cover part of the grid"


def _tie_cameras(W, H):
    """dyadic cameras with voxel size 0.25: every coordinate along the long axis is k + 0.5 exactly, once around the middle of the
    image (|c| > 2^19 when the side is 2^20) and once crossing the far edge (c = side - 0.5 rounds to side: outside); the other
    coordinate is 24.5 - 2z (ties, part of them above the image)"""
    out = []
    wide = W >= H
    n = W if wide else H
    for off in (float(n // 2) + 0.5, float(n) - 100.5):
        if wide:   # u = 8 wx + off = 2x + off, v = 8 wz + 24.5 = 24.5 - 2z
            out.append(np.array([[0, 8, 0, off], [0, 0, 8, 24.5], [0, 0, 0, 1]], F))
        else:      # u = 24.5 - 2z, v = 8 wy + off = 2y + off
            out.append(np.array([[0, 0, 8, 24.5], [8, 0, 0, off], [0, 0, 0, 1]], F))
    return np.stack(out)


@pytest.mark.parametrize("WH", [(65537, 48), (1 << 20, 64), (48, 65537), (40, 1 << 20)], ids=["w65537", "w2p20", "h65537", "h2p20"])
def test_wide_and_tall_images(A, oracle, WH):
    W, H = WH
    rng = np.random.default_rng(W + H)
    # (1) perspective cameras whose projections span the long side; an elliptic silhouette plus 2 % background noise, so every
    #     voxel-view goes through the per-voxel filter
    X, Y, Z = 96, 64, 48
    s = F(0.28 / 96)
    V = 4
    P, _ = _ring(X, Y, Z, s, V, W, H, span=0.9)
    bits = np.stack([_ellipse_bits(W, H, W / 2, H / 2, 0.3 * W, 0.3 * H, rng, int(0.02 * W * H)) for _ in range(V)])
    occ, seen, st = _carve(A, X, Y, Z, s, P, W, H, bits)
    _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen, what="(perspective views)")
    assert 0 < int(oracle.unpack(occ, X).sum()) < X * Y * Z
    # (2) exact .5 ties far from the origin and at the far edge: round half away from zero
    P = _tie_cameras(W, H)
    X, Y, Z = (96, 4, 30) if W >= H else (4, 96, 30)
    s = F(0.25)
    bits = _random_bits(rng, len(P), W, H)
    occ, seen, _ = _carve(A, X, Y, Z, s, P, W, H, bits)
    ro, rs = _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen, what="(tie views)")
    # the far-edge view sees its voxels up to coordinate side - 1.5 and none at side - 0.5 (which rounds to side)
    n = W if W >= H else H
    ok, px, py, uv = oracle.pixel_of(P[1], 50, 50, 12, s, W, H)   # x = 50 (wide) / y = 50 (tall): coordinate side - 0.5
    assert not ok and (px if W >= H else py) == n and float(uv[0 if W >= H else 1]) == n - 0.5


def test_sat_row_offsets_at_the_2p31_limit(A, oracle):
    """W = 2^20: pitch = 1 048 608, so H = 2046 is the tallest accepted image (pitch * (H + 1) < 2^31); one view there (a 4.3 GB
    table) against the oracle"""
    W, H = 1 << 20, 2046
    X, Y, Z = 128, 96, 64
    s = F(0.28 / 128)
    P, _ = _ring(X, Y, Z, s, 1, W, H, span=0.9, seed=41)
    bits = _ellipse_bits(W, H, W / 2 + 0.3, H / 2, 0.3 * W, 0.32 * H, np.random.default_rng(42), 200000)[None]
    with A.VoxelEngine(X, Y, Z, s) as e:
        with pytest.raises(A.VoxCarveError):
            e.set_views(P, W, H + 1)
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        occ, seen, _ = _run_all_modes(e)
    _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen)
    assert 0 < int(oracle.unpack(occ, X).sum()) < X * Y * Z


def test_views_past_2p31_table_elements(A, oracle):
    """256 views of 4096x2160: 4.57 GB of tables, and the tables of views 241..255 start beyond element 2^31"""
    W, H, V = 4096, 2160, 256
    X = Y = Z = 64
    s = F(0.28 / 64)
    assert 241 * (H + 1) * 32 * ((W + 31) // 32 + 1) >= 1 << 31
    P, _ = _ring(X, Y, Z, s, V, W, H, span=0.7, seed=51)
    rng = np.random.default_rng(52)
    bits = np.stack([_ellipse_bits(W, H, W / 2 + rng.uniform(-40, 40), H / 2 + rng.uniform(-40, 40), rng.uniform(0.15, 0.3) * W,
                                   rng.uniform(0.2, 0.4) * H, rng, 3000) for _ in range(V)])
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        occ, seen, _ = _run_all_modes(e)
        _check_oracle(oracle, X, Y, Z, s, P, W, H, bits, occ, seen)
        o, sn, _ = _run_all_modes(e, 241, 256)
        ro, _ = _check_oracle(oracle, X, Y, Z, s, P[241:], W, H, bits[241:], o, sn, what="(views 241..255)")
    assert not oracle.unpack(ro, X).all(), "views 241..255 must carve something"


def test_refused_set_views_leaves_the_engine_as_it_was(A, oracle):
    """after each refusal the engine still has its views, masks and tables and carves them to the same bits"""
    X, Y, Z = 64, 48, 40
    s = F(0.28 / 64)
    W, H, V = 320, 240, 8
    P, M = _ring(X, Y, Z, s, V, W, H, seed=61)
    bits = _view_masks(V, W, H, V, seed=62)
    ro, rs = oracle.carve(X, Y, Z, s, P, W, H, mask_bits=bits, nthreads=0)
    bad = [(257, W, H), (1, (1 << 20) + 1, 16), (1, 1 << 20, 2047), (256, 1 << 20, 256)]   # the last: V H ceil(W/32) = 2^31
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(P, W, H, M)
        e.set_masks_bits(bits)
        occ, seen, _ = _run_all_modes(e)
        assert np.array_equal(occ, ro) and np.array_equal(seen, rs)
        for Vb, Wb, Hb in bad:
            with pytest.raises(A.VoxCarveError):
                e.set_views(np.tile(P[:1], (Vb, 1, 1)), Wb, Hb)
            assert (e.V, e.W, e.H) == (V, W, H)
            assert np.array_equal(e.download_masks(), bits), f"masks changed by the refused call {(Vb, Wb, Hb)}"
            occ, seen, _ = _run_all_modes(e)
            assert np.array_equal(occ, ro) and np.array_equal(seen, rs), f"carve changed by the refused call {(Vb, Wb, Hb)}"
