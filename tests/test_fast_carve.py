"""fastCarve (VoxelCarving.cpp:74-167) on carved sets designed to break the device flood.

vc_fast_carve does not run the reference's BFS: it floods the carved set of vc_carve from voxel (0,0,0) with directional sweeps
(x inside each row with carries across words, then y, then z, both ways) until a batch of rounds changes nothing.  Silhouettes
of convex objects converge in a few rounds and never reach the cases where such a flood goes wrong, so the sets here are chosen
voxel by voxel: one view whose pixel (x + X z, y) belongs to voxel (x, y, z) alone carves exactly the set C its mask marks.

Designed sets: percolation clusters near the cubic site threshold, blobs that touch only along an edge or at a corner, a carved
pocket inside an occupied shell, runs and steps at word edges, combs whose every turn reverses the sweep direction, the origin
cases, a component touching all six faces, grids one voxel thin, two paths of some 300 000 steps (one of them needs about 180 000
sweep rounds), and the full 1024^3 grid of C4.  The device must equal the oracle's literal BFS (oracle.fast_carve) bit for bit, padding
included, with VC_EXACT and VC_EXACT_FLAT.  The CPU tests check the view and the oracle's BFS against the closed form (6-component
of the origin; seen = its dilation plus the origin) on the same sets."""
import time
from collections import deque

import numpy as np
import pytest

from ar_voxel_project_b200.synth import pack_bits

MODES = (0, 2)  # VC_EXACT, VC_EXACT_FLAT


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


# ---- the view that carves any set ---------------------------------------------------------------------------------------------

def carving_view(C):
    """C bool[Z, Y, X] -> (P, W, H, mask_bits) of one view that carves exactly C at voxel size 1.  The world point of voxel
    (x, y, z) is (y, x, -z, 1) (Model.h:134-136), so P = [[0, 1, -X, 0], [1, 0, 0, 0], [0, 0, 0, 1]] projects it to pixel
    (x + X z, y) with depth 1, exactly in f32 and f64, and every voxel has a pixel of its own in a W = X Z by H = Y image."""
    Z, Y, X = C.shape
    P = np.array([[[0, 1, -X, 0], [1, 0, 0, 0], [0, 0, 0, 1]]], np.float32)
    bg = np.ascontiguousarray(C.transpose(1, 0, 2)).reshape(1, Y, Z * X)  # pixel row y = the rows (z, y) side by side
    return P, X * Z, Y, pack_bits(bg)


def packed(b):
    """bool[Z, Y, X] -> the engine's words, padding bits 0"""
    return pack_bits(b)


def closed_form(C):
    """the BFS from the origin in closed form: (carved = 6-component of the origin, seen = its 6-dilation plus the origin)"""
    from scipy import ndimage
    if C[0, 0, 0]:
        lab, _ = ndimage.label(C)  # default structure: 6-connectivity
        comp = lab == lab[0, 0, 0]
    else:
        comp = np.zeros_like(C)
    seen = ndimage.binary_dilation(comp)
    seen[0, 0, 0] = True
    return comp, seen


# ---- designed sets (bool[Z, Y, X], True = carved) -----------------------------------------------------------------------------

PERCOLATION_DIMS = [(1, 1, 1), (1, 1, 40), (1, 9, 40), (33, 5, 7), (64, 1, 9), (95, 17, 13), (257, 31, 3), (128, 64, 64)]
PERCOLATION_P = (0.32, 0.40, 0.55)  # 0.3116: site percolation threshold of the cubic lattice


def percolation(dims, p, seed=0):
    X, Y, Z = dims
    rng = np.random.default_rng([seed, X, Y, Z, int(p * 100)])
    C = rng.random((Z, Y, X)) < p
    C[0, 0, 0] = True
    return C


def contact(kind, x0):
    """blob A = box around the origin ending at x = x0 - 1, y = z = 6; blob B touches A only along an edge parallel to one axis
    or only at a corner, across x0 | x0 - 1 (a word edge for x0 = 32).  -> (C, B)"""
    X, Y, Z = x0 + 20, 14, 14
    C = np.zeros((Z, Y, X), bool)
    C[:7, :7, :x0] = True
    lo = {"edge_z": (0, 7, x0), "edge_y": (7, 0, x0), "edge_x": (7, 7, 0), "corner": (7, 7, x0)}[kind]
    hi = {"edge_x": (14, 14, x0)}.get(kind, (14, 14, x0 + 17))
    B = np.zeros_like(C)
    B[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] = True
    return C | B, B


def cavity():
    """carved exterior; an occupied shell two voxels thick around a carved pocket that straddles the word edge 31 | 32; a second
    pocket behind a shell one voxel thick.  -> (C, pocket, inner shell layers)"""
    X, Y, Z = 70, 20, 18
    C = np.ones((Z, Y, X), bool)
    pocket, inner = np.zeros_like(C), np.zeros_like(C)
    for (x0, x1), t in (((20, 44), 2), ((50, 66), 1)):
        C[3:15, 4:16, x0:x1] = False
        if t == 2:
            inner[4:14, 5:15, x0 + 1:x1 - 1] = True
        pocket[3 + t:15 - t, 4 + t:16 - t, x0 + t:x1 - t] = True
    inner &= ~pocket
    return C | pocket, pocket, inner


def word_edges(X):
    """runs that start and end at 31 | 32, 63 | 64 and X - 1, entered and left by y steps (a staircase in plane z = 0) and by
    z steps (one in row y = Y - 1); a row carved only in its last word, entered at x = X - 1 by a z step; decoys: single
    voxels that touch the path only along an edge, one x step across a word edge away.
    -> (C, decoys, the last-word row's first voxel, the path's end), voxels as (z, y, x)"""
    cuts = sorted({c for c in (0, 31, 32, 63, 64, X - 1) if c < X})
    n = len(cuts)
    Y = Z = n + 2
    C = np.zeros((Z, Y, X), bool)
    for i in range(n - 1):  # row y = i of plane 0 holds [cuts[i], cuts[i + 1]]
        C[0, i, cuts[i]:cuts[i + 1] + 1] = True
    C[0, n - 2:, X - 1] = True  # along y to y = Y - 1
    for i in range(n - 1):  # back in row y = Y - 1: plane z = i holds [cuts[-2 - i], cuts[-1 - i]]
        C[i, Y - 1, cuts[-2 - i]:cuts[-1 - i] + 1] = True
    C[n - 2:, Y - 1, 0] = True  # along z to z = Z - 1
    C[Z - 1, :, 0] = True  # along y to y = 0
    last = (1, n - 1, 32 * ((X - 1) // 32))
    C[1, n - 1, last[2]:] = True  # its only link is (X - 1, n - 1, 0)
    decoys = np.zeros_like(C)
    for z, y, x in np.argwhere(C):
        if x % 32 not in (0, 31):
            continue
        for dz, dy in ((0, 1), (0, -1), (1, 0), (-1, 0)):
            for dx in (-1, 1):
                v = (z + dz, y + dy, x + dx)
                if 0 <= v[0] < Z and 0 <= v[1] < Y and 0 <= v[2] < X and (x + dx) // 32 != x // 32 and not _touches(C | decoys, v):
                    decoys[v] = True
    return C | decoys, decoys, last, (Z - 1, 0, 0)


def _touches(C, v):
    """v or one of its 6-neighbours is set"""
    lo = [max(c - 1, 0) for c in v]
    box = C[lo[0]:v[0] + 2, lo[1]:v[1] + 2, lo[2]:v[2] + 2]
    z, y, x = (c - l for c, l in zip(v, lo))
    return bool(box[z, y, x] or box[:, y, x].any() or box[z, :, x].any() or box[z, y, :].any())


def comb(axis, X=70, n=40):
    """full-length teeth along y (axis 1) or z (axis 0) at x = 0, 2, 4, ..., joined alternately at the far and the near end:
    every turn reverses the direction in which the flood runs along the teeth.  axis 'zy': teeth along z at y = 0, 2, 4, ...
    in the last, partial word (x = X - 1), joined by y steps, so x never moves."""
    if axis == "zy":
        Z, Y = n, 21
        C = np.zeros((Z, Y, 33), bool)
        C[0, 0, :] = True  # from the origin to x = 32
        for i, y in enumerate(range(0, Y, 2)):
            C[:, y, 32] = True
            if y + 2 < Y:
                C[Z - 1 if i % 2 == 0 else 0, y + 1, 32] = True
        return C
    shape = (3, n, X) if axis == 1 else (n, 3, X)
    C = np.zeros(shape, bool)
    for i, x in enumerate(range(0, X, 2)):
        tooth = (0, slice(None), x) if axis == 1 else (slice(None), 0, x)
        C[tooth] = True
        if x + 1 < X:
            end = n - 1 if i % 2 == 0 else 0
            C[(0, end, x + 1) if axis == 1 else (end, 0, x + 1)] = True
    return C


def origin_case(kind):
    C = np.ones((5, 6, 40), bool)
    if kind == "uncarved":  # every neighbour carved: the BFS pops the origin and stops
        C[0, 0, 0] = False
    else:  # carved but isolated: seen = the origin and its 3 neighbours
        C[0, 0, 1] = C[0, 1, 0] = C[1, 0, 0] = False
    return C


def six_faces():
    X, Y, Z = 67, 21, 13
    C = np.random.default_rng(6).random((Z, Y, X)) < 0.25
    cx, cy, cz = X // 2, Y // 2, Z // 2
    C[cz, cy, :] = C[cz, :, cx] = C[:, cy, cx] = True
    C[0, 0, :cx + 1] = C[0, :cy + 1, cx] = True  # origin -> (cx, cy, 0), then the z line
    return C


THIN_DIMS = [(300, 1, 1), (100, 37, 1), (45, 1, 29), (1, 50, 1), (1, 1, 70)]


def long_path(X=1024, Y=64, n_planes=8):
    """a path that turns at nearly every voxel: in each plane z = 0, 2, ..., diagonal staircases x - y in {d, d + 1},
    d = 0, 3, 6, ..., joined end to end alternately along the top and the bottom row; consecutive planes joined by one voxel
    of the odd plane between them, alternately at the plane's path end and at (0, 0).  The y sweep follows a staircase to the
    next word edge in one go, so this needs only some 6 000 rounds."""
    Z = 2 * n_planes - 1
    C = np.zeros((Z, Y, X), bool)
    ys = np.arange(Y)
    ds = list(range(0, X - Y, 3))
    for p in range(n_planes):
        plane = C[2 * p]
        for i, d in enumerate(ds):
            plane[ys, ys + d] = plane[ys, ys + d + 1] = True
            if i + 1 < len(ds):
                if i % 2 == 0:
                    plane[Y - 1, Y + d + 1] = True
                else:
                    plane[0, d + 2] = True
    end = (0, ds[-1]) if len(ds) % 2 == 0 else (Y - 1, Y + ds[-1])
    for p in range(n_planes - 1):
        y, x = end if p % 2 == 0 else (0, 0)
        C[2 * p + 1, y, x] = True
    return C


def serpentine(A, B):
    """cells (a, b) of an A x B plane in path order: staircases a - b in {d, d + 1}, d = 0, 3, 6, ..., run up and down
    alternately and joined by one cell at the top and the bottom row; every other step is along a"""
    cells = []
    ds = list(range(0, A - B, 3))
    for i, d in enumerate(ds):
        if i % 2 == 0:
            for b in range(B):
                cells += [(b + d, b), (b + d + 1, b)]
            if i + 1 < len(ds):
                cells.append((B + d + 1, B - 1))
        else:
            cells.append((B - 1 + d, B - 1))
            for b in range(B - 2, -1, -1):
                cells += [(b + d + 1, b), (b + d, b)]
            cells.pop()  # end on (d + 1, 0), next to the join
            if i + 1 < len(ds):
                cells.append((d + 2, 0))
    return cells


def word_crossing_path(X=1024, Y=192, Z=80):
    """the slowest path for the sweeps: its steps go z, y, x, z, y, x, ..., the reverse of the order of the x, y and z sweeps
    in a round, and every x step crosses a word edge, where only the x sweep carries.  A round then advances the flood about
    1.5 voxels.  Lane k = 1 .. X/32 - 1 follows the serpentine of the y-z plane (backwards for even k) and steps between
    x = 32k - 1 and 32k after every y step; an x run joins the origin to lane 1 and each lane to the next."""
    C = np.zeros((Z, Y, X), bool)
    plane = serpentine(Y, Z)
    x = 0
    for k in range(1, X // 32):
        seq = plane if k % 2 else plane[::-1]
        y0, z0 = seq[0]
        C[z0, y0, min(x, 32 * k - 1):max(x, 32 * k - 1) + 1] = True
        x = 32 * k - 1
        for (ya, _), (yb, zb) in zip(seq, seq[1:]):
            C[zb, yb, x] = True
            if ya != yb:
                x = 32 * k if x == 32 * k - 1 else 32 * k - 1
                C[zb, yb, x] = True
    return C


def geodesic_eccentricity(C):
    """largest BFS distance (in 6-steps) from the origin over its component"""
    Z, Y, X = C.shape
    flat = C.reshape(-1)
    dist = np.full(flat.size, -1, np.int64)
    dist[0] = 0
    q = deque([0])
    far = 0
    while q:
        i = q.popleft()
        z, r = divmod(i, X * Y)
        y, x = divmod(r, X)
        d = dist[i] + 1
        for ok, j in ((x > 0, i - 1), (x < X - 1, i + 1), (y > 0, i - X), (y < Y - 1, i + X), (z > 0, i - X * Y), (z < Z - 1, i + X * Y)):
            if ok and flat[j] and dist[j] < 0:
                dist[j] = d
                far = d
                q.append(j)
    return far


def designed_sets():
    """every designed set at its test size except the long path, by name"""
    sets = {}
    for dims in PERCOLATION_DIMS:
        for p in PERCOLATION_P:
            sets[f"percolation{dims}_p{p}"] = percolation(dims, p)
    for x0 in (10, 32):
        for kind in ("edge_z", "edge_y", "edge_x", "corner"):
            sets[f"contact_{kind}_x{x0}"] = contact(kind, x0)[0]
    sets["cavity"] = cavity()[0]
    for X in (31, 32, 33, 64, 65, 1024):
        sets[f"word_edges_X{X}"] = word_edges(X)[0]
    for axis in (1, 0, "zy"):
        sets[f"comb_{axis}"] = comb(axis)
    for kind in ("uncarved", "isolated"):
        sets[f"origin_{kind}"] = origin_case(kind)
    sets["six_faces"] = six_faces()
    for dims in THIN_DIMS:
        sets[f"thin{dims}"] = percolation(dims, 0.8)
    return sets


# ---- CPU: the view, the oracle's BFS and the designs ---------------------------------------------------------------------------

@pytest.mark.parametrize("dims", [(1, 1, 1), (7, 5, 33), (9, 17, 64), (13, 31, 95)])
def test_view_carves_exactly_the_set(oracle, dims):
    X, Y, Z = dims
    for p in (0.1, 0.5, 0.9):
        C = percolation(dims, p, seed=1)
        P, W, H, bits = carving_view(C)
        occ, seen = oracle.carve(X, Y, Z, 1.0, P, W, H, mask_bits=bits)
        assert np.array_equal(occ, packed(~C)), f"{dims} p={p}: the view does not carve exactly C"
        assert np.array_equal(seen, packed(np.ones_like(C))), f"{dims} p={p}: a voxel is outside the image"


def test_oracle_bfs_is_the_closed_form_on_designed_sets(oracle):
    """extends test_oracle_goldens::test_fast_carve_is_flood_of_carved_set_from_origin from two silhouettes to hostile sets"""
    for name, C in designed_sets().items():
        Z, Y, X = C.shape
        occ, seen = oracle.fast_carve(X, Y, Z, 1.0, *carving_view(C))
        comp, exp_seen = closed_form(C)
        assert np.array_equal(occ, packed(~comp)), f"{name}: occupied is not the complement of the origin's component"
        assert np.array_equal(seen, packed(exp_seen)), f"{name}: seen is not the component's dilation plus the origin"


def test_designs_hold_what_they_claim():
    from scipy import ndimage
    for kind in ("edge_z", "edge_y", "edge_x", "corner"):
        for x0 in (10, 32):
            C, B = contact(kind, x0)
            comp, seen = closed_form(C)
            assert not (comp & B).any() and not (seen & B).any() and ndimage.label(B)[1] == 1, (kind, x0)
            assert (ndimage.binary_dilation(B, np.ones((3, 3, 3), bool)) & comp).any(), (kind, x0)  # they do touch, diagonally
    C, pocket, inner = cavity()
    comp, seen = closed_form(C)
    assert pocket.sum() > 1000 and inner.sum() > 500 and not ((comp | seen) & (pocket | inner)).any()
    assert comp.sum() > 0.5 * C.size
    for X in (31, 32, 33, 64, 65, 1024):
        C, decoys, last, end = word_edges(X)
        comp, _ = closed_form(C)
        assert comp[last] and comp[end] and np.array_equal(C & ~comp, decoys), X
        assert decoys.any() == (X > 32), X
    for axis in (1, 0, "zy"):
        C = comb(axis)
        assert closed_form(C)[0].sum() == C.sum(), axis
    comp = closed_form(six_faces())[0]
    assert comp[0].any() and comp[-1].any() and comp[:, 0].any() and comp[:, -1].any() and comp[..., 0].any() and comp[..., -1].any()
    assert closed_form(origin_case("uncarved"))[1].sum() == 1 and closed_form(origin_case("isolated"))[1].sum() == 4
    big = percolation((128, 64, 64), 0.40)
    assert closed_form(big)[0].sum() > 0.3 * big.size  # a spanning cluster


@pytest.mark.parametrize("design,shape,n,far", [(long_path, (15, 64, 1024), 330239, 322582),
                                                (word_crossing_path, (80, 192, 1024), 284751, 277823)])
def test_long_path_designs(design, shape, n, far):
    """each is one component; `far` = steps from the origin to its farthest voxel"""
    C = design()
    comp, _ = closed_form(C)
    assert C.shape == shape and comp.sum() == C.sum() == n
    assert geodesic_eccentricity(C) == far


# ---- GPU -----------------------------------------------------------------------------------------------------------------------

def _diff(got, exp, X, what):
    from oracle.oracle import unpack
    bad = np.argwhere(unpack(got, X) != unpack(exp, X))
    pad = int(np.count_nonzero(got[..., -1] >> np.uint32(X % 32))) if X % 32 else 0
    return f"{what}: {len(bad)} voxels differ (first (z, y, x) {bad[:4].tolist()}), {pad} words with padding bits set"


def _flood(e, X, mode, ro, rs, name):
    """fast_carve on e (views and masks set) must give the oracle's volumes; -> (flood_rounds, seconds)"""
    t = time.perf_counter()
    e.fast_carve(mode)
    dt = time.perf_counter() - t
    rounds = e.stats()["flood_rounds"]
    occ, seen = e.download_occupied(), e.download_seen()
    what = f"{name} mode {mode} after {rounds} flood rounds"
    assert np.array_equal(occ, ro), _diff(occ, ro, X, what + ", occupied")
    assert np.array_equal(seen, rs), _diff(seen, rs, X, what + ", seen")
    return rounds, dt


def _matches_oracle(A, oracle, C, name):
    Z, Y, X = C.shape
    P, W, H, bits = carving_view(C)
    ro, rs = oracle.fast_carve(X, Y, Z, 1.0, P, W, H, mask_bits=bits)
    with A.VoxelEngine(X, Y, Z, 1.0) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        for mode in MODES:
            _flood(e, X, mode, ro, rs, name)
    return ro, rs


@pytest.mark.gpu
@pytest.mark.parametrize("p", PERCOLATION_P)
@pytest.mark.parametrize("dims", PERCOLATION_DIMS)
def test_percolation_clusters(A, oracle, dims, p):
    _matches_oracle(A, oracle, percolation(dims, p), f"percolation {dims} p={p}")


@pytest.mark.gpu
@pytest.mark.parametrize("x0", [10, 32])
@pytest.mark.parametrize("kind", ["edge_z", "edge_y", "edge_x", "corner"])
def test_edge_and_corner_contacts_do_not_connect(A, oracle, kind, x0):
    C, B = contact(kind, x0)
    ro, rs = _matches_oracle(A, oracle, C, f"contact {kind} x0={x0}")
    X = C.shape[2]
    assert oracle.unpack(ro, X)[B].all() and not oracle.unpack(rs, X)[B].any()


@pytest.mark.gpu
def test_enclosed_cavity_stays_occupied_and_unseen(A, oracle):
    C, pocket, inner = cavity()
    ro, rs = _matches_oracle(A, oracle, C, "cavity")
    X = C.shape[2]
    assert oracle.unpack(ro, X)[pocket].all() and not oracle.unpack(rs, X)[pocket | inner].any()


@pytest.mark.gpu
@pytest.mark.parametrize("X", [31, 32, 33, 64, 65, 1024])
def test_word_edges(A, oracle, X):
    C, decoys, _, _ = word_edges(X)
    ro, _ = _matches_oracle(A, oracle, C, f"word edges X={X}")
    assert np.array_equal(~oracle.unpack(ro, X), C & ~decoys)


@pytest.mark.gpu
@pytest.mark.parametrize("axis", [1, 0, "zy"])
def test_combs_reverse_the_sweep_at_every_turn(A, oracle, axis):
    C = comb(axis)
    ro, _ = _matches_oracle(A, oracle, C, f"comb {axis}")
    assert not (oracle.unpack(ro, C.shape[2]) & C).any()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uncarved", "isolated"])
def test_origin_cases(A, oracle, kind):
    C = origin_case(kind)
    ro, rs = _matches_oracle(A, oracle, C, f"origin {kind}")
    s = oracle.unpack(rs, C.shape[2])
    assert s.sum() == (1 if kind == "uncarved" else 4) and s[0, 0, 0]
    assert oracle.unpack(ro, C.shape[2]).sum() == C.size - (kind == "isolated")


@pytest.mark.gpu
def test_component_touching_all_six_faces(A, oracle):
    _matches_oracle(A, oracle, six_faces(), "six faces")


@pytest.mark.gpu
@pytest.mark.parametrize("dims", THIN_DIMS)
def test_grids_one_voxel_thin(A, oracle, dims):
    _matches_oracle(A, oracle, percolation(dims, 0.8), f"thin {dims}")


@pytest.mark.gpu
@pytest.mark.parametrize("design", ["staircase_planes", "word_crossing"])
def test_long_path_converges(A, oracle, design):
    """components whose farthest voxel is some 300 000 steps away; the word-crossing path needs about 180 000 sweep rounds,
    more than the flood's former cap of 100 000 allowed.  The flood runs until it converges.  Then, on the same engine, the
    same set cut a few voxels from the origin: the flood volume of the previous call must not leak into the new one."""
    C = long_path() if design == "staircase_planes" else word_crossing_path()
    Z, Y, X = C.shape
    P, W, H, bits = carving_view(C)
    ro, rs = oracle.fast_carve(X, Y, Z, 1.0, P, W, H, mask_bits=bits)
    assert (~oracle.unpack(ro, X)).sum() == C.sum()
    C2 = C.copy()
    C2[0, 0, 5] = C2[0, 3, 4] = False  # 5 voxels of the x run to lane 1; 7 of the first staircase
    P2, _, _, bits2 = carving_view(C2)
    ro2, rs2 = oracle.fast_carve(X, Y, Z, 1.0, P2, W, H, mask_bits=bits2)
    assert (~oracle.unpack(ro2, X)).sum() == (7 if design == "staircase_planes" else 5)
    with A.VoxelEngine(X, Y, Z, 1.0) as e:
        e.set_views(P, W, H)
        e.set_masks_bits(bits)
        for mode in MODES:
            rounds, dt = _flood(e, X, mode, ro, rs, design)
            print(f"{design} {X}x{Y}x{Z}, mode {mode}: {rounds} flood rounds, fast_carve {dt:.2f} s")
        e.set_views(P2, W, H)
        e.set_masks_bits(bits2)
        for mode in MODES:
            _flood(e, X, mode, ro2, rs2, design + " cut near the origin")


@pytest.mark.gpu
def test_config4_full_size(A):
    """BASELINE configs[3] (1024^3 x 72 views x 1920x1080).  The oracle's BFS queue would grow to tens of GB here, so the
    reference is the closed form on the engine's own vc_carve, whose parity test_config4_1024cubed_full_size_properties
    establishes.  Plane 0 is carved whole, so the component is the exterior."""
    from scipy import ndimage
    from ar_voxel_project_b200.synth import Workload, CONFIGS, unpack_bits
    N = 1024
    w = Workload(**CONFIGS["C4"])
    with A.VoxelEngine(N, N, N, w.s) as e:
        e.set_views(w.P, w.W, w.H)
        e.set_masks_bits(w.mask_bits)
        e.carve()
        C = ~unpack_bits(e.download_occupied(), N)
        assert C[0].all()
        lab, _ = ndimage.label(C)
        del C
        comp = lab == lab[0, 0, 0]
        del lab
        assert comp.sum() > N ** 3 // 2
        ro = packed(~comp)
        comp = ndimage.binary_dilation(comp)
        comp[0, 0, 0] = True
        rs = packed(comp)
        del comp
        for mode in MODES:
            rounds, dt = _flood(e, N, mode, ro, rs, "C4")
            print(f"C4 1024^3, mode {mode}: {rounds} flood rounds, fast_carve {dt * 1e3:.1f} ms (carve included)")
