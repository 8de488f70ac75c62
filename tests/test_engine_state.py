"""Stateful parity: long-lived engines driven through call sequences, compared with an oracle model after every step.

Callers keep one engine per dataset (the C++ shim, vc::carveToMesh, a streaming capture with vc_append_views, the reference's
-intermediateMesh path that carves view by view into a Model that already holds state).  What such an engine returns depends
on state that every call has to keep right: the cached CUDA graphs of the carve, the ownership of the constant view tables,
the brick flags that vc_mc_classify and the sparse download trust while `flags_valid` is set, the lazy reset, the "have"
flags of colours, cube indices, mesh and text, and the grow-only buffers.  A missed invalidation there does not crash; it
returns stale bits on the second or third call of some sequence.

EngineModel mirrors one engine's observable state and updates it with the CPU oracle; the seeded driver runs random call
sequences against it (VC_STATE_SEEDS=n runs seeds 0 .. n-1, default 10), and the directed tests below pin each cache to the
invariant it must keep."""
import ctypes as C
import os

import numpy as np
import pytest

F = np.float32
S = F(0.01)
VC_ERR_ARG, VC_ERR_STATE = 1, 3


# ---- captures: cameras on a ring around the grid, elliptic silhouettes with background specks ------------------------------
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


def _views(rng, V, W, H, dims):
    """-> (P, M) float32[V, 3, 4]: random cameras around the grid centre (world = (y s, x s, -z s)), the grid inside the image"""
    X, Y, Z = dims
    c = np.array([(Y - 1) * float(S) / 2, (X - 1) * float(S) / 2, -(Z - 1) * float(S) / 2])
    ext = float(S) * max(dims) * 1.5
    dist = 3.0 * ext
    P, M = [], []
    for _ in range(V):
        az, el = rng.uniform(0, 2 * np.pi), np.deg2rad(rng.uniform(15, 65))
        eye = c + dist * np.array([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), -np.sin(el)])
        jx, jy = rng.uniform(-0.5, 0.5, 2)
        p, m = _look_at(eye, c, 0.6 * W * dist / ext, 0.6 * H * dist / ext, W / 2 + jx, H / 2 + jy)
        P.append(p), M.append(m)
    return np.stack(P), np.stack(M)


def _masks(rng, V, W, H, specks=0.003):
    """uint32[V][H][ceil(W/32)] (1 = background): a foreground ellipse of random size plus background specks"""
    from ar_voxel_project_b200.synth import pack_bits
    yy, xx = np.mgrid[0:H, 0:W]
    out = []
    for _ in range(V):
        rx, ry = W * rng.uniform(0.1, 0.2), H * rng.uniform(0.12, 0.25)
        bg = ((xx - W / 2 - rng.uniform(-3, 3)) / rx) ** 2 + ((yy - H / 2 - rng.uniform(-3, 3)) / ry) ** 2 > 1.0
        n = int(specks * W * H)
        bg[rng.integers(0, H, n), rng.integers(0, W, n)] = True
        out.append(pack_bits(bg))
    return np.stack(out)


def _bgr_of_bits(rng, bits, W):
    """8UC3 masks that pack to `bits`: background (0,0,0), foreground any other colour (VoxelCarving.cpp:49-50)"""
    from ar_voxel_project_b200.synth import unpack_bits
    fg = ~unpack_bits(bits, W)
    return (rng.integers(1, 256, (*fg.shape, 3), dtype=np.uint8) * fg[..., None]).astype(np.uint8)


def _valid(X):
    Wx = (X + 31) // 32
    v = np.full(Wx, 0xffffffff, np.uint32)
    if X % 32:
        v[-1] = (1 << (X % 32)) - 1
    return v


def _random_state(rng, X, Y, nz):
    """random volumes with every padding bit set (the upload clears them) and a block of carved-but-unseen voxels"""
    Wx = (X + 31) // 32
    occ = rng.integers(0, 2 ** 32, (nz, Y, Wx), dtype=np.uint64).astype(np.uint32)
    seen = rng.integers(0, 2 ** 32, (nz, Y, Wx), dtype=np.uint64).astype(np.uint32)
    k = int(rng.integers(0, nz))
    occ[k:k + max(1, nz // 4)] = 0xffffffff * int(rng.integers(0, 2))
    seen[k:k + max(1, nz // 4)] = 0
    occ[..., -1] |= ~_valid(X)[-1]
    seen[..., -1] |= ~_valid(X)[-1]
    return occ, seen


def _popcount(a):
    return int(np.unpackbits(np.ascontiguousarray(a).view(np.uint8)).sum())


def _device_bits(bits):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(bits, np.uint32).view(np.int32).copy()).cuda()
    torch.cuda.synchronize()
    return t


def _same(got, want, what):
    assert got.shape == want.shape and np.array_equal(got, want), f"{what} differs from the model"


# ---- the oracle model of one engine ---------------------------------------------------------------------------------------
class EngineModel:
    """What one engine's observable state must be.  Volumes are the slab's words; every operation is restated with the CPU
    oracle.  A carve of views [a, b) onto (o, s) gives (o & ro, s | rs) with (ro, rs) = oracle.carve of those views (DESIGN
    section 2.6).  colors / mc / mesh / text / dense are None while the engine holds none that a download may return."""

    def __init__(self, O, X, Y, Z, z0=0, z1=None, CV=None):
        self.O, self.CV = O, CV
        self.X, self.Y, self.Z = X, Y, Z
        self.z0, self.z1 = z0, Z if z1 is None else z1
        self.whole = self.z0 == 0 and self.z1 == Z
        self.shape = (self.z1 - self.z0, Y, (X + 31) // 32)
        self.P = self.M = self.bits = self.images = None
        self.W = self.H = 0
        self.dense = self.mesh = self.text = None
        self.reset()

    @property
    def V(self):
        return 0 if self.P is None else len(self.P)

    def reset(self):
        self.occ = np.broadcast_to(_valid(self.X), self.shape).copy()
        self.seen = np.zeros(self.shape, np.uint32)
        self.pending = True   # vc_reset not materialised yet (the next VC_EXACT carve is a fresh one)
        self.colors = self.mc = None

    def _volumes_changed(self):
        self.pending = False
        self.colors = self.mc = None

    def carve_result(self, v0, v1):
        return self.O.carve(self.X, self.Y, self.Z, S, self.P[v0:v1], self.W, self.H, mask_bits=self.bits[v0:v1],
                            z0=self.z0, z1=self.z1, nthreads=0)

    def carve(self, v0=0, v1=None):
        v1 = self.V if v1 is None else v1
        ro, rs = self.carve_result(v0, v1)
        self.occ &= ro
        self.seen |= rs
        self._volumes_changed()

    def fast_carve(self):
        self.occ, self.seen = self.O.fast_carve(self.X, self.Y, self.Z, S, self.P, self.W, self.H, mask_bits=self.bits)
        self._volumes_changed()

    def upload(self, occ, seen):
        self.occ, self.seen = occ & _valid(self.X), seen & _valid(self.X)
        self._volumes_changed()

    def color(self, mode):
        self.colors = self.O.color(self.X, self.Y, self.Z, S, self.P, self.M, self.W, self.H, self.images, self.occ, mode)
        self.pending = False

    def color_visible(self, mode, tol):
        self.colors = self.CV.color_visible(self.X, self.Y, self.Z, S, self.P, self.M, self.W, self.H, self.images, self.occ, mode, tol)
        self.pending = False

    def mc_classify(self):
        self.mc = self.O.mc_classify(self.X, self.Y, self.Z, self.occ)
        self.pending = False

    def dense_of_volumes(self, apply_colors, handle_unseen):
        idx, rgbn = self.colors if apply_colors else (None, None)
        return self.O.dense_model(self.X, self.Y, self.Z, self.occ, self.seen if handle_unseen else None, idx, rgbn)

    def set_mesh(self, mesh):
        self.mesh, self.text = mesh, None   # a new mesh: the previous text no longer describes it

    def mesh_from_volumes(self, apply_colors, handle_unseen, closure_k):
        d = self.dense_of_volumes(apply_colors, handle_unseen)
        if closure_k:
            d = self.O.closure(self.X, self.Y, self.Z, d, closure_k)
        self.set_mesh(self.O.marching_cubes(self.X, self.Y, self.Z, d, 0.5))
        self.pending = False

    def dense_from_volumes(self, apply_colors, handle_unseen):
        self.dense = self.dense_of_volumes(apply_colors, handle_unseen)
        self.mesh = None
        self.pending = False

    def dense_upload(self, rgba):
        self.dense = np.ascontiguousarray(rgba, np.float32).reshape(-1, 4).copy()
        self.mesh = None

    def dense_apply_carved(self):
        self.dense[~self.O.unpack(self.occ, self.X).reshape(-1)] = 0   # model.set(x, y, z, 0) (VoxelCarving.cpp:52)
        self.mesh = None
        self.pending = False

    def dense_closure(self, k):
        self.dense = self.O.closure(self.X, self.Y, self.Z, self.dense, k)
        self.mesh = None

    def mc_mesh(self):
        self.set_mesh(self.O.marching_cubes(self.X, self.Y, self.Z, self.dense, 0.5))

    def off_text(self, tmp_path, scale, t):
        p = str(tmp_path / "model.off")
        self.O.write_off(p, self.mesh[0], self.mesh[1], scale, t)
        with open(p, "rb") as f:
            return f.read()


def _state_error(A, code, fn, *a, **kw):
    with pytest.raises(A.VoxCarveError) as ei:
        fn(*a, **kw)
    assert ei.value.code == code, f"expected voxcarve error {code}, got {ei.value.code}: {ei.value}"


def check_engine(A, e, m, volumes=True):
    """everything a caller can observe, against the model: volumes and counts (skipped while a reset is pending: reading them
    would materialise it, and the next carve would no longer be a fresh one), colour records, cube-index histogram, mesh, text
    and dense Model; where the model holds none, the download must be refused with VC_ERR_STATE"""
    if volumes and not m.pending:
        _same(e.download_occupied(), m.occ, "occupied volume")
        _same(e.download_seen(), m.seen, "seen volume")
        assert e.count_occupied() == (_popcount(m.occ), _popcount(m.seen)), "count_occupied differs from the model"
    if m.colors is None:
        _state_error(A, VC_ERR_STATE, e.download_colors)
    else:
        idx, rgbn = e.download_colors()
        _same(idx, m.colors[0], "colour record indices")
        _same(rgbn, m.colors[1], "colour records")
    if m.mc is None:
        _state_error(A, VC_ERR_STATE, e.download_mc)
    else:
        hist, na, nt = e.download_mc()
        _same(hist, m.mc[0], "cube-index histogram")
        assert (na, nt) == (m.mc[1], m.mc[2]), "active cells / triangles differ from the model"
    if m.mesh is None:
        _state_error(A, VC_ERR_STATE, e.download_mesh, 0)
    else:
        v, c = e.download_mesh(len(m.mesh[0]))
        _same(v, m.mesh[0], "mesh vertices")
        _same(c, m.mesh[1], "mesh colours")
    if m.text is None:
        _state_error(A, VC_ERR_STATE, e.download_mesh_off, 0, 0)
    else:
        assert e.download_mesh_off(0, len(m.text)) == m.text, ".off text differs from the model"
    if m.dense is None:
        _state_error(A, VC_ERR_STATE, e.dense_download)
    else:
        _same(e.dense_download().view(np.uint32), m.dense.view(np.uint32), "dense Model")


# ---- 1. the model's accumulation rule (CPU) ---------------------------------------------------------------------------------
@pytest.mark.parametrize("slab", [None, (5, 17)], ids=["grid", "slab"])
def test_model_accumulation_rule_matches_one_carve(oracle, slab):
    """the model folds per-view carves with (o & ro, s | rs); folded view by view in a shuffled order, from the constructor
    state and from a state that holds carved-but-unseen voxels, it must equal one oracle carve of all views"""
    rng = np.random.default_rng(3)
    X, Y, Z = 45, 30, 22
    W, H, V = 96, 72, 7
    z0, z1 = slab or (0, Z)
    P, M = _views(rng, V, W, H, (X, Y, Z))
    bits = _masks(rng, V, W, H)
    m = EngineModel(oracle, X, Y, Z, z0, z1)
    m.P, m.M, m.bits, m.W, m.H = P, M, bits, W, H
    for v in rng.permutation(V):
        m.carve(v, v + 1)
    ro, rs = oracle.carve(X, Y, Z, S, P, W, H, mask_bits=bits, z0=z0, z1=z1)
    _same(m.occ, ro, "occupied of the folded per-view carves")
    _same(m.seen, rs, "seen of the folded per-view carves")
    assert 0 < _popcount(ro) < X * Y * (z1 - z0) and _popcount(rs) > 0
    # from an uploaded state: a carve of all views at once equals the fold in any order
    occ0, seen0 = _random_state(rng, X, Y, z1 - z0)
    m.upload(occ0, seen0)
    for v in rng.permutation(V):
        m.carve(v, v + 1)
    _same(m.occ, occ0 & _valid(X) & ro, "occupied of the folds from an uploaded state")
    _same(m.seen, (seen0 & _valid(X)) | rs, "seen of the folds from an uploaded state")


# ---- 2. the seeded random driver --------------------------------------------------------------------------------------------
_CONFIGS = [
    dict(dims=(45, 30, 20)),
    dict(dims=(100, 20, 18)),               # rows of whole quads: the blind fill of a fresh carve
    dict(dims=(40, 20, 72)),                # nz >= 64: a page-locked carve_download carves in two z-chunks
    dict(dims=(70, 26, 40), slab=(8, 33)),
    dict(dims=(33, 17, 24), many=True),     # appends past 256 views (two view groups)
    dict(dims=(64, 24, 75), slab=(3, 70)),  # a z-slab of 67 planes that also chunks
    dict(dims=(37, 41, 13)),
    dict(dims=(128, 12, 16), slab=(0, 9)),
    dict(dims=(31, 33, 66)),
    dict(dims=(50, 9, 33), many=True),
]
_SEEDS = int(os.environ.get("VC_STATE_SEEDS", "10"))


class Driver:
    def __init__(self, A, O, CV, seed, tmp_path):
        import torch
        self.A, self.O, self.tmp = A, O, tmp_path
        cfg = _CONFIGS[seed % len(_CONFIGS)]
        self.rng = np.random.default_rng(1000 + seed)
        self.X, self.Y, self.Z = cfg["dims"]
        z0, z1 = cfg.get("slab", (0, self.Z))
        self.many = cfg.get("many", False)
        self.geoms = [(64, 48), (70, 41)] if self.many else [(96, 72), (80, 60), (131, 67)]
        self.e = A.VoxelEngine(self.X, self.Y, self.Z, S, z_begin=z0, z_end=z1)
        self.m = EngineModel(O, self.X, self.Y, self.Z, z0, z1, CV)
        self.stream = torch.cuda.Stream()
        self.keep = []   # device masks whose copies may still be queued

    # -- helpers
    def refused(self, code, fn, *a, **kw):
        _state_error(self.A, code, fn, *a, **kw)

    def new_views(self, V=None, geom=None, with_M=None):
        r, m = self.rng, self.m
        W, H = geom or (self.geoms[r.integers(len(self.geoms))] if m.V == 0 or r.random() < 0.5 else (m.W, m.H))
        V = V or int(r.integers(3, 9))
        P, M = _views(r, V, W, H, (self.X, self.Y, self.Z))
        with_M = r.random() < 0.85 if with_M is None else with_M
        return P, (M if with_M else None), W, H

    # -- views and masks
    def op_set_views(self):
        r, e, m = self.rng, self.e, self.m
        kind = ["new P", "new V", "new WxH", "V=257"][r.choice(4, p=[0.45, 0.2, 0.25, 0.1])] if m.V else "first"
        if kind == "V=257":
            P = np.tile(m.P[:1], (257, 1, 1))
            self.refused(VC_ERR_ARG, e.set_views, P, m.W, m.H)
            return "set_views(V=257) refused"
        if kind == "new P" and m.V <= 256:
            P, M, W, H = self.new_views(V=m.V, geom=(m.W, m.H))
        elif kind == "new V":
            P, M, W, H = self.new_views(geom=(m.W, m.H) if m.V else None)
        else:
            P, M, W, H = self.new_views()
        e.set_views(P, W, H, M)
        if (len(P), W, H) != (m.V, m.W, m.H):   # geometry changed: masks and images no longer match
            m.bits = m.images = None
        m.P, m.M, m.W, m.H = P, M, W, H
        return f"set_views(V={len(P)}, {W}x{H}, M={'yes' if M is not None else 'no'})"

    def masks_for(self, n):
        return _masks(self.rng, n, self.m.W, self.m.H, specks=self.rng.choice([0.0, 0.003, 0.02]))

    def op_set_masks(self):
        r, e, m = self.rng, self.e, self.m
        if m.V == 0:
            self.refused(VC_ERR_STATE, e.set_masks_bits, np.zeros(1, np.uint32))
            return "set_masks before set_views refused"
        bits = self.masks_for(m.V)
        fmt = ["bits", "bgr", "device"][r.integers(3)]
        if fmt == "bits":
            e.set_masks_bits(bits)
        elif fmt == "bgr":
            e.set_masks_bgr(_bgr_of_bits(r, bits, m.W))
        else:
            t = _device_bits(bits)
            self.keep.append(t)
            e.set_masks_bits_device(t.data_ptr())
        m.bits = bits
        return f"set_masks({fmt})"

    def op_set_images(self):
        e, m = self.e, self.m
        if m.V == 0:
            self.refused(VC_ERR_STATE, e.set_images, np.zeros(3, np.uint8))
            return "set_images before set_views refused"
        m.images = self.rng.integers(0, 256, (m.V, m.H, m.W, 3), dtype=np.uint8)
        e.set_images(m.images)
        return "set_images"

    def op_append_views(self):
        r, e, m = self.rng, self.e, self.m
        n = int(r.integers(20, 140)) if self.many and r.random() < 0.6 else int(r.integers(1, 5))
        if m.V + n > 320:
            n = int(r.integers(1, 4))
        P, M = _views(r, n, m.W or 64, m.H or 48, (self.X, self.Y, self.Z))
        if m.bits is None:
            self.refused(VC_ERR_STATE, e.append_views, P, M, mask_bits=np.zeros((n, max(m.H, 1), (max(m.W, 1) + 31) // 32), np.uint32))
            return "append_views without masks refused"
        bits = self.masks_for(n)
        imgs = r.integers(0, 256, (n, m.H, m.W, 3), dtype=np.uint8)
        give_M, give_img = m.M is not None, m.images is not None
        if r.random() < 0.15:   # an M or images that do not match the engine
            if r.random() < 0.5:
                give_M = not give_M
            else:
                give_img = not give_img
            self.refused(VC_ERR_ARG, e.append_views, P, M if give_M else None, mask_bits=bits, images_bgr=imgs if give_img else None)
            return f"append_views(n={n}, mismatched M / images) refused"
        fmt = ["bits", "bgr", "device"][r.integers(3)]
        kw = dict(mask_bits=bits) if fmt == "bits" else dict(mask_bgr=_bgr_of_bits(r, bits, m.W)) if fmt == "bgr" else \
            dict(mask_bits=_device_bits(bits))
        if fmt == "device":
            self.keep.append(kw["mask_bits"])
        e.append_views(P, M if give_M else None, images_bgr=imgs if give_img else None, **kw)
        m.P, m.bits = np.concatenate([m.P, P]), np.concatenate([m.bits, bits])
        if give_M:
            m.M = np.concatenate([m.M, M])
        if give_img:
            m.images = np.concatenate([m.images, imgs])
        return f"append_views(n={n}, {fmt}) -> V={m.V}"

    # -- carving
    def op_reset(self):
        self.e.reset()
        self.m.reset()
        return "reset"

    def op_carve(self):
        r, e, m = self.rng, self.e, self.m
        mode = [0, 2][r.integers(2)]
        if m.bits is None:
            self.refused(VC_ERR_STATE, e.carve, mode)
            return f"carve({mode}) without masks refused"
        v0, v1 = 0, m.V
        if r.random() < 0.4:
            v0 = int(r.integers(0, m.V))
            v1 = int(r.integers(v0 + 1, m.V + 1))
        e.carve(mode, v0, v1 if v1 < m.V or r.random() < 0.5 else -1)
        m.carve(v0, v1)
        return f"carve(mode={mode}, [{v0},{v1}))"

    def op_carve_download(self):
        import torch
        r, e, m = self.rng, self.e, self.m
        mode = [0, 2][r.integers(2)]
        if m.bits is None:
            self.refused(VC_ERR_STATE, e.carve_download, mode=mode)
            return "carve_download without masks refused"
        pinned = r.random() < 0.6
        if pinned:
            n = int(np.prod(m.shape))
            o, s = (torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(2))
            e.carve_download(o, s, mode=mode)
            o, s = o.numpy().view(np.uint32).reshape(m.shape), s.numpy().view(np.uint32).reshape(m.shape)
        else:
            o, s = e.carve_download(mode=mode)
        m.carve()
        _same(o, m.occ, "carve_download's occupied")
        _same(s, m.seen, "carve_download's seen")
        return f"carve_download(mode={mode}, {'pinned' if pinned else 'pageable'})"

    def op_sparse(self):
        e, m = self.e, self.m
        if m.bits is None:
            return None
        if not m.pending and self.rng.random() < 0.3:   # the C entry point itself: it describes a fresh carve only
            nbx, nby, nbz = C.c_uint32(), C.c_uint32(), C.c_uint32()
            e._check(e._lib.vc_sparse_dims(e._h, C.byref(nbx), C.byref(nby), C.byref(nbz)))
            nb = nbx.value * nby.value * nbz.value
            flags, listed, words, n = np.empty(nb, np.uint8), np.empty(1, np.uint32), np.empty(128, np.uint32), C.c_uint64()
            rc = e._lib.vc_carve_download_sparse(e._h, flags.ctypes.data, nb, listed.ctypes.data, words.ctypes.data, 1, C.byref(n))
            assert rc == VC_ERR_STATE, f"vc_carve_download_sparse without a pending reset returned {rc}"
            return "vc_carve_download_sparse without a pending reset refused"
        flags, listed, words = e.carve_download_sparse()   # resets first
        m.reset()
        m.carve()
        o, s = e.expand_sparse(flags, listed, words)
        _same(o, m.occ, "sparse download's occupied")
        _same(s, m.seen, "sparse download's seen")
        return f"carve_download_sparse ({len(listed)} listed)"

    def op_fast_carve(self):
        e, m = self.e, self.m
        mode = [0, 2][self.rng.integers(2)]
        if not m.whole or m.bits is None:
            self.refused(VC_ERR_STATE, e.fast_carve, mode)
            return f"fast_carve({mode}) refused ({'slab' if not m.whole else 'no masks'})"
        e.fast_carve(mode)
        m.fast_carve()
        return f"fast_carve({mode})"

    def op_upload(self):
        occ, seen = _random_state(self.rng, self.X, self.Y, self.m.shape[0])
        self.e.upload_volumes(occ, seen)
        self.m.upload(occ, seen)
        return "upload_volumes"

    # -- consumers
    def _colour_refusal(self):
        m = self.m
        if not m.whole:
            return "slab"
        if m.V == 0 or m.images is None:
            return "no images"
        if m.M is None:
            return "no M"
        return None

    def op_color(self):
        mode = int(self.rng.integers(1, 3))
        why = self._colour_refusal()
        if why:
            self.refused(VC_ERR_STATE, self.e.color, mode)
            return f"color({mode}) refused ({why})"
        self.e.color(mode)
        self.m.color(mode)
        return f"color({mode}) -> {len(self.m.colors[0])} records"

    def op_color_visible(self):
        mode = int(self.rng.integers(1, 3))
        tol = [0.0, 2.0, float("inf")][self.rng.integers(3)]
        why = self._colour_refusal()
        if why:
            self.refused(VC_ERR_STATE, self.e.color_visible, mode, tol)
            return f"color_visible({mode}) refused ({why})"
        self.e.color_visible(mode, tol)
        self.m.color_visible(mode, tol)
        return f"color_visible({mode}, {tol}) -> {len(self.m.colors[0])} records"

    def op_mc_classify(self):
        if not self.m.whole:   # a slab without its neighbour planes
            self.refused(VC_ERR_STATE, self.e.mc_classify)
            return "mc_classify refused (slab without halos)"
        self.e.mc_classify()
        self.m.mc_classify()
        return "mc_classify"

    def op_mesh_from_volumes(self):
        r, e, m = self.rng, self.e, self.m
        ac, hu, k = bool(r.integers(2)), bool(r.integers(2)), [0, 0, 3, 5][r.integers(4)]
        if not m.whole or (ac and m.colors is None):
            self.refused(VC_ERR_STATE, e.mesh_from_volumes, ac, hu, k)
            return f"mesh_from_volumes(ac={ac}) refused"
        verts, rgb = e.mesh_from_volumes(ac, hu, k)
        m.mesh_from_volumes(ac, hu, k)
        _same(verts, m.mesh[0], "mesh_from_volumes' vertices")
        _same(rgb, m.mesh[1], "mesh_from_volumes' colours")
        return f"mesh_from_volumes(ac={ac}, hu={hu}, k={k}) -> {len(verts)} triangles"

    def op_format_off(self):
        r, e, m = self.rng, self.e, self.m
        scale = [F(1.0), S, F(0.37)][r.integers(3)]
        t = tuple(F(x) for x in r.uniform(-1, 1, 3)) if r.random() < 0.5 else (F(0), F(0), F(0))
        if m.mesh is None:
            self.refused(VC_ERR_STATE, e.format_off, scale, t)
            return "format_off without a mesh refused"
        n = e.format_off(scale, t)
        m.text = m.off_text(self.tmp, scale, t)
        assert n == len(m.text), f"format_off: {n} bytes, the model {len(m.text)}"
        return f"format_off({n} bytes)"

    def op_dense(self):
        r, e, m = self.rng, self.e, self.m
        kind = ["from_volumes", "upload", "apply_carved", "closure", "mc_mesh"][r.integers(5)]
        if not m.whole:
            fn = {"from_volumes": lambda: e.dense_from_volumes(), "upload": lambda: e.dense_upload(np.zeros((1, 4), np.float32)),
                  "apply_carved": e.dense_apply_carved, "closure": lambda: e.dense_closure(3), "mc_mesh": lambda: e.mc_mesh(0.5)}[kind]
            if kind == "upload":   # the wrapper checks the size of the host buffer first
                fn = lambda: e._check(e._lib.vc_dense_upload(e._h, C.c_void_p(np.zeros(4, np.float32).ctypes.data)))  # noqa: E731
            self.refused(VC_ERR_STATE, fn)
            return f"dense {kind} refused (slab)"
        if kind == "from_volumes":
            ac, hu = bool(r.integers(2)), bool(r.integers(2))
            if ac and m.colors is None:
                self.refused(VC_ERR_STATE, e.dense_from_volumes, True, hu)
                return "dense_from_volumes(apply_colors) without colours refused"
            e.dense_from_volumes(ac, hu)
            m.dense_from_volumes(ac, hu)
            return f"dense_from_volumes(ac={ac}, hu={hu})"
        if kind == "upload":
            n = self.X * self.Y * self.Z
            rgba = np.zeros((n, 4), np.float32)
            rgba[:, :3] = r.integers(0, 256, (n, 3))
            rgba[:, 3] = r.choice([0.0, 0.25, 0.5, 0.75, 1.0], n)
            e.dense_upload(rgba)
            m.dense_upload(rgba)
            return "dense_upload"
        if m.dense is None:
            fn = {"apply_carved": e.dense_apply_carved, "closure": lambda: e.dense_closure(3), "mc_mesh": lambda: e.mc_mesh(0.5)}[kind]
            self.refused(VC_ERR_STATE, fn)
            return f"dense {kind} without a dense Model refused"
        if kind == "apply_carved":
            e.dense_apply_carved()
            m.dense_apply_carved()
            return "dense_apply_carved"
        if kind == "closure":
            k = [3, 5][r.integers(2)]
            e.dense_closure(k)
            m.dense_closure(k)
            return f"dense_closure({k})"
        verts, rgb = e.mc_mesh(0.5)
        m.mc_mesh()
        _same(verts, m.mesh[0], "mc_mesh vertices")
        _same(rgb, m.mesh[1], "mc_mesh colours")
        return f"mc_mesh -> {len(verts)} triangles"

    # -- engine settings
    def op_profiling(self):
        on = bool(self.rng.integers(2))
        self.e.set_profiling(on)
        return f"set_profiling({on})"

    def op_stream(self):
        use = bool(self.rng.integers(2))
        self.e.set_stream(self.stream.cuda_stream if use else None)
        return f"set_stream({'torch stream' if use else 'own'})"

    OPS = [("set_views", 3), ("set_masks", 3), ("set_images", 2), ("append_views", 2), ("reset", 4), ("carve", 7),
           ("carve_download", 3), ("sparse", 2), ("fast_carve", 1), ("upload", 2), ("color", 3), ("color_visible", 2),
           ("mc_classify", 3), ("mesh_from_volumes", 2), ("format_off", 2), ("dense", 4), ("profiling", 1), ("stream", 1)]

    def run(self, seed, n_steps=40):
        names = [n for n, _ in self.OPS]
        p = np.array([w for _, w in self.OPS], float)
        p /= p.sum()
        log = [f"seed {seed}: engine {self.X}x{self.Y}x{self.Z}, slab [{self.m.z0},{self.m.z1})"]
        plan = ["carve", "set_views", "set_masks", "set_images"]   # the cold engine first refuses, then gets its inputs
        i = 0
        try:
            while i < n_steps:
                name = plan.pop(0) if plan else names[self.rng.choice(len(names), p=p)]
                log.append(f"  step {i}: {name}")
                what = getattr(self, "op_" + name)()
                if what is None:
                    log.pop()
                    continue
                log[-1] = f"  step {i}: {what}"
                check_engine(self.A, self.e, self.m)
                i += 1
        except Exception as ex:
            raise AssertionError("\n".join(log) + f"\n  -> failed at the last step: {type(ex).__name__}: {ex}") from ex
        finally:
            self.e.close()
        return log


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(_SEEDS))
def test_random_call_sequences(A, oracle, CV, seed, tmp_path):
    """~40 random calls on one engine, each compared with the oracle model; the failure message replays the sequence"""
    Driver(A, oracle, CV, seed, tmp_path).run(seed)


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


@pytest.fixture(scope="module")
def CV():
    from oracle import color_visible as CV
    CV.build()
    return CV


def _engine_with(A, dims, P, M, W, H, bits, images=None, z0=0, z1=None):
    e = A.VoxelEngine(*dims, S, z_begin=z0, z_end=z1)
    e.set_views(P, W, H, M)
    e.set_masks_bits(bits)
    if images is not None:
        e.set_images(images)
    return e


# ---- 3a. the cached carve graphs -------------------------------------------------------------------------------------------
def _runtime_calls(fn):
    """run fn under torch.profiler -> {"instantiate": graph instantiations, "graph": graph launches, "kernel": kernel launches}:
    the CUDA runtime calls fn made, which tell a captured, a replayed and a plainly launched carve apart"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], acc_events=True) as prof:
        fn()
        torch.cuda.synchronize()
    names = [ev.name for ev in prof.events()]
    return {"instantiate": sum("cudaGraphInstantiate" in n for n in names), "graph": sum(n.startswith("cudaGraphLaunch") for n in names),
            "kernel": sum(n.startswith("cudaLaunchKernel") for n in names)}


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(100, 24, 20), (45, 30, 20)], ids=["quads", "ragged"])
def test_graph_replay_across_input_changes(A, oracle, dims, monkeypatch):
    """a whole-range VC_EXACT carve replays its cached graph while the key (grid, slab, buffers, W x H, view range) is unchanged:
    the graph must then carve with the views and masks uploaded since, and a changed key must recapture.  Each step also checks
    which path it took (graph instantiations / launches among the CUDA runtime calls of the carve)"""
    rng = np.random.default_rng(11)
    W, H, V = 96, 72, 6
    P1, M1 = _views(rng, V, W, H, dims)
    P2, M2 = _views(rng, V, W, H, dims)
    b1, b2 = _masks(rng, V, W, H), _masks(rng, V, W, H, specks=0.02)
    W3, H3 = 80, 60
    P3, M3 = _views(rng, V, W3, H3, dims)
    b3 = _masks(rng, V, W3, H3)
    CAPTURE, REPLAY, PLAIN = (1, 1), (0, 1), (0, 0)   # (instantiations, graph launches)

    def want(P, bits, w, h, v1=V):
        return oracle.carve(*dims, S, P[:v1], w, h, mask_bits=bits[:v1])

    def run(e, graphs):
        def carve(what, path, v0=0, v1=-1):
            c = _runtime_calls(lambda: e.carve(0, v0, v1))
            path = path if graphs else PLAIN
            assert (c["instantiate"], c["graph"]) == path, f"{what}: {c['instantiate']} graph instantiations and {c['graph']} " \
                f"graph launches, expected {path} (VOXCARVE_NO_GRAPH={'0' if graphs else '1'})"
            if path == PLAIN:
                assert c["kernel"] > 0, f"{what}: a plain carve launches its kernels one by one"

        def fresh(what, P, bits, w, h, path):
            e.reset()
            carve(what, path)
            ro, rs = want(P, bits, w, h)
            _same(e.download_occupied(), ro, f"occupied after {what}")
            _same(e.download_seen(), rs, f"seen after {what}")

        fresh("the first fresh carve (graph captured)", P1, b1, W, H, CAPTURE)
        e.set_views(P2, W, H, M2)        # same V / W / H: masks and tables are kept, the key is unchanged
        e.set_masks_bits(b2)
        fresh("new P and masks under the same key (graph replayed against the re-uploaded constants)", P2, b2, W, H, REPLAY)
        # the accumulating graph (slot of non-fresh carves): a sub-range first, then the whole range onto it
        e.reset()
        carve("a fresh sub-range carve", PLAIN, 0, 2)
        carve("the first whole-range carve onto a carved state (accumulating graph captured)", CAPTURE)
        ro, rs = want(P2, b2, W, H)
        _same(e.download_occupied(), ro, "occupied after a sub-range carve + a whole-range accumulating carve")
        e.set_views(P1, W, H, M1)
        e.set_masks_bits(b1)
        e.reset()
        carve("a fresh sub-range carve", PLAIN, 0, 2)
        carve("a whole-range carve onto a carved state with new views (accumulating graph replayed)", REPLAY)
        ro, rs = want(P1, b1, W, H)
        _same(e.download_occupied(), ro, "occupied after the accumulating graph was replayed with new views")
        _same(e.download_seen(), rs, "seen after the accumulating graph was replayed with new views")
        e.set_views(P3, W3, H3, M3)      # new W x H: a new key, recaptured
        e.set_masks_bits(b3)
        fresh("a new W x H (recaptured)", P3, b3, W3, H3, CAPTURE)
        e.set_profiling(True)
        fresh("profiling on (plain launches)", P3, b3, W3, H3, PLAIN)
        assert e.stats()["last_classify_ms"] > 0, "a profiling carve records the classification time"
        e.set_views(P1, W, H, M1)
        e.set_masks_bits(b1)
        fresh("profiling on with the first views", P1, b1, W, H, PLAIN)
        e.set_profiling(False)
        # one cached graph per kind of carve: the fresh slot holds the W3 x H3 key, so the first key is captured again
        fresh("profiling off again (the first key recaptured)", P1, b1, W, H, CAPTURE)
        assert e.stats()["last_classify_ms"] == 0, "a carve without profiling does not split its time"
        fresh("the same carve again (replayed)", P1, b1, W, H, REPLAY)
        e.set_views(P1[:4], W, H, M1[:4])   # fewer views: the view range is part of the key
        e.set_masks_bits(b1[:4])
        e.reset()
        carve("V changed under the same W x H (recaptured)", CAPTURE)
        ro, rs = want(P1, b1, W, H, v1=4)
        _same(e.download_occupied(), ro, "occupied after V changed under the same W x H")

    with A.VoxelEngine(*dims, S) as e:
        e.set_views(P1, W, H, M1)
        e.set_masks_bits(b1)
        run(e, graphs=True)
    monkeypatch.setenv("VOXCARVE_NO_GRAPH", "1")   # read per engine at its first carve
    with A.VoxelEngine(*dims, S) as e:
        e.set_views(P1, W, H, M1)
        e.set_masks_bits(b1)
        run(e, graphs=False)


@pytest.mark.gpu
def test_refused_fast_carve_leaves_the_volumes(A, oracle):
    """vc_fast_carve resets the volumes itself: every refusal must come before that reset and leave the carved state"""
    dims = (45, 30, 20)
    rng = np.random.default_rng(61)
    W, H, V = 96, 72, 5
    P, M = _views(rng, V, W, H, dims)
    bits = _masks(rng, V, W, H)
    ro, rs = oracle.carve(*dims, S, P, W, H, mask_bits=bits)

    def unchanged(e, what):
        _same(e.download_occupied(), ro, f"occupied after {what}")
        _same(e.download_seen(), rs, f"seen after {what}")

    with _engine_with(A, dims, P, M, W, H, bits) as e:
        e.carve(0)
        unchanged(e, "the carve")
        _state_error(A, VC_ERR_ARG, e.fast_carve, 7)
        unchanged(e, "fast_carve with an unknown mode (VC_ERR_ARG)")
        P2, M2 = _views(rng, V, 80, 60, dims)
        e.set_views(P2, 80, 60, M2)          # a new W x H: the masks are dropped
        _state_error(A, VC_ERR_STATE, e.fast_carve, 0)
        unchanged(e, "fast_carve without masks (VC_ERR_STATE)")
    with _engine_with(A, dims, P, M, W, H, bits, z0=0, z1=12) as e:
        e.carve(0)
        _state_error(A, VC_ERR_STATE, e.fast_carve, 0)
        _same(e.download_occupied(), ro[:12], "occupied after fast_carve on a slab (VC_ERR_STATE)")


# ---- 3b. consumers of flags_valid ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flags_valid_consumers_follow_every_state_change(A, oracle):
    """vc_mc_classify takes the brick flags of the last fresh whole-range carve instead of scanning the volumes while
    flags_valid is set.  Every call that changes the volumes or the flags without a fresh carve must clear it; each check here
    compares the histogram with the oracle's on the engine's actual volumes, and the sparse download with the oracle's carve"""
    import torch
    dims = X, Y, Z = (100, 40, 36)
    rng = np.random.default_rng(21)
    W, H, V = 96, 72, 7
    P, M = _views(rng, V, W, H, dims)
    b1, b2 = _masks(rng, V, W, H), _masks(rng, V, W, H, specks=0.02)
    ro1, rs1 = oracle.carve(*dims, S, P, W, H, mask_bits=b1)

    def mc_matches(e, what):
        e.mc_classify()
        hist, na, nt = e.download_mc()
        occ = e.download_occupied()
        rh, rna, rnt = oracle.mc_classify(X, Y, Z, occ)
        assert np.array_equal(hist, rh) and (na, nt) == (rna, rnt), f"flags_valid: cube-index histogram is stale after {what}"
        return occ

    def sparse_matches(e, bits, what):
        flags, listed, words = e.carve_download_sparse()
        o, s = e.expand_sparse(flags, listed, words)
        ro, rs = oracle.carve(*dims, S, P, W, H, mask_bits=bits)
        _same(o, ro, f"sparse download (occupied) after {what}")
        _same(s, rs, f"sparse download (seen) after {what}")

    with _engine_with(A, dims, P, M, W, H, b1) as e, A.VoxelEngine(*dims, S) as scan:
        e.carve(0)
        occ = mc_matches(e, "a fresh carve (flag path)")
        _same(occ, ro1, "occupied of the fresh carve")
        scan.upload_volumes(occ, e.download_seen())   # the same volumes through the scan path
        scan.mc_classify()
        assert all(np.array_equal(a, b) for a, b in zip(scan.download_mc(), e.download_mc())), "flag path and scan path disagree"

        transitions = [
            ("a sub-range carve with new masks and no reset", lambda: (e.set_masks_bits(b2), e.carve(0, 1, 4))),
            ("a whole-range carve with new masks and no reset", lambda: (e.set_masks_bits(b2), e.carve(0))),
            ("upload_volumes", lambda: e.upload_volumes(*_random_state(rng, X, Y, Z))),
            ("fast_carve", lambda: e.fast_carve()),
            ("plan_slabs (classifies without touching the volumes)", lambda: (e.set_masks_bits(b2), e.plan_slabs(2))),
            ("plan_slabs with every pixel background (its flags call every brick carved)",
             lambda: (e.set_masks_bits(np.full_like(b1, 0xffffffff)), e.plan_slabs(2))),
            ("set_slab (volumes reset)", lambda: e.set_slab(0, Z)),
            ("alloc_full_volumes (volumes reset)", lambda: e.alloc_full_volumes()),
        ]
        empty = np.full_like(b1, 0xffffffff)   # every brick carved whole: the flag path answers every interior cell from the flags
        for (what, change), start in [(t, b) for t in transitions for b in (b1, empty)]:
            e.set_masks_bits(start)
            e.reset()
            e.carve(0)
            mc_matches(e, "a fresh carve")
            change()
            mc_matches(e, what)
            e.set_masks_bits(b1)
            sparse_matches(e, b1, what)
            mc_matches(e, f"the sparse download after {what}")
        # caller-owned whole-grid buffers
        n = Z * Y * ((X + 31) // 32)
        bo, bs = torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        e.set_masks_bits(b1)
        e.reset()
        e.carve(0)
        e.bind_volumes(bo.data_ptr(), bs.data_ptr())
        occ = mc_matches(e, "bind_volumes (volumes reset)")
        _same(occ, np.broadcast_to(_valid(X), occ.shape), "occupied after bind_volumes")
        sparse_matches(e, b1, "bind_volumes")
        e.synchronize()
        del bo, bs


# ---- 3c. vc_dense_apply_carved: the -intermediateMesh chain ----------------------------------------------------------------
@pytest.mark.gpu
def test_dense_apply_carved_intermediate_mesh_chain(A, oracle):
    """the reference's -intermediateMesh: carve one view at a time into a Model that already holds state, set every carved
    voxel to 0 (VoxelCarving.cpp:52) and take a mesh of it after each view (VoxelCarving.cpp:65-68)"""
    dims = X, Y, Z = (45, 30, 20)
    rng = np.random.default_rng(31)
    W, H, V = 96, 72, 5
    P, M = _views(rng, V, W, H, dims)
    bits = _masks(rng, V, W, H, specks=0.01)
    n = X * Y * Z
    rgba = np.zeros((n, 4), np.float32)
    rgba[:, :3] = rng.integers(0, 256, (n, 3))
    rgba[:, 3] = rng.choice([0.0, 0.2, 0.45, 0.5, 0.8, 1.0], n)
    m = EngineModel(oracle, X, Y, Z)
    m.P, m.M, m.bits, m.W, m.H = P, M, bits, W, H
    with _engine_with(A, dims, P, M, W, H, bits) as e:
        for start in ("reset", "upload_volumes"):
            if start == "reset":
                e.reset()
                m.reset()
            else:
                occ0, seen0 = _random_state(rng, X, Y, Z)
                e.upload_volumes(occ0, seen0)
                m.upload(occ0, seen0)
            e.dense_upload(rgba)
            m.dense_upload(rgba)
            e.dense_apply_carved()
            m.dense_apply_carved()
            _same(e.dense_download().view(np.uint32), m.dense.view(np.uint32), f"dense Model right after {start}")
            for i in range(V):
                e.carve(0, i, i + 1)
                m.carve(i, i + 1)
                verts, rgb = e.mc_mesh(0.5)        # the mesh of the Model before this view's carve is applied
                e.dense_apply_carved()
                _state_error(A, VC_ERR_STATE, e.download_mesh, len(verts))   # have_mesh: the Model changed under the mesh
                m.dense_apply_carved()
                _same(e.dense_download().view(np.uint32), m.dense.view(np.uint32), f"dense Model after view {i} ({start})")
                verts, rgb = e.mc_mesh(0.5)
                m.mc_mesh()
                _same(verts, m.mesh[0], f"mesh vertices after view {i} ({start})")
                _same(rgb, m.mesh[1], f"mesh colours after view {i} ({start})")
            assert len(verts) > 0
    with _engine_with(A, dims, P, M, W, H, bits) as e:
        _state_error(A, VC_ERR_STATE, e.dense_apply_carved)   # no dense Model yet
    with _engine_with(A, dims, P, M, W, H, bits, z0=4, z1=12) as e:
        e.carve(0)
        _state_error(A, VC_ERR_STATE, e.dense_apply_carved)   # a slab engine


# ---- 3d. caller streams and device masks -----------------------------------------------------------------------------------
def _pack_bits_torch(bgr):
    """8UC3 masks (a CUDA tensor) -> bit masks int32[V][H][ceil(W/32)], 1 = background, with torch ops on the current stream"""
    import torch
    bg = (bgr == 0).all(-1)
    V, H, W = bg.shape
    Ww = (W + 31) // 32
    pad = torch.zeros((V, H, Ww * 32), dtype=torch.int64, device=bgr.device)
    pad[..., :W] = bg.to(torch.int64)
    w = (pad.view(V, H, Ww, 32) << torch.arange(32, device=bgr.device)).sum(-1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32).contiguous()


def _busy(stream, a):
    """a few tens of milliseconds of matrix products queued on `stream`"""
    import torch
    with torch.cuda.stream(stream):
        x = a
        for _ in range(24):
            x = (x @ a) * (1.0 / 64)
    return x


@pytest.mark.gpu
def test_caller_stream_orders_device_masks_and_every_call(A, oracle, tmp_path):
    """with vc_set_stream(s), the engine runs behind whatever the caller queued on s: masks packed on the GPU by torch ops on s,
    behind a long kernel, must be read only once they are written.  set_masks_bits_device queues its copy without a host
    synchronisation, so those scenarios check the ordering; vc_append_views synchronises the stream on entry, so the append
    scenario checks its results only.  The graph carve, the chunked page-locked download, colour, mesh and text all run on s."""
    import torch
    dims = X, Y, Z = (40, 20, 72)
    rng = np.random.default_rng(41)
    W, H, V, n_app = 96, 72, 6, 3
    P, M = _views(rng, V + n_app, W, H, dims)
    bits_a, bits_b = _masks(rng, V + n_app, W, H), _masks(rng, V + n_app, W, H, specks=0.02)
    images = rng.integers(0, 256, (V + n_app, H, W, 3), dtype=np.uint8)
    a = torch.randn(4096, 4096, device="cuda")
    bgr_a = torch.from_numpy(_bgr_of_bits(rng, bits_a, W)).cuda()
    bgr_b = torch.from_numpy(_bgr_of_bits(rng, bits_b, W)).cuda()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    m = EngineModel(oracle, X, Y, Z)
    m.P, m.M, m.W, m.H, m.images = P[:V], M[:V], W, H, images[:V]
    n = Z * Y * ((X + 31) // 32)
    po, ps = (torch.empty(n, dtype=torch.int32).pin_memory() for _ in range(2))
    keep = []

    def queue_masks(bgr):
        _busy(s, a)
        with torch.cuda.stream(s):
            t = _pack_bits_torch(bgr)
        keep.append(t)
        return t

    def check_all(e, what):
        e.reset()
        e.carve(0)                                      # a fresh graph carve on s
        m.reset()
        m.carve()
        _same(e.download_occupied(), m.occ, f"occupied ({what})")
        e.reset()
        e.carve_download(po, ps)                        # two z-chunks, copies on the engine's copy stream behind s
        _same(po.numpy().view(np.uint32).reshape(m.shape), m.occ, f"chunked download's occupied ({what})")
        _same(ps.numpy().view(np.uint32).reshape(m.shape), m.seen, f"chunked download's seen ({what})")
        e.color(2)
        m.color(2)
        verts, rgb = e.mesh_from_volumes(True, True, 3)
        m.mesh_from_volumes(True, True, 3)
        _same(verts, m.mesh[0], f"mesh ({what})")
        nb = e.format_off(S, (F(0.5), F(-0.25), F(0)))
        m.text = m.off_text(tmp_path, S, (F(0.5), F(-0.25), F(0)))
        assert nb == len(m.text)
        check_engine(A, e, m)

    with A.VoxelEngine(X, Y, Z, S) as e:
        e.set_views(P[:V], W, H, M[:V])
        e.set_images(images[:V])
        e.set_stream(s.cuda_stream)
        e.set_masks_bits_device(queue_masks(bgr_a[:V]).data_ptr())   # no host synchronisation in between
        m.bits = bits_a[:V]
        check_all(e, "device masks queued on the caller's stream")
        t = queue_masks(bgr_b[V:])
        e.append_views(P[V:], M[V:], mask_bits=t, images_bgr=images[V:])
        m.P, m.M, m.bits, m.images = P, M, np.concatenate([bits_a[:V], bits_b[V:]]), images
        check_all(e, "device masks appended behind the caller's stream")
        e.set_stream(None)                              # back to the engine's own stream: the graph captured on s replays there
        e.set_masks_bits(bits_b)
        m.bits = bits_b
        check_all(e, "set_stream(None) after the graph was captured on the caller's stream")
    with A.VoxelEngine(X, Y, Z, S) as e:                # captured on the own stream, then replayed on s
        e.set_views(P, W, H, M)
        e.set_images(images)
        e.set_masks_bits(bits_a)
        m.bits = bits_a
        e.carve(0)
        e.set_stream(s.cuda_stream)
        e.set_masks_bits_device(queue_masks(bgr_b).data_ptr())
        m.bits = bits_b
        check_all(e, "a graph captured on the own stream, replayed on the caller's stream")
    torch.cuda.synchronize()


# ---- 3e. grow-only buffers -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_grow_only_buffers_large_small_large(A, oracle, tmp_path):
    """colour records, mesh, text, sparse lists and the shared scratch only ever grow: results must not depend on what an
    earlier, larger or smaller call left in them.  The carve of an uploaded state with carved-but-unseen voxels (which keeps the
    uploaded occupancy in the scratch) runs right after calls that left the scratch at other sizes"""
    dims = X, Y, Z = (70, 40, 30)
    rng = np.random.default_rng(51)
    W, H, V = 96, 72, 6
    P, M = _views(rng, V, W, H, dims)
    images = rng.integers(0, 256, (V, H, W, 3), dtype=np.uint8)
    noisy = _masks(rng, V, W, H, specks=0.05)
    empty = np.full_like(noisy, 0xffffffff)   # every pixel background: every brick is carved whole, none is listed
    m = EngineModel(oracle, X, Y, Z)
    m.P, m.M, m.W, m.H, m.images = P, M, W, H, images
    small_occ = np.zeros((Z, Y, (X + 31) // 32), np.uint32)
    small_occ[10:14, 10:14, 0] = 0xf0
    big_occ, big_seen = _random_state(rng, X, Y, Z)
    sizes = []
    with _engine_with(A, dims, P, M, W, H, noisy, images) as e:
        for label, occ, bits in (("large", big_occ, noisy), ("small", small_occ, empty), ("large again", big_occ, noisy)):
            e.upload_volumes(occ, big_seen)
            m.upload(occ, big_seen)
            e.color(1)
            m.color(1)
            n_records = len(m.colors[0])
            verts, _ = e.mesh_from_volumes(True, False, 3)
            m.mesh_from_volumes(True, False, 3)
            nb = e.format_off(F(1.0))
            m.text = m.off_text(tmp_path, F(1.0), (F(0), F(0), F(0)))
            assert nb == len(m.text)
            check_engine(A, e, m)
            e.set_masks_bits(bits)
            m.bits = bits
            flags, listed, words = e.carve_download_sparse()
            m.reset()
            m.carve()
            o, s = e.expand_sparse(flags, listed, words)
            _same(o, m.occ, f"sparse occupied ({label})")
            _same(s, m.seen, f"sparse seen ({label})")
            sizes.append((n_records, len(verts), nb, len(listed)))
            # the carved-but-unseen carve right after mesh_from_volumes (scratch: counts + dilated volume) ...
            e.mesh_from_volumes(False, False, 5, download=False)
            m.mesh_from_volumes(False, False, 5)
            occ0, seen0 = _random_state(rng, X, Y, Z)
            e.upload_volumes(occ0, seen0)
            m.upload(occ0, seen0)
            e.carve(0)
            m.carve()
            check_engine(A, e, m)
            # ... and right after fast_carve (scratch: flood volume)
            e.fast_carve()
            m.fast_carve()
            check_engine(A, e, m)
            occ0, seen0 = _random_state(rng, X, Y, Z)
            e.upload_volumes(occ0, seen0)
            m.upload(occ0, seen0)
            e.carve(2, 1, V)
            m.carve(1, V)
            check_engine(A, e, m)
    (c0, t0, x0, l0), (c1, t1, x1, l1) = sizes[0], sizes[1]
    assert c1 < c0 and t1 < t0 and x1 < x0 and l1 < l0, f"the small pass must be smaller in every buffer: {sizes}"
