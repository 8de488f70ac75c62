"""VoxelEngine — thin object wrapper over the C ABI (include/voxcarve.h).

Host-side mirror of the reference's hot path: grid = Model(x, y, z, size) (Model.h:108), inputs =
cached per-view P / M matrices and undistorted masks / images (VoxelCarving.cpp:25-36), outputs =
bit-packed occupied / seen volumes, per-surface-voxel colours, cube-index histogram.
All compute happens in libvoxcarve.so on the GPU; this file only marshals pointers.
"""
import ctypes as C

import numpy as np

from . import _lib as L


class VoxCarveError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"voxcarve error {code}: {msg}")
        self.code = code


def _host_ptr(a, dtype, nbytes_min, what):
    """numpy array or CPU torch tensor -> (address, keepalive). Checks dtype, contiguity and size."""
    if hasattr(a, "data_ptr"):  # torch tensor (e.g. pinned host memory)
        if a.is_cuda:
            raise ValueError(f"{what}: expected HOST memory")
        if not a.is_contiguous():
            raise ValueError(f"{what}: tensor must be contiguous")
        nbytes = a.numel() * a.element_size()
        got = np.dtype(str(a.dtype).replace("torch.", ""))
        if got.itemsize != np.dtype(dtype).itemsize or got.kind not in "iu":  # torch has no uint32 arithmetic: int32 is fine
            raise ValueError(f"{what}: dtype {a.dtype}, expected {np.dtype(dtype)}")
        addr, keep = a.data_ptr(), a
    else:
        keep = np.ascontiguousarray(a, dtype=dtype)
        nbytes, addr = keep.nbytes, keep.ctypes.data
    if nbytes < nbytes_min:
        raise ValueError(f"{what}: buffer has {nbytes} bytes, needs {nbytes_min}")
    return addr, keep


def _host_out_ptr(a, nbytes_min, what):
    """OUTPUT buffer (numpy array or CPU torch tensor) -> address.  Never copies: the library writes through this pointer, so
    the buffer must be 4-byte integer typed, C-contiguous and writeable as it stands."""
    if hasattr(a, "data_ptr"):
        addr, _ = _host_ptr(a, np.uint32, nbytes_min, what)
        return addr
    if not isinstance(a, np.ndarray):
        raise TypeError(f"{what}: output buffer must be a numpy array or a CPU torch tensor, got {type(a).__name__}")
    if a.dtype not in (np.dtype(np.uint32), np.dtype(np.int32)):
        raise ValueError(f"{what}: dtype {a.dtype}, expected uint32 (or int32)")
    if not a.flags["C_CONTIGUOUS"] or not a.flags["WRITEABLE"]:
        raise ValueError(f"{what}: output buffer must be C-contiguous and writeable")
    if a.nbytes < nbytes_min:
        raise ValueError(f"{what}: buffer has {a.nbytes} bytes, needs {nbytes_min}")
    return a.ctypes.data


class VoxelEngine:
    """One engine = one GPU = one z-slab [z_begin, z_end) of an X*Y*Z grid."""

    def __init__(self, X, Y, Z, voxel_size, z_begin=0, z_end=None, device=0):
        self._lib = L.load()
        self._h = C.c_void_p()
        z_end = Z if z_end is None else z_end
        g = L.GridDesc(int(X), int(Y), int(Z), float(np.float32(voxel_size)), int(z_begin), int(z_end), int(device))
        rc = self._lib.vc_create(C.byref(g), C.byref(self._h))
        if rc != L.VC_OK:
            msg = self._lib.vc_last_error(None).decode()
            self._h = C.c_void_p()
            raise VoxCarveError(rc, msg)
        self.X, self.Y, self.Z, self.voxel_size = int(X), int(Y), int(Z), np.float32(voxel_size)
        self.z_begin, self.z_end, self.device = int(z_begin), int(z_end), int(device)
        self.Wx = (self.X + 31) // 32
        self.V = self.W = self.H = 0
        self._keep = []

    # -- plumbing ------------------------------------------------------------------------
    def _check(self, rc):
        if rc != L.VC_OK:
            raise VoxCarveError(rc, self._lib.vc_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.vc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.vc_set_stream(self._h, C.c_void_p(cuda_stream_ptr or 0)))

    def set_profiling(self, on=True):
        """plain launches + an event between classification and per-voxel kernel (stats()['last_classify_ms']) instead of one CUDA graph"""
        self._check(self._lib.vc_set_profiling(self._h, int(bool(on))))

    def synchronize(self):
        self._check(self._lib.vc_synchronize(self._h))

    @property
    def slab_shape(self):
        return (self.z_end - self.z_begin, self.Y, self.Wx)

    @property
    def slab_words(self):
        n = C.c_uint64()
        self._check(self._lib.vc_slab_words(self._h, C.byref(n)))
        return n.value

    # -- inputs --------------------------------------------------------------------------
    def set_views(self, P, W, H, M=None):
        P = np.ascontiguousarray(P, np.float32).reshape(-1, 12)
        V = P.shape[0]
        Mp = None
        if M is not None:
            M = np.ascontiguousarray(M, np.float32).reshape(-1, 12)
            if M.shape[0] != V:
                raise ValueError("M and P must have the same number of views")
            Mp = M.ctypes.data
        self._check(self._lib.vc_set_views(self._h, V, int(W), int(H), P.ctypes.data, Mp))
        self.V, self.W, self.H = V, int(W), int(H)

    def append_views(self, P, M=None, mask_bits=None, mask_bgr=None, raw=False, images_bgr=None):
        """append views [V, V+n) of the engine's W x H geometry (vc_append_views): P (and M, iff the engine's views have M), their
        masks (mask_bits uint32[n][H][ceil(W/32)], host array or a CUDA tensor; or mask_bgr uint8[n][H][W][3], distorted if raw),
        and their images iff the engine holds images (raw: distorted, like the masks).  Only the new views' tables are built."""
        P = np.ascontiguousarray(P, np.float32).reshape(-1, 12)
        n = P.shape[0]
        Mp = None
        if M is not None:
            M = np.ascontiguousarray(M, np.float32).reshape(-1, 12)
            if M.shape[0] != n:
                raise ValueError("M and P must have the same number of views")
            Mp = M.ctypes.data
        if (mask_bits is None) == (mask_bgr is None):
            raise ValueError("append_views needs exactly one of mask_bits / mask_bgr")
        Ww = (self.W + 31) // 32
        if mask_bits is not None:
            if raw:
                raise ValueError("raw masks are 8UC3 images: pass them as mask_bgr")
            fmt = L.VC_MASK_BITS
            if hasattr(mask_bits, "is_cuda") and mask_bits.is_cuda:
                if not mask_bits.is_contiguous() or mask_bits.numel() * mask_bits.element_size() < n * self.H * Ww * 4:
                    raise ValueError("device mask bits: must be contiguous and hold n*H*ceil(W/32) words")
                maddr, mkeep = mask_bits.data_ptr(), mask_bits
            else:
                maddr, mkeep = _host_ptr(mask_bits, np.uint32, n * self.H * Ww * 4, "mask bits")
        else:
            fmt = L.VC_MASK_BGR8_RAW if raw else L.VC_MASK_BGR8
            maddr, mkeep = _host_ptr(mask_bgr, np.uint8, n * self.H * self.W * 3, "mask bgr")
        iaddr = None
        if images_bgr is not None:
            iaddr, ikeep = _host_ptr(images_bgr, np.uint8, n * self.H * self.W * 3, "images bgr")
        self._check(self._lib.vc_append_views(self._h, n, P.ctypes.data, Mp, C.c_void_p(maddr), fmt,
                                              None if iaddr is None else C.c_void_p(iaddr)))
        self.V += n

    def set_masks_bits(self, bits):
        """uint32[V][H][ceil(W/32)], 1 = background (carve)."""
        need = self.V * self.H * ((self.W + 31) // 32) * 4
        addr, keep = _host_ptr(bits, np.uint32, need, "mask bits")
        self._check(self._lib.vc_set_masks(self._h, C.c_void_p(addr), L.VC_MASK_BITS))
        self.synchronize()  # host buffer may be pageable / temporary

    def set_masks_bgr(self, bgr, sync=True):
        """uint8[V][H][W][3] undistorted 8UC3 masks (VoxelCarving.cpp:36)."""
        addr, keep = _host_ptr(bgr, np.uint8, self.V * self.H * self.W * 3, "mask bgr")
        self._check(self._lib.vc_set_masks(self._h, C.c_void_p(addr), L.VC_MASK_BGR8))
        if sync:
            self.synchronize()
        else:
            self._keep = [keep]

    def set_masks_bits_async(self, bits):
        need = self.V * self.H * ((self.W + 31) // 32) * 4
        addr, keep = _host_ptr(bits, np.uint32, need, "mask bits")
        self._check(self._lib.vc_set_masks(self._h, C.c_void_p(addr), L.VC_MASK_BITS))
        self._keep = [keep]

    def set_masks_bits_device(self, device_ptr):
        """bit-packed silhouettes already on the GPU (same layout): device-to-device copy + summed-area tables, no host sync"""
        self._check(self._lib.vc_set_masks(self._h, C.c_void_p(int(device_ptr)), L.VC_MASK_BITS))

    def set_calibration(self, K, dist):
        """camera matrix (3x3) and distortion coefficients (4, 5 or 8) for the on-device cv::undistort"""
        K = np.ascontiguousarray(K, np.float64).reshape(9)
        d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())
        self._check(self._lib.vc_set_calibration(self._h, C.c_void_p(K.ctypes.data), C.c_void_p(d.ctypes.data), len(d)))

    def set_masks_raw(self, bgr):
        """distorted 8UC3 masks as cv::imread delivers them; undistorted (VoxelCarving.cpp:36) and packed on the device"""
        addr, keep = _host_ptr(bgr, np.uint8, self.V * self.H * self.W * 3, "raw mask bgr")
        self._check(self._lib.vc_set_masks(self._h, C.c_void_p(addr), L.VC_MASK_BGR8_RAW))
        self.synchronize()

    def set_images_raw(self, images_bgr):
        addr, keep = _host_ptr(images_bgr, np.uint8, self.V * self.H * self.W * 3, "raw images bgr")
        self._check(self._lib.vc_set_images_raw(self._h, C.c_void_p(addr)))

    def download_masks(self):
        out = np.empty((self.V, self.H, (self.W + 31) // 32), np.uint32)
        self._check(self._lib.vc_download_masks(self._h, C.c_void_p(out.ctypes.data)))
        return out

    def download_images(self):
        out = np.empty((self.V, self.H, self.W, 3), np.uint8)
        self._check(self._lib.vc_download_images(self._h, C.c_void_p(out.ctypes.data)))
        return out

    def set_images(self, images_bgr):
        addr, keep = _host_ptr(images_bgr, np.uint8, self.V * self.H * self.W * 3, "images bgr")
        self._check(self._lib.vc_set_images(self._h, C.c_void_p(addr)))
        self.synchronize()

    # -- hot path ------------------------------------------------------------------------
    def reset(self):
        self._check(self._lib.vc_reset(self._h))

    def carve(self, mode=L.VC_EXACT, view_begin=0, view_end=-1, count_executed=False):
        self._check(self._lib.vc_carve(self._h, mode, view_begin, view_end, int(bool(count_executed))))

    def carve_download(self, out_occ=None, out_seen=None, mode=L.VC_EXACT):
        """carve all views and download both volumes, D2H of finished z-chunks overlapped with the carving of the next"""
        n = (self.z_end - self.z_begin) * self.Y * self.Wx
        if out_occ is None:
            out_occ, out_seen = np.empty(self.slab_shape, np.uint32), np.empty(self.slab_shape, np.uint32)
        a = _host_out_ptr(out_occ, n * 4, "occupied buffer")
        b = _host_out_ptr(out_seen, n * 4, "seen buffer")
        self._check(self._lib.vc_carve_download(self._h, mode, C.c_void_p(a), C.c_void_p(b), n))
        return out_occ, out_seen

    def carve_download_sparse(self, flags=None, listed=None, words=None):
        """fresh carve (reset implied) + download in sparse form: (flags uint8[nbz, nby, nbx], listed uint32[n], words uint32[n, 2, 64]).
        Optional preallocated (e.g. pinned) buffers: flags of nbx*nby*nbz bytes, listed / words with room for the listed bricks."""
        nbx, nby, nbz = C.c_uint32(), C.c_uint32(), C.c_uint32()
        self._check(self._lib.vc_sparse_dims(self._h, C.byref(nbx), C.byref(nby), C.byref(nbz)))
        nb = nbx.value * nby.value * nbz.value
        own = flags is None
        if own:
            cap = max(1024, nb // 16)
            flags, listed, words = np.empty(nb, np.uint8), np.empty(cap, np.uint32), np.empty(cap * 128, np.uint32)
        else:
            cap = min(listed.numel() if hasattr(listed, "numel") else listed.size, (words.numel() if hasattr(words, "numel") else words.size) // 128)
        fa = flags.data_ptr() if hasattr(flags, "data_ptr") else flags.ctypes.data
        n = C.c_uint64()
        for attempt in range(2):
            la = listed.data_ptr() if hasattr(listed, "data_ptr") else listed.ctypes.data
            wa = words.data_ptr() if hasattr(words, "data_ptr") else words.ctypes.data
            self.reset()
            rc = self._lib.vc_carve_download_sparse(self._h, C.c_void_p(fa), nb, C.c_void_p(la), C.c_void_p(wa), cap, C.byref(n))
            if rc == L.VC_ERR_CAPACITY and own and n.value > cap and attempt == 0:
                cap = n.value
                listed, words = np.empty(cap, np.uint32), np.empty(cap * 128, np.uint32)
                continue
            self._check(rc)
            break
        k = n.value
        if hasattr(flags, "numpy"):
            flags, listed, words = flags.numpy(), listed.numpy(), words.numpy()
        return (flags[:nb].view(np.uint8).reshape(nbz.value, nby.value, nbx.value), listed[:k].view(np.uint32),
                words[:k * 128].view(np.uint32).reshape(k, 2, 64))

    def expand_sparse(self, flags, listed, words):
        """sparse result -> (occupied, seen) uint32[nz, Y, Wx], the same words carve_download delivers (host side, numpy)"""
        nz, Y, Wx, X = self.z_end - self.z_begin, self.Y, self.Wx, self.X
        nbz, nby, nbx = flags.shape
        valid = np.full(Wx, 0xffffffff, np.uint32)
        if X % 32:
            valid[-1] = (1 << (X % 32)) - 1
        f = np.repeat(np.repeat(flags, 8, axis=0), 8, axis=1)[:nz, :Y]       # per (z, y, word)
        occ = np.where(f & 1, np.uint32(0), valid[None, None, :]).astype(np.uint32)
        seen = np.where(f & 2, valid[None, None, :], np.uint32(0)).astype(np.uint32)
        if len(listed):
            b = listed.astype(np.int64)
            bx, by, bz = b % nbx, (b // nbx) % nby, b // (nbx * nby)
            r = np.arange(64)
            z = (bz[:, None] * 8 + r[None, :] // 8)
            y = (by[:, None] * 8 + r[None, :] % 8)
            ok = (z < nz) & (y < Y)
            xx = np.broadcast_to(bx[:, None], z.shape)
            occ[z[ok], y[ok], xx[ok]] = words[:, 0, :][ok]
            seen[z[ok], y[ok], xx[ok]] = words[:, 1, :][ok]
        return occ, seen

    def fast_carve(self, mode=L.VC_EXACT):
        self._check(self._lib.vc_fast_carve(self._h, mode))

    def color(self, mode):
        self._check(self._lib.vc_color(self._h, int(mode)))

    def color_visible(self, mode, tolerance=2.0):
        """occlusion-aware colouring (vc_color_visible): each surface voxel is coloured from the views that see it; a view is
        occluded when another surface voxel lies more than `tolerance` voxel sizes in front of it.  Whole-grid engines only."""
        self._check(self._lib.vc_color_visible(self._h, int(mode), float(tolerance)))

    def mc_classify(self):
        self._check(self._lib.vc_mc_classify(self._h))

    # -- multi-GPU plumbing --------------------------------------------------------------
    def plan_slabs(self, n_parts):
        """balanced contiguous z-slab boundaries (n_parts + 1 ints) from the super-brick classification of this engine's range"""
        b = (C.c_int32 * (n_parts + 1))()
        self._check(self._lib.vc_plan_slabs(self._h, int(n_parts), b))
        return list(b)

    def set_slab(self, z_begin, z_end):
        self._check(self._lib.vc_set_slab(self._h, int(z_begin), int(z_end)))
        self.z_begin, self.z_end = int(z_begin), int(z_end)

    def bind_volumes(self, d_occ_full_ptr, d_seen_full_ptr):
        self._check(self._lib.vc_bind_volumes(self._h, C.c_void_p(d_occ_full_ptr), C.c_void_p(d_seen_full_ptr)))

    def device_volumes(self):
        a, b = C.c_void_p(), C.c_void_p()
        self._check(self._lib.vc_device_volumes(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_gathered(self, flag=True):
        self._check(self._lib.vc_set_gathered(self._h, int(bool(flag))))

    def alloc_full_volumes(self):
        """engine-owned whole-grid buffers (what gather() fills); resets the state"""
        self._check(self._lib.vc_alloc_full_volumes(self._h))

    # one-plane halos of `occupied` (what the colour / cube-index passes of a slab need from its neighbours)
    def halo_words(self):
        n = C.c_uint64()
        self._check(self._lib.vc_halo_words(self._h, C.byref(n)))
        return n.value

    def export_halo(self, which):
        """device pointer of the slab's first (0) / last (1) plane"""
        p = C.c_void_p()
        self._check(self._lib.vc_export_halo(self._h, int(which), C.byref(p)))
        return p.value

    def import_halo(self, which, device_ptr):
        """copy a neighbour's plane into plane z_begin - 1 (which = 0) / z_end (which = 1); None drops it"""
        self._check(self._lib.vc_import_halo(self._h, int(which), C.c_void_p(device_ptr or 0)))

    # NCCL communicator inside libvoxcarve.so: one rank per GPU, slabs in rank order along z
    def comm_init(self, rank, world, unique_id):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._check(self._lib.vc_comm_init(self._h, int(rank), int(world), buf))

    def comm_destroy(self):
        self._check(self._lib.vc_comm_destroy(self._h))

    def comm_info(self):
        r, w, v = C.c_int32(), C.c_int32(), C.c_int32()
        self._check(self._lib.vc_comm_info(self._h, C.byref(r), C.byref(w), C.byref(v)))
        return {"rank": r.value, "world": w.value, "nccl_version": v.value}

    def exchange_halos(self):
        self._check(self._lib.vc_exchange_halos(self._h))

    def gather(self, bounds, occupied=True, seen=False):
        """assemble the whole grid in the bound / engine-owned whole-grid buffers of every rank (in place, over NCCL)"""
        b = (C.c_int32 * len(bounds))(*[int(x) for x in bounds])
        self._check(self._lib.vc_gather(self._h, (1 if occupied else 0) | (2 if seen else 0), b))

    def download_full(self, which=0):
        """the whole (gathered) grid out of the whole-grid buffers: which = 0 occupied, 1 seen -> uint32[Z, Y, Wx]"""
        out = np.empty((self.Z, self.Y, self.Wx), np.uint32)
        self._check(self._lib.vc_download_full(self._h, int(which), C.c_void_p(out.ctypes.data), out.size))
        return out

    def allreduce_u64(self, values):
        """element-wise sum over the ranks of the communicator -> numpy uint64 (identity without a communicator)"""
        a = np.ascontiguousarray(values, np.uint64).copy()
        self._check(self._lib.vc_comm_allreduce_u64(self._h, C.c_void_p(a.ctypes.data), a.size))
        return a

    def upload_volumes(self, occ_words, seen_words):
        n = (self.z_end - self.z_begin) * self.Y * self.Wx
        a, ka = _host_ptr(occ_words, np.uint32, n * 4, "occupied words")
        b, kb = _host_ptr(seen_words, np.uint32, n * 4, "seen words")
        self._check(self._lib.vc_upload_volumes(self._h, C.c_void_p(a), C.c_void_p(b), n))

    # -- outputs -------------------------------------------------------------------------
    def download_occupied(self, out=None):
        return self._download(self._lib.vc_download_occupied, out)

    def download_seen(self, out=None):
        return self._download(self._lib.vc_download_seen, out)

    def _download(self, fn, out):
        n = (self.z_end - self.z_begin) * self.Y * self.Wx
        if out is None:
            out = np.empty(self.slab_shape, np.uint32)
            addr = out.ctypes.data
        else:
            addr = _host_out_ptr(out, n * 4, "download buffer")
        self._check(fn(self._h, C.c_void_p(addr), n))
        return out

    def count_occupied(self):
        a, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.vc_count_occupied(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def surface_count(self):
        """surface voxels coloured by the last color() call (ColorReconstruction.h:46: occupied and not isInner)"""
        n = C.c_uint64()
        self._check(self._lib.vc_surface_count(self._h, C.byref(n)))
        return int(n.value)

    def download_colors(self):
        n = C.c_uint64()
        self._check(self._lib.vc_surface_count(self._h, C.byref(n)))
        idx = np.empty(n.value, np.uint64)
        rgbn = np.empty((n.value, 4), np.uint8)
        self._check(self._lib.vc_download_colors(self._h, C.c_void_p(idx.ctypes.data), C.c_void_p(rgbn.ctypes.data), n.value))
        return idx, rgbn

    def download_mc(self):
        hist = np.zeros(256, np.uint64)
        na, nt = C.c_uint64(), C.c_uint64()
        self._check(self._lib.vc_download_mc(self._h, C.c_void_p(hist.ctypes.data), C.byref(na), C.byref(nt)))
        return hist, na.value, nt.value

    # -- "next" rows: dense Model, closure, marching-cubes mesh ------------------------
    def dense_upload(self, rgba):
        n = self.X * self.Y * self.Z * 16
        a, keep = _host_ptr(np.ascontiguousarray(rgba, np.float32), np.float32, n, "dense rgba")
        self._check(self._lib.vc_dense_upload(self._h, C.c_void_p(a)))

    def dense_from_volumes(self, apply_colors=False, handle_unseen=False):
        self._check(self._lib.vc_dense_from_volumes(self._h, int(bool(apply_colors)), int(bool(handle_unseen))))

    def dense_apply_carved(self):
        """model.set(x,y,z,0) for every carved voxel on the dense Model already on the device (VoxelCarving.cpp:52)"""
        self._check(self._lib.vc_dense_apply_carved(self._h))

    def dense_closure(self, kernel_size=3):
        self._check(self._lib.vc_dense_closure(self._h, int(kernel_size)))

    def dense_download(self):
        out = np.empty((self.X * self.Y * self.Z, 4), np.float32)
        self._check(self._lib.vc_dense_download(self._h, C.c_void_p(out.ctypes.data)))
        return out

    def mc_mesh(self, threshold=0.5):
        """-> (verts float32[T,3,3] in voxel-index coordinates, rgb uint32[T,3]) in the reference's emission order"""
        n = C.c_uint64()
        self._check(self._lib.vc_mc_mesh(self._h, C.c_float(threshold), C.byref(n)))
        return self.download_mesh(n.value)

    def mesh_from_volumes(self, apply_colors=False, handle_unseen=False, closure_k=0, threshold=0.5, download=True):
        """marchingCubes of the Model dense_from_volumes(apply_colors, handle_unseen) [+ dense_closure(closure_k)] would build,
        from the bit volumes and colour records without the dense Model (closure_k = 0: no closure).  Same (verts, rgb) as
        that chain + mc_mesh(threshold); download=False leaves the mesh on the device and returns its triangle count."""
        n = C.c_uint64()
        self._check(self._lib.vc_mesh_from_volumes(self._h, int(bool(apply_colors)), int(bool(handle_unseen)), int(closure_k),
                                                    C.c_float(threshold), C.byref(n)))
        return self.download_mesh(n.value) if download else int(n.value)

    def download_mesh(self, n_triangles):
        """the mesh the last mc_mesh / mesh_from_volumes left on the device: (verts float32[T,3,3], rgb uint32[T,3])"""
        verts = np.empty((n_triangles, 3, 3), np.float32)
        rgb = np.empty((n_triangles, 3), np.uint32)
        self._check(self._lib.vc_download_mesh(self._h, C.c_void_p(verts.ctypes.data), C.c_void_p(rgb.ctypes.data), n_triangles))
        return verts, rgb

    def format_off(self, scale=1.0, translation=(0.0, 0.0, 0.0)):
        """format the .off text of the mesh on the device (SimpleMesh::WriteMesh, vertex = index coordinates * scale + translation
        in f32) and keep it there; -> its size in bytes"""
        n = C.c_uint64()
        tx, ty, tz = (C.c_float(t) for t in translation)
        self._check(self._lib.vc_mesh_format_off(self._h, C.c_float(scale), tx, ty, tz, C.byref(n)))
        return int(n.value)

    def download_mesh_off(self, offset, n_bytes):
        """bytes [offset, offset + n_bytes) of the text format_off left on the device"""
        out = np.empty(int(n_bytes), np.uint8)
        self._check(self._lib.vc_download_mesh_off(self._h, int(offset), C.c_void_p(out.ctypes.data), int(n_bytes)))
        return out.tobytes()

    def mesh_off(self, scale=1.0, translation=(0.0, 0.0, 0.0)):
        """the whole .off file of the mesh the last mc_mesh / mesh_from_volumes left on the device, formatted on the device"""
        return self.download_mesh_off(0, self.format_off(scale, translation))

    def write_mesh_off(self, path, scale=1.0, translation=(0.0, 0.0, 0.0), chunk=64 << 20):
        """mesh_off written to `path`, downloaded in chunks of `chunk` bytes through one buffer"""
        n = self.format_off(scale, translation)
        buf = np.empty(min(n, int(chunk)), np.uint8)
        with open(path, "wb") as f:
            for o in range(0, n, len(buf)):
                k = min(len(buf), n - o)
                self._check(self._lib.vc_download_mesh_off(self._h, o, C.c_void_p(buf.ctypes.data), k))
                f.write(memoryview(buf)[:k])
        return n

    # -- probes (tests) ------------------------------------------------------------------
    def probe_boxes(self, boxes):
        """the carve's brick classifier on boxes int32[n, 7] = (view, x0, y0, z0, x1, y1, z1), inclusive, global z (vc_probe_boxes)
        -> int32[n, 5] = (code, px0, px1, py0, py1)"""
        b = np.ascontiguousarray(boxes, np.int32).reshape(-1, 7)
        out = np.zeros((len(b), 5), np.int32)
        self._check(self._lib.vc_probe_boxes(self._h, len(b), C.c_void_p(b.ctypes.data), C.c_void_p(out.ctypes.data)))
        return out

    def probe_voxels(self, voxels):
        """the carve's per-voxel filter and exact evaluation on voxel-views int32[n, 4] = (view, x, y, z), global z (vc_probe_voxels)
        -> int32[n, 11] = (decided, inside, px, py, exact inside, exact px, exact py, then the bits of Cu, Cv, hDu, hDv)"""
        v = np.ascontiguousarray(voxels, np.int32).reshape(-1, 4)
        out = np.zeros((len(v), 11), np.int32)
        self._check(self._lib.vc_probe_voxels(self._h, len(v), C.c_void_p(v.ctypes.data), C.c_void_p(out.ctypes.data)))
        return out

    def stats(self):
        s = L.Stats()
        self._check(self._lib.vc_get_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in L.Stats._fields_}


def comm_unique_id():
    """128-byte NCCL id made by rank 0 and handed to every rank's VoxelEngine.comm_init"""
    lib = L.load()
    buf = C.create_string_buffer(128)
    rc = lib.vc_comm_unique_id(buf)
    if rc != L.VC_OK:
        raise VoxCarveError(rc, lib.vc_last_error(None).decode())
    return buf.raw


def exchange_halos_peer(engines):
    """engines of THIS process whose slabs tile a z-range: everyone receives its neighbours' boundary planes (device copies)"""
    lib = L.load()
    arr = (C.c_void_p * len(engines))(*[e._h for e in engines])
    rc = lib.vc_exchange_halos_peer(arr, len(engines))
    if rc != L.VC_OK:
        bad = [e for e in engines if e._lib.vc_last_error(e._h)]
        raise VoxCarveError(rc, "; ".join(e._lib.vc_last_error(e._h).decode() for e in bad))


def gather_peer(engines, occupied=True, seen=False):
    """engines of THIS process whose slabs tile the grid: everyone's whole-grid buffers get all slabs (peer copies over NVLink)"""
    lib = L.load()
    arr = (C.c_void_p * len(engines))(*[e._h for e in engines])
    rc = lib.vc_gather_peer(arr, len(engines), (1 if occupied else 0) | (2 if seen else 0))
    if rc != L.VC_OK:
        raise VoxCarveError(rc, "; ".join(e._lib.vc_last_error(e._h).decode() for e in engines if e._lib.vc_last_error(e._h)))


def measure_peaks(device=0):
    """Measured CUDA-core FFMA / DFMA peaks (TFLOP/s) of `device` — roofline denominators for bench.py."""
    lib = L.load()
    a, b = C.c_double(), C.c_double()
    rc = lib.vc_measure_peaks(int(device), C.byref(a), C.byref(b))
    if rc != L.VC_OK:
        raise VoxCarveError(rc, lib.vc_last_error(None).decode())
    return a.value, b.value


def selftest(which, n, seed=0, device=0):
    """GPU self-test of the arithmetic shortcuts (0: shared-reciprocal divide, 1: pixel index, 2: packed f32 pairs). -> (mismatches, checked)"""
    lib = L.load()
    a, b = C.c_uint64(), C.c_uint64()
    rc = lib.vc_selftest(int(device), int(which), int(n), int(seed), C.byref(a), C.byref(b))
    if rc != L.VC_OK:
        raise VoxCarveError(rc, lib.vc_last_error(None).decode())
    return a.value, b.value


def format_g(values, device=0):
    """printf("%g\\n") of every float32 of `values`, formatted on the GPU with the code of VoxelEngine.format_off -> bytes"""
    lib = L.load()
    v = np.ascontiguousarray(values, np.float32).reshape(-1)
    need = C.c_uint64()
    text = np.empty(13 * len(v), np.uint8)  # at most 12 characters and a newline per value
    rc = lib.vc_format_g(int(device), len(v), C.c_void_p(v.ctypes.data), C.c_void_p(text.ctypes.data), len(text), C.byref(need))
    if rc != L.VC_OK:
        raise VoxCarveError(rc, lib.vc_last_error(None).decode())
    return text[:need.value].tobytes()


def undistort_bgr(images_bgr, K, dist, device=0):
    """cv::undistort of uint8[n,H,W,3] (or [H,W,3]) on the GPU, bit-exact with OpenCV's 8UC3 path"""
    lib = L.load()
    img = np.ascontiguousarray(images_bgr, np.uint8)
    single = img.ndim == 3
    if single:
        img = img[None]
    n, H, W, _ = img.shape
    Kc = np.ascontiguousarray(K, np.float64).reshape(9)
    d = np.ascontiguousarray(np.asarray(dist, np.float64).ravel())
    out = np.empty_like(img)
    rc = lib.vc_undistort_bgr(int(device), n, W, H, C.c_void_p(img.ctypes.data), C.c_void_p(Kc.ctypes.data), C.c_void_p(d.ctypes.data), len(d),
                              C.c_void_p(out.ctypes.data))
    if rc != L.VC_OK:
        raise VoxCarveError(rc, lib.vc_last_error(None).decode())
    return out[0] if single else out
