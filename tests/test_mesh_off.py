"""The .off text formatted on the device (vc_mesh_format_off / vc_download_mesh_off / vc_format_g) against the C library's printf
and the oracle's C writer (SimpleMesh::WriteMesh, MarchingCubes.h:59-87).  Every comparison is of bytes, not parsed numbers."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


@pytest.fixture(scope="module")
def printf_g(tmp_path_factory):
    """values -> the text glibc's snprintf("%g\\n") makes of them (tests/cpp/printf_g.c, one thread per CPU)"""
    so = str(tmp_path_factory.mktemp("printf_g") / "libprintf_g.so")
    subprocess.check_call(["cc", "-O2", "-shared", "-fPIC", "-pthread", os.path.join(ROOT, "tests", "cpp", "printf_g.c"), "-o", so])
    lib = C.CDLL(so)
    lib.ref_format_g.restype = C.c_uint64
    lib.ref_format_g.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_int]

    def fmt(values):
        v = np.ascontiguousarray(values, np.float32).reshape(-1)
        out = np.empty(13 * len(v) + 1, np.uint8)
        n = lib.ref_format_g(v.ctypes.data, len(v), out.ctypes.data, os.cpu_count() or 1)
        return out[:n].tobytes()
    return fmt


def _f32(bits):
    return np.asarray(bits, np.uint64).astype(np.uint32).view(np.float32)


def _same_text(got, exp, what=""):
    if got == exp:
        return
    a, b = got.split(b"\n"), exp.split(b"\n")
    i = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
    pytest.fail(f"{what}: texts differ ({len(got)} vs {len(exp)} bytes, {len(a)} vs {len(b)} lines); first at line {i}: "
                f"{a[i][:120] if i < len(a) else None!r} vs {b[i][:120] if i < len(b) else None!r}")


def _check_g(A, printf_g, values, what):
    values = np.ascontiguousarray(values, np.float32)
    _same_text(A.engine.format_g(values), printf_g(values), what)


# ---- %g of single floats -----------------------------------------------------------------------------------------------
def test_format_g_examples(A):
    vals = [123456.5, 123457.5, 1234565.0, 999999.5, 1e-5, 12345.25, 100000.0, 0.0001, 0.00012345678, 1.5e-45, 3.4028235e38]
    assert A.engine.format_g(np.array(vals, np.float32)) == (
        b"123456\n123458\n1.23456e+06\n1e+06\n1e-05\n12345.2\n100000\n0.0001\n0.000123457\n1.4013e-45\n3.40282e+38\n")
    assert A.engine.format_g(np.zeros(0, np.float32)) == b""


def test_format_g_every_float_from_2p17_to_2p24(A, printf_g):
    """[2^17, 2^24) holds every float with a .5 tie (2^17..2^23) and the integer ties of 7-digit values (2^23..2^24)"""
    lo, hi = np.float32(2.0 ** 17).view(np.uint32), np.float32(2.0 ** 24).view(np.uint32)
    bits = np.arange(int(lo), int(hi), dtype=np.uint32)
    _check_g(A, printf_g, bits.view(np.float32), "[2^17, 2^24)")
    _check_g(A, printf_g, (bits | np.uint32(0x80000000)).view(np.float32)[::7], "-[2^17, 2^24)")


def test_format_g_every_high_half_with_16_low_halves(A, printf_g):
    rng = np.random.default_rng(17)
    low = np.concatenate([np.array([0, 1, 2, 0x7fff, 0x8000, 0xfffe, 0xffff, 0x5555, 0xaaaa], np.uint32),
                          rng.integers(0, 1 << 16, 7, dtype=np.uint32)])
    hi = np.arange(1 << 16, dtype=np.uint32) << np.uint32(16)
    _check_g(A, printf_g, (hi[:, None] | low[None, :]).reshape(-1).view(np.float32), "high halves x low halves")


def test_format_g_random_patterns(A, printf_g):
    bits = np.random.default_rng(2024).integers(0, 1 << 32, 1 << 24, dtype=np.uint64).astype(np.uint32)
    _check_g(A, printf_g, bits.view(np.float32), "2^24 random patterns")


def test_format_g_special_values(A, printf_g):
    bits = [0x0, 0x80000000,                                   # +-0
            0x1, 0x80000001, 0x2, 0x3, 0x7, 0x10, 0x3ff, 0x12345, 0x7fffff, 0x807fffff, 0x400000, 0x00654321,  # denormals
            0x00800000, 0x80800000,                            # FLT_MIN
            0x7f7fffff, 0xff7fffff,                            # +-FLT_MAX
            0x7f800000, 0xff800000,                            # +-inf
            0x7fc00000, 0xffc00000, 0x7f800001, 0xff800001, 0x7fffffff, 0xffffffff, 0x7fa00000]  # quiet / signalling +-NaN
    _check_g(A, printf_g, _f32(bits), "special values")
    vals = np.array([123456.5, 123457.5, 1234565.0, 999999.5, 9999995.0, 99999.95, 0.000099999995, 12345.25, 1e-5, 1e-4,
                     0.0001, 999999.0, 1e6, 1e-38, 1e38, 0.5, 0.1, 2.0 ** -149, 2.0 ** -126, 2.0 ** 127], np.float32)
    _check_g(A, printf_g, np.concatenate([vals, -vals]), "ties and decade edges")


# ---- the .off file ---------------------------------------------------------------------------------------------------
def _oracle_off(oracle, tmp_path, verts, rgb, scale, t):
    p = str(tmp_path / "ref.off")
    oracle.write_off(p, verts, rgb, scale, t)
    with open(p, "rb") as f:
        return f.read()


def _nan(neg):
    return float(_f32([0xffc00000 if neg else 0x7fc00000])[0])


def _transforms(s, X, rng):
    inf = float("inf")
    out = [(np.float32(1.5) * s, (0.5, -0.25, 2.0)),                            # the reference's marchingCubes(&model, 1.5, ...)
           (np.float32(1.0) * s, (0.0, 0.0, 0.0)),
           (np.float32(1.0) * s, (float(np.float32(3 * (X + 2)) * s), 0.0, 0.0))]  # the intermediate mesh of view 3
    for _ in range(2):
        out.append((float(np.float32(rng.uniform(-3, 3))), tuple(float(x) for x in rng.uniform(-100, 100, 3).astype(np.float32))))
    return out


def _special_transforms():
    inf, nan, nnan = float("inf"), _nan(False), _nan(True)
    return [(0.0, (0.0, -0.0, 0.0)), (-0.0, (-0.0, -0.0, 1.0)), (inf, (0.0, 1.0, -inf)), (-inf, (inf, 0.0, 0.0)),
            (nan, (0.0, 0.0, 0.0)), (nnan, (1.0, 2.0, 3.0)), (1.0, (nan, nnan, 0.5)), (3e38, (0.0, -3e38, 1e30)),
            (1e-40, (0.0, 1e-45, -1e-42)), (-1e-30, (1e-7, 123456.5, 999999.5))]


@pytest.mark.parametrize("ds,dims", [("box", (50, 50, 25)), ("human", (100, 100, 100))])
def test_mesh_from_volumes_off_vs_oracle_writer(A, oracle, tmp_path, ds, dims):
    vs = A.ViewSet.from_npz(os.path.join(GOLDEN, f"{ds}_views.npz"))
    X, Y, Z = dims
    s = np.float32(0.28) / np.float32(X)
    rng = np.random.default_rng(X)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(vs.P, vs.W, vs.H, vs.M)
        e.set_masks_bits(vs.mask_bits)
        e.set_images(vs.images_bgr)
        e.carve()
        for cm in (0, 1, 2):
            if cm:
                e.color(cm)
            for k in (0, 3):
                verts, rgb = e.mesh_from_volumes(bool(cm), True, k, 0.5)
                assert len(verts) > 0
                for sc, t in _transforms(s, X, rng):
                    _same_text(e.mesh_off(sc, t), _oracle_off(oracle, tmp_path, verts, rgb, sc, t), (cm, k, sc, t))


def test_mc_mesh_general_alpha_off_vs_oracle_writer(A, oracle, tmp_path):
    """vc_mc_mesh on a dense Model with arbitrary alphas: interpolated vertices and colours above 255"""
    X, Y, Z = 23, 19, 17
    rng = np.random.default_rng(5)
    rgba = np.empty((X * Y * Z, 4), np.float32)
    rgba[:, :3] = rng.integers(0, 70000, (X * Y * Z, 3))
    rgba[:, 3] = rng.random(X * Y * Z)
    with A.VoxelEngine(X, Y, Z, 0.01) as e:
        e.dense_upload(rgba)
        for thr in (0.5, 0.3137):
            verts, rgb = e.mc_mesh(thr)
            assert len(verts) > 0 and rgb.max() > 255
            assert not np.array_equal(verts, np.round(verts))
            for sc, t in _transforms(np.float32(0.01), X, rng) + _special_transforms():
                _same_text(e.mesh_off(sc, t), _oracle_off(oracle, tmp_path, verts, rgb, sc, t), (thr, sc, t))


def test_special_scales_and_translations(A, oracle, tmp_path):
    """+-0, +-inf, +-NaN and overflowing scales on a mesh with vertices at coordinate 0 (0 * inf: x86's default NaN, -nan)"""
    from ar_voxel_project_b200.synth import pack_bits
    X, Y, Z = 21, 18, 16
    rng = np.random.default_rng(8)
    occ = rng.random((Z, Y, X)) < 0.4
    with A.VoxelEngine(X, Y, Z, 0.02) as e:
        e.upload_volumes(pack_bits(occ), pack_bits(np.ones_like(occ)))
        verts, rgb = e.mesh_from_volumes(False, True, 0, 0.5)
        assert (verts == 0).any()
        for sc, t in _special_transforms():
            _same_text(e.mesh_off(sc, t), _oracle_off(oracle, tmp_path, verts, rgb, sc, t), (sc, t))
        # the file on disk, written in small chunks through one buffer
        p = str(tmp_path / "chunked.off")
        n = e.write_mesh_off(p, 0.02, (1.0, 2.0, 3.0), chunk=4096 + 13)
        with open(p, "rb") as f:
            got = f.read()
        assert len(got) == n
        _same_text(got, _oracle_off(oracle, tmp_path, verts, rgb, 0.02, (1.0, 2.0, 3.0)), "write_mesh_off")


def test_empty_mesh(A):
    from ar_voxel_project_b200.synth import pack_bits
    with A.VoxelEngine(20, 20, 20, 0.01) as e:
        e.upload_volumes(pack_bits(np.zeros((20, 20, 20), bool)), pack_bits(np.ones((20, 20, 20), bool)))  # everything carved
        assert e.mesh_from_volumes(False, True, 3, 0.5, download=False) == 0
        assert e.mesh_off(1.0, (0.5, 0.5, 0.5)) == b"OFF\n0 0 0\n"
        e.reset()
        assert e.mesh_from_volumes(False, True, 0, 1.5, download=False) == 0  # threshold above every alpha
        assert e.mesh_off() == b"OFF\n0 0 0\n"
        assert e.write_mesh_off(os.devnull) == len(b"OFF\n0 0 0\n")


def test_refusals_keep_the_previous_text(A, oracle, tmp_path):
    from ar_voxel_project_b200.synth import Workload
    w = Workload(40, 4, 96, 64, seed=1)
    with A.VoxelEngine(40, 40, 40, w.s) as e:
        for call in (lambda: e.format_off(), lambda: e.download_mesh_off(0, 1), lambda: e.download_mesh_off(0, 0)):
            with pytest.raises(A.VoxCarveError) as ei:
                call()
            assert ei.value.code == 3
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(w.images_bgr())
        e.carve()
        e.color(2)
        verts, rgb = e.mesh_from_volumes(True, True, 3, 0.5)
        ref = _oracle_off(oracle, tmp_path, verts, rgb, 0.5, (1.0, 2.0, 3.0))
        n = e.format_off(0.5, (1.0, 2.0, 3.0))
        assert n == len(ref) and e.download_mesh_off(0, n) == ref
        assert e.download_mesh_off(n, 0) == b"" and e.download_mesh_off(n - 5, 5) == ref[-5:] and e.download_mesh_off(7, 9) == ref[7:16]
        for off, k in ((n, 1), (0, n + 1), (n + 1, 0), ((1 << 64) - 1, 2), (5, (1 << 64) - 1)):
            assert e._lib.vc_download_mesh_off(e._h, off, None, k) == 1, (off, k)
        with pytest.raises(A.VoxCarveError) as ei:   # a refused mesh call leaves the mesh and so its text
            e.mesh_from_volumes(True, True, 2, 0.5)
        assert ei.value.code == 1
        assert e.download_mesh_off(0, n) == ref
        e.dense_upload(np.zeros((40 ** 3, 4), np.float32))  # no mesh to format any more, the text of the last one stays
        with pytest.raises(A.VoxCarveError) as ei:
            e.format_off(1.0)
        assert ei.value.code == 3
        assert e.download_mesh_off(0, n) == ref
        e.mesh_from_volumes(False, True, 0, 0.5, download=False)  # a new mesh: the text is stale
        with pytest.raises(A.VoxCarveError) as ei:
            e.download_mesh_off(0, 1)
        assert ei.value.code == 3
        v2, c2 = e.download_mesh(e.mesh_from_volumes(False, True, 0, 0.5, download=False))
        _same_text(e.mesh_off(0.5, (1.0, 2.0, 3.0)), _oracle_off(oracle, tmp_path, v2, c2, 0.5, (1.0, 2.0, 3.0)), "new mesh")


def test_c4_file_equals_the_oracle_writers(A, oracle, tmp_path):
    from ar_voxel_project_b200.synth import CONFIGS, Workload
    w = Workload(**CONFIGS["C4"])
    sc, t = np.float32(1.5) * w.s, (0.5, -0.25, 2.0)
    with A.VoxelEngine(w.X, w.Y, w.Z, w.s) as e:
        e.set_views(w.P, w.W, w.H, w.M)
        e.set_masks_bits(w.mask_bits)
        e.set_images(w.images_bgr())
        e.carve()
        e.color(2)
        verts, rgb = e.mesh_from_volumes(True, True, 3, 0.5)
        got = e.mesh_off(sc, t)
    assert len(verts) > 4_000_000
    _same_text(got, _oracle_off(oracle, tmp_path, verts, rgb, sc, t), "C4")


def _digits(a):
    a = np.asarray(a, np.uint64)
    return 1 + np.searchsorted(np.array([10 ** k for k in range(1, 20)], np.uint64), a, side="right").astype(np.int64)


def test_text_beyond_4_gib(A, printf_g):
    """a checkerboard occupancy of 216^3 voxels: 40 M triangles, more than 2^32 bytes of text.  The line windows around byte
    offsets 2^31 (vertex lines) and 2^32 (face lines) and the end of the file equal the oracle's text for those lines, and the
    total equals the length the C library's formatting gives"""
    from ar_voxel_project_b200.synth import pack_bits
    N = 216
    z, y, x = np.indices((N, N, N), dtype=np.int32)
    occ = ((x + y + z) & 1) == 0
    del x, y, z
    sc, t = np.float32(0.28 / 1024), np.array([0.5, -0.25, 2.0], np.float32)
    with A.VoxelEngine(N, N, N, 0.01) as e:
        e.upload_volumes(pack_bits(occ), pack_bits(np.ones_like(occ)))
        del occ
        T = e.mesh_from_volumes(False, False, 0, 0.5, download=False)
        verts, rgb = e.download_mesh(T)
        n = e.format_off(float(sc), tuple(float(v) for v in t))
        assert n > (1 << 32) + (1 << 28)
        # the length of every line, from the C library's text of every coordinate value (vertices sit on voxels: 0..N)
        grid = np.arange(N + 1, dtype=np.float32)
        lens_axis = [np.array([len(s) for s in printf_g((grid * sc) + t[c]).split(b"\n")[:-1]], np.uint8) for c in range(3)]
        iv = verts.reshape(-1, 3)
        assert np.array_equal(iv, np.round(iv)) and iv.min() >= 0 and iv.max() <= N
        ii = iv.astype(np.int16)
        del iv
        vlen = lens_axis[0][ii[:, 0]] + lens_axis[1][ii[:, 1]] + lens_axis[2][ii[:, 2]] + np.uint8(3)
        del ii
        f = np.arange(T, dtype=np.uint64)
        flen = (2 + _digits(3 * f) + _digits(3 * f + 1) + _digits(3 * f + 2) + 6).astype(np.int64)
        del f
        flen += _digits(rgb[:, 0]) + _digits(rgb[:, 1]) + _digits(rgb[:, 2])
        flen = flen.astype(np.uint8)
        header = b"OFF\n%d %d 0\n" % (3 * T, T)
        assert n == len(header) + int(vlen.sum(dtype=np.int64)) + int(flen.sum(dtype=np.int64))
        starts_v = len(header) + np.concatenate([[0], np.cumsum(vlen, dtype=np.int64)])
        starts_f = starts_v[-1] + np.concatenate([[0], np.cumsum(flen, dtype=np.int64)])
        del vlen, flen

        def vertex_lines(a, b):  # vertex lines [a, b): the oracle writer's text of the triangles holding them
            ta, tb = a // 3, (b + 2) // 3
            p = printf_g((verts[ta:tb].reshape(-1, 3) * sc + t).reshape(-1)).split(b"\n")[:-1]
            lines = [b"%s %s %s\n" % tuple(p[3 * i:3 * i + 3]) for i in range(len(p) // 3)]
            return b"".join(lines[a - 3 * ta:b - 3 * ta])

        def face_lines(a, b):
            return b"".join(b"3 %d %d %d %d %d %d\n" % (3 * i, 3 * i + 1, 3 * i + 2, *rgb[i].tolist()) for i in range(a, b))

        assert starts_v[0] < (1 << 31) < starts_f[0] <= (1 << 32)  # one window in the vertex lines, one in the face lines
        for target, starts, lines, n_lines in ((1 << 31, starts_v, vertex_lines, 3 * T), (1 << 32, starts_f, face_lines, T)):
            j = int(np.searchsorted(starts, target, side="right")) - 1
            a, b = max(j - 40, 0), min(j + 40, n_lines)
            exp, start = lines(a, b), int(starts[a])
            assert start <= target < start + len(exp)
            _same_text(e.download_mesh_off(start, len(exp)), exp, f"window at {target}")
        _same_text(e.download_mesh_off(int(starts_f[T - 50]), n - int(starts_f[T - 50])), face_lines(T - 50, T), "end of file")
        _same_text(e.download_mesh_off(0, int(starts_v[60])), header + vertex_lines(0, 60), "start of file")
