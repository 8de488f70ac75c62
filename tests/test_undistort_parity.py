"""cv::undistort parity against cv2 itself (DESIGN §8 f-4).  The contract is what cv2 4.13.0 computes on x86-64 with its AVX2
code path, for images with both sides below 32767.  The sweep of tests/golden/undistort_hostile_kat.npz (written by
tools/make_goldens.py: undistort_hostile_cases) holds the dataset calibration at three sizes, random calibrations, round-number
camera matrices whose map coordinates sit on rounding ties, distortion strong enough to leave int16 and int32, a rational
denominator that reaches 0 inside the image, and widths for every column count of cv2's scalar tail and for its row stripes.
Every case is a noise image from a seed, so every pixel is checked.

Where cv2 4.13.0 runs with AVX2, the oracle and the device are compared with the live cv2.undistort (and the live answer with
the pinned one); elsewhere with the pinned answers.  The device is then checked through every path raw input takes."""
import hashlib

import numpy as np
import pytest

F = np.float32
KAT = "undistort_hostile_kat.npz"


def _live_cv2():
    try:
        import cv2
    except ImportError:
        return None
    return cv2 if cv2.__version__ == "4.13.0" and cv2.checkHardwareSupport(11) else None  # 11 = CV_CPU_AVX2


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def kat(golden):
    z = golden(KAT)
    cases = []
    for n in z["names"]:
        W, H, seed = (int(v) for v in z[f"{n}_WHseed"])
        cases.append(dict(name=str(n), W=W, H=H, seed=seed, K=z[f"{n}_K"], dist=z[f"{n}_dist"], sha=str(z[f"{n}_sha256"]),
                          src_sha=str(z[f"{n}_src_sha256"]), dst=z[f"{n}_dst"] if f"{n}_dst" in z else None))
    return cases


def _image(c, k=0):
    img = np.random.default_rng(c["seed"] + 7919 * k).integers(0, 256, (c["H"], c["W"], 3), dtype=np.uint8)
    if k == 0:
        assert _sha(img) == c["src_sha"], f"{c['name']}: the seeded input differs from the one the answers were made from"
    return img


def _reference(c, img, k=0):
    """cv2.undistort of the case's k-th image: live where the contract's cv2 runs, else the pinned answer (image 0 only)"""
    cv2 = _live_cv2()
    if cv2 is not None:
        ref = cv2.undistort(img, c["K"], c["dist"])
        if k == 0:
            assert _sha(ref) == c["sha"], f"{c['name']}: live cv2 differs from the pinned answer"
        return ref
    assert k == 0
    return c["dst"]


def _explain(c, got, ref):
    """the first mismatching pixels with the int16 map of both sides"""
    from oracle import oracle as O
    bad = np.argwhere((got != ref).any(-1))
    msg = [f"{c['name']} W={c['W']} H={c['H']} K={c['K'].tolist()} dist={c['dist'].tolist()}: {len(bad)} pixels differ"]
    sxy, frac = O.undistort_map(c["K"], c["dist"], c["W"], c["H"])
    cv2 = _live_cv2()
    stripe = min(max(1, 4096 // c["W"]), c["H"])
    for y, x in bad[:5]:
        line = f"  pixel (x={x}, y={y}): got {got[y, x].tolist()} want {ref[y, x].tolist()}; oracle map {sxy[y, x].tolist()} frac {frac[y, x]}"
        if cv2 is not None:
            y0 = y // stripe * stripe
            Kp = c["K"].copy()
            Kp[1, 2] -= y0
            m1, m2 = cv2.initUndistortRectifyMap(c["K"], c["dist"], None, Kp, (c["W"], min(stripe, c["H"] - y0)), cv2.CV_16SC2)
            line += f"; cv2 map {m1[y - y0, x].tolist()} frac {m2[y - y0, x]}"
        msg.append(line)
    return "\n".join(msg)


# ---- CPU: the oracle against cv2 ------------------------------------------------------------------------------------------
def test_kat_covers_the_hostile_cases(kat, golden):
    """the pinned sweep holds what it claims: every W % 8 twice, W = 1, H = 1, W = 32766, a stripe of one row, stripes that do
    not divide H, map coordinates past int16 and past int32 in the body and in the tail, and pixels whose map is NaN"""
    from oracle import oracle as O
    z = golden(KAT)
    assert str(z["cv2_version"]) == "4.13.0" and str(z["dispatch"]) == "AVX2"
    Ws = [c["W"] for c in kat]
    assert all(sum(W % 8 == r for W in Ws) >= 2 for r in range(8))
    assert 1 in Ws and 32766 in Ws and 1 in [c["H"] for c in kat] and any(W > 4096 for W in Ws)
    assert any(c["H"] % min(max(1, 4096 // c["W"]), c["H"]) for c in kat)
    seen = set()
    for c in kat:
        if c["W"] * c["H"] > 200000:
            continue
        sxy, frac = O.undistort_map(c["K"], c["dist"], c["W"], c["H"])
        W8 = c["W"] - c["W"] % 8
        body, tail = sxy[:, :W8].astype(np.int32), sxy[:, W8:].astype(np.int32)
        if (body == -32768).any() or (body == 32767).any():
            seen.add("body int16")
        if (np.abs(tail) >= 1024).any() and c["name"].startswith("int16"):
            seen.add("tail wraps")
        if c["name"].startswith(("int32", "den0")) and ((sxy == -32768).any() or (tail == 0).any()):
            seen.add(c["name"].split("_")[0])
    assert {"body int16", "tail wraps", "int32", "den0"} <= seen, seen


def test_oracle_matches_cv2_on_the_hostile_sweep(kat, oracle):
    """oracle.undistort == cv2.undistort byte for byte on every case (live cv2 where it is 4.13.0 with AVX2, else the pinned
    output or its SHA-256)"""
    fails = []
    for c in kat:
        img = _image(c)
        got = oracle.undistort(img, c["K"], c["dist"])
        ref = _reference(c, img)
        if ref is None:
            if _sha(got) != c["sha"]:
                fails.append(f"{c['name']}: SHA-256 of the output differs from the pinned answer")
        elif not np.array_equal(got, ref):
            fails.append(_explain(c, got, ref))
    assert not fails, "\n".join(fails)


def test_oracle_map_is_cv2s_map(kat):
    """the oracle's int16 map equals cv2.initUndistortRectifyMap(CV_16SC2) for the first stripe of every case (live cv2 only)"""
    from oracle import oracle as O
    cv2 = _live_cv2()
    if cv2 is None:
        pytest.skip("needs cv2 4.13.0 with AVX2")
    for c in kat:
        rows = min(max(1, 4096 // c["W"]), c["H"])
        sxy, frac = O.undistort_map(c["K"], c["dist"], c["W"], rows)
        m1, m2 = cv2.initUndistortRectifyMap(c["K"], c["dist"], None, c["K"], (c["W"], rows), cv2.CV_16SC2)
        assert np.array_equal(sxy, m1) and np.array_equal(frac, m2), c["name"]


def test_oracle_refuses_what_cv2_refuses(oracle):
    img = np.zeros((2, 32767, 3), np.uint8)
    with pytest.raises(ValueError):
        oracle.undistort(img, np.eye(3), [0.1, 0, 0, 0])
    with pytest.raises(ValueError):
        oracle.undistort(np.zeros((32767, 1, 3), np.uint8), np.eye(3), [0.1, 0, 0, 0])
    cv2 = _live_cv2()
    if cv2 is not None:
        with pytest.raises(cv2.error):
            cv2.undistort(img, np.eye(3), np.array([0.1, 0, 0, 0]))


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def A(lib_built):
    import ar_voxel_project_b200 as A
    return A


@pytest.mark.gpu
def test_device_undistort_matches_cv2_on_the_hostile_sweep(A, kat, oracle):
    """vc_undistort_bgr == cv2.undistort on every case, three images per call (the second and third are compared with live
    cv2, or with the oracle, which the CPU tests hold to cv2)"""
    from ar_voxel_project_b200.engine import undistort_bgr
    fails = []
    for c in kat:
        imgs = np.stack([_image(c, k) for k in range(3)])
        got = undistort_bgr(imgs, c["K"], c["dist"])
        for k in range(3):
            ref = _reference(c, imgs[k], k) if k == 0 or _live_cv2() else oracle.undistort(imgs[k], c["K"], c["dist"])
            if ref is None:
                if _sha(got[k]) != c["sha"]:
                    fails.append(f"{c['name']}: SHA-256 of the device output differs from the pinned answer")
            elif not np.array_equal(got[k], ref):
                fails.append(_explain(c, got[k], ref) + f" (image {k})")
    assert not fails, "\n".join(fails)


# a tie-heavy round-number calibration at the engine's geometry: many map coordinates sit on or next to .5 ties of u * 32, where
# evaluating the map in another order than cv2 flips the rounding (138 pixels of a 163x120 noise image)
TIE_K = np.array([[200.0, 0, 82.0], [0, 200.0, 60.0], [0, 0, 1]])
TIE_DIST = np.array([0.5, 0.0, 0.0, 0.0])
W_E, H_E = 163, 120  # 163 % 8 = 3 columns of scalar tail


def _views(V, seed):
    """V cameras around a 64x48x40 grid, raw 8UC3 masks (an ellipse whose pixels are nonzero noise, background (0,0,0)) and
    raw noise images"""
    from ar_voxel_project_b200.synth import gemm_k_m_f32
    rng = np.random.default_rng(seed)
    X, Y, Z, s = 64, 48, 40, F(0.01)
    c = np.array([(Y - 1) * float(s) / 2, (X - 1) * float(s) / 2, -(Z - 1) * float(s) / 2])
    dist = 3.0 * float(s) * 64 * 1.5
    P, M, masks = [], [], []
    yy, xx = np.mgrid[0:H_E, 0:W_E]
    for v in range(V):
        az, el = 2 * np.pi * (v % 16 + 0.3) / 16 + rng.uniform(-0.01, 0.01), np.deg2rad(25.0 if v % 2 else 55.0)
        eye = c + dist * np.array([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), -np.sin(el)])
        zc = (c - eye) / np.linalg.norm(c - eye)
        xc = np.cross(zc, [0.0, 0.0, -1.0])
        xc /= np.linalg.norm(xc)
        R = np.stack([xc, np.cross(zc, xc), zc])
        m = np.concatenate([R, (-R @ eye)[:, None]], axis=1).astype(F)
        k = np.array([[0.25 * W_E * 3, 0, W_E / 2], [0, 0.25 * W_E * 3, H_E / 2], [0, 0, 1]], F)
        P.append(gemm_k_m_f32(k, m)), M.append(m)
        fg = ((xx - W_E / 2) / (W_E * rng.uniform(0.15, 0.3))) ** 2 + ((yy - H_E / 2) / (H_E * rng.uniform(0.15, 0.3))) ** 2 <= 1
        mk = rng.integers(1, 256, (H_E, W_E, 3), dtype=np.uint8)
        mk[~fg] = 0
        masks.append(mk)
    images = rng.integers(0, 256, (V, H_E, W_E, 3), dtype=np.uint8)
    return (X, Y, Z, s), np.stack(P), np.stack(M), np.stack(masks), images


def _undistorted(x):
    cv2 = _live_cv2()
    from oracle import oracle as O
    return np.stack([cv2.undistort(m, TIE_K, TIE_DIST) if cv2 else O.undistort(m, TIE_K, TIE_DIST) for m in x])


@pytest.mark.gpu
def test_engine_raw_paths_match_cv2_past_256_views(A, oracle):
    """set_masks_raw / set_images_raw for 8 views, then 256 more raw views through vc_append_views: the engine holds exactly
    the cv2-undistorted masks (packed) and images; a carve, an average and a closest colour pass from that raw input equal the
    oracle run on the cv2-undistorted inputs"""
    from ar_voxel_project_b200.synth import pack_bits
    (X, Y, Z, s), P, M, raw_masks, raw_images = _views(264, seed=31)
    und_masks, und_images = _undistorted(raw_masks), _undistorted(raw_images)
    with A.VoxelEngine(X, Y, Z, s) as e:
        e.set_views(P[:8], W_E, H_E, M[:8])
        e.set_calibration(TIE_K, TIE_DIST)
        e.set_masks_raw(raw_masks[:8])
        e.set_images_raw(raw_images[:8])
        assert np.array_equal(e.download_masks(), pack_bits((und_masks[:8] == 0).all(-1)))
        assert np.array_equal(e.download_images(), und_images[:8])
        for v in range(8, 264, 64):
            e.append_views(P[v:v + 64], M[v:v + 64], mask_bgr=raw_masks[v:v + 64], raw=True, images_bgr=raw_images[v:v + 64])
        assert e.V == 264
        assert np.array_equal(e.download_masks(), pack_bits((und_masks == 0).all(-1)))
        assert np.array_equal(e.download_images(), und_images)
        e.reset()
        e.carve()
        occ, seen = e.download_occupied(), e.download_seen()
        colors = {}
        for mode in (A._lib.VC_COLOR_AVG, A._lib.VC_COLOR_CLOSEST):
            e.color(mode)
            colors[mode] = e.download_colors()
    ro, rs = oracle.carve(X, Y, Z, s, P, W_E, H_E, mask_bgr=und_masks, nthreads=0)
    assert np.array_equal(occ, ro) and np.array_equal(seen, rs)
    assert 0 < int(oracle.unpack(ro, X).sum()) < X * Y * Z
    for mode, (idx, rgbn) in colors.items():
        ridx, rrgbn = oracle.color(X, Y, Z, s, P, M, W_E, H_E, und_images, ro, mode)
        assert len(ridx) > 0 and np.array_equal(idx, ridx) and np.array_equal(rgbn, rrgbn), f"colour mode {mode}"


@pytest.mark.gpu
def test_raw_input_of_32767_or_more_is_refused_and_changes_nothing(A):
    """cv::undistort refuses a side of 32767 or more (remap's SHRT_MAX): vc_undistort_bgr, raw vc_set_masks, vc_set_images_raw
    and raw vc_append_views return VC_ERR_ARG, and the engine keeps its views, masks and images"""
    from ar_voxel_project_b200.engine import undistort_bgr
    from ar_voxel_project_b200.synth import pack_bits
    K, dist = np.array([[100.0, 0, 50], [0, 100, 20], [0, 0, 1]]), [0.1, 0, 0, 0]
    for shape in [(1, 2, 32767, 3), (1, 32767, 1, 3)]:
        with pytest.raises(A.VoxCarveError) as ex:
            undistort_bgr(np.zeros(shape, np.uint8), K, dist)
        assert ex.value.code == A._lib.VC_ERR_ARG
    assert undistort_bgr(np.zeros((1, 2, 32766, 3), np.uint8), K, dist).shape == (1, 2, 32766, 3)
    X, Y, Z, s = 32, 8, 8, F(0.01)
    P = np.tile(np.array([[1, 0, 0, 16], [0, 1, 0, 1], [0, 0, 0, 1]], F)[None], (2, 1, 1))
    for W, H in [(32767, 2), (3, 32767)]:
        rng = np.random.default_rng(W)
        bgr = rng.integers(0, 2, (2, H, W, 3), dtype=np.uint8) * 255
        bits = pack_bits((bgr == 0).all(-1))
        with A.VoxelEngine(X, Y, Z, s) as e:
            e.set_views(P, W, H, P)
            e.set_masks_bgr(bgr)
            e.set_images(bgr)
            e.set_calibration(K, dist)
            for call in (lambda: e.set_masks_raw(bgr), lambda: e.set_images_raw(bgr),
                         lambda: e.append_views(P[:1], P[:1], mask_bgr=bgr[:1], raw=True, images_bgr=bgr[:1])):
                with pytest.raises(A.VoxCarveError) as ex:
                    call()
                assert ex.value.code == A._lib.VC_ERR_ARG
                assert (e.V, e.W, e.H) == (2, W, H)
                assert np.array_equal(e.download_masks(), bits) and np.array_equal(e.download_images(), bgr)
            e.append_views(P[:1], P[:1], mask_bgr=bgr[:1], images_bgr=bgr[:1])  # the same append with undistorted masks is taken
            assert e.V == 3 and np.array_equal(e.download_masks()[2], bits[0])
