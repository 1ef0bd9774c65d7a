"""The resize stage's exactness claim (bytes equal to OpenCV's 8-bit cv::resize(INTER_CUBIC)) on tie-dense planes.

On noise almost no output byte depends on the details of cv::resize's vertical pass (its sum order, no FMA, round-half-even,
the float body / integer tail split at (ow/8)*8, the tap table), so a kernel that got one of them wrong would still pass
the noise tests.  oracle/ties.py builds source planes in which hundreds of bytes are witnesses: bytes where the correct
arithmetic and one of its near misses disagree, spread over every tap phase, the first / last row and column, the tile seams
and both sides of the body / tail boundary.  The CPU tests pin the oracle and the tap builder to OpenCV on them and prove
the planes' power; the GPU tests run every resize path of the library on them, bit for bit against the oracle.  A failure
reports the differing bytes by plane and output class."""
import ctypes as C
import functools
import os

import numpy as np
import pytest

from oracle import ties

# name: (sw, sh, scale, integer scale or 0).  ow mod 8 is 0 where the integer-scale kernel is meant to run (it requires it),
# and 1, 3, 4 or 7 elsewhere, so that the tail columns carry witnesses.  x0.95 is a down-scale the tiled kernel takes (32-row
# tiles); x0.62 one it takes with its per-column horizontal pass (quad_ok = 0: 4 output columns span 5 source columns), which
# only a frame narrower than one 64-column tile can reach; x0.5 and x0.3 take the direct kernel.
MOSAICS = {
    "x2_int": (100, 70, 2.0, 2), "x2_tail4": (98, 70, 2.0, 2), "x4_int": (90, 40, 4.0, 4), "x4_tail4": (91, 40, 4.0, 4),
    "x1.5_tail7": (90, 70, 1.5, 0), "x1.25_tail1": (116, 87, 1.25, 0), "x2.7_tail3": (93, 60, 2.7, 0),
    "x0.95_tail3": (138, 90, 0.95, 0), "x0.62_quad_tail3": (70, 34, 0.62, 0),
    "x0.5_tail1": (146, 120, 0.5, 0), "x0.3_tail7": (237, 150, 0.3, 0),
}

# witnesses each generated plane must hold, per class (the generator is seeded: these are floors, not expectations)
FLOOR_ALL = 40
FLOOR_CLASS = 1
FLOOR_PHASE = 5


def dims(name):
    sw, sh, scale, _ = MOSAICS[name]
    return ties.oracle().out_dims(sw, sh, scale)


@functools.lru_cache(maxsize=None)
def grey(name, seed=1):
    sw, sh, scale, si = MOSAICS[name]
    dw, dh = dims(name)
    return ties.tie_plane(sw, sh, dw, dh, seed=seed, colour=False, scale_int=si)


@functools.lru_cache(maxsize=None)
def colour(name, seed=2):
    sw, sh, scale, si = MOSAICS[name]
    dw, dh = dims(name)
    return ties.tie_plane(sw, sh, dw, dh, seed=seed, colour=True, scale_int=si)


def explain(got, want, name):
    """differing bytes of one output plane, by class: 'class: n' for every class with a difference, and the first few"""
    sw, sh, _, si = MOSAICS[name]
    dw, dh = dims(name)
    d = got.astype(np.int16) != want.astype(np.int16)
    if not d.any():
        return "equal"
    parts = ["%d bytes differ" % int(d.sum())]
    for k, m in ties.classes(dw, dh, si).items():
        if (d & m).any():
            parts.append("%s: %d" % (k, int((d & m).sum())))
    simd_w = (dw // 8) * 8
    ys, xs = np.nonzero(d)
    parts.append("body: %d, tail: %d" % (int((xs < simd_w).sum()), int((xs >= simd_w).sum())))
    px, py = ties.phase_ids(sw, dw), ties.phase_ids(sh, dh)
    parts.append("col phases %s, row phases %s" % (sorted(set(px[xs].tolist()))[:12], sorted(set(py[ys].tolist()))[:12]))
    parts.append("first (y, x, got, want): %s" % [(int(y), int(x), int(got[y, x]), int(want[y, x])) for y, x in zip(ys[:6], xs[:6])])
    return "; ".join(parts)


def want_planes(src, name):
    """the oracle's planes: [Y, Cr, Cb] of a BGR source, [plane] of a grey one"""
    o = ties.oracle()
    dw, dh = dims(name)
    if src.ndim == 3:
        ycc = o.bgr2ycrcb(src)
        return [o.resize_cubic(np.ascontiguousarray(ycc[:, :, k]), dw, dh) for k in range(3)]
    return [o.resize_cubic(src, dw, dh)]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulation, the oracle and the tap builder against OpenCV; the generator's power
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["grey", "colour"])
@pytest.mark.parametrize("name", list(MOSAICS))
def test_emulation_oracle_and_cv2_agree_on_tie_planes(name, kind):
    """oracle.resize_cubic == cv2.resize (IPP off) on every plane, and the generator's emulation == both.  The planes hold
    witnesses on the tail columns and next to the (ow/8)*8 boundary: this is where a wrong simd_w split in the oracle shows."""
    import cv2
    cv2.ipp.setUseIPP(False)
    src = grey(name) if kind == "grey" else colour(name)
    dw, dh = dims(name)
    planes = cv2.split(cv2.cvtColor(src, cv2.COLOR_BGR2YCrCb)) if src.ndim == 3 else [src]
    emu = ties.plane_variants(src, dw, dh)
    for k, (p, want) in enumerate(zip(planes, want_planes(src, name))):
        got_cv2 = cv2.resize(np.ascontiguousarray(p), (dw, dh), interpolation=cv2.INTER_CUBIC)
        assert np.array_equal(want, got_cv2), (k, explain(want, got_cv2, name))
        assert np.array_equal(emu[k]["ref"], want), (k, explain(emu[k]["ref"], want, name))


@pytest.mark.parametrize("kind", ["grey", "colour"])
@pytest.mark.parametrize("name", list(MOSAICS))
def test_tie_planes_have_witnesses_in_every_class(name, kind):
    """each generated plane holds witnesses in every class the kernels distinguish, and each near miss of the vertical pass
    changes far more bytes of it than of noise of the same size"""
    sw, sh, scale, si = MOSAICS[name]
    dw, dh = dims(name)
    src = grey(name) if kind == "grey" else colour(name)
    cls, per_mut = ties.witness_counts(ties.plane_variants(src, dw, dh), sw, sh, dw, dh, si)
    assert cls["all"] >= FLOOR_ALL, cls
    low = {k: v for k, v in cls.items() if not k.startswith("min_") and k != "all" and v < FLOOR_CLASS}
    assert not low, (low, cls)
    if si or scale == 0.5:   # a periodic tap table: every phase of both axes
        assert cls["min_per_col_phase"] >= FLOOR_PHASE and cls["min_per_row_phase"] >= FLOOR_PHASE, cls
    rng = np.random.default_rng(9)
    noise = rng.integers(0, 256, src.shape, dtype=np.uint8)
    _, per_noise = ties.witness_counts(ties.plane_variants(noise, dw, dh), sw, sh, dw, dh, si)
    for m in ("int", "half_up"):
        assert per_mut[m] >= 20 and per_mut[m] >= 8 * max(1, per_noise[m]), (m, per_mut, per_noise)
    if dw % 8:
        assert per_mut["float_tail"] >= 1, per_mut
    # FMA contraction and the summation order: every scale but x2 and down-scales by 2 (their products are exact in FP32)
    if scale not in (2.0, 0.5):
        for m in ("fma", "l2r"):
            assert per_mut[m] >= 10 and per_mut[m] >= 8 * max(1, per_noise[m]), (m, per_mut, per_noise)
    elif kind == "grey" and scale == 2.0:
        assert per_mut["l2r"] >= 1, per_mut


def test_tie_planes_are_deterministic():
    ties_a = ties.tie_plane(40, 30, 80, 60, seed=3)
    assert np.array_equal(ties_a, ties.tie_plane(40, 30, 80, 60, seed=3))


def _taps_numpy(src, dst):
    """cv::resize's table builder restated in numpy float32 (IEEE, one rounding per operation, like the C builds)"""
    f32 = np.float32
    A = f32(-0.75)
    sc = 1.0 / (dst / src)
    d = np.arange(dst, dtype=np.float64)
    f = ((d + 0.5) * sc - 0.5).astype(f32)
    s = np.floor(f).astype(np.int64)
    x = (f - s.astype(f32)).astype(f32)
    x1 = x + f32(1)
    c0 = ((A * x1 - f32(5) * A) * x1 + f32(8) * A) * x1 - f32(4) * A
    c1 = ((A + f32(2)) * x - (A + f32(3))) * x * x + f32(1)
    y = f32(1) - x
    c2 = ((A + f32(2)) * y - (A + f32(3))) * y * y + f32(1)
    c3 = f32(1) - c0 - c1 - c2
    c = np.rint(np.stack([c0, c1, c2, c3], -1) * f32(2048)).astype(np.int64)
    return s, np.clip(c, -32768, 32767)


def _lib_taps(src, dst):
    import srcnn_cpp_b200 as S
    f = S.load_library().srcnn_debug_cubic_taps
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    f.restype = C.c_int
    ofs = np.empty(dst, np.int32)
    coef = np.empty((dst, 4), np.int16)
    assert f(src, dst, ofs.ctypes.data, coef.ctypes.data) == 0
    return ofs, coef


TAP_SIZES = [(n, int(np.float32(n) * np.float32(s))) for s in (2.0, 4.0, 1.5, 1.25, 2.7, 0.95, 0.75, 0.5, 0.3)
             for n in (1, 2, 3, 7, 100, 1001, 4097, 21845, 32768)] + [(32768, 65536), (16384, 65536), (43690, 65536),
                                                                      (24272, 65535), (65536, 65536), (65536, 19660)]


def test_tap_builder_matches_oracle_and_numpy_restatement():
    """build_cubic_taps (the library's, through srcnn_debug_cubic_taps) == orc_cubic_taps == the numpy restatement, every
    sample of every table, sizes up to 65536 where (float)((d + 0.5) * sc - 0.5) can land on the other side of an integer"""
    o = ties.oracle()
    for n, d in TAP_SIZES:
        if d <= 0:
            continue
        ofs_o, coef_o = o.cubic_taps(n, d)
        ofs_l, coef_l = _lib_taps(n, d)
        ofs_n, coef_n = _taps_numpy(n, d)
        assert np.array_equal(ofs_o, ofs_l) and np.array_equal(coef_o, coef_l), (n, d)
        assert np.array_equal(ofs_o, ofs_n) and np.array_equal(coef_o.astype(np.int64), coef_n), (n, d)


@pytest.mark.parametrize("n,d", [(32768, 65536), (16384, 65536), (43690, 65536), (24272, 65535), (2047, 6141), (65536, 19660)])
def test_tap_tables_match_cv2_on_long_rows(n, d):
    """what cv2 implies about the horizontal taps: 48 random rows of n pixels resized to d columns (vertical scale 1, taps
    {0, 2048, 0, 0}: every output byte is round(H / 2048), so a tap off by one moves about one byte in 16 per row)"""
    import cv2
    cv2.ipp.setUseIPP(False)
    rng = np.random.default_rng(n + d)
    p = rng.integers(0, 256, (48, n), dtype=np.uint8)
    got = ties.oracle().resize_cubic(p, d, 48)
    want = cv2.resize(p, (d, 48), interpolation=cv2.INTER_CUBIC)
    assert np.array_equal(got, want), int((got != want).sum())


def test_tap_export_refuses_bad_arguments():
    import srcnn_cpp_b200 as S
    f = S.load_library().srcnn_debug_cubic_taps
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    buf = np.zeros(64, np.int32)
    assert f(0, 4, buf.ctypes.data, buf.ctypes.data) != 0 and f(4, 0, buf.ctypes.data, buf.ctypes.data) != 0
    assert f(4, 4, None, buf.ctypes.data) != 0


def all_bgr():
    """one 4096 x 4096 x 3 image holding every 24-bit value once"""
    v = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)


def test_colour_conversion_exhaustive():
    """oracle.bgr2ycrcb and oracle.ycrcb2bgr == cv2.cvtColor on all 2^24 inputs, both directions"""
    import cv2
    cv2.ipp.setUseIPP(False)
    o = ties.oracle()
    img = all_bgr()
    assert np.array_equal(o.bgr2ycrcb(img), cv2.cvtColor(img, cv2.COLOR_BGR2YCrCb))
    assert np.array_equal(o.ycrcb2bgr(img), cv2.cvtColor(img, cv2.COLOR_YCrCb2BGR))
    assert np.array_equal(ties.bgr2ycc(img[::37, ::41]).astype(np.uint8), o.bgr2ycrcb(img[::37, ::41]))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every resize path on the tie planes, bit for bit against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _planes(n, oh, ow):
    import torch
    pitch = (ow + 127) // 128 * 128
    return [torch.full((oh, pitch), 77, dtype=torch.uint8, device="cuda:0")[:, :ow] for _ in range(n)]


def _engine_with(env):
    """a context created with the given knobs in the environment (they are read when a context is created)"""
    import srcnn_cpp_b200 as S
    import torch
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        eng = S.Engine(device=0, variant=S.VARIANT_TC)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    return eng


# the context knobs that change which kernel or tile height an integer scale takes
INT_NAMES = [k for k in MOSAICS if MOSAICS[k][3]]


@pytest.fixture(scope="module", params=["default", "KA_INT=0", "ISR=5", "ISR=8", "ISR=16"])
def eng_knob(request):
    env = {"default": {}, "KA_INT=0": {"SRCNN_KA_INT": "0"}, "ISR=5": {"SRCNN_KA_ISR": "5"}, "ISR=8": {"SRCNN_KA_ISR": "8"},
           "ISR=16": {"SRCNN_KA_ISR": "16"}}[request.param]
    eng = _engine_with(env)
    yield request.param, eng
    eng.close()


def _check_planes(got, want, name, what):
    bad = [(k, explain(g, w, name)) for k, (g, w) in enumerate(zip(got, want)) if not np.array_equal(g, w)]
    assert not bad, (what, name, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MOSAICS))
def test_colour_stage_on_tie_planes(engine, name):
    _colour_stage(("default", engine), name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", INT_NAMES)
def test_colour_stage_knobs(eng_knob, name):
    _colour_stage(eng_knob, name)


def _colour_stage(eng_knob, name):
    """colour + bicubic (integer-scale kernel at x2 / x4 with ow mod 8 == 0, tiled kernel <64|32, 3>, direct kernel <3> for the
    strong down-scales), BGR and RGB order"""
    import srcnn_cpp_b200 as S
    knob, eng = eng_knob
    src = colour(name)
    dw, dh = dims(name)
    want = want_planes(src, name)
    for order, img in ((S.ORDER_BGR, src), (S.ORDER_RGB, src[:, :, ::-1])):
        pl = _planes(3, dh, dw)
        eng.stage_color_bicubic(_dev(img), MOSAICS[name][2], *pl, order=order)
        eng.sync()
        _check_planes([p.cpu().numpy() for p in pl], want, name, (knob, "order", order))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MOSAICS))
def test_grey_plane_on_tie_planes(engine, name):
    _grey_plane(("default", engine), name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", INT_NAMES)
def test_grey_plane_knobs(eng_knob, name):
    _grey_plane(eng_knob, name)


def _grey_plane(eng_knob, name):
    """one-plane resize (k_gray_bicubic_int, tiled <., 1>, direct <1>), from source pointers 0, 1, 4 and 16 bytes past a
    16-byte boundary (32-bit / 128-bit / byte loads)"""
    import torch
    knob, eng = eng_knob
    sw, sh, scale, _ = MOSAICS[name]
    src = grey(name)
    dw, dh = dims(name)
    want = want_planes(src, name)
    for shift in (0, 1, 4, 16):
        stride = (sw + 31) // 32 * 32 + 32
        buf = torch.zeros(sh * stride + 64, dtype=torch.uint8, device="cuda:0")
        view = buf[shift:shift + sh * stride].view(sh, stride)[:, :sw]
        view.copy_(_dev(src))
        out = _planes(1, dh, dw)[0]
        eng.stage_resize_plane(view, scale, out)
        eng.sync()
        _check_planes([out.cpu().numpy()], want, name, (knob, "shift", shift))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MOSAICS))
def test_alpha_plane_of_four_channel_frames(engine, name):
    """BGRA / RGBA: the alpha bytes of the result are the resize of the source's alpha plane (k_color4_bicubic_int, tiled
    <., 4>, direct <4>); the alpha plane is a tie plane, the colour bytes are a colour tie plane"""
    import srcnn_cpp_b200 as S
    import torch
    src = np.concatenate([colour(name), grey(name)[:, :, None]], -1)
    dw, dh = dims(name)
    want = want_planes(grey(name), name)
    for order in (S.ORDER_BGRA, S.ORDER_RGBA):
        dst = torch.zeros((dh, dw, 4), dtype=torch.uint8, device="cuda:0")
        engine.process_device(_dev(src), MOSAICS[name][2], dst, order=order)
        engine.sync()
        _check_planes([dst[:, :, 3].cpu().numpy()], want, name, ("alpha", order))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["x2_int", "x4_int", "x1.5_tail7", "x0.5_tail1"])
def test_alpha_plane_of_a_batch(engine, name):
    """two frames in one launch (blockIdx.z = frame): each frame's alpha is its own tie plane's resize"""
    import srcnn_cpp_b200 as S
    import torch
    sw, sh, scale, si = MOSAICS[name]
    dw, dh = dims(name)
    alphas = [grey(name), ties.tie_plane(sw, sh, dw, dh, seed=5, scale_int=si)]
    src = np.stack([np.concatenate([colour(name), a[:, :, None]], -1) for a in alphas])
    dst = torch.zeros((2, dh, dw, 4), dtype=torch.uint8, device="cuda:0")
    engine.process_batch_device(_dev(src), scale, dst, order=S.ORDER_BGRA)
    engine.sync()
    for f in range(2):
        _check_planes([dst[f, :, :, 3].cpu().numpy()], want_planes(alphas[f], name), name, ("frame", f))


# 4:2:0 / 4:2:2 frames (even sizes, and an output whose chroma plane is half the luma plane): where the luma output is a
# multiple of 16 wide, x2 / x4 take the one-launch integer kernels (k_yuv_bicubic_int), the others
# the generic kernels per plane
YUV_GEOMS = {"x2_int16": (96, 70, 2.0, 2), "x4_int16": (92, 40, 4.0, 4), "x2_tail4": (98, 70, 2.0, 2), "x1.5": (92, 72, 1.5, 0),
             "x2.7": (92, 60, 2.7, 0), "x0.5": (148, 120, 0.5, 0), "x0.3": (240, 160, 0.3, 0)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(YUV_GEOMS))
def test_yuv420_chroma_on_tie_planes(engine, name):
    """NV12 / I420: the output's U and V planes are the cubic resize of the source's (cv::resize's centre-aligned grid)"""
    import srcnn_cpp_b200 as S
    import torch
    sw, sh, scale, si = YUV_GEOMS[name]
    dw, dh = ties.oracle().out_dims(sw, sh, scale)
    assert dw % 2 == 0 and dh % 2 == 0 and ties.oracle().out_dims(sw // 2, sh // 2, scale) == (dw // 2, dh // 2)
    u = ties.tie_plane(sw // 2, sh // 2, dw // 2, dh // 2, seed=11, scale_int=si)
    v = ties.tie_plane(sw // 2, sh // 2, dw // 2, dh // 2, seed=12, scale_int=si)
    o = ties.oracle()
    want = [o.resize_cubic(u, dw // 2, dh // 2), o.resize_cubic(v, dw // 2, dh // 2)]
    rng = np.random.default_rng(1)
    for order in (S.ORDER_NV12, S.ORDER_I420):
        frame = np.zeros((sh * 3 // 2, sw), np.uint8)
        frame[:sh] = rng.integers(0, 256, (sh, sw), dtype=np.uint8)
        dst = torch.zeros((dh * 3 // 2, dw), dtype=torch.uint8, device="cuda:0")
        _, fu, fv = S.yuv420_planes(frame, order)
        fu[:], fv[:] = u, v
        engine.process_device(_dev(frame), scale, dst, order=order)
        engine.sync()
        _, gu, gv = S.yuv420_planes(dst.cpu().numpy(), order)
        for k, (g, w) in enumerate(zip((gu, gv), want)):
            assert np.array_equal(g, w), (order, k, int((g != w).sum()), np.argwhere(g != w)[:6].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(YUV_GEOMS))
def test_yuv422_chroma_on_tie_planes(engine, name):
    """YUY2 / UYVY: the output's U and V planes (ow/2 x oh) are the cubic resize of the source's (w/2 x h)"""
    import srcnn_cpp_b200 as S
    import torch
    sw, sh, scale, si = YUV_GEOMS[name]
    o = ties.oracle()
    dw, dh = o.out_dims(sw, sh, scale)
    assert dw % 2 == 0 and o.out_dims(sw // 2, sh, scale)[0] == dw // 2
    u = ties.tie_plane(sw // 2, sh, dw // 2, dh, seed=13, scale_int=si)
    v = ties.tie_plane(sw // 2, sh, dw // 2, dh, seed=14, scale_int=si)
    want = [o.resize_cubic(u, dw // 2, dh), o.resize_cubic(v, dw // 2, dh)]
    rng = np.random.default_rng(2)
    for order in (S.ORDER_YUY2, S.ORDER_UYVY):
        frame = np.zeros((sh, sw, 2), np.uint8)
        fy, fu, fv = S.yuv422_planes(frame, order)
        fy[:] = rng.integers(0, 256, (sh, sw), dtype=np.uint8)
        fu[:], fv[:] = u, v
        dst = torch.zeros((dh, dw, 2), dtype=torch.uint8, device="cuda:0")
        engine.process_device(_dev(frame), scale, dst, order=order)
        engine.sync()
        _, gu, gv = S.yuv422_planes(dst.cpu().numpy(), order)
        for k, (g, w) in enumerate(zip((gu, gv), want)):
            assert np.array_equal(g, w), (order, k, int((g != w).sum()), np.argwhere(g != w)[:6].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("name,r0,r1", [("x2_int", 1, 2), ("x2_int", 17, 99), ("x4_int", 3, 157), ("x2_tail4", 33, 140),
                                        ("x1.5_tail7", 31, 97), ("x2.7_tail3", 63, 130)])
def test_alpha_of_bands_starting_on_odd_rows(engine, name, r0, r1):
    """a band call's tile grid starts at its first row: the alpha rows of a band are the whole resize's rows [r0, r1)"""
    import srcnn_cpp_b200 as S
    import torch
    sw, sh, scale, _ = MOSAICS[name]
    dw, dh = dims(name)
    src = np.concatenate([colour(name), grey(name)[:, :, None]], -1)
    s0, s1 = S.band_src_rows(sh, scale, r0, r1)
    band = torch.zeros((r1 - r0, dw, 4), dtype=torch.uint8, device="cuda:0")
    engine.process_band_device(_dev(src[s0:s1]), sw, sh, s0, s1, scale, r0, r1, band, order=S.ORDER_BGRA)
    engine.sync()
    want = want_planes(grey(name), name)[0][r0:r1]
    got = band[:, :, 3].cpu().numpy()
    assert np.array_equal(got, want), (int((got != want).sum()), np.argwhere(got != want)[:6].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["x2_int", "x4_int", "x1.5_tail7", "x2_tail4", "x1.25_tail1"])
def test_fp16_luma_written_by_the_resize_kernels(engine, name):
    """The tensor-core path's resize kernels write Y as FP16 (y16) for the CNN themselves.  The staged path builds y16 from
    the u8 plane with k_y8_to_y16 instead, and that u8 plane is pinned to the oracle above.  The CNN is deterministic given
    its input (test_cnn_tc_repeatable, work-cut independence), so process_device == stage_color_bicubic -> stage_cnn(TC) ->
    stage_merge, bit for bit, holds exactly when the in-kernel FP16 write equals the u8 plane on every pixel of the tie plane."""
    import srcnn_cpp_b200 as S
    import torch
    sw, sh, scale, _ = MOSAICS[name]
    dw, dh = dims(name)
    src = _dev(colour(name))
    y, cr, cb = _planes(3, dh, dw)
    ycnn = _planes(1, dh, dw)[0]
    engine.stage_color_bicubic(src, scale, y, cr, cb)
    engine.stage_cnn(y, ycnn, variant=S.VARIANT_TC)
    staged = torch.zeros((dh, dw, 3), dtype=torch.uint8, device="cuda:0")
    engine.stage_merge(ycnn, cr, cb, staged)
    whole = torch.zeros((dh, dw, 3), dtype=torch.uint8, device="cuda:0")
    engine.process_device(src, scale, whole)
    engine.sync()
    a, b = whole.cpu().numpy(), staged.cpu().numpy()
    d = (a != b).any(-1)
    assert not d.any(), explain(d.astype(np.uint8), np.zeros_like(d, np.uint8), name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["x2_int", "x1.5_tail7", "x2_tail4"])
def test_fp32_variant_whole_path_equals_oracle(name):
    """the strict FP32 variant's whole path == oracle.pipeline on colour tie planes"""
    import srcnn_cpp_b200 as S
    import torch
    eng = _engine_with({})
    try:
        eng.set_variant(S.VARIANT_FP32)
        sw, sh, scale, _ = MOSAICS[name]
        dw, dh = dims(name)
        dst = torch.zeros((dh, dw, 3), dtype=torch.uint8, device="cuda:0")
        eng.process_device(_dev(colour(name)), scale, dst)
        eng.sync()
    finally:
        eng.close()
    got, want = dst.cpu().numpy(), ties.oracle().pipeline(colour(name), scale)
    assert np.array_equal(got, want), (int((got != want).any(-1).sum()), np.argwhere((got != want).any(-1))[:6].tolist())


@pytest.mark.gpu
def test_merge_exhaustive(engine):
    """K-C on all 2^24 (Y, Cr, Cb) triples == cv2.cvtColor(YCrCb2BGR), BGR and RGB order"""
    import cv2
    import srcnn_cpp_b200 as S
    import torch
    cv2.ipp.setUseIPP(False)
    ycc = all_bgr()
    want = cv2.cvtColor(ycc, cv2.COLOR_YCrCb2BGR)
    pl = _planes(3, 4096, 4096)
    for k in range(3):
        pl[k].copy_(_dev(ycc[:, :, k]))
    for order, w in ((S.ORDER_BGR, want), (S.ORDER_RGB, want[:, :, ::-1])):
        dst = torch.zeros((4096, 4096, 3), dtype=torch.uint8, device="cuda:0")
        engine.stage_merge(*pl, dst, order=order)
        engine.sync()
        got = dst.cpu().numpy()
        assert np.array_equal(got, w), (order, int((got != w).any(-1).sum()))


@pytest.mark.gpu
def test_colour_conversion_exhaustive_at_scale_one(engine):
    """colour + bicubic at scale 1.0 (taps {0, 2048, 0, 0}: a pure colour conversion) on all 2^24 BGR values ==
    cv2.cvtColor(BGR2YCrCb)"""
    import cv2
    cv2.ipp.setUseIPP(False)
    img = all_bgr()
    want = cv2.cvtColor(img, cv2.COLOR_BGR2YCrCb)
    pl = _planes(3, 4096, 4096)
    engine.stage_color_bicubic(_dev(img), 1.0, *pl)
    engine.sync()
    for k in range(3):
        got = pl[k].cpu().numpy()
        assert np.array_equal(got, want[:, :, k]), (k, int((got != want[:, :, k]).sum()))
