"""The strict FP32 CNN (srcnn_fp32.cu) on witness planes: bit for bit against the oracle where its arithmetic shows.

k_conv55_strict's result is only visible after the (int) truncation, and a near miss of its arithmetic moves the float value
by about 1e-5: on natural content that changes a few bytes per million, and the pixels within 1e-3 of an integer are exactly the
ones a q(v) check has to leave out.  oracle/cnn_witness.py edits one or two bytes of each witness centre's 13x13 field so that
the centre's float value lands on an integer, keeping the edit under which the most near misses (orc_cnn_at modes 1-12) change
the byte.  The tests below check that the witness set does tell each near miss from the reference, and then run the kernels on
it: the stage, conv2's activations, chunk seams of a 65536-wide plane, and the whole grey path at x1 (the cubic resize is then
the identity) through single frames, bands, batches, host sub-bands and a BGR call.  A failure names each differing pixel's
near-miss class (the modes whose byte the kernel reproduced) and where it lies.
"""
import numpy as np
import pytest

from oracle import cnn_witness as cw

DENSITY_MIN = 200   # bytes each of M1-M5 must change over the witness set

# (background, H, W, seed): widths not a multiple of 32 and heights not a multiple of 8 (the kernels' 32x8 CTA tiles)
PLANES = [("natural", 261, 397, 1), ("noise", 203, 331, 2), ("noise", 261, 397, 3), ("noise", 261, 397, 4)]


@pytest.fixture(scope="module")
def witnesses(oracle):
    return [cw.build(cw.background(k, h, w, s), cw.place(h, w), oracle, screen=96, keep=6) for k, h, w, s in PLANES]


def _names(modes):
    return ", ".join(cw.NEAR_MISSES[m] for m in modes) or "no near miss"


def _where(r, c, h, w, seams=(), band_edges=()):
    out = []
    if min(r, c, h - 1 - r, w - 1 - c) < 6:
        out.append("border")
    if any(abs(r - s) <= 2 or abs(r - (s - 1)) <= 2 for s in seams):
        out.append("chunk seam")
    if any(r in (e - 1, e) for e in band_edges):
        out.append("band edge")
    return "/".join(out) or "interior"


def _check_witnesses(label, wit, got, **where):
    """got: the kernel's u8 plane (numpy); every centre of `wit` must carry the exact byte"""
    g = got[wit.rows, wit.cols]
    bad = np.flatnonzero(g != wit.bytes[0])
    h, w = wit.plane.shape
    msg = ["(%d,%d) %s: got %d, want %d (v=%.7f); matches %s" % (
        wit.rows[i], wit.cols[i], _where(wit.rows[i], wit.cols[i], h, w, **where), g[i], wit.bytes[0, i], wit.values[0, i],
        _names([m for m in cw.NEAR_MISSES if wit.bytes[m, i] == g[i]])) for i in bad[:20]]
    assert not len(bad), "%s: %d of %d witness pixels differ\n%s" % (label, len(bad), len(g), "\n".join(msg))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the oracle's listed-pixel CNN and the witness set
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h,w", [(40, 52), (9, 13), (1, 1), (3, 70), (64, 5), (17, 1)])
def test_cnn_at_exact_mode_is_orc_cnn(oracle, h, w):
    y = np.random.default_rng(h * 1000 + w).integers(0, 256, (h, w), dtype=np.uint8)
    r, c = np.indices((h, w))
    _, b = oracle.cnn_at(y, r, c)
    assert np.array_equal(b.reshape(h, w), oracle.cnn(y))
    assert np.array_equal(oracle.act2_at(y, r, c).reshape(h, w, 32).transpose(2, 0, 1), oracle.conv99x11(y))


def test_cnn_at_exact_mode_on_witness_planes(oracle, witnesses):
    """mode 0 == orc_cnn at every centre and on a band of rows through each plane (top and bottom rows included)"""
    for wit in witnesses:
        full = oracle.cnn(wit.plane)
        assert np.array_equal(full[wit.rows, wit.cols], wit.bytes[0])
        h, w = wit.plane.shape
        r, c = np.indices((h, w))
        sel = (r < 3) | (r >= h - 3) | (np.abs(r - h // 2) < 2)
        _, b = oracle.cnn_at(wit.plane, r[sel], c[sel])
        assert np.array_equal(b, full[sel])


def test_cnn_at_refuses_bad_arguments(oracle):
    y = np.zeros((4, 5), np.uint8)
    L, P = oracle.lib, oracle.params
    rows, cols = np.array([0, 4], np.int32), np.array([0, 0], np.int32)
    v, b = np.empty(2, np.float32), np.empty(2, np.uint8)
    assert L.orc_cnn_at(P.ctypes.data, y.ctypes.data, 5, 4, rows.ctypes.data, cols.ctypes.data, 2, 0, v.ctypes.data, b.ctypes.data) == -1
    assert L.orc_cnn_at(P.ctypes.data, y.ctypes.data, 5, 4, rows.ctypes.data, cols.ctypes.data, 1, 13, v.ctypes.data, b.ctypes.data) == -1
    assert L.orc_at_modes() == cw.MODES


def test_builder_is_deterministic(oracle):
    bg = cw.background("natural", 40, 52, 9)
    a = cw.build(bg, cw.place(40, 52), oracle, screen=24, keep=2)
    b = cw.build(bg.copy(), cw.place(40, 52), oracle, screen=24, keep=2)
    assert np.array_equal(a.plane, b.plane) and np.array_equal(a.bytes, b.bytes) and np.array_equal(a.values, b.values)
    assert not np.array_equal(a.plane, bg)                               # it did edit
    assert np.array_equal(cw.background("natural", 40, 52, 9), bg)


def test_placement_covers_the_clamped_rows_and_corners():
    for h, w in ((261, 397), (203, 331), (14, 14)):
        cs = cw.place(h, w)
        r = np.array([p[0] for p in cs])
        c = np.array([p[1] for p in cs])
        d = np.maximum(np.abs(r[:, None] - r[None]), np.abs(c[:, None] - c[None]))
        assert (d[~np.eye(len(cs), dtype=bool)] >= cw.FIELD).all()
        for corner in ((0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1)):
            assert corner in cs or h < 2 * cw.FIELD
        if h > 100:
            for k in (0, 1, h - 2, h - 1):
                assert (r == k).sum() >= 2
            for k in (0, 1, w - 2, w - 1):
                assert (c == k).sum() >= 2


def test_float64_value_is_the_oracle_value(oracle):
    """the float64 value the builder ranks edits with is the oracle's float value to within float32 rounding"""
    y = cw.background("natural", 60, 70, 5)
    cs = cw.place(60, 70)
    r = np.array([p[0] for p in cs], np.int32)
    c = np.array([p[1] for p in cs], np.int32)
    v, _ = cw.value_and_gradient(y, r, c)
    v32, _ = oracle.cnn_at(y, r, c)
    assert np.abs(v - v32).max() < 1e-3


def test_near_misses_change_bytes_on_the_witness_set(oracle, witnesses):
    """Each conv3 near miss M1-M5 changes at least DENSITY_MIN witness bytes; each conv1 / conv2 near miss changes bytes and
    conv2's activations at the centres (a bit-exact act2 comparison fails on every one of them)."""
    n = sum(len(w.rows) for w in witnesses)
    counts = {m: int(sum(w.changed(m).sum() for w in witnesses)) for m in cw.NEAR_MISSES}
    print("WITNESS centres %d, bytes changed %s" % (n, {cw.NEAR_MISSES[m]: k for m, k in counts.items()}))
    for m in cw.CONV3_NEAR_MISSES:
        assert counts[m] >= DENSITY_MIN, (cw.NEAR_MISSES[m], counts[m])
    for m in cw.CONV12_NEAR_MISSES:
        assert counts[m] >= DENSITY_MIN, (cw.NEAR_MISSES[m], counts[m])
        changed = ulps = 0
        for w in witnesses:
            a0 = oracle.act2_at(w.plane, w.rows, w.cols).view(np.int32)
            am = oracle.act2_at(w.plane, w.rows, w.cols, m).view(np.int32)
            changed += int((a0 != am).sum())
            ulps = max(ulps, int(np.abs(a0.astype(np.int64) - am).max()))
        print("WITNESS act2 %s: %d of %d values changed, up to %d ulp" % (cw.NEAR_MISSES[m], changed, 32 * n, ulps))
        assert changed >= n


def test_equivalent_near_misses_change_nothing(witnesses):
    """Two rewrites of conv3 are not near misses: they leave every float value as it is, so no test can or need tell them
    apart.  b3 added in double: temp and b3 are floats, their sum is exact in double (the exponents differ by far less than
    29), and rounding it to float is the float addition.  (n,m) tap order: the 25 products are floats, and a double holds
    their sum exactly whenever the exponent spread of the partial sums stays below 53 - 24 - 5 bits, so the order of the
    inner sum cannot change it.  Neither is counted as covered."""
    for w in witnesses:
        for m in cw.EQUIVALENT_NEAR_MISSES:
            assert np.array_equal(w.values[m], w.values[0]), cw.NEAR_MISSES[m]
            assert not w.changed(m).any()


def test_golden_anchor(oracle, golden):
    """The butterfly's upscaled Y (digest pinned in test_oracle) -> the reference's own CNN output butterfly-srcnn-y.png.
    orc_cnn is that plane; M2-M5 each change it.  A near miss moves the float value by less than 1e-3 - 2e-4, so only pixels
    whose float64 value lies within INT_BAND = 1e-3 of an integer can change; those are evaluated under every near miss.
    M1 (temp kept in double) changes none of the golden bytes: the per-channel float rounding of `temp += temppixel`
    (src/srcnn.cpp:232) is pinned by the C source's semantics and by the witness planes above, not by the golden plane."""
    import hashlib
    import os

    from test_cnn_precision import INT_BAND, cnn_v64
    src, _ = golden
    _, st = oracle.pipeline(src, 1.5, stages=True)
    y = st["up_y"]
    assert hashlib.sha256(y.tobytes()).hexdigest() == "e4862936d82de0eba7d5f49f85e6e478bdeb6cd71fc074494788b660ba463be9"
    import cv2
    want = cv2.imread(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "butterfly-srcnn-y.png"),
                      cv2.IMREAD_UNCHANGED)
    assert np.array_equal(oracle.cnn(y), want)
    v = cnn_v64(y).numpy()
    r, c = np.nonzero(np.abs(v - np.round(v)) < INT_BAND)
    _, b0 = oracle.cnn_at(y, r, c)
    assert np.array_equal(b0, want[r, c])
    diff = {m: int((oracle.cnn_at(y, r, c, m)[1] != want[r, c]).sum()) for m in cw.CONV3_NEAR_MISSES}
    print("GOLDEN %d pixels within INT_BAND; bytes changed %s" % (len(r), {cw.NEAR_MISSES[m]: k for m, k in diff.items()}))
    for m in (2, 3, 4, 5):
        assert diff[m] >= 1, cw.NEAR_MISSES[m]
    assert diff[1] == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the kernels on witness planes, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
def _padded(a, pad=45, dtype=None):
    """a device tensor holding numpy array `a` whose rows are `pad` elements longer than its width"""
    import torch
    h, w = a.shape[:2]
    t = torch.zeros((h, w + pad) + a.shape[2:], dtype=dtype or torch.uint8, device="cuda:0")
    v = t[:, :w]
    if a.size:
        v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
    return v


def _fp32(engine):
    import srcnn_cpp_b200 as S
    engine.set_variant(S.VARIANT_FP32)


def _restore(engine):
    import srcnn_cpp_b200 as S
    engine.set_variant(S.VARIANT_TC)


@pytest.mark.gpu
def test_stage_cnn_fp32_on_witness_planes(engine, oracle, witnesses):
    import srcnn_cpp_b200 as S
    for k, wit in enumerate(witnesses):
        h, w = wit.plane.shape
        out = _padded(np.zeros((h, w), np.uint8), pad=77)
        engine.stage_cnn(_padded(wit.plane), out, variant=S.VARIANT_FP32)
        engine.sync()
        got = out.cpu().numpy()
        _check_witnesses("stage %s" % (PLANES[k],), wit, got)
        assert np.array_equal(got, oracle.cnn(wit.plane)), PLANES[k]


@pytest.mark.gpu
def test_stage_conv99x11_fp32_on_witness_planes(engine, oracle, witnesses):
    """conv2's 32 float planes bit for bit: every conv1 / conv2 near miss changes them (test above)"""
    import torch
    for k, wit in enumerate(witnesses):
        h, w = wit.plane.shape
        act2 = torch.full((32, h, w), float("nan"), dtype=torch.float32, device="cuda:0")
        engine.stage_conv99x11_fp32(_padded(wit.plane), act2)
        engine.sync()
        got = act2.cpu().numpy().view(np.int32)
        want = oracle.conv99x11(wit.plane).view(np.int32)
        bad = np.argwhere(got != want)
        assert not len(bad), (PLANES[k], len(bad), int(np.abs(got.astype(np.int64) - want).max()),
                              [tuple(p) for p in bad[:10].tolist()])


SEAM_ROWS = (58, 59, 60, 61, 62, 118, 119, 120, 121, 122)


@pytest.mark.gpu
def test_fp32_chunk_seams_on_witnesses(engine, oracle):
    """65536 columns: launch_cnn_fp32 works in 60-row chunks whose act2 halo starts at cb - 2, so seams at rows 60 and 120;
    witnesses on rows 58-62 and 118-122, in three column windows (left edge, middle, right edge)"""
    import srcnn_cpp_b200 as S
    h, w = 130, 65536
    bg = cw.background("natural", h, w, 73)
    windows = [(0, 1040), (w // 2 - 520, w // 2 + 520), (w - 1040, w)]
    cs = [(r, c) for r, c in cw.place(h, w, priority_rows=SEAM_ROWS, grid=False)
          if r in SEAM_ROWS and any(a <= c < b for a, b in windows)]
    wit = cw.build(bg, cs, oracle, screen=48, keep=3)
    out = _padded(np.zeros((h, w), np.uint8), pad=128)
    engine.stage_cnn(_padded(wit.plane, pad=128), out, variant=S.VARIANT_FP32)
    engine.sync()
    _check_witnesses("chunk seams", wit, out.cpu().numpy(), seams=(60, 120))


@pytest.mark.gpu
def test_resize_plane_x1_is_the_identity(engine, oracle):
    """at x1 every cubic phase is 0 and its taps are (0, 2048, 0, 0): the whole path's Y is its source"""
    src = cw.background("noise", 203, 331, 5)
    y = _padded(np.zeros_like(src))
    engine.stage_resize_plane(_padded(src), 1.0, y)
    engine.sync()
    assert np.array_equal(y.cpu().numpy(), src)
    ofs, coef = oracle.cubic_taps(331, 331)
    assert np.array_equal(ofs, np.arange(331)) and (coef == np.array([0, 2048, 0, 0], np.int16)).all()


@pytest.mark.gpu
def test_fp32_grey_path_x1_single_frame(engine, oracle, witnesses):
    import srcnn_cpp_b200 as S
    wit = witnesses[0]
    h, w = wit.plane.shape
    out = _padded(np.zeros((h, w), np.uint8), pad=3)
    try:
        _fp32(engine)
        engine.process_device(_padded(wit.plane, pad=9), 1.0, out, order=S.ORDER_GRAY)
        engine.sync()
    finally:
        _restore(engine)
    got = out.cpu().numpy()
    _check_witnesses("process_device", wit, got)
    assert np.array_equal(got, oracle.cnn(wit.plane))


BAND_EDGES = (67, 140)


@pytest.mark.gpu
def test_fp32_grey_path_x1_bands(engine, oracle):
    """process_band_device over three bands whose first and last rows, and the rows just outside them, carry witnesses:
    k_conv99x11_strict reads the band's plane through its gr - yrow0 clamp, k_conv55_strict writes through out_row0"""
    import srcnn_cpp_b200 as S
    h, w = 211, 397
    rows = sorted({e + d for e in BAND_EDGES for d in (-2, -1, 0, 1)})
    wit = cw.build(cw.background("natural", h, w, 21), cw.place(h, w, priority_rows=rows), oracle, screen=48, keep=3)
    src = _padded(wit.plane, pad=11)
    out = np.zeros((h, w), np.uint8)
    edges = (0,) + BAND_EDGES + (h,)
    try:
        _fp32(engine)
        for r0, r1 in zip(edges[:-1], edges[1:]):
            s0, s1 = S.band_src_rows(h, 1.0, r0, r1)
            dst = _padded(np.zeros((r1 - r0, w), np.uint8), pad=5)
            engine.process_band_device(src[s0:s1], w, h, s0, s1, 1.0, r0, r1, dst, order=S.ORDER_GRAY)
            engine.sync()
            out[r0:r1] = dst.cpu().numpy()
    finally:
        _restore(engine)
    _check_witnesses("bands", wit, out, band_edges=BAND_EDGES)
    assert np.array_equal(out, oracle.cnn(wit.plane))


@pytest.mark.gpu
def test_fp32_grey_path_x1_batch(engine, oracle):
    """three frames of different witness planes in one process_batch_device call (FP32 batches run frame by frame)"""
    import torch
    import srcnn_cpp_b200 as S
    h, w = 75, 133
    wits = [cw.build(cw.background(k, h, w, 30 + i), cw.place(h, w), oracle, screen=48, keep=3)
            for i, k in enumerate(("natural", "noise", "natural"))]
    src = torch.from_numpy(np.stack([x.plane for x in wits])).to("cuda:0")
    out = torch.zeros((3, h, w), dtype=torch.uint8, device="cuda:0")
    try:
        _fp32(engine)
        engine.process_batch_device(src, 1.0, out, order=S.ORDER_GRAY)
        engine.sync()
    finally:
        _restore(engine)
    got = out.cpu().numpy()
    for i, x in enumerate(wits):
        _check_witnesses("batch frame %d" % i, x, got[i])
        assert np.array_equal(got[i], oracle.cnn(x.plane)), i


HOST_EDGES = (256, 588)   # a 1024-row frame's sub-bands with 8 host bands, growth 1.3: 256, 332, 436 rows


@pytest.mark.gpu
def test_fp32_grey_path_x1_host_sub_bands(engine, oracle):
    """process_host cuts a frame of >= 1024 rows into sub-bands, each its own copy-in, CNN and copy-out"""
    import srcnn_cpp_b200 as S
    h, w = 1024, 523
    rows = sorted({e + d for e in HOST_EDGES for d in (-2, -1, 0, 1)})
    wit = cw.build(cw.background("natural", h, w, 41), cw.place(h, w, priority_rows=rows, grid=False), oracle,
                   screen=48, keep=3)
    try:
        _fp32(engine)
        got = engine.process(wit.plane, 1.0, order=S.ORDER_GRAY)
    finally:
        _restore(engine)
    _check_witnesses("host sub-bands", wit, got, band_edges=HOST_EDGES)
    assert np.array_equal(got, oracle.cnn(wit.plane))


@pytest.mark.gpu
def test_fp32_bgr_x1_of_a_grey_plane(engine, oracle, witnesses):
    """B = G = R = plane: the 14-bit Y coefficients sum to 16384, so Y is the plane, Cr = Cb = 128, and every output channel
    is the CNN's byte"""
    import srcnn_cpp_b200 as S
    wit = witnesses[0]
    bgr = np.repeat(wit.plane[:, :, None], 3, axis=2)
    assert np.array_equal(oracle.bgr2ycrcb(bgr)[:, :, 0], wit.plane)
    h, w = wit.plane.shape
    out = _padded(np.zeros((h, w, 3), np.uint8), pad=7)
    try:
        _fp32(engine)
        engine.process_device(_padded(bgr, pad=13), 1.0, out, order=S.ORDER_BGR)
        engine.sync()
    finally:
        _restore(engine)
    got = out.cpu().numpy()
    for ch in range(3):
        _check_witnesses("BGR channel %d" % ch, wit, np.ascontiguousarray(got[:, :, ch]))
    assert np.array_equal(got, oracle.pipeline(bgr, 1.0))
