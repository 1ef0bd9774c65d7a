"""The frawscale-compatible stage's bit-identity claim, held by a float64 restatement and by planes that witness it.

oracle/fraw.py restates FrawTable and the two passes of srcnn_fraw_scale_device in numpy float64, operation for operation,
and emulates the near misses a kernel or table builder could quietly drift into (FMA, another summation order, a float
accumulator, reciprocal normalisation, another centre formula, Box's edge, the pass order, a tap too few).  On noise the
near misses that only move a double's last bit almost never show through the float result; the witness planes plant
cancelling pairs of large values so that they do.  The CPU tests pin the restatement to the golden vectors (and to the
compiled reference where it is present), the library's table builder to the restatement on every size pair up to 160 and
on extreme tables, and prove the planes' power.  The GPU tests run every pass order, size edge, special value, the table
cache and the shared scratch buffer bit for bit against the restatement."""
import ctypes as C
import functools
import os
from fractions import Fraction

import numpy as np
import pytest

from oracle import fraw as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILTERS = (F.BOX, F.BILINEAR, F.BICUBIC)

# one-axis (src, dst) witness sizes: ratios that put filter edges on sample centres (2/3, 1/3, 3/7, 5/3, x2, x4, x0.5,
# x0.1) and one that does not (x0.75)
AXIS_SIZES = [(40, 30), (24, 48), (90, 60), (30, 10), (70, 30), (30, 50), (12, 48), (64, 32), (200, 20)]
LINES = 256

# near misses a geometry cannot show away from its borders: table near misses whose table equals the stage's (checked,
# not assumed, in test_witness_planes_catch_every_near_miss), and arithmetic ones where every interior weight is a short
# dyadic fraction, so that products are exact and sums of two are order-free (Box and Bilinear up by 2 and 4, Box down by
# 2, 2/3 and 3/4, Bilinear down by 2 and up by 5/3)
_EXACT = ("fma", "reverse", "pairwise", "f32acc")
ARITH_EXEMPT = {
    (F.BOX, 40, 30): _EXACT, (F.BOX, 24, 48): _EXACT, (F.BOX, 90, 60): _EXACT, (F.BOX, 30, 50): _EXACT,
    (F.BOX, 12, 48): _EXACT, (F.BOX, 64, 32): _EXACT,
    (F.BILINEAR, 24, 48): ("fma", "reverse", "pairwise"), (F.BILINEAR, 12, 48): ("fma", "reverse", "pairwise"),
    (F.BILINEAR, 64, 32): ("fma",), (F.BILINEAR, 30, 50): ("reverse", "pairwise"),
}
# near misses of the last bits of a product or a weight: they must change many times more samples than on noise
LAST_BIT = ("fma", "reverse", "pairwise", "recip")


def _golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "fraw_golden.npz"))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@functools.lru_cache(maxsize=None)
def witness(kind, s, d, axis):
    """axis 'v': a plane of LINES columns resized from s to d rows (k_fraw_vertical alone); 'h': LINES rows, s to d columns"""
    return F.witness_plane(LINES, s, LINES, d, kind, seed=7 * s + d) if axis == "v" else \
        F.witness_plane(s, LINES, d, LINES, kind, seed=7 * s + d + 1)


def _noise(shape, seed=9):
    return (np.random.default_rng(seed).random(shape, dtype=np.float32) * 255).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the restatement, the library's table builder, the planes' power
# ---------------------------------------------------------------------------------------------------------------------
def test_restatement_equals_golden_vectors():
    g = _golden()
    k = 0
    while "cfg%d" % k in g:
        sw, sh, dw, dh, flt = g["cfg%d" % k].tolist()
        got = F.scale(g["src%d" % k], dw, dh, flt)
        assert np.array_equal(_bits(got), g["dst%d" % k].view(np.uint32)), (k, sw, sh, dw, dh, flt)
        k += 1
    assert k >= 10


@pytest.mark.parametrize("kind", FILTERS)
def test_restatement_equals_compiled_reference(kind):
    from oracle.oracle import FrawRef
    if not FrawRef.available():
        pytest.skip("oracle/_ref/libfraw.so not built and /root/reference absent")
    for sw, sh, dw, dh in [(40, 30, 40, 20), (30, 40, 75, 40), (90, 60, 60, 90), (64, 48, 256, 192), (200, 100, 20, 10)]:
        src = witness(kind, sh, dh, "v")[:, :sw] if sw == dw else _noise((sh, sw), sw + dh)
        assert np.array_equal(_bits(F.scale(src, dw, dh, kind)), _bits(FrawRef().scale(src, dw, dh, kind)))


def test_fma_emulation_is_exact():
    """oracle.fraw.fma == round(w * x + acc) computed in rationals, on cancelling and on plain operands"""
    rng = np.random.default_rng(5)
    n = 4000
    w = rng.uniform(-1.5, 1.5, n)
    x = (rng.uniform(-1, 1, n) * np.exp2(rng.integers(-20, 31, n))).astype(np.float32).astype(np.float64)
    acc = np.where(rng.random(n) < 0.6, -(w * x) * (1 + rng.uniform(-1e-9, 1e-9, n)), rng.uniform(-300, 300, n))
    got = F.fma(w, x, acc)
    want = np.array([float(Fraction(a) * Fraction(b) + Fraction(c)) for a, b, c in zip(w, x, acc)])
    assert np.array_equal(got.view(np.int64), want.view(np.int64))
    assert (got != w * x + acc).sum() > 100      # the operands do tell FMA from a multiply and an add


def _lib_table(kind, dst, src):
    import srcnn_cpp_b200 as S
    f = S.load_library().srcnn_debug_fraw_table
    f.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    f.restype = C.c_int
    window = np.zeros(1, np.int32)
    assert f(kind, dst, src, None, None, None, window.ctypes.data) == 0
    left, count = np.empty(dst, np.int32), np.empty(dst, np.int32)
    w = np.empty((dst, int(window[0]) + 1), np.float64)
    assert f(kind, dst, src, left.ctypes.data, count.ctypes.data, w.ctypes.data, window.ctypes.data) == 0
    return int(window[0]), left, count, w


def _assert_tables_equal(kind, dst, src):
    window, left, count, w = _lib_table(kind, dst, src)
    t = F.Table(kind, dst, src)
    assert window == t.window, (kind, dst, src)
    assert np.array_equal(left, t.left) and np.array_equal(count, t.count), (kind, dst, src)
    assert np.array_equal(w.view(np.int64), t.w.view(np.int64)), (kind, dst, src)


@pytest.mark.parametrize("kind", FILTERS)
def test_table_builder_equals_restatement_on_every_small_size(kind):
    """FrawTable (through srcnn_debug_fraw_table) == the restatement, every (src, dst) in 1..160 x 1..160: window, left,
    count and every weight bit, the zeros past each sample's count included"""
    for src in range(1, 161):
        for dst in range(1, 161):
            _assert_tables_equal(kind, dst, src)


@pytest.mark.parametrize("kind", FILTERS)
@pytest.mark.parametrize("src,dst", [(65535, 1), (1, 65535), (65535, 65534), (3, 65535), (4096, 3)])
def test_table_builder_equals_restatement_on_extreme_tables(kind, src, dst):
    _assert_tables_equal(kind, dst, src)
    if (kind, src, dst) == (F.BICUBIC, 4096, 3):
        assert F.Table(kind, dst, src).window == 5463


def test_table_export_refuses_bad_arguments():
    import srcnn_cpp_b200 as S
    f = S.load_library().srcnn_debug_fraw_table
    f.argtypes = [C.c_int, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    f.restype = C.c_int
    b = np.zeros(64, np.float64)
    p = b.ctypes.data
    assert f(3, 4, 4, p, p, p, p) < 0 and f(-1, 4, 4, p, p, p, p) < 0
    assert f(2, 0, 4, p, p, p, p) < 0 and f(2, 4, 0, p, p, p, p) < 0
    assert f(2, 4, 4, p, p, p, None) < 0 and f(2, 4, 4, p, None, p, p) < 0 and f(2, 4, 4, None, None, p, p) < 0


def test_bilinear_edge_is_an_equivalent_change():
    """v <= width instead of v < width in Bilinear adds a tap of weight width - v == +0: the same table, always"""
    for src in (3, 7, 24, 40, 90, 160):
        for dst in (1, 5, 12, 30, 48, 60, 160):
            a, b = F.Table(F.BILINEAR, dst, src), F.Table(F.BILINEAR, dst, src, {"bilinear_le"})
            assert np.array_equal(a.left, b.left) and np.array_equal(a.count, b.count)
            assert np.array_equal(a.w.view(np.int64), b.w.view(np.int64))


def _tables_differ(kind, s, d, v):
    """whether a table near miss changes the linear map (a tap of weight zero, dropped or kept, changes nothing)"""
    return not np.array_equal(F.linear_map(F.table(kind, d, s)), F.linear_map(F.table(kind, d, s, {v})))


@pytest.mark.parametrize("axis", ["v", "h"])
@pytest.mark.parametrize("s,d", AXIS_SIZES)
@pytest.mark.parametrize("kind", FILTERS)
def test_witness_planes_catch_every_near_miss(kind, s, d, axis):
    """every near miss that can change a sample of this geometry changes at least 20 of the witness plane, and the ones of
    the last bit of a product or a weight change at least 8 times as many as on noise of the same size"""
    src = witness(kind, s, d, axis)
    sh, sw = src.shape
    dw, dh = (sw, d) if axis == "v" else (d, sh)
    exempt = ARITH_EXEMPT.get((kind, s, d), ())
    wanted = [v for v in _EXACT if v not in exempt]
    wanted += [v for v in ("centre", "recip", "box_lt", "ratio_mul", "short") if _tables_differ(kind, s, d, v)]
    got = F.witness_counts(src, dw, dh, kind, wanted)
    noise = F.witness_counts(_noise(src.shape), dw, dh, kind, [v for v in wanted if v in LAST_BIT])
    low = {v: n for v, n in got.items() if n < 20 or (v in LAST_BIT and n < 8 * max(1, noise[v]))}
    assert not low, (low, got, noise)


def test_every_near_miss_has_witnesses_somewhere():
    seen = {v: 0 for v in F.VARIANTS if v not in ("bilinear_le", "h_first")}
    for kind in FILTERS:
        for s, d in AXIS_SIZES:
            src = witness(kind, s, d, "v")
            for v, n in F.witness_counts(src, src.shape[1], d, kind, list(seen)).items():
                seen[v] += n
    assert min(seen.values()) >= 100, seen


def test_pass_order_near_miss_on_two_pass_geometries():
    """horizontal first when up-scaling: the intermediate float plane differs, so random content shows it (Box up-scales
    copy samples, so only the other filters can show it)"""
    for kind in (F.BILINEAR, F.BICUBIC):
        src = _noise((40, 30), 3)
        assert F.witness_counts(src, 75, 60, kind, ["h_first"])["h_first"] >= 100, kind


def test_witness_planes_are_deterministic():
    a = F.witness_plane(64, 40, 64, 30, F.BICUBIC, seed=3)
    assert np.array_equal(_bits(a), _bits(F.witness_plane(64, 40, 64, 30, F.BICUBIC, seed=3)))
    assert not np.array_equal(_bits(a), _bits(F.witness_plane(64, 40, 64, 30, F.BICUBIC, seed=4)))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: bit for bit against the restatement
# ---------------------------------------------------------------------------------------------------------------------
def _run(engine, src, dw, dh, kind):
    import torch
    s = torch.from_numpy(np.ascontiguousarray(src, np.float32)).to("cuda:0")
    d = torch.full((dh, dw), float("nan"), dtype=torch.float32, device="cuda:0")
    engine.fraw_scale(s, d, kind)
    engine.sync()
    return d.cpu().numpy()


def _check(engine, src, dw, dh, kind, what=""):
    got, want = _run(engine, src, dw, dh, kind), F.scale(src, dw, dh, kind)
    bad = _bits(got) != _bits(want)
    assert not bad.any(), (what, kind, src.shape, (dh, dw), int(bad.sum()), np.argwhere(bad)[:5].tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("axis", ["v", "h"])
@pytest.mark.parametrize("s,d", AXIS_SIZES)
@pytest.mark.parametrize("kind", FILTERS)
def test_gpu_one_pass_on_witness_planes(engine, kind, s, d, axis):
    """sw == dw: k_fraw_vertical alone; sh == dh: k_fraw_horizontal alone.  Up and down for every filter."""
    src = witness(kind, s, d, axis)
    sh, sw = src.shape
    _check(engine, src, sw if axis == "v" else d, d if axis == "v" else sh, kind)


# (sw, sh, dw, dh): dw <= sw runs horizontal then vertical, dw > sw vertical then horizontal; mixed up / down on the axes
TWO_PASS = [(100, 80, 60, 130), (160, 90, 40, 30), (90, 60, 60, 90), (60, 80, 130, 50), (64, 48, 256, 192),
            (123, 77, 185, 115), (7, 300, 31, 11), (300, 7, 299, 30)]


@pytest.mark.gpu
@pytest.mark.parametrize("geom", TWO_PASS)
@pytest.mark.parametrize("kind", FILTERS)
def test_gpu_two_pass_geometries(engine, kind, geom):
    sw, sh, dw, dh = geom
    rng = np.random.default_rng(sw + 3 * dh + kind)
    src = (rng.standard_normal((sh, sw)) * 100).astype(np.float32)
    _check(engine, src, dw, dh, kind, "two-pass")


@pytest.mark.gpu
def test_gpu_equal_sizes_copy_the_plane(engine):
    rng = np.random.default_rng(4)
    src = rng.integers(0, 1 << 32, (37, 53), dtype=np.uint64).astype(np.uint32).view(np.float32)   # NaN payloads too
    for kind in FILTERS:
        assert np.array_equal(_bits(_run(engine, src, 53, 37, kind)), src.view(np.uint32))


# (sw, sh, dw, dh, filters)
EDGES = [(1, 1, 1, 1), (1, 1, 7, 5), (1, 40, 1, 90), (1, 90, 1, 40), (40, 1, 90, 1), (90, 1, 40, 1), (1, 1, 300, 2),
         (300, 2, 1, 1), (77, 1, 1, 1), (1, 77, 1, 1), (3, 65535, 5, 1000), (2, 1000, 3, 65535), (4, 65535, 4, 7),
         (4096, 7, 3, 7), (5, 4096, 5, 3), (4096, 5, 3, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("edge", EDGES)
def test_gpu_size_edges(engine, edge):
    sw, sh, dw, dh = edge
    src = _noise((sh, sw), sw * 31 + dh)
    for kind in FILTERS:
        _check(engine, src, dw, dh, kind, "edge")


@pytest.mark.gpu
def test_gpu_refuses_65536_rows(engine):
    import srcnn_cpp_b200 as S
    import torch
    buf = torch.zeros(64, dtype=torch.float32, device="cuda:0")
    other = torch.zeros(64, dtype=torch.float32, device="cuda:0")
    L = engine.L
    assert L.srcnn_fraw_scale_device(engine.ctx, S._dptr(buf), 1, 65536, 1, 4, S._dptr(other), 2) == S.E_ARG
    assert L.srcnn_fraw_scale_device(engine.ctx, S._dptr(buf), 1, 4, 1, 65536, S._dptr(other), 2) == S.E_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("geom,kind", [((1920, 1080, 3840, 2160), F.BICUBIC), ((3840, 2160, 15360, 8640), F.BICUBIC),
                                       ((1920, 1080, 1280, 720), F.BILINEAR)])
def test_gpu_full_planes(engine, geom, kind):
    sw, sh, dw, dh = geom
    _check(engine, _noise((sh, sw), sw), dw, dh, kind, "full plane")


def _special_plane(rng, sh, sw):
    fmax = np.finfo(np.float32).max
    vals = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-39, -3e-39, 1.17e-38, np.inf, -np.inf, fmax, -fmax, fmax * 0.9,
                     -1.5, -200.0, 3.0], np.float32)
    src = rng.choice(vals, (sh, sw)).astype(np.float32)
    mask = rng.random((sh, sw)) < 0.5
    src[mask] = _noise((sh, sw), 1)[mask] - 100      # between the specials, ordinary values (negatives too)
    nans = np.array([0x7fc00000, 0xffc00000, 0x7fc12345, 0xffd54321, 0x7f800001], np.uint32).view(np.float32)
    nan_at = rng.random((sh, sw)) < 0.01
    src[nan_at] = rng.choice(nans, int(nan_at.sum()))
    src[:12, :12] = -0.0                              # corners whose outputs are -0, +0 and subnormal
    src[-12:, -12:] = rng.choice(np.array([1e-40, -3e-41, 2e-45, 0.0], np.float32), (12, 12))
    return src


@pytest.mark.gpu
@pytest.mark.parametrize("geom", [(40, 30, 40, 45), (40, 30, 17, 30), (40, 30, 90, 20), (64, 64, 32, 32)])
def test_gpu_special_values(engine, geom):
    """+-0, subnormals, +-Inf, values near FLT_MAX (sums past it become Inf in float), negatives, NaN: equal bits where the
    result is not NaN, NaN in the same places.  Only NaN-ness is promised: which NaN's sign and payload survive a sum of
    several is up to the hardware, and the stage does not pin it."""
    sw, sh, dw, dh = geom
    rng = np.random.default_rng(sw * dh)
    src = _special_plane(rng, sh, sw)
    for kind in FILTERS:
        got, want = _run(engine, src, dw, dh, kind), F.scale(src, dw, dh, kind)
        assert np.array_equal(np.isnan(got), np.isnan(want)), kind
        ok = ~np.isnan(want)
        assert np.array_equal(_bits(got)[ok], _bits(want)[ok]), (kind, int((_bits(got)[ok] != _bits(want)[ok]).sum()))
        tiny = (np.abs(want[ok]) < np.finfo(np.float32).tiny) & (want[ok] != 0)
        assert np.isinf(want).any() and (want[ok] == 0).any() and tiny.any(), kind     # Inf, zero and subnormal results


@pytest.mark.gpu
def test_gpu_table_cache_eviction_and_sharing(engine):
    """more than 8 distinct (filter, dst, src) keys, then the first again (evicted and rebuilt); the same sizes with each
    filter (three keys); a square resize (one key for both axes); every result bit for bit"""
    src = witness(F.BICUBIC, 40, 30, "v")
    for i, dh in enumerate([30, 31, 33, 35, 37, 39, 41, 43, 45, 47, 49, 30]):
        _check(engine, src, LINES, dh, F.BICUBIC, "cache %d" % i)
    for kind in FILTERS + FILTERS:
        _check(engine, _noise((60, 90), kind), 60, 40, kind, "filters")
    sq = _noise((50, 50), 5)
    for kind in FILTERS:
        _check(engine, sq, 80, 80, kind, "square")
        _check(engine, sq, 30, 30, kind, "square")


@pytest.mark.gpu
def test_gpu_scratch_shared_with_whole_path(engine):
    """the intermediate plane lives in act2_buf, which the FP32 variant's whole path uses as well: a small fraw call, a
    larger one (the buffer grows), and fraw calls interleaved with whole-path calls, every result bit for bit"""
    import srcnn_cpp_b200 as S
    import torch
    small, large = _noise((20, 30), 1), _noise((300, 400), 2)
    _check(engine, small, 50, 45, F.BICUBIC, "small")
    _check(engine, large, 700, 600, F.BICUBIC, "large")
    img = np.random.default_rng(3).integers(0, 256, (90, 120, 3), dtype=np.uint8)
    dimg = torch.from_numpy(img).to("cuda:0")
    engine.set_variant(S.VARIANT_FP32)
    try:
        out = torch.zeros((180, 240, 3), dtype=torch.uint8, device="cuda:0")
        engine.process_device(dimg, 2.0, out)
        engine.sync()
        want_path = out.cpu().numpy()
        for i in range(3):
            _check(engine, large if i % 2 else small, 700 if i % 2 else 50, 600 if i % 2 else 45, F.BICUBIC, "interleaved")
            out.zero_()
            engine.process_device(dimg, 2.0, out)
            engine.sync()
            assert np.array_equal(out.cpu().numpy(), want_path), i
    finally:
        engine.set_variant(S.VARIANT_TC)


@pytest.mark.gpu
def test_gpu_no_pass_synchronises(engine):
    """with its tables cached, a two-pass call returns while earlier work on the context's stream is still running"""
    import torch
    src = torch.from_numpy(_noise((200, 300), 6)).to("cuda:0")
    dst = torch.zeros((500, 700), dtype=torch.float32, device="cuda:0")
    engine.fraw_scale(src, dst, F.BICUBIC)
    engine.sync()
    want = _bits(dst.cpu().numpy())
    stream = torch.cuda.current_stream()
    torch.cuda._sleep(2_000_000_000)                      # about a second of one thread spinning on the same stream
    pending = torch.cuda.Event()
    pending.record(stream)
    engine.fraw_scale(src, dst, F.BICUBIC)
    still_pending = not pending.query()
    stream.synchronize()
    assert still_pending, "fraw_scale waited for the stream"
    assert np.array_equal(_bits(dst.cpu().numpy()), want)


@pytest.mark.gpu
def test_gpu_refuses_overlapping_planes(engine):
    """a one-pass resize would read samples other threads are writing: overlapping source and destination are refused"""
    import srcnn_cpp_b200 as S
    import torch
    buf = torch.from_numpy(_noise((200, 64), 8)).to("cuda:0")
    L = engine.L
    p = lambda t: S._dptr(t)
    assert L.srcnn_fraw_scale_device(engine.ctx, p(buf), 64, 100, 64, 90, p(buf[50:]), 2) == S.E_ARG     # vertical only
    assert L.srcnn_fraw_scale_device(engine.ctx, p(buf[10:]), 64, 20, 60, 20, p(buf), 2) == S.E_ARG      # horizontal only
    assert L.srcnn_fraw_scale_device(engine.ctx, p(buf), 64, 40, 64, 40, p(buf), 2) == S.E_ARG           # copy
    assert L.srcnn_fraw_scale_device(engine.ctx, p(buf), 64, 100, 32, 50, p(buf[100:]), 2) == S.OK      # adjacent
    engine.sync()
    want = F.scale(_noise((200, 64), 8)[:100], 32, 50, F.BICUBIC)
    assert np.array_equal(_bits(buf[100:150, :].cpu().numpy().reshape(-1)[:32 * 50].reshape(50, 32)), _bits(want))
