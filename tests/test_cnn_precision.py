"""Per-pixel precision of the CNN kernels against a float64 reference, on whole frames.

The tensor-core kernel (k_srcnn_tc2, srcnn_tc2.cu) multiplies FP16 operands: FP16 weights, FP16 activations after each
ReLU, conv1 / conv2 biases as FP16 hi + lo, accumulators in FP32, b3 added in FP32.  The north_star tolerance the other
tests apply (<= 1 LSB on >= 99.9 % of pixels, max 2) is far looser than what that arithmetic does, and counts how many
pixels are off, not which.  A wrong strip seam lane, ring rotation or segment edge can hide inside it.  So here the kernel
is compared with `cnn_v64(..., emulate=True)`: the same network in float64 with exactly the kernel's FP16 roundings, its
weights decoded from the packed operand image the kernel loads (srcnn_debug_tc2_weights).  What is left between the two
is the order of the kernel's FP32 sums.  Three checks per frame:
  * interval: q(ve - EPS) <= out <= q(ve + EPS) on every pixel (ve: emulated pre-truncation value, q: trunc + clamp);
  * rate: D = fraction of pixels with out != q(ve) is at most D_MAX (plus D_SLACK pixels on tiny planes);
  * no structure: grouped by strip lane (x mod 124), distance from the right / left edge, ring rotation (r mod 11),
    distance from the frame's top / bottom, distance from a segment's first / last row (the work cut of the launch,
    srcnn_debug_tc2_partition) and frame index, no class has a binomial tail probability below 1e-9 under the frame's
    rate together with a rate above 5 D.  Applied to aperiodic content only: a periodic pattern repeats its near-integer
    values with its period, which clusters the off pixels without any fault of the kernel.
The strict FP32 variant (srcnn_fp32.cu) is checked against q(v) of the exact reference on frames cut into several row
chunks, byte for byte against the oracle (orc_cnn_at) on every pixel within INT_BAND of an integer, where q(v) cannot
decide, and byte for byte against the oracle across a chunk seam.  The exact reference itself is pinned to the oracle on
a CPU, and so are the emulation's precision and the packed weight image.

Measured on an NVIDIA B200 (1000 W power limit), unmodified kernel, the whole file in ~11 s:
  geometry                          pixels      D         largest EPS needed   worst class (p)    vs exact: max, exact
  grey x2 3840x2160, ovh 0 and 12   8 294 400   5.19e-4   0.128                none above 5 D     1, 96.17 %
  grey x4 15360x8640                132 710 400 5.22e-4   0.163                none above 5 D     1, 96.56 %
  grey batch 8 x 2560x1440          29 491 200  4.41e-4   0.122                none above 5 D
  stage seams, >= 50 000 pixels     up to 7.1e-4 (420x124 natural)     <= 0.107 (noise)    p >= 2.5e-4
  stage seams, smaller planes       at most 13 pixels off, never more than 0.2 pixel above 2.6e-3 N
  The float64 references cost 0.11 s per 3840x2160 plane and 1.7 s per 15360x8640 plane on the device.
D_MAX is 5 x the largest D seen on a plane of >= 50 000 pixels; no pixel needed more than 0.163 of EPS = 0.25.
"""
import ctypes as C
import json
import time

import numpy as np
import pytest

from conftest import natural_like

EPS = 0.25          # the largest |kernel - emulation| allowed before truncation, in LSB
D_MAX = 0.0035      # the largest fraction of pixels on which the kernel's byte differs from q(emulation)
D_SLACK = 2         # pixels allowed above D_MAX * N (a plane of a few hundred pixels has one or two off)
P_MIN = 1e-9        # a class stands out when its binomial tail is below this ...
RATE_X = 5.0        # ... and its rate is above RATE_X times the frame's
CLASS_MIN_PIXELS = 50_000   # below this the class test has too few pixels to mean anything
BAND_ROWS = 256     # output rows per band of the float64 reference (6 halo rows: a 15360x8640 plane fits in memory)
INT_BAND = 1e-3     # |v - round(v)| below this: float32 summation order decides the reference's byte

STRIP = 124         # output columns per strip of the tensor-core kernel
SLOTS = 11          # im2col ring slots (conv1 weight rotation = absolute row mod 11)

# ORC_* offsets of oracle/srcnn_oracle.c (the layout of srcnn_weights.bin)
W1, B1, W2, B2, W3, B3 = slice(0, 5184), slice(5184, 5248), slice(5248, 7296), slice(7296, 7328), slice(7328, 8128), 8128

# the packed operand image (srcnn_tc2.cu): eleven conv1 rotations of seven [64][16] tiles, conv2 five [32][16] tiles,
# conv3 two [32][16] tiles; element (n, k) of an [N][16] tile at (k/8)*(N*16) + n*16 + (k%8)*2 bytes
IMG_B1_VAR = 7 * 64 * 16 * 2
IMG_B2 = SLOTS * IMG_B1_VAR
IMG_B3 = IMG_B2 + 5 * 32 * 16 * 2
IMG_BYTES = IMG_B3 + 2 * 32 * 16 * 2
ONES_K1 = 110       # conv1 K index of the ones column (bias hi; 111: lo)
ONES_K2 = 64 + 14   # conv2 K index of the ones column in the bias step (hi; 79: lo)


# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------
def q(v):
    """clip(trunc(v), 0, 255): the reference's (int) cast then clamp (src/srcnn.cpp:238)"""
    return v.trunc().clamp(0, 255)


def q_np(v):
    return np.clip(np.trunc(v), 0, 255)


def _f16(a):
    """FP16 rounding of float64 values the way the kernel does it: its FP32 accumulator, then cvt.rn.f16"""
    import torch
    return a.to(torch.float32).to(torch.float16).to(torch.float64)


def _tiles(raw, n, ntiles):
    """[ntiles][2][n][8] FP16 bytes -> [n][16 * ntiles] float64 matrix B[n][k]"""
    t = raw.view(np.float16).reshape(ntiles, 2, n, 8).astype(np.float64)
    return t.transpose(2, 0, 1, 3).reshape(n, 16 * ntiles)


def packed_image():
    """the row-walking kernel's FP16 operand image, packed by the library's host code (no GPU needed)"""
    import srcnn_cpp_b200 as S
    L = S.load_library()
    f = L.srcnn_debug_tc2_weights
    f.argtypes = [C.c_void_p, C.c_size_t]
    f.restype = C.c_int
    img = np.zeros(IMG_BYTES, np.uint8)
    assert f(img.ctypes.data, IMG_BYTES) == 0
    return img


def decode_image(img):
    """-> (B1[11][64][112], B2[32][80], B3[32][32]) as float64"""
    b1 = np.stack([_tiles(img[v * IMG_B1_VAR:(v + 1) * IMG_B1_VAR], 64, 7) for v in range(SLOTS)])
    return b1, _tiles(img[IMG_B2:IMG_B3], 32, 5), _tiles(img[IMG_B3:IMG_BYTES], 32, 2)


_PARAMS = {}


def _params(emulate, device):
    """float64 (w1, b1, w2, b2, w3, b3) as torch tensors: the FP32 file's values, or (emulate) the FP16 values the kernel
    multiplies, taken from the packed image: rotation 0 holds kernel row j in slot j, bias = hi + lo"""
    import torch
    key = (emulate, str(device))
    if key not in _PARAMS:
        from oracle.oracle import load_params
        P = load_params().astype(np.float64)
        b3 = float(P[B3])
        if emulate:
            b1img, b2img, b3img = decode_image(packed_image())
            w1 = b1img[0][:, :90].reshape(64, 9, 10)[:, :, :9].reshape(64, 1, 9, 9)
            b1 = b1img[0][:, ONES_K1] + b1img[0][:, ONES_K1 + 1]
            w2 = b2img[:, :64].reshape(32, 64, 1, 1)
            b2 = b2img[:, ONES_K2] + b2img[:, ONES_K2 + 1]
            w3 = b3img[:25].T.reshape(1, 32, 5, 5)
        else:
            w1, b1 = P[W1].reshape(64, 1, 9, 9), P[B1]
            w2, b2 = P[W2].reshape(32, 64, 1, 1), P[B2]
            w3 = P[W3].reshape(1, 32, 5, 5)
        _PARAMS[key] = tuple(torch.from_numpy(np.ascontiguousarray(a)).to(device) for a in (w1, b1, w2, b2, w3)) + (b3,)
    return _PARAMS[key]


def cnn_v64(y, emulate=False, device="cpu", band=BAND_ROWS):
    """The pre-truncation conv3 value of every pixel of the u8 plane `y` (numpy or torch), float64, on `device`.
    Border semantics are the reference's two clamps: conv1 reads Y replicate-padded by 4, conv3 reads act2 replicate-padded
    by 2.  emulate: FP16 weights and biases from the packed image, act1 / act2 rounded to FP16 after the ReLU.  Computed in
    row bands of `band` output rows (6 halo rows each): the result does not depend on the band height."""
    import torch
    import torch.nn.functional as F
    w1, b1, w2, b2, w3, b3 = _params(emulate, device)
    Y = torch.as_tensor(y).to(device=device, dtype=torch.float64)
    H, W = Y.shape
    out = torch.empty((H, W), dtype=torch.float64, device=device)
    with torch.no_grad():
        for r0 in range(0, H, band):
            r1 = min(r0 + band, H)
            a0, a1 = max(r0 - 2, 0), min(r1 + 2, H)
            rows = torch.arange(a0 - 4, a1 + 4, device=device).clamp_(0, H - 1)
            a = F.relu(F.conv2d(F.pad(Y[rows][None, None], (4, 4, 0, 0), mode="replicate"), w1, b1))
            if emulate:
                a = _f16(a)
            a = F.relu(F.conv2d(a, w2, b2))
            if emulate:
                a = _f16(a)
            rows = torch.arange(r0 - 2, r1 + 2, device=device).clamp_(0, H - 1) - a0
            a = F.pad(a[:, :, rows], (2, 2, 0, 0), mode="replicate")
            out[r0:r1] = F.conv2d(a, w3)[0, 0] + b3
            del a
    return out


# ---------------------------------------------------------------------------------------------------------------------
# content
# ---------------------------------------------------------------------------------------------------------------------
def _content(kind, h, w, seed):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "natural":
        return np.ascontiguousarray(natural_like(rng, h, w)[:, :, 1])
    if kind.startswith("const"):
        return np.full((h, w), int(kind[5:]), np.uint8)
    if kind == "checker":
        return (np.indices((h, w)).sum(axis=0) % 2 * 255).astype(np.uint8)
    if kind == "saturating":   # hard 0 / 255 edges: the network overshoots on both sides (v < 0 and v > 255)
        yy, xx = np.indices((h, w))
        return np.where(((yy // 5) + (xx // 7)) % 2 == 1, 255, 0).astype(np.uint8)
    raise ValueError(kind)


KINDS = ["noise", "natural", "const0", "const128", "const255", "checker", "saturating"]


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests: the references themselves
# ---------------------------------------------------------------------------------------------------------------------
CNN_SHAPES = [(40, 52), (9, 13), (1, 1), (3, 70), (64, 5), (130, 140), (124, 128), (125, 129), (250, 31)]   # test_stage_parity


@pytest.mark.parametrize("h,w", CNN_SHAPES + [(17, 1), (1, 17), (2, 2), (126, 7)])
def test_exact_reference_is_the_oracle(oracle, h, w):
    """q(v) of the float64 reference == the oracle's bytes, except where v lies within INT_BAND of an integer (there the
    reference's own float32 summation order decides); such pixels are rare."""
    for i, kind in enumerate(KINDS):
        y = _content(kind, h, w, h * 1000 + w + i)
        v = cnn_v64(y).numpy()
        want = oracle.cnn(y).astype(np.float64)
        off = q_np(v) != want
        near = np.abs(v - np.round(v)) < INT_BAND
        assert not (off & ~near).any(), (kind, int((off & ~near).sum()))
        assert off.sum() <= 3, (kind, int(off.sum()))


def test_saturating_content_saturates():
    v = cnn_v64(_content("saturating", 40, 52, 0)).numpy()
    assert v.min() < 0 and v.max() > 256


@pytest.mark.parametrize("kind", ["noise", "natural"])
def test_emulation_keeps_the_budgeted_precision(kind):
    """The FP16 emulation against the exact reference: max 1 LSB, 93-99 % exact.  If the weight packing changed its rounding
    (or the activations lost precision), this moves on a CPU."""
    y = _content(kind, 300, 400, 7)
    d = np.abs(q_np(cnn_v64(y, emulate=True).numpy()) - q_np(cnn_v64(y).numpy()))
    exact = float((d == 0).mean())
    assert d.max() == 1 and 0.93 <= exact <= 0.99, (int(d.max()), exact)


@pytest.mark.parametrize("emulate", [False, True])
def test_banded_reference_equals_unbanded(emulate):
    y = _content("natural", 50, 61, 3)
    whole = cnn_v64(y, emulate=emulate, band=50)
    banded = cnn_v64(y, emulate=emulate, band=17)    # three bands: 17 + 17 + 16 rows
    assert float((whole - banded).abs().max()) <= 1e-9


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests: the packed weight image
# ---------------------------------------------------------------------------------------------------------------------
def _fp16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float64)


def _hi_lo(b):
    b = np.asarray(b, np.float32)
    hi = b.astype(np.float16).astype(np.float32)
    return hi.astype(np.float64), (b - hi).astype(np.float16).astype(np.float64)


def test_packed_image_layout():
    from oracle.oracle import load_params
    P = load_params()
    b1img, b2img, b3img = decode_image(packed_image())
    w1 = P[W1].reshape(64, 9, 9)
    hi1, lo1 = _hi_lo(P[B1])
    for v in range(SLOTS):
        want = np.zeros((64, 112))
        for s in range(SLOTS):
            j = (s - v) % SLOTS                  # slot s holds kernel row (s - v) mod 11; rows 9, 10 are outside the window
            if j <= 8:
                want[:, 10 * s:10 * s + 9] = _fp16(w1[:, j, :])
        want[:, ONES_K1], want[:, ONES_K1 + 1] = hi1, lo1
        assert np.array_equal(b1img[v], want), v
    w2 = P[W2].reshape(32, 64)
    hi2, lo2 = _hi_lo(P[B2])
    want = np.zeros((32, 80))
    want[:, :64] = _fp16(w2)
    want[:, ONES_K2], want[:, ONES_K2 + 1] = hi2, lo2
    assert np.array_equal(b2img, want)
    want = np.zeros((32, 32))
    want[:25] = _fp16(P[W3].reshape(32, 25)).T
    assert np.array_equal(b3img, want)
    # hi + lo carries each bias to ~22 bits
    for b, hi, lo in ((P[B1], hi1, lo1), (P[B2], hi2, lo2)):
        b = b.astype(np.float64)
        assert (np.abs(hi + lo - b) <= np.abs(b - hi) * 2.0 ** -11 + 2.0 ** -24).all()


def test_packed_image_export_refuses_a_wrong_size():
    import srcnn_cpp_b200 as S
    f = S.load_library().srcnn_debug_tc2_weights
    f.argtypes = [C.c_void_p, C.c_size_t]
    buf = np.zeros(IMG_BYTES + 16, np.uint8)
    assert f(buf.ctypes.data, IMG_BYTES - 16) != 0 and f(buf.ctypes.data, IMG_BYTES + 16) != 0 and f(None, IMG_BYTES) != 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU checks
# ---------------------------------------------------------------------------------------------------------------------
def _partition(nstrips, hb, nworkers, ovh):
    import srcnn_cpp_b200 as S
    f = S.load_library().srcnn_debug_tc2_partition
    f.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_longlong)]
    b = (C.c_longlong * (nworkers + 1))()
    assert f(nstrips, hb, nworkers, ovh, b) == 0
    return [int(x) for x in b]


def _segment_distances(engine, nframes, H, W, ovh):
    """[nframes * nstrips][H] distances of each row from the first / last row of its segment, for the cut launch_cnn_tc2
    makes: min(SMs, 152, ceil(total / 96)) CTAs of two pipelines each"""
    nstrips = (W + STRIP - 1) // STRIP * nframes
    total = nstrips * H
    grid = min(engine.sm_count, 152, max(1, -(-total // 96)))
    b = _partition(nstrips, H, 2 * grid, ovh)
    ds, de = np.zeros((nstrips, H), np.int64), np.zeros((nstrips, H), np.int64)
    for lo, hi in zip(b[:-1], b[1:]):
        while lo < hi:
            g, ra = divmod(lo, H)
            rb = ra + min(hi - lo, H - ra)
            ds[g, ra:rb] = np.arange(rb - ra)
            de[g, ra:rb] = np.arange(rb - ra)[::-1]
            lo += rb - ra
    return ds, de


def _classes(f, r, x, nframes, H, W, seg):
    """(name, class ids of the given pixels (-1: in no class), pixels per class) for every family of classes"""
    cols, rows = np.arange(W), np.arange(H)
    out = [("x mod 124", x % STRIP, nframes * H * np.bincount(cols % STRIP, minlength=STRIP)),
           ("r mod 11", r % SLOTS, nframes * W * np.bincount(rows % SLOTS, minlength=SLOTS))]
    for name, d, n in (("right edge", W - 1 - x, W), ("left edge", x, W), ("top", r, H), ("bottom", H - 1 - r, H)):
        k = min(6, n)
        out.append((name, np.where(d < k, d, -1), np.full(k, nframes * (H if name.endswith("edge") else W))))
    if nframes > 1:
        out.append(("frame", f, np.full(nframes, H * W)))
    if seg is not None:
        nstrips1 = (W + STRIP - 1) // STRIP
        width = np.minimum(STRIP, W - STRIP * np.arange(nstrips1))
        g = f * nstrips1 + x // STRIP
        for name, tab in (("segment start", seg[0]), ("segment end", seg[1])):
            d = tab[g, r]
            n = np.zeros(12, np.int64)
            for k in range(12):
                n[k] = ((tab == k) * np.tile(width, nframes)[:, None]).sum()
            out.append((name, np.where(d < 12, d, -1), n))
    return out


def _check(label, out, ve, v=None, seg=None, nframes=1, classes=True):
    """out: kernel bytes (torch u8, [F,]H,W), ve: emulated values (float64, same shape), v: exact values (north_star check).
    Returns the stats dict; asserts the interval, the rate and (with `classes`, on enough pixels) the absence of structure."""
    import torch
    from scipy.stats import binom
    o = out.to(ve.device, torch.float64).reshape(nframes, *out.shape[-2:])
    ve = ve.reshape(o.shape)
    H, W = o.shape[-2:]
    N = o.numel()
    mis = o != q(ve)
    idx = mis.nonzero().cpu().numpy()
    f, r, x = idx[:, 0], idx[:, 1], idx[:, 2]
    ov, vv = o[mis], ve[mis]
    need = torch.where(ov > vv.trunc().clamp(0, 255), ov - vv, vv - ov - 1)   # the EPS each off pixel needs
    st = dict(label=label, pixels=N, D=len(f) / N, eps=float(need.max()) if len(f) else 0.0)
    worst = (1.0, None)
    if classes and N >= CLASS_MIN_PIXELS and len(f):
        D = len(f) / N
        for name, ids, n in _classes(f, r, x, nframes, H, W, seg):
            k = np.bincount(ids[ids >= 0], minlength=len(n))
            for c in range(len(n)):
                if n[c] == 0 or k[c] == 0:
                    continue
                p = float(binom.sf(k[c] - 1, int(n[c]), D))
                if k[c] / n[c] > RATE_X * D and p < worst[0]:
                    worst = (p, "%s=%d: %d / %d" % (name, c, k[c], n[c]))
    st["worst_p"], st["worst_class"] = worst
    if v is not None:
        dv = (o - q(v.reshape(o.shape))).abs()
        st["exact_max"] = int(dv.max())
        st["exact_frac"] = float((dv == 0).double().mean())
        st["exact_le1"] = float((dv <= 1).double().mean())
    print("CNN_PRECISION " + json.dumps(st))
    assert st["eps"] <= EPS, st
    assert len(f) <= D_MAX * N + D_SLACK, st
    assert worst[0] >= P_MIN, st
    if v is not None:
        assert st["exact_max"] <= 2 and st["exact_le1"] >= 0.999, st
    return st


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


def _stage_tc(engine, y):
    import torch
    import srcnn_cpp_b200 as S
    out = torch.zeros(y.shape, dtype=torch.uint8, device="cuda:0")
    engine.stage_cnn(_dev(y), out, variant=S.VARIANT_TC)
    engine.sync()
    return out


SEAM_SHAPES = ([(420, w) for w in (123, 124, 125, 126, 127, 128, 247, 248, 249, 250, 251, 252, 373)] +
               [(h, 251) for h in list(range(1, 13)) + [22, 23]] + [(2000, 7), (3, 5000)] + CNN_SHAPES)
GPU_KINDS = ["noise", "natural", "const0", "const128", "const255", "checker", "saturating"]


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SEAM_SHAPES)
def test_tc_stage_on_seams(engine, h, w):
    """stage_cnn, tensor-core variant, on shapes where the last strip has 0-4 real columns or none spare, every ring
    rotation of a short frame, many segments per strip and a very wide frame"""
    engine.set_tc2_seg_ovh(12)
    for i, kind in enumerate(GPU_KINDS):
        y = _content(kind, h, w, 31 * h + w + i)
        out = _stage_tc(engine, y)
        ve = cnn_v64(y, emulate=True, device="cuda:0")
        _check("stage %dx%d %s" % (h, w, kind), out, ve, seg=_segment_distances(engine, 1, h, w, 12),
               classes=kind in ("noise", "natural"))


def _grey_source(h, w, seed):
    return np.ascontiguousarray(natural_like(np.random.default_rng(seed), h, w)[:, :, 1])


def _resized(engine, src, scale):
    import torch
    import srcnn_cpp_b200 as S
    ow, oh = S.out_dims(src.shape[1], src.shape[0], scale)
    y = torch.zeros((oh, ow), dtype=torch.uint8, device="cuda:0")
    engine.stage_resize_plane(src, scale, y)
    engine.sync()
    return y


def _grey_call(engine, src, scale):
    import torch
    import srcnn_cpp_b200 as S
    ow, oh = S.out_dims(src.shape[1], src.shape[0], scale)
    out = torch.zeros((oh, ow), dtype=torch.uint8, device="cuda:0")
    engine.process_device(src, scale, out, order=S.ORDER_GRAY)
    engine.sync()
    return out


def _timed(fn, *a, **k):
    t = time.perf_counter()
    r = fn(*a, **k)
    import torch
    torch.cuda.synchronize()
    print("CNN_PRECISION_TIME %s %.2f s" % (fn.__name__, time.perf_counter() - t))
    return r


@pytest.fixture(scope="module")
def frame_4k(engine):
    """Y of a natural-like 1920x1080 grey frame at x2 (3840x2160, the bench geometry), its exact and emulated values"""
    src = _dev(_grey_source(1080, 1920, 71))
    y = _resized(engine, src, 2.0)
    v = _timed(cnn_v64, y, device="cuda:0")
    ve = _timed(cnn_v64, y, emulate=True, device="cuda:0")
    return src, y, v, ve


@pytest.mark.gpu
@pytest.mark.parametrize("ovh", [0, 12])
def test_tc_full_4k_frame_every_pixel(engine, frame_4k, ovh):
    src, y, v, ve = frame_4k
    try:
        engine.set_tc2_seg_ovh(ovh)
        out = _grey_call(engine, src, 2.0)
    finally:
        engine.set_tc2_seg_ovh(12)
    _check("grey x2 3840x2160 ovh=%d" % ovh, out, ve, v=v, seg=_segment_distances(engine, 1, 2160, 3840, ovh))


@pytest.mark.gpu
def test_tc_full_16k_frame_every_pixel(engine):
    """x4 geometry: a 3840x2160 grey source -> 15360x8640, every pixel against both references"""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 24 * 2**30:
        pytest.skip("needs ~12 GB of device memory")
    engine.set_tc2_seg_ovh(12)
    src = _dev(_grey_source(2160, 3840, 72))
    out = _grey_call(engine, src, 4.0)
    y = _resized(engine, src, 4.0)
    ve = _timed(cnn_v64, y, emulate=True, device="cuda:0")
    v = _timed(cnn_v64, y, device="cuda:0")
    _check("grey x4 15360x8640", out, ve, v=v, seg=_segment_distances(engine, 1, 8640, 15360, 12))
    del ve, v, out, y
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_tc_batch_across_frame_boundaries(engine):
    """An 8-frame grey batch in one launch (1280x720 -> 2560x1440), different content per frame, so that pipelines cross
    from one frame into the next; run on a workspace another geometry has just used"""
    import torch
    engine.set_tc2_seg_ovh(12)
    _grey_call(engine, _dev(_grey_source(333, 517, 5)), 3.0)          # dirty workspace
    frames = [_grey_source(720, 1280, 80 + k) if k % 3 else _content("noise", 720, 1280, 80 + k) for k in range(8)]
    src = _dev(np.stack(frames))
    out = torch.zeros((8, 1440, 2560), dtype=torch.uint8, device="cuda:0")
    import srcnn_cpp_b200 as S
    engine.process_batch_device(src, 2.0, out, order=S.ORDER_GRAY)
    engine.sync()
    ve = torch.stack([cnn_v64(_resized(engine, src[k], 2.0), emulate=True, device="cuda:0") for k in range(8)])
    _check("grey batch 8 x 2560x1440", out, ve, seg=_segment_distances(engine, 8, 1440, 2560, 12), nframes=8)


def _fp32_check(engine, oracle, y, v, seams, cw=320, m=6):
    """FP32 variant on the u8 device plane y: q(v) outside the integer band, the oracle's bytes (orc_cnn_at) on every pixel
    inside it, and the oracle's bytes on a crop around each chunk seam (with m px of context where the image continues)"""
    import torch
    import srcnn_cpp_b200 as S
    H, W = y.shape
    out = torch.zeros((H, W), dtype=torch.uint8, device="cuda:0")
    engine.stage_cnn(y, out, variant=S.VARIANT_FP32)
    engine.sync()
    o = out.to(torch.float64)
    near = (v - v.round()).abs() < INT_BAND
    off = (o != q(v)) & ~near
    assert int(off.sum()) == 0, [tuple(p) for p in off.nonzero()[:10].tolist()]
    got, Y = out.cpu().numpy(), y.cpu().numpy()
    rc = near.nonzero().cpu().numpy()
    _, want = oracle.cnn_at(Y, rc[:, 0], rc[:, 1])
    bad = got[rc[:, 0], rc[:, 1]] != want
    assert not bad.any(), (len(rc), [tuple(p) for p in rc[bad][:10].tolist()])
    for seam in seams:
        r0, r1 = max(seam - 20, 0), min(seam + 20, H)
        c0 = (W - cw) // 2
        ra, rb, ca, cb = max(r0 - m, 0), min(r1 + m, H), max(c0 - m, 0), min(c0 + cw + m, W)
        ref = oracle.cnn(np.ascontiguousarray(Y[ra:rb, ca:cb]))[r0 - ra:r1 - ra, c0 - ca:c0 - ca + cw]
        assert np.array_equal(got[r0:r1, c0:c0 + cw], ref), seam


@pytest.mark.gpu
def test_fp32_chunk_seams_wide_plane(engine, oracle):
    """65536 columns: the FP32 variant works in 60-row chunks (512 MiB / (W * 128 B) - 4), so 130 rows have two seams"""
    y = _dev(_grey_source(130, 65536, 73))
    v = cnn_v64(y, device="cuda:0")
    _fp32_check(engine, oracle, y, v, seams=(60, 120))


@pytest.mark.gpu
def test_fp32_chunk_seam_4k_plane(engine, oracle, frame_4k):
    """3840x2160: one chunk seam, at row 1088"""
    _, y, v, _ = frame_4k
    _fp32_check(engine, oracle, y, v, seams=(1088,))
