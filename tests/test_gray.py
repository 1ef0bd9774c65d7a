"""The greyscale path (SRCNN_ORDER_GRAY): one-channel images end to end on the device.

A grey pixel v replicated to B = G = R = v has Y = v and Cr = Cb = 128, which stay 128 through the resize and convert back to
B = G = R = Y'.  So the grey path must be bit-identical to every channel of the colour path on np.repeat(g, 3, axis=2), and the
FP32 variant must equal oracle.cnn(oracle.resize_cubic(g)) exactly.  Reference path: src/srcnn.cpp:505-659 on a grey image."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import natural_like

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _grey(rng, h, w):
    return np.ascontiguousarray(natural_like(rng, h, w)[:, :, 1])


def _rep3(g):
    return np.ascontiguousarray(np.repeat(g[..., None], 3, axis=-1))


def test_abi_surface():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"SRCNN_ORDER_GRAY\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_GRAY == 2
    L = S.load_library()
    assert hasattr(L, "srcnn_stage_resize_plane_device")
    assert "srcnn_stage_resize_plane_device" in S.ABI_SYMBOLS


# (w, h, scale, dst pitch pad, dst byte offset): reaches the integer x2 / x4 kernel (ow % 8 == 0), the tiled kernel (x2 with
# ow % 8 != 0 or a pitch that is not a multiple of 8, x1.5, x3, x2.7), the direct kernel (0.5, 0.3), 1x1, and a destination the
# word stores cannot take (staged and copied)
RESIZE_GEOS = [(96, 40, 2.0, 0, 0), (64, 30, 4.0, 0, 0), (1000, 70, 2.0, 0, 0), (93, 41, 2.0, 0, 0), (77, 53, 1.5, 0, 0),
               (50, 33, 3.0, 0, 0), (61, 29, 2.7, 0, 0), (120, 90, 0.5, 0, 0), (200, 150, 0.3, 0, 0), (1, 1, 2.0, 0, 0),
               (1, 1, 1.0, 0, 0), (96, 40, 2.0, 4, 0), (96, 40, 2.0, 0, 1), (96, 40, 2.0, 3, 0), (77, 53, 1.5, 1, 3)]


@gpu
@pytest.mark.parametrize("w,h,scale,pad,ofs", RESIZE_GEOS)
def test_stage_resize_plane_bit_exact(engine, oracle, w, h, scale, pad, ofs):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(w * 7 + h)
    g = rng.integers(0, 256, (h, w), dtype=np.uint8)
    ow, oh = S.out_dims(w, h, scale)
    pitch = ow + pad
    buf = torch.full((oh * pitch + ofs + 64,), 77, dtype=torch.uint8, device="cuda:0")
    dst = buf[ofs:ofs + oh * pitch].view(oh, pitch)[:, :ow]
    engine.stage_resize_plane(torch.from_numpy(g).to("cuda:0"), scale, dst)
    engine.sync()
    assert np.array_equal(dst.cpu().numpy(), oracle.resize_cubic(g, ow, oh))
    # nothing outside the plane is written
    assert int(buf[:ofs].ne(77).sum()) == 0 and int(buf[ofs + oh * pitch:].ne(77).sum()) == 0
    assert int(buf[ofs:ofs + oh * pitch].view(oh, pitch)[:, ow:].ne(77).sum()) == 0


def _colour_channels(out3):
    return [out3[..., k] for k in range(3)]


# the x1.5 golden size, x2 / x3 / x4, odd sizes
GEOS = [(384, 384, 1.5), (160, 96, 2.0), (53, 37, 3.0), (64, 48, 4.0), (97, 61, 2.0), (131, 29, 1.25)]


@gpu
@pytest.mark.parametrize("variant_name", ["tc", "fp32"])
def test_grey_equals_every_colour_channel(engine, oracle, variant_name):
    import torch
    import srcnn_cpp_b200 as S
    engine.set_variant(S.VARIANT_FP32 if variant_name == "fp32" else S.VARIANT_TC)
    try:
        rng = np.random.default_rng(11)
        for (w, h, scale) in GEOS:
            g = _grey(rng, h, w)
            ow, oh = S.out_dims(w, h, scale)
            colour = engine.process(_rep3(g), scale)
            host = engine.process(g, scale, order=S.ORDER_GRAY)
            dev = torch.zeros((oh, ow), dtype=torch.uint8, device="cuda:0")
            engine.process_device(torch.from_numpy(g).to("cuda:0"), scale, dev, order=S.ORDER_GRAY)
            engine.sync()
            dev = dev.cpu().numpy()
            assert host.shape == (oh, ow)
            for ch in _colour_channels(colour):
                assert np.array_equal(host, ch), (w, h, scale)
            assert np.array_equal(dev, host), (w, h, scale)
            want = oracle.cnn(oracle.resize_cubic(g, ow, oh))
            if variant_name == "fp32":
                assert np.array_equal(host, want), (w, h, scale)
            else:
                d = np.abs(host.astype(np.int16) - want.astype(np.int16))
                assert d.max() <= 2 and (d <= 1).mean() >= 0.999, (w, h, scale, int(d.max()))
    finally:
        engine.set_variant(S.VARIANT_TC)


@gpu
def test_grey_device_strided_rows(engine):
    """Source and destination rows with padding: strides are in bytes, >= w / ow."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(12)
    g = _grey(rng, 45, 70)
    ow, oh = S.out_dims(70, 45, 2.0)
    src = torch.zeros((45, 77), dtype=torch.uint8, device="cuda:0")
    src[:, :70] = torch.from_numpy(g).to("cuda:0")
    dst = torch.full((oh, ow + 5), 9, dtype=torch.uint8, device="cuda:0")
    engine.process_device(src[:, :70], 2.0, dst[:, :ow], order=S.ORDER_GRAY)
    engine.sync()
    assert np.array_equal(dst[:, :ow].cpu().numpy(), engine.process(g, 2.0, order=S.ORDER_GRAY))
    assert int(dst[:, ow:].ne(9).sum()) == 0


@gpu
@pytest.mark.parametrize("pad", [0, 3])
def test_grey_batches_equal_frame_by_frame(engine, pad):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(13 + pad)
    n, w, h, scale = 5, 96, 56, 2.0
    ow, oh = S.out_dims(w, h, scale)
    frames = np.stack([_grey(rng, h, w) for _ in range(n)])
    want = np.stack([engine.process(f, scale, order=S.ORDER_GRAY) for f in frames])
    assert np.array_equal(engine.process_batch(frames, scale, order=S.ORDER_GRAY), want)
    # padded frame strides (device): frames `pad` rows apart
    src = torch.zeros((n, h + pad, w), dtype=torch.uint8, device="cuda:0")
    src[:, :h] = torch.from_numpy(frames).to("cuda:0")
    dst = torch.zeros((n, oh + pad, ow), dtype=torch.uint8, device="cuda:0")
    engine.process_batch_device(src[:, :h], scale, dst[:, :oh], order=S.ORDER_GRAY)
    engine.sync()
    assert np.array_equal(dst[:, :oh].cpu().numpy(), want)
    # padded frame strides (host)
    hsrc = np.zeros((n, h + pad, w), np.uint8)
    hsrc[:, :h] = frames
    hdst = np.zeros((n, oh + pad, ow), np.uint8)
    assert engine.L.srcnn_process_batch_host(engine.ctx, hsrc.ctypes.data, n, w, h, w, (h + pad) * w, S.ORDER_GRAY, C.c_float(scale),
                                             hdst.ctypes.data, ow, (oh + pad) * ow) == 0
    assert np.array_equal(hdst[:, :oh], want)


@gpu
def test_grey_bands_reassemble(engine):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(14)
    w, h, scale = 120, 100, 2.0
    g = _grey(rng, h, w)
    ow, oh = S.out_dims(w, h, scale)
    whole = engine.process(g, scale, order=S.ORDER_GRAY)
    dg = torch.from_numpy(g).to("cuda:0")
    cuts = [0, 37, 38, 121, oh]
    dev = torch.zeros((oh, ow), dtype=torch.uint8, device="cuda:0")
    host = np.zeros((oh, ow), np.uint8)
    for r0, r1 in zip(cuts[:-1], cuts[1:]):
        s0, s1 = S.band_src_rows(h, scale, r0, r1)
        engine.process_band_device(dg[s0:s1].contiguous(), w, h, s0, s1, scale, r0, r1, dev[r0:r1], order=S.ORDER_GRAY)
        host[r0:r1] = engine.process_band_host(g, scale, r0, r1, order=S.ORDER_GRAY)
    engine.sync()
    assert np.array_equal(dev.cpu().numpy(), whole)
    assert np.array_equal(host, whole)


@gpu
def test_grey_multi_engine(engine):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(15)
    w, h, scale = 100, 76, 2.0
    ow, oh = S.out_dims(w, h, scale)
    g = _grey(rng, h, w)
    frames = np.stack([_grey(rng, h, w) for _ in range(3)])
    whole = engine.process(g, scale, order=S.ORDER_GRAY)
    per_frame = np.stack([engine.process(f, scale, order=S.ORDER_GRAY) for f in frames])
    m = S.MultiEngine(devices=[0, 0])
    try:
        assert np.array_equal(m.process_banded(g, scale, order=S.ORDER_GRAY), whole)
        assert np.array_equal(m.process_batch(frames, scale, order=S.ORDER_GRAY), per_frame)
        plan = m.band_plan(h, scale)
        dg = torch.from_numpy(g).to("cuda:0")
        srcs = [dg[s0:s1].contiguous() for (r0, r1, s0, s1) in plan]
        dst = torch.zeros((oh, ow), dtype=torch.uint8, device="cuda:0")
        dsts = [dst[r0:r1] for (r0, r1, s0, s1) in plan]
        torch.cuda.synchronize()
        m.process_banded_device(srcs, w, h, scale, dsts, order=S.ORDER_GRAY)
        assert np.array_equal(dst.cpu().numpy(), whole)
        df = torch.from_numpy(frames).to("cuda:0")
        dd = torch.zeros((3, oh, ow), dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        m.process_batch_device([df[:2], df[2:]], scale, [dd[:2], dd[2:]], order=S.ORDER_GRAY)
        assert np.array_equal(dd.cpu().numpy(), per_frame)
    finally:
        m.close()


@gpu
def test_grey_tc_call_is_two_launches(engine):
    import torch
    import srcnn_cpp_b200 as S
    src = torch.zeros((90, 128), dtype=torch.uint8, device="cuda:0")
    dst = torch.zeros((180, 256), dtype=torch.uint8, device="cuda:0")
    engine.process_device(src, 2.0, dst, order=S.ORDER_GRAY)     # warm: tap tables, workspace
    n0 = engine.launches
    engine.process_device(src, 2.0, dst, order=S.ORDER_GRAY)
    engine.sync()
    assert engine.launches - n0 == 2


def _overlap(engine, on):
    engine.L.srcnn_debug_overlap.argtypes = [C.c_void_p, C.c_int]
    engine.L.srcnn_debug_overlap.restype = C.c_longlong
    return int(engine.L.srcnn_debug_overlap(engine.ctx, on))


@gpu
def test_grey_call_ends_the_early_start_chain(engine):
    """colour -> grey -> colour -> colour on one stream: results equal the serialised ones; neither the grey call nor the colour
    call right after it starts early, the last one does."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(16)
    w, h, scale = 256, 144, 2.0
    ow, oh = S.out_dims(w, h, scale)
    cols = [torch.from_numpy(natural_like(rng, h, w)).to("cuda:0") for _ in range(3)]
    grey = torch.from_numpy(_grey(rng, h, w)).to("cuda:0")
    seq = [(cols[0], S.ORDER_BGR), (grey, S.ORDER_GRAY), (cols[1], S.ORDER_BGR), (cols[2], S.ORDER_BGR)]

    def outs():
        return [torch.zeros((oh, ow) + (() if o == S.ORDER_GRAY else (3,)), dtype=torch.uint8, device="cuda:0") for _, o in seq]
    try:
        _overlap(engine, 0)
        ref = outs()
        for (src, o), d in zip(seq, ref):
            engine.process_device(src, scale, d, order=o)
            engine.sync()
        _overlap(engine, 1)
        got = outs()
        counts = []
        for (src, o), d in zip(seq, got):
            engine.process_device(src, scale, d, order=o)
            counts.append(_overlap(engine, -1))
        engine.sync()
        for a, b in zip(ref, got):
            assert torch.equal(a, b)
        assert counts[1] == counts[0] and counts[2] == counts[1] and counts[3] == counts[2] + 1
    finally:
        _overlap(engine, 1)


@gpu
def test_grey_after_larger_colour_calls_equals_fresh_context(engine):
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(17)
    engine.process(natural_like(rng, 300, 400), 2.0)
    engine.process(natural_like(rng, 200, 260), 3.0)
    g = _grey(rng, 70, 90)
    got = engine.process(g, 2.0, order=S.ORDER_GRAY)
    fresh = S.Engine(device=0)
    try:
        assert np.array_equal(got, fresh.process(g, 2.0, order=S.ORDER_GRAY))
    finally:
        fresh.close()


@gpu
def test_grey_ignores_fused_merge(engine):
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(18)
    g = _grey(rng, 64, 96)
    want = engine.process(g, 2.0, order=S.ORDER_GRAY)
    frames = np.stack([g, g[::-1].copy()])
    want_b = engine.process_batch(frames, 2.0, order=S.ORDER_GRAY)
    engine.set_fuse_merge(True)
    try:
        assert np.array_equal(engine.process(g, 2.0, order=S.ORDER_GRAY), want)
        assert np.array_equal(engine.process_batch(frames, 2.0, order=S.ORDER_GRAY), want_b)
    finally:
        engine.set_fuse_merge(False)


def _process_srcnn():
    import srcnn_cpp_b200 as S
    fn = S.load_library()._Z12ProcessSRCNNPKhjjjfRPhRj
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.POINTER(C.c_void_p), C.POINTER(C.c_uint)]
    return fn


@gpu
@pytest.mark.parametrize("d", [1, 2])
def test_process_srcnn_grey(engine, oracle, d):
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(19 + d)
    w, h, scale = 46, 30, 2.0
    g = _grey(rng, h, w)
    alpha = rng.integers(0, 256, (h, w), dtype=np.uint8)
    buf = g if d == 1 else np.ascontiguousarray(np.stack([g, alpha], axis=-1))
    out, sz = C.c_void_p(), C.c_uint()
    assert _process_srcnn()(buf.ctypes.data, w, h, d, C.c_float(scale), C.byref(out), C.byref(sz)) == 0
    ow, oh = S.out_dims(w, h, scale)
    assert sz.value == ow * oh * d
    got = np.ctypeslib.as_array((C.c_uint8 * sz.value).from_address(out.value)).reshape(oh, ow, d).copy()
    assert np.array_equal(got[:, :, 0], engine.process(g, scale, order=S.ORDER_GRAY))
    if d == 2:
        assert np.array_equal(got[:, :, 1], oracle.resize_cubic(alpha, ow, oh))


@gpu
def test_grey_argument_checks(engine):
    import torch
    import srcnn_cpp_b200 as S
    L, ctx = engine.L, engine.ctx
    src = torch.zeros((20, 32, 3), dtype=torch.uint8, device="cuda:0")
    y = torch.zeros((40, 64), dtype=torch.uint8, device="cuda:0")
    dst = torch.zeros((40, 64, 3), dtype=torch.uint8, device="cuda:0")
    p = lambda t: C.c_void_p(t.data_ptr())
    assert L.srcnn_stage_color_bicubic_device(ctx, p(src), 32, 20, 96, S.ORDER_GRAY, C.c_float(2.0), p(y), p(y), p(y), 64) == S.E_ARG
    assert L.srcnn_stage_merge_device(ctx, p(y), p(y), p(y), 64, 40, 64, S.ORDER_GRAY, p(dst), 192) == S.E_ARG
    g = torch.zeros((20, 32), dtype=torch.uint8, device="cuda:0")
    assert L.srcnn_process_device(ctx, p(g), 32, 20, 31, S.ORDER_GRAY, C.c_float(2.0), p(y), 64) == S.E_ARG
    assert L.srcnn_process_device(ctx, p(g), 32, 20, 32, S.ORDER_GRAY, C.c_float(2.0), p(y), 63) == S.E_ARG
    assert L.srcnn_stage_resize_plane_device(ctx, p(g), 32, 20, 31, C.c_float(2.0), p(y), 64) == S.E_ARG
    assert L.srcnn_stage_resize_plane_device(ctx, p(g), 32, 20, 32, C.c_float(2.0), p(y), 63) == S.E_ARG
    assert L.srcnn_process_device(ctx, p(g), 32, 20, 32, 3, C.c_float(2.0), p(y), 64) == S.E_ARG
    engine.sync()
