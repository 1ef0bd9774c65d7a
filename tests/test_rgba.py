"""The four-channel path (SRCNN_ORDER_BGRA / SRCNN_ORDER_RGBA): 4-byte pixels end to end on the device.

Contract (include/srcnn_b200.h): bytes 0..2 of every output pixel equal the 3-channel call with the matching order on bytes 0..2
of the source, whatever the alpha byte is; byte 3 equals the one-plane cubic resize of the alpha plane (oracle.resize_cubic,
srcnn_stage_resize_plane_device).  No new tolerance: every check below is byte for byte against an existing call or the oracle."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import natural_like

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _rgba(rng, h, w):
    """colour bytes 0..2 from natural_like, random (non-constant) alpha in byte 3"""
    a = rng.integers(0, 256, (h, w, 1), dtype=np.uint8)
    return np.ascontiguousarray(np.concatenate([natural_like(rng, h, w), a], axis=2))


def _three(order):
    import srcnn_cpp_b200 as S
    return S.ORDER_BGR if order == S.ORDER_BGRA else S.ORDER_RGB


# --------------------------------------------------------------------------------------------------------------------------
# CPU
# --------------------------------------------------------------------------------------------------------------------------
def test_enum_values_match_header():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"SRCNN_ORDER_BGRA\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_BGRA == 3
    assert int(re.search(r"SRCNN_ORDER_RGBA\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_RGBA == 4


def test_library_loads_abi_version_unchanged():
    import srcnn_cpp_b200 as S
    L = S.load_library()
    assert L.srcnn_abi_version() == 2
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"#define SRCNN_B200_ABI_VERSION (\d+)", hdr).group(1)) == 2


def test_host_image_shape_checks():
    import srcnn_cpp_b200 as S
    for order in (S.ORDER_BGRA, S.ORDER_RGBA):
        assert S._pixel_shape(order) == (4,)
        S._check_host_image(np.zeros((5, 7, 4), np.uint8), order, 1)
        S._check_host_image(np.zeros((2, 5, 7, 4), np.uint8), order, 2)
        for bad in (np.zeros((5, 7, 3), np.uint8), np.zeros((5, 7), np.uint8), np.zeros((5, 7, 4), np.float32)):
            with pytest.raises(S.SrcnnError) as e:
                S._check_host_image(bad, order, 1)
            assert e.value.status == S.E_ARG and "HxWx4" in str(e.value)
    with pytest.raises(S.SrcnnError):
        S._check_host_image(np.zeros((5, 7, 4), np.uint8), S.ORDER_BGR, 1)


# --------------------------------------------------------------------------------------------------------------------------
# GPU
# --------------------------------------------------------------------------------------------------------------------------
# the geometries of tests/test_gray.py: the integer x2 / x4 kernel (ow % 8 == 0), the tiled kernel (x2 with ow % 8 != 0, x1.5,
# x3, x2.7, x1.25), the direct kernel (0.5, 0.3), odd sizes and 1x1
GEOS = [(96, 40, 2.0), (64, 30, 4.0), (1000, 70, 2.0), (93, 41, 2.0), (77, 53, 1.5), (50, 33, 3.0), (61, 29, 2.7),
        (120, 90, 0.5), (200, 150, 0.3), (1, 1, 2.0), (1, 1, 1.0), (384, 384, 1.5), (160, 96, 2.0), (53, 37, 3.0),
        (64, 48, 4.0), (97, 61, 2.0), (131, 29, 1.25)]


@gpu
@pytest.mark.parametrize("variant_name", ["tc", "fp32"])
@pytest.mark.parametrize("order_name", ["bgra", "rgba"])
def test_four_channel_matches_colour_call_and_alpha_resize(engine, oracle, variant_name, order_name):
    import torch
    import srcnn_cpp_b200 as S
    order = S.ORDER_BGRA if order_name == "bgra" else S.ORDER_RGBA
    engine.set_variant(S.VARIANT_FP32 if variant_name == "fp32" else S.VARIANT_TC)
    try:
        rng = np.random.default_rng(31 + order)
        for (w, h, scale) in GEOS:
            img = _rgba(rng, h, w)
            ow, oh = S.out_dims(w, h, scale)
            got = engine.process(img, scale, order=order)
            assert got.shape == (oh, ow, 4)
            colour = engine.process(np.ascontiguousarray(img[..., :3]), scale, order=_three(order))
            assert np.array_equal(got[..., :3], colour), (w, h, scale)
            assert np.array_equal(got[..., 3], oracle.resize_cubic(img[..., 3], ow, oh)), (w, h, scale)
            dev = torch.zeros((oh, ow, 4), dtype=torch.uint8, device="cuda:0")
            engine.process_device(torch.from_numpy(img).to("cuda:0"), scale, dev, order=order)
            engine.sync()
            assert np.array_equal(dev.cpu().numpy(), got), (w, h, scale)
            if variant_name == "fp32":
                bgr = img[..., :3] if order == S.ORDER_BGRA else img[..., 2::-1]
                want = oracle.pipeline(np.ascontiguousarray(bgr), scale)
                got_bgr = got[..., :3] if order == S.ORDER_BGRA else got[..., 2::-1]
                assert np.array_equal(got_bgr, want), (w, h, scale)
    finally:
        engine.set_variant(S.VARIANT_TC)


@gpu
def test_alpha_has_no_influence_on_colour(engine):
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(32)
    for (w, h, scale) in [(96, 40, 2.0), (93, 41, 2.0), (77, 53, 1.5), (120, 90, 0.5)]:
        a = _rgba(rng, h, w)
        b = a.copy()
        b[..., 3] = rng.integers(0, 256, (h, w), dtype=np.uint8)
        for order in (S.ORDER_BGRA, S.ORDER_RGBA):
            ra, rb = engine.process(a, scale, order=order), engine.process(b, scale, order=order)
            assert np.array_equal(ra[..., :3], rb[..., :3]), (w, h, scale, order)
            assert not np.array_equal(ra[..., 3], rb[..., 3])


@gpu
@pytest.mark.parametrize("src_ofs,dst_ofs", [(0, 0), (1, 1), (4, 4), (1, 0), (0, 3)])
def test_device_strides_and_alignment(engine, src_ofs, dst_ofs):
    """Padded source / destination rows (strides in bytes) and pointers that are not 16- or 4-byte aligned: the 128-bit,
    32-bit and byte-wise staging of the integer kernel, the wide and the scalar merge.  Nothing outside ow*4 of a row is written."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(33 + src_ofs * 7 + dst_ofs)
    for (w, h, scale) in [(96, 40, 2.0), (77, 53, 1.5), (64, 30, 4.0)]:
        img = _rgba(rng, h, w)
        ow, oh = S.out_dims(w, h, scale)
        want = engine.process(img, scale, order=S.ORDER_BGRA)
        sp, dp = 4 * w + 12, 4 * ow + 20          # row pitches in bytes
        sbuf = torch.zeros(src_ofs + h * sp + 64, dtype=torch.uint8, device="cuda:0")
        sview = sbuf[src_ofs:src_ofs + h * sp].view(h, sp)
        sview[:, :4 * w] = torch.from_numpy(img.reshape(h, 4 * w)).to("cuda:0")
        dbuf = torch.full((dst_ofs + oh * dp + 64,), 201, dtype=torch.uint8, device="cuda:0")
        dview = dbuf[dst_ofs:dst_ofs + oh * dp].view(oh, dp)
        p = lambda t: C.c_void_p(t.data_ptr())
        assert engine.L.srcnn_process_device(engine.ctx, p(sview), w, h, sp, S.ORDER_BGRA, C.c_float(scale), p(dview), dp) == 0
        engine.sync()
        assert np.array_equal(dview[:, :4 * ow].cpu().numpy().reshape(oh, ow, 4), want), (w, h, scale)
        assert int(dview[:, 4 * ow:].ne(201).sum()) == 0
        assert int(dbuf[:dst_ofs].ne(201).sum()) == 0 and int(dbuf[dst_ofs + oh * dp:].ne(201).sum()) == 0


@gpu
@pytest.mark.parametrize("scale", [2.0, 1.5])
def test_batches_equal_frame_by_frame(engine, scale):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(34)
    n, w, h = 5, 96, 56
    ow, oh = S.out_dims(w, h, scale)
    frames = np.stack([_rgba(rng, h, w) for _ in range(n)])
    want = np.stack([engine.process(f, scale, order=S.ORDER_RGBA) for f in frames])
    assert np.array_equal(engine.process_batch(frames, scale, order=S.ORDER_RGBA), want)
    src = torch.from_numpy(frames).to("cuda:0")
    # tight frames: the chunk's results are one tall image, one merge launch
    dst = torch.zeros((n, oh, ow, 4), dtype=torch.uint8, device="cuda:0")
    engine.process_batch_device(src, scale, dst, order=S.ORDER_RGBA)
    engine.sync()
    assert np.array_equal(dst.cpu().numpy(), want)
    # padded frame strides: a merge per frame
    psrc = torch.zeros((n, h + 3, w, 4), dtype=torch.uint8, device="cuda:0")
    psrc[:, :h] = src
    pdst = torch.full((n, oh + 2, ow, 4), 7, dtype=torch.uint8, device="cuda:0")
    engine.process_batch_device(psrc[:, :h], scale, pdst[:, :oh], order=S.ORDER_RGBA)
    engine.sync()
    assert np.array_equal(pdst[:, :oh].cpu().numpy(), want)
    assert int(pdst[:, oh:].ne(7).sum()) == 0
    # padded frame strides, host buffers
    hsrc = np.zeros((n, h + 3, w, 4), np.uint8)
    hsrc[:, :h] = frames
    hdst = np.zeros((n, oh + 2, ow, 4), np.uint8)
    assert engine.L.srcnn_process_batch_host(engine.ctx, hsrc.ctypes.data, n, w, h, 4 * w, (h + 3) * 4 * w, S.ORDER_RGBA,
                                             C.c_float(scale), hdst.ctypes.data, 4 * ow, (oh + 2) * 4 * ow) == 0
    assert np.array_equal(hdst[:, :oh], want)


@gpu
def test_bands_reassemble(engine):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(35)
    w, h, scale = 120, 100, 2.0
    img = _rgba(rng, h, w)
    ow, oh = S.out_dims(w, h, scale)
    whole = engine.process(img, scale, order=S.ORDER_BGRA)
    dimg = torch.from_numpy(img).to("cuda:0")
    cuts = [0, 37, 38, 121, oh]
    dev = torch.zeros((oh, ow, 4), dtype=torch.uint8, device="cuda:0")
    host = np.zeros((oh, ow, 4), np.uint8)
    for r0, r1 in zip(cuts[:-1], cuts[1:]):
        s0, s1 = S.band_src_rows(h, scale, r0, r1)
        engine.process_band_device(dimg[s0:s1].contiguous(), w, h, s0, s1, scale, r0, r1, dev[r0:r1], order=S.ORDER_BGRA)
        host[r0:r1] = engine.process_band_host(img, scale, r0, r1, order=S.ORDER_BGRA)
    engine.sync()
    assert np.array_equal(dev.cpu().numpy(), whole)
    assert np.array_equal(host, whole)


@gpu
def test_multi_engine(engine):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(36)
    w, h, scale = 100, 76, 2.0
    ow, oh = S.out_dims(w, h, scale)
    img = _rgba(rng, h, w)
    frames = np.stack([_rgba(rng, h, w) for _ in range(3)])
    whole = engine.process(img, scale, order=S.ORDER_BGRA)
    per_frame = np.stack([engine.process(f, scale, order=S.ORDER_BGRA) for f in frames])
    m = S.MultiEngine(devices=[0, 0])
    try:
        assert np.array_equal(m.process_banded(img, scale, order=S.ORDER_BGRA), whole)
        assert np.array_equal(m.process_batch(frames, scale, order=S.ORDER_BGRA), per_frame)
        plan = m.band_plan(h, scale)
        dimg = torch.from_numpy(img).to("cuda:0")
        srcs = [dimg[s0:s1].contiguous() for (r0, r1, s0, s1) in plan]
        dst = torch.zeros((oh, ow, 4), dtype=torch.uint8, device="cuda:0")
        dsts = [dst[r0:r1] for (r0, r1, s0, s1) in plan]
        torch.cuda.synchronize()
        m.process_banded_device(srcs, w, h, scale, dsts, order=S.ORDER_BGRA)
        assert np.array_equal(dst.cpu().numpy(), whole)
        df = torch.from_numpy(frames).to("cuda:0")
        dd = torch.zeros((3, oh, ow, 4), dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        m.process_batch_device([df[:2], df[2:]], scale, [dd[:2], dd[2:]], order=S.ORDER_BGRA)
        assert np.array_equal(dd.cpu().numpy(), per_frame)
    finally:
        m.close()


def _overlap(engine, on):
    engine.L.srcnn_debug_overlap.argtypes = [C.c_void_p, C.c_int]
    engine.L.srcnn_debug_overlap.restype = C.c_longlong
    return int(engine.L.srcnn_debug_overlap(engine.ctx, on))


@gpu
def test_overlap_chain_with_mixed_orders(engine):
    """BGRA, BGRA, BGR, BGRA, RGBA on one stream; call 1 reads call 0's result and call 4 reads call 3's (their top-left
    source-sized crop, strides in bytes).  Equal to the same chain fully serialised; the calls with an independent source of the
    same geometry start early (BGR after BGRA, BGRA after BGR), the ones fed by the previous result do not."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(37)
    w, h, scale = 256, 144, 2.0
    ow, oh = S.out_dims(w, h, scale)
    a0 = torch.from_numpy(_rgba(rng, h, w)).to("cuda:0")
    b2 = torch.from_numpy(natural_like(rng, h, w)).to("cuda:0")
    a3 = torch.from_numpy(_rgba(rng, h, w)).to("cuda:0")
    orders = [S.ORDER_BGRA, S.ORDER_BGRA, S.ORDER_BGR, S.ORDER_BGRA, S.ORDER_RGBA]

    def run(serial):
        outs = [torch.zeros((oh, ow, 3 if o == S.ORDER_BGR else 4), dtype=torch.uint8, device="cuda:0") for o in orders]
        srcs = [a0, None, b2, a3, None]
        counts = []
        for i, o in enumerate(orders):
            src = srcs[i] if srcs[i] is not None else outs[i - 1][:h, :w]
            engine.process_device(src, scale, outs[i], order=o)
            counts.append(_overlap(engine, -1))
            if serial:
                engine.sync()
        engine.sync()
        return outs, counts
    try:
        _overlap(engine, 0)
        ref, _ = run(True)
        _overlap(engine, 1)
        got, counts = run(False)
        for a, b in zip(ref, got):
            assert torch.equal(a, b)
        steps = [counts[i] - counts[i - 1] for i in range(1, len(counts))]
        assert steps == [0, 1, 1, 0], counts
    finally:
        _overlap(engine, 1)


@gpu
def test_fused_merge_setting_changes_nothing(engine):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(38)
    img = _rgba(rng, 64, 96)
    want = engine.process(img, 2.0, order=S.ORDER_BGRA)
    frames = np.stack([img, img[::-1].copy()])
    want_b = engine.process_batch(frames, 2.0, order=S.ORDER_BGRA)
    src = torch.from_numpy(img).to("cuda:0")
    dst = torch.zeros((128, 192, 4), dtype=torch.uint8, device="cuda:0")
    engine.process_device(src, 2.0, dst, order=S.ORDER_BGRA)   # warm: tap tables, workspace
    n0 = engine.launches
    engine.process_device(src, 2.0, dst, order=S.ORDER_BGRA)
    engine.sync()
    assert engine.launches - n0 == 3
    engine.set_fuse_merge(True)
    try:
        assert np.array_equal(engine.process(img, 2.0, order=S.ORDER_BGRA), want)
        assert np.array_equal(engine.process_batch(frames, 2.0, order=S.ORDER_BGRA), want_b)
        n0 = engine.launches
        engine.process_device(src, 2.0, dst, order=S.ORDER_BGRA)
        engine.sync()
        assert engine.launches - n0 == 3
        assert np.array_equal(dst.cpu().numpy(), want)
    finally:
        engine.set_fuse_merge(False)


def _process_srcnn():
    import srcnn_cpp_b200 as S
    fn = S.load_library()._Z12ProcessSRCNNPKhjjjfRPhRj
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.POINTER(C.c_void_p), C.POINTER(C.c_uint)]
    return fn


@gpu
@pytest.mark.parametrize("scale", [2.0, 1.5])
def test_process_srcnn_rgba(engine, scale):
    """ProcessSRCNN d = 4 is one RGBA call now; its result is the old composition: the RGB path, the alpha plane through the
    one-plane resize, interleaved."""
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(39)
    w, h = 46, 30
    img = _rgba(rng, h, w)
    out, sz = C.c_void_p(), C.c_uint()
    assert _process_srcnn()(img.ctypes.data, w, h, 4, C.c_float(scale), C.byref(out), C.byref(sz)) == 0
    ow, oh = S.out_dims(w, h, scale)
    assert sz.value == ow * oh * 4
    got = np.ctypeslib.as_array((C.c_uint8 * sz.value).from_address(out.value)).reshape(oh, ow, 4).copy()
    want = np.concatenate([engine.process(np.ascontiguousarray(img[..., :3]), scale, order=S.ORDER_RGB),
                           engine.resize_plane(img[..., 3], scale)[..., None]], axis=2)
    assert np.array_equal(got, want)


@gpu
def test_argument_checks(engine):
    import torch
    import srcnn_cpp_b200 as S
    L, ctx = engine.L, engine.ctx
    p = lambda t: C.c_void_p(t.data_ptr())
    src = torch.zeros((20, 32, 4), dtype=torch.uint8, device="cuda:0")
    dst = torch.zeros((40, 64, 4), dtype=torch.uint8, device="cuda:0")
    y = torch.zeros((40, 64), dtype=torch.uint8, device="cuda:0")
    for order in (S.ORDER_BGRA, S.ORDER_RGBA):
        assert L.srcnn_process_device(ctx, p(src), 32, 20, 127, order, C.c_float(2.0), p(dst), 256) == S.E_ARG
        assert L.srcnn_process_device(ctx, p(src), 32, 20, 96, order, C.c_float(2.0), p(dst), 256) == S.E_ARG
        assert L.srcnn_process_device(ctx, p(src), 32, 20, 128, order, C.c_float(2.0), p(dst), 255) == S.E_ARG
        assert L.srcnn_process_device(ctx, p(src), 32, 20, 128, order, C.c_float(2.0), p(dst), 192) == S.E_ARG
        assert L.srcnn_stage_color_bicubic_device(ctx, p(src), 32, 20, 128, order, C.c_float(2.0), p(y), p(y), p(y), 64) == S.E_ARG
        assert L.srcnn_stage_merge_device(ctx, p(y), p(y), p(y), 64, 40, 64, order, p(dst), 256) == S.E_ARG
    assert L.srcnn_process_device(ctx, p(src), 32, 20, 128, 5, C.c_float(2.0), p(dst), 256) == S.E_ARG
    assert L.srcnn_process_device(ctx, p(src), 32, 20, 128, S.ORDER_BGRA, C.c_float(2.0), p(dst), 256) == 0
    engine.sync()


@gpu
def test_full_size_1080p_to_4k(engine):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(40)
    w, h, scale = 1920, 1080, 2.0
    ow, oh = S.out_dims(w, h, scale)
    img = torch.from_numpy(_rgba(rng, h, w)).to("cuda:0")
    out = torch.zeros((oh, ow, 4), dtype=torch.uint8, device="cuda:0")
    bgr = torch.zeros((oh, ow, 3), dtype=torch.uint8, device="cuda:0")
    alpha = torch.zeros((oh, ow), dtype=torch.uint8, device="cuda:0")
    engine.process_device(img, scale, out, order=S.ORDER_BGRA)
    engine.process_device(img[..., :3].contiguous(), scale, bgr, order=S.ORDER_BGR)
    engine.stage_resize_plane(img[..., 3].contiguous(), scale, alpha)
    engine.sync()
    assert torch.equal(out[..., :3], bgr)
    assert torch.equal(out[..., 3], alpha)
