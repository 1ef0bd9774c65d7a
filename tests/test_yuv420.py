"""The 4:2:0 video path (SRCNN_ORDER_NV12 / SRCNN_ORDER_I420): packed video frames end to end on the device.

No new parity contract: the output's Y plane is the SRCNN_ORDER_GRAY call on the source's Y plane (so the FP32 variant equals
oracle.cnn(oracle.resize_cubic(Y)) exactly), and each chroma plane is oracle.resize_cubic(plane, ow/2, oh/2) -- the one-plane
stage srcnn_stage_resize_plane_device -- with no CNN and no colour matrix."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import natural_like

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
ORDERS = ["nv12", "i420"]


def _order(S, name):
    return S.ORDER_NV12 if name == "nv12" else S.ORDER_I420


def _planes(rng, h, w):
    """a Y plane of natural-looking content and two smooth-ish chroma planes"""
    img = natural_like(rng, h, w)
    y = np.ascontiguousarray(img[:, :, 1])
    u = np.ascontiguousarray(img[::2, ::2, 0])
    v = np.ascontiguousarray(img[1::2, 1::2, 2])
    return y, u, v


def _pack(S, order, y, u, v, stride=None):
    """one (h*3/2) x stride frame holding y, u, v in the layout of `order` (columns past w are padding)"""
    h, w = y.shape
    stride = stride or w
    f = np.full((h * 3 // 2, stride), 213, np.uint8)
    fy, fu, fv = S.yuv420_planes(f, order)
    fy[:, :w] = y
    fu[:, :w // 2] = u
    fv[:, :w // 2] = v
    return f


def _split(S, order, frame, w):
    """(Y, U, V) numpy copies of a frame whose rows may be padded past w"""
    y, u, v = S.yuv420_planes(frame, order)
    return np.array(y[:, :w]), np.array(u[:, :w // 2]), np.array(v[:, :w // 2])


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

def test_enum_values_match_header():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"SRCNN_ORDER_NV12\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_NV12 == 6
    assert int(re.search(r"SRCNN_ORDER_I420\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_I420 == 7


def test_abi_version_unchanged():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"#define SRCNN_B200_ABI_VERSION (\d+)", hdr).group(1)) == 2
    assert S.load_library().srcnn_abi_version() == 2


@pytest.mark.parametrize("name", ORDERS)
def test_python_shape_checks(name):
    """Rejected before any library call: a row count that is not a multiple of 3, a wrong dtype, a wrong rank."""
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    eng = object.__new__(S.Engine)   # the checks run before the context is touched
    for bad, call in [(np.zeros((10, 8), np.uint8), eng.process), (np.zeros((12, 8), np.uint16), eng.process),
                      (np.zeros((12, 8, 3), np.uint8), eng.process), (np.zeros((2, 10, 8), np.uint8), eng.process_batch),
                      (np.zeros((12, 8), np.uint8), eng.process_batch)]:
        with pytest.raises(S.SrcnnError) as e:
            call(bad, 2.0, order=order)
        assert e.value.status == S.E_ARG
    with pytest.raises(S.SrcnnError):
        S.yuv420_planes(np.zeros((10, 8), np.uint8), order)


def test_yuv420_planes_views():
    import torch
    import srcnn_cpp_b200 as S
    h, w, stride = 6, 8, 12
    f = np.arange(h * 3 // 2 * stride, dtype=np.uint8).reshape(h * 3 // 2, stride)
    flat = f.reshape(-1)
    y, u, v = S.yuv420_planes(f[:, :w], S.ORDER_NV12)
    assert y.shape == (h, w) and u.shape == v.shape == (h // 2, w // 2)
    assert np.array_equal(u[1], flat[(h + 1) * stride:(h + 1) * stride + w:2]) and np.array_equal(v[1], flat[(h + 1) * stride + 1:(h + 1) * stride + w:2])
    y, u, v = S.yuv420_planes(f, S.ORDER_I420)
    assert u.shape == v.shape == (h // 2, stride // 2)
    assert np.array_equal(u[1, :w // 2], flat[h * stride + stride // 2:][:w // 2])
    assert np.array_equal(v[0, :w // 2], flat[h * stride + (h // 2) * (stride // 2):][:w // 2])
    u[0, 0] = 1   # views, not copies
    assert flat[h * stride] == 1
    ty, tu, tv = S.yuv420_planes(torch.from_numpy(f), S.ORDER_I420)
    assert np.array_equal(tu.numpy(), u) and np.array_equal(tv.numpy(), v) and np.array_equal(ty.numpy(), f[:h])


# ---- on the GPU ------------------------------------------------------------------------------------------------------------

def _dev(t):
    import torch
    return torch.from_numpy(np.ascontiguousarray(t)).to("cuda:0")


def _chroma_want(engine, oracle, plane, ow, oh, scale):
    want = oracle.resize_cubic(plane, ow // 2, oh // 2)
    import torch
    got = torch.zeros((oh // 2, ow // 2), dtype=torch.uint8, device="cuda:0")
    engine.stage_resize_plane(_dev(plane), scale, got)
    engine.sync()
    assert np.array_equal(got.cpu().numpy(), want)
    return want


# x2 / x4 with ow/2 % 8 == 0 (one launch), x2 with ow/2 % 8 != 0, x1.5, x3 (odd chroma rows: the direct chroma kernel), 2x2, x0.5
GEOS = [(128, 64, 2.0), (104, 40, 2.0), (64, 48, 4.0), (100, 40, 2.0), (384, 384, 1.5), (1280, 720, 1.5), (54, 38, 3.0), (2, 2, 2.0),
        (96, 64, 0.5)]


@gpu
@pytest.mark.parametrize("w,h,scale", GEOS)
def test_parity_across_geometries(engine, oracle, w, h, scale):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(w * 3 + h)
    y, u, v = _planes(rng, h, w)
    ow, oh = S.out_dims(w, h, scale)
    want_y = oracle.cnn(oracle.resize_cubic(y, ow, oh))
    want_u = _chroma_want(engine, oracle, u, ow, oh, scale)
    want_v = _chroma_want(engine, oracle, v, ow, oh, scale)
    try:
        for variant in (S.VARIANT_FP32, S.VARIANT_TC):
            engine.set_variant(variant)
            grey = engine.process(y, scale, order=S.ORDER_GRAY)
            for name in ORDERS:
                order = _order(S, name)
                frame = _pack(S, order, y, u, v)
                host = engine.process(frame, scale, order=order)
                dev = torch.zeros((oh * 3 // 2, ow), dtype=torch.uint8, device="cuda:0")
                engine.process_device(_dev(frame), scale, dev, order=order)
                engine.sync()
                assert host.shape == (oh * 3 // 2, ow)
                assert np.array_equal(dev.cpu().numpy(), host), (name, variant)
                gy, gu, gv = _split(S, order, host, ow)
                assert np.array_equal(gy, grey), (name, variant)
                assert np.array_equal(gu, want_u) and np.array_equal(gv, want_v), (name, variant)
                if variant == S.VARIANT_FP32:
                    assert np.array_equal(gy, want_y), name
                else:
                    d = np.abs(gy.astype(np.int16) - want_y.astype(np.int16))
                    assert d.max() <= 2 and (d <= 1).mean() >= 0.999, (name, int(d.max()))
    finally:
        engine.set_variant(S.VARIANT_TC)


def _written_mask(order, oh, ow, ds, nbytes, ofs):
    """bytes of a dst buffer (frame at byte `ofs`, rows `ds` apart) that a call may write"""
    m = np.zeros(nbytes, bool)
    for r in range(oh):
        m[ofs + r * ds:ofs + r * ds + ow] = True
    base = ofs + oh * ds
    if order == 6:   # NV12
        for r in range(oh // 2):
            m[base + r * ds:base + r * ds + ow] = True
    else:
        for r in range(oh):   # U rows, then V rows, ds/2 apart
            m[base + r * (ds // 2):base + r * (ds // 2) + ow // 2] = True
    return m


# (w, h, scale, src stride pad, src byte offset, dst stride pad, dst byte offset): tight / padded strides on the one-launch path,
# odd offsets that force the generic kernels, an I420 dst stride that is a multiple of 8 but not 16, the fallback scales
STRIDES = [(128, 64, 2.0, 6, 0, 10, 0), (128, 64, 2.0, 0, 1, 0, 3), (128, 64, 2.0, 2, 3, 8, 0), (64, 32, 4.0, 4, 0, 24, 16),
           (128, 64, 2.0, 0, 0, 8, 0), (100, 60, 1.5, 6, 5, 2, 1), (96, 40, 3.0, 2, 0, 14, 7)]


@gpu
@pytest.mark.parametrize("name", ORDERS)
@pytest.mark.parametrize("w,h,scale,spad,sofs,dpad,dofs", STRIDES)
def test_strides_alignment_and_sentinels(engine, name, w, h, scale, spad, sofs, dpad, dofs):
    import torch
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    rng = np.random.default_rng(w + h + spad + dofs)
    y, u, v = _planes(rng, h, w)
    ow, oh = S.out_dims(w, h, scale)
    want = engine.process(_pack(S, order, y, u, v), scale, order=order)
    ss, ds = w + spad, ow + dpad
    sframe = _pack(S, order, y, u, v, stride=ss).reshape(-1)
    sbuf = torch.full((sframe.size + sofs + 64,), 5, dtype=torch.uint8, device="cuda:0")
    sbuf[sofs:sofs + sframe.size] = _dev(sframe)
    nbytes = (oh * 3 // 2) * ds + dofs + 64
    dbuf = torch.full((nbytes,), 77, dtype=torch.uint8, device="cuda:0")
    src = sbuf[sofs:sofs + sframe.size].view(h * 3 // 2, ss)[:, :w]
    dst = dbuf[dofs:dofs + (oh * 3 // 2) * ds].view(oh * 3 // 2, ds)[:, :ow]
    engine.process_device(src, scale, dst, order=order)
    engine.sync()
    full = dbuf.cpu().numpy()
    got = full[dofs:dofs + (oh * 3 // 2) * ds].reshape(oh * 3 // 2, ds)
    for a, b in zip(_split(S, order, got, ow), _split(S, order, want, ow)):
        assert np.array_equal(a, b)
    assert (full[~_written_mask(order, oh, ow, ds, nbytes, dofs)] == 77).all()


@gpu
@pytest.mark.parametrize("name", ORDERS)
@pytest.mark.parametrize("scale", [2.0, 1.5])
def test_batches(engine, name, scale):
    """Device and host batches, tight and padded frame strides, against frame-by-frame calls; a repeated host call on the same
    pinned buffers (replayed as a CUDA graph) equals the first."""
    import torch
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    rng = np.random.default_rng(31)
    n, w, h = 5, 128, 72
    ow, oh = S.out_dims(w, h, scale)
    frames = np.stack([_pack(S, order, *_planes(rng, h, w)) for _ in range(n)])
    single = np.stack([engine.process(f, scale, order=order) for f in frames])
    for pad in (0, 96):
        fr = h * 3 // 2 * w + pad
        sbuf = torch.zeros((n * fr,), dtype=torch.uint8, device="cuda:0")
        for i in range(n):
            sbuf[i * fr:i * fr + frames[i].size] = _dev(frames[i].reshape(-1))
        ofr = oh * 3 // 2 * ow + pad
        dbuf = torch.full((n * ofr,), 77, dtype=torch.uint8, device="cuda:0")
        src = sbuf.as_strided((n, h * 3 // 2, w), (fr, w, 1))
        dst = dbuf.as_strided((n, oh * 3 // 2, ow), (ofr, ow, 1))
        n0 = engine.launches
        engine.process_batch_device(src, scale, dst, order=order)
        engine.sync()
        if scale == 2.0:
            assert engine.launches - n0 == 2    # one chunk: one resize launch, one CNN launch
        assert np.array_equal(dst.cpu().numpy(), single), pad
        if pad:
            assert int(dbuf.view(n, ofr)[:, oh * 3 // 2 * ow:].ne(77).sum()) == 0
    assert np.array_equal(engine.process_batch(frames, scale, order=order), single)
    pin_in = S.PinnedBuffer(frames.nbytes)
    pin_out = S.PinnedBuffer(single.nbytes)
    try:
        pin_in.array[:] = frames.reshape(-1)
        src = pin_in.array.reshape(frames.shape)
        out = pin_out.array.reshape(single.shape)
        for _ in range(3):   # live, captured, replayed
            out[...] = 0
            engine.process_batch(src, scale, order=order, out=out)
            assert np.array_equal(out, single)
    finally:
        pin_in.free()
        pin_out.free()


@gpu
@pytest.mark.parametrize("name", ORDERS)
def test_tall_single_host_frame_in_sub_bands(engine, name):
    """A single host frame tall enough to be cut into several sub-bands equals the device call."""
    import torch
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    rng = np.random.default_rng(41)
    w, h, scale = 256, 1536, 2.0
    ow, oh = S.out_dims(w, h, scale)
    frame = _pack(S, order, *_planes(rng, h, w))
    dev = torch.zeros((oh * 3 // 2, ow), dtype=torch.uint8, device="cuda:0")
    engine.process_device(_dev(frame), scale, dev, order=order)
    engine.sync()
    for bands in (8, 3):
        engine.set_host_bands(bands)
        try:
            assert np.array_equal(engine.process(frame, scale, order=order), dev.cpu().numpy()), bands
        finally:
            engine.set_host_bands(8)


@gpu
@pytest.mark.parametrize("name", ORDERS)
def test_multi_engine_batches(engine, name):
    import torch
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    rng = np.random.default_rng(51)
    n, w, h, scale = 5, 96, 64, 2.0
    ow, oh = S.out_dims(w, h, scale)
    frames = np.stack([_pack(S, order, *_planes(rng, h, w)) for _ in range(n)])
    single = engine.process_batch(frames, scale, order=order)
    m = S.MultiEngine(devices=[0, 0])
    try:
        assert np.array_equal(m.process_batch(frames, scale, order=order), single)
        srcs = [_dev(frames[0::2]), _dev(frames[1::2])]
        dsts = [torch.zeros((s.shape[0], oh * 3 // 2, ow), dtype=torch.uint8, device="cuda:0") for s in srcs]
        m.process_batch_device(srcs, scale, dsts, order=order)
        torch.cuda.synchronize()
        assert np.array_equal(dsts[0].cpu().numpy(), single[0::2]) and np.array_equal(dsts[1].cpu().numpy(), single[1::2])
    finally:
        m.close()


@gpu
def test_launch_count(engine):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(61)
    for name in ORDERS:
        order = _order(S, name)
        for (w, h, scale, most) in [(128, 64, 2.0, 2), (64, 48, 4.0, 2), (100, 40, 2.0, 3), (384, 384, 1.5, 3), (54, 38, 3.0, 3)]:
            ow, oh = S.out_dims(w, h, scale)
            src = _dev(_pack(S, order, *_planes(rng, h, w)))
            dst = torch.zeros((oh * 3 // 2, ow), dtype=torch.uint8, device="cuda:0")
            n0 = engine.launches
            engine.process_device(src, scale, dst, order=order)
            engine.sync()
            if most == 2:
                assert engine.launches - n0 == 2, (name, w, h, scale)
            else:
                assert engine.launches - n0 <= 3, (name, w, h, scale)


def _overlap(engine, on):
    engine.L.srcnn_debug_overlap.argtypes = [C.c_void_p, C.c_int]
    engine.L.srcnn_debug_overlap.restype = C.c_longlong
    return int(engine.L.srcnn_debug_overlap(engine.ctx, on))


@gpu
def test_overlap_chain_and_stale_workspace(engine):
    """BGR -> NV12 -> BGR -> I420 on one stream equals the calls one by one; no colour call after a 4:2:0 call starts early.  A
    context whose workspace was last carved by a larger BGR call gives the same 4:2:0 results."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(71)
    w, h, scale = 256, 128, 2.0
    ow, oh = S.out_dims(w, h, scale)
    bgr = [_dev(natural_like(rng, h, w)) for _ in range(2)]
    nv12 = _dev(_pack(S, S.ORDER_NV12, *_planes(rng, h, w)))
    i420 = _dev(_pack(S, S.ORDER_I420, *_planes(rng, h, w)))
    calls = [(bgr[0], S.ORDER_BGR, (oh, ow, 3)), (nv12, S.ORDER_NV12, (oh * 3 // 2, ow)), (bgr[1], S.ORDER_BGR, (oh, ow, 3)),
             (i420, S.ORDER_I420, (oh * 3 // 2, ow))]
    want = []
    for src, order, shape in calls:
        out = torch.zeros(shape, dtype=torch.uint8, device="cuda:0")
        engine.process_device(src, scale, out, order=order)
        engine.sync()
        want.append(out.cpu().numpy())
    _overlap(engine, 1)
    outs = [torch.zeros(shape, dtype=torch.uint8, device="cuda:0") for _, _, shape in calls]
    engine.process_device(calls[0][0], scale, outs[0], order=calls[0][1])
    e0 = _overlap(engine, -1)
    for (src, order, _), out in zip(calls[1:], outs[1:]):
        engine.process_device(src, scale, out, order=order)
    engine.sync()
    assert _overlap(engine, -1) == e0   # neither the BGR call after NV12 nor the 4:2:0 calls started early
    for got, w_ in zip(outs, want):
        assert np.array_equal(got.cpu().numpy(), w_)
    big = torch.zeros((oh * 2, ow * 2, 3), dtype=torch.uint8, device="cuda:0")
    engine.process_device(_dev(natural_like(rng, h * 2, w * 2)), scale, big, order=S.ORDER_BGR)
    for (src, order, shape), w_ in [(calls[1], want[1]), (calls[3], want[3])]:
        out = torch.zeros(shape, dtype=torch.uint8, device="cuda:0")
        engine.process_device(src, scale, out, order=order)
        engine.sync()
        assert np.array_equal(out.cpu().numpy(), w_)


@gpu
@pytest.mark.parametrize("name", ORDERS)
def test_rejections(engine, name):
    import torch
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    L, ctx = engine.L, engine.ctx
    buf = torch.zeros((1 << 20,), dtype=torch.uint8, device="cuda:0")
    p = C.c_void_p(buf.data_ptr())
    f = C.c_float
    dev = lambda w, h, ss, sc, ds: L.srcnn_process_device(ctx, p, w, h, ss, order, f(sc), p, ds)
    assert dev(64, 32, 64, 2.0, 128) == S.OK
    engine.sync()
    assert dev(63, 32, 64, 2.0, 128) == S.E_ARG                 # odd width
    assert dev(64, 31, 64, 2.0, 128) == S.E_ARG                 # odd height
    assert dev(10, 10, 10, 1.5, 16) == S.E_ARG                  # 15 x 15 output
    assert dev(64, 32, 63, 2.0, 128) == S.E_ARG                 # short source stride
    assert dev(64, 32, 64, 2.0, 127) == S.E_ARG                 # short destination stride
    if order == S.ORDER_I420:
        assert dev(64, 32, 65, 2.0, 128) == S.E_ARG             # odd I420 strides
        assert dev(64, 32, 64, 2.0, 129) == S.E_ARG
    err = (L.srcnn_last_error(ctx) or b"").decode()
    assert "even" in err or "stride" in err
    # batch frame strides below 3/2 frames
    assert L.srcnn_process_batch_device(ctx, p, 2, 64, 32, 64, 64 * 32, order, f(2.0), p, 128, 128 * 96) == S.E_ARG
    assert L.srcnn_process_batch_device(ctx, p, 2, 64, 32, 64, 64 * 48, order, f(2.0), p, 128, 128 * 64) == S.E_ARG
    host = np.zeros(1 << 16, np.uint8)
    assert L.srcnn_process_batch_host(ctx, host.ctypes.data, 2, 64, 32, 64, 64 * 32, order, f(2.0), host.ctypes.data, 128,
                                      128 * 96) == S.E_ARG
    # the band calls, the colour and merge stage calls
    assert L.srcnn_process_band_device(ctx, p, 64, 32, 64, 0, 32, order, f(2.0), 0, 64, p, 128) == S.E_ARG
    assert L.srcnn_process_band_host(ctx, host.ctypes.data, 64, 32, 64, order, f(2.0), 0, 64, host.ctypes.data, 128) == S.E_ARG
    assert L.srcnn_stage_color_bicubic_device(ctx, p, 64, 32, 192, order, f(2.0), p, p, p, 128) == S.E_ARG
    assert L.srcnn_stage_merge_device(ctx, p, p, p, 64, 32, 64, order, p, 192) == S.E_ARG
    m = S.MultiEngine(devices=[0])
    try:
        frame = np.zeros((48, 64), np.uint8)
        with pytest.raises(S.SrcnnError) as e:
            m.process_banded(frame, 2.0, order=order)
        assert e.value.status == S.E_ARG
    finally:
        m.close()


@gpu
def test_full_size_1080p_nv12_to_4k(engine, oracle):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(81)
    w, h, scale = 1920, 1080, 2.0
    ow, oh = S.out_dims(w, h, scale)
    y, u, v = _planes(rng, h, w)
    out = torch.zeros((oh * 3 // 2, ow), dtype=torch.uint8, device="cuda:0")
    n0 = engine.launches
    engine.process_device(_dev(_pack(S, S.ORDER_NV12, y, u, v)), scale, out, order=S.ORDER_NV12)
    engine.sync()
    assert engine.launches - n0 == 2
    gy, gu, gv = _split(S, S.ORDER_NV12, out.cpu().numpy(), ow)
    assert np.array_equal(gu, oracle.resize_cubic(u, ow // 2, oh // 2))
    assert np.array_equal(gv, oracle.resize_cubic(v, ow // 2, oh // 2))
    d = np.abs(gy.astype(np.int16) - oracle.cnn(oracle.resize_cubic(y, ow, oh)).astype(np.int16))
    assert d.max() <= 2 and (d <= 1).mean() >= 0.999, int(d.max())
