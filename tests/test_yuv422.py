"""The packed 4:2:2 path (SRCNN_ORDER_YUY2 / SRCNN_ORDER_UYVY): capture frames end to end on the device.

No new parity contract: the output's Y plane is the SRCNN_ORDER_GRAY call on the source's Y plane (so the FP32 variant equals
oracle.cnn(oracle.resize_cubic(Y)) exactly), and each chroma plane is oracle.resize_cubic(plane, ow/2, oh) -- the one-plane stage
srcnn_stage_resize_plane_device -- with no CNN and no colour matrix.  Unlike 4:2:0, every band call takes these orders."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import natural_like

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
ORDERS = ["yuy2", "uyvy"]


def _order(S, name):
    return S.ORDER_YUY2 if name == "yuy2" else S.ORDER_UYVY


def _planes(rng, h, w):
    """a Y plane of natural-looking content and two smooth-ish h x w/2 chroma planes"""
    img = natural_like(rng, h, w)
    y = np.ascontiguousarray(img[:, :, 1])
    u = np.ascontiguousarray(img[:, ::2, 0])
    v = np.ascontiguousarray(img[:, 1::2, 2])
    return y, u, v


def _pack(S, order, y, u, v, stride=None):
    """an h x stride byte buffer whose first 2*w bytes per row are the frame of `order` (the rest is padding); returns (buffer,
    h x w x 2 view of the frame)"""
    h, w = y.shape
    stride = stride or 2 * w
    buf = np.full((h, stride), 213, np.uint8)
    frame = buf[:, :2 * w].reshape(h, w, 2)
    fy, fu, fv = S.yuv422_planes(frame, order)
    fy[...] = y
    fu[...] = u
    fv[...] = v
    return buf, frame


def _frame(S, order, y, u, v):
    return np.ascontiguousarray(_pack(S, order, y, u, v)[1])


def _split(S, order, frame):
    """(Y, U, V) numpy copies of an h x w x 2 frame"""
    return tuple(np.array(p) for p in S.yuv422_planes(frame, order))


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

def test_enum_values_match_header():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"SRCNN_ORDER_YUY2\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_YUY2 == 8
    assert int(re.search(r"SRCNN_ORDER_UYVY\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_UYVY == 9


def test_abi_version_unchanged():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"#define SRCNN_B200_ABI_VERSION (\d+)", hdr).group(1)) == 2
    assert S.load_library().srcnn_abi_version() == 2


@pytest.mark.parametrize("name", ORDERS)
def test_python_shape_checks(name):
    """Rejected before any library call: a wrong rank, a wrong last dimension, a wrong dtype."""
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    eng = object.__new__(S.Engine)   # the checks run before the context is touched
    for bad, call in [(np.zeros((8, 8), np.uint8), eng.process), (np.zeros((8, 8, 3), np.uint8), eng.process),
                      (np.zeros((8, 8, 2), np.uint16), eng.process), (np.zeros((8, 8, 2), np.uint8), eng.process_batch),
                      (np.zeros((2, 8, 8, 4), np.uint8), eng.process_batch), (np.zeros((8, 8, 4), np.uint8), eng.process_band_host)]:
        with pytest.raises(S.SrcnnError) as e:
            if call == eng.process_band_host:
                call(bad, 2.0, 0, 4, order=order)
            else:
                call(bad, 2.0, order=order)
        assert e.value.status == S.E_ARG
    for bad in (np.zeros((8, 8), np.uint8), np.zeros((8, 7, 2), np.uint8), np.zeros((8, 8, 3), np.uint8)):
        with pytest.raises(S.SrcnnError):
            S.yuv422_planes(bad, order)
    with pytest.raises(S.SrcnnError):
        S.yuv422_planes(np.zeros((8, 8, 2), np.uint8), S.ORDER_NV12)


def test_yuv422_planes_views():
    import torch
    import srcnn_cpp_b200 as S
    h, w, stride = 3, 8, 20
    buf = np.arange(h * stride, dtype=np.uint8).reshape(h, stride)
    frame = buf[:, :2 * w].reshape(h, w, 2)
    row = buf[1]
    y, u, v = S.yuv422_planes(frame, S.ORDER_YUY2)
    assert y.shape == (h, w) and u.shape == v.shape == (h, w // 2)
    assert np.array_equal(y[1], row[0:2 * w:2]) and np.array_equal(u[1], row[1:2 * w:4]) and np.array_equal(v[1], row[3:2 * w:4])
    y, u, v = S.yuv422_planes(frame, S.ORDER_UYVY)
    assert np.array_equal(y[1], row[1:2 * w:2]) and np.array_equal(u[1], row[0:2 * w:4]) and np.array_equal(v[1], row[2:2 * w:4])
    y[2, 3] = 1   # views, not copies
    u[0, 1] = 2
    v[1, 0] = 3
    assert buf[2, 7] == 1 and buf[0, 4] == 2 and buf[1, 2] == 3
    t = torch.from_numpy(buf)[:, :2 * w].reshape(h, w, 2)
    for order in (S.ORDER_YUY2, S.ORDER_UYVY):
        for a, b in zip(S.yuv422_planes(t, order), S.yuv422_planes(frame, order)):
            assert np.array_equal(a.numpy(), b)
    ty, tu, tv = S.yuv422_planes(t, S.ORDER_YUY2)
    tu[2, 3] = 9
    assert buf[2, 13] == 9


# ---- on the GPU ------------------------------------------------------------------------------------------------------------

def _dev(t):
    import torch
    return torch.from_numpy(np.ascontiguousarray(t)).to("cuda:0")


def _chroma_want(engine, oracle, plane, ow, oh, scale):
    want = oracle.resize_cubic(plane, ow // 2, oh)
    import torch
    got = torch.zeros((oh, ow // 2), dtype=torch.uint8, device="cuda:0")
    engine.stage_resize_plane(_dev(plane), scale, got)
    engine.sync()
    assert np.array_equal(got.cpu().numpy(), want)
    return want


def _engine_with(env):
    """a second context created with `env` set, on the test's torch stream"""
    import torch
    import srcnn_cpp_b200 as S
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        eng = S.Engine(device=0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    return eng


# x2 / x4 with ow % 16 == 0 (one launch), x2 with ow/2 % 8 != 0, x1.5, x3, x0.5 (the direct kernels), odd heights, a 2x1 frame
FAST = [(128, 64, 2.0), (64, 48, 4.0), (128, 63, 2.0)]
GEOS = FAST + [(100, 40, 2.0), (108, 40, 2.0), (384, 384, 1.5), (1280, 720, 1.5), (54, 38, 3.0), (96, 33, 3.0), (96, 64, 0.5),
               (2, 1, 2.0)]


def _check_parity(engine, oracle, w, h, scale):
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
                frame = _frame(S, order, y, u, v)
                host = engine.process(frame, scale, order=order)
                dev = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
                engine.process_device(_dev(frame), scale, dev, order=order)
                engine.sync()
                assert host.shape == (oh, ow, 2)
                assert np.array_equal(dev.cpu().numpy(), host), (name, variant)
                gy, gu, gv = _split(S, order, host)
                assert np.array_equal(gy, grey), (name, variant)
                assert np.array_equal(gu, want_u) and np.array_equal(gv, want_v), (name, variant)
                if variant == S.VARIANT_FP32:
                    assert np.array_equal(gy, want_y), name
                else:
                    d = np.abs(gy.astype(np.int16) - want_y.astype(np.int16))
                    assert d.max() <= 2 and (d <= 1).mean() >= 0.999, (name, int(d.max()))
    finally:
        engine.set_variant(S.VARIANT_TC)


@gpu
@pytest.mark.parametrize("w,h,scale", GEOS)
def test_parity_across_geometries(engine, oracle, w, h, scale):
    _check_parity(engine, oracle, w, h, scale)


@gpu
@pytest.mark.parametrize("w,h,scale", FAST)
def test_parity_generic_kernels(oracle, w, h, scale):
    """The one-launch geometries again on a context that never takes the integer-scale kernels (SRCNN_KA_INT=0)."""
    eng = _engine_with({"SRCNN_KA_INT": "0"})
    try:
        _check_parity(eng, oracle, w, h, scale)
    finally:
        eng.close()


def _written_mask(oh, ow, ds, nbytes, ofs):
    """bytes of a dst buffer (frame at byte `ofs`, rows `ds` apart) that a call may write"""
    m = np.zeros(nbytes, bool)
    for r in range(oh):
        m[ofs + r * ds:ofs + r * ds + 2 * ow] = True
    return m


# (w, h, scale, src stride pad, src byte offset, dst stride pad, dst byte offset): padded strides on the one-launch path (8-byte and
# 4-byte aligned sources, a 16-byte aligned destination and one the 128-bit stores cannot take), unaligned pointers, the generic
# and direct kernels
STRIDES = [(128, 64, 2.0, 8, 0, 16, 0), (128, 64, 2.0, 4, 0, 4, 0), (128, 64, 2.0, 0, 1, 0, 3), (128, 64, 2.0, 2, 3, 6, 2),
           (64, 32, 4.0, 4, 0, 32, 16), (100, 60, 1.5, 6, 5, 2, 1), (96, 40, 3.0, 2, 0, 14, 7), (96, 64, 0.5, 2, 1, 2, 1)]


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
    want = engine.process(_frame(S, order, y, u, v), scale, order=order)
    ss, ds = 2 * w + spad, 2 * ow + dpad
    sbytes = _pack(S, order, y, u, v, stride=ss)[0].reshape(-1)
    sbuf = torch.full((sbytes.size + sofs + 64,), 5, dtype=torch.uint8, device="cuda:0")
    sbuf[sofs:sofs + sbytes.size] = _dev(sbytes)
    nbytes = oh * ds + dofs + 64
    dbuf = torch.full((nbytes,), 77, dtype=torch.uint8, device="cuda:0")
    src = sbuf[sofs:sofs + sbytes.size].view(h, ss)[:, :2 * w].view(h, w, 2)
    dst = dbuf[dofs:dofs + oh * ds].view(oh, ds)[:, :2 * ow].view(oh, ow, 2)
    engine.process_device(src, scale, dst, order=order)
    engine.sync()
    full = dbuf.cpu().numpy()
    assert np.array_equal(dst.cpu().numpy(), want)
    assert (full[~_written_mask(oh, ow, ds, nbytes, dofs)] == 77).all()


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
    frames = np.stack([_frame(S, order, *_planes(rng, h, w)) for _ in range(n)])
    single = np.stack([engine.process(f, scale, order=order) for f in frames])
    for pad in (0, 96):
        fr = h * w * 2 + pad
        sbuf = torch.zeros((n * fr,), dtype=torch.uint8, device="cuda:0")
        for i in range(n):
            sbuf[i * fr:i * fr + frames[i].size] = _dev(frames[i].reshape(-1))
        ofr = oh * ow * 2 + pad
        dbuf = torch.full((n * ofr,), 77, dtype=torch.uint8, device="cuda:0")
        src = sbuf.as_strided((n, h, w, 2), (fr, 2 * w, 2, 1))
        dst = dbuf.as_strided((n, oh, ow, 2), (ofr, 2 * ow, 2, 1))
        n0 = engine.launches
        engine.process_batch_device(src, scale, dst, order=order)
        engine.sync()
        if scale == 2.0:   # one chunk: one resize launch, one CNN launch, one pack launch (or one per frame for padded frames)
            assert engine.launches - n0 == (3 if pad == 0 else 2 + n)
        assert np.array_equal(dst.cpu().numpy(), single), pad
        if pad:
            assert int(dbuf.view(n, ofr)[:, oh * ow * 2:].ne(77).sum()) == 0
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
    frame = _frame(S, order, *_planes(rng, h, w))
    dev = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
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
@pytest.mark.parametrize("w,h,scale", [(256, 96, 2.0), (200, 75, 1.5), (64, 40, 4.0)])
def test_bands_union_is_the_whole_frame(engine, name, w, h, scale):
    """process_band_device / process_band_host over several cuts: the union equals the whole-frame call bit for bit (the halo is
    the luma one; chroma needs no more)."""
    import torch
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    rng = np.random.default_rng(w + h)
    ow, oh = S.out_dims(w, h, scale)
    frame = _frame(S, order, *_planes(rng, h, w))
    whole = engine.process(frame, scale, order=order)
    dsrc = _dev(frame)
    for cuts in ([0, oh], [0, 7, oh], [0, oh // 3, oh // 3 + 1, 2 * oh // 3, oh]):
        dev = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
        host = np.zeros((oh, ow, 2), np.uint8)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            s0, s1 = S.band_src_rows(h, scale, r0, r1)
            engine.process_band_device(dsrc[s0:s1], w, h, s0, s1, scale, r0, r1, dev[r0:r1], order=order)
            host[r0:r1] = engine.process_band_host(frame, scale, r0, r1, order=order)
        engine.sync()
        assert np.array_equal(dev.cpu().numpy(), whole), cuts
        assert np.array_equal(host, whole), cuts


@gpu
@pytest.mark.parametrize("name", ORDERS)
def test_multi_engine(engine, name):
    """MultiEngine banded and batch calls, host and device buffers, equal the one-context result."""
    import torch
    import srcnn_cpp_b200 as S
    order = _order(S, name)
    rng = np.random.default_rng(51)
    n, w, h, scale = 5, 96, 64, 2.0
    ow, oh = S.out_dims(w, h, scale)
    frames = np.stack([_frame(S, order, *_planes(rng, h, w)) for _ in range(n)])
    single = engine.process_batch(frames, scale, order=order)
    big = _frame(S, order, *_planes(rng, 150, 128))
    bw, bh = 128, 150
    bow, boh = S.out_dims(bw, bh, scale)
    whole = engine.process(big, scale, order=order)
    m = S.MultiEngine(devices=[0, 0, 0])
    try:
        torch.cuda.synchronize()   # the workers' streams are not ordered against the tensors made on the test's stream
        assert np.array_equal(m.process_batch(frames, scale, order=order), single)
        srcs = [_dev(frames[0::3]), _dev(frames[1::3]), _dev(frames[2::3])]
        dsts = [torch.zeros((s.shape[0], oh, ow, 2), dtype=torch.uint8, device="cuda:0") for s in srcs]
        torch.cuda.synchronize()
        m.process_batch_device(srcs, scale, dsts, order=order)
        torch.cuda.synchronize()
        for i in range(3):
            assert np.array_equal(dsts[i].cpu().numpy(), single[i::3])
        assert np.array_equal(m.process_banded(big, scale, order=order), whole)
        plan = m.band_plan(bh, scale)
        dbig = _dev(big)
        sb = [dbig[s0:s1] for (_, _, s0, s1) in plan]
        db = [torch.zeros((r1 - r0, bow, 2), dtype=torch.uint8, device="cuda:0") for (r0, r1, _, _) in plan]
        torch.cuda.synchronize()
        m.process_banded_device(sb, bw, bh, scale, db, order=order)
        torch.cuda.synchronize()
        assert np.array_equal(torch.cat(db).cpu().numpy(), whole)
    finally:
        m.close()


@gpu
def test_launch_count(engine):
    """tcgen05, single frame: 3 launches (K-A, CNN, pack) on the one-launch path; 4 on the generic tiled path (the Y plane and the
    U / V planes are two resize launches)."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(61)
    for name in ORDERS:
        order = _order(S, name)
        for (w, h, scale, want) in [(128, 64, 2.0, 3), (64, 48, 4.0, 3), (128, 63, 2.0, 3), (100, 40, 2.0, 4), (384, 384, 1.5, 4),
                                    (54, 38, 3.0, 4)]:
            ow, oh = S.out_dims(w, h, scale)
            src = _dev(_frame(S, order, *_planes(rng, h, w)))
            dst = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
            n0 = engine.launches
            engine.process_device(src, scale, dst, order=order)
            engine.sync()
            assert engine.launches - n0 == want, (name, w, h, scale)


def _overlap(engine, on):
    engine.L.srcnn_debug_overlap.argtypes = [C.c_void_p, C.c_int]
    engine.L.srcnn_debug_overlap.restype = C.c_longlong
    return int(engine.L.srcnn_debug_overlap(engine.ctx, on))


@gpu
def test_overlap_chain_and_stale_workspace(engine):
    """BGR, YUY2, UYVY, GRAY, NV12, YUY2 on one stream, the UYVY call reading the YUY2 call's result; equal to the same chain fully
    serialised.  The YUY2 call after BGR (an independent source of the same geometry) starts early; the UYVY call fed by the
    previous result does not, nor does anything after the grey / 4:2:0 calls.  A context whose workspace was last carved by a
    larger BGR call gives the same 4:2:2 results."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(71)
    w, h, scale = 256, 128, 2.0
    ow, oh = S.out_dims(w, h, scale)
    bgr = _dev(natural_like(rng, h, w))
    yuy2 = [_dev(_frame(S, S.ORDER_YUY2, *_planes(rng, h, w))) for _ in range(2)]
    grey = _dev(_planes(rng, h, w)[0])
    nv12 = torch.zeros((h * 3 // 2, w), dtype=torch.uint8, device="cuda:0")
    nv12.copy_(_dev(rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)))
    orders = [S.ORDER_BGR, S.ORDER_YUY2, S.ORDER_UYVY, S.ORDER_GRAY, S.ORDER_NV12, S.ORDER_YUY2]
    shapes = [(oh, ow, 3), (oh, ow, 2), (oh, ow, 2), (oh, ow), (oh * 3 // 2, ow), (oh, ow, 2)]

    def run(serial):
        outs = [torch.zeros(s, dtype=torch.uint8, device="cuda:0") for s in shapes]
        srcs = [bgr, yuy2[0], None, grey, nv12, yuy2[1]]
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
        assert steps == [1, 0, 0, 0, 0], counts
        # each call alone on a fresh chain
        for i in (1, 5):
            out = torch.zeros(shapes[i], dtype=torch.uint8, device="cuda:0")
            engine.process_device([None, yuy2[0], None, None, None, yuy2[1]][i], scale, out, order=orders[i])
            engine.sync()
            assert torch.equal(out, got[i])
        big = torch.zeros((oh * 2, ow * 2, 3), dtype=torch.uint8, device="cuda:0")
        engine.process_device(_dev(natural_like(rng, h * 2, w * 2)), scale, big, order=S.ORDER_BGR)
        for i in (1, 5):
            out = torch.zeros(shapes[i], dtype=torch.uint8, device="cuda:0")
            engine.process_device([None, yuy2[0], None, None, None, yuy2[1]][i], scale, out, order=orders[i])
            engine.sync()
            assert torch.equal(out, got[i])
    finally:
        _overlap(engine, 1)


@gpu
def test_fused_merge_setting_changes_nothing(engine):
    """With the fused merge switched on a 4:2:2 call still takes its pack kernel: same bytes, same launch count."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(38)
    w, h, scale = 128, 64, 2.0
    ow, oh = S.out_dims(w, h, scale)
    for name in ORDERS:
        order = _order(S, name)
        frame = _frame(S, order, *_planes(rng, h, w))
        frames = np.stack([_frame(S, order, *_planes(rng, h, w)) for _ in range(3)])
        want = engine.process(frame, scale, order=order)
        want_b = engine.process_batch(frames, scale, order=order)
        dst = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
        n0 = engine.launches
        engine.process_device(_dev(frame), scale, dst, order=order)
        engine.sync()
        launches = engine.launches - n0
        engine.set_fuse_merge(True)
        try:
            assert np.array_equal(engine.process(frame, scale, order=order), want)
            assert np.array_equal(engine.process_batch(frames, scale, order=order), want_b)
            dst2 = torch.zeros_like(dst)
            n0 = engine.launches
            engine.process_device(_dev(frame), scale, dst2, order=order)
            engine.sync()
            assert engine.launches - n0 == launches == 3
            assert torch.equal(dst, dst2)
        finally:
            engine.set_fuse_merge(False)


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
    assert dev(64, 31, 128, 2.0, 256) == S.OK                   # odd heights are fine
    engine.sync()
    assert dev(63, 32, 128, 2.0, 256) == S.E_ARG                # odd width
    assert "even" in (L.srcnn_last_error(ctx) or b"").decode()
    assert dev(10, 10, 20, 1.5, 32) == S.E_ARG                  # 15-pixel output rows
    assert "odd" in (L.srcnn_last_error(ctx) or b"").decode()
    assert dev(64, 32, 127, 2.0, 256) == S.E_ARG                # short source stride
    assert dev(64, 32, 128, 2.0, 255) == S.E_ARG                # short destination stride
    assert "stride" in (L.srcnn_last_error(ctx) or b"").decode()
    assert L.srcnn_process_device(ctx, None, 64, 32, 128, order, f(2.0), p, 256) == S.E_ARG
    assert L.srcnn_process_device(ctx, p, 64, 32, 128, order, f(2.0), None, 256) == S.E_ARG
    # batch frame strides below one frame
    assert L.srcnn_process_batch_device(ctx, p, 2, 64, 32, 128, 128 * 31, order, f(2.0), p, 256, 256 * 64) == S.E_ARG
    assert L.srcnn_process_batch_device(ctx, p, 2, 64, 32, 128, 128 * 32, order, f(2.0), p, 256, 256 * 63) == S.E_ARG
    host = np.zeros(1 << 16, np.uint8)
    assert L.srcnn_process_batch_host(ctx, host.ctypes.data, 2, 64, 32, 128, 128 * 31, order, f(2.0), host.ctypes.data, 256,
                                      256 * 64) == S.E_ARG
    # the band calls check the same geometry
    assert L.srcnn_process_band_device(ctx, p, 63, 32, 128, 0, 32, order, f(2.0), 0, 64, p, 256) == S.E_ARG
    assert L.srcnn_process_band_host(ctx, host.ctypes.data, 64, 32, 127, order, f(2.0), 0, 64, host.ctypes.data, 256) == S.E_ARG
    # the colour and merge stage calls
    assert L.srcnn_stage_color_bicubic_device(ctx, p, 64, 32, 192, order, f(2.0), p, p, p, 128) == S.E_ARG
    assert L.srcnn_stage_merge_device(ctx, p, p, p, 64, 32, 64, order, p, 192) == S.E_ARG


@gpu
def test_full_size_1080p_yuy2_to_4k(engine, oracle):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(81)
    w, h, scale = 1920, 1080, 2.0
    ow, oh = S.out_dims(w, h, scale)
    y, u, v = _planes(rng, h, w)
    grey = engine.process(y, scale, order=S.ORDER_GRAY)
    out = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
    n0 = engine.launches
    engine.process_device(_dev(_frame(S, S.ORDER_YUY2, y, u, v)), scale, out, order=S.ORDER_YUY2)
    engine.sync()
    assert engine.launches - n0 == 3
    gy, gu, gv = _split(S, S.ORDER_YUY2, out.cpu().numpy())
    assert np.array_equal(gy, grey)
    assert np.array_equal(gu, oracle.resize_cubic(u, ow // 2, oh))
    assert np.array_equal(gv, oracle.resize_cubic(v, ow // 2, oh))
