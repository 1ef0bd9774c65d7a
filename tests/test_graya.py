"""The grey + alpha path (SRCNN_ORDER_GRAYA): 2-byte pixels G A end to end on the device.

No new parity contract: byte 0 of every output pixel is the SRCNN_ORDER_GRAY call on the source's grey plane (so the FP32 variant
equals oracle.cnn(oracle.resize_cubic(g)) exactly), and byte 1 is oracle.resize_cubic(alpha, ow, oh) -- the one-plane stage
srcnn_stage_resize_plane_device -- with no CNN.  Any size and scale; every whole-path call takes the order, band calls included."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import natural_like

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def _planes(rng, h, w):
    """a grey plane of natural-looking content and an alpha plane of noise"""
    g = np.ascontiguousarray(natural_like(rng, h, w)[:, :, 1])
    a = rng.integers(0, 256, (h, w), dtype=np.uint8)
    return g, a


def _frame(g, a):
    return np.ascontiguousarray(np.stack([g, a], axis=-1))


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

def test_enum_value_matches_header():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"SRCNN_ORDER_GRAYA\s*=\s*(\d+)", hdr).group(1)) == S.ORDER_GRAYA == 10
    assert not re.search(r"SRCNN_ORDER_\w+\s*=\s*5\b", hdr)   # 5 stays unassigned


def test_abi_version_unchanged():
    import srcnn_cpp_b200 as S
    hdr = open(os.path.join(ROOT, "include", "srcnn_b200.h")).read()
    assert int(re.search(r"#define SRCNN_B200_ABI_VERSION (\d+)", hdr).group(1)) == 2
    assert S.load_library().srcnn_abi_version() == 2


def test_python_shape_checks():
    """Rejected before any library call: a wrong rank, a wrong last dimension, a wrong dtype."""
    import srcnn_cpp_b200 as S
    order = S.ORDER_GRAYA
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
    assert S._pixel_shape(order) == (2,)


# ---- on the GPU ------------------------------------------------------------------------------------------------------------

def _dev(t):
    import torch
    return torch.from_numpy(np.ascontiguousarray(t)).to("cuda:0")


def _alpha_want(engine, oracle, a, ow, oh, scale):
    """oracle.resize_cubic of the alpha plane, checked against the one-plane stage"""
    import torch
    want = oracle.resize_cubic(a, ow, oh)
    got = torch.zeros((oh, ow), dtype=torch.uint8, device="cuda:0")
    engine.stage_resize_plane(_dev(a), scale, got)
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


# x2 / x4 with ow % 8 == 0 (one launch), x2 with ow % 8 != 0, x1.5, x3, x0.5 (the direct kernels), odd widths and heights, 1x1, 2x1
FAST = [(128, 64, 2.0), (64, 48, 4.0), (128, 63, 2.0), (100, 37, 4.0)]
GEOS = FAST + [(102, 40, 2.0), (45, 31, 2.0), (384, 384, 1.5), (1280, 720, 1.5), (54, 38, 3.0), (97, 33, 3.0), (96, 64, 0.5),
               (33, 17, 0.5), (1, 1, 2.0), (2, 1, 2.0), (1, 1, 4.0)]


def _check_parity(engine, oracle, w, h, scale):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(w * 3 + h)
    g, a = _planes(rng, h, w)
    ow, oh = S.out_dims(w, h, scale)
    want_g = oracle.cnn(oracle.resize_cubic(g, ow, oh))
    want_a = _alpha_want(engine, oracle, a, ow, oh, scale)
    frame = _frame(g, a)
    try:
        for variant in (S.VARIANT_FP32, S.VARIANT_TC):
            engine.set_variant(variant)
            grey = engine.process(g, scale, order=S.ORDER_GRAY)
            host = engine.process(frame, scale, order=S.ORDER_GRAYA)
            dev = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
            engine.process_device(_dev(frame), scale, dev, order=S.ORDER_GRAYA)
            engine.sync()
            assert host.shape == (oh, ow, 2)
            assert np.array_equal(dev.cpu().numpy(), host), variant
            assert np.array_equal(host[..., 0], grey), variant
            assert np.array_equal(host[..., 1], want_a), variant
            if variant == S.VARIANT_FP32:
                assert np.array_equal(host[..., 0], want_g)
            else:
                d = np.abs(host[..., 0].astype(np.int16) - want_g.astype(np.int16))
                assert d.max() <= 2 and (d <= 1).mean() >= 0.999, int(d.max())
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


@gpu
@pytest.mark.parametrize("w,h,scale", [(128, 64, 2.0), (64, 48, 4.0), (102, 40, 2.0), (384, 384, 1.5)])
def test_alpha_has_no_influence_on_grey(engine, w, h, scale):
    """The same grey plane with two different alpha planes: identical bytes 0."""
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(w + h)
    g, a = _planes(rng, h, w)
    one = engine.process(_frame(g, a), scale, order=S.ORDER_GRAYA)
    two = engine.process(_frame(g, 255 - a), scale, order=S.ORDER_GRAYA)
    assert np.array_equal(one[..., 0], two[..., 0])
    assert not np.array_equal(one[..., 1], two[..., 1])


def _written_mask(oh, ow, ds, nbytes, ofs):
    """bytes of a dst buffer (frame at byte `ofs`, rows `ds` apart) that a call may write"""
    m = np.zeros(nbytes, bool)
    for r in range(oh):
        m[ofs + r * ds:ofs + r * ds + 2 * ow] = True
    return m


# (w, h, scale, src stride pad, src byte offset, dst stride pad, dst byte offset): on the one-launch path 8-byte, 4-byte and
# unaligned sources (every class of the group loads), a 16-byte aligned destination and ones the 128-bit stores cannot take; the
# generic and direct kernels; odd widths
STRIDES = [(128, 64, 2.0, 8, 0, 16, 0), (128, 64, 2.0, 4, 0, 4, 0), (128, 64, 2.0, 0, 4, 0, 16), (128, 64, 2.0, 0, 1, 0, 3),
           (128, 64, 2.0, 2, 3, 6, 2), (64, 32, 4.0, 4, 0, 32, 16), (64, 32, 4.0, 1, 2, 3, 1), (100, 60, 1.5, 6, 5, 2, 1),
           (96, 40, 3.0, 2, 0, 14, 7), (96, 64, 0.5, 2, 1, 2, 1), (45, 31, 2.0, 1, 1, 3, 0), (101, 20, 4.0, 3, 0, 8, 16)]


@gpu
@pytest.mark.parametrize("w,h,scale,spad,sofs,dpad,dofs", STRIDES)
def test_strides_alignment_and_sentinels(engine, w, h, scale, spad, sofs, dpad, dofs):
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(w + h + spad + dofs)
    g, a = _planes(rng, h, w)
    ow, oh = S.out_dims(w, h, scale)
    want = engine.process(_frame(g, a), scale, order=S.ORDER_GRAYA)
    ss, ds = 2 * w + spad, 2 * ow + dpad
    sbytes = np.full((h, ss), 213, np.uint8)
    sbytes[:, :2 * w] = _frame(g, a).reshape(h, 2 * w)
    sbytes = sbytes.reshape(-1)
    sbuf = torch.full((sbytes.size + sofs + 64,), 5, dtype=torch.uint8, device="cuda:0")
    sbuf[sofs:sofs + sbytes.size] = _dev(sbytes)
    nbytes = oh * ds + dofs + 64
    dbuf = torch.full((nbytes,), 77, dtype=torch.uint8, device="cuda:0")
    src = sbuf[sofs:sofs + sbytes.size].view(h, ss)[:, :2 * w].view(h, w, 2)
    dst = dbuf[dofs:dofs + oh * ds].view(oh, ds)[:, :2 * ow].view(oh, ow, 2)
    engine.process_device(src, scale, dst, order=S.ORDER_GRAYA)
    engine.sync()
    full = dbuf.cpu().numpy()
    assert np.array_equal(dst.cpu().numpy(), want)
    assert (full[~_written_mask(oh, ow, ds, nbytes, dofs)] == 77).all()
    # the host call on the same padded rows
    hsrc = np.lib.stride_tricks.as_strided(sbytes, shape=(h, w, 2), strides=(ss, 2, 1))
    assert np.array_equal(engine.process(hsrc, scale, order=S.ORDER_GRAYA), want)


@gpu
@pytest.mark.parametrize("w,h,scale", [(128, 72, 2.0), (64, 36, 4.0), (128, 72, 1.5), (77, 35, 2.0)])
def test_batches(engine, w, h, scale):
    """Device and host batches, tight (one tall result) and padded frame strides, against frame-by-frame calls; a repeated host
    call on the same pinned buffers (replayed as a CUDA graph) equals the first."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(31)
    n = 5
    ow, oh = S.out_dims(w, h, scale)
    frames = np.stack([_frame(*_planes(rng, h, w)) for _ in range(n)])
    single = np.stack([engine.process(f, scale, order=S.ORDER_GRAYA) for f in frames])
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
        engine.process_batch_device(src, scale, dst, order=S.ORDER_GRAYA)
        engine.sync()
        if scale != 1.5 and ow % 8 == 0:   # one chunk: one resize launch, one CNN launch, one pack launch (or one per frame when padded)
            assert engine.launches - n0 == (3 if pad == 0 else 2 + n)
        assert np.array_equal(dst.cpu().numpy(), single), pad
        if pad:
            assert int(dbuf.view(n, ofr)[:, oh * ow * 2:].ne(77).sum()) == 0
    assert np.array_equal(engine.process_batch(frames, scale, order=S.ORDER_GRAYA), single)
    pin_in = S.PinnedBuffer(frames.nbytes)
    pin_out = S.PinnedBuffer(single.nbytes)
    try:
        pin_in.array[:] = frames.reshape(-1)
        src = pin_in.array.reshape(frames.shape)
        out = pin_out.array.reshape(single.shape)
        for _ in range(3):   # live, captured, replayed
            out[...] = 0
            engine.process_batch(src, scale, order=S.ORDER_GRAYA, out=out)
            assert np.array_equal(out, single)
    finally:
        pin_in.free()
        pin_out.free()


@gpu
def test_tall_single_host_frame_in_sub_bands(engine):
    """A single host frame tall enough to be cut into several sub-bands equals the device call."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(41)
    w, h, scale = 256, 1536, 2.0
    ow, oh = S.out_dims(w, h, scale)
    frame = _frame(*_planes(rng, h, w))
    dev = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
    engine.process_device(_dev(frame), scale, dev, order=S.ORDER_GRAYA)
    engine.sync()
    for bands in (8, 3):
        engine.set_host_bands(bands)
        try:
            assert np.array_equal(engine.process(frame, scale, order=S.ORDER_GRAYA), dev.cpu().numpy()), bands
        finally:
            engine.set_host_bands(8)


@gpu
@pytest.mark.parametrize("w,h,scale", [(256, 96, 2.0), (201, 75, 1.5), (64, 40, 4.0), (45, 31, 2.0)])
def test_bands_union_is_the_whole_frame(engine, w, h, scale):
    """process_band_device / process_band_host over several cuts: the union equals the whole-frame call bit for bit (the halo is
    the luma one; alpha needs no more)."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(w + h)
    ow, oh = S.out_dims(w, h, scale)
    frame = _frame(*_planes(rng, h, w))
    whole = engine.process(frame, scale, order=S.ORDER_GRAYA)
    dsrc = _dev(frame)
    for cuts in ([0, oh], [0, 7, oh], [0, oh // 3, oh // 3 + 1, 2 * oh // 3, oh]):
        dev = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
        host = np.zeros((oh, ow, 2), np.uint8)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            s0, s1 = S.band_src_rows(h, scale, r0, r1)
            engine.process_band_device(dsrc[s0:s1], w, h, s0, s1, scale, r0, r1, dev[r0:r1], order=S.ORDER_GRAYA)
            host[r0:r1] = engine.process_band_host(frame, scale, r0, r1, order=S.ORDER_GRAYA)
        engine.sync()
        assert np.array_equal(dev.cpu().numpy(), whole), cuts
        assert np.array_equal(host, whole), cuts


@gpu
def test_multi_engine(engine):
    """MultiEngine banded and batch calls, host and device buffers, equal the one-context result."""
    import torch
    import srcnn_cpp_b200 as S
    order = S.ORDER_GRAYA
    rng = np.random.default_rng(51)
    n, w, h, scale = 5, 96, 64, 2.0
    ow, oh = S.out_dims(w, h, scale)
    frames = np.stack([_frame(*_planes(rng, h, w)) for _ in range(n)])
    single = engine.process_batch(frames, scale, order=order)
    bw, bh = 127, 150
    big = _frame(*_planes(rng, bh, bw))
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
    """tcgen05, single frame: 3 launches (K-A, CNN, pack) on the one-launch path; 4 on the generic tiled path (grey and alpha are
    two resize launches)."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(61)
    for (w, h, scale, want) in [(128, 64, 2.0, 3), (64, 48, 4.0, 3), (128, 63, 2.0, 3), (45, 31, 4.0, 4), (102, 40, 2.0, 4),
                                (384, 384, 1.5, 4), (54, 38, 3.0, 4)]:
        ow, oh = S.out_dims(w, h, scale)
        src = _dev(_frame(*_planes(rng, h, w)))
        dst = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
        n0 = engine.launches
        engine.process_device(src, scale, dst, order=S.ORDER_GRAYA)
        engine.sync()
        assert engine.launches - n0 == want, (w, h, scale)


def _overlap(engine, on):
    engine.L.srcnn_debug_overlap.argtypes = [C.c_void_p, C.c_int]
    engine.L.srcnn_debug_overlap.restype = C.c_longlong
    return int(engine.L.srcnn_debug_overlap(engine.ctx, on))


@gpu
def test_overlap_chain_and_stale_workspace(engine):
    """BGR, GRAYA, BGR, GRAYA, GRAYA (reading the previous call's result), GRAY, GRAYA on one stream; equal to the same chain fully
    serialised.  GRAYA after BGR and BGR after GRAYA (independent sources of the same geometry) start early; the GRAYA call fed by
    the previous result does not, nor does anything after the grey call.  A context whose workspace was last carved by a larger BGR
    call gives the same GRAYA results."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(71)
    w, h, scale = 256, 128, 2.0
    ow, oh = S.out_dims(w, h, scale)
    bgr = [_dev(natural_like(rng, h, w)) for _ in range(2)]
    ga = [_dev(_frame(*_planes(rng, h, w))) for _ in range(3)]
    grey = _dev(_planes(rng, h, w)[0])
    orders = [S.ORDER_BGR, S.ORDER_GRAYA, S.ORDER_BGR, S.ORDER_GRAYA, S.ORDER_GRAYA, S.ORDER_GRAY, S.ORDER_GRAYA]
    shapes = [(oh, ow, 3), (oh, ow, 2), (oh, ow, 3), (oh, ow, 2), (oh, ow, 2), (oh, ow), (oh, ow, 2)]
    srcs = [bgr[0], ga[0], bgr[1], ga[1], None, grey, ga[2]]

    def run(serial):
        outs = [torch.zeros(s, dtype=torch.uint8, device="cuda:0") for s in shapes]
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
        assert steps == [1, 1, 1, 0, 0, 0], counts
        # each GRAYA call alone on a fresh chain, then after a larger BGR call has carved the workspace
        for big_first in (False, True):
            if big_first:
                big = torch.zeros((oh * 2, ow * 2, 3), dtype=torch.uint8, device="cuda:0")
                engine.process_device(_dev(natural_like(rng, h * 2, w * 2)), scale, big, order=S.ORDER_BGR)
            for i in (1, 3, 6):
                out = torch.zeros(shapes[i], dtype=torch.uint8, device="cuda:0")
                engine.process_device(srcs[i], scale, out, order=S.ORDER_GRAYA)
                engine.sync()
                assert torch.equal(out, got[i]), (big_first, i)
    finally:
        _overlap(engine, 1)


@gpu
def test_fused_merge_setting_changes_nothing(engine):
    """With the fused merge switched on a GRAYA call still takes its pack kernel: same bytes, same launch count."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(38)
    w, h, scale = 128, 64, 2.0
    ow, oh = S.out_dims(w, h, scale)
    frame = _frame(*_planes(rng, h, w))
    frames = np.stack([_frame(*_planes(rng, h, w)) for _ in range(3)])
    want = engine.process(frame, scale, order=S.ORDER_GRAYA)
    want_b = engine.process_batch(frames, scale, order=S.ORDER_GRAYA)
    dst = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
    n0 = engine.launches
    engine.process_device(_dev(frame), scale, dst, order=S.ORDER_GRAYA)
    engine.sync()
    launches = engine.launches - n0
    engine.set_fuse_merge(True)
    try:
        assert np.array_equal(engine.process(frame, scale, order=S.ORDER_GRAYA), want)
        assert np.array_equal(engine.process_batch(frames, scale, order=S.ORDER_GRAYA), want_b)
        dst2 = torch.zeros_like(dst)
        n0 = engine.launches
        engine.process_device(_dev(frame), scale, dst2, order=S.ORDER_GRAYA)
        engine.sync()
        assert engine.launches - n0 == launches == 3
        assert torch.equal(dst, dst2)
    finally:
        engine.set_fuse_merge(False)


@gpu
def test_rejections(engine):
    import torch
    import srcnn_cpp_b200 as S
    order = S.ORDER_GRAYA
    L, ctx = engine.L, engine.ctx
    buf = torch.zeros((1 << 20,), dtype=torch.uint8, device="cuda:0")
    p = C.c_void_p(buf.data_ptr())
    f = C.c_float
    dev = lambda w, h, ss, sc, ds: L.srcnn_process_device(ctx, p, w, h, ss, order, f(sc), p, ds)
    assert dev(63, 31, 126, 2.0, 252) == S.OK                   # odd sizes are fine
    assert dev(10, 10, 20, 1.5, 30) == S.OK                     # so is an odd output width
    engine.sync()
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
    assert L.srcnn_process_band_device(ctx, p, 64, 32, 127, 0, 32, order, f(2.0), 0, 64, p, 256) == S.E_ARG
    assert L.srcnn_process_band_host(ctx, host.ctypes.data, 64, 32, 128, order, f(2.0), 0, 64, host.ctypes.data, 255) == S.E_ARG
    # the colour and merge stage calls
    assert L.srcnn_stage_color_bicubic_device(ctx, p, 64, 32, 192, order, f(2.0), p, p, p, 128) == S.E_ARG
    assert L.srcnn_stage_merge_device(ctx, p, p, p, 64, 32, 64, order, p, 192) == S.E_ARG
    # 5 stays unassigned, 11 is not an order
    for bad in (5, 11):
        assert L.srcnn_process_device(ctx, p, 64, 32, 256, bad, f(2.0), p, 512) == S.E_ARG


def _process_srcnn():
    import srcnn_cpp_b200 as S
    fn = S.load_library()._Z12ProcessSRCNNPKhjjjfRPhRj
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.POINTER(C.c_void_p), C.POINTER(C.c_uint)]
    return fn


@gpu
@pytest.mark.parametrize("d", [2, 3])
@pytest.mark.parametrize("w,h,scale", [(45, 31, 2.0), (33, 19, 1.5), (23, 11, 4.0)])
def test_process_srcnn_one_call(engine, d, w, h, scale):
    """ProcessSRCNN d = 2 and d = 3 on sizes whose rows are not 4-byte multiples equal the explicit composition: the grey call and
    the one-plane alpha resize interleaved (d = 2), the RGB call (d = 3)."""
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(7 * d + w)
    if d == 2:
        g, a = _planes(rng, h, w)
        img = _frame(g, a)
    else:
        img = np.ascontiguousarray(natural_like(rng, h, w))
    out, sz = C.c_void_p(), C.c_uint()
    assert _process_srcnn()(img.ctypes.data, w, h, d, C.c_float(scale), C.byref(out), C.byref(sz)) == 0
    ow, oh = S.out_dims(w, h, scale)
    assert sz.value == ow * oh * d
    got = np.ctypeslib.as_array((C.c_uint8 * sz.value).from_address(out.value)).reshape(oh, ow, d).copy()
    if d == 2:
        want = np.stack([engine.process(g, scale, order=S.ORDER_GRAY), engine.resize_plane(a, scale)], axis=-1)
    else:
        want = engine.process(img, scale, order=S.ORDER_RGB)
    assert np.array_equal(got, want)


@gpu
def test_full_size_1080p_to_4k(engine, oracle):
    """One full 1080p -> 4K x2 frame: byte 0 against the oracle within the tensor-core tolerance (and equal to the grey call), byte 1
    exactly the oracle's cubic resize of alpha."""
    import torch
    import srcnn_cpp_b200 as S
    rng = np.random.default_rng(81)
    w, h, scale = 1920, 1080, 2.0
    ow, oh = S.out_dims(w, h, scale)
    g, a = _planes(rng, h, w)
    out = torch.zeros((oh, ow, 2), dtype=torch.uint8, device="cuda:0")
    n0 = engine.launches
    engine.process_device(_dev(_frame(g, a)), scale, out, order=S.ORDER_GRAYA)
    engine.sync()
    assert engine.launches - n0 == 3
    got = out.cpu().numpy()
    assert np.array_equal(got[..., 0], engine.process(g, scale, order=S.ORDER_GRAY))
    assert np.array_equal(got[..., 1], oracle.resize_cubic(a, ow, oh))
    want = oracle.cnn(oracle.resize_cubic(g, ow, oh))
    d = np.abs(got[..., 0].astype(np.int16) - want.astype(np.int16))
    assert d.max() <= 2 and (d <= 1).mean() >= 0.999, (int(d.max()), float((d <= 1).mean()))
