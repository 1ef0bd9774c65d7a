#!/usr/bin/env python
"""Four-channel (SRCNN_ORDER_BGRA) against colour (SRCNN_ORDER_BGR) on one box: device time per frame of the device-resident whole
path, the host-buffer end-to-end call, and ProcessSRCNN with d = 4 before and after it became one RGBA call.  One context, the
same seeded images: the BGR input is bytes 0..2 of the BGRA input, whose alpha is seeded noise.  Every line checks that the
BGRA result's colour bytes equal the BGR result.

Timing: CUDA events on the context stream around blocks of back-to-back calls (so both keep their cross-call overlap), BGRA and
BGR blocks alternating, median of the blocks.  Every call of a block reads and writes its own buffer set, and the sets of one
block together are larger than the 126 MB L2.  The host-side lines take a host clock around calls that end in a synchronise.
Every line carries the GPU name and its power limit.

"Before" for ProcessSRCNN d = 4 is the composition the library used until the four-channel path existed, rebuilt here from
Python calls with the same steps: de-interleave on the CPU, srcnn_process_host(RGB) and srcnn_resize_plane_host(alpha) on
pageable buffers, re-interleave on the CPU (numpy does the two CPU loops, so "before" is if anything faster than the C++ was).
"After" is the exported ProcessSRCNN itself.
usage: rgba_bench.py [--quick]"""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import srcnn_cpp_b200 as S

QUICK = "--quick" in sys.argv
L2_BYTES = 126 << 20


def box():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, plim, clk = [x.strip() for x in q[0].split(",")] if q else (torch.cuda.get_device_name(0), "?", "?")
    return dict(gpu=name, power_limit=plim, max_sm_clock=clk)


BOX = box()
st = torch.cuda.Stream()
torch.cuda.set_stream(st)
eng = S.Engine(0, variant=S.VARIANT_TC, stream=st.cuda_stream)


def emit(**kw):
    kw.update(BOX)
    print(json.dumps(kw), flush=True)


def time_blocks(calls, blocks):
    """calls: list of callables run back to back as one block; -> median ms of a block over `blocks` blocks"""
    for fn in calls:
        fn()
    torch.cuda.synchronize()
    ev = []
    for _ in range(blocks):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for fn in calls:
            fn()
        e1.record()
        ev.append((e0, e1))
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def sets_for(bytes_per_set, lo=2, hi=8):
    return int(min(hi, max(lo, -(-2 * L2_BYTES // bytes_per_set))))


def seeded(seed, shape):
    """BGRA frames: colour bytes smooth-ish (low-res noise upsampled), alpha plain noise"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    n, h, w = shape
    small = torch.randint(0, 256, (n, 3, max(2, h // 8), max(2, w // 8)), generator=g, device="cuda", dtype=torch.uint8)
    col = torch.nn.functional.interpolate(small.float(), size=(h, w), mode="bilinear", align_corners=False)
    col = col.round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1)
    alpha = torch.randint(0, 256, (n, h, w, 1), generator=g, device="cuda", dtype=torch.uint8)
    return torch.cat([col, alpha], dim=3).contiguous()


def device_line(name, w, h, scale, n, rounds):
    ow, oh = S.out_dims(w, h, scale)
    nb = sets_for(n * (w * h + ow * oh) * 3)   # enough BGR sets to exceed L2; the BGRA sets are then 4/3 larger still
    quads = [seeded(i, (n, h, w)) for i in range(nb)]
    cols = [q[..., :3].contiguous() for q in quads]
    qout = [torch.zeros((n, oh, ow, 4), dtype=torch.uint8, device="cuda") for _ in range(nb)]
    cout = [torch.zeros((n, oh, ow, 3), dtype=torch.uint8, device="cuda") for _ in range(nb)]
    if n == 1:
        q_calls = [lambda i=i: eng.process_device(quads[i][0], scale, qout[i][0], order=S.ORDER_BGRA) for i in range(nb)]
        c_calls = [lambda i=i: eng.process_device(cols[i][0], scale, cout[i][0]) for i in range(nb)]
    else:
        q_calls = [lambda i=i: eng.process_batch_device(quads[i], scale, qout[i], order=S.ORDER_BGRA) for i in range(nb)]
        c_calls = [lambda i=i: eng.process_batch_device(cols[i], scale, cout[i]) for i in range(nb)]
    qms, cms = [], []
    for _ in range(rounds):   # alternate, so that drift of the box hits both alike
        cms.append(time_blocks(c_calls, 3))
        qms.append(time_blocks(q_calls, 3))
    same = all(torch.equal(qout[i][..., :3], cout[i]) for i in range(nb))
    per = nb * n
    c, q = float(np.median(cms)) / per, float(np.median(qms)) / per
    emit(line=name, src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, frames_per_call=n, buffer_sets=nb,
         bgr_ms_per_frame=round(c, 4), bgra_ms_per_frame=round(q, 4), bgra_over_bgr=round(q / c, 3),
         bgra_colour_bytes_equal_bgr=same)
    del quads, cols, qout, cout
    torch.cuda.empty_cache()


def host_line(w, h, scale, reps):
    ow, oh = S.out_dims(w, h, scale)
    img = seeded(100, (1, h, w))[0].cpu().numpy()
    res = {}
    for order, px in ((S.ORDER_BGR, 3), (S.ORDER_BGRA, 4)):
        src, dst = S.PinnedBuffer(w * h * px), S.PinnedBuffer(ow * oh * px)
        src.array[:] = np.ascontiguousarray(img[..., :px]).reshape(-1)
        call = lambda: eng._check(eng.L.srcnn_process_host(eng.ctx, src.ptr, w, h, w * px, order, C.c_float(scale), dst.ptr, ow * px))
        for _ in range(3):
            call()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        res[order] = (float(np.median(ts)) * 1e3, dst.array.reshape(oh, ow, px)[..., :3].copy())
        src.free()
        dst.free()
    c, q = res[S.ORDER_BGR][0], res[S.ORDER_BGRA][0]
    emit(line="host_e2e", src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, bgr_ms=round(c, 4), bgra_ms=round(q, 4),
         bgra_over_bgr=round(q / c, 3), bgra_colour_bytes_equal_bgr=bool(np.array_equal(res[S.ORDER_BGRA][1], res[S.ORDER_BGR][1])))


def process_srcnn_line(w, h, scale, reps):
    fn = S.load_library()._Z12ProcessSRCNNPKhjjjfRPhRj
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.POINTER(C.c_void_p), C.POINTER(C.c_uint)]
    ow, oh = S.out_dims(w, h, scale)
    rgba = seeded(101, (1, h, w))[0].cpu().numpy()

    def before():   # the old d = 4 composition, step by step
        rgb = np.ascontiguousarray(rgba[..., :3])
        alpha = np.ascontiguousarray(rgba[..., 3])
        out = np.empty((oh, ow, 4), np.uint8)
        out[..., :3] = eng.process(rgb, scale, order=S.ORDER_RGB)
        out[..., 3] = eng.resize_plane(alpha, scale)
        return out

    def after():
        out, sz = C.c_void_p(), C.c_uint()
        if fn(rgba.ctypes.data, w, h, 4, C.c_float(scale), C.byref(out), C.byref(sz)) != 0:
            raise RuntimeError("ProcessSRCNN failed")
        # the caller delete[]s the buffer in C++; here it is copied out and left to the process (a few calls of a benchmark)
        return np.ctypeslib.as_array((C.c_uint8 * sz.value).from_address(out.value)).reshape(oh, ow, 4).copy()

    times = {before: [], after: []}
    for fn_ in (before, after):
        for _ in range(2):
            fn_()
    for _ in range(reps):   # alternating
        for fn_ in (before, after):
            t0 = time.perf_counter()
            fn_()
            times[fn_].append(time.perf_counter() - t0)
    b, a = float(np.median(times[before])) * 1e3, float(np.median(times[after])) * 1e3
    emit(line="ProcessSRCNN_d4", src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, before_ms=round(b, 3), after_ms=round(a, 3),
         after_over_before=round(a / b, 3), bytes_equal=bool(np.array_equal(before(), after())),
         colour_bytes_equal_bgr_path=bool(np.array_equal(after()[..., :3], eng.process(np.ascontiguousarray(rgba[..., :3]), scale,
                                                                                          order=S.ORDER_RGB))))


R = 3 if QUICK else 7
device_line("1080p_to_4K_x2", 1920, 1080, 2.0, 1, R)
device_line("720p_to_1440p_x2_batch", 1280, 720, 2.0, 32 if QUICK else 256, R)
device_line("4K_to_16K_x4", 3840, 2160, 4.0, 1, R)
device_line("1080p_x1.5", 1920, 1080, 1.5, 1, R)
host_line(1920, 1080, 2.0, 10 if QUICK else 30)
process_srcnn_line(1920, 1080, 2.0, 5 if QUICK else 15)
eng.close()
