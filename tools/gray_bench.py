#!/usr/bin/env python
"""Grey (SRCNN_ORDER_GRAY) against colour on one box: device time per frame of the device-resident whole path, the one-plane
resize stage alone, and the host-buffer end-to-end call.  One context, the same seeded images (the grey input is the colour
input's G channel, the colour input is that plane replicated to 3 channels, so both calls compute the same Y').

Timing: CUDA events on the context stream around blocks of back-to-back calls (so the colour path keeps its cross-call overlap),
grey and colour blocks alternating, median of the blocks.  Every call of a block reads and writes its own buffer set, and the
sets of one block together are larger than the 126 MB L2.  Every line carries the GPU name and its power limit.
usage: gray_bench.py [--quick]"""
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
HBM_PEAK = 7.7e12   # B/s, HGX B200 data sheet, one GPU
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


def device_line(name, w, h, scale, n, rounds):
    ow, oh = S.out_dims(w, h, scale)
    rng = np.random.default_rng(0)
    colour_bytes = n * (w * h + ow * oh) * 3
    nb = sets_for(colour_bytes // 3)       # enough grey sets to exceed L2; the colour sets are then 3x larger still
    greys = [torch.from_numpy(rng.integers(0, 256, (n, h, w), dtype=np.uint8)).cuda() for _ in range(nb)]
    cols = [g[..., None].expand(n, h, w, 3).contiguous() for g in greys]
    gout = [torch.zeros((n, oh, ow), dtype=torch.uint8, device="cuda") for _ in range(nb)]
    cout = [torch.zeros((n, oh, ow, 3), dtype=torch.uint8, device="cuda") for _ in range(nb)]
    if n == 1:
        g_calls = [lambda i=i: eng.process_device(greys[i][0], scale, gout[i][0], order=S.ORDER_GRAY) for i in range(nb)]
        c_calls = [lambda i=i: eng.process_device(cols[i][0], scale, cout[i][0]) for i in range(nb)]
    else:
        g_calls = [lambda i=i: eng.process_batch_device(greys[i], scale, gout[i], order=S.ORDER_GRAY) for i in range(nb)]
        c_calls = [lambda i=i: eng.process_batch_device(cols[i], scale, cout[i]) for i in range(nb)]
    gms, cms = [], []
    for _ in range(rounds):   # alternate, so that drift of the box hits both alike
        cms.append(time_blocks(c_calls, 3))
        gms.append(time_blocks(g_calls, 3))
    same = all(torch.equal(gout[i], cout[i][..., 1]) for i in range(nb))
    per = nb * n
    c, g = float(np.median(cms)) / per, float(np.median(gms)) / per
    emit(line=name, src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, frames_per_call=n, buffer_sets=nb,
         colour_ms_per_frame=round(c, 4), grey_ms_per_frame=round(g, 4), grey_over_colour=round(g / c, 3),
         grey_bytes_equal_colour_G=same)
    del greys, cols, gout, cout
    torch.cuda.empty_cache()


def stage_line(w, h, scale, rounds):
    ow, oh = S.out_dims(w, h, scale)
    rng = np.random.default_rng(1)
    nb = sets_for(w * h + ow * oh, hi=16)
    srcs = [torch.from_numpy(rng.integers(0, 256, (h, w), dtype=np.uint8)).cuda() for _ in range(nb)]
    dsts = [torch.zeros((oh, ow), dtype=torch.uint8, device="cuda") for _ in range(nb)]
    calls = [lambda i=i: eng.stage_resize_plane(srcs[i], scale, dsts[i]) for i in range(nb)]
    ms = float(np.median([time_blocks(calls, 3) for _ in range(rounds)])) / nb
    nbytes = w * h + ow * oh
    emit(line="stage_resize_plane", src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, us=round(ms * 1e3, 2),
         bytes=nbytes, TBps=round(nbytes / (ms * 1e-3) / 1e12, 3), share_of_hbm_peak=round(nbytes / (ms * 1e-3) / HBM_PEAK, 3))


def host_line(w, h, scale, reps):
    ow, oh = S.out_dims(w, h, scale)
    rng = np.random.default_rng(2)
    g = rng.integers(0, 256, (h, w), dtype=np.uint8)
    res = {}
    for order, px in ((S.ORDER_BGR, 3), (S.ORDER_GRAY, 1)):
        src, dst = S.PinnedBuffer(w * h * px), S.PinnedBuffer(ow * oh * px)
        src.array[:] = (np.repeat(g[..., None], 3, axis=2) if px == 3 else g).reshape(-1)
        call = lambda: eng._check(eng.L.srcnn_process_host(eng.ctx, src.ptr, w, h, w * px, order, C.c_float(scale), dst.ptr, ow * px))
        for _ in range(3):
            call()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        res[order] = (float(np.median(ts)) * 1e3, dst.array.reshape(oh, ow, px)[..., px // 2].copy())
        src.free()
        dst.free()
    c, g_ = res[S.ORDER_BGR][0], res[S.ORDER_GRAY][0]
    emit(line="host_e2e", src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, colour_ms=round(c, 4), grey_ms=round(g_, 4),
         grey_over_colour=round(g_ / c, 3), grey_bytes_equal_colour_G=bool(np.array_equal(res[S.ORDER_GRAY][1], res[S.ORDER_BGR][1])))


R = 3 if QUICK else 7
device_line("1080p_to_4K_x2", 1920, 1080, 2.0, 1, R)
device_line("720p_to_1440p_x2_batch", 1280, 720, 2.0, 32 if QUICK else 256, R)
device_line("4K_to_16K_x4", 3840, 2160, 4.0, 1, R)
device_line("1080p_x1.5", 1920, 1080, 1.5, 1, R)
stage_line(1920, 1080, 2.0, R)
stage_line(3840, 2160, 4.0, R)
stage_line(1920, 1080, 1.5, R)
host_line(1920, 1080, 2.0, 10 if QUICK else 30)
eng.close()
