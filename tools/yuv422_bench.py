#!/usr/bin/env python
"""Packed 4:2:2 frames (SRCNN_ORDER_YUY2 / _UYVY) on one box: device time per frame of the device-resident whole path against
the grey call on the Y plane alone, the colour (BGR) call on a frame of the same size, and the composition a caller has without
this path -- the grey call on Y plus two srcnn_stage_resize_plane_device calls on already de-interleaved U / V planes (the
de-interleave itself not timed) -- and the host-buffer call, YUY2 against BGR.  One context, seeded images (the 4:2:2 frames, the
Y planes and the U / V planes of one buffer set hold the same content).

Timing: CUDA events on the context stream around blocks of back-to-back calls, the five forms alternating, median of the blocks.
Every call of a block reads and writes its own buffer set, and the sets of one block together are larger than the 126 MB L2.
Every line says whether YUY2 and UYVY gave the composition's bytes, and carries the GPU name and its power limit.
usage: yuv422_bench.py [--quick]"""
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


def pack(y, u, v, order):
    """N x H x W x 2 device frames from N x H x W / N x H x W/2 planes"""
    n, h, w = y.shape
    f = torch.empty((n, h, w, 2), dtype=torch.uint8, device="cuda")
    for i in range(n):
        fy, fu, fv = S.yuv422_planes(f[i], order)
        fy.copy_(y[i])
        fu.copy_(u[i])
        fv.copy_(v[i])
    return f


def device_line(name, w, h, scale, n, rounds):
    ow, oh = S.out_dims(w, h, scale)
    g = torch.Generator(device="cuda").manual_seed(0)
    rnd = lambda *shape: torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=g)
    nb = sets_for(n * (w * h + ow * oh) * 2)
    sets = []
    for _ in range(nb):
        y, u, v = rnd(n, h, w), rnd(n, h, w // 2), rnd(n, h, w // 2)
        sets.append(dict(y=y, u=u, v=v, yuy2=pack(y, u, v, S.ORDER_YUY2), uyvy=pack(y, u, v, S.ORDER_UYVY), bgr=rnd(n, h, w, 3),
                         o_yuy2=torch.zeros((n, oh, ow, 2), dtype=torch.uint8, device="cuda"),
                         o_uyvy=torch.zeros((n, oh, ow, 2), dtype=torch.uint8, device="cuda"),
                         o_y=torch.zeros((n, oh, ow), dtype=torch.uint8, device="cuda"),
                         o_u=torch.zeros((n, oh, ow // 2), dtype=torch.uint8, device="cuda"),
                         o_v=torch.zeros((n, oh, ow // 2), dtype=torch.uint8, device="cuda"),
                         o_bgr=torch.zeros((n, oh, ow, 3), dtype=torch.uint8, device="cuda")))

    def whole(key, out, order):
        if n == 1:
            return [lambda s=s: eng.process_device(s[key][0], scale, s[out][0], order=order) for s in sets]
        return [lambda s=s: eng.process_batch_device(s[key], scale, s[out], order=order) for s in sets]

    def composition(s):
        (eng.process_device(s["y"][0], scale, s["o_y"][0], order=S.ORDER_GRAY) if n == 1 else
         eng.process_batch_device(s["y"], scale, s["o_y"], order=S.ORDER_GRAY))
        for f in range(n):
            eng.stage_resize_plane(s["u"][f], scale, s["o_u"][f])
            eng.stage_resize_plane(s["v"][f], scale, s["o_v"][f])

    forms = dict(yuy2=whole("yuy2", "o_yuy2", S.ORDER_YUY2), uyvy=whole("uyvy", "o_uyvy", S.ORDER_UYVY),
                 grey=whole("y", "o_y", S.ORDER_GRAY), bgr=whole("bgr", "o_bgr", S.ORDER_BGR),
                 composition=[lambda s=s: composition(s) for s in sets])
    ms = {k: [] for k in forms}
    for _ in range(rounds):   # alternate, so that drift of the box hits every form alike
        for k, calls in forms.items():
            ms[k].append(time_blocks(calls, 3))
    same = True
    for s in sets:
        for key, order in (("o_yuy2", S.ORDER_YUY2), ("o_uyvy", S.ORDER_UYVY)):
            for f in range(n):
                yy, uu, vv = S.yuv422_planes(s[key][f], order)
                same &= torch.equal(yy, s["o_y"][f]) and torch.equal(uu, s["o_u"][f]) and torch.equal(vv, s["o_v"][f])
    per = nb * n
    t = {k: float(np.median(v)) / per for k, v in ms.items()}
    emit(line=name, src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, frames_per_call=n, buffer_sets=nb,
         **{k + "_ms_per_frame": round(v, 4) for k, v in t.items()},
         yuy2_over_grey=round(t["yuy2"] / t["grey"], 3), yuy2_over_bgr=round(t["yuy2"] / t["bgr"], 3),
         yuy2_over_composition=round(t["yuy2"] / t["composition"], 3), uyvy_over_yuy2=round(t["uyvy"] / t["yuy2"], 3),
         bytes_equal_composition=bool(same))
    del sets
    torch.cuda.empty_cache()


def host_line(w, h, scale, reps):
    ow, oh = S.out_dims(w, h, scale)
    rng = np.random.default_rng(2)
    res = {}
    for order, src_bytes, dst_bytes, stride, dstride in ((S.ORDER_BGR, w * h * 3, ow * oh * 3, w * 3, ow * 3),
                                                         (S.ORDER_YUY2, w * h * 2, ow * oh * 2, w * 2, ow * 2)):
        src, dst = S.PinnedBuffer(src_bytes), S.PinnedBuffer(dst_bytes)
        src.array[:] = rng.integers(0, 256, src_bytes, dtype=np.uint8)
        call = lambda: eng._check(eng.L.srcnn_process_host(eng.ctx, src.ptr, w, h, stride, order, C.c_float(scale), dst.ptr, dstride))
        for _ in range(3):
            call()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        res[order] = float(np.median(ts)) * 1e3
        src.free()
        dst.free()
    c, v = res[S.ORDER_BGR], res[S.ORDER_YUY2]
    emit(line="host_e2e", src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, bgr_ms=round(c, 4), yuy2_ms=round(v, 4),
         yuy2_over_bgr=round(v / c, 3))


R = 3 if QUICK else 7
device_line("1080p_to_4K_x2", 1920, 1080, 2.0, 1, R)
device_line("720p_to_1440p_x2_batch", 1280, 720, 2.0, 32 if QUICK else 256, R)
device_line("4K_to_16K_x4", 3840, 2160, 4.0, 1, R)
device_line("1080p_x1.5", 1920, 1080, 1.5, 1, R)
host_line(1920, 1080, 2.0, 10 if QUICK else 30)
eng.close()
