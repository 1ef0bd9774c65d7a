#!/usr/bin/env python
"""Each pixel format against the calls it replaces, on one box: device time per frame of the device-resident whole path, the
host-buffer end-to-end call, and a few format-specific lines.  One context, seeded images.

  gray    grey (SRCNN_ORDER_GRAY) against colour; the grey input is the colour input's G channel, the colour input that plane
          replicated to 3 channels, so both compute the same Y'.  Also the one-plane resize stage alone (us, TB/s, share of HBM
          peak).
  rgba    four-channel (SRCNN_ORDER_BGRA) against colour (SRCNN_ORDER_BGR); the BGR input is bytes 0..2 of the BGRA input, whose
          alpha is seeded noise, and every line checks that the BGRA result's colour bytes equal the BGR result.  Also
          ProcessSRCNN with d = 4 before and after it became one RGBA call: "before" is the composition the library used until the
          four-channel path existed, rebuilt from Python calls with the same steps (de-interleave on the CPU,
          srcnn_process_host(RGB) and srcnn_resize_plane_host(alpha) on pageable buffers, re-interleave on the CPU; numpy does the
          two CPU loops, so "before" is if anything faster than the C++ was), "after" is the exported ProcessSRCNN itself.
  yuv420  4:2:0 frames (SRCNN_ORDER_NV12 / _I420) and
  yuv422  packed 4:2:2 frames (SRCNN_ORDER_YUY2 / _UYVY) against the grey call on the Y plane alone, the colour (BGR) call on a
          frame of the same size, and the composition a caller has without the path -- the grey call on Y plus two
          srcnn_stage_resize_plane_device calls on already de-interleaved U / V planes (the de-interleave not timed); the host
          call NV12 / YUY2 against BGR.  The frames, the Y planes and the U / V planes of one buffer set hold the same content,
          and every line says whether both orders gave the composition's bytes.
  graya   grey + alpha (SRCNN_ORDER_GRAYA) against the grey call on the grey plane alone, the colour (BGR) call on a frame of the
          same size, and the composition a caller has without the path -- the grey call plus srcnn_stage_resize_plane_device on an
          already de-interleaved alpha plane (the de-interleave and re-interleave not timed); the host call GRAYA against grey and
          BGR; every line checks that the GRAYA bytes equal the composition's.  Also ProcessSRCNN with d = 2 before and after it
          became one GRAYA call, as for d = 4 above.

Timing: CUDA events on the context stream around blocks of back-to-back calls (so the colour path keeps its cross-call overlap),
the forms of a line alternating, median of the blocks.  Every call of a block reads and writes its own buffer set, and the sets
of one block together are larger than the 126 MB L2.  The host-side lines take a host clock around calls that end in a
synchronise.  Every line carries the GPU name and its power limit.
usage: format_bench.py [--format gray|rgba|yuv420|yuv422|graya|all] [--quick]"""
import argparse
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

FORMATS = ("gray", "rgba", "yuv420", "yuv422", "graya")
ap = argparse.ArgumentParser()
ap.add_argument("--format", choices=FORMATS + ("all",), default="all")
ap.add_argument("--quick", action="store_true")
ARGS = ap.parse_args()
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


def zeros(*shape):
    return torch.zeros(shape, dtype=torch.uint8, device="cuda")


def whole(sets, key, out, order, scale, n):
    """one whole-path call per buffer set: s[key] -> s[out]"""
    if n == 1:
        return [lambda s=s: eng.process_device(s[key][0], scale, s[out][0], order=order) for s in sets]
    return [lambda s=s: eng.process_batch_device(s[key], scale, s[out], order=order) for s in sets]


def rgba_seeded(seed, shape):
    """BGRA frames: colour bytes smooth-ish (low-res noise upsampled), alpha plain noise"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    n, h, w = shape
    small = torch.randint(0, 256, (n, 3, max(2, h // 8), max(2, w // 8)), generator=g, device="cuda", dtype=torch.uint8)
    col = torch.nn.functional.interpolate(small.float(), size=(h, w), mode="bilinear", align_corners=False)
    col = col.round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1)
    alpha = torch.randint(0, 256, (n, h, w, 1), generator=g, device="cuda", dtype=torch.uint8)
    return torch.cat([col, alpha], dim=3).contiguous()


# ---- device lines: each format's buffer sets, the forms timed against each other (in alternation order) and the line's fields
def gray_forms(w, h, ow, oh, scale, n):
    rng = np.random.default_rng(0)
    nb = sets_for(n * (w * h + ow * oh))       # enough grey sets to exceed L2; the colour sets are then 3x larger still
    sets = []
    for _ in range(nb):
        y = torch.from_numpy(rng.integers(0, 256, (n, h, w), dtype=np.uint8)).cuda()
        sets.append(dict(y=y, bgr=y[..., None].expand(n, h, w, 3).contiguous(), o_y=zeros(n, oh, ow), o_bgr=zeros(n, oh, ow, 3)))
    forms = dict(colour=whole(sets, "bgr", "o_bgr", S.ORDER_BGR, scale, n), grey=whole(sets, "y", "o_y", S.ORDER_GRAY, scale, n))

    def fields(t):
        c, g = t["colour"], t["grey"]
        return dict(colour_ms_per_frame=round(c, 4), grey_ms_per_frame=round(g, 4), grey_over_colour=round(g / c, 3),
                    grey_bytes_equal_colour_G=all(torch.equal(s["o_y"], s["o_bgr"][..., 1]) for s in sets))
    return nb, forms, fields


def rgba_forms(w, h, ow, oh, scale, n):
    nb = sets_for(n * (w * h + ow * oh) * 3)   # enough BGR sets to exceed L2; the BGRA sets are then 4/3 larger still
    sets = []
    for i in range(nb):
        q = rgba_seeded(i, (n, h, w))
        sets.append(dict(bgra=q, bgr=q[..., :3].contiguous(), o_bgra=zeros(n, oh, ow, 4), o_bgr=zeros(n, oh, ow, 3)))
    forms = dict(bgr=whole(sets, "bgr", "o_bgr", S.ORDER_BGR, scale, n), bgra=whole(sets, "bgra", "o_bgra", S.ORDER_BGRA, scale, n))

    def fields(t):
        c, q = t["bgr"], t["bgra"]
        return dict(bgr_ms_per_frame=round(c, 4), bgra_ms_per_frame=round(q, 4), bgra_over_bgr=round(q / c, 3),
                    bgra_colour_bytes_equal_bgr=all(torch.equal(s["o_bgra"][..., :3], s["o_bgr"]) for s in sets))
    return nb, forms, fields


def pack420(y, u, v, order):
    """N x (H*3/2) x W device frames from N x H x W / N x H/2 x W/2 planes"""
    n, h, w = y.shape
    f = torch.empty((n, h * 3 // 2, w), dtype=torch.uint8, device="cuda")
    f[:, :h] = y
    if order == S.ORDER_NV12:
        f[:, h:] = torch.stack([u, v], dim=-1).reshape(n, h // 2, w)
    else:
        f[:, h:].view(n, -1)[:] = torch.cat([u.reshape(n, -1), v.reshape(n, -1)], dim=1)
    return f


def pack422(y, u, v, order):
    """N x H x W x 2 device frames from N x H x W / N x H x W/2 planes"""
    n, h, w = y.shape
    f = torch.empty((n, h, w, 2), dtype=torch.uint8, device="cuda")
    for i in range(n):
        fy, fu, fv = S.yuv422_planes(f[i], order)
        fy.copy_(y[i])
        fu.copy_(u[i])
        fv.copy_(v[i])
    return f


def yuv_forms(fmt, w, h, ow, oh, scale, n):
    if fmt == "yuv420":
        (a, oa), (b, ob) = ("nv12", S.ORDER_NV12), ("i420", S.ORDER_I420)
        ch, och, frame, pack, planes = (h // 2, w // 2), (oh // 2, ow // 2), (oh * 3 // 2, ow), pack420, S.yuv420_planes
        nb = sets_for(n * (w * h + ow * oh) * 3 // 2)
    else:
        (a, oa), (b, ob) = ("yuy2", S.ORDER_YUY2), ("uyvy", S.ORDER_UYVY)
        ch, och, frame, pack, planes = (h, w // 2), (oh, ow // 2), (oh, ow, 2), pack422, S.yuv422_planes
        nb = sets_for(n * (w * h + ow * oh) * 2)
    g = torch.Generator(device="cuda").manual_seed(0)
    rnd = lambda *shape: torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=g)
    sets = []
    for _ in range(nb):
        y, u, v = rnd(n, h, w), rnd(n, *ch), rnd(n, *ch)
        sets.append({"y": y, "u": u, "v": v, a: pack(y, u, v, oa), b: pack(y, u, v, ob), "bgr": rnd(n, h, w, 3), "o_" + a: zeros(n, *frame),
                     "o_" + b: zeros(n, *frame), "o_y": zeros(n, oh, ow), "o_u": zeros(n, *och), "o_v": zeros(n, *och),
                     "o_bgr": zeros(n, oh, ow, 3)})

    def composition(s):
        (eng.process_device(s["y"][0], scale, s["o_y"][0], order=S.ORDER_GRAY) if n == 1 else
         eng.process_batch_device(s["y"], scale, s["o_y"], order=S.ORDER_GRAY))
        for f in range(n):
            eng.stage_resize_plane(s["u"][f], scale, s["o_u"][f])
            eng.stage_resize_plane(s["v"][f], scale, s["o_v"][f])

    forms = {a: whole(sets, a, "o_" + a, oa, scale, n), b: whole(sets, b, "o_" + b, ob, scale, n),
             "grey": whole(sets, "y", "o_y", S.ORDER_GRAY, scale, n), "bgr": whole(sets, "bgr", "o_bgr", S.ORDER_BGR, scale, n),
             "composition": [lambda s=s: composition(s) for s in sets]}

    def fields(t):
        same = True
        for s in sets:
            for key, order in (("o_" + a, oa), ("o_" + b, ob)):
                for f in range(n):
                    yy, uu, vv = planes(s[key][f], order)
                    same &= torch.equal(yy, s["o_y"][f]) and torch.equal(uu, s["o_u"][f]) and torch.equal(vv, s["o_v"][f])
        return {**{k + "_ms_per_frame": round(v, 4) for k, v in t.items()}, a + "_over_grey": round(t[a] / t["grey"], 3),
                a + "_over_bgr": round(t[a] / t["bgr"], 3), a + "_over_composition": round(t[a] / t["composition"], 3),
                b + "_over_" + a: round(t[b] / t[a], 3), "bytes_equal_composition": bool(same)}
    return nb, forms, fields


def graya_forms(w, h, ow, oh, scale, n):
    nb = sets_for(n * (w * h + ow * oh) * 2)
    g = torch.Generator(device="cuda").manual_seed(0)
    rnd = lambda *shape: torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=g)
    sets = []
    for _ in range(nb):
        y, a = rnd(n, h, w), rnd(n, h, w)
        sets.append(dict(y=y, a=a, ga=torch.stack([y, a], dim=-1).contiguous(), bgr=rnd(n, h, w, 3), o_ga=zeros(n, oh, ow, 2),
                         o_y=zeros(n, oh, ow), o_a=zeros(n, oh, ow), o_bgr=zeros(n, oh, ow, 3)))

    def composition(s):
        (eng.process_device(s["y"][0], scale, s["o_y"][0], order=S.ORDER_GRAY) if n == 1 else
         eng.process_batch_device(s["y"], scale, s["o_y"], order=S.ORDER_GRAY))
        for f in range(n):
            eng.stage_resize_plane(s["a"][f], scale, s["o_a"][f])

    forms = dict(graya=whole(sets, "ga", "o_ga", S.ORDER_GRAYA, scale, n), grey=whole(sets, "y", "o_y", S.ORDER_GRAY, scale, n),
                 bgr=whole(sets, "bgr", "o_bgr", S.ORDER_BGR, scale, n), composition=[lambda s=s: composition(s) for s in sets])

    def fields(t):
        same = all(torch.equal(s["o_ga"][..., 0], s["o_y"]) and torch.equal(s["o_ga"][..., 1], s["o_a"]) for s in sets)
        return {**{k + "_ms_per_frame": round(v, 4) for k, v in t.items()}, "graya_over_grey": round(t["graya"] / t["grey"], 3),
                "graya_over_bgr": round(t["graya"] / t["bgr"], 3), "graya_over_composition": round(t["graya"] / t["composition"], 3),
                "bytes_equal_composition": bool(same)}
    return nb, forms, fields


FORMS = dict(gray=gray_forms, rgba=rgba_forms, yuv420=lambda *a: yuv_forms("yuv420", *a), yuv422=lambda *a: yuv_forms("yuv422", *a),
             graya=graya_forms)


def device_line(fmt, name, w, h, scale, n, rounds):
    ow, oh = S.out_dims(w, h, scale)
    nb, forms, fields = FORMS[fmt](w, h, ow, oh, scale, n)
    ms = {k: [] for k in forms}
    for _ in range(rounds):   # alternate, so that drift of the box hits every form alike
        for k, calls in forms.items():
            ms[k].append(time_blocks(calls, 3))
    t = {k: float(np.median(v)) / (nb * n) for k, v in ms.items()}
    emit(line=name, src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, frames_per_call=n, buffer_sets=nb, **fields(t))
    del forms, fields
    torch.cuda.empty_cache()


# ---- host lines
def host_ms(src_bytes, w, h, stride, order, scale, dst_bytes, dstride, reps):
    """median ms of srcnn_process_host on pinned buffers; -> (ms, the result bytes)"""
    src, dst = S.PinnedBuffer(src_bytes.size), S.PinnedBuffer(dst_bytes)
    src.array[:] = src_bytes
    call = lambda: eng._check(eng.L.srcnn_process_host(eng.ctx, src.ptr, w, h, stride, order, C.c_float(scale), dst.ptr, dstride))
    for _ in range(3):
        call()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        call()
        ts.append(time.perf_counter() - t0)
    out = dst.array.copy()
    src.free()
    dst.free()
    return float(np.median(ts)) * 1e3, out


def host_line(fmt, w, h, scale, reps):
    ow, oh = S.out_dims(w, h, scale)
    head = dict(line="host_e2e", src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale)
    if fmt == "gray":
        g = np.random.default_rng(2).integers(0, 256, (h, w), dtype=np.uint8)
        c, cb = host_ms(np.repeat(g[..., None], 3, axis=2).reshape(-1), w, h, w * 3, S.ORDER_BGR, scale, ow * oh * 3, ow * 3, reps)
        y, yb = host_ms(g.reshape(-1), w, h, w, S.ORDER_GRAY, scale, ow * oh, ow, reps)
        emit(**head, colour_ms=round(c, 4), grey_ms=round(y, 4), grey_over_colour=round(y / c, 3),
             grey_bytes_equal_colour_G=bool(np.array_equal(yb, cb.reshape(oh, ow, 3)[..., 1].reshape(-1))))
    elif fmt == "rgba":
        img = rgba_seeded(100, (1, h, w))[0].cpu().numpy()
        c, cb = host_ms(np.ascontiguousarray(img[..., :3]).reshape(-1), w, h, w * 3, S.ORDER_BGR, scale, ow * oh * 3, ow * 3, reps)
        q, qb = host_ms(img.reshape(-1), w, h, w * 4, S.ORDER_BGRA, scale, ow * oh * 4, ow * 4, reps)
        emit(**head, bgr_ms=round(c, 4), bgra_ms=round(q, 4), bgra_over_bgr=round(q / c, 3),
             bgra_colour_bytes_equal_bgr=bool(np.array_equal(qb.reshape(oh, ow, 4)[..., :3], cb.reshape(oh, ow, 3))))
    elif fmt == "graya":
        rng = np.random.default_rng(2)
        ga = rng.integers(0, 256, (h, w, 2), dtype=np.uint8)
        c, _ = host_ms(rng.integers(0, 256, w * h * 3, dtype=np.uint8), w, h, w * 3, S.ORDER_BGR, scale, ow * oh * 3, ow * 3, reps)
        y, yb = host_ms(np.ascontiguousarray(ga[..., 0]).reshape(-1), w, h, w, S.ORDER_GRAY, scale, ow * oh, ow, reps)
        q, qb = host_ms(ga.reshape(-1), w, h, w * 2, S.ORDER_GRAYA, scale, ow * oh * 2, ow * 2, reps)
        emit(**head, bgr_ms=round(c, 4), grey_ms=round(y, 4), graya_ms=round(q, 4), graya_over_bgr=round(q / c, 3),
             graya_over_grey=round(q / y, 3), graya_grey_bytes_equal_grey=bool(np.array_equal(qb.reshape(oh, ow, 2)[..., 0], yb.reshape(oh, ow))))
    else:   # 4:2:0: h * 3/2 rows of w bytes; 4:2:2: h rows of 2w bytes
        if fmt == "yuv420":
            name, order, src_bytes, stride, dst_bytes, dstride = "nv12", S.ORDER_NV12, w * h * 3 // 2, w, ow * oh * 3 // 2, ow
        else:
            name, order, src_bytes, stride, dst_bytes, dstride = "yuy2", S.ORDER_YUY2, w * h * 2, w * 2, ow * oh * 2, ow * 2
        rng = np.random.default_rng(2)
        c, _ = host_ms(rng.integers(0, 256, w * h * 3, dtype=np.uint8), w, h, w * 3, S.ORDER_BGR, scale, ow * oh * 3, ow * 3, reps)
        v, _ = host_ms(rng.integers(0, 256, src_bytes, dtype=np.uint8), w, h, stride, order, scale, dst_bytes, dstride, reps)
        emit(**head, bgr_ms=round(c, 4), **{name + "_ms": round(v, 4), name + "_over_bgr": round(v / c, 3)})


# ---- format-specific lines
def stage_line(w, h, scale, rounds):
    ow, oh = S.out_dims(w, h, scale)
    rng = np.random.default_rng(1)
    nb = sets_for(w * h + ow * oh, hi=16)
    srcs = [torch.from_numpy(rng.integers(0, 256, (h, w), dtype=np.uint8)).cuda() for _ in range(nb)]
    dsts = [zeros(oh, ow) for _ in range(nb)]
    calls = [lambda i=i: eng.stage_resize_plane(srcs[i], scale, dsts[i]) for i in range(nb)]
    ms = float(np.median([time_blocks(calls, 3) for _ in range(rounds)])) / nb
    nbytes = w * h + ow * oh
    emit(line="stage_resize_plane", src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, us=round(ms * 1e3, 2),
         bytes=nbytes, TBps=round(nbytes / (ms * 1e-3) / 1e12, 3), share_of_hbm_peak=round(nbytes / (ms * 1e-3) / HBM_PEAK, 3))


def process_srcnn_line(w, h, scale, reps, d=4):
    fn = S.load_library()._Z12ProcessSRCNNPKhjjjfRPhRj
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint, C.c_float, C.POINTER(C.c_void_p), C.POINTER(C.c_uint)]
    ow, oh = S.out_dims(w, h, scale)
    rgba = rgba_seeded(101, (1, h, w))[0].cpu().numpy()
    if d == 2:   # grey + alpha: the G and alpha bytes of the same image
        rgba = np.ascontiguousarray(rgba[..., 1::2])

    def before():   # the old composition, step by step
        col = np.ascontiguousarray(rgba[..., :d - 1]) if d == 4 else np.ascontiguousarray(rgba[..., 0])
        alpha = np.ascontiguousarray(rgba[..., d - 1])
        out = np.empty((oh, ow, d), np.uint8)
        if d == 4:
            out[..., :3] = eng.process(col, scale, order=S.ORDER_RGB)
        else:
            out[..., 0] = eng.process(col, scale, order=S.ORDER_GRAY)
        out[..., d - 1] = eng.resize_plane(alpha, scale)
        return out

    def after():
        out, sz = C.c_void_p(), C.c_uint()
        if fn(rgba.ctypes.data, w, h, d, C.c_float(scale), C.byref(out), C.byref(sz)) != 0:
            raise RuntimeError("ProcessSRCNN failed")
        # the caller delete[]s the buffer in C++; here it is copied out and left to the process (a few calls of a benchmark)
        return np.ctypeslib.as_array((C.c_uint8 * sz.value).from_address(out.value)).reshape(oh, ow, d).copy()

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
    extra = {}
    if d == 4:
        extra["colour_bytes_equal_bgr_path"] = bool(np.array_equal(after()[..., :3], eng.process(np.ascontiguousarray(rgba[..., :3]),
                                                                                                 scale, order=S.ORDER_RGB)))
    emit(line="ProcessSRCNN_d%d" % d, src="%dx%d" % (w, h), dst="%dx%d" % (ow, oh), scale=scale, before_ms=round(b, 3), after_ms=round(a, 3),
         after_over_before=round(a / b, 3), bytes_equal=bool(np.array_equal(before(), after())), **extra)


R = 3 if ARGS.quick else 7
for fmt in FORMATS if ARGS.format == "all" else (ARGS.format,):
    device_line(fmt, "1080p_to_4K_x2", 1920, 1080, 2.0, 1, R)
    device_line(fmt, "720p_to_1440p_x2_batch", 1280, 720, 2.0, 32 if ARGS.quick else 256, R)
    device_line(fmt, "4K_to_16K_x4", 3840, 2160, 4.0, 1, R)
    device_line(fmt, "1080p_x1.5", 1920, 1080, 1.5, 1, R)
    if fmt == "gray":
        stage_line(1920, 1080, 2.0, R)
        stage_line(3840, 2160, 4.0, R)
        stage_line(1920, 1080, 1.5, R)
    host_line(fmt, 1920, 1080, 2.0, 10 if ARGS.quick else 30)
    if fmt in ("rgba", "graya"):
        process_srcnn_line(1920, 1080, 2.0, 5 if ARGS.quick else 15, d=4 if fmt == "rgba" else 2)
eng.close()
