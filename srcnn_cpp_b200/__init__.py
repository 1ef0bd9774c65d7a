"""srcnn_cpp_b200 -- Python front-end of libsrcnn_b200.so (the B200-native SRCNN_Cpp hot path).

The product is the CUDA library behind the C ABI in include/srcnn_b200.h; this module is only the
ctypes binding the tests and bench.py use (PyTorch supplies device buffers, streams and
torch.distributed -- plumbing, not the product).  The reference's own host side is C++ and so is
ours: cli/srcnn_main.cpp (bin/srcnn) and include/libsrcnn.h (ProcessSRCNN).

There is NO CPU fallback and no import of oracle/: if the shared library is missing, or no sm_100
device is present, construction fails loudly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsrcnn_b200.so")

VARIANT_TC = 0
VARIANT_FP32 = 1
ORDER_BGR = 0
ORDER_RGB = 1
ORDER_GRAY = 2   # one channel: HxW (NxHxW) arrays and tensors in and out; the result is the CNN's Y'
ORDER_BGRA = 3   # four channels, straight alpha in byte 3: HxWx4 (NxHxWx4) in and out; colour bytes = the BGR call's,
ORDER_RGBA = 4   # alpha = the one-plane cubic resize of the alpha plane (no CNN)
ORDER_NV12 = 6   # packed 4:2:0 video frames: (H*3/2)xW ((N)x(H*3/2)xW) arrays and tensors in and out; Y plane = the grey call's,
ORDER_I420 = 7   # chroma planes = the one-plane cubic resize of the source's (no CNN).  yuv420_planes() splits a frame
ORDER_YUY2 = 8   # packed 4:2:2 (bytes Y0 U Y1 V / U Y0 V Y1): HxWx2 (NxHxWx2) arrays and tensors in and out, OpenCV's CV_8UC2 shape;
ORDER_UYVY = 9   # Y plane = the grey call's, U / V = the one-plane cubic resize of the source's.  yuv422_planes() splits a frame
ORDER_GRAYA = 10   # grey + straight alpha (bytes G A): HxWx2 (NxHxWx2) arrays and tensors in and out; byte 0 = the grey call's,
                   # byte 1 = the one-plane cubic resize of the alpha plane (no CNN).  img[..., 0] / img[..., 1] are the planes

OK = 0
E_RATIO = -1
E_ARG = -20
E_NODEVICE = -30
E_CUDA = -31
E_NOMEM = -32
E_KERNEL = -33

# every symbol include/srcnn_b200.h declares (tests/test_abi.py checks the library exports them all)
ABI_SYMBOLS = [
    "srcnn_abi_version", "srcnn_strerror", "srcnn_create", "srcnn_destroy", "srcnn_last_error",
    "srcnn_set_variant", "srcnn_get_variant", "srcnn_set_stream", "srcnn_get_stream", "srcnn_sync",
    "srcnn_launch_count", "srcnn_device_sm_count", "srcnn_profile_enable", "srcnn_profile_read", "srcnn_out_dims", "srcnn_host_alloc", "srcnn_host_free",
    "srcnn_process_host", "srcnn_process_device", "srcnn_process_batch_device", "srcnn_process_batch_host",
    "srcnn_band_src_rows", "srcnn_process_band_device", "srcnn_stage_color_bicubic_device",
    "srcnn_stage_cnn_device", "srcnn_stage_conv99x11_fp32_device", "srcnn_stage_merge_device",
    "srcnn_fraw_scale_device",
    "srcnn_last_failed_stage", "srcnn_get_device", "srcnn_host_register", "srcnn_host_unregister",
    "srcnn_process_band_host", "srcnn_resize_plane_host", "srcnn_stage_resize_plane_device",
    "srcnn_mgpu_create", "srcnn_mgpu_destroy", "srcnn_mgpu_device_count", "srcnn_mgpu_context", "srcnn_mgpu_last_error",
    "srcnn_mgpu_band_plan", "srcnn_mgpu_process_batch_host", "srcnn_mgpu_process_banded_host",
    "srcnn_mgpu_process_batch_device", "srcnn_mgpu_process_banded_device", "srcnn_mgpu_last_timing",
    "srcnn_jpeg_stream_create", "srcnn_jpeg_stream_destroy", "srcnn_jpeg_stream_last_error", "srcnn_jpeg_stream_process", "srcnn_jpeg_free",
]


class SrcnnError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("srcnn status %d: %s" % (status, msg))
        self.status = status


_lib = None


def load_library():
    """dlopen libsrcnn_b200.so and declare the C ABI.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("SRCNN_B200_LIB", LIB_PATH)   # override: A/B runs of two builds of the library (tools/ab_libs.sh)
    if not os.path.exists(path):
        raise FileNotFoundError(
            path + " is missing: run `make` (or __graft_entry__.build()). There is no CPU fallback.")
    L = C.CDLL(path)
    vp, u8p, i32p, sz = C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.c_size_t
    L.srcnn_abi_version.restype = C.c_int
    L.srcnn_strerror.restype = C.c_char_p
    L.srcnn_strerror.argtypes = [C.c_int]
    L.srcnn_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int]
    L.srcnn_destroy.argtypes = [vp]
    L.srcnn_last_error.restype = C.c_char_p
    L.srcnn_last_error.argtypes = [vp]
    L.srcnn_set_variant.argtypes = [vp, C.c_int]
    L.srcnn_get_variant.argtypes = [vp]
    L.srcnn_set_stream.argtypes = [vp, vp]
    L.srcnn_get_stream.restype = vp
    L.srcnn_get_stream.argtypes = [vp]
    L.srcnn_sync.argtypes = [vp]
    L.srcnn_launch_count.restype = C.c_longlong
    L.srcnn_launch_count.argtypes = [vp]
    L.srcnn_device_sm_count.argtypes = [vp]
    L.srcnn_profile_enable.argtypes = [vp, C.c_int]
    L.srcnn_profile_read.argtypes = [vp, C.POINTER(C.c_double), i32p]
    L.srcnn_out_dims.argtypes = [C.c_int, C.c_int, C.c_float, i32p, i32p]
    L.srcnn_host_alloc.argtypes = [C.POINTER(vp), sz]
    L.srcnn_host_free.argtypes = [vp]
    L.srcnn_process_host.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_int, C.c_float, u8p, sz]
    L.srcnn_process_device.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_int, C.c_float, u8p, sz]
    L.srcnn_process_batch_device.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, sz, sz, C.c_int, C.c_float, u8p, sz, sz]
    L.srcnn_process_batch_host.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, sz, sz, C.c_int, C.c_float, u8p, sz, sz]
    L.srcnn_band_src_rows.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, i32p, i32p]
    L.srcnn_process_band_device.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_int, C.c_int, C.c_int, C.c_float,
                                            C.c_int, C.c_int, u8p, sz]
    L.srcnn_stage_color_bicubic_device.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_int, C.c_float, u8p, u8p, u8p, sz]
    L.srcnn_stage_cnn_device.argtypes = [vp, C.c_int, u8p, C.c_int, C.c_int, sz, u8p, sz]
    L.srcnn_stage_conv99x11_fp32_device.argtypes = [vp, u8p, C.c_int, C.c_int, sz, vp]
    L.srcnn_stage_merge_device.argtypes = [vp, u8p, u8p, u8p, C.c_int, C.c_int, sz, C.c_int, u8p, sz]
    L.srcnn_fraw_scale_device.argtypes = [vp, vp, C.c_uint, C.c_uint, C.c_uint, C.c_uint, vp, C.c_int]
    L.srcnn_last_failed_stage.argtypes = [vp]
    L.srcnn_get_device.argtypes = [vp]
    L.srcnn_host_register.argtypes = [vp, sz]
    L.srcnn_host_unregister.argtypes = [vp]
    L.srcnn_process_band_host.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_int, C.c_float, C.c_int, C.c_int, u8p, sz]
    L.srcnn_resize_plane_host.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_float, u8p, sz]
    L.srcnn_stage_resize_plane_device.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_float, u8p, sz]
    L.srcnn_mgpu_create.argtypes = [C.POINTER(vp), i32p, C.c_int, C.c_int]
    L.srcnn_mgpu_destroy.argtypes = [vp]
    L.srcnn_mgpu_device_count.argtypes = [vp]
    L.srcnn_mgpu_context.restype = vp
    L.srcnn_mgpu_context.argtypes = [vp, C.c_int]
    L.srcnn_mgpu_last_error.restype = C.c_char_p
    L.srcnn_mgpu_last_error.argtypes = [vp]
    L.srcnn_mgpu_band_plan.argtypes = [C.c_int, C.c_int, C.c_float, C.c_int, i32p, i32p, i32p, i32p]
    L.srcnn_mgpu_process_batch_host.argtypes = [vp, u8p, C.c_int, C.c_int, C.c_int, sz, sz, C.c_int, C.c_float, u8p, sz, sz]
    L.srcnn_mgpu_process_banded_host.argtypes = [vp, u8p, C.c_int, C.c_int, sz, C.c_int, C.c_float, u8p, sz]
    L.srcnn_mgpu_process_batch_device.argtypes = [vp, C.POINTER(vp), i32p, C.c_int, C.c_int, sz, sz, C.c_int, C.c_float,
                                                  C.POINTER(vp), sz, sz]
    L.srcnn_mgpu_process_banded_device.argtypes = [vp, C.POINTER(vp), C.c_int, C.c_int, sz, C.c_int, C.c_float, C.POINTER(vp), sz]
    L.srcnn_mgpu_last_timing.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.srcnn_jpeg_stream_create.argtypes = [C.POINTER(vp), vp, C.c_int]
    L.srcnn_jpeg_stream_destroy.argtypes = [vp]
    L.srcnn_jpeg_stream_last_error.restype = C.c_char_p
    L.srcnn_jpeg_stream_last_error.argtypes = [vp]
    L.srcnn_jpeg_stream_process.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(sz), C.c_int, C.c_float, C.POINTER(vp), C.POINTER(sz), i32p, i32p]
    L.srcnn_jpeg_free.restype = None
    L.srcnn_jpeg_free.argtypes = [vp]
    _lib = L
    return L


def out_dims(w, h, scale):
    """(ow, oh) = ((int)((float)w*scale), (int)((float)h*scale)) -- src/srcnn.cpp:573-575."""
    L = load_library()
    ow, oh = C.c_int(), C.c_int()
    rc = L.srcnn_out_dims(w, h, C.c_float(scale), C.byref(ow), C.byref(oh))
    if rc != OK:
        raise SrcnnError(rc, L.srcnn_strerror(rc).decode())
    return ow.value, oh.value


def band_src_rows(h, scale, r0, r1):
    L = load_library()
    s0, s1 = C.c_int(), C.c_int()
    rc = L.srcnn_band_src_rows(h, C.c_float(scale), r0, r1, C.byref(s0), C.byref(s1))
    if rc != OK:
        raise SrcnnError(rc, L.srcnn_strerror(rc).decode())
    return s0.value, s1.value


class PinnedBuffer:
    """Page-locked host memory from srcnn_host_alloc, viewed as a numpy uint8 array."""

    def __init__(self, nbytes):
        L = load_library()
        p = C.c_void_p()
        rc = L.srcnn_host_alloc(C.byref(p), nbytes)
        if rc != OK:
            raise SrcnnError(rc, "srcnn_host_alloc(%d)" % nbytes)
        self.ptr = p.value
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p.value))

    def free(self):
        if self.ptr:
            load_library().srcnn_host_free(self.ptr)
            self.ptr = None
            self.array = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _pixel_shape(order):
    """trailing shape of one pixel: () for ORDER_GRAY and the 4:2:0 orders, (4,) for ORDER_BGRA / ORDER_RGBA, (2,) for the 4:2:2
    orders and ORDER_GRAYA, (3,) for the colour orders"""
    if order in (ORDER_GRAY, ORDER_NV12, ORDER_I420):
        return ()
    if order in (ORDER_YUY2, ORDER_UYVY, ORDER_GRAYA):
        return (2,)
    return (4,) if order in (ORDER_BGRA, ORDER_RGBA) else (3,)


def _is_yuv420(order):
    return order in (ORDER_NV12, ORDER_I420)


def _frame_h(order, rows):
    """image height of a frame of `rows` rows in memory: rows*2/3 for a 4:2:0 frame (Y rows, then h/2 chroma rows)"""
    if not _is_yuv420(order):
        return rows
    if rows % 3:
        raise SrcnnError(E_ARG, "a 4:2:0 frame has H*3/2 rows; %d is not a multiple of 3" % rows)
    return rows * 2 // 3


def _out_rows(order, oh):
    return oh * 3 // 2 if _is_yuv420(order) else oh


def yuv420_planes(frame, order):
    """(Y, U, V) views of one packed 4:2:0 frame: an (H*3/2)xW uint8 numpy array or torch tensor whose rows may be padded
    (row stride >= W; I420: even).  NV12: U and V are the even / odd bytes of the interleaved chroma rows.  I420: H/2 x W/2 planes
    whose rows are stride/2 apart, V after U."""
    if order not in (ORDER_NV12, ORDER_I420) or len(frame.shape) != 2:
        raise SrcnnError(E_ARG, "expected one (H*3/2)xW frame and ORDER_NV12 / ORDER_I420")
    rows, w = frame.shape
    h = _frame_h(order, rows)
    y, c = frame[:h], frame[h:]
    if order == ORDER_NV12:
        return y, c[:, 0::2], c[:, 1::2]
    torch_like = hasattr(frame, "storage_offset")
    s = frame.stride(0) if torch_like else frame.strides[0]
    if s % 2:
        raise SrcnnError(E_ARG, "I420 rows must be an even number of bytes apart")
    shape, first, second = (h // 2, w // 2), h * s, h * s + (h // 2) * (s // 2)
    if torch_like:
        o = frame.storage_offset()
        return y, frame.as_strided(shape, (s // 2, 1), o + first), frame.as_strided(shape, (s // 2, 1), o + second)
    flat = np.lib.stride_tricks.as_strided(frame, shape=(second + (h // 2) * (s // 2),), strides=(1,))
    as_plane = lambda k: np.lib.stride_tricks.as_strided(flat[k:], shape=shape, strides=(s // 2, 1))
    return y, as_plane(first), as_plane(second)


def yuv422_planes(frame, order):
    """(Y, U, V) views of one packed 4:2:2 frame: an HxWx2 uint8 numpy array or torch tensor (W even; rows may be padded).  Y is
    HxW (byte 0 of each pixel with ORDER_YUY2, byte 1 with ORDER_UYVY), U and V are HxW/2 (bytes 1 / 3 of each 4-byte macropixel
    with ORDER_YUY2, bytes 0 / 2 with ORDER_UYVY).  Strided views of the frame's memory, not copies."""
    if order not in (ORDER_YUY2, ORDER_UYVY) or len(frame.shape) != 3 or frame.shape[2] != 2 or frame.shape[1] % 2:
        raise SrcnnError(E_ARG, "expected one HxWx2 frame with an even W and ORDER_YUY2 / ORDER_UYVY")
    y_byte, u_byte = (0, 1) if order == ORDER_YUY2 else (1, 0)
    mp = frame[:, 0::2, :]                       # H x W/2 x 2: the first two bytes of each macropixel
    mq = frame[:, 1::2, :]                       # ... and the last two
    return frame[:, :, y_byte], mp[:, :, u_byte], mq[:, :, u_byte]


def _check_host_image(a, order, lead):
    """a: numpy uint8 array of `lead` leading dims (1: HxW[xC], 2: NxHxW[xC]) in the layout `order` implies"""
    px = _pixel_shape(order)
    if a.dtype != np.uint8 or a.ndim != lead + 1 + len(px) or tuple(a.shape[lead + 1:]) != px:
        raise SrcnnError(E_ARG, "expected a %s uint8 array" % ("x".join(["N"] * (lead - 1) + ["H", "W"] + [str(c) for c in px])))


def _dptr(t):
    """device pointer of a torch CUDA uint8/float tensor (must be contiguous in its last dim)"""
    return C.c_void_p(t.data_ptr())


class Engine:
    """One srcnn_ctx: a device, a stream, workspace and packed weights (include/srcnn_b200.h)."""

    def __init__(self, device=0, variant=VARIANT_TC, stream=None):
        self.L = load_library()
        self.ctx = C.c_void_p()
        rc = self.L.srcnn_create(C.byref(self.ctx), int(device), int(variant))
        if rc != OK:
            self.ctx = None
            raise SrcnnError(rc, self.L.srcnn_strerror(rc).decode())
        self.device = int(device)
        if stream is not None:
            self.set_stream(stream)

    def close(self):
        if getattr(self, "ctx", None):
            self.L.srcnn_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise SrcnnError(rc, (self.L.srcnn_last_error(self.ctx) or b"").decode() or self.L.srcnn_strerror(rc).decode())

    # -- context knobs ---------------------------------------------------------------------------
    def set_variant(self, variant):
        self._check(self.L.srcnn_set_variant(self.ctx, int(variant)))

    def set_stream(self, cuda_stream_ptr):
        """cuda_stream_ptr: int (cudaStream_t), e.g. torch.cuda.current_stream().cuda_stream; 0/None = own stream"""
        self._check(self.L.srcnn_set_stream(self.ctx, C.c_void_p(cuda_stream_ptr or None)))

    def sync(self):
        self._check(self.L.srcnn_sync(self.ctx))

    def profile_enable(self, on=True):
        """on: False / True (events around all three stages: the stages then run strictly one after another) / 2 (events around
        the CNN stage only: the merge of one call and the colour+bicubic of the next stay adjacent and may overlap)"""
        self._check(self.L.srcnn_profile_enable(self.ctx, 2 if on == 2 else (1 if on else 0)))

    def profile_read(self):
        """-> ([ms colour+bicubic, ms fused SRCNN, ms merge], number of whole-path calls); in mode 2: [ms between consecutive CNN
        launches (merge of call i beside colour+bicubic of call i+1), ms fused SRCNN, 0]"""
        ms = (C.c_double * 3)()
        n = C.c_int()
        self._check(self.L.srcnn_profile_read(self.ctx, ms, C.byref(n)))
        return [ms[0], ms[1], ms[2]], n.value

    @property
    def launches(self):
        return int(self.L.srcnn_launch_count(self.ctx))

    @property
    def sm_count(self):
        return int(self.L.srcnn_device_sm_count(self.ctx))

    # -- whole path, host buffers (numpy) ----------------------------------------------------------
    def process(self, img, scale, order=ORDER_BGR, out=None):
        """img: HxWx3 uint8 numpy array (BGR by default, like cv::imread), HxW with order=ORDER_GRAY, HxWx4 with
        order=ORDER_BGRA / ORDER_RGBA, an (H*3/2)xW frame with ORDER_NV12 / ORDER_I420, or HxWx2 with ORDER_YUY2 / ORDER_UYVY /
        ORDER_GRAYA.
        Returns OHxOWx3 (OHxOW, OHxOWx4, (OH*3/2)xOW, OHxOWx2) uint8."""
        img = np.asarray(img)
        _check_host_image(img, order, 1)
        if not img.flags.c_contiguous:
            img = np.ascontiguousarray(img)
        h, w = _frame_h(order, img.shape[0]), img.shape[1]
        ow, oh = out_dims(w, h, scale)
        if out is None:
            out = np.empty((_out_rows(order, oh), ow) + _pixel_shape(order), np.uint8)
        self._check(self.L.srcnn_process_host(self.ctx, img.ctypes.data, w, h, img.strides[0], order, C.c_float(scale),
                                              out.ctypes.data, out.strides[0]))
        return out

    def process_batch(self, frames, scale, order=ORDER_BGR, out=None):
        """frames: NxHxWx3 (NxHxW with order=ORDER_GRAY, NxHxWx4 with ORDER_BGRA / ORDER_RGBA, NxHxWx2 with ORDER_YUY2 /
        ORDER_UYVY / ORDER_GRAYA) uint8 numpy array -> NxOHxOWx3 (NxOHxOW, NxOHxOWx4, NxOHxOWx2)."""
        frames = np.ascontiguousarray(frames)
        _check_host_image(frames, order, 2)
        n, h, w = frames.shape[0], _frame_h(order, frames.shape[1]), frames.shape[2]
        ow, oh = out_dims(w, h, scale)
        if out is None:
            out = np.empty((n, _out_rows(order, oh), ow) + _pixel_shape(order), np.uint8)
        self._check(self.L.srcnn_process_batch_host(self.ctx, frames.ctypes.data, n, w, h, frames.strides[1],
                                                    frames.strides[0], order, C.c_float(scale), out.ctypes.data,
                                                    out.strides[1], out.strides[0]))
        return out

    # -- whole path, device buffers (torch CUDA tensors) -------------------------------------------
    def process_device(self, src, scale, dst, order=ORDER_BGR):
        """src: HxWx3 (HxW with order=ORDER_GRAY, HxWx4 with ORDER_BGRA / ORDER_RGBA) uint8 device tensor; dst: OHxOWx3
        (OHxOW, OHxOWx4); (H*3/2)xW and (OH*3/2)xOW frames with ORDER_NV12 / ORDER_I420; HxWx2 and OHxOWx2 with ORDER_YUY2 /
        ORDER_UYVY / ORDER_GRAYA."""
        h, w = _frame_h(order, src.shape[0]), src.shape[1]
        self._check(self.L.srcnn_process_device(self.ctx, _dptr(src), w, h, src.stride(0), order, C.c_float(scale),
                                                _dptr(dst), dst.stride(0)))
        return dst

    def process_batch_device(self, src, scale, dst, order=ORDER_BGR):
        n, h, w = src.shape[0], _frame_h(order, src.shape[1]), src.shape[2]
        self._check(self.L.srcnn_process_batch_device(self.ctx, _dptr(src), n, w, h, src.stride(1), src.stride(0), order,
                                                      C.c_float(scale), _dptr(dst), dst.stride(1), dst.stride(0)))
        return dst

    def process_band_device(self, src_rows, w, h, s0, s1, scale, r0, r1, dst_rows, order=ORDER_BGR):
        """src_rows: (s1-s0)xWx3 device tensor holding source rows [s0,s1); dst_rows: (r1-r0)xOWx3 (no x3 with ORDER_GRAY, x4
        with ORDER_BGRA / ORDER_RGBA, x2 with ORDER_YUY2 / ORDER_UYVY / ORDER_GRAYA)."""
        self._check(self.L.srcnn_process_band_device(self.ctx, _dptr(src_rows), w, h, src_rows.stride(0), s0, s1, order,
                                                     C.c_float(scale), r0, r1, _dptr(dst_rows), dst_rows.stride(0)))
        return dst_rows

    # -- stages (torch CUDA tensors) ---------------------------------------------------------------
    def stage_color_bicubic(self, src, scale, y, cr, cb, order=ORDER_BGR):
        h, w, _ = src.shape
        self._check(self.L.srcnn_stage_color_bicubic_device(self.ctx, _dptr(src), w, h, src.stride(0), order,
                                                            C.c_float(scale), _dptr(y), _dptr(cr), _dptr(cb), y.stride(0)))

    def stage_resize_plane(self, src, scale, dst):
        """One HxW uint8 device plane through the path's cubic resize (cv::resize INTER_CUBIC) into dst (OHxOW, any stride)."""
        h, w = src.shape
        self._check(self.L.srcnn_stage_resize_plane_device(self.ctx, _dptr(src), w, h, src.stride(0), C.c_float(scale),
                                                           _dptr(dst), dst.stride(0)))
        return dst

    def stage_cnn(self, y, out, variant=None):
        h, w = y.shape
        v = self.L.srcnn_get_variant(self.ctx) if variant is None else variant
        self._check(self.L.srcnn_stage_cnn_device(self.ctx, int(v), _dptr(y), w, h, y.stride(0), _dptr(out), out.stride(0)))
        return out

    def set_host_bands(self, bands):
        """Tuning hook: most sub-bands the host-buffer pipeline cuts a single frame into."""
        self.L.srcnn_debug_set_host_bands.argtypes = [C.c_void_p, C.c_int]
        self._check(self.L.srcnn_debug_set_host_bands(self.ctx, int(bands)))

    def process_band_host(self, img, scale, r0, r1, out_rows=None, order=ORDER_BGR):
        """img: the WHOLE HxWx3 (HxW, HxWx4, HxWx2) source image; returns output rows [r0, r1) as an (r1-r0)xOWx3 ((r1-r0)xOW,
        (r1-r0)xOWx4, (r1-r0)xOWx2) array."""
        img = np.ascontiguousarray(img)
        _check_host_image(img, order, 1)
        h, w = img.shape[:2]
        ow, oh = out_dims(w, h, scale)
        if out_rows is None:
            out_rows = np.empty((r1 - r0, ow) + _pixel_shape(order), np.uint8)
        self._check(self.L.srcnn_process_band_host(self.ctx, img.ctypes.data, w, h, img.strides[0], order, C.c_float(scale),
                                                   r0, r1, out_rows.ctypes.data, out_rows.strides[0]))
        return out_rows

    def resize_plane(self, plane, scale):
        """One uint8 plane through the path's cubic resize (cv::resize INTER_CUBIC semantics), host buffers."""
        plane = np.ascontiguousarray(plane)
        h, w = plane.shape
        ow, oh = out_dims(w, h, scale)
        out = np.empty((oh, ow), np.uint8)
        self._check(self.L.srcnn_resize_plane_host(self.ctx, plane.ctypes.data, w, h, plane.strides[0], C.c_float(scale),
                                                   out.ctypes.data, out.strides[0]))
        return out

    def set_tc2_seg_ovh(self, ovh):
        """Test hook: cost of opening a segment in the row-walking kernel's work cut (0 = equal row counts)."""
        self.L.srcnn_debug_set_tc2_seg_ovh.argtypes = [C.c_void_p, C.c_int]
        self._check(self.L.srcnn_debug_set_tc2_seg_ovh(self.ctx, int(ovh)))

    def set_fuse_merge(self, on):
        """Test hook: merge + colour-back inside the fused tcgen05 kernel, or as a separate launch (default)."""
        self.L.srcnn_debug_set_fuse_merge.argtypes = [C.c_void_p, C.c_int]
        self._check(self.L.srcnn_debug_set_fuse_merge(self.ctx, int(bool(on))))

    def stage_conv99x11_fp32(self, y, act2):
        h, w = y.shape
        self._check(self.L.srcnn_stage_conv99x11_fp32_device(self.ctx, _dptr(y), w, h, y.stride(0), _dptr(act2)))
        return act2

    def fraw_scale(self, src, dst, filter=2):
        """frawscale-compatible resize of a float32 device plane (src/frawscale.cpp:162-286); filter 0/1/2 = box/bilinear/bicubic"""
        sh, sw = src.shape
        dh, dw = dst.shape
        self._check(self.L.srcnn_fraw_scale_device(self.ctx, _dptr(src), sw, sh, dw, dh, _dptr(dst), int(filter)))
        return dst

    def stage_merge(self, y, cr, cb, dst, order=ORDER_BGR):
        h, w = y.shape
        self._check(self.L.srcnn_stage_merge_device(self.ctx, _dptr(y), _dptr(cr), _dptr(cb), w, h, y.stride(0), order,
                                                    _dptr(dst), dst.stride(0)))
        return dst


def mgpu_band_plan(n_workers, h, scale, i):
    """Worker i's share of a banded image: (r0, r1, s0, s1).  Pure host arithmetic."""
    L = load_library()
    v = [C.c_int() for _ in range(4)]
    rc = L.srcnn_mgpu_band_plan(n_workers, h, C.c_float(scale), i, *[C.byref(x) for x in v])
    if rc != OK:
        raise SrcnnError(rc, L.srcnn_strerror(rc).decode())
    return tuple(x.value for x in v)


class MultiEngine:
    """srcnn_mgpu: a device list behind one call -- one host thread, context and stream set per device
    (include/srcnn_b200.h).  Frames go to worker f mod n, a single image is cut into n row bands."""

    def __init__(self, devices=None, variant=VARIANT_TC):
        self.L = load_library()
        self.h = C.c_void_p()
        if devices is None:
            arr, n = None, 0
        else:
            n = len(devices)
            arr = (C.c_int * n)(*devices)
        rc = self.L.srcnn_mgpu_create(C.byref(self.h), arr, n, int(variant))
        if rc != OK:
            self.h = None
            raise SrcnnError(rc, self.L.srcnn_strerror(rc).decode())
        self.n = int(self.L.srcnn_mgpu_device_count(self.h))
        self.devices = [int(self.L.srcnn_get_device(self.L.srcnn_mgpu_context(self.h, i))) for i in range(self.n)]

    def close(self):
        if getattr(self, "h", None):
            self.L.srcnn_mgpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise SrcnnError(rc, (self.L.srcnn_mgpu_last_error(self.h) or b"").decode() or self.L.srcnn_strerror(rc).decode())

    def set_variant(self, variant):
        for i in range(self.n):
            self.L.srcnn_set_variant(self.L.srcnn_mgpu_context(self.h, i), int(variant))

    def launches(self):
        return sum(int(self.L.srcnn_launch_count(self.L.srcnn_mgpu_context(self.h, i))) for i in range(self.n))

    def last_timing(self):
        """-> (per-worker ms of its share, wall ms of the call)"""
        ms = (C.c_double * self.n)()
        wall = C.c_double()
        self._check(self.L.srcnn_mgpu_last_timing(self.h, ms, C.byref(wall)))
        return list(ms), wall.value

    def band_plan(self, h, scale):
        return [mgpu_band_plan(self.n, h, scale, i) for i in range(self.n)]

    # -- host buffers (numpy, or raw pointers for pinned memory) -------------------------------------
    def process_banded(self, img, scale, order=ORDER_BGR, out=None):
        img = np.ascontiguousarray(img)
        _check_host_image(img, order, 1)
        h, w = img.shape[:2]
        ow, oh = out_dims(w, h, scale)
        if out is None:
            out = np.empty((oh, ow) + _pixel_shape(order), np.uint8)
        self._check(self.L.srcnn_mgpu_process_banded_host(self.h, img.ctypes.data, w, h, img.strides[0], order, C.c_float(scale),
                                                          out.ctypes.data, out.strides[0]))
        return out

    def process_batch(self, frames, scale, order=ORDER_BGR, out=None):
        frames = np.ascontiguousarray(frames)
        _check_host_image(frames, order, 2)
        n, h, w = frames.shape[0], _frame_h(order, frames.shape[1]), frames.shape[2]
        ow, oh = out_dims(w, h, scale)
        if out is None:
            out = np.empty((n, _out_rows(order, oh), ow) + _pixel_shape(order), np.uint8)
        self._check(self.L.srcnn_mgpu_process_batch_host(self.h, frames.ctypes.data, n, w, h, frames.strides[1], frames.strides[0],
                                                         order, C.c_float(scale), out.ctypes.data, out.strides[1], out.strides[0]))
        return out

    # -- device-resident shares (torch CUDA tensors, one per worker, each on that worker's device) -----
    def process_batch_device(self, srcs, scale, dsts, order=ORDER_BGR):
        """srcs[i]: n_i x H x W x 3 (no x 3 with ORDER_GRAY, x 4 with ORDER_BGRA / ORDER_RGBA, x 2 with ORDER_YUY2 / ORDER_UYVY /
        ORDER_GRAYA) on worker i's device (n_i may be
        0 -> pass None); dsts[i]: n_i x OH x OW x 3 (likewise)."""
        ref = next(t for t in srcs if t is not None)
        h, w = _frame_h(order, ref.shape[1]), ref.shape[2]
        dref = next(t for t in dsts if t is not None)
        ps = (C.c_void_p * self.n)(*[t.data_ptr() if t is not None else None for t in srcs])
        pd = (C.c_void_p * self.n)(*[t.data_ptr() if t is not None else None for t in dsts])
        cnt = (C.c_int * self.n)(*[t.shape[0] if t is not None else 0 for t in srcs])
        self._check(self.L.srcnn_mgpu_process_batch_device(self.h, ps, cnt, w, h, ref.stride(1), ref.stride(0), order, C.c_float(scale),
                                                           pd, dref.stride(1), dref.stride(0)))

    def process_banded_device(self, src_bands, w, h, scale, dst_bands, order=ORDER_BGR):
        """src_bands[i]: (s1_i-s0_i) x W x 3 (x 4, x 2, or no channel dim, per `order`) holding the source rows of band_plan()[i];
        dst_bands[i]: (r1_i-r0_i) x OW x 3 (likewise)."""
        ps = (C.c_void_p * self.n)(*[t.data_ptr() if t is not None else None for t in src_bands])
        pd = (C.c_void_p * self.n)(*[t.data_ptr() if t is not None else None for t in dst_bands])
        sref = next(t for t in src_bands if t is not None)
        dref = next(t for t in dst_bands if t is not None)
        self._check(self.L.srcnn_mgpu_process_banded_device(self.h, ps, w, h, sref.stride(0), order, C.c_float(scale), pd, dref.stride(0)))


class JpegStream:
    """srcnn_jpeg_stream: a stream of same-sized JPEG frames through decode -> whole path -> encode, all on the device."""

    def __init__(self, engine, quality=95):
        self.L, self.engine = engine.L, engine
        self.h = C.c_void_p()
        rc = self.L.srcnn_jpeg_stream_create(C.byref(self.h), engine.ctx, int(quality))
        if rc != OK:
            self.h = None
            raise SrcnnError(rc, self.L.srcnn_strerror(rc).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.srcnn_jpeg_stream_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def process(self, jpegs, scale):
        """jpegs: list of bytes objects -> (list of bytes objects, (ow, oh))"""
        n = len(jpegs)
        arr = (C.c_char_p * n)(*jpegs)
        sizes = (C.c_size_t * n)(*[len(j) for j in jpegs])
        out = (C.c_void_p * n)()
        osz = (C.c_size_t * n)()
        ow, oh = C.c_int(), C.c_int()
        rc = self.L.srcnn_jpeg_stream_process(self.h, arr, sizes, n, C.c_float(scale), out, osz, C.byref(ow), C.byref(oh))
        if rc != OK:
            raise SrcnnError(rc, (self.L.srcnn_jpeg_stream_last_error(self.h) or b"").decode())
        res = []
        for i in range(n):
            res.append(C.string_at(out[i], osz[i]))
            self.L.srcnn_jpeg_free(out[i])
        return res, (ow.value, oh.value)
