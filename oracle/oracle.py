"""ctypes front-end of the CHECKERS under oracle/ -- test infrastructure, never product code.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module.  The product package (srcnn_cpp_b200) must never import it.

Three checkers, strongest first:
  * RefLib      oracle/_ref/libref.so  -- the reference's own src/srcnn.cpp conv functions
                (Convolution99x11 src/srcnn.cpp:254-325, Convolution55 :189-243) compiled unmodified.
  * cv2 stages  python cv2 with IPP off = the OpenCV arithmetic the reference calls at
                src/srcnn.cpp:509, :540, :577-582, :639, :657 (third-party, not vendored).
  * Oracle      oracle/_build/liboracle.so -- our C restatement of the whole path (srcnn_oracle.c),
                pinned against the two above and the butterfly golden vector (tests/test_oracle.py).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
WEIGHTS_BIN = os.path.join(_ROOT, "srcnn_cpp_b200", "data", "srcnn_weights.bin")

_u8p = C.POINTER(C.c_uint8)
_f32p = C.POINTER(C.c_float)


def build(quiet=True):
    """(Re)build the checker libraries; _ref only when /root/reference is present."""
    subprocess.run(["make", "-C", _HERE], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def load_params():
    p = np.fromfile(WEIGHTS_BIN, dtype=np.float32)
    assert p.size == 8129, p.size
    return p


def _ptr(a, t):
    return a.ctypes.data_as(t)


class Oracle:
    """Our C restatement (oracle/srcnn_oracle.c)."""

    def __init__(self):
        path = os.path.join(_HERE, "_build", "liboracle.so")
        if not os.path.exists(path):
            build()
        L = self.lib = C.CDLL(path)
        L.orc_scaled_dim.restype = C.c_int
        L.orc_scaled_dim.argtypes = [C.c_int, C.c_float]
        L.orc_max_threads.restype = C.c_int
        L.orc_bgr2ycrcb.argtypes = [_u8p, C.c_size_t, C.c_int, C.c_int, _u8p, C.c_size_t]
        L.orc_ycrcb2bgr.argtypes = [_u8p, C.c_size_t, C.c_int, C.c_int, _u8p, C.c_size_t]
        L.orc_resize_cubic.argtypes = [_u8p, C.c_size_t, C.c_int, C.c_int, _u8p, C.c_size_t, C.c_int, C.c_int]
        L.orc_cubic_taps.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int16)]
        L.orc_conv99x11.argtypes = [_f32p, _u8p, C.c_int, C.c_int, _f32p]
        L.orc_conv55.argtypes = [_f32p, _f32p, C.c_int, C.c_int, _u8p]
        L.orc_cnn.restype = C.c_int
        L.orc_cnn.argtypes = [_f32p, _u8p, C.c_int, C.c_int, _u8p, _f32p]
        L.orc_pipeline.restype = C.c_int
        L.orc_pipeline.argtypes = [_f32p, _u8p, C.c_size_t, C.c_int, C.c_int, C.c_float, _u8p, C.c_size_t,
                                   _u8p, _u8p, _u8p, _u8p]
        vp = C.c_void_p
        L.orc_at_modes.restype = C.c_int
        L.orc_cnn_at.restype = C.c_int
        L.orc_cnn_at.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, vp, vp]
        L.orc_act2_at.restype = C.c_int
        L.orc_act2_at.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, vp]
        self.params = load_params()

    def threads(self):
        return int(self.lib.orc_max_threads())

    def out_dims(self, w, h, scale):
        return int(self.lib.orc_scaled_dim(w, scale)), int(self.lib.orc_scaled_dim(h, scale))

    def bgr2ycrcb(self, bgr):
        bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
        h, w, _ = bgr.shape
        out = np.empty_like(bgr)
        self.lib.orc_bgr2ycrcb(_ptr(bgr, _u8p), 3 * w, w, h, _ptr(out, _u8p), 3 * w)
        return out

    def ycrcb2bgr(self, ycc):
        ycc = np.ascontiguousarray(ycc, dtype=np.uint8)
        h, w, _ = ycc.shape
        out = np.empty_like(ycc)
        self.lib.orc_ycrcb2bgr(_ptr(ycc, _u8p), 3 * w, w, h, _ptr(out, _u8p), 3 * w)
        return out

    def resize_cubic(self, plane, dw, dh):
        plane = np.ascontiguousarray(plane, dtype=np.uint8)
        sh, sw = plane.shape
        out = np.empty((dh, dw), np.uint8)
        self.lib.orc_resize_cubic(_ptr(plane, _u8p), sw, sw, sh, _ptr(out, _u8p), dw, dw, dh)
        return out

    def cubic_taps(self, src, dst):
        ofs = np.empty(dst, np.int32)
        coef = np.empty((dst, 4), np.int16)
        self.lib.orc_cubic_taps(src, dst, _ptr(ofs, C.POINTER(C.c_int)), _ptr(coef, C.POINTER(C.c_int16)))
        return ofs, coef

    def conv99x11(self, y):
        y = np.ascontiguousarray(y, dtype=np.uint8)
        h, w = y.shape
        act2 = np.empty((32, h, w), np.float32)
        self.lib.orc_conv99x11(_ptr(self.params, _f32p), _ptr(y, _u8p), w, h, _ptr(act2, _f32p))
        return act2

    def conv55(self, act2):
        act2 = np.ascontiguousarray(act2, dtype=np.float32)
        _, h, w = act2.shape
        out = np.empty((h, w), np.uint8)
        self.lib.orc_conv55(_ptr(self.params, _f32p), _ptr(act2, _f32p), w, h, _ptr(out, _u8p))
        return out

    def cnn(self, y):
        y = np.ascontiguousarray(y, dtype=np.uint8)
        h, w = y.shape
        out = np.empty((h, w), np.uint8)
        rc = self.lib.orc_cnn(_ptr(self.params, _f32p), _ptr(y, _u8p), w, h, _ptr(out, _u8p), None)
        assert rc == 0
        return out

    # orc_cnn_at modes (oracle/srcnn_oracle.c): 0 is orc_cnn, the others near misses of its arithmetic
    AT_EXACT, AT_TEMP_DOUBLE, AT_INNER_FLOAT, AT_EXACT_PRODUCTS, AT_CHANNELS_REVERSED, AT_FMA_DOUBLE, AT_TAPS_NM, \
        AT_B3_DOUBLE, AT_CONV1_FMA, AT_CONV1_BIAS_FIRST, AT_CONV1_JI, AT_CONV2_FMA, AT_CONV2_REVERSED = range(13)

    def _at_args(self, y, rows, cols):
        y = np.ascontiguousarray(y, dtype=np.uint8)
        rows = np.ascontiguousarray(rows, dtype=np.int32).ravel()
        cols = np.ascontiguousarray(cols, dtype=np.int32).ravel()
        assert rows.shape == cols.shape
        return y, rows, cols

    def cnn_at(self, y, rows, cols, mode=0):
        """The CNN at pixels (rows[p], cols[p]) of the u8 plane y -> (temp + b3 as float32, the byte), both [n]"""
        y, rows, cols = self._at_args(y, rows, cols)
        h, w = y.shape
        v = np.empty(rows.size, np.float32)
        b = np.empty(rows.size, np.uint8)
        rc = self.lib.orc_cnn_at(self.params.ctypes.data, y.ctypes.data, w, h, rows.ctypes.data, cols.ctypes.data,
                                 rows.size, int(mode), v.ctypes.data, b.ctypes.data)
        assert rc == 0, (rc, mode)
        return v, b

    def act2_at(self, y, rows, cols, mode=0):
        """conv2's activations at the listed pixels, [n][32] float32 (mode 0 or a conv1 / conv2 near miss)"""
        y, rows, cols = self._at_args(y, rows, cols)
        h, w = y.shape
        out = np.empty((rows.size, 32), np.float32)
        rc = self.lib.orc_act2_at(self.params.ctypes.data, y.ctypes.data, w, h, rows.ctypes.data, cols.ctypes.data,
                                  rows.size, int(mode), out.ctypes.data)
        assert rc == 0, (rc, mode)
        return out

    def pipeline(self, bgr, scale, stages=False):
        """BGR8 HWC -> BGR8 HWC (the reference's timed region, src/srcnn.cpp:505-659)."""
        bgr = np.ascontiguousarray(bgr, dtype=np.uint8)
        h, w, _ = bgr.shape
        ow, oh = self.out_dims(w, h, scale)
        out = np.empty((oh, ow, 3), np.uint8)
        taps = [np.empty((oh, ow), np.uint8) for _ in range(4)] if stages else [None] * 4
        rc = self.lib.orc_pipeline(_ptr(self.params, _f32p), _ptr(bgr, _u8p), 3 * w, w, h, C.c_float(scale),
                                   _ptr(out, _u8p), 3 * ow,
                                   *[(_ptr(t, _u8p) if t is not None else None) for t in taps])
        if rc != 0:
            raise ValueError("orc_pipeline rc=%d" % rc)
        if stages:
            return out, dict(up_y=taps[0], up_cr=taps[1], up_cb=taps[2], cnn_y=taps[3])
        return out


class RefLib:
    """The reference's own conv code (oracle/_ref/libref.so, built by oracle/Makefile from
    /root/reference/src/srcnn.cpp, unmodified).  opt='O3' or 'O0' (the reference Makefile's flags)."""

    def __init__(self, opt="O3"):
        name = "libref.so" if opt == "O3" else "libref_O0.so"
        path = os.path.join(_HERE, "_ref", name)
        if not os.path.exists(path):
            if os.path.exists("/root/reference/src/srcnn.cpp"):
                build()
            else:
                raise FileNotFoundError(path + " (built only where /root/reference exists)")
        L = self.lib = C.CDLL(path)
        L.ref_max_threads.restype = C.c_int
        L.ref_conv99x11.argtypes = [_u8p, C.c_int, C.c_int, _f32p]
        L.ref_conv55.argtypes = [_f32p, C.c_int, C.c_int, _u8p]
        L.ref_cnn.restype = C.c_int
        L.ref_cnn.argtypes = [_u8p, C.c_int, C.c_int, _u8p, _f32p]
        L.ref_params.argtypes = [_f32p]

    @staticmethod
    def available():
        return os.path.exists(os.path.join(_HERE, "_ref", "libref.so")) or os.path.exists("/root/reference/src/srcnn.cpp")

    def threads(self):
        return int(self.lib.ref_max_threads())

    def params(self):
        p = np.empty(8129, np.float32)
        self.lib.ref_params(_ptr(p, _f32p))
        return p

    def conv99x11(self, y):
        y = np.ascontiguousarray(y, dtype=np.uint8)
        h, w = y.shape
        act2 = np.empty((32, h, w), np.float32)
        self.lib.ref_conv99x11(_ptr(y, _u8p), h, w, _ptr(act2, _f32p))
        return act2

    def conv55(self, act2):
        act2 = np.ascontiguousarray(act2, dtype=np.float32)
        _, h, w = act2.shape
        out = np.empty((h, w), np.uint8)
        self.lib.ref_conv55(_ptr(act2, _f32p), h, w, _ptr(out, _u8p))
        return out

    def cnn(self, y, want_act2=False):
        y = np.ascontiguousarray(y, dtype=np.uint8)
        h, w = y.shape
        out = np.empty((h, w), np.uint8)
        act2 = np.empty((32, h, w), np.float32) if want_act2 else None
        rc = self.lib.ref_cnn(_ptr(y, _u8p), h, w, _ptr(out, _u8p), _ptr(act2, _f32p) if want_act2 else None)
        assert rc == 0
        return (out, act2) if want_act2 else out


def cv2_pipeline(bgr, scale, cnn, stages=False):
    """The reference pipeline with REAL OpenCV (python cv2, IPP off) for the OpenCV stages and `cnn`
    (a callable Y u8 plane -> Y' u8 plane, e.g. RefLib().cnn) for the conv stage -- SURVEY Appendix B."""
    import cv2
    cv2.ipp.setUseIPP(False)
    h, w, _ = bgr.shape
    ow = int(np.float32(w) * np.float32(scale))
    oh = int(np.float32(h) * np.float32(scale))
    ycc = cv2.cvtColor(bgr, cv2.COLOR_BGR2YCrCb)
    up = [cv2.resize(np.ascontiguousarray(ycc[:, :, i]), (ow, oh), interpolation=cv2.INTER_CUBIC) for i in range(3)]
    y2 = cnn(up[0])
    out = cv2.cvtColor(cv2.merge([y2, up[1], up[2]]), cv2.COLOR_YCrCb2BGR)
    if stages:
        return out, dict(up_y=up[0], up_cr=up[1], up_cb=up[2], cnn_y=y2)
    return out


class FrawRef:
    """The reference's own float resampler, FRAWResizeEngine::scale (src/frawscale.cpp:162-286), compiled
    unmodified into oracle/_ref/libfraw.so (oracle/fraw_wrap.cpp).  filter: 0 box, 1 bilinear, 2 bicubic."""

    def __init__(self):
        path = os.path.join(_HERE, "_ref", "libfraw.so")
        if not os.path.exists(path):
            if os.path.exists("/root/reference/src/frawscale.cpp"):
                build()
            else:
                raise FileNotFoundError(path + " (built only where /root/reference exists)")
        self.lib = C.CDLL(path)
        self.lib.ref_fraw_scale.restype = C.c_uint
        self.lib.ref_fraw_scale.argtypes = [_f32p, C.c_uint, C.c_uint, C.c_uint, C.c_uint, _f32p, C.c_int]

    @staticmethod
    def available():
        return os.path.exists(os.path.join(_HERE, "_ref", "libfraw.so")) or os.path.exists("/root/reference/src/frawscale.cpp")

    def scale(self, src, dw, dh, filter=2):
        src = np.ascontiguousarray(src, dtype=np.float32)
        sh, sw = src.shape
        dst = np.zeros((dh, dw), np.float32)
        n = self.lib.ref_fraw_scale(_ptr(src, _f32p), sw, sh, dw, dh, _ptr(dst, _f32p), int(filter))
        assert n != 0
        return dst
