"""Tie-dense test planes for cv::resize(INTER_CUBIC) on 8-bit planes -- test infrastructure, like the rest of oracle/.

The colour+bicubic stage claims bytes equal to cv::resize's, and those bytes hang on four details of the vertical pass:
the sum order H0*b0 + (H1*b1 + (H2*b2 + H3*b3)) with every product and sum rounded on its own (no FMA), round-half-even,
the float form on columns dx < (dw/8)*8 against the integer form (sum + 2^21) >> 22 on the rest, and the tap table.
On noise almost no output byte depends on them (a few per million).  The planes built here make many bytes depend on
them: a *witness* is an output byte on which the correct arithmetic and one of its near misses disagree.

`variants` emulates the vertical pass exactly: every float32 value there is a multiple of 2^-22 below 2^32 in those
units, so each rounding is done on exact int64 sums, one rounding to float32 at a time.  Its "ref" output equals
`Oracle.resize_cubic` (asserted by the tests).

`tie_plane` builds a source plane (grey, or BGR whose Y / Cr / Cb planes carry the witnesses) in place: output pixels
are chosen on a grid whose 4x4 source windows do not overlap (first / last row and column, tile seams and the columns
around the (dw/8)*8 boundary first), each window is filled at random, and two of its pixels are then solved over all
65536 value pairs for a sum on or next to a half-integer that separates the most near misses.
"""
import numpy as np

from .oracle import Oracle

U22 = 1 << 22                      # the vertical pass's fixed point: H * coef is the value in units of 2^-22
MUTATIONS = ("int", "fma", "l2r", "half_up", "float_tail")
# int:        the integer form on every column
# fma:        the vertical pass contracted into an FMA chain (body columns)
# l2r:        ((t0 + t1) + t2) + t3 instead of t0 + (t1 + (t2 + t3)) (body columns)
# half_up:    floor(v + 0.5) instead of round-half-even (body columns)
# float_tail: the float form on the last dw mod 8 columns as well

_oracle = None


def oracle():
    global _oracle
    if _oracle is None:
        _oracle = Oracle()
    return _oracle


def axis_taps(src, dst):
    """(idx, coef): the clamped source index and the 11-bit tap of each of the 4 taps of each output sample, int64"""
    ofs, coef = oracle().cubic_taps(src, dst)
    idx = np.clip(ofs.astype(np.int64)[:, None] - 1 + np.arange(4)[None], 0, src - 1)
    return idx, coef.astype(np.int64)


def _f32(x):
    """round an exact int64 value (units of 2^-22) to float32; the result, back in the same units, is exact"""
    return np.asarray(x, np.float64).astype(np.float32).astype(np.int64)


def _rne(v):
    return np.clip(np.rint(v.astype(np.float64) / U22), 0, 255).astype(np.int64)


def vertical(H, cy, body):
    """Every variant of the vertical pass.  H: 4 int64 arrays of horizontal sums (broadcastable), cy: 4 int64 taps (same),
    body: bool, the columns of the float form.  -> {name: output byte array} for "ref" and MUTATIONS."""
    t = [_f32(H[k] * cy[k]) for k in range(4)]
    ref_f = _f32(t[0] + _f32(t[1] + _f32(t[2] + t[3])))
    fma_f = _f32(H[0] * cy[0] + _f32(H[1] * cy[1] + _f32(H[2] * cy[2] + t[3])))
    l2r_f = _f32(_f32(_f32(t[0] + t[1]) + t[2]) + t[3])
    s = H[0] * cy[0] + H[1] * cy[1] + H[2] * cy[2] + H[3] * cy[3]
    intv = np.clip((s + (1 << 21)) >> 22, 0, 255)
    fl = _rne(ref_f)
    out = {"ref": np.where(body, fl, intv), "int": intv + 0 * fl,
           "fma": np.where(body, _rne(fma_f), intv), "l2r": np.where(body, _rne(l2r_f), intv),
           "half_up": np.where(body, np.clip(np.floor(ref_f.astype(np.float64) / U22 + 0.5), 0, 255).astype(np.int64), intv),
           "float_tail": fl + 0 * intv}
    return out


def variants(plane, dw, dh):
    """plane: (sh, sw) uint8 -> {name: (dh, dw) int64 output} for "ref" (== cv::resize) and every MUTATION"""
    plane = np.asarray(plane)
    sh, sw = plane.shape
    xi, xc = axis_taps(sw, dw)
    yi, yc = axis_taps(sh, dh)
    Hrows = (plane[:, xi].astype(np.int64) * xc[None]).sum(-1)            # (sh, dw)
    H = [Hrows[yi[:, k]] for k in range(4)]                               # (dh, dw) each
    cy = [yc[:, k][:, None] for k in range(4)]
    body = (np.arange(dw) < (dw // 8) * 8)[None, :]
    return vertical(H, cy, body)


# ---------------------------------------------------------------------------------------------------------------------
# colour: OpenCV's 8-bit BGR -> YCrCb (the oracle's orc_bgr2ycrcb), vectorised
# ---------------------------------------------------------------------------------------------------------------------
def bgr2ycc(bgr):
    b, g, r = (bgr[..., k].astype(np.int64) for k in range(3))
    y = (1868 * b + 9617 * g + 4899 * r + 8192) >> 14
    cr = np.clip(((r - y) * 11682 + (128 << 14) + 8192) >> 14, 0, 255)
    cb = np.clip(((b - y) * 9241 + (128 << 14) + 8192) >> 14, 0, 255)
    return np.stack([y, cr, cb], -1)


# ---------------------------------------------------------------------------------------------------------------------
# output classes the kernels treat differently
# ---------------------------------------------------------------------------------------------------------------------
SEAM_COLS = (64, 256)              # tiled kernel: 64-column tiles; integer-scale kernel: 256-column tiles
SEAM_ROWS = (32, 64)               # tiled kernel: 32- / 64-row tiles (integer-scale kernel: isr * S rows, isr = 5, 8, 16)


def _near(period, total):
    """indices within one of a positive multiple of `period` (the last row / column of one tile and the first of the next)"""
    i = np.arange(total)
    m = i % period
    return (i >= period - 1) & ((m == period - 1) | (m == 0)) & (i > 0)


def classes(dw, dh, scale_int=0):
    """name -> (dh, dw) bool mask of the output classes a witness must cover"""
    simd_w = (dw // 8) * 8
    xs, ys = np.arange(dw)[None, :], np.arange(dh)[:, None]
    full = np.ones((dh, dw), bool)
    c = {"first_col": full & (xs == 0), "last_col": full & (xs == dw - 1),
         "first_row": full & (ys == 0), "last_row": full & (ys == dh - 1),
         "body_at_boundary": full & (xs >= simd_w - 4) & (xs < simd_w)}
    if simd_w < dw:
        c["tail"] = full & (xs >= simd_w)
    for p in SEAM_COLS:
        if dw > p:
            c["seam_col_%d" % p] = full & _near(p, dw)[None, :]
    for p in SEAM_ROWS:
        if dh > p:
            c["seam_row_%d" % p] = full & _near(p, dh)[:, None]
    if scale_int:
        for isr in (5, 8, 16):
            p = isr * scale_int
            if dh > p:
                c["seam_row_isr%d" % isr] = full & _near(p, dh)[:, None]
    return c


def phase_ids(src, dst):
    """per output sample: the index of its tap tuple among the distinct tuples of the axis"""
    _, coef = oracle().cubic_taps(src, dst)
    _, inv = np.unique(coef, axis=0, return_inverse=True)
    return inv.reshape(-1)


def witness_counts(planes_out, sw, sh, dw, dh, scale_int=0):
    """planes_out: list of variants() dicts (one per plane) -> ({class: witnesses, plus the fewest witnesses of any column /
    row tap phase and the total}, {mutation: bytes it changes}).  A witness is an output byte where "ref" differs from at least one mutation."""
    wit = np.zeros((dh, dw), np.int64)
    per_mut = {m: 0 for m in MUTATIONS}
    for v in planes_out:
        any_ = np.zeros((dh, dw), bool)
        for m in MUTATIONS:
            d = v[m] != v["ref"]
            per_mut[m] += int(d.sum())
            any_ |= d
        wit += any_
    cls = {k: int(wit[m].sum()) for k, m in classes(dw, dh, scale_int).items()}
    px, py = phase_ids(sw, dw), phase_ids(sh, dh)
    cls["min_per_col_phase"] = int(min(wit[:, px == k].sum() for k in range(px.max() + 1)))
    cls["min_per_row_phase"] = int(min(wit[py == k].sum() for k in range(py.max() + 1)))
    cls["all"] = int(wit.sum())
    return cls, per_mut


# ---------------------------------------------------------------------------------------------------------------------
# the generator
# ---------------------------------------------------------------------------------------------------------------------
def _pick(idx, priority, rot, k0=0):
    """output samples of one axis whose (clamped) source windows are pairwise disjoint: `priority` first, then a sweep;
    the sweep steps `k mod rot` samples past the first free one so that every tap phase gets its turn"""
    lo, hi = idx.min(1), idx.max(1)
    taken = []
    used = np.zeros(int(hi.max()) + 2, bool)

    def free(d):
        return not used[lo[d]:hi[d] + 1].any()

    def take(d):
        taken.append(d)
        used[lo[d]:hi[d] + 1] = True

    for d in priority:
        if 0 <= d < len(idx) and free(d):
            take(d)
    n, d, k = len(idx), 0, k0
    while d < n:
        if free(d):
            e = d
            for _ in range(k % rot):
                if e + 1 < n and free(e + 1):
                    e += 1
            take(e)
            k += 1
            d = e + 1
        else:
            d += 1
    return sorted(taken)


_WEIGHT = {"int": 1.0, "fma": 3.0, "l2r": 3.0, "half_up": 1.0, "float_tail": 1.0}


def _solve(src, ry, cyv, rx, cxv, pl, colour, body, rng):
    """set two pixels of one target's window (plane pl's value through channel G / R / B for Y / Cr / Cb) to the value pair
    whose vertical sum separates the most near misses; True when that pair makes the target a witness"""
    av = np.arange(256)
    # effective weight of each distinct source pixel of the window (clamped taps add up)
    wr = {}
    for a in range(4):
        for b in range(4):
            key = (int(ry[a]), int(rx[b]))
            wr[key] = wr.get(key, 0) + int(cyv[a]) * int(cxv[b])
    keys = sorted(wr, key=lambda k: -abs(wr[k]))
    k1 = keys[0]
    # the second pixel: the one whose weight has the smallest common factor with the first's (the finest lattice of sums)
    rest = [k for k in keys[1:] if wr[k] != 0 and abs(wr[k]) != abs(wr[k1])]
    if not rest:
        return False
    k2 = min(rest, key=lambda k: (np.gcd(wr[k], wr[k1]), -abs(wr[k])))
    # plane value of each pixel, and of the two solved pixels for every value of their varied channel
    ch = (1, 2, 0)[pl]                    # Y <- G, Cr <- R, Cb <- B
    win = src[ry.min():ry.max() + 1, rx.min():rx.max() + 1]
    vals = bgr2ycc(win)[..., pl] if colour else win.astype(np.int64)
    V = []
    for (r, c) in (k1, k2):
        if colour:
            px = np.repeat(src[r, c][None], 256, 0)
            px[:, ch] = av
            V.append(bgr2ycc(px)[:, pl])
        else:
            V.append(av.astype(np.int64))
    # horizontal sums of the 4 tap rows, without the two solved pixels, then with every (a, b)
    Hb = np.zeros(4, np.int64)
    for a in range(4):
        for b in range(4):
            r, c = int(ry[a]), int(rx[b])
            if (r, c) not in (k1, k2):
                Hb[a] += int(vals[r - ry.min(), c - rx.min()]) * int(cxv[b])
    dH = [np.zeros((4, 256), np.int64) for _ in range(2)]
    for n, (r, c) in enumerate((k1, k2)):
        for a in range(4):
            for b in range(4):
                if int(ry[a]) == r and int(rx[b]) == c:
                    dH[n][a] += V[n] * int(cxv[b])
    cy = [int(c) for c in cyv]
    s = (sum(Hb[a] * cy[a] for a in range(4)) + sum(dH[0][a] * cy[a] for a in range(4))[:, None]
         + sum(dH[1][a] * cy[a] for a in range(4))[None, :]).reshape(-1)
    dist = np.abs((s & (U22 - 1)) - (U22 >> 1))
    ok = (s > U22) & (s < 254 * U22)
    cand = np.flatnonzero(ok & (dist < 2048))
    if len(cand) == 0:
        cand = np.flatnonzero(ok)
        if len(cand) == 0:
            return False
        cand = cand[np.argsort(dist[cand])[:64]]
    ia, ib = cand >> 8, cand & 255
    Hc = [Hb[a] + dH[0][a][ia] + dH[1][a][ib] for a in range(4)]
    v = vertical(Hc, cy, body)
    score = sum(_WEIGHT[m] * (v[m] != v["ref"]) for m in MUTATIONS) + rng.random(len(cand)) * 0.1
    best = cand[int(np.argmax(score))]
    a, b = divmod(int(best), 256)
    for (r, c), val in ((k1, a), (k2, b)):
        if colour:
            src[r, c, ch] = val
        else:
            src[r, c] = val
    return bool(score[int(np.argmax(score))] >= 1)


def tie_plane(sw, sh, dw, dh, seed=0, colour=False, scale_int=0):
    """A (sh, sw) uint8 plane (colour: (sh, sw, 3) BGR) whose resize to (dw, dh) is dense in witnesses."""
    rng = np.random.default_rng(seed)
    xi, xc = axis_taps(sw, dw)
    yi, yc = axis_taps(sh, dh)
    simd_w = (dw // 8) * 8
    seams = []
    for p in SEAM_COLS:
        for m in range(p, dw, p):
            seams += [m - 1, m]
    tail = list(range(simd_w, dw))
    # four column sets, one per target row in turn (rows do not share windows, so each row may use its own columns): the
    # image edges, the tail and the tile seams in two, the body columns at the (dw/8)*8 boundary in the other two
    prio = [[0, dw - 1] + tail, [simd_w - 1, simd_w - 2, simd_w - 3, simd_w - 4] + tail[::-1],
            [dw - 1, 0] + seams + tail[1:], [simd_w - 2, simd_w - 1] + seams[::-1] + tail]
    pr = [0, dh - 1]
    for p in SEAM_ROWS + tuple(isr * scale_int for isr in (5, 8, 16) if scale_int):
        for m in range(p, dh, p):
            pr += [m - 1, m]
    rot = max(2, min(4, int(np.ceil(dw / sw))))
    colsets = [_pick(xi, prio[k], rot, k) for k in range(4)]
    rows = _pick(yi, pr, max(2, min(4, int(np.ceil(dh / sh)))), 0)
    src = rng.integers(0, 256, (sh, sw, 3) if colour else (sh, sw), dtype=np.uint8)
    for i, dy in enumerate(rows):
        for j, dx in enumerate(colsets[i % 4]):
            pl = (i + j) % 3 if colour else 0
            ry, rx = yi[dy], xi[dx]
            for attempt in range(4):     # a window without a witness is filled afresh (windows of targets never overlap)
                if attempt:
                    win = src[ry.min():ry.max() + 1, rx.min():rx.max() + 1]
                    win[...] = rng.integers(0, 256, win.shape, dtype=np.uint8)
                if _solve(src, ry, yc[dy], rx, xc[dx], pl, colour, dx < simd_w, rng):
                    break
    return src


def plane_variants(src, dw, dh):
    """the variants of every plane the stage resizes: [Y, Cr, Cb] of a BGR source, [plane] of a grey one"""
    if src.ndim == 3:
        ycc = bgr2ycc(src).astype(np.uint8)
        return [variants(ycc[..., k], dw, dh) for k in range(3)]
    return [variants(src, dw, dh)]
