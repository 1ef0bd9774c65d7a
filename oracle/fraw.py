"""frawscale's resampler (FRAWResizeEngine::scale, src/frawscale.cpp:8-385) restated in numpy float64, its near misses, and
witness planes that tell them apart.  Test infrastructure only: the product never imports it.

The restatement follows srcnn_cpp_b200/csrc/fraw_resize.cu operation for operation: every double operation is one numpy
float64 operation (IEEE, rounded once), every sum is a loop over taps in tap order, vectorised across samples only.  No
np.sum / np.dot / @ / einsum anywhere: np.sum sums pairwise and BLAS contracts into FMA.

Near misses (`variant`, a set of names; an empty set is the stage itself):
  table   centre       centre of destination sample u as (u + 0.5) / ratio - 0.5
          recip        renormalise by * (1 / total) instead of / total
          box_lt       Box filter with v < width instead of v <= width
          bilinear_le  Bilinear filter with v <= width instead of v < width (equivalent: width - v is 0 at v == width)
          ratio_mul    inv = src / dst, and every / ratio of the builder as * inv
          short        one trailing tap too few
  passes  f32acc       accumulator kept in float: acc = (float)(acc + w * x)
          fma          acc = fma(w, x, acc), rounded once (DFMA)
          reverse      taps summed last to first
          pairwise     taps summed as a balanced tree
          h_first      horizontal pass first when up-scaling as well
"""
import numpy as np

TABLE_VARIANTS = ("centre", "recip", "box_lt", "bilinear_le", "ratio_mul", "short")
PASS_VARIANTS = ("f32acc", "fma", "reverse", "pairwise", "h_first")
VARIANTS = TABLE_VARIANTS + PASS_VARIANTS
BOX, BILINEAR, BICUBIC = 0, 1, 2
_WIDTH = {BOX: 0.5, BILINEAR: 1.0, BICUBIC: 2.0}


def _mitchell():
    b = 1 / 3.0
    c = 1 / 3.0                                           # src/frawscale.h:93
    return ((6 - 2 * b) / 6, (-18 + 12 * b + 6 * c) / 6, (12 - 9 * b - 6 * c) / 6,
            (8 * b + 24 * c) / 6, (-12 * b - 48 * c) / 6, (6 * b + 30 * c) / 6, (-b - 6 * c) / 6)


def filter_eval(kind, x, variant=frozenset()):
    """FrawFilter::eval on a float64 array"""
    v = np.abs(x)
    width = _WIDTH[kind]
    if kind == BOX:
        inside = v < width if "box_lt" in variant else v <= width
        return np.where(inside, 1.0, 0.0)
    if kind == BILINEAR:
        inside = v <= width if "bilinear_le" in variant else v < width
        return np.where(inside, width - v, 0.0)
    p0, p2, p3, q0, q1, q2, q3 = _mitchell()
    near = p0 + v * v * (p2 + v * p3)
    far = q0 + v * (q1 + v * (q2 + v * q3))
    return np.where(v < 1, near, np.where(v < 2, far, 0.0))


class Table:
    """FrawTable for one axis: left[dst], count[dst], w[dst, window + 1] (the device layout), window"""

    def __init__(self, kind, dst, src, variant=frozenset()):
        variant = frozenset(variant)
        width = _WIDTH[kind]
        if "ratio_mul" in variant:
            inv = float(src) / float(dst)
            ratio = 1.0 / inv
            down = ratio < 1.0
            support = width * inv if down else width
            shift = (0.5 * inv) - 0.5
            centre_of = lambda u: u * inv + shift
        else:
            ratio = float(dst) / float(src)
            down = ratio < 1.0
            support = width / ratio if down else width
            shift = (0.5 / ratio) - 0.5
            centre_of = lambda u: u / ratio + shift
        arg_scale = ratio if down else 1.0
        window = 2 * int(np.ceil(support)) + 1
        u = np.arange(dst, dtype=np.float64)
        centre = (u + 0.5) / ratio - 0.5 if "centre" in variant else centre_of(u)
        first = np.maximum(0, np.floor(centre - support).astype(np.int64))
        last = np.minimum(np.ceil(centre + support).astype(np.int64), src - 1)
        first = first + (last - first + 1 > window)        # always the left end that gives way (fraw_resize.cu)
        n = last - first + 1
        w = np.zeros((dst, window + 1), np.float64)
        total = np.zeros(dst, np.float64)
        for k in range(window):
            on = k < n
            wk = arg_scale * filter_eval(kind, arg_scale * (centre - (first + k).astype(np.float64)), variant)
            w[:, k] = np.where(on, wk, 0.0)
            total = np.where(on, total + wk, total)
        norm = (total > 0) & (total != 1)
        rows = np.nonzero(norm)[0]
        if "recip" in variant:
            w[rows] = w[rows] * (1.0 / total[rows])[:, None]
        else:
            w[rows] = w[rows] / total[rows][:, None]
        count = n.copy()
        trimming = norm.copy()
        while trimming.any():                               # trailing zero taps dropped, never the first
            r = np.nonzero(trimming)[0]
            z = (w[r, count[r] - 1] == 0) & (count[r] > 1)
            count[r[z]] -= 1
            trimming[:] = False
            trimming[r[z]] = True
        if "short" in variant:
            count = count - 1
        self.kind, self.dst, self.src, self.window = kind, dst, src, window
        self.left, self.count, self.w = first.astype(np.int32), count.astype(np.int32), w


_TABLES = {}


def table(kind, dst, src, variant=frozenset()):
    key = (kind, dst, src, frozenset(variant) & frozenset(TABLE_VARIANTS))
    if key not in _TABLES:
        if len(_TABLES) > 256:
            _TABLES.clear()
        _TABLES[key] = Table(kind, dst, src, key[3])
    return _TABLES[key]


# ---------------------------------------------------------------------------------------------------------------------
# exact fused multiply-add, vectorised (Python 3.12 has no math.fma; np.longdouble is not exact for this)
# ---------------------------------------------------------------------------------------------------------------------
def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def _split(a):
    """Veltkamp: a = hi + lo exactly, each with at most 26 significant bits"""
    t = a * 134217729.0
    hi = t - (t - a)
    return hi, a - hi


def fma(w, x, acc):
    """round(w * x + acc) once, for float64 w and acc and float32-valued x (exact products: x has 24 bits, w's halves 26).
    Boldo & Melquiond's emulation: acc + (ph + pl) with the low part rounded to odd, then one round to nearest."""
    with np.errstate(all="ignore"):
        hi, lo = _split(w)
        ph, pl = _two_sum(x * hi, x * lo)                  # ph + pl == w * x exactly
        th, tl = _two_sum(acc, ph)
        v, e = _two_sum(tl, pl)
        bits = v.view(np.int64)
        even = (bits & 1) == 0
        fix = (e != 0) & even & np.isfinite(v) & (v != 0)
        v = np.where(fix, np.nextafter(v, np.where(e > 0, np.inf, -np.inf)), v)
        r = th + v
        plain = w * x + acc                                 # non-finite operands: the IEEE result of the plain expression
        return np.where(np.isfinite(w) & np.isfinite(x) & np.isfinite(acc) & np.isfinite(r), r, plain)


# ---------------------------------------------------------------------------------------------------------------------
# the two passes
# ---------------------------------------------------------------------------------------------------------------------
def accumulate(w, x, count, variant=frozenset()):
    """float32 results of sum_i w[:, i] * x[:, i] over i < count, in the stage's arithmetic (or a near miss of it).
    w: [N, >= max count] float64, x: [N, >= max count] float32-valued float64, count: [N]."""
    n = int(count.max()) if count.size else 0
    with np.errstate(all="ignore"):
        if "pairwise" in variant:
            out = np.zeros(count.shape, np.float64)
            for c in np.unique(count):
                r = count == c
                terms = [w[r, i] * x[r, i] for i in range(c)]
                out[r] = _tree(terms) if c else 0.0
            return out.astype(np.float32)
        if "f32acc" in variant:
            acc = np.zeros(count.shape, np.float32)
            for i in range(n):
                acc = np.where(i < count, (acc.astype(np.float64) + w[:, i] * x[:, i]).astype(np.float32), acc)
            return acc
        acc = np.zeros(count.shape, np.float64)
        for j in range(n):
            if "reverse" in variant:
                i = np.maximum(count - 1 - j, 0)[:, None]
                wi, xi = np.take_along_axis(w, i, 1)[:, 0], np.take_along_axis(x, i, 1)[:, 0]
            else:
                wi, xi = w[:, j], x[:, j]
            nxt = fma(wi, xi, acc) if "fma" in variant else acc + wi * xi
            acc = np.where(j < count, nxt, acc)
        return acc.astype(np.float32)


def _tree(terms):
    if len(terms) == 1:
        return terms[0]
    m = len(terms) // 2
    return _tree(terms[:m]) + _tree(terms[m:])


def _gather(t, src_len):
    """per destination sample, the source indices of its taps (clamped into range; masked by count later)"""
    k = np.arange(max(int(t.count.max()), 1))
    return np.clip(t.left[:, None] + np.minimum(k[None, :], np.maximum(t.count[:, None] - 1, 0)), 0, src_len - 1), k.size


def vertical(src, t, variant=frozenset(), rows_per_chunk=None):
    """[sh, W] float32 -> [dh, W] float32 (k_fraw_vertical)"""
    sh, wd = src.shape
    idx, n = _gather(t, sh)
    out = np.empty((t.dst, wd), np.float32)
    step = rows_per_chunk or max(1, (1 << 22) // max(1, wd * n))
    for y0 in range(0, t.dst, step):
        y1 = min(t.dst, y0 + step)
        x = src[idx[y0:y1]].astype(np.float64)                                      # [rows, n, W]
        rows = y1 - y0
        xw = x.transpose(0, 2, 1).reshape(rows * wd, n)
        w = np.repeat(t.w[y0:y1, :n], wd, axis=0)
        c = np.repeat(t.count[y0:y1], wd)
        out[y0:y1] = accumulate(w, xw, c, variant).reshape(rows, wd)
    return out


def horizontal(src, t, variant=frozenset()):
    """[H, sw] float32 -> [H, dw] float32 (k_fraw_horizontal)"""
    h, sw = src.shape
    idx, n = _gather(t, sw)
    out = np.empty((h, t.dst), np.float32)
    step = max(1, (1 << 22) // max(1, t.dst * n))
    for r0 in range(0, h, step):
        r1 = min(h, r0 + step)
        x = src[r0:r1][:, idx].astype(np.float64)                                  # [rows, dw, n]
        rows = r1 - r0
        w = np.tile(t.w[:, :n], (rows, 1))
        c = np.tile(t.count, rows)
        out[r0:r1] = accumulate(w, x.reshape(rows * t.dst, n), c, variant).reshape(rows, t.dst)
    return out


def scale(src, dw, dh, kind, variant=frozenset()):
    """srcnn_fraw_scale_device on a host float32 plane [sh, sw] -> [dh, dw]"""
    with np.errstate(all="ignore"):       # NaN, Inf and overflow to Inf are part of what is restated
        return _scale(src, dw, dh, kind, frozenset(variant))


def _scale(src, dw, dh, kind, variant):
    src = np.ascontiguousarray(src, np.float32)
    sh, sw = src.shape
    if sw == dw and sh == dh:
        return src.copy()                                  # the documented deviation: the whole plane is copied
    th = table(kind, dw, sw, variant) if sw != dw else None
    tv = table(kind, dh, sh, variant) if sh != dh else None
    if dw <= sw or "h_first" in variant:
        mid = src if th is None else horizontal(src, th, variant)
        return mid if tv is None else vertical(mid, tv, variant)
    mid = src if tv is None else vertical(src, tv, variant)
    return horizontal(mid, th, variant)


# ---------------------------------------------------------------------------------------------------------------------
# witness planes
# ---------------------------------------------------------------------------------------------------------------------
# near misses the candidate search scores (the table ones through their own weights of the same sample)
_SCORED = ("fma", "reverse", "pairwise", "f32acc", "recip", "centre", "ratio_mul")


def linear_map(t):
    """[dst, src] float64: the weight each source sample has in each destination sample (zero-weight taps vanish)"""
    m = np.zeros((t.dst, t.src))
    for k in range(int(t.count.max()) if t.count.size else 0):
        on = np.nonzero(k < t.count)[0]
        m[on, t.left[on] + k] = t.w[on, k]
    return m


def witness_lines(kind, src_len, dst_len, lines, seed, tries=192):
    """[lines, src_len] float32: each line, resized along its length to dst_len, holds witnesses in the destination samples
    whose footprints it plants.  Every tap of a planted footprint gets a modest value; two of them instead get a large float
    X1 and X2 ~ -w_a X1 / w_b, X1 chosen among `tries` candidates so that the two products cancel, and a third (the last
    tap where it can) is set so that the result lands near 2^-30 of the large products, where the 2^-53 rounding of a
    product, the order of the sum or the last bit of a weight decides the float result.  Samples where a table near miss
    builds another table are planted first, those of the rarest near miss first; footprints of planted samples are disjoint (two zero samples apart), so every
    planted sample is independent of the others."""
    rng = np.random.default_rng(seed)
    t = table(kind, dst_len, src_len)
    alt = {v: table(kind, dst_len, src_len, {v}) for v in ("recip", "centre", "ratio_mul", "box_lt", "short")}
    ref = linear_map(t)
    moved = [np.nonzero(np.any(linear_map(ta) != ref, axis=1))[0] for ta in alt.values()]
    moved = sorted((m for m in moved if m.size), key=len)        # the rarest first: they must not be crowded out
    # samples whose weights are short dyadic fractions (exact products, order-free pairs) come last: they witness less
    dyadic = np.all(np.mod(t.w * 4096.0, 1.0) == 0, axis=1)
    out = np.zeros((lines, src_len), np.float32)
    for start in range(3):
        ln = np.arange(start, lines, 3)
        if not ln.size:
            continue
        pri = [rng.permutation(m) for m in moved] if start != 2 else []
        rest = [np.arange(start, dst_len)[~dyadic[start:]], np.arange(start, dst_len)[dyadic[start:]]]
        taken = np.zeros(src_len + 4, bool)
        for u in np.concatenate(pri + rest + [[dst_len - 1]]).astype(int):
            l, n = int(t.left[u]), int(t.count[u])
            lo, hi = max(0, l - 2), min(src_len, l + n + 2)
            if n < 1 or taken[lo:hi].any():
                continue
            taken[lo:hi] = True
            _plant(out, ln, l, n, t.w[u, :n], u, alt, rng, tries)
    return out


def _plant(out, ln, l, n, wu, u, alt, rng, tries):
    m = ln.size
    base = (rng.uniform(1, 4, (m, n))).astype(np.float32).astype(np.float64)
    good = np.nonzero(np.abs(wu) > 1e-6)[0]
    if good.size < 2:
        out[ln, l:l + n] = base.astype(np.float32)
        return
    a = np.empty(m, int)
    b = np.empty(m, int)
    c = np.full(m, -1)
    # a tap whose weight a table near miss changes in its last bits carries a large value, where the change shows
    moved = [k for k in good for ta in alt.values()
             if int(ta.left[u]) == l and int(ta.count[u]) == n and ta.w[u, k] != wu[k]]
    for j in range(m):
        p = rng.permutation(good)
        if moved and rng.random() < 0.75:
            k = moved[int(rng.integers(0, len(moved)))]
            p = np.concatenate([[k], [q for q in p if q != k]])
        a[j], b[j] = p[0], p[1]
        rest = [k for k in good[::-1] if k not in (p[0], p[1])]
        if rest:
            c[j] = rest[0] if rng.random() < 0.5 else rest[int(rng.integers(0, len(rest)))]
    rows = np.arange(m)[:, None]
    cols = np.arange(tries)[None, :]
    vals = np.repeat(base[:, None, :], tries, axis=1)
    mag = np.exp2(rng.uniform(20, 30, (m, tries)))
    x1 = (mag * rng.choice([-1.0, 1.0], (m, tries))).astype(np.float32).astype(np.float64)
    wa, wb = wu[a][:, None], wu[b][:, None]
    x2 = (-(wa * x1) / wb).astype(np.float32).astype(np.float64)
    vals[rows, cols, a[:, None]] = x1
    vals[rows, cols, b[:, None]] = x2
    has_c = c >= 0
    cc = np.maximum(c, 0)
    vals[rows, cols, cc[:, None]] = np.where(has_c[:, None], 0.0, vals[rows, cols, cc[:, None]])
    partial = np.zeros((m, tries))
    for k in range(n):
        partial = partial + wu[k] * vals[:, :, k]
    target = np.abs(wa * x1) * np.exp2(rng.uniform(-33, -27, (m, tries))) * rng.choice([-1.0, 1.0], (m, tries))
    wc = np.where(has_c, wu[cc], 1.0)[:, None]
    x3 = ((target - partial) / wc).astype(np.float32).astype(np.float64)
    vals[rows, cols, cc[:, None]] = np.where(has_c[:, None], x3, vals[rows, cols, cc[:, None]])
    flat = vals.reshape(m * tries, n)
    cnt = np.full(m * tries, n)
    w = np.broadcast_to(wu, (m * tries, n))
    ref = accumulate(w, flat, cnt).view(np.uint32)
    score = np.zeros(m * tries)
    for v in _SCORED:
        if v in alt:
            ta = alt[v]
            if int(ta.left[u]) != l or int(ta.count[u]) != n:
                continue
            got = accumulate(np.broadcast_to(ta.w[u, :n], (m * tries, n)), flat, cnt)
        else:
            got = accumulate(w, flat, cnt, {v})
        score += got.view(np.uint32) != ref
    r = ref.view(np.float32)
    score = np.where(np.isfinite(r) & (r != 0), score, -1).reshape(m, tries)
    best = np.argmax(score + rng.uniform(0, 0.5, score.shape), axis=1)
    out[ln, l:l + n] = vals[np.arange(m), best].astype(np.float32)


def witness_plane(sw, sh, dw, dh, kind, seed=0):
    """[sh, sw] float32 plane for a one-axis resize (sw == dw: a vertical pass, every column its own witness line;
    sh == dh: a horizontal pass, every row one)"""
    if sw == dw:
        return np.ascontiguousarray(witness_lines(kind, sh, dh, sw, seed).T)
    assert sh == dh, "witness planes are for one-axis resizes"
    return witness_lines(kind, sw, dw, sh, seed)


def witness_counts(src, dw, dh, kind, variants=VARIANTS):
    """{near miss: number of output samples whose bits differ from the stage's}"""
    ref = scale(src, dw, dh, kind).view(np.uint32)
    return {v: int((scale(src, dw, dh, kind, {v}).view(np.uint32) != ref).sum()) for v in variants}
