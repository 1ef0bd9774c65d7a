"""Witness planes for the strict FP32 CNN -- test infrastructure, never product code.

conv3's result is only visible after the (int) truncation (src/srcnn.cpp:238), and a near miss of its arithmetic (a sum kept in
double, a float inner sum, an FMA, another order) moves the float value by about 1e-5.  That changes a byte only where the value
lies within about 1e-5 of an integer: a few pixels per million of natural content.  A witness plane puts such pixels where a test
wants them.

The network is piecewise linear in Y (conv -> ReLU -> conv -> ReLU -> conv), so around a plane the value of one pixel is, while no
ReLU changes state, v + sum_p g_p * dY_p over its clamped 13x13 field.  For each witness centre the builder takes v and g in
float64 and ranks one- and two-pixel integer edits of the field by how close they bring v to an integer.  A one-byte edit flips
some ReLUs and the float32 value differs from the float64 one by up to ~1e-4, so the ranking only narrows the search: the best
SCREEN edits are evaluated exactly with orc_cnn_at under the reference's arithmetic, the KEEP whose float value lies closest to
an integer are evaluated under every near miss, and the edit under which the most near misses change the byte is kept.  Centres
are at least 13 apart in both directions (Chebyshev), so their fields, and their edits, are disjoint: every centre's edit is
chosen on its own and all are applied to one plane.

M3 (products exact in double) and M5 (fma into the double sum) are one arithmetic: a product of two floats is exact in double,
so both round w * a + tp once.  They are kept apart because a kernel reaches them by different code.
"""
import numpy as np

from .oracle import Oracle, load_params

FIELD = 13          # conv1 9x9 under conv3 5x5: a pixel reads Y at clamp(r - 6 .. r + 6)
MAX_STEP = 24       # largest change of one Y byte an edit makes
SCREEN = 48         # predicted edits per centre whose exact value is computed
KEEP = 3            # of those, the closest to an integer, evaluated under every near miss

# orc_cnn_at's near misses, by mode (oracle/srcnn_oracle.c)
CONV3_NEAR_MISSES = {1: "M1 temp kept in double", 2: "M2 inner sum in float", 3: "M3 products exact in double",
                     4: "M4 channels reversed", 5: "M5 fma into the double sum"}
EQUIVALENT_NEAR_MISSES = {6: "conv3 (n,m) tap order", 7: "b3 added in double"}
CONV12_NEAR_MISSES = {8: "conv1 fmaf", 9: "conv1 bias first", 10: "conv1 (j,i) order", 11: "conv2 fmaf", 12: "conv2 reversed"}
NEAR_MISSES = {**CONV3_NEAR_MISSES, **EQUIVALENT_NEAR_MISSES, **CONV12_NEAR_MISSES}
MODES = 13
_SCORED = sorted(set(CONV3_NEAR_MISSES) | set(CONV12_NEAR_MISSES))

_W = None


def _weights():
    global _W
    if _W is None:
        P = load_params().astype(np.float64)
        _W = (P[0:5184].reshape(64, 81), P[5184:5248], P[5248:7296].reshape(32, 64), P[7296:7328],
              P[7328:8128].reshape(32, 25), float(P[8128]))
    return _W


def _field(h, w, rows, cols):
    """[N, 25, 81] (row, col) of the Y byte behind conv1 tap (i, j) under conv3 tap (m, n), with the reference's two clamps
    (conv3 reads act2 at clamp(r + m - 2), conv1 reads Y at clamp(that + i - 4))"""
    d5, d9 = np.arange(5) - 2, np.arange(9) - 4
    ar = np.clip(rows[:, None] + d5, 0, h - 1)
    ac = np.clip(cols[:, None] + d5, 0, w - 1)
    yr = np.clip(ar[:, :, None] + d9, 0, h - 1)                       # [N, m, i]
    yc = np.clip(ac[:, :, None] + d9, 0, w - 1)                       # [N, n, j]
    n = len(rows)
    fr = np.broadcast_to(yr[:, :, None, :, None], (n, 5, 5, 9, 9)).reshape(n, 25, 81)
    fc = np.broadcast_to(yc[:, None, :, None, :], (n, 5, 5, 9, 9)).reshape(n, 25, 81)
    return fr, fc


def value_and_gradient(y, rows, cols):
    """float64 value of each centre and its gradient over the centre's 13x13 window (rows r-6..r+6, cols c-6..c+6; zero where
    the window leaves the plane): (v [N], g [N, 13, 13])"""
    W1, b1, W2, b2, W3, b3 = _weights()
    h, w = y.shape
    rows, cols = np.asarray(rows, np.int64), np.asarray(cols, np.int64)
    fr, fc = _field(h, w, rows, cols)
    G = y[fr, fc].astype(np.float64)
    a1 = G @ W1.T + b1
    m1 = a1 > 0
    a2 = (a1 * m1) @ W2.T + b2
    m2 = a2 > 0
    v = np.einsum("npk,kp->n", a2 * m2, W3) + b3
    gG = (((m2 * W3.T[None]) @ W2) * m1) @ W1                           # dv / dG, [N, 25, 81]
    local = (fr - rows[:, None, None] + 6) * FIELD + (fc - cols[:, None, None] + 6)
    flat = (np.arange(len(rows))[:, None, None] * FIELD * FIELD + local).ravel()
    g = np.bincount(flat, weights=gG.ravel(), minlength=len(rows) * FIELD * FIELD)
    return v, g.reshape(len(rows), FIELD, FIELD)


def _edits(v, g, window, k):
    """the k one- or two-pixel edits of one centre whose predicted value lands closest to an integer in [1, 255]:
    a list of ((dr, dc, d), ...) with offsets into the window"""
    idx, steps = [], []
    for p in np.flatnonzero(g.ravel() != 0):
        y0 = int(window.flat[p])
        d = np.arange(max(-MAX_STEP, -y0), min(MAX_STEP, 255 - y0) + 1)
        d = d[d != 0]
        idx.append(np.full(d.size, p))
        steps.append(d)
    if not idx:
        return []
    p, d = np.concatenate(idx), np.concatenate(steps)
    s = g.ravel()[p] * d
    t = np.mod(v + s, 1.0)
    order = np.argsort(t, kind="stable")
    ts = t[order]
    q = np.mod(-s, 1.0)                                                   # a second edit b wants t_a close to -s_b mod 1
    pos = np.searchsorted(ts, q)
    best = []
    for off in (-1, 0):
        a = order[(pos + off) % len(ts)]
        pred = v + s[a] + s
        dist = np.abs(pred - np.round(pred))
        ok = (p[a] != p) & (np.round(pred) >= 1) & (np.round(pred) <= 255)
        best.append((np.where(ok, dist, np.inf), a))
    one = v + s
    dist1 = np.where((np.round(one) >= 1) & (np.round(one) <= 255), np.abs(one - np.round(one)), np.inf)
    cand = [(dist1[b], ((p[b], d[b]),)) for b in np.argsort(dist1, kind="stable")[:k]]
    for dist, a in best:
        for b in np.argsort(dist, kind="stable")[:k]:
            cand.append((dist[b], ((p[a[b]], d[a[b]]), (p[b], d[b]))))
    cand.sort(key=lambda e: e[0])
    out, seen = [], set()
    for dist, e in cand:
        key = tuple(sorted((int(pp), int(dd)) for pp, dd in e))
        if not np.isfinite(dist) or key in seen:
            continue
        seen.add(key)
        out.append(tuple((int(pp) // FIELD - 6, int(pp) % FIELD - 6, int(dd)) for pp, dd in key))
        if len(out) == k:
            break
    return out


def _apply(y, r, c, edit):
    for dr, dc, d in edit:
        y[r + dr, c + dc] = np.uint8(int(y[r + dr, c + dc]) + d)


def evaluate(oracle, y, rows, cols):
    """(values [MODES, N] float32, bytes [MODES, N] u8) of the centres under every orc_cnn_at mode"""
    vb = [oracle.cnn_at(y, rows, cols, m) for m in range(MODES)]
    return np.stack([a for a, _ in vb]), np.stack([b for _, b in vb])


class Witness:
    """plane: the edited u8 plane; rows, cols: the centres; values / bytes: [MODES, N] under every orc_cnn_at mode (0 exact)"""

    def __init__(self, plane, rows, cols, values, bytes_):
        self.plane, self.rows, self.cols, self.values, self.bytes = plane, rows, cols, values, bytes_

    def changed(self, mode):
        """centres whose byte differs from the exact one under near miss `mode`"""
        return self.bytes[mode] != self.bytes[0]


def build(background, centres, oracle=None, screen=SCREEN, keep=KEEP):
    """Edit `background` (u8 HxW) around each (row, col) of `centres` (pairwise Chebyshev distance >= 13)."""
    oracle = oracle or Oracle()
    y = np.array(background, dtype=np.uint8, copy=True)
    rows = np.array([r for r, _ in centres], np.int32)
    cols = np.array([c for _, c in centres], np.int32)
    v, g = value_and_gradient(y, rows, cols)
    pad = np.pad(y, 6, mode="constant")
    cand = [_edits(v[i], g[i], pad[rows[i]:rows[i] + FIELD, cols[i]:cols[i] + FIELD], screen) for i in range(len(rows))]

    def edited(pick):
        t = y.copy()
        for i, e in enumerate(cand):
            if 0 <= pick[i] < len(e):
                _apply(t, rows[i], cols[i], e[pick[i]])
        return t

    # the float32 value lands within ~1e-4 of the float64 prediction: screen many edits exactly, under the reference's
    # arithmetic only, and keep the few whose float value is closest to an integer
    dist = np.full((len(rows), screen), np.inf)
    n_cand = np.array([len(e) for e in cand])
    for j in range(screen):
        vj, _ = oracle.cnn_at(edited(np.full(len(rows), j)), rows, cols, 0)
        k = np.round(vj.astype(np.float64))
        dist[:, j] = np.where((j < n_cand) & (k >= 1) & (k <= 255), np.abs(vj - k), np.inf)
    top = np.argsort(dist, axis=1, kind="stable")[:, :keep]
    best = np.full(len(rows), -1)
    score = np.zeros(len(rows), np.int64)
    for j in range(keep):
        pick = np.where(np.isfinite(dist[np.arange(len(rows)), top[:, j]]), top[:, j], -1)
        _, b = evaluate(oracle, edited(pick), rows, cols)
        sc = (b[_SCORED] != b[0]).sum(axis=0)
        better = (pick >= 0) & (sc > score)
        best[better], score[better] = pick[better], sc[better]
    y = edited(best)
    values, bytes_ = evaluate(oracle, y, rows, cols)
    return Witness(y, rows, cols, values, bytes_)


def place(h, w, priority_rows=(), grid=True):
    """Centres at Chebyshev distance >= 13: the corners first, then rows and columns 0, 1, h-2, h-1, then every row of
    `priority_rows` (staggered so that neighbouring rows take different columns), then a 13-pitch grid where room is left."""
    blocked = np.zeros((h, w), bool)
    out = []

    def take(r, c):
        if 0 <= r < h and 0 <= c < w and not blocked[r, c]:
            out.append((r, c))
            blocked[max(r - FIELD + 1, 0):r + FIELD, max(c - FIELD + 1, 0):c + FIELD] = True

    for r in (0, h - 1):
        for c in (0, w - 1):
            take(r, c)
    edge_r = sorted({0, 1, h - 2, h - 1} & set(range(h)))
    edge_c = sorted({0, 1, w - 2, w - 1} & set(range(w)))
    for k, r in enumerate(edge_r):
        for c in range(FIELD * (k + 1), w, FIELD * len(edge_r)):
            take(r, c)
    for k, c in enumerate(edge_c):
        for r in range(FIELD * (k + 1), h, FIELD * len(edge_c)):
            take(r, c)
    pr = list(priority_rows)
    for k, r in enumerate(pr):
        for c in range(FIELD * k, w, FIELD * len(pr)):
            take(r, c)
    if grid:
        for r in range(FIELD // 2, h, FIELD):
            for c in range(FIELD // 2, w, FIELD):
                take(r, c)
    return out


def background(kind, h, w, seed):
    """'noise': uniform bytes; 'natural': smooth content with gradients and grain (tests/conftest.natural_like's recipe)"""
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    import cv2
    small = rng.integers(0, 256, (max(2, h // 8), max(2, w // 8)), dtype=np.uint8)
    img = cv2.resize(small, (w, h), interpolation=cv2.INTER_CUBIC).astype(np.int16)
    img += np.linspace(0, 40, w).astype(np.int16)[None, :] + np.linspace(0, 25, h).astype(np.int16)[:, None]
    img += rng.integers(-6, 7, (h, w), dtype=np.int16)
    return np.clip(img, 0, 255).astype(np.uint8)
