"""Reference for detection scores (cv2 detectMultiScale2's numDetections, detectMultiScale3(outputRejectLevels=True)'s
levelWeights), built on the CPU oracle's per-level artefacts and restated here in numpy with the oracle's arithmetic.

  - raw candidates: the windows whose depth code in oracle.eval_pyramid is "passed every stage", in the oracle's order
    (level, row, column); their rectangles are the oracle's;
  - a window's weight is the double sum of its LAST stage's leaves in XML order (cascadedetect.cpp keeps the sum of the
    stage a window left last); the feature values are the oracle's float arithmetic (float products and sums, times the
    float variance factor from a double square root; none for LBP models), vectorised over the candidates;
  - grouping: cv::partition's classes (connected components of SimilarRects, numbered by first member), class size and
    the largest member weight (groupRectangles with levelWeights); the rectangles and sizes are checked against
    oracle.group_rectangles, and the final list against oracle.detect_multiscale.
"""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

import oracle as O

EPS = 0.2


def _corner(img, y, x):
    return img[y, x].astype(np.int64)


def _rect_sums(s, y, x, rx, ry, rw, rh):
    return (_corner(s, y + ry, x + rx) - _corner(s, y + ry, x + rx + rw) - _corner(s, y + ry + rh, x + rx)
            + _corner(s, y + ry + rh, x + rx + rw))


def _tilted_sums(t, y, x, rx, ry, rw, rh):
    return (_corner(t, y + ry, x + rx) - _corner(t, y + ry + rh, x + rx - rh) - _corner(t, y + ry + rw, x + rx + rw)
            + _corner(t, y + ry + rw + rh, x + rx + rw - rh))


def _feature(d, f, s, t, y, x):
    """Un-normalised float feature value of feature f[i] at window (x[i], y[i]) (ora_feature)."""
    r = d["feat_rect"][f]                                   # [m, 3, 4]
    wt = d["feat_weight"][f].astype(np.float32)             # [m, 3]
    tilted = d["feat_tilted"][f].astype(bool)
    v = np.zeros(len(f), np.float32)
    for k in range(3):
        rs = np.zeros(len(f), np.int64)
        up = ~tilted
        if up.any():
            rs[up] = _rect_sums(s, y[up], x[up], r[up, k, 0], r[up, k, 1], r[up, k, 2], r[up, k, 3])
        if tilted.any():
            rs[tilted] = _tilted_sums(t, y[tilted], x[tilted], r[tilted, k, 0], r[tilted, k, 1], r[tilted, k, 2], r[tilted, k, 3])
        term = wt[:, k] * rs.astype(np.int32).astype(np.float32)
        use = wt[:, 2] != 0 if k == 2 else np.ones(len(f), bool)
        v = np.where(use, term if k == 0 else v + term, v).astype(np.float32)
    return v


def _lbp_code(d, f, s, y, x):
    r = d["feat_rect"][f][:, 0]                             # x, y, w, h of the cell
    cx, cy, cw, ch = r[:, 0], r[:, 1], r[:, 2], r[:, 3]
    c = [[_rect_sums(s, y, x, cx + i * cw, cy + j * ch, cw, ch) for i in range(3)] for j in range(3)]
    cv = c[1][1]
    code = np.zeros(len(f), np.int64)
    for bit, (j, i) in zip((128, 64, 32, 16, 8, 4, 2, 1), ((0, 0), (0, 1), (0, 2), (1, 2), (2, 2), (2, 1), (2, 0), (1, 0))):
        code |= np.where(c[j][i] >= cv, bit, 0)
    return code


def _vnf(casc, s, q, y, x):
    nw, nh = casc.win_w - 2, casc.win_h - 2
    valsum = _rect_sums(s, y, x, 1, 1, nw, nh)
    qq = q.astype(np.uint32)
    valsq = (qq[y + 1, x + 1] - qq[y + 1, x + 1 + nw] - qq[y + 1 + nh, x + 1] + qq[y + 1 + nh, x + 1 + nw]).astype(np.uint32)
    area = float(nw * nh)
    nf = area * valsq.astype(np.float64) - valsum.astype(np.float64) * valsum.astype(np.float64)
    return (1.0 / np.sqrt(nf)).astype(np.float32)


def last_stage_weights(casc, s, q, t, y, x):
    """Sum of the last stage's leaves (double, XML order) at windows (x[i], y[i]) of one level."""
    d = casc.d
    ntr = d["tree_nnodes"]
    t0 = int(np.sum(d["stage_ntrees"][:-1]))
    node0 = int(np.sum(ntr[:t0])); leaf0 = int(np.sum(ntr[:t0] + 1))
    vnf = None if casc.lbp else _vnf(casc, s, q, y, x)
    subset = d["node_subset"].astype(np.int64) & 0xffffffff
    w = np.zeros(len(y), np.float64)
    for tr in range(t0, len(ntr)):
        idx = np.zeros(len(y), np.int64)
        active = np.ones(len(y), bool)
        while active.any():
            n = node0 + idx[active]
            fa = d["node_feat"][n]
            ya, xa = y[active], x[active]
            if casc.lbp:
                code = _lbp_code(d, fa, s, ya, xa)
                left = (subset[n, code >> 5] >> (code & 31)) & 1
                nxt = np.where(left == 1, d["node_left"][n], d["node_right"][n])
            else:
                v = (_feature(d, fa, s, t, ya, xa) * vnf[active]).astype(np.float32)
                nxt = np.where(v < d["node_thr"][n], d["node_left"][n], d["node_right"][n])
            idx[active] = nxt
            active = idx > 0
        w = w + d["leaves"][leaf0 - idx].astype(np.float64)
        node0 += int(ntr[tr]); leaf0 += int(ntr[tr]) + 1
    return w


def raw_candidates(gray, casc, scale_factor, min_size=(0, 0), max_size=(0, 0)):
    """(rects [n, 4] int32, weights [n] float64) of every window that passes all stages, in the oracle's order."""
    rects, weights = [], []
    for lv in O.eval_pyramid(gray, casc, scale_factor, min_size, max_size, keep_integrals=True):
        iy, ix = np.nonzero(lv["depth"] == 1)               # row-major: the order of the oracle's candidate list
        assert len(iy) == len(lv["cand"])
        ys = lv["ystep"]
        weights.append(last_stage_weights(casc, lv["sum"], lv["sqsum"], lv["tilted"], iy * ys, ix * ys))
        rects.append(lv["cand"])
    if not rects:
        return np.zeros((0, 4), np.int32), np.zeros(0, np.float64)
    return np.concatenate(rects).astype(np.int32), np.concatenate(weights)


def _similar_pairs(r, eps):
    """All pairs (i, j), i != j, of cv::SimilarRects(eps); candidates sorted by x, compared within a window of x."""
    n = len(r)
    order = np.argsort(r[:, 0], kind="stable")
    rs = r[order].astype(np.int64)
    xs = rs[:, 0]
    ii, jj = [], []
    for a in range(0, n, 512):
        b = min(n, a + 512)
        reach = int(np.ceil(eps * (rs[a:b, 2].max() + rs[a:b, 3].max()) * 0.5)) + 1
        lo, hi = np.searchsorted(xs, xs[a] - reach, "left"), np.searchsorted(xs, xs[b - 1] + reach, "right")
        A, B = rs[a:b, None, :], rs[None, lo:hi, :]
        delta = eps * (np.minimum(A[..., 2], B[..., 2]) + np.minimum(A[..., 3], B[..., 3])).astype(np.float64) * 0.5
        sim = ((np.abs(A[..., 0] - B[..., 0]) <= delta) & (np.abs(A[..., 1] - B[..., 1]) <= delta) &
               (np.abs(A[..., 0] + A[..., 2] - B[..., 0] - B[..., 2]) <= delta) &
               (np.abs(A[..., 1] + A[..., 3] - B[..., 1] - B[..., 3]) <= delta))
        p, q = np.nonzero(sim)
        ii.append(order[a + p]); jj.append(order[lo + q])
    return np.concatenate(ii), np.concatenate(jj)


def group_weighted(rects, weights, thr, eps=EPS):
    """groupRectangles(rects, thr, eps) with levelWeights: (rects, class sizes, largest member weight per kept class)."""
    r = np.asarray(rects, np.int32).reshape(-1, 4)
    weights = np.asarray(weights, np.float64)
    n = len(r)
    if thr <= 0 or n == 0:
        return r.copy(), np.ones(n, np.int32), weights.copy()
    i, j = _similar_pairs(r, eps)
    _, comp = connected_components(coo_matrix((np.ones(len(i)), (i, j)), shape=(n, n)), directed=False)
    first = np.full(comp.max() + 1, n); np.minimum.at(first, comp, np.arange(n))
    rank = np.empty_like(first); rank[np.argsort(first)] = np.arange(len(first))
    lab = rank[comp]                                        # classes numbered by their first member
    ncls = len(first)
    cnt = np.bincount(lab, minlength=ncls)
    acc = np.stack([np.bincount(lab, weights=r[:, k].astype(np.float64), minlength=ncls).astype(np.int64) for k in range(4)], 1)
    wmax = np.full(ncls, -np.inf); np.maximum.at(wmax, lab, weights)
    s = (np.float32(1) / cnt.astype(np.float32)).astype(np.float32)
    avg = np.rint(acc.astype(np.float32) * s[:, None]).astype(np.int64)
    out_r, out_n, out_w = [], [], []
    for a in range(ncls):
        n1 = cnt[a]
        if n1 <= thr:
            continue
        keep = True
        for b in range(ncls):
            n2 = cnt[b]
            if b == a or n2 <= thr:
                continue
            dx, dy = int(np.rint(avg[b, 2] * eps)), int(np.rint(avg[b, 3] * eps))
            if (avg[a, 0] >= avg[b, 0] - dx and avg[a, 1] >= avg[b, 1] - dy and avg[a, 0] + avg[a, 2] <= avg[b, 0] + avg[b, 2] + dx
                    and avg[a, 1] + avg[a, 3] <= avg[b, 1] + avg[b, 3] + dy and (n2 > max(3, n1) or n1 < 3)):
                keep = False
                break
        if keep:
            out_r.append(avg[a]); out_n.append(n1); out_w.append(wmax[a])
    out_r = np.asarray(out_r, np.int32).reshape(-1, 4)
    er, en = O.group_rectangles(r, thr, eps)               # the oracle's own grouping: same rectangles, same sizes
    assert (er == out_r).all() and (en == out_n).all()
    return out_r, np.asarray(out_n, np.int32), np.asarray(out_w, np.float64)


def detect_multiscale_scores(gray, casc, scale_factor=1.1, min_neighbors=3, min_size=(0, 0), max_size=(0, 0)):
    """cv2 detectMultiScale2 / detectMultiScale3(outputRejectLevels=True) on the oracle: (rects, num_detections,
    level_weights); rectangles clipped to the image, empty intersections dropped with their scores (clipObjects)."""
    gray = np.ascontiguousarray(gray, np.uint8)
    H, W = gray.shape
    raw, w = raw_candidates(gray, casc, scale_factor, min_size, max_size)
    r, n, lw = group_weighted(raw, w, min_neighbors)
    x0, y0 = np.maximum(r[:, 0], 0), np.maximum(r[:, 1], 0)
    x1, y1 = np.minimum(r[:, 0] + r[:, 2], W), np.minimum(r[:, 1] + r[:, 3], H)
    keep = (x1 > x0) & (y1 > y0)
    r = np.stack([x0, y0, x1 - x0, y1 - y0], 1)[keep].astype(np.int32).reshape(-1, 4)
    assert (r == O.detect_multiscale(gray, casc, scale_factor, min_neighbors, min_size, max_size)).all()
    return r, n[keep], lw[keep]
