"""numpy restatement of the merge by spectral and shape heterogeneity (TEST INFRASTRUCTURE; Baatz & Schaepe 2000,
the fusion criterion of multiresolution segmentation).  There is no reference code for it -- the reference only reads
the attribute columns the segmentation software wrote (MyUtils1.py:79-114) -- so the parity is CUDA == this
restatement (DESIGN.md section 2).  The raster stages it starts from are oracle_np's."""
from __future__ import annotations

import numpy as np

from oracle.oracle_np import M32, build_rag, pack_keys, pool_bands, region_bbox, relabel, unpack_keys


def _sigma(n, S, Q):
    m = S / n
    v = Q / n - m * m
    return np.sqrt(np.where(v < 0.0, 0.0, v))


def _box_border(box):
    b = np.asarray(box, np.int64)
    return (2 * ((b[..., 2] - b[..., 0] + 1) + (b[..., 3] - b[..., 1] + 1))).astype(np.float64)


def spectral_fusion(area, perim, bsum, bsq, bbox, keys, blen, w_shape=0.1, w_cmpct=0.5, band_w=None):
    """Fusion value f of every edge (include/deepmerge_b200.h, dm_score_spectral), vectorised fp64 in the header's
    operation order, every step rounded once -> float32 [E].  w_shape, w_cmpct and band_w are float32 values widened."""
    lo, hi = unpack_keys(keys)
    area = np.asarray(area, np.int64)
    perim = np.asarray(perim, np.int64)
    bsum = np.asarray(bsum).astype(np.uint64).astype(np.int64)
    bsq = np.asarray(bsq).astype(np.uint64).astype(np.int64)
    bbox = np.asarray(bbox, np.int32)
    C = bsum.shape[1]
    ws = float(np.float32(w_shape))
    wc = float(np.float32(w_cmpct))
    bw = np.ones(C, np.float64) if band_w is None else np.asarray(band_w, np.float32).astype(np.float64)
    na, nb = area[lo], area[hi]
    da, db, dm = na.astype(np.float64), nb.astype(np.float64), (na + nb).astype(np.float64)
    hc = np.zeros(lo.shape[0], np.float64)
    for c in range(C):
        Sa, Sb, Qa, Qb = bsum[lo, c], bsum[hi, c], bsq[lo, c], bsq[hi, c]
        ta = da * _sigma(da, Sa.astype(np.float64), Qa.astype(np.float64))
        tb = db * _sigma(db, Sb.astype(np.float64), Qb.astype(np.float64))
        tm = dm * _sigma(dm, (Sa + Sb).astype(np.float64), (Qa + Qb).astype(np.float64))
        hc = hc + bw[c] * (tm - (ta + tb))
    la, lb = perim[lo], perim[hi]
    fa, fb = la.astype(np.float64), lb.astype(np.float64)
    fm = (la + lb - 2 * np.asarray(blen, np.int64)).astype(np.float64)
    ba, bb = bbox[lo], bbox[hi]
    bm = np.stack([np.minimum(ba[:, 0], bb[:, 0]), np.minimum(ba[:, 1], bb[:, 1]),
                   np.maximum(ba[:, 2], bb[:, 2]), np.maximum(ba[:, 3], bb[:, 3])], axis=1)
    cm = lambda n, l: (n * l) / np.sqrt(n)
    sm = lambda n, l, b: (n * l) / _box_border(b)
    h_cmpct = cm(dm, fm) - (cm(da, fa) + cm(db, fb))
    h_smooth = sm(dm, fm, bm) - (sm(da, fa, ba) + sm(db, fb, bb))
    h_shape = wc * h_cmpct + (1.0 - wc) * h_smooth
    return ((1.0 - ws) * hc + ws * h_shape).astype(np.float32)


def mutual_keys(scores):
    """(ordered fp32 bits << 32 | edge index) of every edge: unsigned order = (score, index) order, -0 == +0."""
    s = np.asarray(scores, np.float32)
    u = s.view(np.uint32).astype(np.uint64)
    u = np.where(s == 0, np.uint64(0x80000000), np.where(u & np.uint64(0x80000000), ~u & M32, u | np.uint64(0x80000000)))
    return (u << np.uint64(32)) | np.arange(s.shape[0], dtype=np.uint64)


def select_mutual(scores, keys, threshold, n_regions):
    """Local mutual best fitting (dm_merge_select_mutual): score < threshold (fp32) and the minimum (score, edge index)
    at both endpoints among the edges below the threshold -> bool [E]."""
    s = np.asarray(scores, np.float32)
    lo, hi = unpack_keys(keys)
    cand = s < np.float32(threshold)
    k = mutual_keys(s)
    best = np.full(n_regions, np.iinfo(np.uint64).max, np.uint64)
    np.minimum.at(best, lo[cand], k[cand])
    np.minimum.at(best, hi[cand], k[cand])
    return cand & (best[lo] == k) & (best[hi] == k)


def merge_spectral(area, perim, bsum, bsq, bbox, keys, blen, threshold, w_shape=0.1, w_cmpct=0.5, band_w=None,
                   max_rounds=None):
    """Merge loop by spectral and shape heterogeneity (spec of this build, in the style of merge_graph): score every
    live edge (spectral_fusion), select local mutual best pairs below `threshold` (float32, = scale^2), stop when none
    is selected or after max_rounds (None: no limit); merge each pair into its smaller id -- area, perimeter, band sums
    and sums of squares added, boxes united -- re-key the edges (self loops removed, 2 len off the perimeter, lengths
    summed).  Returns dict(root, rounds, merges, area, perim, bsum, bsq, bbox, keys, blen, scores)."""
    R = np.asarray(area).shape[0]
    area = np.asarray(area, np.int64).copy()
    perim = np.asarray(perim, np.int64).copy()
    bsum = np.asarray(bsum).astype(np.uint64).copy()
    bsq = np.asarray(bsq).astype(np.uint64).copy()
    bbox = np.asarray(bbox, np.int32).copy()
    keys = np.asarray(keys, np.uint64).copy()
    blen = np.asarray(blen, np.int64).copy()
    root = np.arange(R, dtype=np.int64)
    rounds = merges = 0
    while True:
        scores = spectral_fusion(area, perim, bsum, bsq, bbox, keys, blen, w_shape, w_cmpct, band_w)
        sel = select_mutual(scores, keys, threshold, R)
        if rounds == max_rounds or not sel.any():
            break
        rounds += 1
        lo, hi = unpack_keys(keys)
        a, b = lo[sel], hi[sel]                  # disjoint pairs, a < b: b joins a
        comp = np.arange(R, dtype=np.int64)
        comp[b] = a
        merges += b.size
        area[a] += area[b]
        perim[a] += perim[b]
        bsum[a] += bsum[b]
        bsq[a] += bsq[b]
        bbox[a, :2] = np.minimum(bbox[a, :2], bbox[b, :2])
        bbox[a, 2:] = np.maximum(bbox[a, 2:], bbox[b, 2:])
        nlo, nhi = comp[lo], comp[hi]
        loop = nlo == nhi
        np.add.at(perim, nlo[loop], -2 * blen[loop])
        nk = pack_keys(nlo[~loop], nhi[~loop])
        keys, inv = np.unique(nk, return_inverse=True)
        blen = np.bincount(inv, weights=blen[~loop].astype(np.float64), minlength=keys.size).astype(np.int64)
        root = comp[root]
    return dict(root=root.astype(np.int32), rounds=rounds, merges=merges, area=area, perim=perim, bsum=bsum, bsq=bsq,
                bbox=bbox, keys=keys, blen=blen.astype(np.uint32), scores=scores)


def merge_scene_spectral(labels, image, n_regions, scale, w_shape=0.1, w_cmpct=0.5, band_w=None, max_rounds=None):
    """End to end: RAG, band sums, boxes -> merge_spectral with threshold float32(scale^2) -> relabel."""
    keys, blen, area, perim = build_rag(labels, n_regions)
    s, q = pool_bands(labels, image, n_regions)
    box = region_bbox(labels, n_regions)
    g = merge_spectral(area, perim, s, q, box, keys, blen, np.float32(float(scale) * float(scale)), w_shape, w_cmpct,
                       band_w, max_rounds)
    g["labels"] = relabel(labels, g["root"])
    return g
