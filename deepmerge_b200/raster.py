"""Raster-native entry points of the region-merging hot path (SURVEY.md section 8(b)).

Thin PyTorch host code over the C ABI (include/deepmerge_b200.h): torch only owns device
memory and streams; every computation is a hand-written sm_100a kernel in
libdeepmerge_b200.so.  No CPU / eager fallback exists: tensors must live on a CUDA device.

Edge keys are returned as int64 tensors holding (min << 32) | max (ids < 2^31, so the
signed view orders like the unsigned key).
"""
from __future__ import annotations

from dataclasses import dataclass, replace
from typing import Optional, Sequence

import torch

from ._lib import lib

_I64, _I32, _U8, _F32 = torch.int64, torch.int32, torch.uint8, torch.float32

# Slots of the int64 counter array the raster pass and the merge kernels write (dm_shard_round_flags reads this layout):
# edges, raw entries needed, overflow flag, status (1 = bad label, >= 2 = internal error / pair-MLP status), selected, merged
_EDGES, _RAW_NEEDED, _OVERFLOW, _STATUS, _SELECTED, _MERGED = range(6)


def _check_raster_flags(c):
    """Raises on the raster pass's flags in read-back counters; OverflowError(raw entries needed) when the edges overflowed."""
    if c[_STATUS] == 1:
        raise ValueError("labels contain ids >= n_regions")
    if c[_STATUS] != 0:
        raise RuntimeError("dm_rag_build: internal pipeline error")
    if c[_OVERFLOW] != 0:
        raise OverflowError(int(c[_RAW_NEEDED]))


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise ValueError("deepmerge_b200 kernels need CUDA tensors (there is no CPU path)")


def _labels_2d(labels):
    if labels.dim() != 2 or labels.dtype != _I32:
        raise ValueError("labels must be an int32 [H, W] tensor")
    if labels.stride(1) != 1:
        labels = labels.contiguous()
    return labels


@dataclass
class RAG:
    edge_keys: torch.Tensor       # int64 [E] sorted unique (min<<32)|max
    boundary_len: torch.Tensor    # int32 [E] (uint32 counts)
    area: torch.Tensor            # int64 [R]
    perimeter: torch.Tensor       # int64 [R]
    border: torch.Tensor          # int64 [R] sides facing the image border / nodata
    band_sum: Optional[torch.Tensor] = None    # int64 [R, C] (uint64 values)
    band_sumsq: Optional[torch.Tensor] = None  # int64 [R, C]
    bbox: Optional[torch.Tensor] = None        # int32 [R, 4] (min col, min row, max col, max row); build_rag(bbox=True)

    @property
    def n_edges(self):
        return self.edge_keys.shape[0]

    def endpoints(self):
        return self.edge_keys >> 32, self.edge_keys & 0xFFFFFFFF

    def attributes(self):
        """The designed polygon attributes of the reference's tables (MyUtils1.py:79-114) that follow from this
        pass alone (SURVEY.md 8(f) N2, first part): `area` (pixels), `peri` (pixel sides facing another label, nodata
        or the image border), per band `mean<c>` and `std<c>` (population deviation) and `bright` (mean of the band
        means) -> dict of float32 tensors [R] ([R, C] for mean / std), NaN for regions without pixels.

        With `bbox` (build_rag(..., bbox=True)) the bounding-box attributes follow.  The reference only READS these
        columns (they were written by the segmentation software, their formulas are not in the repository), so the
        definitions are this build's, the usual object-based ones, restated in oracle_np.shape_attributes:
        `len` / `width` = longer / shorter side of the axis-aligned bounding box in pixels, `smooth` = peri over the
        bounding box's border 2 (w + h), `shapeness` = peri / (4 sqrt(area)), `compact` = len * width / area,
        `border` = peri / (2 (len + area / len))."""
        area = self.area.to(torch.float64)
        out = {"area": area.to(_F32), "peri": self.perimeter.to(_F32)}
        if self.bbox is not None:
            b = self.bbox.to(torch.float64)
            nan = torch.full_like(area, float("nan"))
            has = area > 0
            w = torch.where(has, b[:, 2] - b[:, 0] + 1, nan)
            h = torch.where(has, b[:, 3] - b[:, 1] + 1, nan)
            a = torch.where(has, area, nan)
            peri = self.perimeter.to(torch.float64)
            ln, wd = torch.maximum(w, h), torch.minimum(w, h)
            out["len"], out["width"] = ln.to(_F32), wd.to(_F32)
            out["smooth"] = (peri / (2.0 * (w + h))).to(_F32)
            out["shapeness"] = (peri / (4.0 * torch.sqrt(a))).to(_F32)
            out["compact"] = (ln * wd / a).to(_F32)
            out["border"] = (peri / (2.0 * (ln + a / ln))).to(_F32)
        if self.band_sum is not None:
            n = torch.where(area > 0, area, torch.full_like(area, float("nan")))[:, None]
            mean = self.band_sum.to(torch.float64) / n
            var = self.band_sumsq.to(torch.float64) / n - mean * mean
            out["mean"] = mean.to(_F32)
            out["std"] = torch.sqrt(torch.clamp(var, min=0.0)).to(_F32)
            out["bright"] = mean.mean(dim=1).to(_F32)
        return out


def default_edge_capacity(n_regions, H, W):
    return int(max(1 << 16, min(2 * H * W, 8 * n_regions + 4 * (H + W))))


def build_rag(labels: torch.Tensor, n_regions: int, image: Optional[torch.Tensor] = None, *, rows_own=None,
              top_border=True, bottom_border=True, capacity=None, return_raw=False, bbox=False) -> RAG:
    """RAG of a label raster, fused with band pooling when `image` (uint8 [H,W,C]) is given.

    Replaces the edge list the reference reads from lines.shp (MyUtils2.py:155-193) and the
    area / peri / mean / std polygon attributes (MyUtils1.py:79-114).  `rows_own` < H marks
    the last row as a halo (row-tile sharding, SURVEY.md section 8(e))."""
    L = lib()
    labels = _labels_2d(labels)
    _need_cuda(labels, image)
    H, W = labels.shape
    own = H if rows_own is None else int(rows_own)
    if own not in (H, H - 1):
        raise ValueError("rows_own must be H or H-1 (one halo row)")
    dev = labels.device
    C = 0
    if image is not None:
        if image.dtype != _U8 or image.dim() != 3 or image.shape[0] < own or image.shape[1] != W:
            raise ValueError("image must be uint8 [H, W, C]")
        image = image.contiguous()
        C = image.shape[2]
    cap = default_edge_capacity(n_regions, H, W) if capacity is None else int(capacity)
    with torch.cuda.device(dev):
        while True:
            area = torch.zeros(n_regions, dtype=_I64, device=dev)
            border = torch.zeros(n_regions, dtype=_I64, device=dev)
            bsum = torch.zeros((n_regions, C), dtype=_I64, device=dev) if C else None
            bsq = torch.zeros((n_regions, C), dtype=_I64, device=dev) if C else None
            keys = torch.empty(max(cap, 1), dtype=_I64, device=dev)
            blen = torch.empty(max(cap, 1), dtype=_I32, device=dev)
            counts = torch.zeros(4, dtype=_I64, device=dev)
            ws_bytes = L.dm_rag_workspace_bytes(cap)
            ws = torch.empty(ws_bytes, dtype=_U8, device=dev)
            L.check(L.dm_rag_build(_p(labels), own, H, W, labels.stride(0), _p(image), C, W * C if C else 0, n_regions,
                                   int(top_border), int(bottom_border), _p(area), _p(border), _p(bsum), _p(bsq),
                                   _p(keys), _p(blen), cap, _p(counts), _p(ws), ws_bytes, _stream()), "dm_rag_build")
            c = counts.tolist()
            try:
                _check_raster_flags(c)
                break
            except OverflowError as ov:
                cap = int(ov.args[0]) + 1024    # the exact raw size needed
        E = int(c[_EDGES])
        perim = torch.empty(n_regions, dtype=_I64, device=dev)
        L.check(L.dm_perimeter(_p(keys), _p(blen), _p(counts), cap, _p(border), _p(perim), n_regions, _stream()),
                "dm_perimeter")
    rag = RAG(keys[:E], blen[:E], area, perim, border, bsum, bsq)
    if bbox:
        rag.bbox = region_bbox(labels[:own], n_regions)
    if return_raw:
        return rag, int(c[_RAW_NEEDED])
    return rag


def region_bbox(labels, n_regions):
    """Bounding box of every region -> int32 [R, 4] (min column, min row, max column, max row; (INT32_MAX, INT32_MAX,
    -1, -1) for a region without pixels).  Input of the bounding-box attributes of RAG.attributes (SURVEY.md 8(f) N2)."""
    L = lib()
    labels = _labels_2d(labels)
    _need_cuda(labels)
    H, W = labels.shape
    with torch.cuda.device(labels.device):
        box = torch.empty((n_regions, 4), dtype=_I32, device=labels.device)
        bad = torch.zeros(1, dtype=_I64, device=labels.device)
        L.check(L.dm_region_bbox(_p(labels), H, W, labels.stride(0), n_regions, _p(box), _p(bad), _stream()),
                "dm_region_bbox")
        if int(bad.item()):
            raise ValueError("labels contain ids >= n_regions")
    return box


def pool_bands(labels, image, n_regions):
    """Per-region band sums / sums of squares (uint64 exact) -> (sum, sumsq) int64 [R, C]."""
    r = build_rag(labels, n_regions, image, capacity=None)
    return r.band_sum, r.band_sumsq


def merge_edge_lists(keys: torch.Tensor, lens: torch.Tensor, n_regions: int):
    """Sort + unique (summing lengths) a concatenation of per-tile edge lists."""
    L = lib()
    _need_cuda(keys, lens)
    n = keys.shape[0]
    keys = keys.clone()
    lens = lens.clone()
    dev = keys.device
    with torch.cuda.device(dev):
        cnt = torch.tensor([n, 0], dtype=_I64, device=dev)
        wsb = L.dm_edges_unique_workspace_bytes(n)
        ws = torch.empty(wsb, dtype=_U8, device=dev)
        L.check(L.dm_edges_sort_unique(_p(keys), _p(lens), _p(cnt), n, n_regions, cnt[1:].data_ptr(), _p(ws), wsb,
                                       _stream()), "dm_edges_sort_unique")
        E = int(cnt[1].item())
    return keys[:E], lens[:E]


def points_region(labels, xs, ys):
    """region_of_point[i] = labels[ys[i], xs[i]] (-1 outside / nodata): the raster form of the
    PointID membership (ExtractFeatures.py:175-179)."""
    L = lib()
    labels = _labels_2d(labels)
    _need_cuda(labels, xs, ys)
    H, W = labels.shape
    n = xs.shape[0]
    out = torch.empty(n, dtype=_I32, device=labels.device)
    with torch.cuda.device(labels.device):
        L.check(L.dm_points_region(_p(labels), H, W, labels.stride(0), _p(xs.contiguous()), _p(ys.contiguous()), n,
                                   _p(out), _stream()), "dm_points_region")
    return out


def csr_from_region_of_point(region_of_point, n_regions):
    """-> (offsets int64 [R+1], point_ids int32 [N_valid]), ascending point id per region."""
    L = lib()
    _need_cuda(region_of_point)
    rop = region_of_point.contiguous()
    n = rop.shape[0]
    dev = rop.device
    offsets = torch.empty(n_regions + 1, dtype=_I64, device=dev)
    pids = torch.empty(max(n, 1), dtype=_I32, device=dev)
    with torch.cuda.device(dev):
        wsb = L.dm_csr_workspace_bytes(n, n_regions)
        ws = torch.empty(wsb, dtype=_U8, device=dev)
        L.check(L.dm_csr_build(_p(rop), n, n_regions, _p(offsets), _p(pids), _p(ws), wsb, _stream()), "dm_csr_build")
    return offsets, pids


def pool_points_csr(offsets, point_ids, feats):
    """Mean pooling of member-point embeddings, ExtractFeatures.py:188-212 semantics
    (membership order, sequential fp32 sum, one fp32 division) -> (sum [R,D], cnt [R])."""
    L = lib()
    _need_cuda(offsets, point_ids, feats)
    if feats.dtype != _F32 or feats.dim() != 2 or feats.stride(1) != 1:
        raise ValueError("feats must be a float32 [N, D] tensor with unit inner stride")
    R = offsets.shape[0] - 1
    D = feats.shape[1]
    dev = feats.device
    s = torch.empty((R, D), dtype=_F32, device=dev)
    c = torch.empty(R, dtype=_I32, device=dev)
    with torch.cuda.device(dev):
        L.check(L.dm_pool_points_csr(_p(offsets), _p(point_ids), _p(feats), feats.stride(0), R, D, _p(s), _p(c),
                                     _stream()), "dm_pool_points_csr")
    return s, c


def pool_points(region_of_point, feats, n_regions):
    """-> (sum fp32 [R,D], cnt int32 [R]) from a per-point region id."""
    off, ids = csr_from_region_of_point(region_of_point, n_regions)
    return pool_points_csr(off, ids, feats)


def region_mean(sum_, cnt, only=None, out=None):
    """-> (mean fp32 [R,D], norm2 fp32 [R]); mean = sum / max(cnt, 1)."""
    L = lib()
    _need_cuda(sum_, cnt)
    R, D = sum_.shape
    mean, n2 = out if out is not None else (torch.empty_like(sum_), torch.empty(R, dtype=_F32, device=sum_.device))
    with torch.cuda.device(sum_.device):
        L.check(L.dm_region_mean(_p(sum_), _p(cnt), R, D, _p(mean), _p(n2), _p(only), _stream()), "dm_region_mean")
    return mean, n2


def pool_dense(labels, emb, n_regions):
    """Per-pixel embedding pooling: emb fp32 / bf16 [H,W,D] -> (sum fp32 [R,D], cnt int32 [R])."""
    L = lib()
    labels = _labels_2d(labels)
    _need_cuda(labels, emb)
    H, W = labels.shape
    if emb.shape[:2] != labels.shape or emb.dtype not in (_F32, torch.bfloat16):
        raise ValueError("emb must be float32 or bfloat16 [H, W, D]")
    emb = emb.contiguous()
    D = emb.shape[2]
    s = torch.zeros((n_regions, D), dtype=_F32, device=labels.device)
    c = torch.zeros(n_regions, dtype=_I32, device=labels.device)
    with torch.cuda.device(labels.device):
        L.check(L.dm_pool_dense(_p(labels), H, W, labels.stride(0), _p(emb), int(emb.dtype == torch.bfloat16), D,
                                n_regions, _p(s), _p(c), _stream()), "dm_pool_dense")
    return s, c


def pool_boundary(labels, emb, edge_keys):
    """Per-boundary pooling: for every 4-adjacent pixel pair straddling two regions, both pixels'
    embeddings go to that edge -> (sum fp32 [E, D], cnt int32 [E] = 2 * boundary_len)."""
    L = lib()
    labels = _labels_2d(labels)
    _need_cuda(labels, emb, edge_keys)
    H, W = labels.shape
    if emb.shape[:2] != labels.shape or emb.dtype not in (_F32, torch.bfloat16):
        raise ValueError("emb must be float32 or bfloat16 [H, W, D]")
    emb = emb.contiguous()
    D = emb.shape[2]
    E = edge_keys.shape[0]
    dev = labels.device
    s = torch.zeros((E, D), dtype=_F32, device=dev)
    c = torch.zeros(E, dtype=_I32, device=dev)
    with torch.cuda.device(dev):
        n = torch.tensor([E], dtype=_I64, device=dev)
        L.check(L.dm_pool_boundary(_p(labels), H, H, W, labels.stride(0), _p(emb), int(emb.dtype == torch.bfloat16), D,
                                   _p(edge_keys.contiguous()), _p(n), E, _p(s), _p(c), _stream()), "dm_pool_boundary")
    return s, c


def score_l2(mean, edge_keys, norm2=None):
    """Euclidean distance between the pooled means of every edge's endpoints, the
    reference's formula (ExtractFeatures.py:139-147) -> fp32 [E]."""
    L = lib()
    _need_cuda(mean, edge_keys)
    if mean.dtype != _F32 or not mean.is_contiguous():
        raise ValueError("mean must be a contiguous float32 [R, D] tensor")
    R, D = mean.shape
    dev = mean.device
    E = edge_keys.shape[0]
    if norm2 is None:
        ones = torch.ones(R, dtype=_I32, device=dev)
        _, norm2 = region_mean(mean, ones)
    scores = torch.empty(E, dtype=_F32, device=dev)
    with torch.cuda.device(dev):
        n = torch.tensor([E], dtype=_I64, device=dev)
        L.check(L.dm_score_l2(_p(mean), _p(norm2), D, _p(edge_keys.contiguous()), _p(n), E, None, _p(scores), _stream()),
                "dm_score_l2")
    return scores


def _spectral_params(C, shape, compactness, band_weights, scale=None):
    """Checks the parameters of the spectral criterion -> (w_shape, w_cmpct, band weights float32 [C] on the CPU or None,
    threshold = float32(scale^2) or None)."""
    import math

    def real(v, name, ok):
        try:
            f = float(v)
        except (TypeError, ValueError):
            f = math.nan
        if not ok(f):
            raise ValueError(name)
        return f
    thr = None
    if scale is not None:
        scale = real(scale, "scale must be a finite number > 0", lambda f: math.isfinite(f) and f > 0)
        thr = float(torch.tensor(scale * scale, dtype=torch.float64).to(_F32))
    w_shape = real(shape, "shape must be in [0, 1]", lambda f: 0.0 <= f <= 1.0)
    w_cmpct = real(compactness, "compactness must be in [0, 1]", lambda f: 0.0 <= f <= 1.0)
    bw = None
    if band_weights is not None:
        bw = torch.as_tensor(band_weights).detach().cpu().to(_F32).reshape(-1)
        if bw.numel() != C or not bool(torch.isfinite(bw).all()) or bool((bw < 0).any()):
            raise ValueError("band_weights must be %d finite values >= 0" % C)
    return w_shape, w_cmpct, bw, thr


def score_spectral(rag: RAG, shape=0.1, compactness=0.5, band_weights=None):
    """Fusion values (Baatz & Schaepe 2000, multiresolution segmentation) of every edge of a RAG built with an image and
    bbox=True: (1 - shape) h_color + shape (compactness h_cmpct + (1 - compactness) h_smooth) of the merged candidate,
    fp64 from the integer statistics, rounded to fp32 (include/deepmerge_b200.h, dm_score_spectral) -> fp32 [E]."""
    L = lib()
    if rag.band_sum is None or rag.bbox is None:
        raise ValueError("score_spectral needs a RAG built with an image and bbox=True")
    _need_cuda(rag.edge_keys, rag.band_sum, rag.bbox)
    C = rag.band_sum.shape[1]
    w_shape, w_cmpct, bw, _ = _spectral_params(C, shape, compactness, band_weights)
    dev = rag.edge_keys.device
    E = rag.n_edges
    scores = torch.empty(E, dtype=_F32, device=dev)
    with torch.cuda.device(dev):
        n = torch.tensor([E], dtype=_I64, device=dev)
        bw_d = None if bw is None else bw.to(dev)
        L.check(L.dm_score_spectral(_p(rag.edge_keys.contiguous()), _p(rag.boundary_len.contiguous()), _p(n), E,
                                    _p(rag.area), _p(rag.perimeter), _p(rag.band_sum.contiguous()),
                                    _p(rag.band_sumsq.contiguous()), C, _p(rag.bbox.contiguous()), _p(bw_d), w_shape, w_cmpct,
                                    None, _p(scores), _stream()), "dm_score_spectral")
    return scores


class PackedMLP:
    """bf16 weights of a Nets.MLP-structured network (Nets.py:11-35) in the padded tensor-core
    layout dm_score_mlp_bf16 / dm_mlp_forward_bf16 read (dm_mlp_pack).  hidden <= 256, n_out <= 16."""

    def __init__(self, W1, b1, W2, b2, W3, b3):
        L = lib()
        ws = [W1, b1, W2, b2, W3, b3]
        _need_cuda(*ws)
        ws = [w.detach().contiguous().float() for w in ws]
        self.hidden, self.in_features = ws[0].shape
        self.n_out = ws[4].shape[0]
        if ws[2].shape != (self.hidden, self.hidden) or ws[4].shape[1] != self.hidden or ws[1].shape != (self.hidden,) \
                or ws[3].shape != (self.hidden,) or ws[5].shape != (self.n_out,):
            raise ValueError("weights do not have the Linear(in,h) / Linear(h,h) / Linear(h,out) shapes of Nets.MLP")
        nbytes = L.dm_mlp_packed_bytes(self.in_features, self.hidden, self.n_out)
        if nbytes == 0:
            raise ValueError("unsupported MLP dimensions (hidden <= 256, n_out <= 16)")
        dev = ws[0].device
        self.blob = torch.empty(nbytes, dtype=_U8, device=dev)
        with torch.cuda.device(dev):
            L.check(L.dm_mlp_pack(*[_p(w) for w in ws], self.in_features, self.hidden, self.n_out, _p(self.blob),
                                  _stream()), "dm_mlp_pack")
        off = L.dm_mlp_status_offset(self.in_features, self.hidden, self.n_out)
        self.status = self.blob[off:off + 4].view(torch.int32)      # 1 = a bounded wait inside the kernel expired

    def check(self):
        """Synchronises and raises if the kernel reported a lost signal (its outputs are invalid then)."""
        if int(self.status.item()) != 0:
            raise RuntimeError("pair-MLP kernel: a bounded wait expired (lost TMA / tensor-core signal); outputs are invalid")


def _check_pair_mlp(mlp, D):
    if mlp is not None and mlp.in_features != 2 * D:
        raise ValueError("the pair-MLP takes concat(mean[lo], mean[hi]): in_features must be 2 D")


def score_mlp(mean, edge_keys, mlp: PackedMLP, want_h2=False, n_edges_dev=None, out=None, check=False):
    """Pair-MLP scores of every edge: x_e = concat(mean[lo], mean[hi]) through the three
    Linear + leaky_relu layers of Nets.MLP.forward (Nets.py:28-35), bf16 operands / fp32
    accumulation on tcgen05 -> (o fp32 [E, n_out], h2 fp32 [E, hidden] or None).
    Asynchronous; check=True synchronises and raises if the kernel reported a lost signal (mlp.check())."""
    L = lib()
    _need_cuda(mean, edge_keys)
    if mean.dtype != _F32 or not mean.is_contiguous():
        raise ValueError("mean must be a contiguous float32 [R, D] tensor")
    R, D = mean.shape
    _check_pair_mlp(mlp, D)
    dev = mean.device
    E = edge_keys.shape[0]
    o = out if out is not None else torch.empty((E, mlp.n_out), dtype=_F32, device=dev)
    h2 = torch.empty((E, mlp.hidden), dtype=_F32, device=dev) if want_h2 else None
    with torch.cuda.device(dev):
        n = n_edges_dev if n_edges_dev is not None else torch.tensor([E], dtype=_I64, device=dev)
        L.check(L.dm_score_mlp_bf16(_p(mean), D, _p(edge_keys.contiguous()), _p(n), E, _p(mlp.blob), mlp.in_features,
                                    mlp.hidden, mlp.n_out, _p(o), _p(h2), _stream()), "dm_score_mlp_bf16")
    if check:
        mlp.check()
    return o, h2


def mlp_forward(x, mlp: PackedMLP, want_h2=True, check=False):
    """Nets.MLP()(x): x fp32 [B, in_features] -> (fc3 [B, n_out], fc2 [B, hidden])."""
    L = lib()
    _need_cuda(x)
    x = x.contiguous().float()
    B, K = x.shape
    if K != mlp.in_features:
        raise ValueError("x has %d features, the network takes %d" % (K, mlp.in_features))
    o = torch.empty((B, mlp.n_out), dtype=_F32, device=x.device)
    h2 = torch.empty((B, mlp.hidden), dtype=_F32, device=x.device) if want_h2 else None
    with torch.cuda.device(x.device):
        L.check(L.dm_mlp_forward_bf16(_p(x), B, _p(mlp.blob), K, mlp.hidden, mlp.n_out, _p(o), _p(h2), _stream()),
                "dm_mlp_forward_bf16")
    if check:
        mlp.check()
    return o, h2


def relabel(labels, root):
    """labels'[p] = root[labels[p]] (nodata kept)."""
    L = lib()
    labels = _labels_2d(labels)
    _need_cuda(labels, root)
    H, W = labels.shape
    out = torch.empty((H, W), dtype=_I32, device=labels.device)
    with torch.cuda.device(labels.device):
        L.check(L.dm_relabel(_p(labels), H, W, labels.stride(0), _p(root), root.shape[0], _p(out), W, _stream()),
                "dm_relabel")
    return out


def compact_roots(root):
    """roots -> 0..R'-1 in ascending root order; returns (compact int32 [R], R')."""
    L = lib()
    _need_cuda(root)
    R = root.shape[0]
    dev = root.device
    out = torch.empty(R, dtype=_I32, device=dev)
    n = torch.zeros(1, dtype=_I64, device=dev)
    with torch.cuda.device(dev):
        wsb = L.dm_compact_roots_workspace_bytes(R)
        ws = torch.empty(wsb, dtype=_U8, device=dev)
        L.check(L.dm_compact_roots(_p(root), R, _p(out), _p(n), _p(ws), wsb, _stream()), "dm_compact_roots")
    return out, int(n.item())


@dataclass
class MergeResult:
    labels: torch.Tensor            # int32 [H, W] final label map (root ids)
    root: torch.Tensor              # int32 [R]
    rounds: int
    merges: int
    edge_keys: torch.Tensor         # final live edges
    boundary_len: torch.Tensor
    scores: torch.Tensor
    area: torch.Tensor
    perimeter: torch.Tensor
    sum: torch.Tensor
    cnt: torch.Tensor
    rag: Optional[RAG] = None       # the initial graph
    band_sum: Optional[torch.Tensor] = None     # int64 [R, C] merged band sums (run_spectral)
    band_sumsq: Optional[torch.Tensor] = None   # int64 [R, C]
    bbox: Optional[torch.Tensor] = None         # int32 [R, 4] merged bounding boxes


class MergeEngine:
    """Pre-allocated end-to-end pipeline for one raster (tile): RAG + band pooling -> point
    pooling -> edge scoring -> iterative union-find merge -> relabel.  All buffers and
    workspaces are allocated once; a run makes one host read-back per merge round (the
    selected-edge count that decides whether the loop continues)."""

    def __init__(self, H, W, n_regions, D, C=0, n_points=0, edge_capacity=None, device=None):
        self.L = lib()
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.H, self.W, self.R, self.D, self.C, self.N = int(H), int(W), int(n_regions), int(D), int(C), int(n_points)
        self.cap = default_edge_capacity(n_regions, H, W) if edge_capacity is None else int(edge_capacity)
        self.logits = None
        self.use_graphs = True                           # False once a capture was refused: plain launches from then on
        self.pool_id_range, self.id_range = False, None  # a row tile's engine (sharded.py) pools only the id interval of its points
        self.sbox = None                                  # buffers of run_spectral, allocated by its first call
        self._alloc()

    def _alloc(self):
        L, dev, R, D, C, N, cap = self.L, self.dev, self.R, self.D, self.C, self.N, self.cap
        self._graphs = {}                                 # captured round bodies point into the buffers below
        z = lambda *s, dt: torch.zeros(*s, dtype=dt, device=dev)
        e = lambda *s, dt: torch.empty(*s, dtype=dt, device=dev)
        with torch.cuda.device(dev):
            self.stats = z(3 * R + 2 * R * max(C, 1), dt=_I64)           # area | border | band_sum | band_sumsq | perimeter
            self.area, self.border = self.stats[:R], self.stats[R:2 * R]
            self.bsum = self.stats[2 * R:2 * R + R * C].view(R, C) if C else None
            self.bsq = self.stats[2 * R + R * max(C, 1):2 * R + R * max(C, 1) + R * C].view(R, C) if C else None
            self.perim = self.stats[2 * R + 2 * R * max(C, 1):]          # (one buffer -> one all-reduce when sharded)
            self.keys, self.blen, self.scores = e(cap, dt=_I64), e(cap, dt=_I32), e(cap, dt=_F32)
            self.selected = e(cap, dt=_U8)
            self.counts = z(8, dt=_I64)       # slots _EDGES .. _MERGED
            self.n_edges, self.n_selected, self.n_merged = (self.counts[i:i + 1] for i in (_EDGES, _SELECTED, _MERGED))
            self.host_counts = torch.zeros(8, dtype=_I64).pin_memory()
            self.rop = e(max(N, 1), dt=_I32)
            self.offsets, self.pids = e(R + 1, dt=_I64), e(max(N, 1), dt=_I32)
            self.sum, self.cnt = e((R, D), dt=_F32), e(R, dt=_I32)
            self.mean, self.norm2 = e((R, D), dt=_F32), e(R, dt=_F32)
            self.parent = e(R, dt=_I32)
            self.iota = torch.arange(R, dtype=_I32, device=dev)
            self.alive, self.changed = e(R, dt=_U8), e(R, dt=_U8)
            self.out = e((self.H, self.W), dt=_I32)
            # the raster pass (dm_rag_build / dm_rag_scan) and the edge re-keying are the calls that use ws
            self.ws_bytes = max(L.dm_rag_workspace_bytes(cap), L.dm_edges_rekey_workspace_bytes(cap))
            self.ws = e(self.ws_bytes, dt=_U8)
            # pooling runs on its own stream beside the raster pass (independent until the merge loop): own workspace
            self.ws_pool_bytes = L.dm_csr_workspace_bytes(N, R)
            self.ws_pool = e(self.ws_pool_bytes, dt=_U8)
            self.ws_side_bytes = L.dm_merge_apply_workspace_bytes(R)
            self.ws_side = e(self.ws_side_bytes, dt=_U8)
            self.side = torch.cuda.Stream(dev)
            self.done = torch.cuda.Event()

    # ---- stages -------------------------------------------------------------------------
    def _rag(self, labels, image, rows_own, top_border, bottom_border):
        L, s = self.L, _stream()
        self.stats.zero_()
        H = labels.shape[0]
        own = H if rows_own is None else rows_own
        L.check(L.dm_rag_build(_p(labels), own, H, self.W, labels.stride(0), _p(image), self.C, self.W * self.C, self.R,
                               int(top_border), int(bottom_border), _p(self.area), _p(self.border), _p(self.bsum),
                               _p(self.bsq), _p(self.keys), _p(self.blen), self.cap, _p(self.counts), _p(self.ws),
                               self.ws_bytes, s), "dm_rag_build")
        L.check(L.dm_perimeter(_p(self.keys), _p(self.blen), _p(self.counts), self.cap, _p(self.border), _p(self.perim),
                               self.R, s), "dm_perimeter")

    def _pool(self, labels, xs, ys, region_of_point, feats):
        """membership -> CSR -> per-region sums, and for a whole raster the means and norms (in the same pass when
        D <= 128).  A row tile's engine leaves the means to the sharded loop: they need the other tiles' partial sums."""
        L, s = self.L, _stream()
        N = feats.shape[0]
        if N > self.N:
            raise ValueError("more points than the engine was sized for")
        ld = feats.stride(0) if N else self.D        # a [0, D] tensor may report any strides (0 from numpy); no row is read
        if region_of_point is None:
            L.check(L.dm_points_region(_p(labels), labels.shape[0], self.W, labels.stride(0), _p(xs), _p(ys), N,
                                       _p(self.rop), s), "dm_points_region")
            region_of_point = self.rop
        L.check(L.dm_csr_build(_p(region_of_point), N, self.R, _p(self.offsets), _p(self.pids), _p(self.ws_pool),
                               self.ws_pool_bytes, s), "dm_csr_build")
        if not self.pool_id_range and self.D <= 128:
            L.check(L.dm_pool_points_csr_mean(_p(self.offsets), _p(self.pids), _p(feats), ld, self.R, self.D,
                                              _p(self.sum), _p(self.cnt), _p(self.mean), _p(self.norm2), s),
                    "dm_pool_points_csr_mean")
            return
        rng = None
        if self.pool_id_range:          # a row tile's engine: only the id interval that holds the tile's points is visited
            if self.id_range is None:
                self.id_range = torch.zeros(2, dtype=_I64, device=self.dev)
            L.check(L.dm_points_id_range(_p(region_of_point), N, self.R, _p(self.id_range), s), "dm_points_id_range")
            rng = self.id_range
        L.check(L.dm_pool_points_csr_tile(_p(self.offsets), _p(self.pids), _p(feats), ld, self.R, self.D,
                                          _p(self.sum), _p(self.cnt), _p(rng), s), "dm_pool_points_csr_tile")
        if not self.pool_id_range:
            self._mean_all()

    def _mean_all(self):
        L = self.L
        L.check(L.dm_region_mean(_p(self.sum), _p(self.cnt), self.R, self.D, _p(self.mean), _p(self.norm2), None, _stream()),
                "dm_region_mean")

    def _read_counts(self, after_enqueue=None):
        """The loop's host read-back; after_enqueue() is called between the enqueue of the copy and the wait for it."""
        self.host_counts.copy_(self.counts, non_blocking=True)
        self.done.record()
        if after_enqueue is not None:
            after_enqueue()
        self.done.synchronize()
        return self.host_counts.tolist()

    def load_graph(self, sum_, cnt, area, perimeter, edge_keys, boundary_len):
        """Load an explicit region graph (e.g. the all-gathered graph of a sharded scene)."""
        E = edge_keys.shape[0]
        if E > self.cap:
            self.cap = E + 1024
            self._alloc()
        self.sum.copy_(sum_)
        self.cnt.copy_(cnt)
        self.area.copy_(area)
        self.perim.copy_(perimeter)
        self.keys[:E].copy_(edge_keys)
        self.blen[:E].copy_(boundary_len)
        self.counts.zero_()
        self.counts[_EDGES] = E

    def merge_loaded_graph(self, tau, max_rounds=64, mlp=None):
        rule = _EmbeddingRule(tau, mlp)
        with torch.cuda.device(self.dev):
            rule.prepare(self)
            self._merge_init()
            self._mean_all()
            rounds, merges = self._merge_loop(rule, max_rounds)
        return self._result(None, rounds, merges)

    def run(self, labels, feats, tau, *, image=None, xs=None, ys=None, region_of_point=None, max_rounds=64,
            rows_own=None, top_border=True, bottom_border=True, relabel=True, mlp=None):
        labels = _labels_2d(labels)
        _need_cuda(labels, feats, image, xs, ys, region_of_point)
        if feats.dtype != _F32 or feats.dim() != 2 or feats.shape[1] != self.D or feats.stride(1) != 1:
            raise ValueError("feats must be float32 [N, D]")
        if (image is None) != (self.C == 0):
            raise ValueError("engine was sized for C=%d bands" % self.C)
        return self._run(_EmbeddingRule(tau, mlp), labels, image, max_rounds, relabel, rows_own, top_border, bottom_border,
                         points=(xs, ys, region_of_point, feats))

    def run_spectral(self, labels, image, scale, *, shape=0.1, compactness=0.5, band_weights=None, max_rounds=None,
                     relabel=True) -> MergeResult:
        """Merge by spectral and shape heterogeneity, without embeddings (the engine may be built with D = 0 and
        n_points = 0): RAG, band sums and boxes of the label raster, then rounds of local mutual best fitting on the
        fusion values of Baatz & Schaepe until no adjacent pair fuses below scale^2 (or max_rounds rounds; None = no
        limit).  shape / compactness are MRS's weights, band_weights one weight per band (None = ones).  `scores` of
        the result are the final fusion values; band_sum / band_sumsq / bbox the merged statistics."""
        labels = _labels_2d(labels)
        _need_cuda(labels, image)
        if image is None or image.dtype != _U8 or image.dim() != 3 or image.shape[2] < 1:
            raise ValueError("image must be a uint8 [H, W, C >= 1] tensor")
        if tuple(labels.shape) != (self.H, self.W) or tuple(image.shape) != (self.H, self.W, self.C):
            raise ValueError("engine was sized for [%d, %d] labels and a [%d, %d, %d] image" % (self.H, self.W, self.H,
                                                                                                self.W, self.C))
        w_shape, w_cmpct, bw, thr = _spectral_params(self.C, shape, compactness, band_weights, scale)
        res = self._run(_SpectralRule(thr, w_shape, w_cmpct, bw), labels, image.contiguous(), max_rounds, relabel)
        return replace(res, sum=None, cnt=None, band_sum=self.bsum, band_sumsq=self.bsq, bbox=self.sbox)

    def _run(self, rule, labels, image, max_rounds, relabel, rows_own=None, top_border=True, bottom_border=True,
             points=None):
        """Raster pass (and point pooling beside it), merge loop of `rule`, relabel; reruns when the edges outgrew `cap`."""
        own = labels.shape[0] if rows_own is None else rows_own
        # The relabel is enqueued behind every selection, right AFTER the copy of the counters the host waits for and
        # gated on the device by the selection's count: when the loop ends it is already running (no idle device
        # during the last read-back), when it goes on the kernel returns at once.  The host never waits for it.
        after_read = (lambda last: self._relabel_gated(labels, own, None if last else self.n_selected)) if relabel else None
        with torch.cuda.device(self.dev):
            while True:
                rule.prepare(self)
                if points is None:
                    self._merge_init()
                    self._rag(labels, image, rows_own, top_border, bottom_border)
                else:
                    # point pooling (membership, CSR, segment sums) only needs the labels: it runs on a side stream while
                    # the raster pass -- instruction-issue bound, light on memory -- and its edge sort occupy the main one
                    cur = torch.cuda.current_stream(self.dev)
                    self.side.wait_stream(cur)
                    with torch.cuda.stream(self.side):
                        self._merge_init()
                        self._pool(labels, *points)
                    self._rag(labels, image, rows_own, top_border, bottom_border)
                    cur.wait_stream(self.side)
                rule.after_raster(self, labels)
                try:
                    rounds, merges = self._merge_loop(rule, max_rounds, after_read)
                    break
                except OverflowError as ov:            # raw edge list outgrew the capacity: resize, rerun
                    self.cap = int(ov.args[0]) + 1024
                    self._alloc()
        return self._result(self.out[:own] if relabel else None, rounds, merges)

    def _result(self, labels, rounds, merges):
        E = int(self.host_counts[_EDGES])
        return MergeResult(labels, self.parent, rounds, merges, self.keys[:E], self.blen[:E], self.scores[:E], self.area,
                           self.perim, self.sum, self.cnt)

    def _relabel_gated(self, labels, rows, gate):
        """out = parent[labels] over `rows` rows; the kernel returns at once when the int64 `gate` is nonzero (None: never)."""
        self.L.check(self.L.dm_relabel_gated(_p(labels), rows, self.W, labels.stride(0), _p(self.parent), self.R,
                                             _p(self.out), self.W, _p(gate), _stream()), "dm_relabel_gated")

    def _merge_init(self):
        """A new merge loop: parent = identity, everything alive, round counters zero."""
        self.parent.copy_(self.iota)
        self.alive.fill_(1)
        self.counts[_MERGED:].zero_()

    def _merge_loop(self, rule, max_rounds, after_read=None):
        """The merge rounds of `rule` on the engine's graph; after_read(last) is enqueued behind each read-back's copy."""
        rule.score(self, None)
        rule.select(self)
        rounds = merges = 0
        while True:
            c = self._read_counts(None if after_read is None else (lambda: after_read(rounds == max_rounds)))
            if rounds == 0:
                _check_raster_flags(c)
            if c[_STATUS] > 1:
                raise RuntimeError("pair-MLP kernel: a bounded wait expired (lost TMA / tensor-core signal)")
            merges += int(c[_MERGED])                 # members absorbed by the previous round
            if c[_SELECTED] == 0 or rounds == max_rounds:
                break
            rounds += 1
            self._graph_launch(lambda: self._round_body(rule), rule)
        return rounds, merges

    def _rekey(self):
        L = self.L
        L.check(L.dm_edges_rekey(_p(self.parent), _p(self.keys), _p(self.blen), _p(self.scores), _p(self.n_edges), self.cap,
                                 self.R, _p(self.perim), _p(self.ws), self.ws_bytes, _stream()), "dm_edges_rekey")

    def _round_body(self, rule):
        """One merge round between two read-backs: unions of the selected edges, merged statistics, re-keyed edge list,
        scores of what changed, the next selection."""
        L, s = self.L, _stream()
        L.check(L.dm_uf_union(_p(self.parent), _p(self.keys), _p(self.selected), _p(self.n_edges), self.cap, s), "dm_uf_union")
        L.check(L.dm_uf_compress(_p(self.parent), self.R, s), "dm_uf_compress")
        rule.merge_and_rescore(self, None)
        rule.select(self)

    def _graph_launch(self, body, rule, *extra):
        """Runs a round body as ONE CUDA graph launch: a round is a dozen (sharded: ~35) short kernels whose launch gaps
        otherwise show.  The body only touches the engine's own buffers, so it is captured once per (rule.key, capacity,
        *extra) and replayed until _alloc re-allocates them.  Returns what the captured body returned.  A refused capture
        (driver / library in use) switches to plain launches from then on: the same kernels in the same order."""
        if not self.use_graphs:
            return body()
        key = rule.key + (self.cap,) + extra
        ent = self._graphs.get(key)
        if ent is None:
            g = torch.cuda.CUDAGraph()
            n0 = self.L.dm_launch_count()
            try:
                with torch.cuda.graph(g, capture_error_mode="thread_local"):
                    out = body()
            except Exception:
                self.use_graphs = False
                return body()
            ent = (g, self.L.dm_launch_count() - n0, out)
            if len(self._graphs) >= 8:
                self._graphs.clear()
            self._graphs[key] = ent
        ent[0].replay()
        self.L.dm_launch_count_add(ent[1])          # the library's counter saw the capture only
        return ent[2]


class _EmbeddingRule:
    """Merge criterion of run, merge_graph and the sharded loop: L2 distance of the pooled means below tau, or -- when a
    PackedMLP is given -- its pair decision (logit 1 > logit 0).  Embedding sums and counts, area and perimeter are merged."""

    def __init__(self, tau, mlp):
        self.tau, self.mlp = float(tau), mlp
        self.key = (self.tau, None if mlp is None else (id(mlp), mlp.blob.data_ptr()))

    def prepare(self, eng):
        mlp = self.mlp
        _check_pair_mlp(mlp, eng.D)
        if mlp is not None and (eng.logits is None or eng.logits.shape != (eng.cap, mlp.n_out)):
            eng.logits = torch.empty((eng.cap, mlp.n_out), dtype=_F32, device=eng.dev)

    def after_raster(self, eng, labels):
        pass                                       # the means come from the pooling pass

    def score(self, eng, only):
        """L2 distance (R6) of the live edges with an endpoint in `only` (None: all), or the pair-MLP logits (R8), which
        re-score every live edge each round (one tensor-core pass)."""
        L, s, mlp = eng.L, _stream(), self.mlp
        if mlp is None:
            L.check(L.dm_score_l2(_p(eng.mean), _p(eng.norm2), eng.D, _p(eng.keys), _p(eng.n_edges), eng.cap, _p(only),
                                  _p(eng.scores), s), "dm_score_l2")
            return
        L.check(L.dm_score_mlp_bf16(_p(eng.mean), eng.D, _p(eng.keys), _p(eng.n_edges), eng.cap, _p(mlp.blob),
                                    mlp.in_features, mlp.hidden, mlp.n_out, _p(eng.logits), None, s), "dm_score_mlp_bf16")
        eng.counts[_STATUS:_STATUS + 1].add_(mlp.status.to(_I64) << 1)     # the kernel's status word travels with the read-back

    def select(self, eng):
        L, s = eng.L, _stream()
        if self.mlp is None:
            L.check(L.dm_merge_select_l2(_p(eng.scores), self.tau, _p(eng.n_edges), eng.cap, _p(eng.selected),
                                         _p(eng.n_selected), s), "dm_merge_select_l2")
        else:
            L.check(L.dm_merge_select_mlp(_p(eng.logits), self.mlp.n_out, _p(eng.n_edges), eng.cap, _p(eng.selected),
                                          _p(eng.n_selected), s), "dm_merge_select_mlp")

    def merge_and_rescore(self, eng, root_mask):
        """Merged statistics, re-keyed edge list, means and scores of what changed.  root_mask (a row tile's engine):
        embedding sums are merged only for the components it flags."""
        L, R, D = eng.L, eng.R, eng.D
        # merged statistics (side stream) and edge re-keying (main stream) only share the parent array and integer
        # atomics on the perimeter: two chains of small kernels that fill the GPU better together
        cur = torch.cuda.current_stream(eng.dev)
        eng.side.wait_stream(cur)
        with torch.cuda.stream(eng.side):
            L.check(L.dm_merge_apply_masked(_p(eng.parent), _p(eng.alive), _p(eng.changed), _p(eng.sum), _p(eng.cnt),
                                            _p(eng.area), _p(eng.perim), R, D, _p(eng.n_merged), _p(root_mask),
                                            _p(eng.ws_side), eng.ws_side_bytes, _stream()), "dm_merge_apply_masked")
        eng._rekey()
        cur.wait_stream(eng.side)
        L.check(L.dm_region_mean(_p(eng.sum), _p(eng.cnt), R, D, _p(eng.mean), _p(eng.norm2), _p(eng.changed), _stream()),
                "dm_region_mean")
        self.score(eng, eng.changed)


class _SpectralRule:
    """Merge criterion of run_spectral: fusion values of Baatz & Schaepe, local mutual best pairs below thr = scale^2;
    area, perimeter, band sums and boxes are merged (integers)."""

    def __init__(self, thr, w_shape, w_cmpct, bw):
        self.thr, self.w_shape, self.w_cmpct, self.bw = thr, w_shape, w_cmpct, bw
        self.key = (thr, w_shape, w_cmpct, None if bw is None else tuple(bw.tolist()))

    def prepare(self, eng):
        if eng.sbox is None:                 # first spectral run: its buffers (existing engines do not pay for them)
            eng.sbox = torch.empty((eng.R, 4), dtype=_I32, device=eng.dev)
            eng.sbox_bad = torch.zeros(1, dtype=_I64, device=eng.dev)
            eng.band_w = torch.empty(eng.C, dtype=_F32, device=eng.dev)
            eng.ws_mutual_bytes = eng.L.dm_merge_select_mutual_workspace_bytes(eng.R)
            eng.ws_mutual = torch.empty(eng.ws_mutual_bytes, dtype=_U8, device=eng.dev)
        if self.bw is not None:
            eng.band_w.copy_(self.bw)

    def after_raster(self, eng, labels):
        eng.L.check(eng.L.dm_region_bbox(_p(labels), eng.H, eng.W, labels.stride(0), eng.R, _p(eng.sbox), _p(eng.sbox_bad),
                                         _stream()), "dm_region_bbox")

    def score(self, eng, only):
        eng.L.check(eng.L.dm_score_spectral(_p(eng.keys), _p(eng.blen), _p(eng.n_edges), eng.cap, _p(eng.area), _p(eng.perim),
                                            _p(eng.bsum), _p(eng.bsq), eng.C, _p(eng.sbox),
                                            None if self.bw is None else _p(eng.band_w), self.w_shape, self.w_cmpct, _p(only),
                                            _p(eng.scores), _stream()), "dm_score_spectral")

    def select(self, eng):
        eng.L.check(eng.L.dm_merge_select_mutual(_p(eng.scores), self.thr, _p(eng.keys), _p(eng.n_edges), eng.cap, eng.R,
                                                 _p(eng.selected), _p(eng.n_selected), _p(eng.ws_mutual),
                                                 eng.ws_mutual_bytes, _stream()), "dm_merge_select_mutual")

    def merge_and_rescore(self, eng, root_mask):
        eng.L.check(eng.L.dm_merge_apply_regions(_p(eng.parent), _p(eng.alive), _p(eng.changed), _p(eng.area), _p(eng.perim),
                                                 _p(eng.bsum), _p(eng.bsq), eng.C, _p(eng.sbox), eng.R, _p(eng.n_merged),
                                                 _stream()), "dm_merge_apply_regions")
        eng._rekey()
        self.score(eng, eng.changed)

class ScenePipeline:
    """Throughput mode for a stream of same-sized HOST scenes (the public API behind bench.py's `e2e`):
    the pinned host -> device copy of scene k+1 and the device -> host copy of label map k-1 run on their
    own CUDA streams while scene k computes, so a step costs max(H2D, D2H + compute) instead of their
    sum (PCIe is full duplex).  Inputs and outputs are double buffered on the device; every scene still
    pays its own H2D and D2H.

        pipe = ScenePipeline(engine)
        for labels_host in pipe.run(scenes, tau):      # scenes: iterable of dicts of pinned CPU tensors
            ...                                        # labels_host: pinned int32 [H, W], valid until the
                                                       # second-next iteration
    """

    KEYS = ("labels", "image", "feats", "xs", "ys")

    def __init__(self, engine: "MergeEngine", run_fn=None):
        """run_fn(device_inputs: dict, tau, **kw) -> result with .labels living in engine.out; default: engine.run.
        A ShardedMergeEngine passes its own run (engine = its tile engine): every rank then pipelines its tile."""
        self.eng = engine
        self.run_fn = run_fn or (lambda d, tau, **kw: engine.run(d["labels"], d["feats"], tau, image=d.get("image"),
                                                                  xs=d.get("xs"), ys=d.get("ys"), **kw))
        dev = engine.dev
        with torch.cuda.device(dev):
            self.s_in, self.s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        self.dev_in = [None, None]
        self.dev_out = [torch.empty((engine.H, engine.W), dtype=_I32, device=dev) for _ in range(2)]
        self.host_out = [torch.empty((engine.H, engine.W), dtype=_I32).pin_memory() for _ in range(2)]
        self.in_ready = [torch.cuda.Event() for _ in range(2)]
        self.in_free = [None, None]          # compute finished with dev_in[i]
        self.out_done = [None, None]         # D2H of dev_out[i] finished
        self.h2d_bytes = self.d2h_bytes = 0

    def _upload(self, i, scene):
        """enqueue the H2D of one scene into input buffer i on the copy-in stream"""
        dev = self.eng.dev
        with torch.cuda.stream(self.s_in):
            if self.in_free[i] is not None:
                self.s_in.wait_event(self.in_free[i])
            if self.dev_in[i] is None:
                self.dev_in[i] = {k: torch.empty(scene[k].shape, dtype=scene[k].dtype, device=dev)
                                  for k in self.KEYS if scene.get(k) is not None}
            for k, d in self.dev_in[i].items():
                d.copy_(scene[k], non_blocking=True)
                self.h2d_bytes += d.numel() * d.element_size()
            self.in_ready[i].record(self.s_in)

    def run(self, scenes, tau, **kw):
        eng = self.eng
        cur = torch.cuda.current_stream(eng.dev)
        it = iter(scenes)
        nxt = next(it, None)
        if nxt is None:
            return
        self._upload(0, nxt)
        k = 0
        pending = []                                         # (event, host buffer) of label maps on their way out
        while nxt is not None:
            i = k & 1
            nxt = next(it, None)
            if nxt is not None:
                self._upload(i ^ 1, nxt)                     # scene k+1 travels while scene k computes
            cur.wait_event(self.in_ready[i])
            if self.out_done[i] is not None:
                cur.wait_event(self.out_done[i])             # label map k-2 has left dev_out[i]
            d = self.dev_in[i]
            eng.out = self.dev_out[i]
            res = self.run_fn(d, tau, **kw)
            done = torch.cuda.Event()
            done.record(cur)
            self.in_free[i] = done
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(done)
                self.host_out[i].copy_(res.labels, non_blocking=True)
                self.d2h_bytes += res.labels.numel() * 4
                ev = torch.cuda.Event()
                ev.record(self.s_out)
            self.out_done[i] = ev
            pending.append((ev, self.host_out[i]))
            if len(pending) > 1:                             # hand out label map k-1 once it has landed
                e0, h0 = pending.pop(0)
                e0.synchronize()
                yield h0
            k += 1
        for e0, h0 in pending:
            e0.synchronize()
            yield h0


def merge_graph(sum_, cnt, area, perimeter, edge_keys, boundary_len, tau, max_rounds=64, mlp=None):
    """Merge loop on an explicit region graph (spec SURVEY.md section 8(a) R9): edges with L2 score < tau
    are contracted, or -- when a PackedMLP is given -- edges whose pair-MLP logit 1 exceeds logit 0."""
    _need_cuda(sum_, cnt, area, perimeter, edge_keys, boundary_len)
    R, D = sum_.shape
    eng = MergeEngine(1, 1, R, D, C=0, n_points=0, edge_capacity=max(edge_keys.shape[0], 1), device=sum_.device)
    with torch.cuda.device(sum_.device):
        eng.load_graph(sum_, cnt, area, perimeter, edge_keys, boundary_len)
    return eng.merge_loaded_graph(tau, max_rounds, mlp)


def _stage(x, dt):
    """A host input (numpy array or CPU tensor) -> dtype dt on the current device, staged through pinned memory; CUDA
    tensors stay on the device, None stays None."""
    import numpy as np
    if x is None:
        return None
    t = torch.from_numpy(np.ascontiguousarray(x)) if isinstance(x, np.ndarray) else x
    if t.dtype != dt:
        t = t.to(dt)
    return t if t.is_cuda else t.pin_memory().to(torch.device("cuda", torch.cuda.current_device()), non_blocking=True)


def _to_host_like(res, labels):
    """The label map and roots of `res` go back to the host when the input `labels` came from there."""
    if not (isinstance(labels, torch.Tensor) and labels.is_cuda):
        res.labels, res.root = res.labels.cpu(), res.root.cpu()
    return res


def merge_scene(labels, feats, tau, *, n_regions, image=None, xs=None, ys=None, region_of_point=None, max_rounds=64,
                engine: Optional[MergeEngine] = None, mlp=None) -> MergeResult:
    """End to end on one GPU: label raster (+ optional image bands) and sample-point
    embeddings -> merged label map.  Host (CPU / numpy) inputs are staged through pinned
    memory and the label map comes back on the host, so the call is a drop-in for a CPU
    pipeline; CUDA inputs stay on the device."""
    labels_d, feats_d, image_d = _stage(labels, _I32), _stage(feats, _F32), _stage(image, _U8)
    xs_d, ys_d, rop_d = _stage(xs, _I32), _stage(ys, _I32), _stage(region_of_point, _I32)
    H, W = labels_d.shape
    if engine is None:
        engine = MergeEngine(H, W, n_regions, feats_d.shape[1], C=0 if image_d is None else image_d.shape[2],
                             n_points=feats_d.shape[0], device=labels_d.device)
    res = engine.run(labels_d, feats_d, tau, image=image_d, xs=xs_d, ys=ys_d, region_of_point=rop_d, max_rounds=max_rounds,
                     mlp=mlp)
    return _to_host_like(res, labels)


def merge_scene_spectral(labels, image, *, n_regions, scale, shape=0.1, compactness=0.5, band_weights=None,
                         max_rounds=None, engine: Optional[MergeEngine] = None) -> MergeResult:
    """Merge by spectral and shape heterogeneity end to end on one GPU (MergeEngine.run_spectral): label raster and
    uint8 [H, W, C] image -> merged label map, no embeddings.  Host (CPU / numpy) inputs are staged through pinned
    memory and the label map and roots come back on the host, as with merge_scene; CUDA inputs stay on the device."""
    if image is None or str(image.dtype) not in ("uint8", "torch.uint8") or len(image.shape) != 3 or image.shape[2] < 1 \
            or len(labels.shape) != 2 or tuple(image.shape[:2]) != tuple(labels.shape):
        raise ValueError("merge_scene_spectral needs labels [H, W] and the image as uint8 [H, W, C >= 1]")
    _spectral_params(image.shape[2], shape, compactness, band_weights, scale)
    labels_d, image_d = _stage(labels, _I32), _stage(image, _U8)
    H, W = labels_d.shape
    if engine is None:
        engine = MergeEngine(H, W, n_regions, 0, C=image_d.shape[2], n_points=0, device=labels_d.device)
    res = engine.run_spectral(labels_d, image_d, scale, shape=shape, compactness=compactness, band_weights=band_weights,
                              max_rounds=max_rounds)
    return _to_host_like(res, labels)
