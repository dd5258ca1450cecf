"""Label raster -> polygons (dm_polygonize): the way back from a merged label map to one polygon per segment, as the
reference's tile.shp holds them.  shapefile.write_polygonized writes the result."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from ._lib import lib
from .raster import _I32, _I64, _U8, _labels_2d, _need_cuda, _p, _stream

_MAX_CAPACITY = (1 << 31) - 1


@dataclass
class Polygons:
    """Rings of every region present, in canonical order (include/deepmerge_b200.h, dm_polygonize): ring k of
    region ring_region[k] has the vertices vertices[ring_offsets[k]:ring_offsets[k + 1]] (pixel corners (x, y), y down,
    corners only, not closed, the region on the right); the rings of region r are region_rings[r]:region_rings[r + 1].
    ring_area is signed: outer rings positive, holes negative."""
    ring_region: torch.Tensor    # int32 [n_rings]
    ring_offsets: torch.Tensor   # int64 [n_rings + 1]
    ring_area: torch.Tensor      # int64 [n_rings]
    vertices: torch.Tensor       # int32 [n_vertices, 2]
    region_rings: torch.Tensor   # int64 [n_regions + 1]
    boundary_sides: int

    @property
    def n_rings(self):
        return self.ring_region.shape[0]

    def shapes(self, geotransform):
        """-> (region_ids int64 [k], rings_per_region): for every region present, ascending, its rings as float64
        [n + 1, 2] closed rings in map coordinates X = gt0 + x gt1, Y = gt3 + y gt5, outer rings clockwise and holes
        counter-clockwise in (X, Y) as the shapefile specification requires.  North-up geotransforms only."""
        gt = [float(v) for v in geotransform]
        if gt[2] != 0.0 or gt[4] != 0.0 or gt[1] == 0.0 or gt[5] == 0.0:
            raise ValueError("Polygons.shapes needs a north-up geotransform")
        rr = self.region_rings.cpu().numpy()
        off = self.ring_offsets.cpu().numpy()
        v = self.vertices.cpu().numpy().astype(np.float64)
        xy = np.stack([gt[0] + v[:, 0] * gt[1], gt[3] + v[:, 1] * gt[5]], axis=1)
        # outer rings have positive area in pixel coordinates; in (X, Y) the sign is multiplied by that of gt1 gt5, and
        # clockwise means negative there
        flip = gt[1] * gt[5] > 0
        ids = np.flatnonzero(np.diff(rr) > 0)
        out = []
        for r in ids:
            rings = []
            for k in range(rr[r], rr[r + 1]):
                ring = xy[off[k]:off[k + 1]]
                if flip:
                    ring = np.concatenate([ring[:1], ring[:0:-1]])
                rings.append(np.concatenate([ring, ring[:1]]))
            out.append(rings)
        return ids.astype(np.int64), out

    def region_area(self, n_regions=None):
        """int64 [n_regions]: sum of the signed ring areas of every region = its pixel count."""
        n = self.region_rings.shape[0] - 1 if n_regions is None else int(n_regions)
        area = torch.zeros(n, dtype=_I64, device=self.ring_area.device)
        return area.index_add_(0, self.ring_region.long(), self.ring_area)


def default_capacity(n_regions, H, W):
    return int(min(4 * H * W, max(1 << 16, 8 * (H + W) + 256 * n_regions), _MAX_CAPACITY))


def polygonize(labels: torch.Tensor, n_regions: int, *, capacity=None) -> Polygons:
    """Rings of every region of an int32 label raster [H, W] on the GPU (strided row views accepted); negative labels
    are nodata.  Regions are 4-connected; see Polygons for the layout.  `capacity` bounds the boundary sides; when it
    is too small the call is repeated once with the exact count."""
    L = lib()
    _need_cuda(labels)
    labels = _labels_2d(labels)
    H, W = labels.shape
    n_regions = int(n_regions)
    dev = labels.device
    ld = labels.stride(0) if H > 1 else W          # the row stride of a tensor with one row or none is arbitrary
    cap = default_capacity(n_regions, H, W) if capacity is None else int(capacity)
    with torch.cuda.device(dev):
        for attempt in range(2):
            ring_cap = cap // 4
            ring_region = torch.empty(max(ring_cap, 1), dtype=_I32, device=dev)
            ring_offsets = torch.empty(ring_cap + 1, dtype=_I64, device=dev)
            ring_area = torch.empty(max(ring_cap, 1), dtype=_I64, device=dev)
            vertices = torch.empty((max(cap, 1), 2), dtype=_I32, device=dev)
            region_rings = torch.empty(n_regions + 1, dtype=_I64, device=dev)
            counts = torch.zeros(4, dtype=_I64, device=dev)
            ws_bytes = L.dm_polygonize_workspace_bytes(H, W, n_regions, cap)
            ws = torch.empty(max(ws_bytes, 1), dtype=_U8, device=dev)
            L.check(L.dm_polygonize(_p(labels), H, W, ld, n_regions, cap, _p(ring_region), _p(ring_offsets),
                                    _p(ring_area), _p(vertices), _p(region_rings), _p(counts), _p(ws), ws_bytes,
                                    _stream()), "dm_polygonize")
            c = counts.tolist()
            if c[3] == 1:
                raise ValueError("labels contain ids >= n_regions")
            if c[3] == 2 and attempt == 0:
                if c[2] > _MAX_CAPACITY:
                    raise ValueError("the raster has %d boundary sides, more than 2^31 - 1" % c[2])
                cap = int(c[2])
                continue
            if c[3] != 0:
                raise RuntimeError("dm_polygonize: status %d" % c[3])
            break
    k, v = int(c[0]), int(c[1])
    return Polygons(ring_region[:k], ring_offsets[:k + 1], ring_area[:k], vertices[:v], region_rings, int(c[2]))
