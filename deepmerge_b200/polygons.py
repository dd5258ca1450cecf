"""Label raster -> polygons (dm_polygonize) and boundary lines (dm_lines): the way back from a merged label map to one
polygon per segment, as the reference's tile.shp holds them, and to one polyline per shared boundary, as its lines.shp
holds them.  shapefile.write_polygonized and shapefile.write_boundary_lines write the results.  Polygons -> label raster
(dm_rasterize): the way in, from the polygons shapefile.read_polygons / read_polygon_rings read."""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch

from ._lib import lib
from .raster import _I32, _I64, _U8, _labels_2d, _need_cuda, _p, _stream
from .shapefile import PolygonRings

_MAX_CAPACITY = (1 << 31) - 1


def _tolerance(tolerance):
    """() for the unsimplified tracer, else (tolerance,): the extra argument of its _simplified entry point."""
    if tolerance is None:
        return ()
    t = float(tolerance)
    if not math.isfinite(t) or t < 0:
        raise ValueError("tolerance must be finite and >= 0, got %r" % (tolerance,))
    return (t,)


def _trace(labels, n_regions, capacity, default_capacity, outputs, entry, workspace_bytes, elements, extra=()):
    """Runs the library's tracer `entry` (dm_polygonize or dm_lines, whose arguments are labels, H, W, ld, n_regions,
    capacity, the output buffers, counts, workspace, stream; their _simplified forms take `extra`, the tolerance, after
    capacity) -> (counts as a list, the output buffers).
    outputs(cap, device) allocates the buffers for a capacity of cap boundary elements (`elements` names them);
    workspace_bytes(lib, H, W, n_regions, cap) is the tracer's workspace query.  When the capacity is too small the call
    is repeated once with the exact count."""
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
            outs = outputs(cap, dev)
            counts = torch.zeros(4, dtype=_I64, device=dev)
            ws_bytes = workspace_bytes(L, H, W, n_regions, cap)
            ws = torch.empty(max(ws_bytes, 1), dtype=_U8, device=dev)
            L.check(getattr(L, entry)(_p(labels), H, W, ld, n_regions, cap, *extra, *[_p(t) for t in outs], _p(counts),
                                      _p(ws), ws_bytes, _stream()), entry)
            c = counts.tolist()
            if c[3] == 1:
                raise ValueError("labels contain ids >= n_regions")
            if c[3] == 2 and attempt == 0:
                if c[2] > _MAX_CAPACITY:
                    raise ValueError("the raster has %d %s, more than 2^31 - 1" % (c[2], elements))
                cap = int(c[2])
                continue
            if c[3] != 0:
                raise RuntimeError("%s: status %d" % (entry, c[3]))
            return c, outs


def _map_xy(shapes, geotransform):
    """-> (float64 [n, 2] map coordinates X = gt0 + x gt1, Y = gt3 + y gt5 of shapes.vertices, whether the transform
    mirrors: gt1 gt5 > 0).  North-up geotransforms only."""
    gt = [float(v) for v in geotransform]
    if gt[2] != 0.0 or gt[4] != 0.0 or gt[1] == 0.0 or gt[5] == 0.0:
        raise ValueError("%s.shapes needs a north-up geotransform" % type(shapes).__name__)
    v = shapes.vertices.cpu().numpy().astype(np.float64)
    return np.stack([gt[0] + v[:, 0] * gt[1], gt[3] + v[:, 1] * gt[5]], axis=1), gt[1] * gt[5] > 0


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
        # outer rings have positive area in pixel coordinates; in (X, Y) the sign is multiplied by that of gt1 gt5, and
        # clockwise means negative there
        xy, flip = _map_xy(self, geotransform)
        rr = self.region_rings.cpu().numpy()
        off = self.ring_offsets.cpu().numpy()
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


def polygonize(labels: torch.Tensor, n_regions: int, *, tolerance=None, capacity=None) -> Polygons:
    """Rings of every region of an int32 label raster [H, W] on the GPU (strided row views accepted); negative labels
    are nodata.  Regions are 4-connected; see Polygons for the layout.  `capacity` bounds the boundary sides; when it
    is too small the call is repeated once with the exact count.

    tolerance (pixels, finite, >= 0): Douglas-Peucker simplification (dm_polygonize_simplified in
    include/deepmerge_b200.h) that keeps every shared boundary identical on both of its sides and the same as
    boundary_lines(..., tolerance=) gives it: nodes, the image border and the start of a ring without nodes are kept,
    and no ring drops below 3 vertices.  Vertices stay pixel corners; a ring may then hold a vertex where it does not
    turn (a node).  ring_area stays the pixel count.  For a tolerance in map units: tolerance = metres / |gt1|.
    W and H must be below 2^26.  None: corners only, as without simplification."""
    extra = _tolerance(tolerance)
    def outputs(cap, dev):
        ring_cap = cap // 4
        return (torch.empty(max(ring_cap, 1), dtype=_I32, device=dev),       # ring_region
                torch.empty(ring_cap + 1, dtype=_I64, device=dev),           # ring_offsets
                torch.empty(max(ring_cap, 1), dtype=_I64, device=dev),       # ring_area
                torch.empty((max(cap, 1), 2), dtype=_I32, device=dev),       # vertices
                torch.empty(int(n_regions) + 1, dtype=_I64, device=dev))     # region_rings

    entry = "dm_polygonize_simplified" if extra else "dm_polygonize"
    c, (ring_region, ring_offsets, ring_area, vertices, region_rings) = _trace(
        labels, n_regions, capacity, default_capacity, outputs, entry,
        lambda L, H, W, R, cap: getattr(L, entry + "_workspace_bytes")(H, W, R, cap), "boundary sides", extra)
    k, v = int(c[0]), int(c[1])
    return Polygons(ring_region[:k], ring_offsets[:k + 1], ring_area[:k], vertices[:v], region_rings, int(c[2]))


@dataclass
class Lines:
    """Boundary lines in canonical order (include/deepmerge_b200.h, dm_lines): line k separates the values
    line_left[k] (-1: nodata or outside) and line_right[k] (>= 0, the larger), which lie on its left and right (pixel
    coordinates, y down), and has the vertices vertices[line_offsets[k]:line_offsets[k + 1]] (start, corners, end; a
    closed line repeats its start) and line_length[k] unit segments."""
    line_left: torch.Tensor      # int32 [n_lines]
    line_right: torch.Tensor     # int32 [n_lines]
    line_length: torch.Tensor    # int64 [n_lines]
    line_offsets: torch.Tensor   # int64 [n_lines + 1]
    vertices: torch.Tensor       # int32 [n_vertices, 2]
    boundary_segments: int

    @property
    def n_lines(self):
        return self.line_left.shape[0]

    def shapes(self, geotransform):
        """-> one float64 [n, 2] polyline per line in map coordinates X = gt0 + x gt1, Y = gt3 + y gt5, with line_right
        on the right of the direction of travel in (X, Y) too: a mirroring transform (gt1 gt5 > 0) reverses the vertex
        order.  North-up geotransforms only."""
        xy, flip = _map_xy(self, geotransform)
        off = self.line_offsets.cpu().numpy()
        return [xy[off[k]:off[k + 1]][::-1 if flip else 1] for k in range(len(off) - 1)]


def default_line_capacity(n_regions, H, W):
    return int(min(2 * H * W + H + W, max(1 << 16, 4 * (H + W) + 128 * n_regions), _MAX_CAPACITY))


def boundary_lines(labels: torch.Tensor, n_regions: int, *, tolerance=None, capacity=None) -> Lines:
    """Boundary lines of an int32 label raster [H, W] on the GPU (strided row views accepted); negative labels are
    nodata: one polyline per maximal chain of pixel sides between two values, ending where three or more boundaries
    meet; see Lines for the layout.  `capacity` bounds the boundary segments; when it is too small the call is repeated
    once with the exact count.

    tolerance (pixels, finite, >= 0): Douglas-Peucker simplification (dm_lines_simplified in include/deepmerge_b200.h),
    the same on every line as polygonize(..., tolerance=) applies to the rings on both of its sides.  A line keeps its
    ends and its vertices on the image border; line_length stays the number of unit segments.  For a tolerance in map
    units: tolerance = metres / |gt1|.  W and H must be below 2^26.  None: every corner, as without simplification."""
    extra = _tolerance(tolerance)
    def outputs(cap, dev):
        return (torch.empty(max(cap, 1), dtype=_I32, device=dev),            # left
                torch.empty(max(cap, 1), dtype=_I32, device=dev),            # right
                torch.empty(max(cap, 1), dtype=_I64, device=dev),            # length
                torch.empty(cap + 1, dtype=_I64, device=dev),                # offsets
                torch.empty((max(2 * cap, 1), 2), dtype=_I32, device=dev))   # vertices

    entry = "dm_lines_simplified" if extra else "dm_lines"
    c, (left, right, length, offsets, vertices) = _trace(
        labels, n_regions, capacity, default_line_capacity, outputs, entry,
        lambda L, H, W, R, cap: getattr(L, entry + "_workspace_bytes")(H, W, cap), "boundary segments", extra)
    k, v = int(c[0]), int(c[1])
    return Lines(left[:k], right[:k], length[:k], offsets[:k + 1], vertices[:v], int(c[2]))


def _flat_rings(polygons, dev):
    """(xy float64 [n, 2], ring_offsets int64 [k + 1], ring_record int32 [k], n_records) on dev from PolygonRings (used in
    place when its arrays are already such tensors on dev) or from a list of records, each a list of [n, 2] rings."""
    if isinstance(polygons, PolygonRings):
        xy, off, rec, n_records = polygons
    else:
        rings = [np.asarray(r, np.float64).reshape(-1, 2) for rings in polygons for r in rings]
        n_records = len(polygons)
        xy = np.concatenate(rings) if rings else np.zeros((0, 2))
        off = np.zeros(len(rings) + 1, np.int64)
        np.cumsum([len(r) for r in rings], out=off[1:])
        rec = np.repeat(np.arange(n_records, dtype=np.int32), [len(r) for r in polygons])
    t = lambda a, dt: torch.as_tensor(a).to(device=dev, dtype=dt).contiguous()    # noqa: E731  (no copy when it fits)
    xy, off, rec = t(xy, torch.float64), t(off, _I64), t(rec, _I32)
    if xy.dim() != 2 or xy.shape[1] != 2 or off.dim() != 1 or rec.dim() != 1 or off.shape[0] != rec.shape[0] + 1:
        raise ValueError("rings: xy must be [n, 2] and ring_offsets one longer than ring_record")
    return xy, off, rec, int(n_records)


def default_raster_capacity(n_vertices, H):
    return int(min(max(1 << 16, 2 * n_vertices + 2 * H), _MAX_CAPACITY))


def rasterize(polygons, geotransform, height, width, *, nodata=-1, ids=None, capacity=None, device=None) -> torch.Tensor:
    """int32 [height, width] label raster on the GPU, bit for bit shapefile.rasterize_polygons: a pixel takes ids[fid]
    (default: fid) of the last polygon whose even-odd fill contains its centre, and nodata where there is none.
    `polygons` is what shapefile.read_polygons returns (one list of rings per record) or shapefile.PolygonRings, whose
    arrays may already be CUDA tensors.  North-up geotransforms only.  A non-finite coordinate raises ValueError.
    `capacity` bounds the row crossings of all segments; when it is too small the call is repeated once with the exact
    count."""
    L = lib()
    gt = [float(v) for v in geotransform]
    if gt[2] != 0.0 or gt[4] != 0.0 or gt[1] == 0.0 or gt[5] == 0.0:
        raise ValueError("rasterize needs a north-up geotransform")
    H, W, nodata = int(height), int(width), int(nodata)
    if H < 0 or W < 0:
        raise ValueError("negative raster size")
    if not -(1 << 31) <= nodata < (1 << 31):
        raise ValueError("nodata must fit int32")
    if device is None:
        first = getattr(polygons, "xy", None)
        device = first.device if isinstance(first, torch.Tensor) and first.is_cuda else torch.device("cuda")
    dev = torch.device(device)
    if dev.type != "cuda":
        raise ValueError("deepmerge_b200 kernels need CUDA tensors (there is no CPU path)")
    with torch.cuda.device(dev):
        xy, off, rec, n_records = _flat_rings(polygons, dev)
        if ids is not None:
            ids = torch.as_tensor(ids)
            if ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool or ids.dim() != 1:
                raise ValueError("ids must be a 1-D integer array")
            if ids.shape[0] < n_records:
                raise ValueError("ids has %d entries for %d records" % (ids.shape[0], n_records))
            if ids.numel() and (int(ids.min()) < -(1 << 31) or int(ids.max()) >= (1 << 31)):
                raise ValueError("ids must fit int32")
            ids = ids.to(device=dev, dtype=_I32).contiguous()
        n_v, n_rings = xy.shape[0], rec.shape[0]
        cap = default_raster_capacity(n_v, H) if capacity is None else int(capacity)
        out = torch.empty((H, W), dtype=_I32, device=dev)
        for attempt in range(2):
            counts = torch.zeros(4, dtype=_I64, device=dev)
            ws_bytes = L.dm_rasterize_workspace_bytes(n_v, n_records, cap)
            ws = torch.empty(max(ws_bytes, 1), dtype=_U8, device=dev)
            L.check(L.dm_rasterize(_p(xy), n_v, _p(off), _p(rec), n_rings, n_records, gt[0], gt[1], gt[3], gt[5], _p(ids),
                                   nodata, H, W, W, cap, _p(out), _p(counts), _p(ws), ws_bytes, _stream()), "dm_rasterize")
            c = counts.tolist()
            if c[3] == 1:
                raise ValueError("rasterize: a coordinate is not finite, or a crossing overflows float64")
            if c[3] == 4:
                raise ValueError("rasterize: a ring offset or ring record is out of range")
            if c[3] == 2 and attempt == 0:
                if c[2] > _MAX_CAPACITY:
                    raise ValueError("the polygons cross %d rows, more than 2^31 - 1" % c[2])
                cap = int(c[2])
                continue
            if c[3] != 0:
                raise RuntimeError("dm_rasterize: status %d" % c[3])
            return out
