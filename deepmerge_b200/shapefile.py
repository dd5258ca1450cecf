"""On-disk adaptor for the shapefiles the reference reads and writes on the hot path (SURVEY.md
section 8(f) N3), without GDAL.

The reference goes through OGR for three things on this path:
  * `lines.shp` attributes LEFT_FID / RIGHT_FID -> the RAG edge list      (MyUtils2.py:155-193)
  * polygon attributes `PointID` (space separated), `join` / `Points` (comma separated) -> membership
    and neighbour lists                                                  (ExtractFeatures.py:175-179,
                                                                          MyUtils.py:110-117)
  * the score written back as the OFTReal attribute `simi` of the line   (ExtractFeatures.py:181-186,
                                                                          217-219)
and for the sample-point coordinates of `PointsGCS.shp` (MyUtils2.py:236-242).  All of it lives in
the .dbf attribute table (dBase III, fixed-width ASCII records) and, for the points, in fixed-size
.shp records -- both simple published formats, restated here in plain Python + numpy:

  DbfTable        the attribute table: vectorised column reads / writes (whole-column numpy parsing,
                  which is what feeds the GPU path), field creation, in-place record updates
  read_points     X / Y of a Point / PointZ / PointM .shp
  ShapefileLayer  the subset of the OGR layer / feature interface the reference calls on this path
                  (ResetReading, GetNextFeature, GetFeature, GetFeatureCount, GetLayerDefn().GetFieldIndex,
                  CreateField, SetFeature; feature.GetField / SetField / GetFID / GetGeometryRef().GetX/GetY),
                  so the reference-shaped classes (deepmerge_b200.MyUtils2.PolygonConnectPointDataset) run on
                  real files when `osgeo` is not installed
  write_dbf / write_point_shp   writers (tests, and exporting a raster-derived RAG for GIS tools)

Conventions follow the OGR "ESRI Shapefile" driver: FID = record index, trailing blanks of strings
are stripped, N fields without decimals are integers, blank / '*' filled numbers are null (None),
OFTReal is created as N(24,15), deleted records ('*' flag) are skipped by iteration.
"""
from __future__ import annotations

import datetime
import os
import struct

import numpy as np

OFTInteger, OFTReal, OFTString, OFTInteger64 = 0, 2, 4, 12      # the OGR field type codes the reference uses


class FieldDefn:
    """Name + dBase type ('C', 'N', 'F', 'L', 'D') + width + decimals of one attribute column."""

    def __init__(self, name, ftype="N", width=None, decimals=None):
        if isinstance(ftype, int):                                  # an OGR type code, as in ogr.FieldDefn(name, ogr.OFTReal)
            ftype, width, decimals = {OFTInteger: ("N", width or 9, 0), OFTInteger64: ("N", width or 18, 0),
                                      OFTReal: ("N", width or 24, 15 if decimals is None else decimals),
                                      OFTString: ("C", width or 80, 0)}[ftype]
        self.name, self.type = str(name), str(ftype).upper()
        self.width = int(width if width is not None else {"C": 80, "N": 24, "F": 24, "L": 1, "D": 8}[self.type])
        self.decimals = int(decimals or 0)
        if len(self.name.encode("ascii")) > 10:
            raise ValueError("dBase field names are at most 10 bytes: %r" % self.name)
        if not 1 <= self.width <= 254:
            raise ValueError("field width out of range: %d" % self.width)

    def GetName(self):
        return self.name

    def GetNameRef(self):
        return self.name

    @property
    def is_integer(self):
        return self.type == "N" and self.decimals == 0

    @property
    def is_real(self):
        return self.type == "F" or (self.type == "N" and self.decimals > 0)


class DbfTable:
    """A .dbf file held as one [n_records, record_length] byte matrix (numpy), parsed column-wise."""

    def __init__(self, path, update=False):
        self.path, self.update = path, bool(update)
        try:
            with open(path, "rb") as f:
                raw = f.read()
        except OSError as e:
            raise ValueError("Can not open {0}".format(path)) from e
        if len(raw) < 33:
            raise ValueError("Can not open {0}".format(path))
        self.version = raw[0]
        n, hlen, rlen = struct.unpack_from("<IHH", raw, 4)
        self.ldid = raw[29]
        self.fields = []
        off = 32
        while off + 32 <= hlen and raw[off] != 0x0D:
            name = raw[off:off + 11].split(b"\0", 1)[0].decode("ascii", "replace")
            ftype, width, dec = chr(raw[off + 11]), raw[off + 16], raw[off + 17]
            if ftype == "C":                                       # long character fields keep the high byte here
                width, dec = width + 256 * dec, 0
            fd = FieldDefn(name, ftype, max(1, min(width, 254)), dec)
            fd.width = width
            self.fields.append(fd)
            off += 32
        if rlen != 1 + sum(f.width for f in self.fields):
            raise ValueError("Can not open {0}".format(path))      # corrupt header
        avail = max(0, (len(raw) - hlen) // rlen) if rlen else 0
        n = min(n, avail)
        self.header_len, self.record_len = hlen, rlen
        self.records = np.frombuffer(raw, np.uint8, n * rlen, hlen).reshape(n, rlen).copy()
        self._dirty = False

    # ---- structure ----------------------------------------------------------------------------
    def __len__(self):
        return self.records.shape[0]

    def field_index(self, name):
        for i, f in enumerate(self.fields):
            if f.name.upper() == str(name).upper():                 # OGR matches field names case-insensitively
                return i
        return -1

    def _col(self, name_or_index):
        i = name_or_index if isinstance(name_or_index, int) else self.field_index(name_or_index)
        if i < 0 or i >= len(self.fields):
            raise KeyError(name_or_index)
        start = 1 + sum(f.width for f in self.fields[:i])
        return self.fields[i], start

    @property
    def deleted(self):
        """bool [n]: records carrying the dBase deletion flag."""
        return self.records[:, 0] == ord("*") if len(self) else np.zeros(0, bool)

    # ---- column reads (vectorised) ------------------------------------------------------------
    def column_bytes(self, name):
        """The fixed-width raw column as a numpy 'S<width>' array (padding included)."""
        f, s = self._col(name)
        return np.ascontiguousarray(self.records[:, s:s + f.width]).view("S%d" % f.width).reshape(-1)

    def column_str(self, name):
        """list[str] with trailing blanks stripped, as OGR returns string fields."""
        return [b.decode("utf-8", "replace").rstrip(" \0") for b in self.column_bytes(name).tolist()]

    def column_int(self, name, null=-1):
        """int64 [n] of a numeric column; blank / '*' (null) entries become `null`."""
        col = np.char.strip(self.column_bytes(name))
        bad = (col == b"") | (np.char.startswith(col, b"*"))
        out = np.full(col.shape, null, np.int64)
        if (~bad).any():
            good = col[~bad]
            try:
                out[~bad] = good.astype(np.int64)
            except ValueError:                                      # '12.000' style integers
                out[~bad] = good.astype(np.float64).astype(np.int64)
        return out

    def column_float(self, name, null=np.nan):
        col = np.char.strip(self.column_bytes(name))
        bad = (col == b"") | (np.char.startswith(col, b"*"))
        out = np.full(col.shape, null, np.float64)
        if (~bad).any():
            out[~bad] = col[~bad].astype(np.float64)
        return out

    def value(self, rec, name_or_index):
        """One cell with OGR's typing: int / float / str / None (null)."""
        f, s = self._col(name_or_index)
        raw = bytes(self.records[rec, s:s + f.width])
        if f.type == "C":
            return raw.decode("utf-8", "replace").rstrip(" \0")
        txt = raw.strip(b" \0")
        if txt == b"" or txt.startswith(b"*"):
            return None
        if f.type in ("N", "F"):
            if f.is_integer:
                try:
                    return int(txt)
                except ValueError:
                    return int(float(txt))
            return float(txt)
        if f.type == "L":
            return txt[:1] in b"YyTt"
        return txt.decode("ascii", "replace")                      # 'D' and anything else: the text

    # ---- writes -------------------------------------------------------------------------------
    @staticmethod
    def _format(f, v):
        if v is None:
            return b" " * f.width
        if f.type == "C":
            b = str(v).encode("utf-8")[:f.width]
            return b + b" " * (f.width - len(b))
        if f.type in ("N", "F"):
            txt = ("%d" % int(v)) if f.is_integer else ("%.*f" % (f.decimals, float(v)))
            if len(txt) > f.width:                                  # OGR truncates decimals before giving up
                txt = ("%.*g" % (max(1, f.width - 7), float(v)))[:f.width]
            return txt.rjust(f.width).encode("ascii")
        if f.type == "L":
            return (b"T" if v else b"F").ljust(f.width)
        return str(v).encode("ascii")[:f.width].ljust(f.width)

    def set_value(self, rec, name_or_index, v):
        f, s = self._col(name_or_index)
        self.records[rec, s:s + f.width] = np.frombuffer(self._format(f, v), np.uint8)
        self._dirty = True

    def set_column(self, name, values, rows=None):
        """Write a whole column (or the records `rows`) from a sequence / numpy array -- vectorised for numbers."""
        f, s = self._col(name)
        rows = np.arange(len(self)) if rows is None else np.asarray(rows, np.int64)
        values = np.asarray(values)
        if values.shape[0] != rows.shape[0]:
            raise ValueError("one value per record expected")
        if rows.size == 0:
            return
        if f.type in ("N", "F") and values.dtype.kind in "iuf":
            if f.is_integer:
                txt = np.char.mod("%d", values.astype(np.int64))
            else:
                txt = np.char.mod("%%.%df" % f.decimals, values.astype(np.float64))
            txt = np.char.rjust(txt, f.width).astype("S")
            if txt.dtype.itemsize != f.width:
                raise ValueError("a value does not fit field %s N(%d,%d)" % (f.name, f.width, f.decimals))
            self.records[rows, s:s + f.width] = txt.view(np.uint8).reshape(-1, f.width)
        else:
            for r, v in zip(rows.tolist(), values.tolist()):
                self.records[r, s:s + f.width] = np.frombuffer(self._format(f, v), np.uint8)
        self._dirty = True

    def add_field(self, defn: FieldDefn):
        """Append a column (all null), as OGR's CreateField does on a shapefile layer."""
        if self.field_index(defn.name) >= 0:
            raise ValueError("field %s exists" % defn.name)
        self.fields.append(defn)
        pad = np.full((len(self), defn.width), ord(" "), np.uint8)
        self.records = np.concatenate([self.records, pad], axis=1)
        self.record_len += defn.width
        self.header_len = 32 + 32 * len(self.fields) + 1
        self._dirty = True

    def flush(self):
        if not self._dirty:
            return
        if not self.update:
            raise ValueError("{0} was opened read-only".format(self.path))
        write_dbf(self.path, self.fields, records=self.records, ldid=self.ldid)
        self._dirty = False


def _header_bytes(fields, n_records, ldid=0):
    today = datetime.date.today()
    rlen = 1 + sum(f.width for f in fields)
    hlen = 32 + 32 * len(fields) + 1
    head = bytearray(32)
    head[0] = 0x03
    head[1:4] = bytes([today.year - 1900, today.month, today.day])
    struct.pack_into("<IHH", head, 4, n_records, hlen, rlen)
    head[29] = ldid
    out = bytes(head)
    for f in fields:
        d = bytearray(32)
        nm = f.name.encode("ascii")
        d[:len(nm)] = nm
        d[11] = ord(f.type)
        d[16] = f.width & 0xFF
        d[17] = (f.width >> 8) if f.type == "C" else f.decimals
        out += bytes(d)
    return out + b"\x0D"


def write_dbf(path, fields, columns=None, records=None, ldid=0):
    """Write a dBase III table.  Either `columns` = {field name: sequence} or a ready
    [n, record_length] uint8 `records` matrix."""
    fields = [f if isinstance(f, FieldDefn) else FieldDefn(*f) for f in fields]
    if records is None:
        n = len(next(iter(columns.values()))) if columns else 0
        rlen = 1 + sum(f.width for f in fields)
        records = np.full((n, rlen), ord(" "), np.uint8)
        off = 1
        for f in fields:
            vals = columns[f.name]
            if len(vals) != n:
                raise ValueError("column %s has %d values, expected %d" % (f.name, len(vals), n))
            for r, v in enumerate(vals):
                records[r, off:off + f.width] = np.frombuffer(DbfTable._format(f, v), np.uint8)
            off += f.width
    tmp = path + ".tmp"
    with open(tmp, "wb") as fh:
        fh.write(_header_bytes(fields, records.shape[0], ldid))
        fh.write(np.ascontiguousarray(records).tobytes())
        fh.write(b"\x1A")
    os.replace(tmp, path)


# ---------------------------------------------------------------------------------------------
# .shp geometry (points)
# ---------------------------------------------------------------------------------------------
_POINT_TYPES = (1, 11, 21)          # Point, PointZ, PointM


def _shp_header(path):
    try:
        with open(path, "rb") as f:
            raw = f.read()
    except OSError as e:
        raise ValueError("Can not open {0}".format(path)) from e
    if len(raw) < 100 or struct.unpack_from(">i", raw, 0)[0] != 9994:
        raise ValueError("Can not open {0}".format(path))
    return raw, struct.unpack_from("<i", raw, 32)[0]


def read_points(path):
    """-> (X float64 [n], Y float64 [n]) of a point shapefile; null shapes give NaN."""
    raw, shape_type = _shp_header(path)
    if shape_type not in _POINT_TYPES:
        raise ValueError("{0} is not a point shapefile (shape type {1})".format(path, shape_type))
    xs, ys = [], []
    off, end = 100, len(raw)
    while off + 8 <= end:
        (clen,) = struct.unpack_from(">i", raw, off + 4)
        body = off + 8
        (st,) = struct.unpack_from("<i", raw, body) if body + 4 <= end else (0,)
        if st in _POINT_TYPES and body + 20 <= end:
            x, y = struct.unpack_from("<dd", raw, body + 4)
        else:
            x = y = float("nan")
        xs.append(x)
        ys.append(y)
        off = body + 2 * clen
    return np.asarray(xs, np.float64), np.asarray(ys, np.float64)


def shape_type(path):
    return _shp_header(path)[1]


def write_point_shp(path, X, Y):
    """Point .shp + .shx for coordinates X, Y (tests; exporting sample points)."""
    X, Y = np.asarray(X, np.float64), np.asarray(Y, np.float64)
    n = X.shape[0]
    bbox = (float(X.min()), float(Y.min()), float(X.max()), float(Y.max())) if n else (0.0, 0.0, 0.0, 0.0)

    def header(file_words):
        h = bytearray(100)
        struct.pack_into(">i", h, 0, 9994)
        struct.pack_into(">i", h, 24, file_words)
        struct.pack_into("<ii", h, 28, 1000, 1)
        struct.pack_into("<dddd", h, 36, *bbox)
        return bytes(h)

    recs, idx = bytearray(), bytearray()
    for i in range(n):
        idx += struct.pack(">ii", (100 + len(recs)) // 2, 10)
        recs += struct.pack(">ii", i + 1, 10) + struct.pack("<idd", 1, X[i], Y[i])
    base = path[:-4] if path.lower().endswith(".shp") else path
    with open(base + ".shp", "wb") as f:
        f.write(header((100 + len(recs)) // 2) + bytes(recs))
    with open(base + ".shx", "wb") as f:
        f.write(header((100 + len(idx)) // 2) + bytes(idx))


# ---------------------------------------------------------------------------------------------
# the OGR-shaped view the reference's code paths call
# ---------------------------------------------------------------------------------------------
class _Point:
    def __init__(self, x, y):
        self._x, self._y = float(x), float(y)

    def GetX(self, i=0):
        return self._x

    def GetY(self, i=0):
        return self._y


class Feature:
    def __init__(self, layer, fid):
        self._layer, self._fid, self._pending = layer, int(fid), {}

    def GetFID(self):
        return self._fid

    def GetField(self, name_or_index):
        i = name_or_index if isinstance(name_or_index, int) else self._layer.table.field_index(name_or_index)
        if i < 0:
            raise KeyError("no field %r" % (name_or_index,))       # OGR raises too (KeyError since GDAL 3.x)
        if i in self._pending:
            return self._pending[i]
        return self._layer.table.value(self._fid, i)

    def GetFieldAsString(self, name_or_index):
        v = self.GetField(name_or_index)
        return "" if v is None else str(v)

    def SetField(self, name_or_index, value):
        i = name_or_index if isinstance(name_or_index, int) else self._layer.table.field_index(name_or_index)
        if i < 0:
            raise KeyError("no field %r" % (name_or_index,))
        self._pending[i] = value

    def GetGeometryRef(self):
        xy = self._layer.points
        if xy is None or self._fid >= xy[0].shape[0] or np.isnan(xy[0][self._fid]):
            return None
        return _Point(xy[0][self._fid], xy[1][self._fid])


class _LayerDefn:
    def __init__(self, table):
        self._t = table

    def GetFieldIndex(self, name):
        return self._t.field_index(name)

    def GetFieldCount(self):
        return len(self._t.fields)

    def GetFieldDefn(self, i):
        return self._t.fields[i]


class ShapefileLayer:
    """`drv.Open(path, update).GetLayer(0)` of the reference, for the calls made on this path."""

    def __init__(self, path, update=0):
        base = path[:-4] if path.lower().endswith((".shp", ".dbf")) else path
        self.path = path
        self.table = DbfTable(base + ".dbf", update=bool(update))
        self._shp = base + ".shp"
        self._points = False            # not loaded yet
        self._cursor = 0

    @property
    def points(self):
        if self._points is False:
            self._points = None
            if os.path.exists(self._shp) and shape_type(self._shp) in _POINT_TYPES:
                self._points = read_points(self._shp)
        return self._points

    def GetLayerDefn(self):
        return _LayerDefn(self.table)

    def GetFeatureCount(self, force=1):
        return int((~self.table.deleted).sum())

    def ResetReading(self):
        self._cursor = 0

    def GetNextFeature(self):
        n, dele = len(self.table), self.table.deleted
        while self._cursor < n and dele[self._cursor]:
            self._cursor += 1
        if self._cursor >= n:
            return None
        self._cursor += 1
        return Feature(self, self._cursor - 1)

    def __iter__(self):
        self.ResetReading()
        while True:
            f = self.GetNextFeature()
            if f is None:
                return
            yield f

    def GetFeature(self, fid):
        fid = int(fid)
        if fid < 0 or fid >= len(self.table) or self.table.deleted[fid]:
            return None                                             # OGR returns None for a missing FID
        return Feature(self, fid)

    def CreateField(self, defn, approx_ok=1):
        if not isinstance(defn, FieldDefn):                         # a real ogr.FieldDefn
            defn = FieldDefn(defn.GetName(), defn.GetType(), defn.GetWidth() or None, defn.GetPrecision() or None)
        if not self.table.update:
            return 6                                                # OGRERR_FAILURE: layer not opened for update
        self.table.add_field(defn)
        self.table.flush()
        return 0

    def SetFeature(self, feature):
        if not self.table.update:
            return 6
        for i, v in feature._pending.items():
            self.table.set_value(feature.GetFID(), i, v)
        feature._pending.clear()
        self.table.flush()
        return 0

    def SyncToDisk(self):
        self.table.flush()
        return 0


class ShapefileDataSource:
    """`ogr.GetDriverByName("ESRI Shapefile").Open(path, update)`: one layer."""

    def __init__(self, path, update=0):
        self._layer = ShapefileLayer(path, update)

    def GetLayer(self, i=0):
        return self._layer if i == 0 else None

    def GetLayerCount(self):
        return 1


def Open(path, update=0):
    """None when the file cannot be opened, like the OGR driver (callers raise "Can not open ...")."""
    try:
        return ShapefileDataSource(path, update)
    except ValueError:
        return None


# ---------------------------------------------------------------------------------------------
# polygon geometry -> label raster (the step from the reference's vector artefacts to the raster-native path)
# ---------------------------------------------------------------------------------------------
_POLY_TYPES = (5, 15, 25)           # Polygon, PolygonZ, PolygonM


def read_polygons(path):
    """-> list (one entry per record, FID order) of lists of rings, each ring a float64 [k, 2] array of (X, Y);
    null shapes give an empty list.  Outer rings and holes are not distinguished: filling uses the even-odd rule."""
    raw, st = _shp_header(path)
    if st not in _POLY_TYPES:
        raise ValueError("{0} is not a polygon shapefile (shape type {1})".format(path, st))
    out = []
    off, end = 100, len(raw)
    while off + 8 <= end:
        (clen,) = struct.unpack_from(">i", raw, off + 4)
        body = off + 8
        rings = []
        if body + 44 <= end and struct.unpack_from("<i", raw, body)[0] in _POLY_TYPES:
            n_parts, n_points = struct.unpack_from("<ii", raw, body + 36)
            parts = list(struct.unpack_from("<%di" % n_parts, raw, body + 44)) + [n_points]
            pts = np.frombuffer(raw, "<f8", 2 * n_points, body + 44 + 4 * n_parts).reshape(n_points, 2)
            rings = [pts[parts[i]:parts[i + 1]].copy() for i in range(n_parts)]
        out.append(rings)
        off = body + 2 * clen
    return out


def write_polygon_shp(path, polygons):
    """Polygon .shp + .shx; `polygons` = list of lists of rings ([k, 2] arrays, closed or not)."""
    def closed(r):
        r = np.asarray(r, np.float64).reshape(-1, 2)
        return r if len(r) and np.array_equal(r[0], r[-1]) else np.concatenate([r, r[:1]])

    polys = [[closed(r) for r in rings] for rings in polygons]
    allpts = np.concatenate([r for rings in polys for r in rings]) if any(polys) else np.zeros((1, 2))
    bbox = (allpts[:, 0].min(), allpts[:, 1].min(), allpts[:, 0].max(), allpts[:, 1].max())

    def header(file_words):
        h = bytearray(100)
        struct.pack_into(">i", h, 0, 9994)
        struct.pack_into(">i", h, 24, file_words)
        struct.pack_into("<ii", h, 28, 1000, 5)
        struct.pack_into("<dddd", h, 36, *bbox)
        return bytes(h)

    recs, idx = bytearray(), bytearray()
    for i, rings in enumerate(polys):
        if rings:
            pts = np.concatenate(rings)
            starts = np.cumsum([0] + [len(r) for r in rings[:-1]])
            content = struct.pack("<i4dii", 5, pts[:, 0].min(), pts[:, 1].min(), pts[:, 0].max(), pts[:, 1].max(),
                                  len(rings), len(pts))
            content += struct.pack("<%di" % len(rings), *starts.tolist()) + np.ascontiguousarray(pts, "<f8").tobytes()
        else:
            content = struct.pack("<i", 0)
        idx += struct.pack(">ii", (100 + len(recs)) // 2, len(content) // 2)
        recs += struct.pack(">ii", i + 1, len(content) // 2) + content
    base = path[:-4] if path.lower().endswith(".shp") else path
    with open(base + ".shp", "wb") as f:
        f.write(header((100 + len(recs)) // 2) + bytes(recs))
    with open(base + ".shx", "wb") as f:
        f.write(header((100 + len(idx)) // 2) + bytes(idx))


def rasterize_polygons(polygons, geotransform, height, width, nodata=-1, ids=None):
    """int32 [height, width] label raster: a pixel takes the id (default: the polygon's FID) of the polygon that
    contains its CENTRE (even-odd rule over all rings of the polygon, so holes stay empty; the later polygon wins
    where two overlap; pixels in no polygon keep `nodata`, which the RAG kernels treat like the reference's -1 ids).
    North-up rasters only (geotransform[2] == geotransform[4] == 0)."""
    gt = [float(v) for v in geotransform]
    if gt[2] != 0.0 or gt[4] != 0.0 or gt[1] == 0.0 or gt[5] == 0.0:
        raise ValueError("rasterize_polygons needs a north-up geotransform")
    out = np.full((int(height), int(width)), nodata, np.int32)
    for fid, rings in enumerate(polygons):
        if not rings:
            continue
        label = fid if ids is None else int(ids[fid])
        # pixel-space coordinates in which pixel (r, c) has its centre at (c + 0.5, r + 0.5)
        segs = []
        for r in rings:
            r = np.asarray(r, np.float64).reshape(-1, 2)
            if len(r) < 3:
                continue
            px = (r[:, 0] - gt[0]) / gt[1]
            py = (r[:, 1] - gt[3]) / gt[5]
            if px[0] != px[-1] or py[0] != py[-1]:
                px, py = np.append(px, px[0]), np.append(py, py[0])
            segs.append(np.stack([px[:-1], py[:-1], px[1:], py[1:]], axis=1))
        if not segs:
            continue
        s = np.concatenate(segs)
        r0 = max(0, int(np.ceil(min(s[:, 1].min(), s[:, 3].min()) - 0.5)))
        r1 = min(int(height) - 1, int(np.floor(max(s[:, 1].max(), s[:, 3].max()) - 0.5)))
        if r1 < r0:
            continue
        yc = np.arange(r0, r1 + 1, dtype=np.float64) + 0.5                     # [rows]
        x0, y0, x1, y1 = s[:, 0:1], s[:, 1:2], s[:, 2:3], s[:, 3:4]            # [segments, 1]
        crosses = (y0 <= yc) != (y1 <= yc)                                     # half-open rule: no double count at vertices
        with np.errstate(divide="ignore", invalid="ignore"):
            xi = x0 + (yc - y0) * (x1 - x0) / (y1 - y0)
        xi = np.where(crosses, xi, np.inf)
        xi.sort(axis=0)                                                        # crossings of every row, ascending
        n_pairs = int(crosses.sum(axis=0).max()) // 2
        if n_pairs == 0:
            continue
        xa, xb = xi[0:2 * n_pairs:2], xi[1:2 * n_pairs:2]                      # [pairs, rows]: fill [xa, xb)
        ok = np.isfinite(xa) & np.isfinite(xb)
        ca = np.clip(np.ceil(np.where(ok, xa, 0.0) - 0.5), 0, width).astype(np.int64)    # first column with centre >= xa
        cb = np.clip(np.ceil(np.where(ok, xb, 0.0) - 0.5), 0, width).astype(np.int64)    # first column with centre >= xb
        ok &= cb > ca
        if not ok.any():
            continue
        c_lo, c_hi = int(ca[ok].min()), int(cb[ok].max())
        rows = np.broadcast_to(np.arange(yc.shape[0]), ok.shape)[ok]
        d = np.zeros((yc.shape[0], c_hi - c_lo + 1), np.int32)                 # +1 / -1 marks, then a running sum per row
        np.add.at(d, (rows, ca[ok] - c_lo), 1)
        np.add.at(d, (rows, cb[ok] - c_lo), -1)
        inside = np.cumsum(d, axis=1)[:, :-1] > 0
        out[r0:r1 + 1, c_lo:c_hi][inside] = label
    return out


def write_polygonized(path, polys, geotransform, columns=None):
    """Write the rings of a polygonized label raster (deepmerge_b200.polygonize -> Polygons) as a polygon shapefile:
    one record per region present, in ascending id order, with the attributes REGION (the label id) and AREA (pixels)
    and any `columns` = {field name: array indexed by region id} (e.g. MergeResult.perimeter).  A region made of several
    pieces is one multi-ring record (label = record, as in rasterize_polygons), unlike gdal.Polygonize, which writes one
    feature per connected piece."""
    ids, rings = polys.shapes(geotransform)
    base = path[:-4] if path.lower().endswith(".shp") else path
    write_polygon_shp(base + ".shp", rings)
    region = polys.ring_region.cpu().numpy().astype(np.int64)
    area = np.zeros(int(ids.max()) + 1 if len(ids) else 0, np.int64)
    np.add.at(area, region, polys.ring_area.cpu().numpy())
    fields = [FieldDefn("REGION", "N", 11, 0), FieldDefn("AREA", "N", 18, 0)]
    cols = {"REGION": ids, "AREA": area[ids]}
    for name, values in (columns or {}).items():
        a = np.asarray(values.cpu() if hasattr(values, "cpu") else values)[ids]
        fields.append(FieldDefn(name, "N", 18, 0) if np.issubdtype(a.dtype, np.integer) else FieldDefn(name, OFTReal))
        cols[name] = a
    write_dbf(base + ".dbf", fields, cols)
