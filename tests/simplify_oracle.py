"""Loader of tests/simplify_oracle.c, the sequential simplifier the tests and tools/time_simplify.py compare
dm_polygonize_simplified and dm_lines_simplified against.  TEST INFRASTRUCTURE ONLY.  c_oracle.load builds it; the
unsimplified rings and lines come from polygon_oracle and lines_oracle."""
from __future__ import annotations

import ctypes

import numpy as np

import lines_oracle as lo
import polygon_oracle as po
from c_oracle import load


def lib():
    p, i64, i, d = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_double
    return load("simplify_oracle", {"dmo_simplify": (i64, [p, i64, i64, p, i, i64, i64, d, p]),
                                    "dmo_ring_nodes": (i64, [p, i64, i64, p, p, i64, p, p, p])})


def keep(vertices, offsets, H, W, t, node=None):
    """bool [n] kept vertices of the chains vertices[offsets[k]:offsets[k + 1]]: rings (cyclic, nodes flagged in
    `node`) when node is given, else lines."""
    v = np.ascontiguousarray(vertices, np.int32)
    off = np.ascontiguousarray(offsets, np.int64)
    out = np.zeros(len(v) + 1, np.uint8)
    nd = None if node is None else np.ascontiguousarray(node, np.uint8)
    r = lib().dmo_simplify(v.ctypes.data, off.ctypes.data, len(off) - 1, None if nd is None else nd.ctypes.data,
                           int(nd is not None), H, W, float(t), out.ctypes.data)
    if r < 0:
        raise ValueError("tolerance must be finite and >= 0")
    return out[:len(v)].astype(bool)


def compact(vertices, offsets, k):
    """(vertices [k.sum(), 2], offsets) of the kept vertices k"""
    rank = np.concatenate([[0], np.cumsum(k)]).astype(np.int64)
    return vertices[k], rank[offsets]


def ring_nodes(labels, P):
    """(vertices, offsets, node flags) of the rings of polygon_oracle's P with their nodes added as vertices"""
    L = np.ascontiguousarray(labels, np.int32)
    H, W = L.shape
    v, off = np.ascontiguousarray(P["vertices"], np.int32), np.ascontiguousarray(P["ring_offsets"], np.int64)
    n_max = int(P["counts"][2]) + 1          # at most one vertex per boundary side
    vo, oo, no = np.zeros((n_max, 2), np.int32), np.zeros(len(off), np.int64), np.zeros(n_max, np.uint8)
    n = lib().dmo_ring_nodes(L.ctypes.data, H, W, v.ctypes.data, off.ctypes.data, len(off) - 1, vo.ctypes.data,
                             oo.ctypes.data, no.ctypes.data)
    return vo[:n], oo, no[:n]


def polygons(labels, n_regions, t):
    """dm_polygonize_simplified's outputs as a dict (polygon_oracle.polygonize's keys), plus 'full': the rings with
    their nodes before simplification (vertices, offsets, node flags)."""
    L = np.ascontiguousarray(labels, np.int32)
    H, W = L.shape
    P = po.polygonize(L, n_regions)
    v, off, node = ring_nodes(L, P)
    k = keep(v, off, H, W, t, node)
    P["vertices"], P["ring_offsets"] = compact(v, off, k)
    P["counts"][1] = len(P["vertices"])
    P["full"] = (v, off, node)
    return P


def lines(labels, n_regions, t):
    """dm_lines_simplified's outputs as a dict (lines_oracle.lines' keys), plus 'full': the unsimplified
    (vertices, offsets)."""
    L = np.ascontiguousarray(labels, np.int32)
    H, W = L.shape
    P = lo.lines(L, n_regions)
    v, off = P["vertices"], P["line_offsets"]
    k = keep(v, off, H, W, t)
    P["full"] = (v, off)
    P["vertices"], P["line_offsets"] = compact(v, off, k)
    P["counts"][1] = len(P["vertices"])
    return P
