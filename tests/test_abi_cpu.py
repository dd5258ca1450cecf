"""CPU: the C-ABI library loads, exports every symbol include/deepmerge_b200.h declares, and
rejects bad arguments before touching CUDA.  No compute calls (there is no GPU here)."""
import ctypes
import os
import re

import pytest

from deepmerge_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    from deepmerge_b200 import build
    build.build()
    return _lib.lib()


def test_every_declared_symbol_is_exported(L):
    protos = _lib.parse_header()
    with open(os.path.join(ROOT, "include", "deepmerge_b200.h")) as f:
        declared = set(re.findall(r"\b(dm_\w+)\s*\(", f.read()))
    declared -= {"dm_stream_t"}
    assert declared == set(protos), declared ^ set(protos)
    assert len(protos) >= 45
    for name in protos:
        assert hasattr(L.cdll, name)


def test_the_scene_generator_is_a_library_of_its_own():
    """dm_synth_* (bench / test data) are not part of the product ABI: their own header, their own .so."""
    S = _lib.synth_lib()
    assert set(S.protos) == {"dm_synth_labels", "dm_synth_region_objects", "dm_synth_image", "dm_synth_points", "dm_synth_feats"}
    assert not any(n.startswith("dm_synth") for n in _lib.parse_header())
    product = ctypes.CDLL(_lib.LIB_PATH)
    assert not hasattr(product, "dm_synth_labels")
    assert S.dm_synth_labels(None, 0, -1, 4, 4, 4, 1, 0, None) == _lib.DM_ERR_BAD_ARG


def test_version_and_error_strings(L):
    assert L.dm_version() == 100
    assert L.dm_error_string(0) == b"ok"
    assert b"argument" in L.dm_error_string(_lib.DM_ERR_BAD_ARG)
    assert b"workspace" in L.dm_error_string(_lib.DM_ERR_WORKSPACE)
    assert L.dm_launch_count() == 0                       # nothing has been launched in this process


def test_workspace_queries_are_pure(L):
    a, b = L.dm_rag_workspace_bytes(1000), L.dm_rag_workspace_bytes(100000)
    assert 0 < a < b
    assert L.dm_edges_rekey_workspace_bytes(1 << 20) > (1 << 20) * 8
    assert L.dm_csr_workspace_bytes(0, 5) > 0 and L.dm_merge_apply_workspace_bytes(0) > 0
    assert L.dm_csr_workspace_bytes(1000, 10**6) > L.dm_csr_workspace_bytes(1000, 10)    # per-id arrays for every region
    assert L.dm_sort_edges_workspace_bytes(4096) > 4096 * 12


def test_bad_arguments_are_rejected_without_cuda(L):
    bad = _lib.DM_ERR_BAD_ARG
    assert L.dm_relabel(None, -1, 4, 4, None, 4, None, 4, None) == bad            # negative extent
    assert L.dm_relabel(None, 4, 4, 2, None, 4, None, 4, None) == bad             # pitch < width
    assert L.dm_relabel(None, 4, 4, 4, None, 4, None, 4, None) == bad             # null pointers with work to do
    assert L.dm_relabel(None, 0, 4, 4, None, 0, None, 4, None) == 0               # empty raster is fine
    assert L.dm_score_l2(None, None, 0, None, None, 10, None, None, None) == bad  # D <= 0
    assert L.dm_pool_points_csr(None, None, None, 3, 5, 100, None, None, None) == bad   # ld < D
    assert L.dm_rag_scan(None, 4, 6, 4, 4, None, 0, 0, 4, 1, 1, None, None, None, None, 10, None, None, 0, None) == bad
    assert L.dm_contrastive_fwd_bwd(None, None, None, 0, 100, 1.0, None, None, None, None) == bad
    assert L.dm_resize_area(None, 4, 50, 32, 0, None, None, None, None) == bad        # mode 0 needs an integer factor
    assert L.dm_resize_area(None, 4, 50, 32, 1, None, None, None, None) == bad        # tables / buffers missing
    assert L.dm_resize_area(None, 0, 64, 32, 0, None, None, None, None) == 0          # nothing to do
    # entry points added in round 2
    assert L.dm_relabel_gated(None, 4, 4, 2, None, 4, None, 4, None, None) == bad     # pitch < width
    assert L.dm_relabel_gated(None, 0, 4, 4, None, 0, None, 4, None, None) == 0
    assert L.dm_pool_points_csr_mean(None, None, None, 200, 5, 200, None, None, None, None, None) == _lib.DM_ERR_UNSUPPORTED
    assert L.dm_pool_points_csr_mean(None, None, None, 3, 5, 100, None, None, None, None, None) == bad   # ld < D
    assert L.dm_pool_points_csr_tile(None, None, None, 100, 5, 100, None, None, None, None) == bad       # null pointers
    assert L.dm_peer_allreduce_i32(None, 2, 2, 0, 8, 0, None) == bad                  # rank outside the world
    assert L.dm_peer_allreduce_i32(None, 2, 0, 0, 6, 0, None) == bad                  # n not a multiple of 4
    assert L.dm_peer_allreduce_i32(None, 2, 0, 8, 8, 0, None) == bad                  # offset not a multiple of 16
    assert L.dm_peer_allreduce_i32(None, 2, 0, 0, 8, 2, None) == bad                  # unknown op
    assert L.dm_peer_allreduce_i32(None, 2, 0, 0, 0, 1, None) == 0                    # nothing to reduce
    assert L.dm_slots_word_max(None, 2, 80, 12, None, None) == bad                    # unaligned word / no output
    assert L.dm_region_bbox(None, 4, 4, 2, 3, None, None, None) == bad                # pitch < width
    assert L.dm_points_id_range(None, -1, 3, None, None) == bad
    with pytest.raises(ValueError):
        L.check(bad, "x")
    with pytest.raises(RuntimeError):
        L.check(_lib.DM_ERR_WORKSPACE, "x")


def test_missing_library_fails_loudly(tmp_path):
    with pytest.raises(RuntimeError, match="no CPU or PyTorch fallback"):
        _lib.Library(str(tmp_path / "libnope.so"))


def test_cpu_tensors_are_refused():
    import torch
    from deepmerge_b200 import build_rag, score_l2
    with pytest.raises(ValueError):
        build_rag(torch.zeros((4, 4), dtype=torch.int32), 2)
    with pytest.raises(ValueError):
        score_l2(torch.zeros((2, 4)), torch.zeros(1, dtype=torch.int64))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "deepmerge_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                with open(os.path.join(dirpath, fn)) as f:
                    src = f.read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn
                assert "/root/reference" not in src, fn


def test_no_work_is_enqueued_before_an_argument_error(L):
    """An entry point checks every argument, the workspace size included, before it enqueues anything: a call that
    returns DM_ERR_BAD_ARG or DM_ERR_WORKSPACE has launched no kernel and written no output."""
    import torch
    cuda = torch.cuda.is_available()
    probes = []

    def buf(nbytes):
        # With CUDA: device memory holding a sentinel of its own, which must survive the call.  Without: an address
        # that nothing may dereference -- every CUDA call fails there first (DM_ERR_CUDA), so a bad-argument result
        # shows that no CUDA call was made.
        if not cuda:
            return 16
        t = torch.full((nbytes,), 0x41 + len(probes), dtype=torch.uint8, device="cuda")
        probes.append((t, t.clone()))
        return t.data_ptr()

    bad, short = _lib.DM_ERR_BAD_ARG, _lib.DM_ERR_WORKSPACE
    R, D, cap, H, W = 10, 4, 10, 4, 4
    merge_ws, rag_ws = L.dm_merge_apply_workspace_bytes(R), L.dm_rag_workspace_bytes(cap)

    def merge_stats():      # alive, changed, sum, cnt, area, perimeter, R, D, n_merged
        return buf(R), buf(R), buf(4 * R * D), buf(4 * R), buf(8 * R), buf(8 * R), R, D, buf(8)

    def rag_head(labels):   # labels, rows_own, rows_avail, W, ld, image, C, pitch, n_regions, borders, area, border, bands
        return labels, H, H, W, W, None, 0, 0, R, 1, 1, buf(8 * R), buf(8 * R), None, None

    cases = [
        ("dm_merge_select_l2", bad, lambda: L.dm_merge_select_l2(None, 0.5, buf(8), cap, buf(cap), buf(8), None)),
        ("dm_merge_select_mlp", bad, lambda: L.dm_merge_select_mlp(None, 2, buf(8), cap, buf(cap), buf(8), None)),
        ("dm_merge_apply_masked", bad,
         lambda: L.dm_merge_apply_masked(None, *merge_stats(), None, buf(merge_ws), merge_ws, None)),
        ("dm_merge_apply", bad, lambda: L.dm_merge_apply(None, *merge_stats(), buf(merge_ws), merge_ws, None)),
        ("dm_merge_apply_masked workspace", short,
         lambda: L.dm_merge_apply_masked(buf(4 * R), *merge_stats(), None, buf(merge_ws), merge_ws - 1, None)),
        ("dm_rows_pack", bad, lambda: L.dm_rows_pack(None, buf(4 * R * D), R, D, buf(4 * cap), buf(4 * cap * D), cap,
                                                      buf(8), None)),
        ("dm_shard_frontier_pairs", bad,
         lambda: L.dm_shard_frontier_pairs(None, buf(R), buf(4 * R), 0, R, buf(80 + 8 * cap), cap, None)),
        ("dm_perimeter", bad, lambda: L.dm_perimeter(None, buf(4 * cap), buf(8), cap, buf(8 * R), buf(8 * R), R, None)),
        ("dm_points_id_range", bad, lambda: L.dm_points_id_range(None, 10, R, buf(16), None)),
        ("dm_region_bbox", bad, lambda: L.dm_region_bbox(None, H, W, W, R, buf(16 * R), buf(8), None)),
        ("dm_rag_scan", bad, lambda: L.dm_rag_scan(*rag_head(None), cap, buf(32), buf(rag_ws), rag_ws, None)),
        ("dm_rag_build", bad, lambda: L.dm_rag_build(*rag_head(None), buf(8 * cap), buf(4 * cap), cap, buf(32),
                                                      buf(rag_ws), rag_ws, None)),
        ("dm_rag_scan workspace", short,
         lambda: L.dm_rag_scan(*rag_head(buf(4 * H * W)), cap, buf(32), buf(rag_ws), rag_ws - 1, None)),
    ]
    for name, want, call in cases:
        del probes[:]
        n0 = L.dm_launch_count()
        assert call() == want, name
        assert L.dm_launch_count() == n0, name
        if cuda:
            torch.cuda.synchronize()
            assert all(torch.equal(t, t0) for t, t0 in probes), name


def _csrc():
    """file name -> text of every CUDA source of the library"""
    csrc = os.path.join(ROOT, "deepmerge_b200", "csrc")
    srcs = {}
    for fn in sorted(os.listdir(csrc)):
        if fn.endswith((".cu", ".cuh")):
            with open(os.path.join(csrc, fn)) as f:
                srcs[fn] = f.read()
    return srcs


def test_every_launch_goes_through_the_launch_helper():
    """Kernels are launched only by launch() and launch_cooperative() of common.cuh, which count a launch once the
    runtime accepted it and read and clear its error; the grid rule of the grid-stride kernels is defined there once."""
    srcs = _csrc()
    for fn, src in srcs.items():
        for token in ("<<<", "cudaLaunch"):
            assert src.count(token) == (1 if fn == "common.cuh" else 0), (fn, token)
        assert "DM_COUNT_LAUNCH" not in src and "DM_LAUNCH_CHECK" not in src, fn
    body = lambda name: re.search(r"\bint %s\(.*?\n\}" % name, srcs["common.cuh"], flags=re.S).group(0)
    assert "<<<" in body("launch") and "cudaLaunch" in body("launch_cooperative")
    defs = [fn for fn, src in srcs.items() for _ in re.finditer(r"\bgrid_for\s*\(\s*(const\s+)?(int64_t|long long|int)\s", src)]
    assert defs == ["common.cuh"], defs


def test_workspace_queries_measure_the_carve():
    """A workspace query returns the extent of the carve that lays the workspace out, so the bytes a caller allocates
    and the pieces an entry point takes cannot disagree: no query sums piece sizes by hand, and only Carver rounds."""
    srcs = _csrc()
    assert [fn for fn, src in srcs.items() if re.search(r"\balign_up\b", src)] == ["common.cuh"]
    queries = {}
    for fn, src in srcs.items():
        for m in re.finditer(r'extern "C" size_t (dm_\w+_workspace_bytes)\(([^)]*)\)\s*\{(.*?)\n?\}\n', src, flags=re.S):
            queries[m.group(1)] = m.group(3)
    with open(os.path.join(ROOT, "include", "deepmerge_b200.h")) as f:
        assert set(queries) == set(re.findall(r"\b(dm_\w+_workspace_bytes)\s*\(", f.read()))
    for name, body in queries.items():
        assert not re.search(r"[+*]", body), name
        returns = re.findall(r"\breturn\b([^;]*);", body)
        # the last return measures a carve; an earlier one may only answer 0 for extents the entry point rejects
        assert returns and all(r.strip() == "0" for r in returns[:-1]), (name, returns)
        assert re.fullmatch(r"\s*[\w:]+\(.*\)(\.bytes)?\s*", returns[-1], flags=re.S), (name, returns[-1])
