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
