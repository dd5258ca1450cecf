"""CPU: the C ABI of the spectral merge (dm_score_spectral, dm_merge_select_mutual, dm_merge_apply_regions) is
exported and rejects bad arguments before it enqueues anything; the Python entry points reject bad parameters before
any launch."""
import numpy as np
import pytest
import torch

from deepmerge_b200 import _lib

NAMES = ("dm_score_spectral", "dm_merge_select_mutual_workspace_bytes", "dm_merge_select_mutual", "dm_merge_apply_regions")


@pytest.fixture(scope="module")
def L():
    from deepmerge_b200 import build
    build.build()
    return _lib.lib()


def test_the_new_symbols_are_declared_and_exported(L):
    protos = _lib.parse_header()
    for name in NAMES:
        assert name in protos and hasattr(L.cdll, name), name


def test_workspace_query_is_a_slot_per_region(L):
    assert L.dm_merge_select_mutual_workspace_bytes(0) > 0
    assert L.dm_merge_select_mutual_workspace_bytes(10 ** 5) >= 8 * 10 ** 5
    assert L.dm_merge_select_mutual_workspace_bytes(10 ** 5) < L.dm_merge_select_mutual_workspace_bytes(10 ** 6)


def test_bad_arguments_are_rejected_before_anything_is_enqueued(L):
    """The probe of test_abi_cpu.test_no_work_is_enqueued_before_an_argument_error: with CUDA, device buffers holding a
    sentinel that must survive the call; without, an address nothing may dereference (every CUDA call would fail there
    first with DM_ERR_CUDA), so a bad-argument result shows that no CUDA call was made.  No kernel is counted either."""
    cuda = torch.cuda.is_available()
    probes = []

    def buf(nbytes):
        if not cuda:
            return 16
        # at least one byte and at most 1 MiB: the bad-extent cases (capacity -1 or 2^32) need an address to pass, not
        # the bytes their extent implies
        t = torch.full((min(max(nbytes, 1), 1 << 20),), 0x41 + len(probes), dtype=torch.uint8, device="cuda")
        probes.append((t, t.clone()))
        return t.data_ptr()

    bad, short = _lib.DM_ERR_BAD_ARG, _lib.DM_ERR_WORKSPACE
    R, C, cap = 10, 3, 10
    ws = L.dm_merge_select_mutual_workspace_bytes(R)

    def score(C=C, cap=cap, keys=True, w_shape=0.1, w_cmpct=0.5):
        return L.dm_score_spectral(buf(8 * cap) if keys else None, buf(4 * cap), buf(8), cap, buf(8 * R), buf(8 * R),
                                   buf(8 * R * 3), buf(8 * R * 3), C, buf(16 * R), None, w_shape, w_cmpct, None, buf(4 * cap),
                                   None)

    def select(cap=cap, R=R, scores=True, ws_bytes=ws, n_sel=True):
        return L.dm_merge_select_mutual(buf(4 * cap) if scores else None, 1.0, buf(8 * cap), buf(8), cap, R, buf(cap),
                                        buf(8) if n_sel else None, buf(ws), ws_bytes, None)

    def apply(C=C, R=R, parent=True):
        return L.dm_merge_apply_regions(buf(4 * R) if parent else None, buf(R), buf(R), buf(8 * R), buf(8 * R),
                                        buf(8 * R * 3), buf(8 * R * 3), C, buf(16 * R), R, buf(8), None)

    cases = [
        ("score C = 0", bad, lambda: score(C=0)),
        ("score C < 0", bad, lambda: score(C=-2)),
        ("score negative capacity", bad, lambda: score(cap=-1)),
        ("score null keys", bad, lambda: score(keys=False)),
        ("score shape weight above 1", bad, lambda: score(w_shape=1.5)),
        ("score NaN compactness", bad, lambda: score(w_cmpct=float("nan"))),
        ("select negative capacity", bad, lambda: select(cap=-1)),
        ("select negative regions", bad, lambda: select(R=-1)),
        ("select capacity above 2^32 - 1", bad, lambda: select(cap=1 << 32)),
        ("select null scores", bad, lambda: select(scores=False)),
        ("select no count", bad, lambda: select(n_sel=False)),
        ("select workspace", short, lambda: select(ws_bytes=ws - 1)),
        ("apply C = 0", bad, lambda: apply(C=0)),
        ("apply negative regions", bad, lambda: apply(R=-1)),
        ("apply null parent", bad, lambda: apply(parent=False)),
    ]
    for name, want, call in cases:
        del probes[:]
        n0 = L.dm_launch_count()
        assert call() == want, name
        assert L.dm_launch_count() == n0, name
        if cuda:
            torch.cuda.synchronize()
            assert all(torch.equal(t, t0) for t, t0 in probes), name


def test_python_parameters_are_checked_before_any_launch():
    from deepmerge_b200 import merge_scene_spectral
    lab = np.zeros((4, 4), np.int32)
    img = np.zeros((4, 4, 3), np.uint8)
    ok = dict(n_regions=1, scale=10.0)
    for kw in (dict(scale=0.0), dict(scale=-1.0), dict(scale=float("inf")), dict(scale=float("nan")), dict(scale="x"),
               dict(shape=1.5), dict(shape=-0.1), dict(compactness=2.0), dict(compactness=float("nan")),
               dict(band_weights=[1.0, 1.0]), dict(band_weights=[1.0, -1.0, 1.0]), dict(band_weights=[1.0, float("inf"), 1.0]),
               dict(band_weights=[1.0, 1.0, 1e39])):
        with pytest.raises(ValueError):
            merge_scene_spectral(lab, img, **dict(ok, **kw))
    for image in (None, img.astype(np.float32), img[..., 0], np.zeros((4, 4, 0), np.uint8), np.zeros((4, 5, 3), np.uint8)):
        with pytest.raises(ValueError):
            merge_scene_spectral(lab, image, **ok)


def test_cpu_tensors_are_refused():
    from deepmerge_b200 import RAG, score_spectral
    z = lambda *s, dt=torch.int64: torch.zeros(*s, dtype=dt)
    rag = RAG(z(1), z(1, dt=torch.int32), z(2), z(2), z(2), z(2, 3), z(2, 3), z(2, 4, dt=torch.int32))
    with pytest.raises(ValueError):
        score_spectral(rag)
    with pytest.raises(ValueError):
        score_spectral(RAG(z(1), z(1, dt=torch.int32), z(2), z(2), z(2)))            # no bands / boxes
