"""The ABI checks both tracers of the boundary-chain pipeline (dm_polygonize and dm_lines, deepmerge_b200/csrc/chain.cuh)
must pass: test_polygonize_cpu and test_lines_cpu run each of them on their own entry point.  The two entry points take
the same arguments around their outputs, so every check either one had applies to both."""

# entry point -> its workspace query as (lib, H, W, n_regions, capacity), the byte sizes of its output buffers for a
# capacity and n_regions, the index of vertices among them, and whether its workspace grows with n_regions
TRACERS = {
    "dm_polygonize": dict(ws=lambda L, H, W, R, cap: L.dm_polygonize_workspace_bytes(H, W, R, cap),
                          # ring_region, ring_offsets, ring_area, vertices, region_rings
                          outputs=lambda cap, R: (4 * (cap // 4), 8 * (cap // 4) + 8, 8 * (cap // 4), 8 * cap, 8 * R + 8),
                          vertices=3, per_region_ws=True),
    "dm_lines": dict(ws=lambda L, H, W, R, cap: L.dm_lines_workspace_bytes(H, W, cap),
                     # left, right, length, offsets, vertices
                     outputs=lambda cap, R: (4 * cap, 4 * cap, 8 * cap, 8 * cap + 8, 16 * cap),
                     vertices=4, per_region_ws=False),
}


def check_rejects_bad_arguments(entry):
    """The scalar checks, the empty raster and the workspace query of `entry`, without CUDA."""
    from deepmerge_b200 import _lib
    L = _lib.lib()
    bad = _lib.DM_ERR_BAD_ARG
    f = getattr(L, entry)
    ws = lambda H, W, cap, R=10: TRACERS[entry]["ws"](L, H, W, R, cap)    # noqa: E731
    nul = [None] * 6
    assert f(None, 4, 4, 4, 3, 64, *nul, None, 0, None) == bad                  # null pointers with work to do
    assert f(None, -1, 4, 4, 3, 64, *nul, None, 0, None) == bad                 # negative extent
    assert f(None, 4, -1, 4, 3, 64, *nul, None, 0, None) == bad
    assert f(None, 4, 4, 3, 3, 64, *nul, None, 0, None) == bad                  # ld < W
    assert f(None, 4, 4, 4, 3, 1 << 31, *nul, None, 0, None) == bad             # capacity >= 2^31
    assert f(None, 4, 4, 4, 3, -1, *nul, None, 0, None) == bad                  # negative capacity
    assert f(None, 4, 4, 4, -1, 64, *nul, None, 0, None) == bad                 # negative region count
    assert f(None, 1 << 20, 1 << 20, 1 << 20, 3, 64, *nul, None, 0, None) == bad    # more than 2^32 vertices
    assert f(None, 0, 4, 4, 3, 64, *nul, None, 0, None) == 0                    # empty raster
    assert f(None, 4, 0, 0, 3, 64, *nul, None, 0, None) == 0
    assert ws(64, 64, -1) == 0
    assert 0 < ws(64, 64, 1000) < ws(64, 64, 100000)
    assert ws(1024, 1024, 1000) >= 1024 * 1024 // 2     # 4 bits of boundary elements per pixel
    # the polygonizer's workspace holds its bucket sort by region
    assert (ws(64, 64, 1000, R=1 << 22) > ws(64, 64, 1000)) == TRACERS[entry]["per_region_ws"]


def check_no_work_before_an_argument_error(entry):
    """The tracer checks every argument, the workspace size included, before it enqueues anything: a call that returns
    DM_ERR_BAD_ARG or DM_ERR_WORKSPACE has launched no kernel and written no output."""
    import torch
    from deepmerge_b200 import _lib
    L = _lib.lib()
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
    tracer, f = TRACERS[entry], getattr(L, entry)
    R, cap, H, W = 10, 64, 4, 4
    ws = tracer["ws"](L, H, W, R, cap)

    def outs(null=None):    # the output buffers, the one at index `null` a null pointer, then counts
        return [None if k == null else buf(n) for k, n in enumerate(tracer["outputs"](cap, R))] + [buf(32)]

    cases = [
        ("labels", bad, lambda: f(None, H, W, W, R, cap, *outs(), buf(ws), ws, None)),
        ("vertices", bad, lambda: f(buf(4 * H * W), H, W, W, R, cap, *outs(tracer["vertices"]), buf(ws), ws, None)),
        ("workspace pointer", bad, lambda: f(buf(4 * H * W), H, W, W, R, cap, *outs(), None, ws, None)),
        ("ld", bad, lambda: f(buf(4 * H * W), H, W, W - 1, R, cap, *outs(), buf(ws), ws, None)),
        ("workspace", short, lambda: f(buf(4 * H * W), H, W, W, R, cap, *outs(), buf(ws), ws - 1, None)),
    ]
    for name, want, call in cases:
        del probes[:]
        n0 = L.dm_launch_count()
        assert call() == want, name
        assert L.dm_launch_count() == n0, name
        if cuda:
            torch.cuda.synchronize()
            assert all(torch.equal(t, t0) for t, t0 in probes), name
