#!/usr/bin/env python
"""bench.py -- headline benchmark of the region-merging hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

A step = one end-to-end pass (RAG + band pooling -> point pooling -> L2 edge scoring ->
iterative union-find merge -> relabel) over the synthetic scene of SURVEY.md section 8(d).
N=1 workload: BASELINE.json configs[1] (10k x 10k, 4 bands, ~100k segments).  Prints ONE
JSON line (rank 0).  `value` = Mpx/s with inputs resident in HBM; `e2e` = the same through
the public API with HOST buffers (H2D of labels/image/points/embeddings and D2H of the label
map inside the timed region); `roofline` = the fused RAG+pool raster kernel against the
measured HBM peak; `cpu_baseline` = the oracle port timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CFG = dict(H=10000, W=10000, R=100000, C=4, P=4, D=100, tau=0.5, seed=1234)
WORKLOAD = "configs[1]: 10k x 10k 4-band synthetic scene, ~100k segments, single B200 RAG+pool+score+merge"
FALLBACK_HBM_GBS = 6650.0


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed ncu capture
    (profiles/traffic.json, written by tools/profile_summary.py for the same workload); None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return float(json.load(f)[kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region with NVML (in-process thread,
    ~2 ms period; nvidia-smi is too slow to start for a region this short)."""

    def __init__(self, index=0):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        except Exception as e:          # no NVML: report that, never fake a clock record
            self.err = repr(e)
        return self

    def _run(self):
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def __exit__(self, *a):
        self._stop.set()
        if self._t:
            self._t.join(timeout=1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle port on a bounded sample of the same workload
# ----------------------------------------------------------------------------------------------
def cpu_sample_dims(cfg, side):
    """A side x side crop-equivalent of the workload: same region pitch, bands, P and D."""
    scale = (side * side) / (cfg["H"] * cfg["W"])
    return dict(cfg, H=side, W=side, R=max(4, int(round(cfg["R"] * scale))))


def run_cpu_port(cfg, steps=1, warmup=0):
    """Times oracle_np.merge_scene + band pooling (numpy, 1 thread) on the given scene."""
    from oracle import oracle_np as o
    sc = o.synth_scene(cfg["H"], cfg["W"], cfg["R"], C=cfg["C"], P=cfg["P"], D=cfg["D"], seed=cfg["seed"])
    times = []
    res = None
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        res = o.merge_scene(sc["labels"], sc["n_regions"], sc["region_of_point"], sc["feats"], tau=cfg["tau"])
        o.pool_bands(sc["labels"], sc["image"], sc["n_regions"])
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return float(np.min(times)), res["merges"], sc["n_regions"]


_BARRIER = None


def _cpu_init(barrier):
    global _BARRIER
    _BARRIER = barrier
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[k] = "1"


def _cpu_worker(args):
    """One process = one sample scene: generate it, then `warmup` untimed and `steps` timed passes; every pass starts at
    a barrier of all processes, and (start, end) of every timed pass is returned."""
    cfg, steps, warmup = args
    from oracle import oracle_np as o
    sc = o.synth_scene(cfg["H"], cfg["W"], cfg["R"], C=cfg["C"], P=cfg["P"], D=cfg["D"], seed=cfg["seed"])
    spans = []
    for k in range(warmup + steps):
        _BARRIER.wait()
        t0 = time.time()
        res = o.merge_scene(sc["labels"], sc["n_regions"], sc["region_of_point"], sc["feats"], tau=cfg["tau"])
        o.pool_bands(sc["labels"], sc["image"], sc["n_regions"])
        if k >= warmup:
            spans.append((t0, time.time()))
    return spans, res["merges"], sc["n_regions"]


def run_cpu_port_parallel(cfg, steps=1, procs=None, warmup=1):
    """The oracle port on ALL host cores: the numpy path is single-threaded, so `procs` processes each
    run it on their own sample scene (different seeds) side by side; a pass takes (last finish - first start) over the
    processes, and the BEST of the `steps` timed passes after `warmup` untimed ones is reported (BASELINE.md section 4:
    one warm-up, best of 3).  Returns (seconds per step, merges of one sample, segments, procs)."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64) if procs is None else procs)
    if procs == 1:
        sec, merges, R = run_cpu_port(cfg, steps=steps, warmup=warmup)
        return sec, merges, R, 1
    ctx = mp.get_context("spawn")
    jobs = [(dict(cfg, seed=cfg["seed"] + i), steps, warmup) for i in range(procs)]
    with ctx.Pool(procs, initializer=_cpu_init, initargs=(ctx.Barrier(procs),)) as pool:
        out = pool.map(_cpu_worker, jobs, chunksize=1)
    walls = [max(o[0][k][1] for o in out) - min(o[0][k][0] for o in out) for k in range(steps)]
    return min(walls), out[0][1], out[0][2], procs


def cpu_baseline_record(cfg, side, steps=3, warmup=1):
    ccfg = cpu_sample_dims(cfg, side)
    sec, merges, R, procs = run_cpu_port_parallel(ccfg, steps=steps, warmup=warmup)
    mpx = procs * ccfg["H"] * ccfg["W"] / sec / 1e6
    sample = (f"{procs} x {ccfg['H']}x{ccfg['W']} scenes at the workload's region pitch ({R} segments each), "
              f"{ccfg['C']} bands; numpy oracle port, one process per scene on {procs} of {os.cpu_count()} host cores; "
              f"{warmup} warm-up pass, best of {steps}")
    return {"value": mpx, "unit": "Mpx/s", "cores": procs, "kind": "port", "sample": sample}, sec, merges * procs


DUMP_MAX_ELEMS = 1 << 19        # per array: the 13 files written for a MergeResult stay below 64 MB in all


def dump_outputs(path, res, seed=0):
    """Writes every field of a MergeResult as path/<field>.npy so that two builds can be compared output for output:
    integers as float64 (exact below 2**53), floats as float32.  An array of more than DUMP_MAX_ELEMS elements is
    replaced by a sample of its flattened elements at seeded positions, the same in every run of the same workload.
    A float field holds NaN by design where a region has no sample points (its mean is NaN, its edges score NaN and are
    never selected): such values are written as 0, and path/<field>_finite.npy holds 1 where the value is finite and 0
    where it is not, so every file holds finite numbers and nothing is lost."""
    import dataclasses
    import torch
    os.makedirs(path, exist_ok=True)
    for f in dataclasses.fields(res):
        v = getattr(res, f.name)
        if isinstance(v, int):
            v = torch.tensor(v)
        if not isinstance(v, torch.Tensor):         # MergeEngine.run leaves the initial graph out (rag is None)
            continue
        if v.numel() > DUMP_MAX_ELEMS:
            idx = np.unique(np.random.default_rng(seed).integers(0, v.numel(), DUMP_MAX_ELEMS))
            v = v.reshape(-1)[torch.from_numpy(idx).to(v.device)]
        a = v.cpu().numpy()
        if a.dtype.kind == "f":
            ok = np.isfinite(a)
            np.save(os.path.join(path, f.name + "_finite.npy"), ok.astype(np.float32))
            a = np.where(ok, a, 0).astype(np.float32)
        else:
            a = a.astype(np.float64)
        np.save(os.path.join(path, f.name + ".npy"), a)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(args.warmup, 0)
    rec, sec, merges = cpu_baseline_record(CFG, args.cpu_side, steps=steps, warmup=warmup)
    line = {
        "impl": "reference", "metric": "megapixels/sec end-to-end (RAG+pool+score+merge+relabel)", "value": rec["value"],
        "unit": "Mpx/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32/u8 index + fp32 scores",
        "data": "synthetic", "config": {"workload": WORKLOAD, "sample": rec["sample"]},
        "cpu_baseline": rec,
        "e2e": {"value": rec["value"], "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "merged_edges_per_s": merges / sec,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def b200_arm(args):
    import torch
    import torch.distributed as dist
    from deepmerge_b200 import MergeEngine, _lib
    from deepmerge_b200.raster import _p, _stream
    from deepmerge_b200.synth import synth_scene

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        from deepmerge_b200.sharded import bench_sharded
        if world != 8 or args.config2 or args.side:
            return bench_sharded(args, CFG, WORKLOAD, dist, dev, ClockSampler, measured_peaks)
        # N = 8: the weak-scaling line (the contract's metric), and BASELINE.json configs[2] -- ONE 40k x 40k scene with 1M
        # segments over the 8 GPUs, the north-star target -- measured in the same job as the extra key "config2"
        line = bench_sharded(args, CFG, WORKLOAD, dist, dev, ClockSampler, measured_peaks, emit=False)
        import copy
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        a2 = copy.copy(args)
        a2.config2, a2.steps = True, max(3, args.steps // 2)
        l2 = bench_sharded(a2, CFG, WORKLOAD, dist, dev, ClockSampler, measured_peaks, emit=False)
        if rank == 0:
            line["config2"] = {k: l2[k] for k in ("value", "unit", "ms_per_step", "steps", "scaling", "parity_ok", "parity",
                                                  "ms_per_step_gathered", "rounds", "segments_after", "gpu_launches")}
            line["config2"]["workload"] = l2["config"]["workload"]
            line["config2"]["e2e_ms_per_step"] = l2["e2e"]["ms_per_step"]
            print(json.dumps(line), flush=True)
        dist.barrier()
        dist.destroy_process_group()
        return

    L = _lib.lib()
    cfg = dict(CFG)
    if args.side:
        cfg = cpu_sample_dims(CFG, args.side)
    H, W, C, D = cfg["H"], cfg["W"], cfg["C"], cfg["D"]
    sc = synth_scene(H, W, cfg["R"], C=C, P=cfg["P"], D=D, seed=cfg["seed"], device=dev)
    R, N = sc.n_regions, sc.feats.shape[0]
    eng = MergeEngine(H, W, R, D, C=C, n_points=N, device=dev)

    def step():
        return eng.run(sc.labels, sc.feats, cfg["tau"], image=sc.image, xs=sc.xs, ys=sc.ys)

    for _ in range(max(args.warmup, 3)):
        res = step()
    torch.cuda.synchronize()
    E0 = None

    # ---- device-resident timing: exactly K steps in one bracket ------------------------------------
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = L.dm_launch_count()
    with ClockSampler(local) as clocks:
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            res = step()
        ev1.record()
        torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = (L.dm_launch_count() - launches0)
    mpx = H * W / ms / 1e3
    if args.dump_outputs:               # res holds views of the engine's buffers: write them before anything else runs
        dump_outputs(args.dump_outputs, res)

    # ---- the dominant kernel alone (fused RAG + band pooling raster pass), CUDA events -------------
    s = _stream()
    k0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    k1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for i in range(args.steps):
        eng.stats.zero_()
        k0[i].record()
        L.check(L.dm_rag_scan(_p(sc.labels), H, H, W, W, _p(sc.image), C, W * C, R, 1, 1, _p(eng.area), _p(eng.border),
                              _p(eng.bsum), _p(eng.bsq), eng.cap, _p(eng.counts), _p(eng.ws), eng.ws_bytes, s), "scan")
        k1[i].record()
    torch.cuda.synchronize()
    rag_ms = float(np.mean([a.elapsed_time(b) for a, b in zip(k0, k1)]))
    rag = eng.run(sc.labels, sc.feats, cfg["tau"], image=sc.image, xs=sc.xs, ys=sc.ys, max_rounds=0)
    E0 = int(rag.edge_keys.shape[0])
    alg_bytes = (4 + C) * H * W + 12 * E0 + 16 * R * C
    peak, peak_kind = measured_peaks()
    achieved = alg_bytes / (rag_ms * 1e-3) / 1e9
    res = step()
    # (a MergeResult holds views of the engine's buffers: keep what the line reports before the engine runs anything else)
    root_l2 = res.root.clone()
    n_roots = int((root_l2 == torch.arange(R, device=dev, dtype=torch.int32)).sum())
    res_rounds, res_merges = res.rounds, res.merges

    # ---- end to end through the public API with HOST buffers -----------------------------------------
    # ScenePipeline: every step copies its inputs from pinned host memory and its label map back; the
    # copies of neighbouring steps overlap the compute on separate streams (full-duplex PCIe).  The
    # un-pipelined single call (merge_scene semantics) is reported next to it.
    from deepmerge_b200 import ScenePipeline
    host = {k: getattr(sc, k).cpu().pin_memory() for k in ("labels", "image", "feats", "xs", "ys")}
    h2d = sum(t.numel() * t.element_size() for t in host.values())
    d2h = H * W * 4
    pipe = ScenePipeline(eng)
    for _ in pipe.run((host for _ in range(3)), cfg["tau"]):
        pass
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_out = 0
    for lab in pipe.run((host for _ in range(args.steps)), cfg["tau"]):
        n_out += 1
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    assert n_out == args.steps
    eng.out = pipe.dev_out[0]

    out_host = pipe.host_out[0]

    def e2e_step():
        d = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        r = eng.run(d["labels"], d["feats"], cfg["tau"], image=d["image"], xs=d["xs"], ys=d["ys"])
        out_host.copy_(r.labels, non_blocking=True)
        torch.cuda.synchronize()
        return r

    e2e_step()
    t0 = time.perf_counter()
    for _ in range(max(1, args.steps // 3)):
        e2e_step()
    e2e_single_ms = (time.perf_counter() - t0) * 1e3 / max(1, args.steps // 3)

    # ---- the pair-MLP scorer (R8) on the scene's edges: tcgen05 kernel timed alone ------------------------------
    mlp_rec = None
    try:
        from deepmerge_b200 import PackedMLP
        g = torch.Generator(device="cpu").manual_seed(1)
        hid, n_out = 250, 2
        mk = lambda *sh: (torch.randn(*sh, generator=g) / (sh[-1] ** 0.5)).to(dev)
        mlp = PackedMLP(mk(hid, 2 * D), mk(hid), mk(hid, hid), mk(hid), mk(n_out, hid), mk(n_out))
        keys0 = rag.edge_keys.contiguous()
        n0 = torch.tensor([E0], dtype=torch.int64, device=dev)
        o_buf = torch.empty((E0, n_out), dtype=torch.float32, device=dev)
        m0 = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        m1 = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
        for i in range(6):
            m0[i].record()
            L.check(L.dm_score_mlp_bf16(_p(eng.mean), D, _p(keys0), _p(n0), E0, _p(mlp.blob), 2 * D, hid, n_out, _p(o_buf),
                                        None, s), "mlp")
            m1[i].record()
        torch.cuda.synchronize()
        mlp_ms = float(np.mean([a.elapsed_time(b) for a, b in zip(m0[1:], m1[1:])]))
        useful = 2.0 * E0 * (2 * D * hid + hid * hid + hid * n_out)
        padded = 2.0 * E0 * (256 * 256 + 256 * 256 + 256 * 16)
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                tpeak = float(json.load(f)["bf16_tflops"])
        except Exception:
            tpeak = 1590.0
        mlp_rec = {"kernel": "pair_mlp_kernel (tcgen05, 200->250->250->2 on every edge)", "ms": mlp_ms, "edges": E0,
                   "tflops_useful": useful / mlp_ms / 1e9, "tflops_padded": padded / mlp_ms / 1e9, "peak_bf16_tflops": tpeak,
                   "frac_useful": useful / mlp_ms / 1e9 / tpeak, "frac_padded": padded / mlp_ms / 1e9 / tpeak,
                   "scored_edges_per_s": E0 / (mlp_ms * 1e-3)}
    except Exception as ex:                              # never hide it: the record says what failed
        mlp_rec = {"error": repr(ex)}

    # ---- the whole step with the pair-MLP as the scorer (R8 inside the merge loop) --------------------------------
    # a hand-made "same object?" network: logit 0 = L1 distance of the two pooled embeddings (leaky-ReLU pairs), logit 1
    # a constant -- it takes the same decisions as the L2 scorer on this scene, so the two steps do the same merges
    mlp_step = None
    try:
        from deepmerge_b200 import PackedMLP
        W1 = torch.zeros((2 * D, 2 * D))
        i = torch.arange(D)
        W1[i, i], W1[i, D + i], W1[D + i, i], W1[D + i, D + i] = 1.0, -1.0, -1.0, 1.0
        W3 = torch.zeros((2, 2 * D))
        W3[0] = 1.0
        l1net = PackedMLP(W1.to(dev), torch.zeros(2 * D, device=dev), torch.eye(2 * D, device=dev),
                          torch.zeros(2 * D, device=dev), W3.to(dev), torch.tensor([0.0, 4.0], device=dev))

        def step_m():
            return eng.run(sc.labels, sc.feats, 0.0, image=sc.image, xs=sc.xs, ys=sc.ys, mlp=l1net)

        for _ in range(3):
            rm = step_m()
        km = max(3, args.steps // 3)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(km):
            rm = step_m()
        ev1.record()
        torch.cuda.synchronize()
        l1net.check()
        mlp_step = {"scorer": "pair-MLP 200->200->200->2 (tcgen05), every live edge every round", "ms_per_step": ev0.elapsed_time(ev1) / km,
                    "value": H * W / (ev0.elapsed_time(ev1) / km) / 1e3, "unit": "Mpx/s", "rounds": rm.rounds, "merges": rm.merges,
                    "same_roots_as_l2": bool(torch.equal(rm.root, root_l2))}
    except Exception as ex:
        mlp_step = {"error": repr(ex)}

    # ---- a multi-round workload: embeddings whose merges cascade over three rounds (deepmerge_b200.synth.cascade_feats) ---
    multi = None
    try:
        from deepmerge_b200.synth import CASCADE_TAU, cascade_feats
        cf = cascade_feats(sc, D)

        def step_c(mr=64):
            return eng.run(sc.labels, cf, CASCADE_TAU, image=sc.image, xs=sc.xs, ys=sc.ys, max_rounds=mr)

        kc = max(3, args.steps // 3)
        cum, edges_live = [], []
        for mr in (0, 1, 2, 3, 64):
            for _ in range(2):
                rc = step_c(mr)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(kc):
                rc = step_c(mr)
            ev1.record()
            torch.cuda.synchronize()
            cum.append(ev0.elapsed_time(ev1) / kc)
            edges_live.append(int(rc.edge_keys.shape[0]))
        ms_c = cum[-1]
        scored = sum(edges_live[:rc.rounds + 1])                    # E_0 (all edges) + the live edges after every round but the last
        multi = {"workload": f"{H}x{W}, {R} segments, cascade embeddings (regions -> objects -> 4x4 groups -> 4x4 groups of groups), "
                             f"tau {CASCADE_TAU}", "rounds": rc.rounds, "ms_per_step": ms_c, "value": H * W / ms_c / 1e3, "unit": "Mpx/s",
                 "merges": rc.merges, "segments_after": int((rc.root == torch.arange(R, device=dev, dtype=torch.int32)).sum()),
                 "live_edges_after_round_0_1_2_3": edges_live[:4], "ms_with_max_rounds_0_1_2_3": cum[:4],
                 "ms_per_round_1_2_3": [cum[i + 1] - cum[i] for i in range(3)],
                 "scored_edges": scored, "scored_edges_per_s": scored / (ms_c * 1e-3), "merged_edges_per_s": rc.merges / (ms_c * 1e-3)}
    except Exception as ex:
        multi = {"error": repr(ex)}

    # ---- configs[3] micro-bench: adjacent-pair sampling + row gather + contrastive loss forward / backward at B = 960 -----
    train = None
    try:
        import random
        from deepmerge_b200 import MyUtils1
        from deepmerge_b200.Losses import Loss
        B = 960
        lo_all, hi_all = rag.edge_keys >> 32, rag.edge_keys & 0xFFFFFFFF
        npairs = min(100000, int(lo_all.shape[0]))
        lo_h, hi_h = lo_all[:npairs].cpu().numpy(), hi_all[:npairs].cpu().numpy()
        obj = sc.region_obj.cpu().numpy()
        flags = (obj[lo_h] == obj[hi_h]).astype(np.int64)
        off = np.zeros(R + 1, np.int64)
        rop_h = sc.region_of_point.cpu().numpy()
        order = np.argsort(np.where(rop_h >= 0, rop_h, R), kind="stable")
        np.cumsum(np.bincount(rop_h[rop_h >= 0], minlength=R), out=off[1:])
        fields = {}

        class Fields:                               # PointID strings of the polygons, built when a pair asks for them
            def __getitem__(self, r):
                f = fields.get(r)
                if f is None:
                    f = fields[r] = " ".join(str(int(v)) for v in order[off[r]:off[r + 1]]) or "0"
                return f

        crit = Loss(1.0, 0.1, 0)
        random.seed(1)
        sel = np.random.default_rng(1).integers(0, npairs, size=(8, B))

        def train_step(k):
            pairs = [(int(lo_h[j]), int(hi_h[j])) for j in sel[k % 8]]
            left, right, _ = MyUtils1.pairs_to_arrays(MyUtils1.sample_pairs(Fields(), pairs, 0))
            flag = flags[sel[k % 8]]
            li, ri = torch.from_numpy(left).to(dev, non_blocking=True), torch.from_numpy(right).to(dev, non_blocking=True)
            a_rows = torch.empty((B, D), dtype=torch.float32, device=dev)
            b_rows = torch.empty((B, D), dtype=torch.float32, device=dev)
            L.check(L.dm_gather_rows(_p(sc.feats), D, _p(li), B, _p(a_rows), s), "dm_gather_rows")
            L.check(L.dm_gather_rows(_p(sc.feats), D, _p(ri), B, _p(b_rows), s), "dm_gather_rows")
            a_rows.requires_grad_(True)
            loss = crit(a_rows, b_rows, torch.from_numpy(flag).to(dev, non_blocking=True))
            loss.backward()
            return loss

        for k in range(3):
            train_step(k)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        kt = max(8, args.steps)
        for k in range(kt):
            lossv = train_step(k)
        torch.cuda.synchronize()
        tms = (time.perf_counter() - t0) * 1e3 / kt
        train = {"workload": "configs[3] micro-bench: per step 960 labelled adjacent pairs -> one random member point per side "
                             "(random.randint, as MyUtils1.py:278-279) -> dm_gather_rows x 2 -> Loss forward + backward",
                 "batch": B, "ms_per_step": tms, "pairs_per_s": B / (tms * 1e-3), "loss": float(lossv.item()),
                 "note": "host-bound: the reference's per-pair Python sampling dominates (the three kernels take ~20 us)"}
    except Exception as ex:
        train = {"error": repr(ex)}

    # ---- configs[0]: 1024 x 1024, 3 bands, ~2k segments, MLP merge -- next to the reference-STYLE CPU path --------------
    # (the embeddings are the synthetic ones: the ShiftScaleFormer that produces them in the reference is outside this
    # build, and it is left out of BOTH arms)
    config0 = None
    try:
        s0 = synth_scene(1024, 1024, 2000, C=3, P=cfg["P"], D=D, seed=cfg["seed"], device=dev)
        e0 = MergeEngine(1024, 1024, s0.n_regions, D, C=3, n_points=s0.feats.shape[0], device=dev)

        def step0(mlp_):
            return e0.run(s0.labels, s0.feats, 0.0 if mlp_ is not None else cfg["tau"], image=s0.image, xs=s0.xs, ys=s0.ys, mlp=mlp_)

        rec0 = {}
        for name, m_ in (("mlp", l1net), ("l2", None)):
            for _ in range(3):
                r0 = step0(m_)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(20):
                r0 = step0(m_)
            ev1.record()
            torch.cuda.synchronize()
            rec0[name] = {"ms_per_step": ev0.elapsed_time(ev1) / 20, "rounds": r0.rounds, "merges": r0.merges}
        # reference-style CPU path (BASELINE.md section 4.1): the per-edge loop of ExtractFeatures.py:164-222, one thread
        cpu0 = None
        if not args.no_cpu:
            from oracle import oracle_np as o
            g0 = e0.run(s0.labels, s0.feats, cfg["tau"], image=s0.image, xs=s0.xs, ys=s0.ys, max_rounds=0)
            k0h = g0.edge_keys.cpu().numpy()
            lo0, hi0 = (k0h >> 32).astype(np.int64), (k0h & 0xFFFFFFFF).astype(np.int64)
            rop0 = s0.region_of_point.cpu().numpy()
            off0, ids0 = o.csr_from_region_of_point(rop0, s0.n_regions)
            fields0 = [" ".join(str(int(v)) for v in ids0[off0[r]:off0[r + 1]]) for r in range(s0.n_regions)]
            ok = np.array([fields0[a] != "" and fields0[b] != "" for a, b in zip(lo0, hi0)])
            store0 = s0.feats.cpu().numpy()
            t0 = time.perf_counter()
            simi0 = o.edge_loop_reference_style(store0, fields0, lo0[ok], hi0[ok])
            loop_s = time.perf_counter() - t0
            t0 = time.perf_counter()
            o.merge_scene(s0.labels.cpu().numpy(), s0.n_regions, rop0, store0, tau=cfg["tau"])
            port_s = time.perf_counter() - t0
            cpu0 = {"reference_style_edge_loop_s": loop_s, "edges": int(ok.sum()), "edges_per_s": float(ok.sum()) / loop_s,
                    "kind": "port of ExtractFeatures.py:164-222 (per-edge gather by np.concatenate, np.mean, Euclidean_distance), "
                            "1 host core, scores only", "vectorised_port_whole_step_s": port_s,
                    "max_abs_diff_vs_gpu_scores": float(np.nanmax(np.abs(simi0 - g0.scores.cpu().numpy()[: len(k0h)][ok])))}
        config0 = {"workload": "configs[0]: 1024 x 1024 3-band tile, %d segments, %d edges, synthetic embeddings (no ShiftScaleFormer in "
                               "either arm)" % (s0.n_regions, int(e0.run(s0.labels, s0.feats, cfg["tau"], image=s0.image, xs=s0.xs, ys=s0.ys,
                                                                          max_rounds=0).edge_keys.shape[0])),
                   "gpu_step_pair_mlp": rec0["mlp"], "gpu_step_l2": rec0["l2"], "cpu": cpu0}
        del e0, s0
    except Exception as ex:
        config0 = {"error": repr(ex)}

    # ---- CPU baseline: the oracle port on a bounded sample, same box, all host cores ---------------------------
    cpu = None
    if not args.no_cpu:
        cpu, _, _ = cpu_baseline_record(cfg, min(args.cpu_side, H), steps=3, warmup=1)

    line = {
        "metric": "megapixels/sec end-to-end (RAG+pool+score+merge+relabel)", "value": mpx, "unit": "Mpx/s",
        "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32/u8 index + fp32 scores", "data": "synthetic",
        "config": {"workload": WORKLOAD if not args.side else f"{H}x{W} reduced scene", "H": H, "W": W, "bands": C,
                   "segments": R, "edges": E0, "points": N, "embed_dim": D, "tau": cfg["tau"],
                   "l2_policy": "inputs (labels+image 800 MB) larger than L2, no flush needed"},
        "merged_edges_per_s": res_merges / (ms * 1e-3), "scored_edges_per_s": E0 / (ms * 1e-3),
        "segments_after": n_roots, "rounds": res_rounds,
        "e2e": {"value": H * W / e2e_ms / 1e3, "unit": "Mpx/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "api": "ScenePipeline.run (H2D / compute / D2H of neighbouring steps overlap)",
                "unpipelined_ms_per_step": e2e_single_ms, "unpipelined_value": H * W / e2e_single_ms / 1e3},
        "gpu_launches": launches,
        "roofline": {"kernel": "rag_blocks_kernel (fused RAG + band pooling raster pass)", "bound": "hbm",
                     "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": achieved / peak,
                     "frac_of_nominal_8TBs": achieved / 8000.0, "ms": rag_ms, "algorithmic_bytes": alg_bytes,
                     "traffic": ncu_traffic("rag_blocks_kernel") if not args.side else None,
                     "traffic_source": "profiles/traffic.json (ncu --set full capture of this kernel on this workload)"},
        "mlp": mlp_rec, "mlp_step": mlp_step, "multi_round": multi, "train_pairs": train, "config0": config0, "cpu_baseline": cpu,
        "clocks": clocks.summary(),
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--side", type=int, default=0, help="debug: run a reduced side x side scene instead of configs[1]")
    ap.add_argument("--cpu-side", type=int, default=3000,
                    help="side of the bounded CPU sample scenes (one per host core; ~1.4 s of numpy work each per step)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true",
                    help="N > 1: skip the (untimed) check of the sharded answer against the single-GPU engine on rank 0")
    ap.add_argument("--config2", action="store_true",
                    help="N > 1 only: run BASELINE.json configs[2] (ONE 40k x 40k scene, ~1M segments, split over the ranks) "
                         "instead of the weak-scaling stack of configs[1] tiles")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="single GPU: write the result of the last timed step as DIR/<field>.npy (float32 / float64; "
                         "fields above %d elements as a fixed, seeded sample; non-finite floats as 0, flagged in "
                         "DIR/<field>_finite.npy)" % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs the single-GPU b200 run")
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
