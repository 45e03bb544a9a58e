#!/usr/bin/env python
"""bench.py -- SOM-codebook hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU, torchrun for N > 1)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)
    python bench.py --gpus 1 --steps K --dump-outputs DIR    # + the last timed step's codebook and loss as DIR/*.npy

Headline workload at every N (BASELINE.json `metric` = patches/sec BMU+update; configs[3], C4): ONE SOM training step
of /root/reference/train_codebook.py:225-249 -- BMU search + neighbourhood-weighted update + Adam -- at P=4 (D=64),
K=16 384 units, on a FIXED GLOBAL batch of 16 384 synthetic 4x32x32 feature maps = 1 048 576 patches per step, split
over the N ranks (patch-sharded data parallel, STRONG scaling).  Every step of every N > 1 run contains the NCCL
all-reduce of the packed per-unit accumulators (4 MB) inside the timed region; the whole step is a CUDA graph.
`value` has the batches resident in HBM; `e2e` feeds the same step from pinned HOST memory through somcb.HostTrainer
(H2D copy of every batch and D2H read of every loss inside the timed region).  `extra` carries BASELINE configs[1]
(C2, BMU-only tokenisation, with its own roofline and e2e), configs[4] (C5, unit-sharded search + histogram over the
N ranks), C1 / C3 step times, and -- for N > 1 -- in-run parity checks (replicas identical, DP == 1-GPU trainer,
sharded search == unsharded search).  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "quantized-autoregression-image-generator_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# NCCL prints "NCCL version ..." on STDOUT at NCCL_DEBUG=VERSION (and INFO); the contract is ONE JSON line there.
# An explicit INFO / TRACE request is left alone.
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

import torch  # noqa: E402

METRIC = "patches/sec BMU+update (SOM training step P=4 D=64 K=16384, 1 048 576 patches per step over all GPUs)"
UNIT = "patches/s"
C4 = dict(n_fmaps=16384, patch=(4, 4), K=16384, C=4, H=32, W=32, D=64, seq=64, lr=1e-4, neighbourhood_step=200)
C2 = dict(n_fmaps=39063, patch=(2, 2), K=4096, C=4, H=32, W=32)
WORKLOAD = ("BASELINE configs[3] (C4): SOM training step (BMU + neighbourhood update + Adam, "
            "train_codebook.py:225-249), P=4 (D=64), K=16384 trained-like codebook, range 8192, fixed global batch of "
            "16 384 synthetic 4x32x32 fmaps = 1 048 576 patches per step, patch-sharded over the GPUs")
CONFIG = {"workload": WORKLOAD, "global_patches_per_step": C4["n_fmaps"] * C4["seq"], "D": 64, "K": 16384,
          "parallelism": "patch-sharded data parallel, one all-reduce of the packed accumulators per step"}
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
L2_BYTES = 126 << 20


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        d["_source"] = "measured (MEASURED_PEAKS.json)"
        return d
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback (B200_PROFILING.md)"
    return d


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML (~1 kHz) while the timed region runs."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = str(e)

    def _loop(self):
        nv = self.nv
        names = {}
        for nm in dir(nv):
            if nm.startswith("nvmlClocksEventReason") or nm.startswith("nvmlClocksThrottleReason"):
                val = getattr(nv, nm)
                if isinstance(val, int) and val:
                    names.setdefault(val, nm.replace("nvmlClocksEventReason", "")
                                     .replace("nvmlClocksThrottleReason", ""))
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if mask & bit and bit & (bit - 1) == 0:
                        self.reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.001)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "no NVML samples"}
        s = sorted(self.samples)
        reasons = sorted(r for r in self.reasons if r not in ("GpuIdle", "None", "ApplicationsClocksSetting"))
        return {"sm_mhz": s[len(s) // 2], "sm_min_mhz": s[0], "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md 8d): tanh(randn) fmaps, trained-like codebooks -- restated here so that the measured
# arm imports nothing from oracle/
# ---------------------------------------------------------------------------------------------------------------
def _trained_like_codebook(k, patch, seed=7):
    import somcb
    p_h, p_w = patch
    seq = (32 // p_h) * (32 // p_w)
    n_fmaps = max(2, (2 * k + seq - 1) // seq)
    g = torch.Generator().manual_seed(1000 + seed)
    pool = somcb.patchify(torch.tanh(torch.randn(n_fmaps, 4, 32, 32, generator=g)), patch)
    pool = pool.reshape(-1, pool.shape[-1])
    g2 = torch.Generator().manual_seed(int(seed))
    pick = torch.randperm(pool.shape[0], generator=g2)[:k]
    return pool[pick].clone().contiguous()


def _fmaps(n, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.empty(n, 4, 32, 32, device=dev)
    for lo in range(0, n, 8192):
        hi = min(n, lo + 8192)
        x[lo:hi] = torch.tanh(torch.randn(hi - lo, 4, 32, 32, generator=g, device=dev))
    return x


def _codebook(k, patch, dev, rng=None, seed=7):
    import somcb
    cb = somcb.Codebook(patch_dim=patch, image_dim=(32, 32), image_channel=4, num_embeddings=k,
                        init_neighbour_range=k // 2 if rng is None else rng)
    with torch.no_grad():
        cb.codebook.weight.copy_(_trained_like_codebook(k, patch, seed))
    return cb.to(dev) if dev is not None else cb


def _timed(fn, reps, warm=2):
    """Average device time of fn (ms), CUDA events on the current stream."""
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _log(msg):
    """Progress on stderr (rank 0): a hang shows where it happened; stdout stays ONE JSON line."""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def _max_over_ranks(ms, dev, world):
    import torch.distributed as dist
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


# ---------------------------------------------------------------------------------------------------------------
# the reference arm: the reference's own CPU implementation of the step (oracle port) on a 128-fmap sample of the
# batch, for as many steps as --steps asks
# ---------------------------------------------------------------------------------------------------------------
def _cpu_reference_step(steps, warmup, sample_fmaps=128, min_seconds=0.0):
    """train_codebook.py:225-249 on the host cores at the C4 shape, 8192 patches per step (the reference's dense N x K
    temporaries need 16*N*K bytes, BASELINE.md 3): patches/s."""
    from oracle.step_oracle import (make_oracle_codebook, make_reference_optimizer, reference_step,
                                    synthetic_fmaps, trained_like_codebook)
    torch.set_num_threads(os.cpu_count() or 1)
    w = trained_like_codebook(C4["K"], C4["patch"], 7)
    cb = make_oracle_codebook(w, C4["patch"], (32, 32), 4, C4["K"] // 2)
    opt = make_reference_optimizer(cb, C4["lr"])
    x = synthetic_fmaps(sample_fmaps, 123)
    n_p = sample_fmaps * C4["seq"]
    for _ in range(warmup):
        reference_step(cb, opt, x)
    t0 = time.perf_counter()
    done = 0
    while done < steps or (time.perf_counter() - t0) < min_seconds:
        reference_step(cb, opt, x)
        done += 1
    dt = time.perf_counter() - t0
    return {"value": n_p * done / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{done} steps x {n_p} patches (a {sample_fmaps}-fmap sample of the 16 384-fmap step; the "
                      f"reference's dense N x K temporaries do not fit more), oracle restatement of "
                      f"train_codebook.py:225-249 + models/Codebook.py on torch {torch.__version__} CPU, {dt:.1f} s"}, \
        dt / done


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    base, s_per_step = _cpu_reference_step(steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": CONFIG, "cpu_baseline": base,
            "steps_run": steps,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
# headline: the C4 step, strong-scaled
# ---------------------------------------------------------------------------------------------------------------
def _make_trainer(cb, world, graph=True, tail="auto", wt="full"):
    import somcb
    kw = dict(lr=C4["lr"], neighbourhood_step=C4["neighbourhood_step"], use_cuda_graph="alias" if graph else False)
    return somcb.DataParallelSom(cb, tail=tail, wt=wt, **kw) if world > 1 else somcb.SomTrainer(cb, **kw)


def run_headline(args, dev, world, rank, peaks):
    import somcb
    import torch.distributed as dist
    from somcb import ops
    lib = somcb._lib.load()
    lo, hi = somcb.shard_bounds(C4["n_fmaps"], world, rank)
    share = hi - lo
    share_bytes = share * 4 * 32 * 32 * 4
    n_rot = max(2, -(-(256 << 20) // share_bytes))           # rotate through >= 256 MB of distinct batches (> L2)
    n_rot = min(n_rot, 8)
    # global batch b = fmaps of seed 5000 + b (generated per rank for its own contiguous share: seeds differ per rank)
    xs = [_fmaps(share, 5000 + 131 * b + rank, dev) for b in range(n_rot)]
    cb = _codebook(C4["K"], C4["patch"], dev)
    tr = _make_trainer(cb, world, tail=args.tail, wt=args.wt)
    if world > 1:
        tr.broadcast_weights(0)
    tail_mode = getattr(tr, "tail", "single")
    _log(f"trainer ready (tail: {tail_mode})")
    # set-up (untimed, before the warm-up): one eager step (kernel attributes, NCCL communicator), then one graph
    # capture per rotation buffer
    l0 = lib.som_launch_count()
    tr.step(xs[0])
    launches_per_step = int(lib.som_launch_count() - l0)
    for b in range(n_rot):
        tr.step(xs[b])
    torch.cuda.synchronize()
    it = 0
    for _ in range(args.warmup):
        tr.step(xs[it % n_rot])
        it += 1
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    with ClockSampler(dev.index) as clk:
        e0.record()
        for _ in range(args.steps):
            loss = tr.step(xs[it % n_rot])
            it += 1
        e1.record()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms_step = _max_over_ranks(e0.elapsed_time(e1), dev, world) / args.steps
    n_global = C4["n_fmaps"] * C4["seq"]
    value = n_global / (ms_step * 1e-3)
    # what a caller holds after the last timed step: the codebook it updated in place and the loss it returned (read
    # here, before the end-to-end run below trains the same codebook further)
    outputs = {"codebook_weight": cb.codebook.weight.detach().cpu().numpy(),
               "loss": loss.detach().reshape(1).cpu().numpy()} if args.dump_outputs else None
    loss = float(loss)
    assert loss == loss and 0.0 < loss < float("inf"), f"implausible loss {loss}"

    _log(f"headline timed: {ms_step:.3f} ms/step")
    # ---- end to end: pinned host batches -> H2D -> step -> loss D2H, every step ----------------------------------
    e2e_steps = args.e2e_steps or min(args.steps, 20)
    cpus_before = os.sched_getaffinity(0)
    numa_node = somcb.bind_host_to_gpu_node(dev)
    hosts = [torch.empty(share, 4, 32, 32, pin_memory=True) for _ in range(2)]
    for b in range(2):
        hosts[b].copy_(xs[b])
    ht = somcb.HostTrainer(tr, depth=2)
    pend = None
    for b in range(4):                                       # graph capture on the two staging buffers + warm-up
        pend = ht.step(hosts[b % 2])
    pend.item()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    prev = None
    for b in range(e2e_steps):
        cur = ht.step(hosts[b % 2])
        if prev is not None:
            prev.item()                                      # the host reads every step's loss (one step behind)
        prev = cur
    last_loss = prev.item()
    f1.record()
    torch.cuda.synchronize()
    e2e_ms = _max_over_ranks(f0.elapsed_time(f1), dev, world) / e2e_steps
    # copy floor: the same H2D bytes alone, all ranks at once
    dst = torch.empty_like(xs[0])

    def h2d():
        dst.copy_(hosts[0], non_blocking=True)
    if world > 1:
        dist.barrier()
    floor_ms = _max_over_ranks(_timed(h2d, 5, warm=1), dev, world)
    os.sched_setaffinity(0, cpus_before)
    del hosts, ht, dst
    e2e = {"value": n_global / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms, "steps": e2e_steps,
           "h2d_bytes_per_step": share * 4 * 32 * 32 * 4, "d2h_bytes_per_step": 8,
           "bytes_note": "per rank: its share of the step's fmaps in, the loss scalar out",
           "copy_floor_ms": floor_ms, "frac_of_copy_floor": floor_ms / e2e_ms,
           "api": "somcb.HostTrainer(trainer).step(pinned fmaps) -> PendingLoss.item()", "host_numa_node": numa_node,
           "last_loss": last_loss}

    _log(f"e2e timed: {e2e_ms:.3f} ms/step (copy floor {floor_ms:.3f})")
    # ---- per-kernel breakdown of one rank's step (each op timed alone, CUDA events) ------------------------------
    x = xs[0]
    geom = ops.geometry(x.shape, C4["patch"])
    w = cb.codebook.weight.data
    k, d, rng = C4["K"], C4["D"], cb.neighbourhood_range
    cn = ops.prepare_codebook(w)
    wt = ops.neighbourhood_filter(w, rng)
    bmu = ops.bmu(x, geom, w, cn)
    packed = torch.empty(k * d + 4, dtype=torch.float32, device=dev)
    ops.accumulate_packed(x, geom, bmu, wt, k, packed=packed)
    wc, mc, vc = w.clone(), torch.zeros_like(w), torch.zeros_like(w)
    tdev = torch.tensor([1, 0], dtype=torch.int64, device=dev)
    grad = ops.neighbourhood_filter(packed[:k * d].view(k, d), rng)
    reps = 10
    parts = {"filter_W": _timed(lambda: ops.neighbourhood_filter(w, rng), reps),
             "norms": _timed(lambda: ops.prepare_codebook(w), reps),
             "bmu": _timed(lambda: ops.bmu(x, geom, w, cn), reps),
             "accumulate": _timed(lambda: ops.accumulate_packed(x, geom, bmu, wt, k, packed=packed), reps),
             "filter_Rbar": _timed(lambda: ops.neighbourhood_filter(packed[:k * d].view(k, d), rng), reps),
             "adam": _timed(lambda: ops.adam_step_dp(wc, mc, vc, grad, d, 1e-4, tdev, packed[k * d:]), reps)}
    if world > 1:
        scratch = packed.clone()
        dist.barrier()
        parts["nccl_all_reduce_4MB (reference point)"] = _timed(lambda: dist.all_reduce(scratch), reps)
    if world > 1 and tail_mode == "peer":
        # the sharded tail replaces filter_W / filter_Rbar / adam / all_reduce above by their per-slice forms
        lo_u, hi_u, g0, g1, max_own, max_halo = tr._slices(ops.filter_half_width(k, rng))
        if 4 * max_halo <= 3 * k and hi_u > lo_u:
            pm, mc = tr.peer, tr._mc
            sig, rk = pm.signal_ptrs, pm.rank
            rsum = torch.empty(g1 - g0, d, dtype=torch.float32, device=dev)
            tl = torch.empty(4, dtype=torch.float32, device=dev)
            wth = ops.neighbourhood_filter(w[g0:g1], rng)
            mm, vv = torch.zeros(hi_u - lo_u, d, device=dev), torch.zeros(hi_u - lo_u, d, device=dev)
            ops.peer_reduce_rows(mc["packed"], tr._peer_packed, k, d, g0, g1, max_halo, rsum, tl, rk, world, sig, 1)
            gh = ops.neighbourhood_filter(rsum, rng)
            dist.barrier()
            for name in ("filter_Rbar", "adam"):
                parts.pop(name)
            if tr.wt_mode == "slice":
                parts.pop("filter_W")
                parts["slice: filter_W rows"] = _timed(lambda: ops.neighbourhood_filter(w[g0:g1], rng), reps)
                parts["slice: multicast W~ rows + barrier"] = _timed(
                    lambda: ops.peer_bcast_rows(wth[lo_u - g0:hi_u - g0], mc["wt"] + lo_u * d * 4, max_own * d, rk, world, sig, 0), reps)
            scratch = torch.empty(max_halo, d, dtype=torch.float32, device=dev)
            parts["slice: filter_Rbar rows, in-switch reduce of the rows + halo fused into its read"] = _timed(
                lambda: ops.peer_reduce_filter_rows(mc["packed"], tr._peer_packed, k, d, g0, g1, max_halo, rng, scratch, gh,
                                                    tl, rk, world, sig, 1), reps)
            # (Adam here re-broadcasts the CURRENT rows: lr = 0 keeps the replicas' weights unchanged)
            parts["slice: adam + multicast W rows + barrier"] = _timed(
                lambda: ops.peer_adam_slice(w[lo_u:hi_u], mc["w"] + lo_u * d * 4, mm, vv, gh[lo_u - g0:hi_u - g0], max_own * d,
                                            d, 0.0, tdev, tl, rk, world, sig, 2), reps)
    parts = {kk: _max_over_ranks(v, dev, world) for kk, v in parts.items()}
    ksum = sum(v for kk, v in parts.items() if "reference point" not in kk)
    breakdown = {kk: {"ms": v, "pct_of_step": 100.0 * v / ms_step} for kk, v in parts.items()}
    breakdown["sum_of_parts_ms"] = ksum
    breakdown["graph_step_ms"] = ms_step
    breakdown["note"] = ("each op timed alone (eager, its own pre-pass launches included) on one rank's share, max "
                         "over ranks; the step itself is one CUDA-graph replay.  Ops of a few microseconds are bound by "
                         "the eager launch path here (a filter call: ~32 us eager, 15-32 us on the GPU): "
                         "tools/graph_time.py has their GPU times from graph replay")

    # ---- roofline of the dominant kernel (BMU) --------------------------------------------------------------------
    n_local = share * C4["seq"]
    flops = 2.0 * k * d * n_local
    achieved = flops / (parts["bmu"] * 1e-3) / 1e12
    mode = os.environ.get("SOM_BMU_VARIANT_NOTE", "")
    split = lib.som_bmu_split_mode(n_local, d, k) if hasattr(lib, "som_bmu_split_mode") else 0
    f16 = split == 1
    peak_burst = peaks["bf16_tflops"] / (3.0 if f16 else 6.0)
    peak_sust = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]) / (3.0 if f16 else 6.0)
    traffic, pipe_pct, src = None, None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        key = "bmu_c4_f16" if f16 else "bmu_c4"
        per_patch = tj.get(key + "_dram_bytes_per_patch")
        traffic = per_patch * n_local if per_patch else None
        pipe_pct = tj.get(key + "_tensor_pipe_active_pct")
        src = tj.get(key + "_source")
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak_burst, "unit": "TFLOP/s",
                "frac": achieved / peak_burst, "traffic": traffic,
                "traffic_source": (f"DRAM bytes per patch of one ncu --set full capture x the patches of this launch: "
                                   f"{src}; not measured in this run" if traffic is not None else None),
                "kernel": ("bmu_tc_l16 (tcgen05 kind::f16, FP16 hi/lo split x3 products, fp32 accumulate in TMEM)" if f16
                           else "bmu_tc_l (tcgen05 kind::tf32 x3)"),
                "peak_basis": (f"{peaks['_source']}: BURST cuBLAS bf16 {peaks['bf16_tflops']} TFLOP/s / 3 (three 16-bit "
                               "products per fp32-faithful product)" if f16 else
                               f"{peaks['_source']}: BURST cuBLAS bf16 / 2 (tf32) / 3 (3xTF32)"),
                "frac_of_sustained_basis": achieved / peak_sust,
                "launch_ms": parts["bmu"], "patches_per_launch": n_local,
                "algorithmic_flops_per_patch": 2 * k * d, "algorithmic_bytes_per_patch": 4 * d + 8,
                "hbm_frac": (4 * d + 8) * n_local / (parts["bmu"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "tensor_pipe_active_pct_ncu": pipe_pct, "note": mode or None}
    head = {"value": value, "ms_per_step": ms_step, "loss": loss, "outputs": outputs, "clocks": clk.summary(), "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps, "roofline": roofline, "breakdown": breakdown,
            "details": {"fmaps_per_rank": share, "patches_per_rank": n_local, "rotation_buffers": n_rot,
                        "launches_per_step": launches_per_step,
                        "launch_note": "kernels of libsomcb per step, replayed from one CUDA graph per rotation buffer "
                                       "(+ the NCCL all-reduce kernel for N > 1)",
                        "l2": f"each rank rotates through {n_rot} distinct resident batches "
                              f"({n_rot * share_bytes >> 20} MB > the 126 MB L2), so no step re-reads a batch that is "
                              "still L2 resident",
                        "dp_tail": tail_mode,
                        "allreduce_bytes_per_step": (k * d + 4) * 4 if world > 1 else 0}}
    return head, tr, cb, xs


# ---------------------------------------------------------------------------------------------------------------
# in-run parity checks at N > 1
# ---------------------------------------------------------------------------------------------------------------
def run_checks(tr, cb, dev, world, rank):
    import somcb
    import torch.distributed as dist
    from somcb import ops
    out = {}
    # (1) replicas bit-identical after the timed steps
    w = cb.codebook.weight.data
    ref = w.clone()
    dist.broadcast(ref, src=0)
    same = torch.tensor([1 if torch.equal(ref, w) else 0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    out["replicas_bit_identical_after_timed_steps"] = bool(int(same))
    # (2) DP over the ranks == a 1-GPU trainer on the whole 65 536-patch batch (2 steps, same start)
    x = _fmaps(1024, 777, dev)                               # same seed on every rank: the same global batch
    cb_dp, cb_one = _codebook(C4["K"], C4["patch"], dev), _codebook(C4["K"], C4["patch"], dev)
    dp = somcb.DataParallelSom(cb_dp, lr=1e-4, neighbourhood_step=200)
    one = somcb.SomTrainer(cb_one, lr=1e-4, neighbourhood_step=200)
    rel_l = 0.0
    for _ in range(2):
        l_dp = dp.step(somcb.split_batch(x, world, rank).contiguous())
        l_one = one.step(x)
        rel_l = max(rel_l, abs(float(l_dp) - float(l_one)) / abs(float(l_one)))
    w_dp, w_one = cb_dp.codebook.weight.data.double(), cb_one.codebook.weight.data.double()
    rel_w = torch.tensor([float((w_dp - w_one).norm() / w_one.norm()), rel_l], device=dev, dtype=torch.float64)
    dist.all_reduce(rel_w, op=dist.ReduceOp.MAX)
    # weights: 1e-6 (SURVEY 8c.4).  loss: 5e-6 -- the sharded tail filters W per slice with the FFMA kernel where the
    # one-GPU trainer uses the tensor-core (3xTF32) filter on the whole codebook; the two agree to ~3e-7 on W~, which
    # shows up 2x in the squared error (the reduction of the loss itself is exact: fp64 over the ranks' tails)
    out["dp_vs_single_gpu_2_steps_65536_patches"] = {"weights_rel_fro": float(rel_w[0]), "loss_rel": float(rel_w[1]),
                                                     "tolerance": {"weights": 1e-6, "loss": 5e-6},
                                                     "ok": bool(rel_w[0] <= 1e-6 and rel_w[1] <= 5e-6)}
    # (3) unit-sharded search over the ranks == the unsharded search (same codebook, 65 536 patches)
    wfull = cb_one.codebook.weight.data
    geom = ops.geometry(x.shape, C4["patch"])
    full = ops.bmu(x, geom, wfull)
    lo, hi = somcb.shard_bounds(C4["K"], world, rank)
    got = somcb.sharded_bmu(x, geom, wfull[lo:hi].contiguous(), lo)
    diff = torch.nonzero(got != full).flatten()
    ok = True
    if diff.numel():
        flat = somcb.patchify(x, C4["patch"]).reshape(-1, 64)[diff].double()
        da = (flat - wfull[got[diff]].double()).norm(dim=1)
        db = (flat - wfull[full[diff]].double()).norm(dim=1)
        ok = bool(((da - db).abs() <= 1e-6 * db).all())
    flag = torch.tensor([1 if ok else 0, int(diff.numel())], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["sharded_bmu_vs_unsharded_65536_patches"] = {"index_differences": int(diff.numel()),
                                                    "all_within_1e-6_fp64_distance": bool(int(flag[0]))}
    out["all_ok"] = bool(out["replicas_bit_identical_after_timed_steps"] and
                         out["dp_vs_single_gpu_2_steps_65536_patches"]["ok"] and int(flag[0]))
    return out


# ---------------------------------------------------------------------------------------------------------------
# extras: C2 (BMU-only tokenisation), C5 (unit-sharded search + histogram), C1 / C3
# ---------------------------------------------------------------------------------------------------------------
def extra_c2(dev, peaks, steps=10):
    import somcb
    lib = somcb._lib.load()
    cb = _codebook(C2["K"], C2["patch"], dev)
    cb.eval()
    x = _fmaps(C2["n_fmaps"], 123, dev)
    n_p = C2["n_fmaps"] * 256
    with torch.no_grad():
        ms = _timed(lambda: cb.get_patches_bmu(x, reshape=True), steps, warm=3)
        idx = cb.get_patches_bmu(x, reshape=True)
    counts = somcb.ops.histogram(idx.reshape(-1), C2["K"])
    assert int(counts.sum()) == n_p
    host = torch.empty(C2["n_fmaps"], 4, 32, 32, pin_memory=True)
    host.copy_(x)
    out_host = torch.empty(C2["n_fmaps"], 256, dtype=torch.int64, pin_memory=True)
    tok = somcb.HostTokenizer(cb, chunk_fmaps=4096, depth=3)
    e2e_ms = _timed(lambda: tok.tokenize(host, out_host), 5, warm=2)
    assert torch.equal(out_host, idx.cpu()), "e2e indices differ from the resident-input run"
    dst = torch.empty_like(x)
    floor_ms = _timed(lambda: dst.copy_(host, non_blocking=True), 3, warm=1)
    flops = 2.0 * C2["K"] * 16 * n_p
    achieved = flops / (ms * 1e-3) / 1e12
    f16 = (lib.som_bmu_split_mode(n_p, 16, C2["K"]) == 1) if hasattr(lib, "som_bmu_split_mode") else True
    peak = peaks["bf16_tflops"] / (3.0 if f16 else 6.0)
    return {"workload": "BASELINE configs[1] (C2): 39 063 fmaps, P=2 (D=16), K=4096, 10 000 128 patches, BMU only",
            "value": n_p / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
            "dtype": "f32 (fp16 hi/lo x3 screen, fp32 accumulate, exact fp32 resolve of the winning chunk)",
            "e2e": {"value": n_p / (e2e_ms * 1e-3), "ms_per_step": e2e_ms, "h2d_bytes_per_step": host.numel() * 4,
                    "d2h_bytes_per_step": out_host.numel() * 8, "copy_floor_ms": floor_ms,
                    "frac_of_copy_floor": floor_ms / e2e_ms,
                    "api": "somcb.HostTokenizer.tokenize(pinned fmaps) -> pinned int64 indices (synchronous)"},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak,
                         "peak_basis": f"{peaks['_source']}: BURST cuBLAS bf16 / 3 (three 16-bit products)",
                         "kernel": "bmu_tc_s<F16> (tcgen05 kind::f16)"}}


def extra_c5(dev, world, rank):
    """configs[4]: D=256, K=262 144 units sharded over the ranks (K/N per GPU), 1 048 576 replicated patches (a
    131 072-patch sample when one GPU holds all units), all-gather + merge + sharded histogram."""
    import somcb
    import torch.distributed as dist
    from somcb import ops
    from somcb.distributed import sharded_bmu, sharded_histogram
    k_total = 262144
    lo, hi = somcb.shard_bounds(k_total, world, rank)
    n_f = 65536 if world >= 4 else 8192 * world
    x = _fmaps(n_f, 123, dev)
    gw = torch.Generator(device=dev).manual_seed(500 + rank)
    w_shard = torch.tanh(torch.randn(hi - lo, 256, generator=gw, device=dev))
    geom = ops.geometry(x.shape, (8, 8))
    cn = ops.prepare_codebook(w_shard)
    state = {}

    def search():
        idx = sharded_bmu(x, geom, w_shard, lo, c_norm2=cn)
        state["counts"] = sharded_histogram(idx, lo, hi)

    search()
    if world > 1:
        dist.barrier()
    ms = _max_over_ranks(_timed(search, 2, warm=0), dev, world)
    n_p = ops.n_patches_of(geom)
    tot = state["counts"].sum().to(torch.int64)
    if world > 1:
        dist.all_reduce(tot)
    assert int(tot) == n_p, f"sharded histogram sums to {int(tot)}, expected {n_p}"
    return {"workload": f"BASELINE configs[4] (C5): D=256, K=262 144 units in {world} shard(s) of {hi - lo}, "
                        f"{n_p} patches, candidates all-gathered and merged, sharded hit histogram",
            "ms": ms, "patches_per_s": n_p / (ms * 1e-3), "unit_patch_pairs_per_s": n_p * k_total / (ms * 1e-3),
            "fp32_faithful_tflops_all_gpus": 2.0 * 256 * k_total * n_p / (ms * 1e-3) / 1e12}


def extra_small_configs(dev):
    import somcb
    from somcb import ops
    out = {}
    x1, cb1 = _fmaps(8, 123, dev), _codebook(1024, (4, 4), dev)
    tr1 = somcb.SomTrainer(cb1, lr=1e-4, neighbourhood_step=10 ** 9, use_cuda_graph="alias")
    out["C1_step_cuda_graph_us"] = 1e3 * _timed(lambda: tr1.step(x1), 100, warm=5)
    x3, cb3 = _fmaps(4096, 123, dev), _codebook(512, (32, 32), dev)
    w3 = cb3.codebook.weight.data
    g3 = ops.geometry(x3.shape, (32, 32))
    cn3 = ops.prepare_codebook(w3)
    out["C3_bmu_ms"] = _timed(lambda: ops.bmu(x3, g3, w3, cn3), 20)
    tr3 = somcb.SomTrainer(cb3, lr=1e-4, neighbourhood_step=10 ** 9, use_cuda_graph="alias")
    out["C3_step_ms"] = _timed(lambda: tr3.step(x3), 20)
    out["shapes"] = "C1: 512 patches D=64 K=1024 (BASELINE configs[0]); C3: 4096 patches D=4096 K=512 (configs[2])"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=96)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0: min(steps, 20)")
    ap.add_argument("--wt", default="full", choices=["slice", "full"],
                    help="peer tail: W~ = T @ W per slice + multicast, or the whole filter on every rank")
    ap.add_argument("--tail", default="auto", choices=["auto", "peer", "nccl"],
                    help="data-parallel tail: sharded over NVSwitch multicast peer memory, or NCCL all-reduce + replicated")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed (the codebook it updated and "
                         "its loss) as DIR/<name>.npy; the inputs are seeded, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of our arm's step; --impl reference has none to write")
        run_reference(args)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: somcb has no CPU fallback")
    # stdout carries ONE JSON line: NCCL writes its version banner to file descriptor 1 whatever NCCL_DEBUG says, so
    # everything else that lands on fd 1 during the run is sent to stderr and the line goes to the saved descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import somcb  # noqa: F401
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = _peaks()

    head, tr, cb, xs = run_headline(args, dev, world, rank, peaks)
    _log("headline + breakdown done")
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in head["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        _log(f"outputs of the last timed step written to {args.dump_outputs}")

    extra = {}
    if not args.no_extra:
        if world > 1:
            try:
                extra["checks"] = run_checks(tr, cb, dev, world, rank)
            except Exception as e:  # noqa: BLE001
                extra["checks"] = {"error": repr(e), "all_ok": False}
            _log(f"checks done: {extra['checks'].get('all_ok')}")
    # captured CUDA graphs hold NCCL kernels: release them before anything tears the communicator down
    tr._graphs.clear()
    del tr, cb, xs
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    if not args.no_extra:
        try:
            extra["C5_sharded_search"] = extra_c5(dev, world, rank)
        except Exception as e:  # noqa: BLE001
            extra["C5_sharded_search"] = {"error": repr(e)}
        _log("C5 done")
        torch.cuda.empty_cache()
        if world == 1:
            for name, fn in (("C2_bmu", lambda: extra_c2(dev, peaks)), ("small_configs", lambda: extra_small_configs(dev))):
                try:
                    extra[name] = fn()
                except Exception as e:  # noqa: BLE001
                    extra[name] = {"error": repr(e)}
                torch.cuda.empty_cache()

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base, _ = _cpu_reference_step(steps=3, warmup=1, min_seconds=10.0)

    if rank == 0:
        line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None,
                "dtype": "f32 (BMU: fp16 hi/lo split x3 products on tcgen05, fp32 accumulate; update, filters and Adam "
                         "fp32; filters 3xTF32)",
                "data": "synthetic", "config": CONFIG, "details": head["details"], "loss": head["loss"],
                "clocks": head["clocks"], "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
                "roofline": head["roofline"], "breakdown": head["breakdown"], "cpu_baseline": cpu_base,
                "extra": extra or None}
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        # no destroy_process_group(): NCCL's communicator teardown can block behind CUDA-graph-captured collectives
        # (seen on this stack: the process printed its result and then never exited).  The result is out; leave.
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
