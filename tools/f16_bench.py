"""fp32 against 16-bit (fp16 or bf16) feature maps, alternating inside one process, timed with CUDA events after
warm-up:

  * C4 BMU alone (1 048 576 patches, D = 64, K = 16 384), with the FP16-split kernel's issuer wait counters
  * the C4 training step, graph-replayed (SomTrainer, or DataParallelSom on this rank's share under torchrun)
  * C4 end to end from pinned host batches through HostTrainer, and the host-to-device copy floor of each dtype
  * C2 end to end from a pinned host array through HostTokenizer (D = 16, K = 4096), with its copy floor
  * C5 shard BMU (D = 256, 32 768 units, 262 144 patches)

Every arm rotates through device inputs of more than 126 MB (the L2) per dtype.  At each size the 16-bit outputs are
checked against the fp32 outputs on the upcast inputs: indices, and weights / losses after the timed steps.  For the
C4 and C5 batches it also reports the share of FP16-split (tile, 64-feature block) pairs that keep the A_lo x B_hi
product group, from a host emulation of the kernel's row scale and lo flag (tests/test_f16_input_host.py).
usage: python tools/f16_bench.py OUT.json [--rounds R] [--half {float16,bfloat16}]      (N GPUs: python -m
       torch.distributed.run --nproc-per-node=N tools/f16_bench.py OUT.json ...; rank 0 writes)"""
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "quantized-autoregression-image-generator_b200"), os.path.join(ROOT, "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import somcb  # noqa: E402
from somcb import ops  # noqa: E402
from somcb.host_pipeline import HostTokenizer, HostTrainer  # noqa: E402
import bench  # noqa: E402
from oracle import patchify  # noqa: E402
from test_f16_input_host import _codebook_scales, _row_scale  # noqa: E402

OUT = sys.argv[1]
ROUNDS = int(sys.argv[sys.argv.index("--rounds") + 1]) if "--rounds" in sys.argv else 5
HALF_NAME = sys.argv[sys.argv.index("--half") + 1] if "--half" in sys.argv else "float16"
HALF = {"float16": torch.float16, "bfloat16": torch.bfloat16}[HALF_NAME]
H = {"float16": "f16", "bfloat16": "bf16"}[HALF_NAME]           # the 16-bit arm's key in the results
WORLD = int(os.environ.get("WORLD_SIZE", "1"))
RANK = int(os.environ.get("RANK", "0"))
dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
torch.cuda.set_device(dev)
if WORLD > 1:
    dist.init_process_group("nccl", device_id=dev)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(dev.index)],
                       capture_output=True, text=True)
    return dict(zip(q.split(","), (v.strip() for v in r.stdout.strip().split(",")))) if r.returncode == 0 else {}


def timed(fn, reps):
    """ms per call of ``fn`` over ``reps`` calls, device events"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def ab(arms, reps, warm=2):
    """{name: sorted ms per call}: the arms alternate A B B A per round after ``warm`` untimed calls each"""
    for fn in arms.values():
        for i in range(warm):
            fn(i)
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    names = list(arms)
    for r in range(ROUNDS):
        for k in (names if r % 2 == 0 else names[::-1]):
            res[k].append(timed(arms[k], reps))
    return {k: sorted(v) for k, v in res.items()}


def summary(v):
    return {"median_ms": v[len(v) // 2], "min_ms": v[0], "max_ms": v[-1], "rounds": len(v)}


def device_batches(n_f, n_buf, seed, patch=(4, 4)):
    x32 = [bench._fmaps(n_f, seed + b, dev).to(HALF).float() for b in range(n_buf)]   # values the 16-bit type holds
    return x32, [x.to(HALF) for x in x32]


def kept_third_product(x32, patch, w):
    """Share of (128-patch tile, 64-feature block) pairs whose lo flag is set, so that the FP16-split kernel keeps
    their A_lo x B_hi products: host emulation of the row scale on the batch's patch rows."""
    v = patchify(x32, patch).reshape(-1, patch[0] * patch[1] * x32.shape[1]).cpu().numpy()
    _, tc_exp = _codebook_scales(w.cpu().numpy())
    with np.errstate(invalid="ignore", over="ignore"):
        s = v * _row_scale(v, tc_exp)[:, None]
        lo = s - s.astype(np.float16).astype(np.float32)
    bad = (lo != 0) | np.isnan(lo)
    n, d = bad.shape
    rows = -(-n // 128) * 128
    bad = np.concatenate([bad, np.zeros((rows - n, d), bool)]) if rows > n else bad
    dp = -(-d // 64) * 64
    bad = np.concatenate([bad, np.zeros((rows, dp - d), bool)], 1) if dp > d else bad
    flags = bad.reshape(rows // 128, 128, dp // 64, 64).any(axis=(1, 3))
    return {"tile_blocks": int(flags.size), "kept": int(flags.sum()), "share": float(flags.mean())}


def l16_cycles():
    buf = (ctypes.c_longlong * 5)()
    somcb._lib.load().som_debug_tc_l16_cycles(buf)
    return {"cycles": buf[0], "tiles": buf[1], "wait_acc": buf[2], "wait_b": buf[3], "wait_a": buf[4]}


result = {"device": gpu_info(), "world": WORLD, "rounds": ROUNDS, "half": HALF_NAME, "checks": {}}
C4 = bench.C4
seq4 = C4["seq"]

# ---- C4 BMU alone ------------------------------------------------------------------------------------------------
n_f = C4["n_fmaps"] // WORLD
x32, x16 = device_batches(n_f, 2, 9000)                  # 2 x 268 MB fp32, 2 x 134 MB fp16 / bf16
cb = bench._codebook(C4["K"], C4["patch"], dev)
w = cb.codebook.weight.detach()
cn = ops.prepare_codebook(w)
geom = ops.geometry(x32[0].shape, C4["patch"])
out = {k: torch.empty(n_f * seq4, dtype=torch.int64, device=dev) for k in ("f32", H)}
arms = {"f32": lambda i: ops.bmu(x32[i % 2], geom, w, cn, out=out["f32"]),
        H: lambda i: ops.bmu(x16[i % 2], geom, w, cn, out=out[H])}
t = ab(arms, 20)
cyc = {}
for k in ("f32", H):
    arms[k](0)
    torch.cuda.synchronize()
    cyc[k] = l16_cycles()
ok = all(torch.equal(ops.bmu(x16[b], geom, w, cn), ops.bmu(x32[b], geom, w, cn)) for b in range(2))
result["c4_bmu"] = {"patches": n_f * seq4, "native_f16": ops.bmu_f16_native(geom, C4["K"]),
                    "kept_third_product": kept_third_product(x32[0], C4["patch"], w),
                    "f32": summary(t["f32"]), H: summary(t[H]), "issuer_cta0": cyc,
                    "speedup": t["f32"][len(t["f32"]) // 2] / t[H][len(t[H]) // 2]}
result["checks"]["c4_bmu_idx_equal"] = ok

# ---- C4 graph step ------------------------------------------------------------------------------------------------
trainers = {}
for k in ("f32", H):
    c = bench._codebook(C4["K"], C4["patch"], dev)
    if WORLD > 1:
        trainers[k] = somcb.DataParallelSom(c, lr=C4["lr"], neighbourhood_step=10 ** 9, use_cuda_graph="alias")
    else:
        trainers[k] = somcb.SomTrainer(c, lr=C4["lr"], neighbourhood_step=10 ** 9, use_cuda_graph="alias")
xs = {"f32": x32, H: x16}
loss = {}


def step_arm(k):
    def f(i):
        loss[k] = trainers[k].step(xs[k][i % 2])
    return f


t = ab({k: step_arm(k) for k in ("f32", H)}, 10)
same_w = torch.equal(trainers["f32"].cb.codebook.weight.data, trainers[H].cb.codebook.weight.data)
result["c4_graph_step"] = {"patches_per_rank": n_f * seq4, "f32": summary(t["f32"]), H: summary(t[H]),
                           "speedup": t["f32"][len(t["f32"]) // 2] / t[H][len(t[H]) // 2]}
result["checks"]["c4_step_weights_equal"] = same_w
result["checks"]["c4_step_loss_equal"] = float(loss["f32"]) == float(loss[H])
del trainers

# ---- C4 end to end from pinned host batches ---------------------------------------------------------------------
host = {"f32": [x.cpu().pin_memory() for x in x32], H: [x.cpu().pin_memory() for x in x16]}
del x32, x16, xs
torch.cuda.empty_cache()
hts = {}
for k in ("f32", H):
    c = bench._codebook(C4["K"], C4["patch"], dev)
    tr = (somcb.DataParallelSom if WORLD > 1 else somcb.SomTrainer)(c, lr=C4["lr"], neighbourhood_step=10 ** 9,
                                                                   use_cuda_graph="alias")
    hts[k] = HostTrainer(tr)
pend = {}


def host_arm(k):
    def f(i):
        pend[k] = hts[k].step(host[k][i % 2])
    return f


t = ab({k: host_arm(k) for k in ("f32", H)}, 10)
same_w = torch.equal(hts["f32"].tr.cb.codebook.weight.data, hts[H].tr.cb.codebook.weight.data)
result["checks"]["c4_host_weights_equal"] = same_w
result["checks"]["c4_host_loss_equal"] = pend["f32"].item() == pend[H].item()
dst = {k: torch.empty(host[k][0].shape, dtype=host[k][0].dtype, device=dev) for k in ("f32", H)}
floor = ab({k: (lambda k: lambda i: dst[k].copy_(host[k][i % 2], non_blocking=True))(k) for k in ("f32", H)}, 10)
result["c4_host_e2e"] = {k: {"step": summary(t[k]), "h2d_copy_floor": summary(floor[k]),
                             "bytes_per_step": host[k][0].numel() * host[k][0].element_size()} for k in t}
result["c4_host_e2e"]["speedup"] = t["f32"][len(t["f32"]) // 2] / t[H][len(t[H]) // 2]
del hts, host, dst
torch.cuda.empty_cache()

# ---- C2 end to end through HostTokenizer (one GPU's work; rank 0 only) ---------------------------------------------
if RANK == 0:
    C2 = bench.C2
    h32 = bench._fmaps(C2["n_fmaps"], 4242, dev).to(HALF).float().cpu().pin_memory()
    h16 = h32.to(HALF).pin_memory()
    c2cb = bench._codebook(C2["K"], C2["patch"], dev)
    tok = {k: HostTokenizer(c2cb) for k in ("f32", H)}
    hin = {"f32": h32, H: h16}
    seq2 = (32 // C2["patch"][0]) * (32 // C2["patch"][1])
    outs = {k: torch.empty(C2["n_fmaps"], seq2, dtype=torch.int64, pin_memory=True) for k in ("f32", H)}
    t = ab({k: (lambda k: lambda i: tok[k].tokenize(hin[k], out_host=outs[k]))(k) for k in ("f32", H)}, 2, warm=1)
    result["checks"]["c2_tokens_equal"] = torch.equal(outs["f32"], outs[H])
    d_in = {k: torch.empty(hin[k].shape, dtype=hin[k].dtype, device=dev) for k in hin}
    d_out = torch.empty(outs["f32"].shape, dtype=torch.int64, device=dev)

    def copies(k):
        def f(i):
            d_in[k].copy_(hin[k], non_blocking=True)
            outs[k].copy_(d_out, non_blocking=True)
        return f
    floor = ab({k: copies(k) for k in ("f32", H)}, 2, warm=1)
    n_p = C2["n_fmaps"] * seq2
    result["c2_host_e2e"] = {k: {"tokenize": summary(t[k]), "copy_floor_h2d_plus_d2h": summary(floor[k]),
                                 "patches_per_s": n_p / (t[k][len(t[k]) // 2] * 1e-3)} for k in t}
    result["c2_host_e2e"]["speedup"] = t["f32"][len(t["f32"]) // 2] / t[H][len(t[H]) // 2]
    del h32, h16, d_in, d_out, tok
    torch.cuda.empty_cache()

    # ---- C5 shard BMU ----------------------------------------------------------------------------------------------
    k5, p5 = 32768, (8, 8)
    x32, x16 = device_batches(16384, 2, 777)
    w5 = bench._codebook(k5, p5, dev).codebook.weight.detach()
    cn5 = ops.prepare_codebook(w5)
    g5 = ops.geometry(x32[0].shape, p5)
    o5 = {k: torch.empty(ops.n_patches_of(g5), dtype=torch.int64, device=dev) for k in ("f32", H)}
    t = ab({"f32": lambda i: ops.bmu(x32[i % 2], g5, w5, cn5, out=o5["f32"]),
            H: lambda i: ops.bmu(x16[i % 2], g5, w5, cn5, out=o5[H])}, 10)
    result["checks"]["c5_idx_equal"] = all(torch.equal(ops.bmu(x16[b], g5, w5, cn5), ops.bmu(x32[b], g5, w5, cn5))
                                           for b in range(2))
    result["c5_shard_bmu"] = {"patches": ops.n_patches_of(g5), "K": k5, "D": 256,
                              "native_f16": ops.bmu_f16_native(g5, k5), "f32": summary(t["f32"]),
                              "kept_third_product": kept_third_product(x32[0], p5, w5),
                              H: summary(t[H]),
                              "speedup": t["f32"][len(t["f32"]) // 2] / t[H][len(t[H]) // 2]}

    result["device_after"] = gpu_info()
    with open(OUT, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k in ("checks", "device")}))
    print(json.dumps({k: result[k].get("speedup") for k in result if isinstance(result[k], dict)
                      and "speedup" in result[k]}))
if WORLD > 1:
    dist.destroy_process_group()
if not all(result["checks"].values()):
    sys.exit(f"{HALF_NAME} outputs differ from the fp32 outputs on the upcast inputs")
