"""16-bit codebooks against fp32 codebooks holding the same values, in one process, arms alternating on the same
batches.  Search arms use bf16 feature maps (the case where both operands are 16-bit: 17 instead of 33 MMAs per tile at
D = 256 when every B flag is clear); decode gathers the codebook in its own dtype.  Every batch is larger than the
126 MB L2.  Outputs are compared at every timed size; the JSON records the device, its power limit and SM clock, CUDA
event times, the FP16-split issuer's cycles per tile (som_debug_tc_l16_cycles, CTA 0) and the host-emulated share of
(tile, block) pairs that keep B_lo.

    python tools/w16_bench.py [--rounds 3] [--iters 5] [--out profiles/w16_bench.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "quantized-autoregression-image-generator_b200"), os.path.join(ROOT, "tests"), ROOT]
import somcb  # noqa: E402
from somcb import ops  # noqa: E402
from test_w16_codebook_host import kept_share  # noqa: E402

DEV = "cuda:0"


def device_record():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def issuer_cycles():
    fn = somcb._lib.load().som_debug_tc_l16_cycles
    out = (ctypes.c_longlong * 5)()
    fn(out)
    return {"cycles": out[0], "tiles": out[1], "cycles_per_tile": out[0] / max(1, out[1]),
            "wait_acc": out[2], "wait_b": out[3], "wait_a": out[4]}


def timed(fn, iters):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def tanh_codebook(k, d, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.tanh(torch.randn(k, d, generator=g, device=DEV)).to(torch.bfloat16)


def bmu_case(name, n_img, c, p, k, rounds, iters):
    g = torch.Generator(device=DEV).manual_seed(n_img + k)
    x = torch.tanh(torch.randn(n_img, c, 32, 32, generator=g, device=DEV)).to(torch.bfloat16)
    geom = ops.geometry(x.shape, (p, p))
    w16 = tanh_codebook(k, c * p * p, k)
    w32 = w16.float()
    arms = {"fp32": w32, "bf16": w16}
    res = {"name": name, "n_patches": ops.n_patches_of(geom), "D": c * p * p, "K": k, "x": "bf16",
           "x_bytes": x.numel() * 2, "kept_B_lo_share": kept_share(w16.float().cpu().numpy()),
           "ms": {a: [] for a in arms}, "issuer": {}}
    outs = {}
    for a, w in arms.items():
        outs[a] = ops.bmu(x, geom, w, want_rd=True)
        torch.cuda.synchronize()
        res["issuer"][a] = issuer_cycles()
    res["equal"] = bool(torch.equal(outs["fp32"][0], outs["bf16"][0]) and torch.equal(outs["fp32"][1], outs["bf16"][1]))
    for _ in range(rounds):
        for a, w in arms.items():
            cn = ops.prepare_codebook(w)
            res["ms"][a].append(timed(lambda: ops.bmu(x, geom, w, cn), iters))
    return res


def tokenizer_case(rounds, iters):
    k, pd = 16384, (4, 4)
    host = torch.tanh(torch.randn(65536, 4, 32, 32)).to(torch.bfloat16).pin_memory()     # 512 MB of bf16
    res = {"name": "C2_host_tokenizer", "fmaps": host.shape[0], "K": k, "D": 64, "x": "bf16", "ms": {}}
    outs = {}
    for a, wd in (("fp32", torch.float32), ("bf16", torch.bfloat16)):
        cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4, num_embeddings=k,
                            init_neighbour_range=k // 2).to(DEV)
        with torch.no_grad():
            cb.codebook.weight.copy_(tanh_codebook(k, 64, 1).float())
        cb = cb.to(wd)
        tok = HostTok(cb)
        outs[a] = tok.run(host).clone()
        res["ms"][a] = []
        arms = res.setdefault("_toks", {})
        arms[a] = tok
    res["equal"] = bool(torch.equal(outs["fp32"], outs["bf16"]))
    for _ in range(rounds):
        for a in ("fp32", "bf16"):
            res["ms"][a].append(timed(lambda: res["_toks"][a].run(host), max(1, iters // 5)))
    del res["_toks"]
    return res


class HostTok:
    def __init__(self, cb):
        self.tok = somcb.HostTokenizer(cb, chunk_fmaps=4096)
        self.out = None

    def run(self, host):
        self.out = self.tok.tokenize(host, out_host=self.out)
        return self.out


def decode_case(rounds, iters):
    k, n = 16384, 16384                        # C4 shape (D = 64, 4 x 32 x 32 maps) x 4: fp32 output 268 MB
    w16 = tanh_codebook(k, 64, 2)
    idx = torch.randint(0, k, (n * 64,), device=DEV)
    geom = ops.geometry((n, 4, 32, 32), (4, 4))
    arms = {"fp32": w16.float(), "bf16": w16}
    res = {"name": "C4_decode", "images": n, "K": k, "out_bytes": {a: n * 4096 * w.element_size() for a, w in arms.items()},
           "ms": {a: [] for a in arms}}
    outs = {a: ops.quantize(idx, w, geom) for a, w in arms.items()}
    res["equal"] = bool(torch.equal(outs["fp32"], outs["bf16"].float()))
    for _ in range(rounds):
        for a, w in arms.items():
            o = outs[a]
            res["ms"][a].append(timed(lambda: ops.quantize(idx, w, geom, out=o), iters * 4))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "w16_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("w16_bench needs a CUDA device")
    rec = {"device": device_record(), "rounds": a.rounds, "iters": a.iters, "cases": []}
    rec["cases"].append(bmu_case("C5_shard_bmu", 16384, 16, 4, 32768, a.rounds, a.iters))    # 2^20 patches, D = 256
    rec["cases"].append(bmu_case("D128_bmu", 16384, 8, 4, 16384, a.rounds, a.iters))         # 2^20 patches, D = 128
    rec["cases"].append(bmu_case("C4_bmu", 16384, 4, 4, 16384, a.rounds, a.iters))           # 2^20 patches, D = 64
    rec["cases"].append(tokenizer_case(a.rounds, a.iters))
    rec["cases"].append(decode_case(a.rounds, a.iters))
    for c in rec["cases"]:
        c["median_ms"] = {k: sorted(v)[len(v) // 2] for k, v in c["ms"].items()}
        c["speedup"] = c["median_ms"]["fp32"] / c["median_ms"]["bf16"]
        print(json.dumps({k: c[k] for k in ("name", "median_ms", "speedup", "equal")}))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    assert all(c["equal"] for c in rec["cases"]), "16-bit and fp32 codebook outputs differ"


if __name__ == "__main__":
    main()
