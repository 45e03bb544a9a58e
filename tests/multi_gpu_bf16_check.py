"""N-GPU check of bf16 feature maps (launch with torch.distributed.run):
  * DataParallelSom (NCCL tail and the default tail, the peer tail where multicast memory is available) on bf16
    shares == the same trainer on the fp32 shares of the upcast data, bit for bit, with bit-identical replicas
  * unit-sharded search (sharded_bmu) on a bf16 batch == the same search on the fp32 upcast
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "quantized-autoregression-image-generator_b200"), os.path.join(ROOT, "tests")]
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import somcb  # noqa: E402
from somcb import ops  # noqa: E402
from somcb.distributed import shard_bounds, sharded_bmu  # noqa: E402
from oracle.step_oracle import synthetic_fmaps, trained_like_codebook  # noqa: E402


def make_cb(w, pd, dev):
    cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4, num_embeddings=w.shape[0],
                        init_neighbour_range=w.shape[0] // 2)
    with torch.no_grad():
        cb.codebook.weight.copy_(w)
    return cb.to(dev)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ok = True

    # ---- data parallel: 1024 fmaps per rank -> 65 536 patches, the native FP16-split search with staging ------------
    pd, k = (4, 4), 16384
    w0 = trained_like_codebook(k, pd, 7)
    for tail in ("nccl", "auto"):
        runs = []
        for half in (True, False):
            cb = make_cb(w0, pd, dev)
            tr = somcb.DataParallelSom(cb, lr=1e-4, neighbourhood_step=3, tail=tail)
            losses = []
            for step in range(4):
                x = synthetic_fmaps(1024 * world, 600 + step).bfloat16().to(dev)
                share = somcb.split_batch(x, world, rank).contiguous()
                losses.append(float(tr.step(share if half else share.float())))
            torch.cuda.synchronize()
            runs.append((cb.codebook.weight.data.clone(), losses, tr.tail))
        (w16, l16, used), (w32, l32, _) = runs
        same = torch.equal(w16.view(torch.int32), w32.view(torch.int32)) and l16 == l32
        gathered = [torch.empty_like(w16) for _ in range(world)]
        dist.all_gather(gathered, w16)
        replicas = all(torch.equal(g.view(torch.int32), w16.view(torch.int32)) for g in gathered)
        if rank == 0:
            print(f"[dp {tail} -> {used}] bf16 == fp32 on upcast: {same}; replicas identical: {replicas}")
        ok &= same and replicas

    # ---- unit-sharded search on a bf16 batch ----------------------------------------------------------------------
    k = 32768
    w = trained_like_codebook(k, pd, 9).to(dev)
    xb = synthetic_fmaps(1024, 77).bfloat16().to(dev)
    geom = ops.geometry(xb.shape, pd)
    lo, hi = shard_bounds(k, world, rank)
    got = sharded_bmu(xb, geom, w[lo:hi].contiguous(), lo)
    want = sharded_bmu(xb.float(), geom, w[lo:hi].contiguous(), lo)
    same = torch.equal(got, want)
    if rank == 0:
        print(f"[sharded] fp16 == fp32 on upcast: {same}")
    ok &= same

    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTI_GPU_BF16_CHECK", "PASS" if int(flag) else "FAIL", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
