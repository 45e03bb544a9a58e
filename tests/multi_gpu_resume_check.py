"""N-GPU check of save and resume of DataParallelSom (launch with torch.distributed.run):
  * on the NCCL tail and on the peer tail, eagerly and replayed from CUDA graphs: a run split by
    checkpoint_dict(C, with_state=True) -> torch.save -> torch.load -> resume into a new codebook and trainer is
    bit-identical to the run that was not interrupted (weights, full moments, device step count, losses, lr,
    global_steps, range), and the replicas are bit-identical after the resume;
  * the saved moments are complete: equal to every rank's own rows [lo, hi) put together, where the rows a rank does
    not own are stale in its own m and v (the peer tail's Adam updates only its slice);
  * a state saved at N ranks resumes on one GPU and a state saved on one GPU resumes at N ranks, equal to the straight
    one-GPU run to 1e-6 (the tolerance between the data-parallel and the one-GPU step of multi_gpu_check.py).
"""
import io
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "quantized-autoregression-image-generator_b200"), os.path.join(ROOT, "tests")]
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import somcb  # noqa: E402
from oracle.step_oracle import synthetic_fmaps, trained_like_codebook  # noqa: E402

PD, K, C, RANGE, N = (4, 4), 4096, 4, 64, 3        # range 64: band half-width ~50 rows, so the peer tail slices
SCHED = dict(lr=1e-3, neighbourhood_step=2, lr_step=3)    # range and lr change on both sides of the split


def make_cb(dev, w0=None):
    cb = somcb.Codebook(patch_dim=PD, image_dim=(32, 32), image_channel=C, num_embeddings=K, init_neighbour_range=RANGE)
    with torch.no_grad():
        cb.codebook.weight.copy_(trained_like_codebook(K, PD, 7) if w0 is None else w0)
    return cb.to(dev)


def run(tr, batches, part):
    """Losses of the steps on ``batches``; ``part(x)`` is the share of the global batch x this trainer takes."""
    return torch.cat([tr.step(part(x)).clone().reshape(1) for x in batches])


def save_load(tr):
    buf = io.BytesIO()
    torch.save(tr.checkpoint_dict(C, with_state=True), buf)      # collective on the peer tail
    buf.seek(0)
    return torch.load(buf)


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    ok = True

    def report(what, good):
        nonlocal ok
        ok &= bool(good)
        if rank == 0:
            print(f"[resume] {what}: {'ok' if good else 'FAILED'}", flush=True)

    def share(x):
        return somcb.split_batch(x, world, rank).contiguous()

    def whole(x):
        return x

    batches = [synthetic_fmaps(64 * world, 500 + s).to(dev) for s in range(2 * N)]
    single = somcb.SomTrainer(make_cb(dev), **SCHED)
    want_single = run(single, batches, whole)

    # tail="auto" takes the peer tail wherever NVSwitch multicast symmetric memory is available to the group
    tails = ["nccl"] + (["peer"] if somcb.DataParallelSom(make_cb(dev), **SCHED).tail == "peer" else [])
    if rank == 0 and "peer" not in tails:
        print("[resume] NVSwitch multicast symmetric memory not available: peer tail not checked", flush=True)
    graphs = []
    saved_at_n = None
    for tail in tails:
        for graph in (False, True):
            name = f"tail={tail} use_cuda_graph={graph}"
            straight = somcb.DataParallelSom(make_cb(dev), tail=tail, use_cuda_graph=graph, **SCHED)
            first = somcb.DataParallelSom(make_cb(dev), tail=tail, use_cuda_graph=graph, **SCHED)
            graphs += [straight, first]
            assert straight.tail == tail and first.tail == tail
            want = run(straight, batches, share)
            run(first, batches[:N], share)
            ck = save_load(first)
            st = ck["trainer"]
            # the saved moments are every rank's own rows put together (broadcast from their owners here)
            parts_m, parts_v = [], []
            for r in range(world):
                lo, hi = somcb.shard_bounds(K, world, r)
                pm = first.m[lo:hi].clone() if r == rank else torch.empty(hi - lo, first.m.shape[1], device=dev)
                pv = first.v[lo:hi].clone() if r == rank else torch.empty(hi - lo, first.v.shape[1], device=dev)
                dist.broadcast(pm, src=r)
                dist.broadcast(pv, src=r)
                parts_m.append(pm)
                parts_v.append(pv)
            full = torch.equal(st["m"], torch.cat(parts_m).cpu()) and torch.equal(st["v"], torch.cat(parts_v).cpu())
            report(f"{name}: saved moments == the owners' rows put together", full)
            if tail == "peer":
                stale = torch.tensor([0 if torch.equal(first.m.cpu(), st["m"]) else 1], device=dev)
                dist.all_reduce(stale)
                report(f"{name}: the ranks' own m hold stale rows outside their slice ({int(stale)} of {world})",
                       int(stale) > 0)
            second = somcb.DataParallelSom(make_cb(dev, torch.zeros(K, C * PD[0] * PD[1])), lr=0.5, neighbourhood_step=1,
                                           tail=tail, use_cuda_graph=graph)
            graphs.append(second)
            second.resume(ck)
            got = run(second, batches[N:], share)
            s_got, s_want = second.state_dict(), straight.state_dict()
            same = torch.equal(got, want[N:]) and \
                torch.equal(second.cb.codebook.weight.data, straight.cb.codebook.weight.data) and \
                all(torch.equal(s_got[key], s_want[key]) if torch.is_tensor(s_want[key]) else
                    s_got[key] == s_want[key] for key in s_want)
            report(f"{name}: split run == straight run, bit for bit", same)
            w_all = [torch.empty_like(second.cb.codebook.weight.data) for _ in range(world)]
            dist.all_gather(w_all, second.cb.codebook.weight.data)
            report(f"{name}: replicas identical after the resume", all(torch.equal(w_all[0], w) for w in w_all))
            if saved_at_n is None or tail == "peer":
                saved_at_n = ck

    # saved at N, resumed on one GPU (every rank does it on its own device)
    one = somcb.SomTrainer(make_cb(dev, torch.zeros(K, C * PD[0] * PD[1])), lr=0.5, neighbourhood_step=1)
    one.resume(saved_at_n)
    got = run(one, batches[N:], whole)
    r_w, r_l = rel(one.cb.codebook.weight.data, single.cb.codebook.weight.data), rel(got, want_single[N:])
    report(f"saved at {world} GPUs, resumed on one: weights rel {r_w:.2e}, losses rel {r_l:.2e} vs the one-GPU run",
           r_w <= 1e-6 and r_l <= 1e-6 and one.cb.neighbourhood_range == single.cb.neighbourhood_range
           and one.lr == single.lr and one.global_steps == single.global_steps)

    # saved on one GPU, resumed at N ranks
    half = somcb.SomTrainer(make_cb(dev), **SCHED)
    run(half, batches[:N], whole)
    ck1 = save_load(half)
    dp = somcb.DataParallelSom(make_cb(dev, torch.zeros(K, C * PD[0] * PD[1])), lr=0.5, neighbourhood_step=1,
                               tail=tails[-1])
    dp.resume(ck1)
    got = run(dp, batches[N:], share)
    r_w, r_l = rel(dp.cb.codebook.weight.data, single.cb.codebook.weight.data), rel(got, want_single[N:])
    w_all = [torch.empty_like(dp.cb.codebook.weight.data) for _ in range(world)]
    dist.all_gather(w_all, dp.cb.codebook.weight.data)
    report(f"saved on one GPU, resumed at {world} ({dp.tail} tail): weights rel {r_w:.2e}, losses rel {r_l:.2e}",
           r_w <= 1e-6 and r_l <= 1e-6 and all(torch.equal(w_all[0], w) for w in w_all)
           and dp.cb.neighbourhood_range == single.cb.neighbourhood_range and dp.lr == single.lr)

    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTI_GPU_RESUME_CHECK", "PASS" if int(flag) else "FAIL", flush=True)
    # captured CUDA graphs hold NCCL kernels and destroy_process_group() can block behind them: release the graphs
    # and leave without tearing the communicator down
    for tr in graphs:
        tr._graphs.clear()
    torch.cuda.synchronize()
    dist.barrier()
    sys.stdout.flush()
    os._exit(0 if int(flag) else 1)


if __name__ == "__main__":
    main()
