"""Save and resume of the fused trainers on the GPU.  In every regime the step can take (the one-kernel small step, the
separate kernels eagerly, replayed from a CUDA graph captured on a static or on the caller's buffer, fp16 and bf16 feature
maps, the W~ filter beside the search or in front of it) a run split by checkpoint_dict(C, with_state=True) ->
torch.save -> torch.load -> resume into a new Codebook and trainer is bit-identical to the run that was not interrupted:
weights, Adam's moments, the device step count, every loss after the split, lr, global_steps and neighbourhood range.
Loading into a trainer that has already captured graphs copies in place: the next replay runs on the loaded state.
A state taken while HostTrainer steps are still in flight equals the state after a device synchronise."""
import io
import os
import subprocess
import sys

import pytest
import torch

import somcb
from somcb import ops
from oracle.step_oracle import synthetic_fmaps, trained_like_codebook

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PD, C = (4, 4), 4
LR = 1e-3


def _cb(k, w0=None):
    cb = somcb.Codebook(patch_dim=PD, image_dim=(32, 32), image_channel=C, num_embeddings=k,
                        init_neighbour_range=k // 2)
    with torch.no_grad():
        cb.codebook.weight.copy_(trained_like_codebook(k, PD, 7) if w0 is None else w0)
    return cb.to(DEV)


def _batches(n_f, dtype, steps, seed=500):
    return [synthetic_fmaps(n_f, seed + s).to(DEV, dtype) for s in range(steps)]


def _run(tr, batches, staging=None):
    """Losses of the steps on ``batches`` (through ``staging`` when given: the buffer an "alias" trainer replays on)."""
    out = []
    for x in batches:
        if staging is not None:
            staging.copy_(x)
            x = staging
        out.append(tr.step(x).clone())
    return torch.stack(out)


def _resume_from(tr, **kw):
    """A new Codebook (other weights) and trainer (other lr and schedule), resumed from ``tr``'s saved checkpoint."""
    buf = io.BytesIO()
    torch.save(tr.checkpoint_dict(C, with_state=True), buf)
    buf.seek(0)
    k = tr.cb.num_embeddings
    new = somcb.SomTrainer(_cb(k, torch.zeros(k, C * PD[0] * PD[1])), lr=0.5, neighbourhood_step=1, **kw)
    new.resume(torch.load(buf))
    return new


def _assert_same_state(a, b):
    for name in ("m", "v", "t_dev"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert torch.equal(a.cb.codebook.weight.data, b.cb.codebook.weight.data), "W"
    assert (a.t, a.lr, a.global_steps, a.cb.neighbourhood_range) == (b.t, b.lr, b.global_steps, b.cb.neighbourhood_range)
    assert type(a.cb.neighbourhood_range) is type(b.cb.neighbourhood_range)


# (id, K, feature maps per step, batch dtype, trainer options, one-kernel small step expected)
REGIMES = [
    ("small_step", 1024, 8, torch.float32, {}, True),                  # config 1: 512 patches, one cooperative kernel
    ("small_step_graph", 1024, 8, torch.float32, {"use_cuda_graph": True}, True),
    ("small_step_f16", 1024, 8, torch.float16, {}, True),
    ("separate_eager", 2048, 64, torch.float32, {}, False),            # 4096 patches: the separate kernels
    ("separate_graph", 2048, 64, torch.float32, {"use_cuda_graph": True}, False),
    ("separate_alias", 2048, 64, torch.float32, {"use_cuda_graph": "alias"}, False),
    ("separate_f16", 2048, 64, torch.float16, {}, False),
    ("separate_bf16_graph", 2048, 64, torch.bfloat16, {"use_cuda_graph": True}, False),
    ("no_overlap_filter", 2048, 64, torch.float32, {"overlap_filter": False}, False),
    ("no_overlap_filter_graph", 2048, 64, torch.float32, {"overlap_filter": False, "use_cuda_graph": True}, False),
]


@pytest.mark.parametrize("k,n_f,dtype,kw,small", [r[1:] for r in REGIMES], ids=[r[0] for r in REGIMES])
def test_split_run_equals_straight_run(k, n_f, dtype, kw, small, monkeypatch):
    """8 steps straight against 4 + save + resume + 4: the range shrinks at steps 3 and 6 and lr halves at step 6
    (new graph keys on both sides of the split)."""
    n = 4
    sched = dict(neighbourhood_step=3, lr_step=5)
    batches = _batches(n_f, dtype, 2 * n)
    geom = ops.geometry(batches[0].shape, PD)
    alias = kw.get("use_cuda_graph") == "alias"
    small_calls = []
    step_small = ops.step_small
    monkeypatch.setattr(ops, "step_small", lambda *a, **k_: small_calls.append(1) or step_small(*a, **k_))

    straight = somcb.SomTrainer(_cb(k), lr=LR, **sched, **kw)
    buffers = {id(straight): torch.empty_like(batches[0]) if alias else None}
    want = []
    for x in batches:
        # the regime this row names, at the range of every step
        assert ops.step_small_supported(geom, k, straight.cb.neighbourhood_range) == small
        want.append(_run(straight, [x], buffers[id(straight)]))
    want = torch.cat(want)
    assert bool(small_calls) == small      # the one-kernel step ran (eagerly or under capture), or it did not

    first = somcb.SomTrainer(_cb(k), lr=LR, **sched, **kw)
    _run(first, batches[:n], torch.empty_like(batches[0]) if alias else None)
    second = _resume_from(first, **kw)
    assert second.t == n and second._graphs == {}
    buffers[id(second)] = torch.empty_like(batches[0]) if alias else None
    got = _run(second, batches[n:], buffers[id(second)])

    assert torch.equal(got, want[n:])
    _assert_same_state(second, straight)
    assert straight.lr == LR / 2 and straight.cb.neighbourhood_range == k // 2 - 2
    for tr in (straight, second):
        if kw.get("use_cuda_graph"):
            assert tr._graphs, "no graph was captured"
        if alias:
            assert all(entry[1] is buffers[id(tr)] for entry in tr._graphs.values())
        assert (tr._side is not None) == (kw.get("overlap_filter", True) and not small)


@pytest.mark.parametrize("graph", [True, "alias"])
@pytest.mark.parametrize("same_key", [True, False], ids=["same_graph", "new_graph"])
def test_load_into_a_trainer_that_holds_graphs(graph, same_key):
    """No new trainer: the state is loaded into one that has captured graphs already.  With the lr and range its graph
    was captured for, the next step replays that graph (none is captured) on the loaded W, m, v and t_dev: rebinding the
    tensors instead of copying into them would leave the graph on the old ones.  With another lr and range, the loaded
    state selects a graph of its own (captured at the next step).  Either way the result is the uninterrupted run."""
    k, n = 2048, 3
    sched = dict(neighbourhood_step=10 ** 6, lr_step=10 ** 6) if same_key else dict(neighbourhood_step=2, lr_step=2)
    batches = _batches(64, torch.float32, 2 * n)
    staging = torch.empty_like(batches[0]) if graph == "alias" else None

    straight = somcb.SomTrainer(_cb(k), lr=LR, use_cuda_graph=graph, **sched)
    want = _run(straight, batches, staging)
    donor = somcb.SomTrainer(_cb(k), lr=LR, use_cuda_graph=graph, **sched)
    _run(donor, batches[:n], staging)

    target = somcb.SomTrainer(_cb(k, trained_like_codebook(k, PD, 99)), lr=LR, neighbourhood_step=10 ** 6,
                              lr_step=10 ** 6, use_cuda_graph=graph)
    _run(target, _batches(64, torch.float32, 3, seed=900), staging)
    graphs = dict(target._graphs)
    assert len(graphs) == 1 and target.t == 3
    buffers = [target.m.data_ptr(), target.v.data_ptr(), target.t_dev.data_ptr(),
               target.cb.codebook.weight.data.data_ptr()]

    buf = io.BytesIO()
    torch.save(donor.checkpoint_dict(C, with_state=True), buf)
    buf.seek(0)
    target.resume(torch.load(buf))
    assert buffers == [target.m.data_ptr(), target.v.data_ptr(), target.t_dev.data_ptr(),
                       target.cb.codebook.weight.data.data_ptr()]
    got = _run(target, batches[n:], staging)

    assert torch.equal(got, want[n:])
    _assert_same_state(target, straight)
    assert all(target._graphs.get(key) is entry for key, entry in graphs.items())     # kept, not re-captured
    if same_key:
        assert list(target._graphs) == list(graphs)
    else:
        assert len(target._graphs) > len(graphs)
        assert (target.lr, target.cb.neighbourhood_range) != (LR, k // 2)


def test_state_saved_behind_pending_host_trainer_steps():
    """state_dict right after HostTrainer.step calls whose losses have not been read, called from another stream: it
    synchronises the device first, so the state equals the one after torch.cuda.synchronize() and the resident run's."""
    k = 16384
    w0 = trained_like_codebook(k, PD, 7)
    hosts = [synthetic_fmaps(2048, 40 + i).pin_memory() for i in range(5)]        # 131 072 patches per step
    tr = somcb.SomTrainer(_cb(k, w0), lr=LR, neighbourhood_step=2, use_cuda_graph="alias")
    ht = somcb.HostTrainer(tr, depth=len(hosts))     # no staging slot (and its pinned loss) is reused
    ht.step(hosts[0]).item()                 # capture-free first (eager) step
    pending = [ht.step(h) for h in hosts[1:]]
    with torch.cuda.stream(torch.cuda.Stream(DEV)):
        early = tr.state_dict()
    torch.cuda.synchronize()
    late = tr.state_dict()
    for key, val in late.items():
        assert torch.equal(early[key], val) if torch.is_tensor(val) else early[key] == val, key
    resident = somcb.SomTrainer(_cb(k, w0), lr=LR, neighbourhood_step=2, use_cuda_graph="alias")
    want = [float(resident.step(h.to(DEV))) for h in hosts]
    assert [p.item() for p in pending] == want[1:]
    assert torch.equal(early["m"], resident.m.cpu()) and torch.equal(early["v"], resident.v.cpu())
    assert early["t_dev"] == int(resident.t_dev[0]) == early["t"] == 5
    assert (early["lr"], early["global_steps"], early["neighbourhood_range"]) == \
        (resident.lr, resident.global_steps, resident.cb.neighbourhood_range)


def test_multi_gpu_resume_under_torchrun():
    """With at least two GPUs visible: tests/multi_gpu_resume_check.py under torch.distributed.run -- split run ==
    straight run on the NCCL and the peer tail, full moments in the saved state, and a state saved at N GPUs resumed at
    one and the other way round.  Skips on a one-GPU box (the gloo test covers the host logic on CPU)."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    world = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29737",
                        os.path.join(root, "tests", "multi_gpu_resume_check.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "MULTI_GPU_RESUME_CHECK PASS" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
