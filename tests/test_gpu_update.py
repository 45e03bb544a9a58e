"""GPU parity of the neighbourhood-weighted update (K2, K3, K4, quantise) through the C-ABI:
per-kernel checks against dense fp64 forms, the drop-in autograd path and the fused SomTrainer
against the reference's golden step, and the 100-step free run of BASELINE config 1."""
import pytest
import torch
import torch.nn.functional as F

import somcb
from somcb import ops
from oracle import neighbourhood_two_var
from oracle.step_oracle import synthetic_fmaps
from _helpers import (CASES, assert_bmu_parity, assert_close_norm, assert_weights_parity, flat_patches,
                      fp64_truth_step, golden_rows, load_case, load_golden, rel_fro)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _gpu_cb(rec, weight_key="weight", rng=None):
    cb = somcb.Codebook(patch_dim=rec["patch_dim"], image_dim=rec["image_dim"],
                        image_channel=rec["channels"], num_embeddings=rec[weight_key].shape[0],
                        init_neighbour_range=rec["neighbourhood_range"] if rng is None else rng)
    with torch.no_grad():
        cb.codebook.weight.copy_(rec[weight_key])
    return cb.to(DEV)


def _dense_t(k, rng):
    ids = torch.arange(k)
    return torch.exp(-(((ids.unsqueeze(0) - ids.unsqueeze(1)) ** 2) / neighbourhood_two_var(rng))).double()


@pytest.mark.parametrize("k,d,rng", [(1024, 64, 512), (1024, 64, 1.0), (37, 18, 5), (4096, 16, 2048),
                                     (512, 4096, 256), (100, 33, 100), (2048, 256, 7)])
def test_filter_matches_dense_toeplitz(k, d, rng):
    g = torch.Generator().manual_seed(k + d)
    w = torch.randn(k, d, generator=g)
    want = _dense_t(k, rng) @ w.double()
    got = ops.neighbourhood_filter(w.to(DEV), rng)
    assert_close_norm(got, want, 2e-6, "T@W")
    got2 = ops.neighbourhood_filter(w.to(DEV), rng, scale=0.125)
    assert_close_norm(got2, want * 0.125, 2e-6, "scaled T@W")


@pytest.mark.parametrize("k,d,rng", [(1024, 64, 512), (512, 4096, 256), (300, 50, 40), (4100, 50, 40), (1000, 530, 3),
                                     (300, 4096, 0.5), (4096, 64, 2048), (2100, 200, 4000.0), (640, 64, 1.0)])
def test_filter_tensor_core_and_ffma_kernels_agree(k, d, rng):
    """K >= 256, D >= 48 and at least 32 tiles take the tcgen05 banded-Toeplitz GEMM (fp32-faithful 3xTF32; here
    cases 2, 4, 5, 6, 7 and 8): both kernels must agree
    with the dense fp64 product -- partial unit tiles, feature counts that are not multiples of 4 / 32 / the tile,
    bands from one unit to wider than the codebook, a non-trivial scale, guard bands around the output."""
    g = torch.Generator().manual_seed(k * 7 + d)
    w = torch.randn(k, d, generator=g)
    want = 0.37 * (_dense_t(k, rng) @ w.double())
    wd = w.to(DEV)
    for tc in (True, False):
        buf = torch.full((k * d + 8,), 7.0, device=DEV)
        out = (buf[4:-4] if k % 2 else buf[5:-3]).view(k, d)          # 16-byte aligned / 4-byte aligned output
        ops.neighbourhood_filter(wd, rng, scale=0.37, out=out, tensor_cores=tc)
        assert_close_norm(out, want, 2e-6, f"T@W tensor_cores={tc}")
        assert float((out.double().cpu() - want).abs().max()) <= 2e-6 * float(want.abs().max())
        assert bool((buf[:4] == 7.0).all()) and bool((buf[-3:] == 7.0).all())
    a = ops.neighbourhood_filter(wd, rng)
    b = ops.neighbourhood_filter(wd, rng)
    assert torch.equal(a, b)                                     # deterministic


def test_filter_c4_shape_tensor_core_vs_ffma():
    """BASELINE C4 codebook (K = 16384, D = 64, range 8192: band 1217): too large for the dense fp64 check, so the
    two kernels are compared with each other."""
    g = torch.Generator().manual_seed(5)
    w = torch.randn(16384, 64, generator=g).to(DEV)
    a = ops.neighbourhood_filter(w, 8192)
    b = ops.neighbourhood_filter(w, 8192, tensor_cores=False)
    assert_close_norm(a, b.double().cpu(), 2e-6, "tensor-core vs FFMA filter")


@pytest.mark.parametrize("name", CASES)
def test_accumulate_matches_index_add(name):
    rec = load_case(name)
    x = rec["x"].to(DEV)
    geom = ops.geometry(x.shape, rec["patch_dim"])
    k, d = rec["weight"].shape
    flat = flat_patches(rec["x"], rec["patch_dim"]).double()
    bmu = rec["bmu"]
    table = torch.randn(k, d, generator=torch.Generator().manual_seed(5))
    # residual mode
    rbar, counts, sse = ops.accumulate(x, geom, bmu.to(DEV), table.to(DEV), k, want_counts=True, want_sse=True)
    r = table.double()[bmu] - flat
    want = torch.zeros(k, d, dtype=torch.float64).index_add_(0, bmu, r)
    assert_close_norm(rbar, want, 2e-6, "Rbar")
    assert torch.equal(counts.cpu(), torch.bincount(bmu, minlength=k))
    assert abs(float(sse) - float((r ** 2).sum())) <= 2e-6 * float((r ** 2).sum())
    # plain-sum mode (autograd backward)
    xbar, _, _ = ops.accumulate(x, geom, bmu.to(DEV), None, k)
    want2 = torch.zeros(k, d, dtype=torch.float64).index_add_(0, bmu, flat)
    assert_close_norm(xbar, want2, 2e-6, "Xbar")
    # deterministic: bit-identical on a second run
    rbar2, _, sse2 = ops.accumulate(x, geom, bmu.to(DEV), table.to(DEV), k, want_sse=True)
    assert torch.equal(rbar, rbar2) and torch.equal(sse, sse2)


@pytest.mark.parametrize("pattern", ["one_unit", "two_units", "sorted_runs", "random_sparse"])
def test_accumulate_skewed_segments(pattern):
    """Heavy hitters spanning many chunks, empty units, segments ending on chunk edges."""
    n_f, pd, k = 96, (4, 4), 300
    x = synthetic_fmaps(n_f, 77)
    flat = flat_patches(x, pd).double()
    n = flat.shape[0]
    g = torch.Generator().manual_seed(3)
    if pattern == "one_unit":
        bmu = torch.full((n,), 123, dtype=torch.int64)
    elif pattern == "two_units":
        bmu = torch.where(torch.arange(n) % 3 == 0, 7, 299).to(torch.int64)
    elif pattern == "sorted_runs":
        bmu = (torch.arange(n) // 64 % k).to(torch.int64)
    else:
        bmu = torch.randint(0, k, (n,), generator=g) // 50 * 50
    table = torch.randn(k, 64, generator=g)
    xd = x.to(DEV)
    geom = ops.geometry(x.shape, pd)
    rbar, counts, sse = ops.accumulate(xd, geom, bmu.to(DEV), table.to(DEV), k, want_counts=True, want_sse=True)
    r = table.double()[bmu] - flat
    want = torch.zeros(k, 64, dtype=torch.float64).index_add_(0, bmu, r)
    assert_close_norm(rbar, want, 5e-6, "Rbar")
    assert torch.equal(counts.cpu(), torch.bincount(bmu, minlength=k))
    empty = torch.bincount(bmu, minlength=k) == 0
    assert float(rbar.cpu()[empty].abs().max()) == 0.0
    assert abs(float(sse) - float((r ** 2).sum())) <= 5e-6 * float((r ** 2).sum())


@pytest.mark.parametrize("fmaps,k", [(33, 300), (79, 300), (128, 16384), (129, 300), (20, 70000), (1, 70000)])
def test_accumulate_small_and_medium_batches(fmaps, k):
    """64 to 8256 patches, codebooks of 300 to 70000 units (K = 70000 keeps tiny batches off the scan path, so the
    sorted path also sees them): fp64 index_add, counts, empty units exactly zero, SSE, bit-identical repeat."""
    pd = (4, 4)
    x = synthetic_fmaps(fmaps, 5 + fmaps)
    flat = flat_patches(x, pd).double()
    n = flat.shape[0]
    g = torch.Generator().manual_seed(n)
    bmu = torch.randint(0, k, (n,), generator=g)
    bmu[::3] = bmu[0]                                       # a heavy hitter
    table = torch.randn(k, 64, generator=g)
    xd, geom = x.to(DEV), ops.geometry(x.shape, pd)
    rbar, counts, sse = ops.accumulate(xd, geom, bmu.to(DEV), table.to(DEV), k, want_counts=True, want_sse=True)
    r = table.double()[bmu] - flat
    want = torch.zeros(k, 64, dtype=torch.float64).index_add_(0, bmu, r)
    assert_close_norm(rbar, want, 5e-6, "Rbar")
    hits = torch.bincount(bmu, minlength=k)
    assert torch.equal(counts.cpu(), hits)
    if bool((hits == 0).any()):
        assert float(rbar.cpu()[hits == 0].abs().max()) == 0.0
    assert abs(float(sse) - float((r ** 2).sum())) <= 5e-6 * float((r ** 2).sum())
    rbar2, _, sse2 = ops.accumulate(xd, geom, bmu.to(DEV), table.to(DEV), k, want_sse=True)
    assert torch.equal(rbar, rbar2) and torch.equal(sse, sse2)


@pytest.mark.parametrize("fmaps,k,skew", [(128, 16384, False), (2048, 16384, False), (2500, 16384, True), (515, 5000, True),
                                          (4096, 300, True)])
def test_accumulate_counting_sort_equals_radix_sort_path(fmaps, k, skew):
    """Codebooks of up to 16 384 units sort the (unit, patch) pairs with the library's own one-pass stable counting sort,
    larger ones with cub's radix sort.  Both are stable, so the segmented sums must be BIT-identical: the same hits are
    accumulated once with K units and once with K + 16 385 units (the extra units stay empty and push the call onto
    the radix path).  Covers several sort blocks, more than one block per SM's worth of patches, and a heavy hitter."""
    pd = (4, 4)
    x = synthetic_fmaps(fmaps, 901 + fmaps).to(DEV)
    geom = ops.geometry(x.shape, pd)
    n = ops.n_patches_of(geom)
    g = torch.Generator().manual_seed(n + k)
    bmu = torch.randint(0, k, (n,), generator=g)
    if skew:
        bmu[::2] = k - 1                                     # half of the batch on the last unit
        bmu[1::64] = 0
    k_big = k + 16385
    table = torch.randn(k_big, 64, generator=g).to(DEV)
    bmu = bmu.to(DEV)
    small, c_small, sse_small = ops.accumulate(x, geom, bmu, table[:k].contiguous(), k, want_counts=True, want_sse=True)
    big, c_big, sse_big = ops.accumulate(x, geom, bmu, table, k_big, want_counts=True, want_sse=True)
    assert torch.equal(small, big[:k])
    assert float(big[k:].abs().max()) == 0.0
    assert torch.equal(c_small, c_big[:k]) and int(c_big[k:].sum()) == 0
    assert torch.equal(sse_small, sse_big)


def _teacher_force(monkeypatch, rec):
    """Make the drop-in module's BMU search return the reference's own indices (teacher forcing, SURVEY 8c.2): from
    the reference's fresh init a near-tie may resolve differently, and the quantise / autograd outputs are only
    comparable element-wise on the same BMUs.  The rest of the path (_FilterFn, _GatherFn, backward) runs unchanged."""
    import somcb.codebook as cbmod
    golden = rec["bmu"].to(DEV)
    real = cbmod.ops.bmu

    def forced(x, geom, weight, c_norm2=None, **kw):
        real(x, geom, weight, c_norm2, **kw)               # the kernel still runs (and must not fail)
        return golden.clone()
    monkeypatch.setattr(cbmod.ops, "bmu", forced)


@pytest.mark.parametrize("name", CASES)
def test_quantize_paths_match_reference(name, monkeypatch):
    rec = load_case(name)
    cb = _gpu_cb(rec)
    x = rec["x"].to(DEV)
    with torch.no_grad():
        bmu = cb.get_patches_bmu(x)
        if not torch.equal(bmu.cpu(), rec["bmu"]):
            assert_bmu_parity(bmu, rec["bmu"], flat_patches(rec["x"], rec["patch_dim"]), rec["weight"])
            _teacher_force(monkeypatch, rec)
        assert torch.equal(*golden_rows(rec, "quant_hard", cb.get_quantized_patches(x, use_gaussian=False).cpu()))
        assert torch.equal(*golden_rows(rec, "quant_image", cb.get_quantized_image(rec["bmu_reshaped"].to(DEV)).cpu()))
        qi = cb.get_quantized_image(rec["bmu_reshaped"].to(DEV), unpatchify_input=False)
        assert torch.equal(*golden_rows(rec, "quant_hard", qi.cpu()))
        assert_close_norm(*golden_rows(rec, "quant_gauss", cb.get_quantized_patches(x).cpu()), 1e-5, "quant_gauss")
        assert_close_norm(*golden_rows(rec, "forward_gauss", cb(x).cpu()), 1e-5, "forward")


@pytest.mark.parametrize("name", CASES)
def test_dropin_autograd_step_matches_reference(name, monkeypatch):
    """The literal step body of train_codebook.py:227-242 with somcb.Codebook in place of the
    reference class and torch.optim.Adam owning the update.  Where a fresh-init near-tie resolves differently
    from the reference the step is teacher-forced with the reference's BMU (the gradient still flows through
    _GatherFn.backward and _FilterFn.backward)."""
    rec = load_case(name)
    cb = _gpu_cb(rec)
    opt = torch.optim.Adam(cb.parameters(), lr=1e-4, betas=(0.5, 0.999))
    x = rec["x"].to(DEV)
    with torch.no_grad():
        if not torch.equal(cb.get_patches_bmu(x).cpu(), rec["bmu"]):
            _teacher_force(monkeypatch, rec)
    cb.train()
    opt.zero_grad()
    quant = cb(x, use_gaussian=True)
    loss = F.mse_loss(quant, x)
    assert not torch.isnan(loss)
    loss.backward()
    grad = cb.codebook.weight.grad
    assert grad is not None
    g, g_ref = golden_rows(rec, "grad", grad)
    assert g.shape == g_ref.shape
    opt.step()
    assert_close_norm(loss, rec["loss"], 1e-5, "loss")
    assert_close_norm(g, g_ref, 1e-5, "grad")
    w_truth, _, _ = fp64_truth_step(rec)
    w, w_truth, w_ref = golden_rows(rec, "weight_after_step", cb.codebook.weight.detach(), w_truth)
    assert_weights_parity(w, w_ref, w_truth)


@pytest.mark.parametrize("name", CASES)
def test_fused_trainer_step_teacher_forced(name):
    """SomTrainer.step with the reference's own BMU (teacher forcing, SURVEY 8c.2)."""
    rec = load_case(name)
    cb = _gpu_cb(rec)
    tr = somcb.SomTrainer(cb, lr=1e-4, neighbourhood_step=10 ** 9)
    loss = tr.step(rec["x"].to(DEV), bmu=rec["bmu"].to(DEV))
    assert_close_norm(loss, rec["loss"], 1e-5, "loss")
    w_truth, _, _ = fp64_truth_step(rec)
    w, w_truth, w_ref = golden_rows(rec, "weight_after_step", cb.codebook.weight.detach(), w_truth)
    assert_weights_parity(w, w_ref, w_truth)


@pytest.mark.parametrize("path", ["fused", "dropin"])
def test_free_run_100_steps_c1(path):
    """BASELINE config 1 (B=8, P=4, K=1024, 100 steps) from a trained-like init, free-running."""
    run = load_golden("run_c1_trained_100.pt")
    rec = {"patch_dim": run["patch_dim"], "image_dim": run["image_dim"], "channels": run["channels"],
           "weight": run["weight0"], "neighbourhood_range": run["range0"]}
    cb = _gpu_cb(rec)
    if path == "fused":
        tr = somcb.SomTrainer(cb, lr=run["lr"], neighbourhood_step=run["neighbourhood_step"])
    else:
        opt = torch.optim.Adam(cb.parameters(), lr=run["lr"], betas=(0.5, 0.999))
        gs = 0
    for step in range(100):
        x = synthetic_fmaps(8, 123 + step).to(DEV)
        if path == "fused":
            loss = tr.step(x)
        else:
            opt.zero_grad()
            loss = F.mse_loss(cb(x, use_gaussian=True), x)
            loss.backward()
            opt.step()
            gs += 1
            if gs % run["neighbourhood_step"] == 0:
                cb.decrease_neighbourhood(steps=1)
        ref_loss = float(run["losses"][step])
        assert abs(float(loss) - ref_loss) <= 1e-5 * abs(ref_loss), f"loss at step {step}"
        assert cb.neighbourhood_range == run["ranges"][step]
        if step + 1 in run["weights"]:
            w, snaps = golden_rows(run, "weights", cb.codebook.weight.detach())
            assert_close_norm(w, snaps[step + 1], 1e-5, f"weights@{step + 1}")


def test_adam_kernel_matches_torch_adam():
    g = torch.Generator().manual_seed(11)
    w0 = torch.randn(257, 33, generator=g)
    p = torch.nn.Parameter(w0.clone())
    opt = torch.optim.Adam([p], lr=3e-3, betas=(0.5, 0.999))
    w = w0.clone().to(DEV)
    m = torch.zeros_like(w)
    v = torch.zeros_like(w)
    for t in range(1, 8):
        grad = torch.randn(257, 33, generator=g) * (10.0 ** (-t))
        p.grad = grad.clone()
        opt.step()
        ops.adam_step(w, m, v, grad.to(DEV), 3e-3, t)
        assert rel_fro(w, p.detach()) <= 2e-7


def test_cuda_graph_trainer_matches_eager_trainer():
    """SomTrainer(use_cuda_graph=True): 60 steps of config 1 with the neighbourhood range shrinking every 20
    steps (forces two re-captures) against the eager fused trainer -- same losses and weights."""
    from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
    pd, k = (4, 4), 1024
    w0 = trained_like_codebook(k, pd, 7)
    trainers = []
    for graph in (False, True, "alias"):
        cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4, num_embeddings=k,
                            init_neighbour_range=k // 2)
        with torch.no_grad():
            cb.codebook.weight.copy_(w0)
        cb = cb.to(DEV)
        trainers.append(somcb.SomTrainer(cb, lr=1e-4, neighbourhood_step=20, use_cuda_graph=graph))
    staging = torch.empty(8, 4, 32, 32, device=DEV)        # the "alias" trainer replays on this buffer
    for step in range(60):
        x = synthetic_fmaps(8, 123 + step).to(DEV)
        staging.copy_(x)
        l0 = float(trainers[0].step(x))
        l1 = float(trainers[1].step(x))
        l2 = float(trainers[2].step(staging))
        assert abs(l0 - l1) <= 1e-6 * abs(l0), f"step {step}: loss {l0} vs {l1}"
        assert abs(l0 - l2) <= 1e-6 * abs(l0), f"step {step}: loss {l0} vs {l2} (alias)"
    for tr in trainers[1:]:
        assert len(tr._graphs) == 3 and tr.t == 60 and int(tr.t_dev[0]) == 60
        assert trainers[0].cb.neighbourhood_range == tr.cb.neighbourhood_range == k // 2 - 3
        assert_close_norm(tr.cb.codebook.weight.data, trainers[0].cb.codebook.weight.data,
                          what="weights after 60 graph-replayed steps")
    assert all(entry[1] is staging for entry in trainers[2]._graphs.values())
    # an eager (teacher-forced) step between replays shares the device-resident Adam step count with the graph
    x = synthetic_fmaps(8, 999).to(DEV)
    forced = trainers[0].cb.get_patches_bmu(x)
    for tr in trainers[:2]:
        tr.step(x, bmu=forced)
        tr.step(x)
    assert trainers[1].t == 62 and int(trainers[1].t_dev[0]) == 62
    assert_close_norm(trainers[1].cb.codebook.weight.data, trainers[0].cb.codebook.weight.data,
                      what="weights after an eager step between graph replays")


@pytest.mark.parametrize("graph", [False, True])
def test_filter_on_a_side_stream_gives_the_same_step(graph):
    """W~ = T @ W runs on a side stream beside the search (SomTrainer(overlap_filter=True), fork / join by stream waits,
    also inside a captured graph): same kernels on the same data, so losses and weights must be BIT-identical to the
    one-stream order, step after step (a missing join would show up as a stale or half-written W~)."""
    from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
    pd, k = (4, 4), 2048
    w0 = trained_like_codebook(k, pd, 11)
    trainers = []
    for overlap in (True, False):
        cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4, num_embeddings=k,
                            init_neighbour_range=k // 2)
        with torch.no_grad():
            cb.codebook.weight.copy_(w0)
        trainers.append(somcb.SomTrainer(cb.to(DEV), lr=1e-3, neighbourhood_step=4, use_cuda_graph=graph,
                                         overlap_filter=overlap, small_step_kernel=False))
    for step in range(12):
        x = synthetic_fmaps(64, 500 + step).to(DEV)           # 4096 patches: the separate-kernel path
        la, lb = trainers[0].step(x), trainers[1].step(x)
        assert float(la) == float(lb), f"step {step}: loss {float(la)} vs {float(lb)}"
        assert torch.equal(trainers[0].cb.codebook.weight.data, trainers[1].cb.codebook.weight.data), f"step {step}"
    assert trainers[0]._side is not None and trainers[1]._side is None


def test_trainer_nan_guard():
    """check_nan=True restores the reference's guard (train_codebook.py:237-238)."""
    from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
    cb = somcb.Codebook(patch_dim=(4, 4), image_dim=(32, 32), image_channel=4, num_embeddings=1024,
                        init_neighbour_range=512)
    with torch.no_grad():
        cb.codebook.weight.copy_(trained_like_codebook(1024, (4, 4), 7))
    cb = cb.to(DEV)
    tr = somcb.SomTrainer(cb, lr=1e-4, neighbourhood_step=10 ** 9, check_nan=True)
    x = synthetic_fmaps(8, 1).to(DEV)
    tr.step(x)
    x[0, 0, 0, 0] = float("nan")
    with pytest.raises(Exception, match="NaN encountered during training"):
        tr.step(x)


def test_packed_accumulate_and_device_scaled_adam_match_the_host_scaled_path():
    """som_accumulate_packed_nchw_f32 + som_adam_dp_f32 (batch size and loss on the device) against
    som_accumulate_nchw_f32 + host-scaled filter + som_adam_f32: bit-identical weights, loss to fp64 rounding."""
    from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
    pd, k, d = (4, 4), 2048, 64
    x = synthetic_fmaps(96, 5).to(DEV)
    w = trained_like_codebook(k, pd, 7).to(DEV)
    geom = ops.geometry(x.shape, pd)
    wt = ops.neighbourhood_filter(w, 300)
    bmu = ops.bmu(x, geom, w)
    rbar, _, sse = ops.accumulate(x, geom, bmu, wt, k, want_sse=True)
    packed = ops.accumulate_packed(x, geom, bmu, wt, k)
    assert torch.equal(packed[:k * d].view(k, d), rbar)
    n = ops.n_patches_of(geom)
    assert float(packed[k * d + 2]) * 4096 + float(packed[k * d + 3]) == n
    assert abs(float(packed[k * d].double() + packed[k * d + 1].double()) - float(sse)) <= 1e-12 * float(sse)
    numel = x.numel()
    w_a, m_a, v_a = w.clone(), torch.zeros_like(w), torch.zeros_like(w)
    w_b, m_b, v_b = w.clone(), torch.zeros_like(w), torch.zeros_like(w)
    t_dev = torch.zeros(2, dtype=torch.int64, device=DEV)
    for t in (1, 2, 3):
        g_a = ops.neighbourhood_filter(rbar, 300, scale=2.0 / numel)
        ops.adam_step(w_a, m_a, v_a, g_a, 1e-4, t)
        g_b = ops.neighbourhood_filter(rbar, 300, scale=1.0)
        loss = ops.adam_step_dp(w_b, m_b, v_b, g_b, d, 1e-4, t_dev, packed[k * d:])
        assert torch.equal(w_a, w_b) and torch.equal(v_a, v_b)
    assert int(t_dev[0]) == 3 and int(t_dev[1]) == 0
    assert abs(float(loss) - float(sse) / numel) <= 1e-12 * float(loss)


def test_staging_copy_from_the_bmu_kernel_feeds_the_accumulation():
    """Large batches of 16 < D <= 256: the FP16-split BMU kernel also writes the patch-major copy of the patch rows
    (som_bmu_stage_nchw_f32); the copy equals patchify(x) bit for bit, the accumulation from it equals the
    accumulation from NCHW bit for bit, and a trainer step through it matches the step that reads NCHW."""
    from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
    for p, k, n_f in ((4, 2048, 320), (8, 1024, 2400)):
        pd, d = (p, p), 4 * p * p
        x = synthetic_fmaps(n_f, 31).to(DEV)
        w = trained_like_codebook(k, pd, 7).to(DEV)
        geom = ops.geometry(x.shape, pd)
        npat = ops.n_patches_of(geom)
        assert ops.bmu_can_stage(geom, k)
        stage = torch.empty(npat, d, device=DEV)
        idx = ops.bmu(x, geom, w, stage=stage)
        assert torch.equal(idx, ops.bmu(x, geom, w))
        assert torch.equal(stage, somcb.patchify(x, pd).reshape(npat, d))
        wt = ops.neighbourhood_filter(w, k // 4)
        a = ops.accumulate_packed(x, geom, idx, wt, k)
        b = ops.accumulate_packed(stage, ops.flat_geometry(npat, d), idx, wt, k)
        assert torch.equal(a, b)
    assert not ops.bmu_can_stage(ops.geometry((8, 4, 32, 32), (4, 4)), 1024)      # small batch: 3xTF32 kernel
    with pytest.raises(somcb._lib.SomError):
        xs = synthetic_fmaps(8, 1).to(DEV)
        g8 = ops.geometry(xs.shape, (4, 4))
        ops.bmu(xs, g8, trained_like_codebook(1024, (4, 4), 7).to(DEV), stage=torch.empty(512, 64, device=DEV))


@pytest.mark.parametrize("p,k,n_f,rng", [(4, 1024, 8, 512), (2, 512, 4, 256), (8, 300, 16, 32), (4, 4096, 8, 512),
                                         (4, 1024, 32, 100)])
def test_one_kernel_small_step_matches_the_separate_kernels(p, k, n_f, rng):
    """som_step_small_f32 (BASELINE config 1's whole step as one cooperative kernel) against the step built from the
    separate kernels: 12 free-running steps with the neighbourhood range shrinking, same losses, weights and BMUs; also
    captured in a CUDA graph."""
    from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
    pd = (p, p)
    w0 = trained_like_codebook(k, pd, 7)
    trainers = []
    for small, graph in ((True, False), (False, False), (True, True)):
        cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4, num_embeddings=k,
                            init_neighbour_range=rng)
        with torch.no_grad():
            cb.codebook.weight.copy_(w0)
        trainers.append(somcb.SomTrainer(cb.to(DEV), lr=1e-4, neighbourhood_step=5, small_step_kernel=small,
                                         use_cuda_graph=graph))
    geom = ops.geometry((n_f, 4, 32, 32), pd)
    assert ops.step_small_supported(geom, k, rng)
    for step in range(12):
        x = synthetic_fmaps(n_f, 700 + step).to(DEV)
        ls = [float(tr.step(x)) for tr in trainers]
        assert abs(ls[0] - ls[1]) <= 2e-6 * abs(ls[1]), f"step {step}: loss {ls[0]} vs {ls[1]}"
        assert ls[0] == ls[2], f"step {step}: graph replay {ls[2]} vs eager {ls[0]}"
        if step == 0:
            flat = flat_patches(x.cpu(), pd)
            assert_bmu_parity(trainers[0].last_bmu, trainers[1].last_bmu, flat, w0)
    assert trainers[0].t == 12 and int(trainers[0].t_dev[0]) == 12
    assert_close_norm(trainers[0].cb.codebook.weight.data, trainers[1].cb.codebook.weight.data, 1e-6,
                      "one-kernel step vs separate kernels")
    assert torch.equal(trainers[0].cb.codebook.weight.data, trainers[2].cb.codebook.weight.data)
    # not covered: more than 2048 patches, or a band whose staged rows do not fit in shared memory
    assert not ops.step_small_supported(ops.geometry((64, 4, 32, 32), (2, 2)), 512, 256)
    assert not ops.step_small_supported(ops.geometry((8, 4, 32, 32), (8, 8)), 300, 150)
