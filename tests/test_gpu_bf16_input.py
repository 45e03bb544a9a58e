"""bf16 feature maps on the GPU: every result must be BIT-identical to the fp32 path on x.float() -- the native
FP16-split kernel (whose bf16 tiles skip the A_lo x B_hi products where every lo operand is zero, and keep them where
one is not), the upcast route of every other kernel, the trainers, the host pipeline and the drop-in Codebook."""
import os

import pytest
import torch

import somcb
from somcb import ops
from somcb.fmap_shards import ShardReader, shard_torch_dtype, write_shard
from somcb.host_pipeline import HostTokenizer, HostTrainer
from somcb.tokenizer import tokenize_pair
from oracle.step_oracle import make_oracle_codebook, make_reference_optimizer, reference_step, synthetic_fmaps
from oracle.step_oracle import trained_like_codebook
from _helpers import assert_bmu_parity, assert_close_norm, flat_patches
from test_bf16_input_host import KINDS, _special_rows
from test_gpu_f16_input import NATIVE, UPCAST, _assert_same_search, _bits, _cb, _codebook

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _fmaps_bf16(n, c, seed, hw=32):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.tanh(torch.randn(n, c, hw, hw, device=DEV, generator=g)).bfloat16()


@pytest.mark.parametrize("c,pd,n,k,variant,off", NATIVE)
def test_native_bf16_kernel_equals_fp32_on_upcast(c, pd, n, k, variant, off):
    xb = _fmaps_bf16(n, c, 1 + n)
    geom = ops.geometry(xb.shape, pd)
    w = _codebook(k, ops.dim_of(geom), 2)
    assert ops.bmu_f16_native(geom, k, variant)
    _assert_same_search(xb, geom, w, variant, unit_offset=off)


@pytest.mark.parametrize("n_rows,variant", [(4096, ops.SOM_BMU_TC_F16), (20480, ops.SOM_BMU_AUTO)])
def test_special_rows_inside_one_tile(n_rows, variant):
    """Every row kind of the host emulation in the second tile (bf16 rows below 2^-23 of their max, subnormals, the
    clamped scale, NaN, inf: tiles that keep the third product) and, in the third tile, the kinds that let a tile
    drop it."""
    d, k = 64, 1024
    special = torch.from_numpy(_special_rows(d)).bfloat16()
    x = flat_patches(synthetic_fmaps(n_rows // 64, 5), (4, 4)).bfloat16()
    x[130:130 + special.shape[0]] = special
    clean = [i for i, keep in enumerate(KINDS.values()) if not keep]
    x[260:260 + len(clean)] = special[clean]
    w = trained_like_codebook(k, (4, 4), 7)
    geom = ops.flat_geometry(n_rows, d)
    xb, wd = x.to(DEV).contiguous(), w.to(DEV)
    assert ops.bmu_f16_native(geom, k, variant)
    idx = _assert_same_search(xb, geom, wd, variant).cpu()
    nan_row = 130 + list(KINDS).index("nan")
    assert int(idx[nan_row]) == 0, "a patch holding a NaN gets unit 0"
    finite = torch.isfinite(x.float()).all(1)
    flat = x.float()[finite]
    w64 = w.double()
    ref = ((w64 * w64).sum(1)[None, :] - 2 * flat.double() @ w64.T).argmin(1)
    assert_bmu_parity(idx[finite], ref, flat, w)


@pytest.mark.parametrize("c,pd,n,k,variant", UPCAST)
def test_upcast_route_equals_fp32_on_upcast(c, pd, n, k, variant):
    xb = _fmaps_bf16(n, c, 3 + n)
    geom = ops.geometry(xb.shape, pd)
    w = _codebook(k, ops.dim_of(geom), 4)
    assert not ops.bmu_f16_native(geom, k, variant)
    _assert_same_search(xb, geom, w, variant, stage=False)


def test_upcast_bf16_is_exact_and_handles_unaligned_tails():
    bits = torch.arange(0, 65536, dtype=torch.int32).to(torch.int16).to(DEV)
    h = bits.view(torch.bfloat16)
    want = (bits.to(torch.int32) << 16).view(torch.float32)              # bf16 -> fp32 is the bit pattern << 16

    def same(a, b):                                                   # every value bit for bit, NaN as NaN
        nan = torch.isnan(b)
        return torch.equal(torch.isnan(a), nan) and torch.equal(_bits(a)[~nan], _bits(b)[~nan])

    assert same(h.float(), want)
    for lo, hi in ((0, 65536), (1, 65536), (3, 65533), (8, 17)):
        assert same(ops.upcast_bf16(h[lo:hi].contiguous()), want[lo:hi])
        out = torch.empty(hi - lo + 1, device=DEV)[1:]               # 4-byte but not 16-byte aligned output
        ops.upcast_bf16(h[lo:hi].contiguous(), out=out)
        assert same(out, want[lo:hi])
    with pytest.raises(TypeError):
        ops.upcast_bf16(h.view(torch.float16))
    with pytest.raises(TypeError):
        ops.upcast_f16(h)


@pytest.mark.parametrize("n,k,graph", [(1024, 16384, False), (1024, 16384, True), (1024, 16384, "alias"),
                                       (8, 1024, False), (8, 1024, "alias")])
def test_trainer_bf16_steps_equal_fp32_on_upcast(n, k, graph):
    pd = (4, 4)
    w0 = trained_like_codebook(k, pd, 7)
    batches = [_fmaps_bf16(n, 4, 50 + s) for s in range(5)]
    out = []
    for half in (True, False):
        cb = _cb(w0, pd, 4, k // 2)
        tr = somcb.SomTrainer(cb, lr=1e-4, neighbourhood_step=3, use_cuda_graph=graph)
        losses = []
        for xb in batches:
            x = xb if half else xb.float()
            losses.append(tr.step(x).clone())
        torch.cuda.synchronize()
        out.append((cb.codebook.weight.detach().clone(), torch.stack(losses)))
    (wb, lb), (w32, l32) = out
    assert torch.equal(_bits(wb), _bits(w32)), "weights differ after 5 steps"
    assert torch.equal(lb.view(torch.int64), l32.view(torch.int64)), "losses differ"


@pytest.mark.parametrize("graph", [True, "alias"])
def test_fp16_and_bf16_batches_capture_separate_graphs(graph):
    pd, k, n = (4, 4), 16384, 1024
    w0 = trained_like_codebook(k, pd, 7)
    src = [_fmaps_bf16(n, 4, 80 + s).float() for s in range(4)]
    batches = [x.half() if s % 2 == 0 else x.bfloat16() for s, x in enumerate(src)]
    out = []
    for half in (True, False):
        cb = _cb(w0, pd, 4, k // 2)
        tr = somcb.SomTrainer(cb, lr=1e-4, neighbourhood_step=3, use_cuda_graph=graph)
        losses = [tr.step(x if half else x.float()).clone() for x in batches]
        torch.cuda.synchronize()
        out.append((cb.codebook.weight.detach().clone(), torch.stack(losses), {key[1] for key in tr._graphs}))
    (wh, lh, dtypes), (w32, l32, _) = out
    assert dtypes == {torch.float16, torch.bfloat16}, "one graph per 16-bit dtype"
    assert torch.equal(_bits(wh), _bits(w32)) and torch.equal(lh.view(torch.int64), l32.view(torch.int64))


def test_c1_bf16_run_matches_the_oracle_on_upcast_inputs():
    pd, k, lr = (4, 4), 1024, 1e-4
    w0 = trained_like_codebook(k, pd, 7)
    ocb = make_oracle_codebook(w0, pd, (32, 32), 4, k // 2)
    opt = make_reference_optimizer(ocb, lr)
    cb = _cb(w0, pd, 4, k // 2)
    tr = somcb.SomTrainer(cb, lr=lr, neighbourhood_step=10 ** 6)
    for step in range(20):
        xb = synthetic_fmaps(8, 123 + step).bfloat16()
        ref = float(reference_step(ocb, opt, xb.float()))
        got = float(tr.step(xb.to(DEV)))
        assert abs(got - ref) <= 1e-5 * abs(ref), f"loss at step {step}"
    assert_close_norm(cb.codebook.weight.detach().cpu(), ocb.codebook.weight.detach(), 1e-5, "weights@20")


def test_host_trainer_with_bf16_pinned_batches_equals_resident_run():
    pd, k = (4, 4), 16384
    w0 = trained_like_codebook(k, pd, 7)
    host = [synthetic_fmaps(512, 70 + s).bfloat16().pin_memory() for s in range(4)]  # 32 768 patches: native
    cb_h = _cb(w0, pd, 4, k // 2)
    ht = HostTrainer(somcb.SomTrainer(cb_h, lr=1e-4, neighbourhood_step=3, use_cuda_graph="alias"))
    lh = [ht.step(b).item() for b in host]
    cb_r = _cb(w0, pd, 4, k // 2)
    tr = somcb.SomTrainer(cb_r, lr=1e-4, neighbourhood_step=3, use_cuda_graph="alias")
    resident = [b.float().to(DEV) for b in host]
    lr_ = [float(tr.step(x)) for x in resident]
    assert lh == lr_
    assert torch.equal(_bits(cb_h.codebook.weight.detach()), _bits(cb_r.codebook.weight.detach()))
    assert ht._slots[1][0]["x"].dtype == torch.bfloat16


def test_host_tokenizer_and_bf16_shards_equal_resident_search(tmp_path):
    pd, k = (2, 2), 4096
    cb = _cb(trained_like_codebook(k, pd, 7), pd, 4, k // 2)
    xb = synthetic_fmaps(600, 9).bfloat16()
    want = cb.get_patches_bmu(xb.float().to(DEV), reshape=True).cpu()
    tok = HostTokenizer(cb, chunk_fmaps=256)
    assert torch.equal(tok.tokenize(xb.pin_memory()), want)
    assert tok._bufs[1][0][0]["x"].dtype == torch.bfloat16
    paths = []
    for i, (lo, hi) in enumerate(((0, 250), (250, 600))):
        paths.append(os.path.join(tmp_path, f"s{i}.shard"))
        write_shard(paths[-1], xb[lo:hi], dtype=torch.bfloat16)
        assert shard_torch_dtype(paths[-1]) == torch.bfloat16
    reader = ShardReader(paths, batch_fmaps=256)
    got = torch.cat([tok.tokenize(b).clone() for _, _, b in reader.batches()])
    assert torch.equal(got, want)
    # fp32 values rounded by write_shard: the same bf16 values
    q = os.path.join(tmp_path, "r.shard")
    write_shard(q, xb.float().numpy(), dtype=torch.bfloat16)
    assert torch.equal(tok.tokenize(ShardReader(q).read_all()), want)


def test_codebook_and_tokenize_pair_on_bf16():
    lr_cb = _cb(trained_like_codebook(1024, (4, 4), 3), (4, 4), 4, 512)
    hr_cb = _cb(trained_like_codebook(16384, (2, 2), 5), (2, 2), 4, 8192)
    xb = _fmaps_bf16(1024, 4, 17)
    assert torch.equal(hr_cb.get_patches_bmu(xb, reshape=True), hr_cb.get_patches_bmu(xb.float(), reshape=True))
    lr_cb16 = _cb(trained_like_codebook(16384, (4, 4), 3), (4, 4), 4, 8192)
    assert torch.equal(lr_cb16.get_patches_bmu(xb), lr_cb16.get_patches_bmu(xb.float()))
    for base in (True, False):
        a = tokenize_pair(lr_cb, hr_cb, xb, base)
        b = tokenize_pair(lr_cb, hr_cb, xb.float(), base)
        for u, v in zip(a, b):
            assert (u is None and v is None) or torch.equal(u, v)
    with pytest.raises(TypeError):
        lr_cb(xb)
    with pytest.raises(TypeError):
        lr_cb.get_quantized_patches(xb)


def test_multi_gpu_bf16_under_torchrun():
    """With at least two GPUs: tests/multi_gpu_bf16_check.py -- DataParallelSom (NCCL and peer tails) on bf16 shares
    equals the fp32 shares of the upcast data with bit-identical replicas; sharded_bmu on bf16 equals fp32."""
    import subprocess
    import sys
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    world = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29743",
                        os.path.join(root, "tests", "multi_gpu_bf16_check.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "MULTI_GPU_BF16_CHECK PASS" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
