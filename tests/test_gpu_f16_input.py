"""fp16 feature maps on the GPU: every result must be BIT-identical to the fp32 path on x.half().float() -- the native
FP16-split kernel (which skips the A_lo x B_hi products of tiles whose lo operands are all zero), the upcast route of
every other kernel, the trainers, the host pipeline and the drop-in Codebook.  The equalities rest on a tcgen05.mma
whose A operand is all zero leaving the fp32 accumulator unchanged."""
import os

import numpy as np
import pytest
import torch

import somcb
from somcb import ops
from somcb.fmap_shards import ShardReader, write_shard
from somcb.host_pipeline import HostTokenizer, HostTrainer
from somcb.tokenizer import tokenize_pair
from oracle.step_oracle import make_oracle_codebook, make_reference_optimizer, reference_step, synthetic_fmaps
from oracle.step_oracle import trained_like_codebook
from _helpers import assert_bmu_parity, assert_close_norm, flat_patches

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _fmaps16(n, c, seed, hw=32):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.tanh(torch.randn(n, c, hw, hw, device=DEV, generator=g)).half()


def _codebook(k, d, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (0.7 * torch.tanh(torch.randn(k, d, device=DEV, generator=g))).contiguous()


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_same_search(x16, geom, w, variant=ops.SOM_BMU_AUTO, unit_offset=0, stage=None):
    """ops.bmu on the fp16 batch and on its upcast: idx, rd (and the staging rows) bit for bit."""
    d, k = ops.dim_of(geom), w.shape[0]
    npat = ops.n_patches_of(geom)
    x32 = x16.float()
    if stage is None:
        stage = ops.bmu_can_stage(geom, k, variant)
    s16 = torch.full((npat, d), float("nan"), device=DEV) if stage else None
    s32 = torch.full((npat, d), float("nan"), device=DEV) if stage else None
    i16, r16 = ops.bmu(x16, geom, w, unit_offset=unit_offset, want_rd=True, variant=variant, stage=s16)
    i32, r32 = ops.bmu(x32, geom, w, unit_offset=unit_offset, want_rd=True, variant=variant, stage=s32)
    assert torch.equal(i16, i32), f"{int((i16 != i32).sum())} of {npat} indices differ"
    assert torch.equal(_bits(r16), _bits(r32)), "reduced distances differ"
    if stage:
        assert torch.equal(_bits(s16), _bits(s32)), "staging rows differ"
        from oracle import patchify
        want = patchify(x32.cpu().reshape(geom[:4]), (geom[4], geom[5])).reshape(npat, d)
        assert torch.equal(_bits(s16.cpu()), _bits(want)), "staging rows are not patchify(x.float())"
    return i16


# (C, patch, fmaps, K, variant): D = C * pH * pW; 128-patch tiles against the 148 SMs decide CTA pairs
NATIVE = [
    (4, (4, 2), 320, 1024, ops.SOM_BMU_AUTO, 0),             # D = 32, pW = 2 loads, CTA pairs, merged
    (3, (4, 4), 320, 32768, ops.SOM_BMU_AUTO, 0),            # D = 48 (partial k-steps), single CTAs, merged
    (4, (4, 4), 320, 16384, ops.SOM_BMU_AUTO, 0),            # D = 64 (C4), single CTAs, merged
    (4, (4, 4), 1024, 16384, ops.SOM_BMU_AUTO, 4096),        # D = 64, CTA pairs, unit_offset
    (8, (4, 4), 640, 16384, ops.SOM_BMU_AUTO, 0),            # D = 128, CTA pairs, merged
    (4, (8, 8), 2560, 32768, ops.SOM_BMU_AUTO, 0),           # D = 256 (C5), CTA pairs, separate rings
    (4, (4, 4), 16, 1024, ops.SOM_BMU_TC_F16, 0),            # forced at a small batch, single CTA
    (4, (8, 8), 32, 1024, ops.SOM_BMU_TC_F16, 7),            # forced, D = 256
]


@pytest.mark.parametrize("c,pd,n,k,variant,off", NATIVE)
def test_native_fp16_kernel_equals_fp32_on_upcast(c, pd, n, k, variant, off):
    x16 = _fmaps16(n, c, 1 + n)
    geom = ops.geometry(x16.shape, pd)
    w = _codebook(k, ops.dim_of(geom), 2)
    assert ops.bmu_f16_native(geom, k, variant)
    _assert_same_search(x16, geom, w, variant, unit_offset=off)


def _special_rows(d):
    rng = np.random.default_rng(3)
    rows = [np.tanh(rng.standard_normal(d))]
    for mag in (1e-6, 1e-3, 1.0, 100.0, 127.9, 128.0, 1e3, 6e4):
        rows.append(rng.uniform(-mag, mag, d))
    rows.append(np.float16(2.0 ** -24) * rng.integers(-1023, 1024, d))
    rows.append(np.where(rng.random(d) < 0.5, 65504.0, -65504.0))
    wide = rng.uniform(-1, 1, d)
    wide[0], wide[1] = 6e4, 2.0 ** -24
    rows.append(wide)
    rows.append(np.zeros(d))
    for col, val in ((5, np.nan), (7, np.inf), (9, -np.inf)):
        r = np.tanh(rng.standard_normal(d))
        r[col] = val
        rows.append(r)
    return torch.from_numpy(np.stack(rows).astype(np.float16))


@pytest.mark.parametrize("n_rows,variant", [(4096, ops.SOM_BMU_TC_F16), (20480, ops.SOM_BMU_AUTO)])
def test_fallback_rows_inside_one_tile(n_rows, variant):
    d, k = 64, 1024
    special = _special_rows(d)
    x = flat_patches(synthetic_fmaps(n_rows // 64, 5), (4, 4)).half()
    x[130:130 + special.shape[0]] = special                          # all in the second tile
    w = trained_like_codebook(k, (4, 4), 7)
    geom = ops.flat_geometry(n_rows, d)
    x16, wd = x.to(DEV).contiguous(), w.to(DEV)
    assert ops.bmu_f16_native(geom, k, variant)
    idx = _assert_same_search(x16, geom, wd, variant).cpu()
    nan_row = 130 + 13
    assert int(idx[nan_row]) == 0, "a patch holding a NaN gets unit 0"
    finite = torch.isfinite(x.float()).all(1)
    flat = x.float()[finite]
    w64 = w.double()
    ref = ((w64 * w64).sum(1)[None, :] - 2 * flat.double() @ w64.T).argmin(1)
    assert_bmu_parity(idx[finite], ref, flat, w)


UPCAST = [
    (4, (2, 2), 256, 4096, ops.SOM_BMU_TC_TF32),             # D = 16, config S, 3xTF32, 65 536 patches
    (4, (2, 2), 256, 4096, ops.SOM_BMU_TC_F16),              # D = 16, config S, FP16 split
    (4, (2, 2), 256, 4096, ops.SOM_BMU_AUTO),
    (4, (4, 4), 8, 1024, ops.SOM_BMU_AUTO),                  # C1
    (4, (32, 32), 64, 512, ops.SOM_BMU_AUTO),                # C3: D = 4096
    (4, (4, 4), 64, 1000, ops.SOM_BMU_FFMA),
    (4, (4, 4), 1024, 16384, ops.SOM_BMU_TC_TF32),           # an l16 shape with 3xTF32 forced
]


@pytest.mark.parametrize("c,pd,n,k,variant", UPCAST)
def test_upcast_route_equals_fp32_on_upcast(c, pd, n, k, variant):
    x16 = _fmaps16(n, c, 3 + n)
    geom = ops.geometry(x16.shape, pd)
    w = _codebook(k, ops.dim_of(geom), 4)
    assert not ops.bmu_f16_native(geom, k, variant)
    _assert_same_search(x16, geom, w, variant, stage=False)


def test_upcast_kernel_is_exact_and_handles_unaligned_tails():
    bits = torch.arange(0, 65536, dtype=torch.int32).to(torch.int16).to(DEV)
    h = bits.view(torch.float16)
    want = h.float()

    def same(a, b):                                                   # every value bit for bit, NaN as NaN
        nan = torch.isnan(b)
        return torch.equal(torch.isnan(a), nan) and torch.equal(_bits(a)[~nan], _bits(b)[~nan])

    for lo, hi in ((0, 65536), (1, 65536), (3, 65533), (8, 17)):
        assert same(ops.upcast_f16(h[lo:hi].contiguous()), want[lo:hi])
        out = torch.empty(hi - lo + 1, device=DEV)[1:]               # 4-byte but not 16-byte aligned output
        ops.upcast_f16(h[lo:hi].contiguous(), out=out)
        assert same(out, want[lo:hi])


def _cb(w, pd, channels, rng, variant=ops.SOM_BMU_AUTO):
    cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=channels, num_embeddings=w.shape[0],
                        init_neighbour_range=rng)
    with torch.no_grad():
        cb.codebook.weight.copy_(w)
    cb = cb.to(DEV)
    cb.bmu_variant = variant
    return cb


@pytest.mark.parametrize("n,k,graph", [(1024, 16384, False), (1024, 16384, True), (1024, 16384, "alias"),
                                       (8, 1024, False), (8, 1024, "alias")])
def test_trainer_fp16_steps_equal_fp32_on_upcast(n, k, graph):
    pd = (4, 4)
    w0 = trained_like_codebook(k, pd, 7)
    batches = [_fmaps16(n, 4, 50 + s) for s in range(5)]
    out = []
    for half in (True, False):
        cb = _cb(w0, pd, 4, k // 2)
        tr = somcb.SomTrainer(cb, lr=1e-4, neighbourhood_step=3, use_cuda_graph=graph)
        losses = []
        for xb in batches:
            x = xb if half else xb.float()
            losses.append(tr.step(x).clone())
        torch.cuda.synchronize()
        out.append((cb.codebook.weight.detach().clone(), torch.stack(losses), tr.last_bmu))
    (w16, l16, _), (w32, l32, _) = out
    assert torch.equal(_bits(w16), _bits(w32)), "weights differ after 5 steps"
    assert torch.equal(l16.view(torch.int64), l32.view(torch.int64)), "losses differ"


def test_c1_fp16_run_matches_the_oracle_on_upcast_inputs():
    pd, k, lr = (4, 4), 1024, 1e-4
    w0 = trained_like_codebook(k, pd, 7)
    ocb = make_oracle_codebook(w0, pd, (32, 32), 4, k // 2)
    opt = make_reference_optimizer(ocb, lr)
    cb = _cb(w0, pd, 4, k // 2)
    tr = somcb.SomTrainer(cb, lr=lr, neighbourhood_step=10 ** 6)
    for step in range(20):
        x16 = synthetic_fmaps(8, 123 + step).half()
        ref = float(reference_step(ocb, opt, x16.float()))
        got = float(tr.step(x16.to(DEV)))
        assert abs(got - ref) <= 1e-5 * abs(ref), f"loss at step {step}"
    assert_close_norm(cb.codebook.weight.detach().cpu(), ocb.codebook.weight.detach(), 1e-5, "weights@20")


def test_host_trainer_with_fp16_pinned_batches_equals_resident_run():
    pd, k = (4, 4), 16384
    w0 = trained_like_codebook(k, pd, 7)
    host = [synthetic_fmaps(512, 70 + s).half().pin_memory() for s in range(4)]      # 32 768 patches: native
    cb_h = _cb(w0, pd, 4, k // 2)
    ht = HostTrainer(somcb.SomTrainer(cb_h, lr=1e-4, neighbourhood_step=3, use_cuda_graph="alias"))
    lh = [ht.step(b).item() for b in host]
    cb_r = _cb(w0, pd, 4, k // 2)
    tr = somcb.SomTrainer(cb_r, lr=1e-4, neighbourhood_step=3, use_cuda_graph="alias")
    resident = [b.float().to(DEV) for b in host]
    lr_ = [float(tr.step(x)) for x in resident]
    assert lh == lr_
    assert torch.equal(_bits(cb_h.codebook.weight.detach()), _bits(cb_r.codebook.weight.detach()))
    assert ht._slots[1][0]["x"].dtype == torch.float16


def test_host_tokenizer_and_fp16_shards_equal_resident_search(tmp_path):
    pd, k = (2, 2), 4096
    cb = _cb(trained_like_codebook(k, pd, 7), pd, 4, k // 2)
    x16 = synthetic_fmaps(600, 9).half()
    want = cb.get_patches_bmu(x16.float().to(DEV), reshape=True).cpu()
    tok = HostTokenizer(cb, chunk_fmaps=256)
    assert torch.equal(tok.tokenize(x16.pin_memory()), want)
    paths = []
    for i, (lo, hi) in enumerate(((0, 250), (250, 600))):
        paths.append(os.path.join(tmp_path, f"s{i}.shard"))
        write_shard(paths[-1], x16[lo:hi].numpy(), dtype=np.float16)
    reader = ShardReader(paths, batch_fmaps=256)
    got = torch.cat([tok.tokenize(b).clone() for _, _, b in reader.batches()])
    assert torch.equal(got, want)


def test_codebook_and_tokenize_pair_on_fp16():
    lr_cb = _cb(trained_like_codebook(1024, (4, 4), 3), (4, 4), 4, 512)
    hr_cb = _cb(trained_like_codebook(16384, (2, 2), 5), (2, 2), 4, 8192)
    x16 = _fmaps16(1024, 4, 17)
    assert torch.equal(hr_cb.get_patches_bmu(x16, reshape=True), hr_cb.get_patches_bmu(x16.float(), reshape=True))
    lr_cb16 = _cb(trained_like_codebook(16384, (4, 4), 3), (4, 4), 4, 8192)
    assert torch.equal(lr_cb16.get_patches_bmu(x16), lr_cb16.get_patches_bmu(x16.float()))
    for base in (True, False):
        a = tokenize_pair(lr_cb, hr_cb, x16, base)
        b = tokenize_pair(lr_cb, hr_cb, x16.float(), base)
        for u, v in zip(a, b):
            assert (u is None and v is None) or torch.equal(u, v)
    with pytest.raises(TypeError):
        lr_cb(x16)
    with pytest.raises(TypeError):
        lr_cb.get_quantized_patches(x16)


def test_multi_gpu_fp16_under_torchrun():
    """With at least two GPUs: tests/multi_gpu_f16_check.py -- DataParallelSom (NCCL and peer tails) on fp16 shares
    equals the fp32 shares of the upcast data with bit-identical replicas; sharded_bmu on fp16 equals unsharded."""
    import subprocess
    import sys
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least two GPUs")
    world = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                        "--master-addr", "127.0.0.1", "--master-port", "29741",
                        os.path.join(root, "tests", "multi_gpu_f16_check.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "MULTI_GPU_F16_CHECK PASS" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
