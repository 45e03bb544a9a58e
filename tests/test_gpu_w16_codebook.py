"""16-bit codebooks on the GPU: every result of a fp16 / bf16 codebook equals the fp32 search on weight.float().

On the exact lattice of tests/_lattice.py every regime row of test_gpu_bmu_regimes.py, every variant and every
feature-map dtype must give the lowest-index fp64 argmin and the fp32 module's reduced distance; lattice codebooks
clear every B flag of the FP16-split kernel, so they exercise the skipped B_lo path.  The kept path runs on the
flag-setting codebooks of test_w16_codebook_host.py (their flags asserted set by the host emulation) and must equal
the fp32 search bit for bit, as must tanh-range codebooks (all flags clear).  The module API on 16-bit modules
(search, decoding, pruning, histograms, tokenisers) is checked against the fp32 module holding the same values."""
import copy
import os

import numpy as np
import pytest
import torch

import somcb
from somcb import ops
from somcb.fmap_shards import ShardReader, write_shard
from somcb.host_pipeline import HostTokenizer
from somcb.tokenizer import tokenize_pair
from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
import _lattice as L
from test_gpu_bmu_regimes import ROWS, _assert_plan, _lattice, _row, _variants, plan
from test_w16_codebook_host import b_flags, flag_setting_codebooks, tanh_codebook

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
W16 = (torch.float16, torch.bfloat16)
XS = (torch.float32, torch.float16, torch.bfloat16)
L16_ROWS = [n for n in ROWS if n.startswith("l16_")]


def _same_rd(a, b):
    """Equal values, NaN where the other has NaN."""
    return bool(((a == b) | (a.isnan() & b.isnan())).all())


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _check_equal(x, geom, w16, variant, what, unit_offset=0):
    """ops.bmu with the 16-bit codebook == ops.bmu with its fp32 copy (idx and rd); returns the result."""
    idx, rd = ops.bmu(x, geom, w16, want_rd=True, variant=variant, unit_offset=unit_offset)
    ridx, rrd = ops.bmu(x, geom, w16.float(), want_rd=True, variant=variant, unit_offset=unit_offset)
    assert torch.equal(idx, ridx), f"{what}: {int((idx != ridx).sum())} indices differ from the fp32 codebook"
    assert _same_rd(rd, rrd), f"{what}: rd differs from the fp32 codebook"
    return idx, rd


@pytest.mark.parametrize("name", list(ROWS))
def test_regime_is_exact_on_the_lattice_with_16bit_codebooks(name):
    row = _row(name)
    geom = row.ops_geom()
    _assert_plan(row, plan(row.n, row.d, row.k, row.variant), name)
    x, flat, w = _lattice(row, "narrow", 1 + len(name))
    assert L.zero_unit_share(flat, w, L.fp64_bmu(flat, w)[0]) <= L.MAX_ZERO_SHARE
    ref, ref_rd = L.fp64_bmu(flat, w)
    assert not b_flags(w.cpu().numpy()).any()
    for wd in W16:
        w16 = w.to(wd)
        assert torch.equal(w16.float(), w), "lattice values are exact in both formats"
        assert torch.equal(ops.prepare_codebook(w16), ops.prepare_codebook(w)), f"{name} {wd}: norms"
        for xd in XS:
            for v in _variants(row):
                what = f"{name} x={xd} W={wd} variant {v}"
                idx, rd = _check_equal(x.to(xd), geom, w16, v, what)
                assert torch.equal(idx, ref), f"{what}: {int((idx != ref).sum())} indices differ from the fp64 argmin"
                assert torch.equal(rd.double(), ref_rd), f"{what}: rd differs from the fp64 reduced distance"
    # a 64-bit unit offset, and a 3-way uneven unit-shard split merged == the unsharded answer (bf16 codebook, bf16 x)
    w16, xb = w.to(torch.bfloat16), x.to(torch.bfloat16)
    off = 3 << 31
    assert torch.equal(ops.bmu(xb, geom, w16, unit_offset=off, variant=row.variant), ref + off), f"{name}: unit_offset"
    k = row.k
    cuts = [0, k // 7 + 1, k // 7 + 1 + k // 2, k]
    parts = [ops.bmu(xb, geom, w16[lo:hi].contiguous(), unit_offset=lo, want_rd=True) for lo, hi in zip(cuts, cuts[1:])]
    m_idx, m_rd = ops.merge_candidates(torch.stack([p[1] for p in parts]), torch.stack([p[0] for p in parts]))
    assert torch.equal(m_idx, ref) and torch.equal(m_rd.double(), ref_rd), f"{name}: shard merge"


def _tanh_batch(row):
    """A tanh batch of the row's geometry."""
    g = torch.Generator(device=DEV).manual_seed(row.n)
    return row.batch(torch.tanh(torch.randn(row.n, row.d, generator=g, device=DEV)))


@pytest.mark.parametrize("name", L16_ROWS)
def test_fp16_split_skip_and_keep_paths_equal_the_fp32_codebook(name):
    """Real-valued codebooks on every FP16-split instantiation: tanh-range (every B flag clear: B_lo skipped) and the
    flag-setting codebooks (B_lo kept where the host emulation sets the flag)."""
    row = _row(name)
    geom = row.ops_geom()
    x = _tanh_batch(row)
    cases = [(f"tanh {wd}", wd, tanh_codebook(row.k, row.d, row.k, wd), set()) for wd in W16]
    cases += [(n, wd, w, planted) for n, wd, w, planted in flag_setting_codebooks(row.d)]
    for what, wd, w_np, planted in cases:
        k = w_np.shape[0]
        p = plan(row.n, row.d, k, row.variant)
        if p is None or p["family"] != "L16":
            p = plan(row.n, row.d, k, ops.SOM_BMU_TC_F16)
            variant = ops.SOM_BMU_TC_F16
        else:
            variant = row.variant
        assert p is not None and p["family"] == "L16", f"{name} {what}: {p}"
        f = b_flags(w_np)
        if planted:
            assert {(int(a), int(b)) for a, b in zip(*np.nonzero(f))} >= planted, f"{name} {what}"
        else:                                                   # tanh range: (almost) every pair skips B_lo
            assert f.mean() <= 0.01, f"{name} {what}: flags {np.argwhere(f).tolist()}"
        w16 = torch.from_numpy(w_np).to(wd).to(DEV)
        for xd in XS:
            _check_equal(x.to(xd), geom, w16, variant, f"{name} {what} x={xd}")


def test_special_rows_units_and_empty_batch():
    """NaN and +-inf patch rows and units inside one tile, bf16 subnormal units, and an empty batch."""
    row = _row("l16_pairs_d96")
    geom = row.ops_geom()
    flat = torch.tanh(torch.randn(row.n, row.d, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3)))
    flat[5, 7] = float("nan")
    flat[9, 0] = float("inf")
    flat[11, 3] = float("-inf")
    x = row.batch(flat)
    w = tanh_codebook(row.k, row.d, 4, torch.bfloat16)
    w[300, 2] = np.nan
    w[301, :] = np.inf
    w[302, 5] = -np.inf
    w[303, :8] = 3 * 2.0 ** -133                                 # bf16 subnormals
    for wd in W16:
        w16 = torch.from_numpy(w).to(wd).to(DEV)
        for xd in XS:
            idx, _ = _check_equal(x.to(xd), geom, w16, row.variant, f"special W={wd} x={xd}")
            assert int(idx[5]) == 0, "a NaN patch takes unit 0"
    empty = torch.empty(0, *x.shape[1:], device=DEV)
    for wd in W16:
        w16 = torch.from_numpy(w).to(wd).to(DEV)
        for xd in XS:
            out = ops.bmu(empty.to(xd), ops.geometry(empty.shape, (row.geom[2], row.geom[3])), w16)
            assert out.numel() == 0 and out.dtype == torch.int64


def _modules(k, pd, wd, seed):
    cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4, num_embeddings=k,
                        init_neighbour_range=k // 2)
    with torch.no_grad():
        cb.codebook.weight.copy_(trained_like_codebook(k, pd, seed))
    cb16 = copy.deepcopy(cb).to(DEV).to(wd)
    ref = copy.deepcopy(cb).to(DEV)
    with torch.no_grad():
        ref.codebook.weight.copy_(cb16.codebook.weight.float())
    return cb16, ref


@pytest.mark.parametrize("wd", W16)
def test_module_api_on_16bit_modules(wd):
    pd, k = (4, 4), 4096
    cb16, ref = _modules(k, pd, wd, 7)
    x = synthetic_fmaps(640, 5).to(DEV)                           # 40 960 patches of D = 64: the FP16-split kernel
    for xd in XS:
        xx = x.to(xd)
        idx = cb16.get_patches_bmu(xx, reshape=True)
        assert torch.equal(idx, ref.get_patches_bmu(xx, reshape=True)), f"get_patches_bmu x={xd}"
    idx = cb16.get_patches_bmu(x, reshape=True)
    w = cb16.codebook.weight.detach()
    img = cb16.get_quantized_image(idx)
    want = L.unpatchify(w[idx.reshape(-1)], 4, 4, 4, 8, 8)
    assert img.dtype == wd and not img.requires_grad and torch.equal(_bits(img), _bits(want))
    seq = cb16.get_quantized_image(idx, unpatchify_input=False)
    assert seq.dtype == wd and torch.equal(_bits(seq), _bits(w[idx.reshape(-1)].reshape(idx.shape[0], -1, 64)))
    assert torch.equal(img.float(), ref.get_quantized_image(idx).detach())
    counts = somcb.bmu_histogram(cb16, [x[:320], x[320:].to(torch.bfloat16)])
    assert torch.equal(counts, somcb.bmu_histogram(ref, [x[:320], x[320:].to(torch.bfloat16)]))
    new, keep, ck = somcb.prune_codebook(cb16, counts, 2)
    new_r, keep_r, ck_r = somcb.prune_codebook(ref, counts, 2)
    assert torch.equal(keep, keep_r) and 0 < keep.numel() < k
    assert new.codebook.weight.dtype == wd and torch.equal(_bits(new.codebook.weight.detach()), _bits(w[keep]))
    assert set(ck) == set(ck_r) and list(ck["checkpoint"]) == ["codebook.weight"]
    assert ck["checkpoint"]["codebook.weight"].dtype == wd
    assert torch.equal(ck["checkpoint"]["codebook.weight"].float(), ck_r["checkpoint"]["codebook.weight"])
    assert {kk: v for kk, v in ck.items() if kk != "checkpoint"} == {kk: v for kk, v in ck_r.items() if kk != "checkpoint"}
    with pytest.raises(TypeError, match="float32 weights"):
        cb16(x)
    with pytest.raises(TypeError, match="float32 weights"):
        cb16.get_quantized_patches(x)
    with pytest.raises(TypeError):
        somcb.SomTrainer(cb16, lr=1e-4, neighbourhood_step=3).step(x)
    with pytest.raises(ValueError):
        ops.bmu(x, ops.geometry(x.shape, pd), w, stage=torch.empty(40960, 64, device=DEV))


def test_tokenize_pair_and_host_tokenizer_over_a_bf16_shard(tmp_path):
    lr16, lr = _modules(1024, (4, 4), torch.float16, 3)
    hr16, hr = _modules(16384, (2, 2), torch.bfloat16, 5)
    xb = synthetic_fmaps(1024, 17).bfloat16().to(DEV)
    for base in (True, False):
        a = tokenize_pair(lr16, hr16, xb, base)
        b = tokenize_pair(lr, hr, xb, base)
        for u, v in zip(a, b):
            assert (u is None and v is None) or torch.equal(u, v)
    host = xb[:600].cpu()
    want = hr.get_patches_bmu(host.to(DEV), reshape=True).cpu()
    path = os.path.join(tmp_path, "s.shard")
    write_shard(path, host, dtype=torch.bfloat16)
    tok = HostTokenizer(hr16, chunk_fmaps=256)
    got = torch.cat([tok.tokenize(bt).clone() for _, _, bt in ShardReader(path, batch_fmaps=256).batches()])
    assert torch.equal(got, want)
