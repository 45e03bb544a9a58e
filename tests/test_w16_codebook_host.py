"""16-bit codebooks on the host side: the B-side flag of the FP16-split kernel (csrc/som_bmu_tc_l16.cu,
split_w_l16_kernel with W16), emulated in numpy.

For a 16-bit codebook the kernel splits -2 s_c c into FP16 hi + lo exactly as for an fp32 one, and sets one flag per
(256-unit tile, 64-feature block) where some lo is non-zero (NaN counts).  Where a flag is clear every B_lo operand of
that block is exactly zero, so skipping its A_hi x B_lo products leaves every sum unchanged.
  fp16 : -2 s_c c is exact in FP16 for every finite c whenever s_c >= 1 (largest unit norm below 256); it stays exact
         for normal values down to s_c = 1/2, and below that a small element falls off FP16's 2^-24 grid.
  bf16 : an element is exact when its lowest significand bit lands on FP16's 2^-24 grid after the scale, i.e. when it
         lies within about 2^-23 of the codebook's largest |s_c c|; tiny units, subnormals, inf and NaN keep lo."""
import numpy as np
import pytest
import torch

import _lattice as L

F32, F16 = np.float32, np.float16
TN, KBLK = 256, 64


def scales_from_max_norm(w):
    """(s_c, t_c) of scales_from_max_norm from max ||c||^2 (NaN norms dropped, as fmaxf does; an infinite or all-zero
    codebook keeps both at 1)."""
    with np.errstate(over="ignore", invalid="ignore"):
        n2 = (w.astype(np.float64) ** 2).sum(1).astype(F32)
    mn = np.fmax.reduce(n2, initial=F32(0))
    en = int((np.asarray(mn, F32).view(np.uint32) >> 23) & 0xFF)
    e = g = 0
    if mn > 0 and en not in (0, 0xFF):
        e2 = en - 127
        e = max(-60, min(60, 7 - (e2 >> 1)))
        g = max(-60, min(60, 14 - (e2 + e)))
    return F32(2.0 ** e), F32(2.0 ** g)


def f16_split(v):
    """hi = fp16(v), lo = v - hi (fp32), as som_tc_split.cuh's f16_split"""
    with np.errstate(over="ignore", invalid="ignore"):
        hi = v.astype(F16).astype(F32)
        return hi, v - hi


def b_flags(w):
    """(NT, DB) bool: whether unit tile n, feature block fb keeps B_lo.  ``w``: (K, D) float array holding the
    codebook's values.  Rows are padded to whole tiles with copies of unit K - 1 and features with zeros, as the
    pre-split codebook is."""
    w = np.asarray(w, dtype=F32)
    k, d = w.shape
    nt, db = -(-k // TN), -(-d // KBLK)
    wp = np.zeros((nt * TN, db * KBLK), dtype=F32)
    wp[:k, :d] = w
    wp[k:, :d] = w[k - 1]
    sc, _ = scales_from_max_norm(w)
    with np.errstate(over="ignore", invalid="ignore"):
        b = F32(-2.0) * sc * wp
    _, lo = f16_split(b)
    nz = (lo != 0) | np.isnan(lo)
    return nz.reshape(nt, TN, db, KBLK).any(axis=(1, 3))


def kept_share(w):
    """Share of (tile, block) pairs that keep B_lo."""
    return float(b_flags(w).mean())


def _as(dtype, a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=F32)).to(dtype).float().numpy()


def tanh_codebook(k, d, seed, dtype):
    rng = np.random.default_rng(seed)
    return _as(dtype, np.tanh(rng.standard_normal((k, d))))


def flag_setting_codebooks(d):
    """Codebooks whose B flags are set in some (tile, block) pairs and clear in others, as (name, dtype, values, the
    (tile, block) pairs planted to be set).  Tile 1 keeps only values on a coarse grid, so it stays clear."""
    rng = np.random.default_rng(d)
    k = 3 * TN + 17
    out = []
    base = np.round(np.tanh(rng.standard_normal((k, d))) * 64) / 64          # multiples of 2^-6: exact at any scale here
    # fp16, largest norm >= 512 (s_c = 2^-2): odd FP16 subnormals halve off the 2^-24 grid
    w = base.copy()
    w[0, :] = 0
    w[0, 0] = 600.0
    w[2 * TN + 5, 1] = 3 * 2.0 ** -24
    out.append(("fp16_big_norm_tiny_elements", torch.float16, _as(torch.float16, w), {(2, 0)}))
    # bf16: units far below the largest (lowest bit under the 2^-24 grid after s_c = 8), a subnormal, inf and NaN
    w = base.copy()
    last = d - 1
    w[TN * 2 + 3, last] = 129 * 2.0 ** -33
    out.append(("bf16_far_below", torch.bfloat16, _as(torch.bfloat16, w), {(2, last // KBLK)}))
    w = base.copy()
    w[3 * TN + 1, 0] = 3 * 2.0 ** -133                                       # bf16 subnormal
    out.append(("bf16_subnormal", torch.bfloat16, _as(torch.bfloat16, w), {(3, 0)}))
    w = base.copy()
    w[7, 0] = np.inf
    w[2 * TN, min(d - 1, 70)] = np.nan
    out.append(("bf16_inf_nan_units", torch.bfloat16, _as(torch.bfloat16, w), {(0, 0), (2, min(d - 1, 70) // KBLK)}))
    return out


@pytest.mark.parametrize("d", [20, 64, 128, 200, 256])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_tanh_range_codebooks_clear_every_flag(d, dtype):
    w = tanh_codebook(4096 + 37, d, d, dtype)
    assert np.sqrt((w.astype(np.float64) ** 2).sum(1).max()) < 256
    assert not b_flags(w).any()


@pytest.mark.parametrize("d", [64, 200, 256])
def test_flag_setting_codebooks_set_exactly_the_planted_pairs(d):
    for name, _, w, planted in flag_setting_codebooks(d):
        f = b_flags(w)
        got = {(int(n), int(b)) for n, b in zip(*np.nonzero(f))}
        assert planted <= got, f"{name}: planted {planted}, set {got}"
        assert not f[1].any(), f"{name}: the coarse-grid tile must stay clear"


def test_fp16_stays_exact_down_to_half_scale():
    """fp16 values with s_c = 1/2 (largest norm in [256, 512)): -2 s_c c = -c, exact, even for subnormals."""
    w = np.zeros((TN, 64), dtype=F32)
    w[0, 0] = 300.0
    w[1, :] = 3 * 2.0 ** -24
    w = _as(torch.float16, w)
    assert scales_from_max_norm(w)[0] == F32(0.5)
    assert not b_flags(w).any()


@pytest.mark.parametrize("e", L.SCALES)
def test_lattice_codebooks_never_set_a_flag(e):
    """The exact-lattice codebooks (|b| <= 8, one power of two) have lo = 0 everywhere in both formats: on them the
    GPU tests see only the skip; the keep path is covered by the flag-setting codebooks above."""
    _, b = L.lattice_ints(4096, 200, 3000, "narrow", seed=e + 100)
    w = L.to_float(b, e).numpy()
    for dtype in (torch.float16, torch.bfloat16):
        assert np.array_equal(_as(dtype, w), w)
        assert not b_flags(w).any()


def test_flag_clear_means_exactly_zero_lo_operand():
    """Where a flag is clear the FP16-rounded B_lo (what the kernel stores) is zero too."""
    for _, _, w, _ in flag_setting_codebooks(256):
        k, d = w.shape
        sc, _ = scales_from_max_norm(w)
        with np.errstate(over="ignore", invalid="ignore"):
            _, lo = f16_split(F32(-2.0) * sc * w)
            lo16 = lo.astype(F16)
        f = b_flags(w)
        for n in range(f.shape[0]):
            for fb in range(f.shape[1]):
                if not f[n, fb]:
                    blk = lo16[n * TN:(n + 1) * TN, fb * KBLK:(fb + 1) * KBLK]
                    assert not np.any(blk.astype(np.float64)), (n, fb)
