"""CPU proof of the exact-lattice premise (tests/_lattice.py) before any GPU time is spent: on lattice inputs the three
operand splits of the tensor-core BMU kernels -- 3xTF32 (som_bmu_tc_l.cu / config S TF32), config-S FP16
(som_bmu_tc_s.cu) and the FP16-split kernel (som_bmu_tc_l16.cu) -- form exactly the fp64 reduced distance for every
(patch, unit) pair, so any kernel that returns something else is wrong, with no tolerance to hide it."""
import numpy as np
import pytest
import torch

import _lattice as L
from oracle import patchify
from test_f16_input_host import _codebook_scales, _row_scale
from test_fp16_split_scheme import fp16_split_rd

CASES = [(3, "narrow"), (16, "narrow"), (20, "narrow"), (48, "wide"), (64, "wide"), (200, "narrow"), (200, "wide"),
         (256, "wide")]


def _case(d, kind, e, n=300, k=700, seed=0):
    a, b = L.lattice_ints(n, d, k, kind, seed=seed + d)
    L.check_bound(a, b)
    return a, b, L.to_float(a, e), L.to_float(b, e)


def _rd64(x, w):
    return torch.cat([rd for _, rd in L.fp64_rd(x, w)])


def _tf32_rna(v):
    """cvt.rna.tf32.f32: round to 10 stored mantissa bits, ties away from zero (fp32 in, fp32 out)"""
    u = v.contiguous().view(torch.int32)
    return ((u + 0x1000) & ~0x1FFF).view(torch.float32)


def _3xtf32_terms(x, w):
    """The products and the norm tail that the 3xTF32 kernels sum, and the dropped lo . lo product (fp64)."""
    cn = (w * w).sum(1)                                         # prepare_codebook (exact on a lattice)
    xh = _tf32_rna(x)
    xl = _tf32_rna(x - xh)
    wh = _tf32_rna(w)
    wl = _tf32_rna(w - wh)
    n1 = _tf32_rna(cn)
    n2 = _tf32_rna(cn - n1)
    n3 = _tf32_rna(cn - n1 - n2)
    f = torch.float64
    prods = (xh.to(f) @ (-2 * wh).to(f).T, xl.to(f) @ (-2 * wh).to(f).T, xh.to(f) @ (-2 * wl).to(f).T)
    tail = (n1.to(f) + n2.to(f) + n3.to(f))[None, :]
    return prods, tail, xl.to(f) @ (-2 * wl).to(f).T, (xh, xl, wh, wl)


@pytest.mark.parametrize("e", L.SCALES)
@pytest.mark.parametrize("d,kind", CASES)
def test_3xtf32_split_is_exact_on_the_lattice(d, kind, e):
    _, _, x, w = _case(d, kind, e)
    prods, tail, dropped, (xh, xl, wh, wl) = _3xtf32_terms(x, w)
    assert bool((wl == 0).all()) and bool((dropped == 0).all())
    assert bool((xl != 0).any()) == (kind == "wide")
    rd = tail + prods[0] + prods[1] + prods[2]
    assert torch.equal(rd, _rd64(x, w))
    # the same sum in an fp32 accumulator, feature by feature (one order of many the kernels use): still exact
    acc = tail.float().expand(x.shape[0], -1).clone()
    for j in range(d):
        for xa, wb in ((xh, wh), (xl, wh), (xh, wl)):
            acc += xa[:, j:j + 1] * (-2 * wb[:, j])[None, :]
    assert torch.equal(acc.double(), rd)


@pytest.mark.parametrize("e", L.SCALES)
@pytest.mark.parametrize("kind", ["narrow", "wide"])
def test_config_s_fp16_split_is_exact_on_the_lattice(kind, e):
    """s_c, t_c and the per-patch scale of config S (test_fp16_split_scheme.fp16_split_rd) at D = 16."""
    _, _, x, w = _case(16, kind, e)
    acc, factor = fp16_split_rd(x, w)
    assert torch.equal(acc / factor[:, None], _rd64(x, w))


def _l16_rd(x, w):
    """rd as the FP16-split kernel forms and un-scales it: row scale s_p with its clamps, codebook scales s_c / t_c,
    hi / lo of s_p x and -2 s_c c in FP16, the three-half norm tail a_p (n1 + n2 + n3); products summed in fp64."""
    xv, wv = x.numpy(), w.numpy()
    sc, tc_exp = _codebook_scales(wv)
    sp = _row_scale(xv, tc_exp)
    es = np.log2(sp).astype(np.int64)
    ka = es - tc_exp
    far = ka < -24                                             # (the row scale keeps es = ep there: a_p = 0)
    ka = np.minimum(ka, 15)
    ap = np.where(far, 0.0, np.ldexp(1.0, ka))
    assert np.array_equal(ap.astype(np.float16).astype(np.float64), ap)
    s = xv * sp[:, None]
    h = s.astype(np.float16)
    lo = (s - h.astype(np.float32)).astype(np.float16)
    assert np.array_equal(lo.astype(np.float32), s - h.astype(np.float32)), "lo(s_p x) is not exact in FP16"
    bb = np.float32(-2) * sc * wv
    bh = bb.astype(np.float16)
    bl = (bb - bh.astype(np.float32)).astype(np.float16)
    cn = (wv * wv).sum(1, dtype=np.float32)
    nrm = cn * sc * np.float32(2.0 ** tc_exp)
    n1 = nrm.astype(np.float16).astype(np.float32)
    n2 = (nrm - n1).astype(np.float16).astype(np.float32)
    n3 = (nrm - n1 - n2).astype(np.float16)
    assert np.array_equal(n3.astype(np.float32), nrm - n1 - n2), "the norm tail is not exact in three halves"
    f = np.float64
    acc = (ap[:, None] * (n1.astype(f) + n2.astype(f) + n3.astype(f))[None, :]
           + h.astype(f) @ bh.astype(f).T + lo.astype(f) @ bh.astype(f).T + h.astype(f) @ bl.astype(f).T)
    sc_exp = int(np.log2(sc))
    return torch.from_numpy(np.ldexp(acc, -(es + sc_exp)[:, None])), bool((lo != 0).any()), bool((bl != 0).any())


@pytest.mark.parametrize("e", L.SCALES)
@pytest.mark.parametrize("d,kind", [c for c in CASES if c[0] > 16])
def test_l16_fp16_split_is_exact_on_the_lattice(d, kind, e):
    _, _, x, w = _case(d, kind, e)
    rd, x_lo, c_lo = _l16_rd(x, w)
    assert not c_lo, "a codebook lo part is non-zero: the dropped lo . lo product would not be 0"
    assert x_lo == (kind == "wide")
    assert torch.equal(rd, _rd64(x, w))


@pytest.mark.parametrize("d", [3, 64, 1102, 4096, 8192])
def test_narrow_lattice_bound_and_bit_widths(d):
    a, b = L.lattice_ints(64, d, 300, "narrow", seed=d)
    assert L.check_bound(a, b) < L.BOUND
    assert int(a.abs().max()) <= 8 and int(b.abs().max()) <= 8
    for e in L.SCALES:
        x = L.to_float(a, e)
        for dt in (torch.float16, torch.bfloat16):
            assert torch.equal(x.to(dt).float(), x), f"narrow x not exact in {dt} at e = {e}"


@pytest.mark.parametrize("d", [20, 64, 200, 512, 4096, 8192])
def test_wide_lattice_bound_and_bit_widths(d):
    a, b = L.lattice_ints(256, d, 300, "wide", seed=d)
    assert L.check_bound(a, b) < L.BOUND
    assert int(b.abs().max()) <= 8
    big = a.abs().amax(1)
    assert int(big.max()) < L.WIDE_HI
    assert int((big >= L.WIDE_LO).sum()) >= 3 * 256 // 4 - 3          # less the planted zero patches
    x = L.to_float(a, 0)
    assert bool((x - _tf32_rna(x) != 0).any()), "no wide entry has a TF32 lo part"


def test_bound_check_rejects_what_it_should():
    a = torch.full((4, 300), 8191, dtype=torch.int64)
    b = torch.full((5, 300), 8, dtype=torch.int64)
    with pytest.raises(AssertionError):
        L.check_bound(a, b)


def test_planted_ties_are_exact_ties_and_the_reference_takes_the_lowest_index():
    d, k = 20, 700
    a, b = L.lattice_ints(300, d, k, "narrow", seed=1)
    x, w = L.to_float(a, 0), L.to_float(b, 0)
    rd = _rd64(x, w)
    idx, best = L.fp64_bmu(x, w)
    ties = (rd == best[:, None]).sum(1)
    assert int((ties >= 2).sum()) >= 5, "too few exact ties"
    first = torch.argmax((rd == best[:, None]).int(), dim=1)
    assert torch.equal(idx, first)
    zero_units = torch.nonzero((b == 0).all(1)).flatten()
    assert zero_units.numel() >= 2
    for p in (0, 150, 299):
        assert int(idx[p]) == int(zero_units[0]) and float(best[p]) == 0.0
    # a mirror pair: two different rows at exactly the same distance from a patch
    mirrors = 0
    for p in range(300):
        tied = torch.nonzero(rd[p] == best[p]).flatten()
        rows = {tuple(b[u].tolist()) for u in tied.tolist()}
        mirrors += len(rows) >= 2
    assert mirrors >= 1


@pytest.mark.parametrize("d,k", [(16, 4096), (48, 700), (128, 4096), (256, 1024), (1102, 777), (8192, 300), (512, 7)])
def test_narrow_lattice_answers_depend_on_the_data(d, k):
    """The argmin of a non-zero patch must come from the distance arithmetic, not from the planted all-zero units
    (rd = 0): with independent random rows it would be a zero unit for nearly every patch from D ~ 64 on."""
    a, b = L.lattice_ints(512, d, k, "narrow", seed=d + k)
    idx, best = L.fp64_bmu(L.to_float(a, 0), L.to_float(b, 0))
    assert L.zero_unit_share(a, b, idx) <= L.MAX_ZERO_SHARE
    nz = (a != 0).any(1)
    assert float((best[nz] < 0).float().mean()) > 0.9
    # independent random rows: the degenerate case this guards against
    g = torch.Generator().manual_seed(d)
    ar, br = torch.randint(-8, 9, (512, d), generator=g), torch.randint(-8, 9, (k, d), generator=g)
    br[5] = 0
    idx_r, _ = L.fp64_bmu(L.to_float(ar, 0), L.to_float(br, 0))
    if d >= 128:
        assert L.zero_unit_share(ar, br, idx_r) > 0.5


@pytest.mark.parametrize("c,ph,pw,gh,gw", [(5, 2, 2, 4, 4), (16, 4, 3, 4, 8), (24, 4, 1, 8, 32), (40, 4, 2, 2, 3)])
def test_unpatchify_inverts_patchify(c, ph, pw, gh, gw):
    rows = torch.arange(3 * gh * gw * c * ph * pw, dtype=torch.float32).reshape(3 * gh * gw, c * ph * pw)
    x = L.unpatchify(rows, c, ph, pw, gh, gw)
    assert torch.equal(patchify(x, (ph, pw)).reshape(rows.shape), rows)
