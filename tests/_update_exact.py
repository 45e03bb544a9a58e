"""Exact expected values for the update half of the step: the neighbourhood filter on impulse inputs and the
per-unit accumulation on the lattice.

Filter.  The filter treats every feature column on its own.  Column d holds impulses in[j][d] = +-2^k (k in [0, 7],
the sign and k varying per impulse) at rows j = phase_d + m P, with period P = 2h + 1 and zeros elsewhere.  Any window
of 2h + 1 rows holds exactly one impulse, so each output element out[a][d] has at most one non-zero term,
w(|a - j|) * v: none only where that impulse row lies outside the codebook.  The phases spread evenly over the period, so
across the columns the impulse rows cover every position of a 32-row k-block, and every output row (every TMEM lane of
a unit tile) has a term inside the codebook.  v * w is exact for a power of two v.  So the FFMA kernels must return fl32(scale * v w)
and the tensor-core kernels fl32(scale * v (hi + lo)), with hi = tf32_rna(w), lo = tf32_rna(w - hi): hi + lo has at most
24 significant bits, lo(v) = 0, and a sum of one such product with exact zeros never rounds.

Accumulation.  x = a 2^e and W~ = b 2^e with small integers a, b.  Rbar, the counts and the squared error are then
integers times a power of two; while every fp32 partial sum a path forms stays below 2^24 units (`check_accum_bound`,
on the path's own grouping), every path must return them exactly.
"""
import math

import torch

from _lattice import tf32_rna as tf32

BOUND = 1 << 24


# ---- the neighbourhood filter -------------------------------------------------------------------------------------
def two_var(neighbourhood_range):
    """filter_two_var (csrc/som_step_rules.cuh): the double computation, one rounding to fp32"""
    variance = -(neighbourhood_range / (2.0 * math.log(0.1)))
    return torch.tensor(2.0 * variance, dtype=torch.float64).float()


def weights64(neighbourhood_range, n):
    """exp(-fl32(fl32(t^2) / two_var)) for t in [0, n), in fp64 (the argument as band_weight rounds it)"""
    t = torch.arange(n, dtype=torch.int64)
    sq = (t * t).to(torch.float32)
    q = (sq.double() / two_var(neighbourhood_range).double()).float()       # fp32 division, correctly rounded
    return torch.exp(-q.double())


def check_weight_table(w_dev, neighbourhood_range, h):
    """The device weights w[0..n) against fp64: 2 ulp where w is normal, 2 * 2^-149 where it is subnormal (expf's
    bound); w[h] > 0 and w[t] = 0 beyond h."""
    n = w_dev.numel()
    w = w_dev.double().cpu()
    ref = weights64(neighbourhood_range, n)
    inside = torch.arange(n) <= h
    assert bool((w[~inside] == 0).all()), "non-zero weight beyond the band"
    if h < n:
        assert float(w[h]) > 0.0, f"w[h = {h}] is zero"
    tiny = 2.0 ** -126
    ulp = torch.where(ref.abs() >= tiny, torch.ldexp(torch.ones_like(ref), torch.frexp(ref)[1] - 24),
                      torch.full_like(ref, 2.0 ** -149))
    err = (w - ref).abs()[inside]
    assert bool((err <= 2 * ulp[inside]).all()), f"weight error {float((err / ulp[inside]).max()):.2f} ulp"


def impulse_phases(d, h):
    """phase of each column's impulses: the columns spread evenly over one period P = 2h + 1, so that no gap between
    impulse rows exceeds ceil(P / D)"""
    p = 2 * h + 1
    return (torch.arange(d, dtype=torch.int64) * p) // d if d < p else torch.arange(d, dtype=torch.int64) % p


def impulse_case(k, d, h, seed=0):
    """(in (k, d) fp32, src (k, d) int64): the impulse input and, per output element, the row of its one non-zero
    term (-1 where it has none)."""
    p = 2 * h + 1
    phase = impulse_phases(d, h)
    j = torch.arange(k, dtype=torch.int64)[:, None]
    on = (j - phase[None, :]) % p == 0
    g = torch.Generator().manual_seed(seed + 7919 * k + d)
    mag = torch.randint(0, 8, (k, d), generator=g)
    sign = torch.randint(0, 2, (k, d), generator=g) * 2 - 1
    vals = torch.where(on, torch.ldexp(sign.double(), mag.double()), torch.zeros((), dtype=torch.float64)).float()
    # the one impulse row of [a - h, a + h] in column d
    a = torch.arange(k, dtype=torch.int64)[:, None]
    src = a + h - ((a + h - phase[None, :]) % p)
    src = torch.where((src >= 0) & (src < k), src, torch.full_like(src, -1))
    return vals, src


def terms_per_output(vals, src, h):
    """the number of non-zero terms of every output element, counted by brute force (a check of `impulse_case`)"""
    k, d = vals.shape
    nz = (vals != 0).to(torch.int64)
    c = torch.cat([torch.zeros(1, d, dtype=torch.int64), nz.cumsum(0)])
    a = torch.arange(k)
    lo, hi = (a - h).clamp(0, k), (a + h + 1).clamp(0, k)
    return c[hi] - c[lo]


def filter_expected(vals, src, wtab, scale):
    """fl32(scale * v * wtab[|a - j|]) at every element with a term, 0 elsewhere (wtab: fp32 weights per distance,
    the device table for the FFMA kernels, hi + lo for the tensor-core kernels)"""
    k, d = vals.shape
    dev = vals.device
    a = torch.arange(k, device=dev)[:, None]
    has = src >= 0
    j = src.clamp(min=0)
    t = (a - j).abs().clamp(max=wtab.numel() - 1)
    v = torch.gather(vals, 0, j)
    prod = v * wtab[t]                                          # exact: v is a power of two
    out = torch.where(has, prod, torch.zeros((), device=dev))
    return out * torch.tensor(scale, dtype=torch.float32, device=dev)


def tc_weights(w):
    """(hi + lo, subnormal): the weights the tensor-core filter multiplies with, and where hi or lo is subnormal"""
    hi = tf32(w)
    lo = tf32(w - hi)
    s = hi + lo
    assert torch.equal(s.double(), hi.double() + lo.double()), "hi + lo is not an fp32 value"
    tiny = 2.0 ** -126
    sub = ((hi != 0) & (hi.abs() < tiny)) | ((lo != 0) & (lo.abs() < tiny))
    return s, sub


def tc_weights_flushed(w):
    """hi + lo with every subnormal hi or lo operand read as zero"""
    hi = tf32(w)
    lo = tf32(w - hi)
    tiny = 2.0 ** -126
    hi = torch.where(hi.abs() < tiny, torch.zeros_like(hi), hi)
    lo = torch.where(lo.abs() < tiny, torch.zeros_like(lo), lo)
    return hi + lo


def tc_plan_model(k, h, sms, tiles_n):
    """nkb, q, na, ks of the tensor-core filter (csrc/som_filter_tc.cu make_plan) for `tiles_n` feature tiles"""
    nkb = (128 + 2 * h + 31) // 32
    q = (nkb + 3) // 4
    na = (nkb + q - 1) // q
    tiles = (k + 127) // 128 * tiles_n
    return nkb, q, na, (na if tiles * 2 <= sms else 1)


def tc_hits(vals, h, nkb, q):
    """the (unit tile, k-block, chain) triples whose B block holds an impulse of some column: tile ut, k-block kb reads
    the input rows [128 ut + 32 kb - h, 128 ut + 32 kb - h + 32)"""
    k = vals.shape[0]
    rows = torch.nonzero((vals != 0).any(1)).flatten().tolist()
    hit = set()
    n_ut = (k + 127) // 128
    for j in rows:
        jp = j + h                                              # padded inner index
        for ut in range(max(0, (jp - 32 * nkb) // 128), min(n_ut, jp // 128 + 1)):
            kb = (jp - 128 * ut) // 32
            if 0 <= kb < nkb:
                hit.add((ut, kb, kb // q))
    return hit


def tc_all_blocks(k, h, nkb, q):
    """every (unit tile, k-block, chain) whose 32 rows all lie inside the codebook"""
    out = set()
    for ut in range((k + 127) // 128):
        for kb in range(nkb):
            lo = 128 * ut + 32 * kb - h
            if lo >= 0 and lo + 32 <= k:
                out.add((ut, kb, kb // q))
    return out


# ---- the accumulation -------------------------------------------------------------------------------------------
def segment_bmu(n, k, s, seed):
    """BMUs with the segment structure the sorted paths care about, for chunks of s sorted positions: units 0 and k - 1
    empty, a heavy hitter of 9 s + 3 hits starting on a chunk edge, a segment ending on one, one that starts and ends on
    edges, the rest spread at random; patch order scrambled (a unit's patches are not consecutive)."""
    g = torch.Generator().manual_seed(seed)
    counts = torch.zeros(k, dtype=torch.int64)
    fixed = [(1, 9 * s + 3), (2, s - 3), (3, 2 * s)]
    used = 0
    for u, c in fixed:
        if u < k - 1 and used + c <= n:
            counts[u] = c
            used += c
    rest = n - used
    if rest > 0:
        lo = 4 if k > 5 else 1
        hi = max(lo + 1, k - 1)
        counts += torch.bincount(torch.randint(lo, hi, (rest,), generator=g), minlength=k)[:k]
    assert int(counts.sum()) == n
    units = torch.repeat_interleave(torch.arange(k), counts)
    return units[torch.randperm(n, generator=g)]


def accum_reference(a, b, bmu, k):
    """int64 (Rbar residual, Rbar plain, counts, sse) on the integer lattice: r = b[bmu] - a"""
    r = b[bmu] - a
    rbar = torch.zeros(k, a.shape[1], dtype=torch.int64, device=a.device).index_add_(0, bmu, r)
    xbar = torch.zeros(k, a.shape[1], dtype=torch.int64, device=a.device).index_add_(0, bmu, a)
    counts = torch.bincount(bmu, minlength=k)
    return rbar, xbar, counts, int((r * r).sum())


def check_accum_bound(a, b, bmu, k, path, vec, s=None):
    """Assert that every fp32 partial sum of the accumulation path stays below 2^24 units: per segment for Rbar (residual
    and plain), per (unit, 256 vec-feature slice) CTA on the scan path and per (chunk of s sorted positions, 32 vec-feature
    slice) warp on the sorted paths for the squared error.  Returns the largest partial sum."""
    r = b[bmu] - a
    n, d = a.shape
    worst = 0
    for t in (r.abs(), a.abs()):
        seg = torch.zeros(k, d, dtype=torch.int64, device=a.device).index_add_(0, bmu, t)
        worst = max(worst, int(seg.max()) if seg.numel() else 0)
    width = (256 if path == "scan" else 32) * vec
    n_sl = (d + width - 1) // width
    pad = n_sl * width - d
    r2 = torch.nn.functional.pad(r * r, (0, pad)).reshape(n, n_sl, width).sum(2)
    if path == "scan":
        grp = torch.zeros(k, n_sl, dtype=torch.int64, device=a.device).index_add_(0, bmu, r2)
    else:
        order = torch.sort(bmu, stable=True).indices
        chunk = torch.arange(n, device=a.device) // s
        n_ch = (n + s - 1) // s
        grp = torch.zeros(n_ch, n_sl, dtype=torch.int64, device=a.device).index_add_(0, chunk, r2[order])
    worst = max(worst, int(grp.max()) if grp.numel() else 0)
    assert worst < BOUND, f"accumulation partial sum {worst} >= 2^24"
    return worst


def packed_tail(sse, n):
    """pack_tail (csrc/som_step_rules.cuh): [fl32(sse), fl32(sse - hi), n / 4096, n % 4096]"""
    hi = torch.tensor(sse, dtype=torch.float64).float()
    lo = torch.tensor(sse - float(hi), dtype=torch.float64).float()
    return torch.stack([hi, lo, torch.tensor(float(n >> 12)), torch.tensor(float(n & 4095))])
