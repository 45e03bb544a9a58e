"""Exact expected values for the optimizer half of the training step: a correctly rounded CPU emulation of the rules of
csrc/som_step_rules.cuh (Adam, the packed tail) in torch fp64, vectorised.

The library is built without fast math or flush-to-zero, so every rule is a fixed sequence of IEEE fp32 operations plus
two fp64 `pow` calls, and the kernels' bits are fully determined by it:

* a + b, a - b, a * b, a / b and sqrt(a) of fp32 operands: evaluated in fp64 and rounded once more to fp32.  Rounding
  twice is innocuous for these five operations because 53 >= 2 * 24 + 2.
* fma(a, b, c): a * b is exact in fp64, but the fp64 sum a * b + c can land exactly on the midpoint between two fp32
  values while the exact sum does not, and the second rounding then goes the wrong way (`FMA_TRAP` is such a case).  So
  the sum is formed with its TwoSum error e, rounded to fp32, and moved to the other neighbour only when the fp64 sum is
  such a midpoint and e points to that neighbour's side.  This also holds at subnormal spacing and at the overflow
  threshold, where 2^128 stands in for the neighbour above the largest float.
* `adam_scalars`: the same double expressions as the header, then narrowed.  The device evaluates `pow` in three of the
  four Adam entry points and CUDA's double `pow` is only within 2 ulp, so every (lr, betas, t) the GPU tests use must
  narrow to the same fp32 scalars whatever `pow` returns within 4 ulp (`scalar_margin`, asserted on the CPU for every row
  in `gpu_scalar_rows`).

Powers of two are built by multiplication, never with torch.ldexp (1 ulp off on CUDA tensors for negative exponents).
"""
import math
from dataclasses import dataclass

import torch

F32, F64 = torch.float32, torch.float64
TWO128 = 2.0 ** 128
POW_ULPS = 4                   # the device pow's 2 ulp, doubled
MIN_MARGIN = 2.0 ** 10         # fp64 ulps between a scalar and the nearest fp32 rounding boundary

# a = 1 + 2^-23, b = 2^-24 (1 - 2^-23), c = a: fl64(a b + c) = 1 + 3 * 2^-24 is an fp32 midpoint, the exact sum lies just
# below it, so the correct fp32 FMA is 0x1.000002p+0 while fl32(fl64(a b + c)) is 0x1.000004p+0
FMA_TRAP = (1.0 + 2.0 ** -23, 2.0 ** -24 * (1.0 - 2.0 ** -23), 1.0 + 2.0 ** -23)


# ---- fp32 operations ------------------------------------------------------------------------------------------------
def _d(x):
    return torch.as_tensor(x, dtype=F32).to(F64)


def _r(x):
    return x.to(F32)


def fadd(a, b):
    return _r(_d(a) + _d(b))


def fsub(a, b):
    return _r(_d(a) - _d(b))


def fmul(a, b):
    return _r(_d(a) * _d(b))


def fdiv(a, b):
    return _r(_d(a) / _d(b))


def fsqrt(a):
    return _r(torch.sqrt(_d(a)))


def _value(x32):
    """an fp32 tensor as fp64, with +-2^128 in place of +-inf (the 'next float' past the largest one)"""
    return torch.where(torch.isinf(x32), torch.copysign(torch.full_like(x32, TWO128, dtype=F64), x32.to(F64)),
                       x32.to(F64))


def fma(a, b, c):
    """fp32 fma(a, b, c), correctly rounded (one rounding of the exact a * b + c)"""
    p = _d(a) * _d(b)                              # exact: 24 + 24 bits, far inside fp64's exponent range
    c = _d(c)
    p, c = torch.broadcast_tensors(p, c)
    s = p + c
    bb = s - p                                     # TwoSum: s + e == p + c exactly
    e = (p - (s - bb)) + (c - bb)
    r = _r(s)
    rd = _value(r)
    fin = torch.isfinite(s)
    other = torch.nextafter(r, torch.where(rd < s, torch.tensor(math.inf), torch.tensor(-math.inf)).to(F32))
    od = _value(other)
    mid = fin & ((rd + od) * 0.5 == s)
    fix = mid & (e != 0) & ((od - rd) * e > 0)
    return torch.where(fix, other, r)


# ---- Adam -----------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class AdamScalars:
    w1: float
    b2: float
    one_m_b2: float
    step_size: float
    bc2_sqrt: float
    eps: float


def _f32(x):
    return float(torch.tensor(x, dtype=F64).to(F32))


def scalars64(lr, b1, b2, t, pow_fn=math.pow):
    """the two fp64 values adam_scalars narrows: lr / (1 - b1^t), sqrt(1 - b2^t)"""
    return lr / (1.0 - pow_fn(b1, t)), math.sqrt(1.0 - pow_fn(b2, t))


def adam_scalars(lr, b1, b2, eps, t):
    step_size, bc2_sqrt = scalars64(lr, b1, b2, float(t))
    return AdamScalars(_f32(1.0 - b1), _f32(b2), _f32(1.0 - b2), _f32(step_size), _f32(bc2_sqrt), _f32(eps))


def adam_update(a, g, m, v, w, gscale=None):
    """(m, v, w) after one step of the header's adam_update on fp32 tensors; `gscale`: the SCALED form (g * gscale is
    rounded once first)"""
    if gscale is not None:
        g = fmul(g, gscale)
    g, m, v, w = (torch.as_tensor(x, dtype=F32) for x in (g, m, v, w))
    diff = fsub(g, m)
    if a.w1 < 0.5:
        m = fma(a.w1, diff, m)
    else:
        m = fma(-diff, fsub(1.0, a.w1), g)
    v = fma(fmul(a.one_m_b2, g), g, fmul(v, a.b2))
    denom = fadd(fdiv(fsqrt(v), a.bc2_sqrt), a.eps)
    w = fma(-a.step_size, fdiv(m, denom), w)
    return m, v, w


def _boundary_distance(x):
    """fp64 ulps between x > 0 and the nearest midpoint of two adjacent fp32 values"""
    r = torch.tensor(x, dtype=F64).to(F32)
    lo = torch.nextafter(r, torch.tensor(0.0, dtype=F32))
    hi = torch.nextafter(r, torch.tensor(math.inf, dtype=F32))
    mids = ((float(r) + float(lo)) * 0.5, (float(r) + float(hi)) * 0.5)
    return min(abs(x - mp) for mp in mids) / math.ulp(x)


def scalar_margin(lr, b1, b2, t):
    """(fp64 ulps from step_size and bc2_sqrt to the nearest fp32 rounding boundary, whether the narrowed pair is the
    same for every pow result within POW_ULPS ulp of the host's)"""
    exact = scalars64(lr, b1, b2, float(t))
    narrowed = tuple(_f32(x) for x in exact)
    stable = True
    for k in (-POW_ULPS, POW_ULPS):                # the map is monotone in pow: its two ends bound every value between
        def off(b, tt, k=k):
            y = math.pow(b, tt)
            for _ in range(abs(k)):
                y = math.nextafter(y, math.inf if k > 0 else -math.inf)
            return max(y, 0.0)
        stable &= tuple(_f32(x) for x in scalars64(lr, b1, b2, float(t), off)) == narrowed
    return min(_boundary_distance(x) for x in exact), stable


# ---- the packed tail [sse_hi, sse_lo, n / 4096, n % 4096] -------------------------------------------------------------
def pack_tail(sse, n):
    hi = _f32(sse)
    return torch.tensor([hi, _f32(sse - hi), float(n >> 12), float(n & 4095)], dtype=F32)


def tail_count(hi, lo):
    return float(hi) * 4096.0 + float(lo)


def tail_totals(tail, d):
    """(numel, gscale) of a (reduced) tail: numel = D * patch count, gscale = fl32(2 / numel)"""
    numel = tail_count(tail[2], tail[3]) * float(d)
    return numel, _f32(2.0 / numel)


def tail_loss(tail, numel):
    return (float(tail[0]) + float(tail[1])) / numel


# ---- the (lr, betas, t) the GPU tests run ---------------------------------------------------------------------------
LR = 3e-3
BETAS = ((0.5, 0.999), (0.9, 0.999))
T_LARGE = 1_000_000            # b^t underflows to 0 for both betas: step_size = fl32(lr), bc2_sqrt = 1
STEPS = 4                      # consecutive steps per row
TRAINER_LR, TRAINER_STEPS = 1e-2, 7
COMPOSED_LR = 2e-3


def gpu_scalar_rows():
    """every (lr, b1, b2, t) whose scalars a GPU test of tests/test_gpu_adam_exact.py evaluates on the device"""
    rows = set()
    for b1, b2 in BETAS:
        for t0 in (1, T_LARGE):
            rows.update((LR, b1, b2, t0 + s) for s in range(STEPS + 1))
    # graph replays: 5 replays after an eager step
    rows.update((LR, 0.5, 0.999, t) for t in range(1, 8))
    # the trainer: lr halved after steps 3 and 5 (1-based), t = 1 .. 7
    for t in range(1, TRAINER_STEPS + 1):
        for j in range(3):
            rows.add((TRAINER_LR * 0.5 ** j, 0.5, 0.999, t))
    rows.update((COMPOSED_LR, 0.5, 0.999, t) for t in range(1, STEPS + 1))
    return sorted(rows)
