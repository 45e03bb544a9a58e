"""The premises of tests/test_gpu_adam_exact.py, on the CPU: the fp32 emulation of tests/_adam_exact.py against exact
rational arithmetic, the pow margin of every (lr, betas, t) the GPU tests evaluate on the device, and the packed tail's
count fields."""
import math
import random
import struct
from fractions import Fraction

import pytest
import torch

import _adam_exact as E

TWO = Fraction(2)


def round_f32(q, neg_zero=False):
    """a rational rounded to the nearest fp32 value, ties to even, with gradual underflow and overflow to inf"""
    if q == 0:
        return -0.0 if neg_zero else 0.0
    sign = -1.0 if q < 0 else 1.0
    q = abs(q)
    e = q.numerator.bit_length() - q.denominator.bit_length()
    if q < TWO ** e:
        e -= 1
    if q >= TWO ** (e + 1):
        e += 1
    quantum = TWO ** (max(e, -126) - 23)
    n = q / quantum
    k = n.numerator // n.denominator
    rem = n - k
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and k % 2 == 1):
        k += 1
    r = k * quantum
    if r >= TWO ** 128:
        return sign * math.inf
    return sign * float(r)        # k < 2^24: exact in a double, and so is the product with a power of two


def sqrt_f32(q):
    """the correctly rounded fp32 square root of a non-negative rational"""
    if q == 0:
        return 0.0
    k = 200                       # sqrt(q) >= 2^-75 for an fp32 q, so 2^-200 resolves every fp32 rounding boundary
    big = q * 4 ** k
    s = math.isqrt(big.numerator // big.denominator)
    if Fraction(s * s) == big:
        return round_f32(Fraction(s, 2 ** k))
    return round_f32(Fraction(2 * s + 1, 2 ** (k + 1)))     # strictly between s and s + 1: no boundary lies there


def fma_ref(a, b, c):
    exact = Fraction(a) * Fraction(b) + Fraction(c)
    if exact == 0:
        # an exact zero sum is -0 only when both addends are -0 (round to nearest)
        p_neg = (a == 0 or b == 0) and math.copysign(1.0, a) * math.copysign(1.0, b) < 0
        return -0.0 if (p_neg and c == 0 and math.copysign(1.0, c) < 0) else 0.0
    return round_f32(exact, neg_zero=exact < 0)


def bits(x):
    return struct.unpack("<I", struct.pack("<f", x))[0]


def f32(x):
    return float(torch.tensor(x, dtype=torch.float64).float())


def _emulated_fma(triples):
    a, b, c = (torch.tensor([t[i] for t in triples], dtype=torch.float32) for i in range(3))
    return E.fma(a, b, c).tolist()


def _check_fma(triples, what):
    got = _emulated_fma(triples)
    bad = [(t, g, fma_ref(*t)) for t, g in zip(triples, got) if bits(g) != bits(fma_ref(*t))]
    assert not bad, f"{what}: {len(bad)} of {len(triples)} differ, e.g. {bad[:3]}"


def test_fma_trap_is_rounded_once():
    a, b, c = E.FMA_TRAP
    assert (f32(a), f32(b), f32(c)) == (a, b, c)
    naive = f32(a * b + c)
    assert naive.hex() == "0x1.0000040000000p+0"
    assert fma_ref(a, b, c).hex() == "0x1.0000020000000p+0"
    assert E.fma(torch.tensor(a), torch.tensor(b), torch.tensor(c)).item() == fma_ref(a, b, c)


def _midpoint_cases():
    """fp64 sums that land exactly on an fp32 midpoint while the exact sum lies just below or just above it: both
    signs, normal scales from 2^-100 to 2^100, odd and even neighbours, and the largest (odd) subnormals"""
    u = 2.0 ** -23
    out = []
    for scale in (2.0 ** -100, 2.0 ** -20, 1.0, 2.0 ** 20, 2.0 ** 100):
        for r in (1.0 + u, 1.0 + 3 * u, 1.5 + u, 1.0 + 2 * u, 1.75):
            for sa in (1.0, -1.0):
                for sc in (1.0, -1.0):
                    out.append((sa * (1.0 + u) * scale, 2.0 ** -24 * (1.0 - u), sc * r * scale))
    # subnormal spacing: a b = 2^-150 (1 - 2^-46), c = m 2^-149 with m large and odd
    for m in ((1 << 23) - 1, (1 << 23) - 3, (1 << 22) + 1, (1 << 22) + 2):
        for sa in (1.0, -1.0):
            for sc in (1.0, -1.0):
                out.append((sa * 2.0 ** -75 * (1.0 + u), 2.0 ** -75 * (1.0 - u), sc * m * 2.0 ** -149))
    return out


def test_fma_midpoint_cases_match_exact_rounding():
    cases = _midpoint_cases()
    for a, b, c in cases:
        assert (f32(a), f32(b), f32(c)) == (a, b, c)
    # the construction does reach the double-rounding trap for a good share of them
    trapped = sum(bits(f32(a * b + c)) != bits(fma_ref(a, b, c)) for a, b, c in cases)
    assert trapped >= len(cases) // 4, trapped
    _check_fma(cases, "midpoints")


def _rand_f32(rng, lo_exp, hi_exp):
    m = rng.randrange(1 << 23, 1 << 24)
    e = rng.randint(lo_exp, hi_exp)
    return f32(rng.choice((1.0, -1.0)) * m * 2.0 ** (e - 23))


def test_fma_random_inputs_match_exact_rounding():
    rng = random.Random(5)
    cases = []
    for _ in range(4000):
        a, b = _rand_f32(rng, -30, 30), _rand_f32(rng, -30, 30)
        kind = rng.randrange(4)
        if kind == 0:
            c = _rand_f32(rng, -60, 60)
        elif kind == 1:                                   # near cancellation
            c = f32(-a * b * (1.0 + rng.uniform(-1e-6, 1e-6)))
        elif kind == 2:                                   # c dominates, a b is a few ulps of it
            c = _rand_f32(rng, 0, 10)
            b = f32(b * 2.0 ** -40)
        else:                                             # a b dominates
            c = _rand_f32(rng, -50, -40)
        cases.append((a, b, c))
    _check_fma(cases, "random")


def test_fma_subnormal_results_and_exact_cancellation_match():
    rng = random.Random(6)
    cases = []
    for _ in range(2000):
        a, b = _rand_f32(rng, -80, -60), _rand_f32(rng, -80, -60)        # a b in [2^-160, 2^-120)
        c = f32(rng.choice((1.0, -1.0)) * rng.randrange(0, 1 << 23) * 2.0 ** -149)
        cases.append((a, b, c))
    for _ in range(500):                                                    # a b exact in fp32: exact zero
        a = f32(rng.randrange(1, 1 << 12) * 2.0 ** rng.randint(-20, 20))
        b = f32(rng.choice((1.0, -1.0)) * rng.randrange(1, 1 << 12) * 2.0 ** rng.randint(-20, 20))
        cases.append((a, b, -a * b))
        # a b not exact in fp32: the result is the product's rounding error, exactly
        a2, b2 = _rand_f32(rng, -5, 5), _rand_f32(rng, -5, 5)
        cases.append((a2, b2, -f32(a2 * b2)))
    cases += [(0.0, 1.0, -0.0), (-0.0, 1.0, -0.0), (-0.0, -1.0, -0.0), (1.0, -0.0, 0.0), (2.0 ** -75, 2.0 ** -75, 0.0),
              (-(2.0 ** -75), 2.0 ** -75, 0.0), (2.0 ** -75, 2.0 ** -76, 2.0 ** -149), (3.0 * 2.0 ** -76, 2.0 ** -75, 0.0),
              (2.0 ** 127, 4.0, -(2.0 ** 127)), (2.0 ** 64, 2.0 ** 64, 3.4e38)]
    got = _emulated_fma(cases)
    assert any(g != 0 and abs(g) < 2.0 ** -126 for g in got)
    assert any(bits(g) == 0 for g in got) and any(bits(g) == 0x80000000 for g in got)
    _check_fma(cases, "subnormal / cancellation")


def test_fma_overflow_threshold():
    """the midpoint between the largest float and 2^128: exact sums just below it stay finite, at or above it overflow"""
    top = f32(3.4028234663852886e38)
    u = 2.0 ** -23
    for sa in (1.0, -1.0):
        for b, c in ((2.0 ** 103 * (1.0 - u), top), (2.0 ** 103, top), (2.0 ** 103 * (1.0 + u), top)):
            cases = [(sa * (1.0 + u), b, sa * c)]
            _check_fma(cases, "overflow")


def _adam_ref(a, g, m, v, w, gscale=None):
    """one element of the header's adam_update in exact rational arithmetic, rounded where the fp32 code rounds"""
    F = Fraction
    if gscale is not None:
        g = round_f32(F(g) * F(gscale))
    diff = round_f32(F(g) - F(m))
    if a.w1 < 0.5:
        m = round_f32(F(a.w1) * F(diff) + F(m))
    else:
        m = round_f32(-F(diff) * F(round_f32(1 - F(a.w1))) + F(g))
    v = round_f32(F(round_f32(F(a.one_m_b2) * F(g))) * F(g) + F(round_f32(F(v) * F(a.b2))))
    denom = round_f32(F(round_f32(F(sqrt_f32(F(v))) / F(a.bc2_sqrt))) + F(a.eps))
    w = round_f32(-F(a.step_size) * F(round_f32(F(m) / F(denom))) + F(w))
    return m, v, w


@pytest.mark.parametrize("b1,eps,t,scaled", [(0.5, 1e-8, 1, False), (0.9, 1e-8, 3, True), (0.5, 0.0, 2, True),
                                             (0.9, 1e-3, E.T_LARGE, False)])
def test_adam_update_matches_exact_rational_evaluation(b1, eps, t, scaled):
    a = E.adam_scalars(E.LR, b1, 0.999, eps, t)
    rng = random.Random(int(b1 * 10) + t)
    n = 300
    g = [_rand_f32(rng, -20, 5) for _ in range(n)]
    g[:4] = [0.0, 1e-40, -3e-42, 2.0 ** -140]            # zero and subnormal gradients
    m = [_rand_f32(rng, -20, 5) for _ in range(n)]
    m[4:8] = [0.0, 1e-41, g[6], -g[7]]
    v = [abs(_rand_f32(rng, -40, 10)) for _ in range(n)]
    v[8:10] = [1e-44, 2.0 ** -126]
    if eps == 0.0:
        v = [x if x != 0 else 1e-30 for x in v]
    w = [_rand_f32(rng, -10, 3) for _ in range(n)]
    gscale = f32(2.0 / (64 * 4099)) if scaled else None
    T = [torch.tensor(x, dtype=torch.float32) for x in (g, m, v, w)]
    em, ev, ew = E.adam_update(a, *T, gscale=gscale)
    for i in range(n):
        want = _adam_ref(a, g[i], m[i], v[i], w[i], gscale)
        got = (em[i].item(), ev[i].item(), ew[i].item())
        assert got == want, f"element {i}: g={g[i]!r} m={m[i]!r} v={v[i]!r} w={w[i]!r}: {got} != {want}"


def test_adam_scalars_narrow_the_header_expressions():
    a = E.adam_scalars(E.LR, 0.5, 0.999, 1e-8, 1)
    assert a.w1 == 0.5 and a.b2 == f32(0.999) and a.one_m_b2 == f32(1.0 - 0.999) and a.eps == f32(1e-8)
    assert a.step_size == f32(E.LR / 0.5) and a.bc2_sqrt == f32(math.sqrt(1.0 - 0.999))
    big = E.adam_scalars(E.LR, 0.9, 0.999, 0.0, E.T_LARGE)
    assert big.step_size == f32(E.LR) and big.bc2_sqrt == 1.0 and big.w1 == f32(0.1)
    assert math.pow(0.999, E.T_LARGE) == 0.0 and math.pow(0.9, E.T_LARGE) == 0.0


@pytest.mark.parametrize("row", E.gpu_scalar_rows(), ids=lambda r: f"lr{r[0]:g}_b{r[1]:g}_t{r[3]}")
def test_every_gpu_row_narrows_the_same_whatever_the_device_pow_returns(row):
    margin, stable = E.scalar_margin(*row)
    assert margin >= E.MIN_MARGIN, f"{row}: {margin:.0f} fp64 ulps from an fp32 rounding boundary"
    assert stable, f"{row}: a pow result within {E.POW_ULPS} ulp narrows differently"


def test_pack_tail_count_round_trips_every_int32_count():
    """n = (n >> 12) 4096 + (n & 4095): both fields are exact fp32 integers for every n <= INT32_MAX (hi < 2^19, lo <
    4096), and hi 4096 + lo is exact in fp64.  The two fields vary independently, so checking every value of each field
    checks every n; the ends of the range are also checked as whole counts."""
    hi = torch.arange(0, 1 << 19, dtype=torch.int64)
    lo = torch.arange(0, 4096, dtype=torch.int64)
    assert torch.equal(hi.float().to(torch.int64), hi) and torch.equal(lo.float().to(torch.int64), lo)
    ends = torch.cat([torch.arange(0, 1 << 16), torch.arange((1 << 31) - (1 << 16), 1 << 31)])
    for n in ends[::97].tolist() + [0, 4095, 4096, 2 ** 30, 2 ** 31 - 1]:
        t = E.pack_tail(0.0, n)
        assert E.tail_count(t[2], t[3]) == n
    big = torch.arange(0, 1 << 31, 12289, dtype=torch.int64)
    h, l = (big >> 12).float(), (big & 4095).float()
    assert torch.equal(h.double() * 4096.0 + l.double(), big.double())


def test_sums_of_eight_tails_carry_the_global_count():
    """an fp32 sum, in any order, of the tails of 8 ranks: every partial sum of the count fields is an integer below
    2^24, so the reduced fields give the exact global count (8 ranks of 2^30 patches: a hi field of 2^21)"""
    rng = random.Random(8)
    shares = [[2 ** 30] * 8, [2 ** 31 - 1] * 8, [0] * 7 + [2 ** 31 - 1], [4095] * 8, [4096] * 8]
    shares += [[rng.randrange(0, 2 ** 31) for _ in range(8)] for _ in range(200)]
    for ns in shares:
        tails = torch.stack([E.pack_tail(0.0, n) for n in ns])
        for order in (list(range(8)), list(range(7, -1, -1))):
            acc = torch.zeros(4, dtype=torch.float32)
            for i in order:
                acc = acc + tails[i]
            assert E.tail_count(acc[2], acc[3]) == sum(ns), ns


def test_tail_totals_and_loss():
    sse = 12345.678901234567
    t = E.pack_tail(sse, 3 * 4096 + 5)
    assert float(t[0]) == f32(sse) and float(t[0]) + float(t[1]) != float(t[0])
    assert abs(float(t[0]) + float(t[1]) - sse) <= 2.0 ** -40 * sse
    numel, gscale = E.tail_totals(t, 64)
    assert numel == 64.0 * (3 * 4096 + 5) and gscale == f32(2.0 / numel)
    assert E.tail_loss(t, numel) == (float(t[0]) + float(t[1])) / numel
