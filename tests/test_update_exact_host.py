"""CPU proof of the exact-value premises of tests/test_gpu_update_exact.py (helpers in tests/_update_exact.py): the
impulse input gives every filter output at most one term and exercises every tensor-core block, the expected values are
exact fp32 results, and the lattice bound check of the accumulation accepts and rejects what it should."""
import pytest
import torch

import _lattice as L
import _update_exact as U


@pytest.mark.parametrize("k,d,h", [(300, 18, 0), (1000, 33, 7), (4096, 64, 20), (300, 512, 300), (4100, 50, 41),
                                   (6000, 96, 1400), (777, 200, 150)])
def test_impulses_give_each_output_exactly_its_one_term(k, d, h):
    vals, src = U.impulse_case(k, d, h)
    terms = U.terms_per_output(vals, src, h)
    assert bool((terms <= 1).all())
    assert torch.equal(terms == 1, src >= 0)
    a = torch.arange(k)[:, None]
    j = src.clamp(min=0)
    assert bool(((a - j).abs()[src >= 0] <= h).all())
    assert bool((torch.gather(vals, 0, j)[src >= 0] != 0).all())
    # the values are +-2^k, k in [0, 7], with both signs and several exponents
    v = vals[vals != 0]
    m, e = torch.frexp(v)
    assert bool((m.abs() == 0.5).all()) and int(e.min()) == 1 and int(e.max()) == 8
    assert bool((v > 0).any()) and bool((v < 0).any())
    # inside the codebook, away from its ends, every output has its term
    if k > 4 * h + 2:
        assert bool((src[2 * h + 1:k - 2 * h - 1] >= 0).all())
    # the impulse rows cover every position of a k-block
    rows = torch.nonzero(vals != 0)[:, 0]
    assert len(set(((rows + h) % 32).tolist())) == 32


@pytest.mark.parametrize("k,d,h,sms", [(4096, 64, 0, 148), (2048, 128, 20, 148), (4096, 64, 512, 148),
                                       (300, 512, 300, 148), (6000, 96, 1400, 148), (4100, 50, 41, 148),
                                       (16384, 64, 100, 148), (12800, 96, 100, 148)])
def test_impulses_reach_every_tensor_core_block(k, d, h, sms):
    """every (unit tile, k-block, accumulation chain) of the modelled plan holds an impulse of some column"""
    nkb, q, na, ks = U.tc_plan_model(k, h, sms, (d + (127 if d > 64 else 63)) // (128 if d > 64 else 64))
    assert na <= 4 and (na - 1) * q < nkb <= na * q
    vals, _ = U.impulse_case(k, d, h)
    want = U.tc_all_blocks(k, h, nkb, q)
    got = U.tc_hits(vals, h, nkb, q)
    assert want <= got, f"{len(want - got)} blocks without an impulse"
    assert {c for _, _, c in got} == set(range(na))
    assert {t for t, _, _ in got} == set(range((k + 127) // 128))


@pytest.mark.parametrize("rng", [0.01, 5.0, 40.0, 512.0, 8192.0, 1e5, 6.6e6])
def test_tensor_core_expected_values_are_exact(rng):
    """hi + lo is an fp32 value, v (hi + lo) is exact for every impulse value, and so is the sum with zeros in any
    association; the subnormal class (hi or lo subnormal) lies in the outer band"""
    h = 4000
    w = U.weights64(rng, h + 1).float()
    s, sub = U.tc_weights(w)
    assert torch.equal(L.tf32_rna(w - L.tf32_rna(w)) + L.tf32_rna(w), s)
    for k in range(8):
        for sign in (1.0, -1.0):
            v = sign * 2.0 ** k
            p = s * v
            assert torch.equal(p.double(), s.double() * v)
            assert torch.equal(((p + 0.0) + 0.0) + 0.0, p)
    # hi + lo is w to 21 bits or better down to 2^-100 (below, w - hi may be subnormal); the subnormal class lies in
    # that far band, and flushing its operands moves a weight by less than 2^-126
    normal = w.abs() >= 2.0 ** -100
    assert bool(((s - w).abs()[normal] <= w.abs()[normal] * 2.0 ** -21).all())
    assert bool((w[sub] < 2.0 ** -100).all())
    assert bool(((U.tc_weights_flushed(w) - s).abs()[sub] < 2.0 ** -126).all())


def test_weight_table_check_catches_a_wrong_weight():
    w = U.weights64(40.0, 200).float()
    h = int(torch.nonzero(w > 0).max())
    U.check_weight_table(w, 40.0, h)
    bad = w.clone()
    bad[17] = torch.nextafter(torch.nextafter(torch.nextafter(bad[17], torch.tensor(2.0)), torch.tensor(2.0)),
                              torch.tensor(2.0))
    with pytest.raises(AssertionError):
        U.check_weight_table(bad, 40.0, h)


def test_filter_expected_is_the_dense_product_on_impulses():
    k, d, h, rng = 257, 40, 9, 10.0
    vals, src = U.impulse_case(k, d, h)
    w = U.weights64(rng, k).float()
    w[h + 1:] = 0
    dense = w[(torch.arange(k)[:, None] - torch.arange(k)[None, :]).abs()].double() @ vals.double()
    got = U.filter_expected(vals, src, w, 0.37)
    assert torch.equal(got, (dense.float() * torch.tensor(0.37, dtype=torch.float32)))


@pytest.mark.parametrize("n,k,s", [(4096, 300, 8), (40000, 1000, 16), (300000, 5000, 64)])
def test_segment_bmu_structure(n, k, s):
    bmu = U.segment_bmu(n, k, s, seed=n)
    counts = torch.bincount(bmu, minlength=k)
    assert int(counts[0]) == 0 and int(counts[k - 1]) == 0
    starts = torch.cumsum(counts, 0) - counts
    assert int(counts[1]) == 9 * s + 3 and int(starts[1]) % s == 0
    assert int(starts[2] + counts[2]) % s == 0
    assert int(starts[3]) % s == 0 and int(counts[3]) % s == 0


def test_accum_bound_accepts_the_lattice_and_rejects_an_overflow():
    g = torch.Generator().manual_seed(3)
    n, d, k = 5000, 64, 300
    a = torch.randint(-3, 4, (n, d), generator=g)
    b = torch.randint(-3, 4, (k, d), generator=g)
    bmu = U.segment_bmu(n, k, 8, seed=1)
    for path, vec in (("scan", 4), ("sorted", 2), ("sorted", 1)):
        assert U.check_accum_bound(a, b, bmu, k, path, vec, s=8) < U.BOUND
    # a heavy hitter whose residual sum in one feature reaches 2^24 units
    a2 = a.clone()
    a2[:, 0] = -4000
    bmu2 = torch.zeros(n, dtype=torch.int64)
    with pytest.raises(AssertionError):
        U.check_accum_bound(a2, b, bmu2, k, "sorted", 1, s=64)
    # a scan-path CTA whose squared error over 1024 features reaches 2^24 units
    a3 = torch.full((2048, 1024), 3, dtype=torch.int64)
    b3 = torch.full((4, 1024), -1, dtype=torch.int64)
    with pytest.raises(AssertionError):
        U.check_accum_bound(a3, b3, torch.zeros(2048, dtype=torch.int64), 4, "scan", 4)


def test_accum_reference_and_packed_tail():
    g = torch.Generator().manual_seed(5)
    a = torch.randint(-3, 4, (100, 8), generator=g)
    b = torch.randint(-3, 4, (10, 8), generator=g)
    bmu = torch.randint(0, 10, (100,), generator=g)
    rbar, xbar, counts, sse = U.accum_reference(a, b, bmu, 10)
    r = b[bmu] - a
    assert torch.equal(rbar, torch.stack([r[bmu == u].sum(0) for u in range(10)]))
    assert torch.equal(xbar, torch.stack([a[bmu == u].sum(0) for u in range(10)]))
    assert int(counts.sum()) == 100 and sse == int((r * r).sum())
    t = U.packed_tail(2.0 ** 30 + 3.0, 5000)
    assert float(t[0].double() + t[1].double()) == 2.0 ** 30 + 3.0
    assert float(t[2]) * 4096 + float(t[3]) == 5000
