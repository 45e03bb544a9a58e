"""Exact-lattice BMU cases and an fp64 reference with the lowest-index tie rule.

On a lattice every BMU kernel's arithmetic is exact, so every kernel must return the lowest-index true argmin and the
true reduced distance rd = ||c||^2 - 2 x.c bit for bit.  A case is

    x = a * 2^e,  W = b * 2^e,   a, b integers, one shared power of two e

* narrow: |a|, |b| <= 8, data-like: patches and units scatter around shared centres (`_clustered`), so the true argmin
  depends on x (`zero_unit_share` measures how often it does not).  Every operand is exact in the TF32 and FP16 hi
  parts after any power-of-two row or codebook scale (4 significant bits), so every lo part is 0.  The values are exact
  in fp16 and bf16 too.
* wide-x: |b| <= 8, and some |a| in [2^11, 2^13): x then has a non-zero lo part in both splits (13 > 11 significant
  bits), which exercises the x_lo . c_hi product.  c_lo = 0, so the dropped lo . lo product is exactly 0.

Bound: for every (patch, unit) pair sum_d |2 a b| + sum_d b^2 < 2^24.  Every partial sum of ||c||^2 - 2 x.c is then an
integer multiple of 2^(2e) below 2^24 of them, exact in an fp32 accumulator in any order and any split of the feature
axis, and so is ||c||^2 itself (the three-part norm tails carry 33 bits).  `check_bound` asserts it on the data.

Planted structure (positions chosen per case, see `plant`): exact copies of a unit inside its 8-unit chunk, in another
256-unit tile, in the padded last unit tile and near the end of the codebook (another unit split or shard); mirror
pairs x_p + e_j and x_p - e_j of sampled patches (two different rows at exactly the same distance); all-zero patches
and all-zero units.
"""
import torch

SCALES = (-12, 0, 12)
BOUND = 1 << 24
WIDE_LO, WIDE_HI = 1 << 11, 1 << 13
WIDE_PER_ROW = 64                  # wide entries per wide row: keeps the bound at every D up to 8192


def _ints(gen, shape, lim):
    return torch.randint(-lim, lim + 1, shape, generator=gen, dtype=torch.int64)


def _clustered(gen, n, k, d):
    """Data-like narrow rows: patches and units both scatter (+-1 on a third of the features each way, clamped to
    [-8, 8]) around a few shared random centres.  Every patch then has units of its own centre at a distance far below
    ||x||, so its true argmin has rd < 0 and depends on x; with independent random rows rd = ||c - x||^2 - ||x||^2 would
    be positive for almost every unit beyond D ~ 32, and the planted all-zero units (rd = 0) would answer nearly every
    patch whatever the kernel read."""
    m = max(1, min(64, k // 8))
    centres = _ints(gen, (m, d), 7)

    def draw(rows, first):
        cid = torch.randint(0, m, (rows,), generator=gen)
        if first:
            cid[:min(rows, m)] = torch.arange(min(rows, m))         # every centre has units
        return (centres[cid] + torch.randint(-1, 2, (rows, d), generator=gen)).clamp(-8, 8)

    return draw(n, False), draw(k, True)


def lattice_ints(n, d, k, kind, seed, plant_ties=True):
    """Integer matrices (A (n, d), B (k, d), int64) of a lattice case with its planted structure."""
    assert kind in ("narrow", "wide")
    gen = torch.Generator().manual_seed(seed)
    a, b = _clustered(gen, n, k, d)
    if kind == "wide":
        # three rows in four carry WIDE_PER_ROW (or all d, if fewer) entries of magnitude [2^11, 2^13); the fourth stays
        # narrow so that mirror pairs can be planted around it with |b| <= 8
        wide_rows = torch.arange(n) % 4 != 3
        m = min(WIDE_PER_ROW, d)
        cols = torch.argsort(torch.rand(n, d, generator=gen), dim=1)[:, :m]
        mag = torch.randint(WIDE_LO, WIDE_HI, (n, m), generator=gen, dtype=torch.int64)
        sign = torch.randint(0, 2, (n, m), generator=gen, dtype=torch.int64) * 2 - 1
        big = a.clone()
        big.scatter_(1, cols, mag * sign)
        a = torch.where(wide_rows[:, None], big, a)
    if plant_ties:
        plant(a, b, gen)
    return a, b


def plant(a, b, gen):
    """Plant ties into B (in place) and zero patches into A."""
    n, d = a.shape
    k = b.shape[0]
    # all-zero patches: rd = ||c||^2, so the all-zero units below tie at 0
    for p in (0, n // 2, n - 1):
        a[p] = 0
    zero_units = sorted({min(k - 1, u) for u in (5, k // 3 + 1, k - 2)})
    # mirror pairs around narrow patches, each unit of a pair at a different position class
    # (the patch is pulled into [-7, 7] first, so that both mirrors keep |b| <= 8)
    narrow = torch.nonzero((a.abs().amax(1) <= 8) & (a != 0).any(1)).flatten()
    sites = _sites(k)
    n_pairs = min(len(sites) // 2, narrow.numel())
    pick = narrow[torch.randperm(narrow.numel(), generator=gen)[:n_pairs]]
    used = set(zero_units)
    for t, p in enumerate(pick.tolist()):
        u1, u2 = sites[2 * t], sites[2 * t + 1]
        if u1 in used or u2 in used or u1 == u2:
            continue
        used.update((u1, u2))
        a[p] = a[p].clamp(-7, 7)
        j = int(torch.randint(0, d, (1,), generator=gen))
        b[u1] = a[p]
        b[u2] = a[p]
        b[u1, j] += 1
        b[u2, j] -= 1
    # exact copies of some units: in the same 8-unit chunk, another 256-unit tile, the padded last tile, the far end
    for src in sorted(used - set(zero_units))[:4]:
        for dst in (src - src % 8 + (src % 8 + 3) % 8, (src + 256 * 3 + 1) % k, k - 1 - (src % 3), k - 7):
            if 0 <= dst < k and dst not in used:
                b[dst] = b[src]
    for u in zero_units:
        b[u] = 0


def _sites(k):
    """Unit positions for planted mirror pairs: early, chunk-adjacent, across tiles, in the last (padded) tile."""
    cand = [1, 2, 9, 10, 250, 258, 511, 600, k // 2, k // 2 + 8, k - 300, k - 260, k - 5, k - 3]
    out = []
    for u in cand:
        if 0 <= u < k and u not in out:
            out.append(u)
    return out


def zero_unit_share(a, b, idx):
    """Share of the non-zero patches (rows of A) whose answer `idx` is an all-zero unit of B: a case where this is
    large tests little but the tie rule among the zero units."""
    zero_units = (b == 0).all(1).to(idx.device)
    nz = (a != 0).any(1).to(idx.device)
    return float(zero_units[idx][nz].float().mean()) if bool(nz.any()) else 0.0


MAX_ZERO_SHARE = 0.02


def check_bound(a, b):
    """Assert sum_d |2 a b| + sum_d b^2 < 2^24 for every (patch, unit) pair; returns the largest value."""
    aa, ba = a.abs(), b.abs()
    nb = int((b * b).sum(1).max())
    # cheap form: sum_d |a_d b_d| <= max|b| * max_p sum_d |a_pd|
    cheap = 2 * int(ba.max()) * int(aa.sum(1).max()) + nb
    if cheap < BOUND:
        return cheap
    worst = 0
    for i in range(0, a.shape[0], 4096):
        m = (aa[i:i + 4096].double() @ ba.double().T) * 2 + (b * b).sum(1).double()[None, :]
        worst = max(worst, int(m.max()))
    assert worst < BOUND, f"lattice bound {worst} >= 2^24"
    return worst


def to_float(ints, e, dtype=torch.float32):
    """ints * 2^e, exactly (every |value| here is below 2^24)."""
    return torch.ldexp(ints.to(torch.float64), torch.tensor(float(e), dtype=torch.float64)).to(dtype)


def unpatchify(rows, c, ph, pw, gh, gw):
    """(n_img * gh * gw, c * ph * pw) patch rows -> the (n_img, c, gh * ph, gw * pw) batch they come from."""
    n_img = rows.shape[0] // (gh * gw)
    t = rows.reshape(n_img, gh, gw, c, ph, pw).permute(0, 3, 1, 4, 2, 5)
    return t.reshape(n_img, c, gh * ph, gw * pw).contiguous()


def fp64_rd(x, w, chunk=2048):
    """rd64 = ||c||^2 - 2 x.c in fp64 per (patch, unit), as a generator of (row0, rd) blocks of at most `chunk` rows."""
    w64 = w.double()
    cn = (w64 * w64).sum(1)
    for i in range(0, x.shape[0], chunk):
        yield i, cn[None, :] - 2.0 * (x[i:i + chunk].double() @ w64.T)


def fp64_bmu(x, w, chunk=2048):
    """(lowest index of the fp64 minimum of rd, that minimum) per patch.  The index comes from a masked min, so it does
    not depend on torch.argmin's tie rule."""
    k = w.shape[0]
    idx = torch.empty(x.shape[0], dtype=torch.int64, device=x.device)
    best = torch.empty(x.shape[0], dtype=torch.float64, device=x.device)
    ar = torch.arange(k, device=x.device)
    for i, rd in fp64_rd(x, w, chunk):
        m = rd.min(1).values
        idx[i:i + rd.shape[0]] = torch.where(rd == m[:, None], ar[None, :], k).min(1).values
        best[i:i + rd.shape[0]] = m
    return idx, best
