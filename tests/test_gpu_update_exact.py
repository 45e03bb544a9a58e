"""The training step's update path, exactly, in every regime: the neighbourhood filter on impulse inputs, the per-unit
accumulation on the integer lattice, and the one-kernel step against the same step composed of the separate kernels.

Which kernel runs depends on K, D, the band half-width h, 16-byte alignment, the workspace and the SM count
(csrc/som_filter.cu, som_filter_tc.cu, som_accumulate.cu, som_step_small.cu).  Every row first asserts through the
test hooks som_debug_filter_plan / som_debug_accumulate_plan / som_debug_step_small_plan that its shape reaches its
regime on this part, then compares with zero tolerance (expected values: tests/_update_exact.py):

* filter: the device weight table against fp64 expf, then every output element (and the guard bands around `out`)
  against its one exact term: fl32(scale v w) for the FFMA kernels, fl32(scale v (hi + lo)) for the tensor-core kernels.
  Where hi or lo is subnormal the tensor pipe keeps the operand (SUBNORMAL_RULE, DESIGN.md section 2);
* accumulation: Rbar (residual and plain sum), the counts, the squared error and the packed tail against int64;
* one-kernel step: W, m, v, the BMUs and the step count bit-identical to the scalar filter, the scan accumulation, the
  scaled scalar filter and adam_step_dev, step after step; on the lattice at h = 0 the loss is the exact squared error.

The last tests derive the reachable kernel sets from the hooks and assert that the rows reach all of them."""
import ctypes
from dataclasses import dataclass

import pytest
import torch

from somcb import _lib, ops
import _lattice as L
import _update_exact as U

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SCALE = 0.37
# how tcgen05.mma kind::tf32 treats a subnormal A operand (hi or lo of a far-band weight): "kept" exactly or "flushed"
SUBNORMAL_RULE = "kept"


def _hook(name, argtypes):
    fn = getattr(_lib.load(), name)
    fn.restype = ctypes.c_int
    fn.argtypes = argtypes
    return fn


FILTER_FIELDS = ("kernel", "h", "smem", "nkb", "q", "na", "ks", "Kp")          # csrc/som_common.cuh: FilterPlanField
KERNELS = {0: "scalar", 1: "tile64", 2: "tile128", 3: "tc64", 4: "tc128"}
ACCUM_FIELDS = ("path", "vec", "S", "n_chunks", "n_slices", "cs_per", "cs_blocks")   # AccumPlanField
PATHS = {0: "scan", 1: "counting", 2: "radix"}
STEP_FIELDS = ("grid", "R", "RB", "slot", "UC", "PG", "PPG", "h")


def filter_plan(k, d, rng, with_ws, aligned):
    fn = _hook("som_debug_filter_plan", [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int,
                                         ctypes.POINTER(ctypes.c_int64), ctypes.c_int])
    out = (ctypes.c_int64 * len(FILTER_FIELDS))()
    rc = fn(k, d, rng, int(with_ws), int(aligned), out, len(FILTER_FIELDS))
    assert rc == 0, _lib.load().som_last_error()
    p = dict(zip(FILTER_FIELDS, list(out)))
    p["kernel"] = KERNELS[p["kernel"]]
    return p


def accum_plan(x_ptr, geom, wt_ptr, k, rbar_ptr):
    fn = _hook("som_debug_accumulate_plan", [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                             ctypes.POINTER(ctypes.c_int64), ctypes.c_int])
    out = (ctypes.c_int64 * len(ACCUM_FIELDS))()
    rc = fn(x_ptr, *geom, wt_ptr, k, rbar_ptr, out, len(ACCUM_FIELDS))
    assert rc == 0, _lib.load().som_last_error()
    p = dict(zip(ACCUM_FIELDS, list(out)))
    p["path"] = PATHS[p["path"]]
    return p


def step_plan(n, d, k, rng):
    fn = _hook("som_debug_step_small_plan", [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                             ctypes.POINTER(ctypes.c_int64), ctypes.c_int])
    out = (ctypes.c_int64 * len(STEP_FIELDS))()
    assert fn(n, d, k, rng, out, len(STEP_FIELDS)) == 0
    p = dict(zip(STEP_FIELDS, list(out)))
    return None if p["grid"] < 0 else p


def range_for_h(k, h):
    """a neighbourhood range whose band half-width (som_filter_half_width) is exactly h"""
    lo, hi = 1e-6, 1e9
    for _ in range(200):
        mid = (lo * hi) ** 0.5
        if ops.filter_half_width(k, mid) >= h:
            hi = mid
        else:
            lo = mid
    assert ops.filter_half_width(k, hi) == h, f"no range gives h = {h} at K = {k}"
    return hi


def _sms():
    return ops.device_info()[0]


def _guarded(n, off):
    buf = torch.full((n + 128 + 1,), -777.0, device=DEV)
    return buf, buf[64 + off:64 + off + n]


def _guard_ok(buf, n, off):
    return bool((buf[:64 + off] == -777.0).all()) and bool((buf[64 + off + n:] == -777.0).all())


# ================================================ filter ============================================================
@dataclass
class FRow:
    k: int
    d: int
    rng: object             # a range, or ("h", target)
    ws: bool                # through som_filter_ws_f32 with a workspace (tensor_cores=True)
    aligned: bool           # 16-byte aligned out (else offset by 4 bytes)
    expect: dict
    check: object = None

    def range(self):
        return range_for_h(self.k, self.rng[1]) if isinstance(self.rng, tuple) else self.rng


def _ks_split(p):
    return p["ks"] > 1 and p["ks"] == p["na"]


# shapes follow the SM count s where the rule does (148 on a B200: the comments give those values)
FROWS = {
    "scalar_d18": lambda s: FRow(1000, 18, 40.0, True, True, {"kernel": "scalar"}),
    "scalar_d33": lambda s: FRow(777, 33, 5.0, False, True, {"kernel": "scalar"}),
    "scalar_d64_misaligned": lambda s: FRow(1500, 64, 100.0, False, False, {"kernel": "scalar"}),
    # h ~ 6720: the table needs more than 48 KB of shared memory
    "scalar_opt_in": lambda s: FRow(7000, 20, 1e6, True, True, {"kernel": "scalar"}, lambda p: p["smem"] > 48 * 1024),
    "tile64_d48": lambda s: FRow(1000, 48, 50.0, False, True, {"kernel": "tile64"}),
    "tile64_d64": lambda s: FRow(999, 64, 30.0, False, True, {"kernel": "tile64"}),
    "tile128_d128": lambda s: FRow(1001, 128, 60.0, False, True, {"kernel": "tile128"}),
    "tile128_d200": lambda s: FRow(1003, 200, 20.0, False, True, {"kernel": "tile128"}),
    # s / 2 unit tiles: the last tile count that k-splits (2 tiles <= s), then one more tile
    "tc64_ksplit": lambda s: FRow(128 * (s // 2), 64, 512.0, True, True, {"kernel": "tc64"}, _ks_split),
    "tc64_one_cta": lambda s: FRow(128 * (s // 2 + 1), 64, 512.0, True, True, {"kernel": "tc64", "ks": 1}),
    "tc128_d96_ksplit": lambda s: FRow(128 * (s // 2) - 5, 96, 200.0, True, True, {"kernel": "tc128"}, _ks_split),
    "tc128_d96_one_cta": lambda s: FRow(128 * (s // 2) + 7, 96, 200.0, True, True, {"kernel": "tc128", "ks": 1}),
    "tc64_c4_shape": lambda s: FRow(16384, 64, 100.0, True, True, {"kernel": "tc64", "ks": 1}),
    # D % 32 != 0: the epilogue's scalar store path on the last feature tile
    "tc128_d530": lambda s: FRow(1000, 530, 3.0, True, True, {"kernel": "tc128"}),
    "tc_h0": lambda s: FRow(4096, 64, 0.01, True, True, {"kernel": "tc64", "h": 0, "nkb": 4, "q": 1, "na": 4}),
    "tc_partial_strip": lambda s: FRow(2048, 128, ("h", 20), True, True,
                                       {"kernel": "tc128", "h": 20, "nkb": 6, "q": 2, "na": 3}),
    "tc_h1400": lambda s: FRow(6000, 96, ("h", 1400), True, True, {"kernel": "tc128", "h": 1400}),
    "ffma_h1401": lambda s: FRow(6000, 96, ("h", 1401), True, True, {"kernel": "tile64", "h": 1401}),
    "tc_band_wider_than_codebook": lambda s: FRow(300, 512, 1e5, True, True, {"kernel": "tc128", "h": 300}),
    "ffma_band_wider_than_codebook": lambda s: FRow(300, 512, 1e5, False, True, {"kernel": "tile128", "h": 300}),
    "tc_partial_tile_misaligned": lambda s: FRow(4100, 50, 40.0, True, False, {"kernel": "tc64"}),
    # the tile kernels' table and ring exceed 200 KB from h = 17 208 at TD = 128: the scalar kernel takes the shape
    "scalar_wide_band_fallback": lambda s: FRow(20000, 128, ("h", 17208), False, True, {"kernel": "scalar", "h": 17208}),
}


def _frow(name):
    return FROWS[name](_sms())


def _assert_plan(p, expect, check, what):
    for f, v in expect.items():
        assert p[f] == v, f"{what}: plan {f} = {p[f]}, expected {v} ({p})"
    if check is not None:
        assert check(p), f"{what}: plan misses the row's edge: {p}"


_WTAB = {}


def device_weights(k, rng):
    """the device's band_weight table w[0..k): the scalar kernel on a unit impulse at row 0 with scale 1"""
    key = (k, rng)
    if key not in _WTAB:
        e = torch.zeros(k, 1, device=DEV)
        e[0, 0] = 1.0
        _WTAB[key] = ops.neighbourhood_filter(e, rng, tensor_cores=False)[:, 0].clone()
    return _WTAB[key]


@pytest.mark.parametrize("name", list(FROWS))
def test_filter_regime_is_exact_on_impulses(name):
    row = _frow(name)
    k, d = row.k, row.d
    rng = row.range()
    p = filter_plan(k, d, rng, row.ws, row.aligned)
    _assert_plan(p, row.expect, row.check, name)
    h = p["h"]
    assert h == ops.filter_half_width(k, rng)
    w = device_weights(k, rng)
    U.check_weight_table(w, rng, h)
    vals, src = U.impulse_case(k, d, h, seed=len(name))
    vin, src = vals.to(DEV), src.to(DEV)
    off = 0 if row.aligned else 1
    buf, flat = _guarded(k * d, off)
    out = flat.view(k, d)
    ops.neighbourhood_filter(vin, rng, scale=SCALE, out=out, tensor_cores=row.ws)
    torch.cuda.synchronize()
    assert _guard_ok(buf, k * d, off), f"{name}: guard band written"
    tc = p["kernel"].startswith("tc")
    if not tc:
        want = U.filter_expected(vin, src, w, SCALE)
        bad = int((out != want).sum())
        assert bad == 0, f"{name}: {bad} of {k * d} elements differ"
        return
    s, sub = U.tc_weights(w)
    want = U.filter_expected(vin, src, s, SCALE)
    t = (torch.arange(k, device=DEV)[:, None] - src.clamp(min=0)).abs()
    in_sub = (src >= 0) & sub[t]
    bad = int(((out != want) & ~in_sub).sum())
    assert bad == 0, f"{name}: {bad} of {k * d} elements differ where hi and lo are normal or zero"
    if bool(in_sub.any()):
        rule = want if SUBNORMAL_RULE == "kept" else U.filter_expected(vin, src, U.tc_weights_flushed(w), SCALE)
        kept = int((out == want)[in_sub].sum())
        n_sub = int(in_sub.sum())
        assert torch.equal(out[in_sub], rule[in_sub]), (
            f"{name}: subnormal tf32 operands are not {SUBNORMAL_RULE}: {kept} of {n_sub} elements match 'kept'")
    # every (unit tile, k-block, chain) whose rows lie inside the codebook carried an impulse
    hits = U.tc_hits(vals, h, p["nkb"], p["q"])
    assert U.tc_all_blocks(k, h, p["nkb"], p["q"]) <= hits
    assert {c for _, _, c in hits} == set(range(p["na"]))


def test_filter_rows_reach_every_kernel():
    seen = set()
    for name in FROWS:
        row = _frow(name)
        p = filter_plan(row.k, row.d, row.range(), row.ws, row.aligned)
        _assert_plan(p, row.expect, row.check, name)
        seen.add(p["kernel"])
        if p["kernel"].startswith("tc"):
            seen.add(("tc", p["ks"] > 1))
            seen.add(("na", p["na"]))
            # the band reaches weights whose TF32 hi or lo is subnormal (the class SUBNORMAL_RULE pins)
            _, sub = U.tc_weights(device_weights(row.k, row.range()))
            seen.add(("subnormal tf32 operand", bool(sub[:min(p["h"], row.k - 1) + 1].any())))
        if p["kernel"] == "scalar":
            seen.add(("scalar opt-in", p["smem"] > 48 * 1024))
    want = set(KERNELS.values()) | {("tc", True), ("tc", False), ("na", 3), ("na", 4), ("scalar opt-in", True),
                                    ("scalar opt-in", False), ("subnormal tf32 operand", True)}
    assert want <= seen, f"unreached: {want - seen}"


def test_filter_wide_band_takes_the_scalar_kernel_until_its_table_does_not_fit():
    """h in [17 208, 25 583] at TD = 128 and [21 304, 25 583] at TD = 64: the scalar kernel; beyond, SOM_E_SHAPE"""
    for d, h_first in ((128, 17208), (64, 21304)):
        k = 60000
        assert filter_plan(k, d, range_for_h(k, h_first - 1), False, True)["kernel"] == ("tile128" if d == 128
                                                                                        else "tile64")
        for h in (h_first, 25583):
            assert filter_plan(k, d, range_for_h(k, h), False, True)["kernel"] == "scalar"
    fn = _hook("som_debug_filter_plan", [ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_int,
                                         ctypes.POINTER(ctypes.c_int64), ctypes.c_int])
    out = (ctypes.c_int64 * len(FILTER_FIELDS))()
    assert fn(60000, 128, range_for_h(60000, 25584), 0, 1, out, len(FILTER_FIELDS)) != 0


# ============================================== accumulation ========================================================
@dataclass
class ARow:
    geom: tuple             # ("nchw", C, pH, pW, gH, gW, n_img) or ("flat", n, D)
    k: int
    expect: dict
    check: object = None
    wt_off: int = 0         # float offset of W~ (1: 4-byte aligned only)
    rbar_off: int = 0
    lim: int = 2

    @property
    def n(self):
        g = self.geom
        return g[1] if g[0] == "flat" else g[4] * g[5] * g[6]

    @property
    def d(self):
        g = self.geom
        return g[2] if g[0] == "flat" else g[1] * g[2] * g[3]

    def ops_geom(self):
        g = self.geom
        if g[0] == "flat":
            return ops.flat_geometry(g[1], g[2])
        _, c, ph, pw, gh, gw, n_img = g
        return n_img, c, gh * ph, gw * pw, ph, pw

    def batch(self, rows):
        g = self.geom
        if g[0] == "flat":
            return rows.contiguous()
        _, c, ph, pw, gh, gw, _ = g
        return L.unpatchify(rows, c, ph, pw, gh, gw)


AROWS = {
    "scan_vec4": ARow(("nchw", 4, 4, 4, 8, 8, 20), 300, {"path": "scan", "vec": 4}),
    "scan_vec2": ARow(("nchw", 3, 2, 2, 16, 16, 7), 1000, {"path": "scan", "vec": 2}),
    "scan_vec1_pw3": ARow(("nchw", 4, 3, 3, 5, 5, 40), 500, {"path": "scan", "vec": 1}),
    "scan_two_slices": ARow(("flat", 700, 1100), 64, {"path": "scan", "vec": 4, "n_slices": 2}),
    "scan_wt_misaligned": ARow(("nchw", 4, 4, 4, 8, 8, 20), 300, {"path": "scan", "vec": 1}, wt_off=1),
    "scan_rbar_misaligned": ARow(("nchw", 4, 4, 4, 8, 8, 20), 300, {"path": "scan", "vec": 1}, rbar_off=1),
    "counting_s16_vec2": ARow(("flat", 40000, 64), 1000, {"path": "counting", "vec": 2, "S": 16, "cs_per": 2048}),
    "counting_s32_rbar_misaligned": ARow(("flat", 40000, 256), 1000, {"path": "counting", "vec": 1, "S": 32},
                                         rbar_off=1),
    "counting_s32_wt_misaligned": ARow(("flat", 40000, 256), 1000, {"path": "counting", "vec": 1, "S": 32}, wt_off=1),
    "counting_wide_blocks": ARow(("nchw", 4, 2, 2, 10, 10, 4000), 5000, {"path": "counting", "vec": 1, "S": 64},
                                 lambda p: p["cs_per"] > 2048),
    "counting_pw3": ARow(("nchw", 2, 3, 3, 4, 4, 300), 2000, {"path": "counting", "vec": 1, "S": 8}),
    "counting_pw4_halved": ARow(("nchw", 4, 4, 4, 8, 8, 100), 3000, {"path": "counting", "vec": 2, "S": 8}),
    "radix_k16385": ARow(("flat", 5000, 128), 16385, {"path": "radix", "vec": 4, "S": 8}),
    "radix_large_batch": ARow(("flat", (1 << 22) + 100, 4), 100, {"path": "radix", "vec": 1, "S": 64}),
}


def _accum_case(row, seed):
    n, d, k = row.n, row.d, row.k
    g = torch.Generator().manual_seed(seed)
    a = torch.randint(-row.lim, row.lim + 1, (n, d), generator=g)
    b = torch.randint(-row.lim, row.lim + 1, (k, d), generator=g)
    return a, b


@pytest.mark.parametrize("name", list(AROWS))
def test_accumulate_regime_is_exact_on_the_lattice(name):
    row = AROWS[name]
    n, d, k = row.n, row.d, row.k
    geom = row.ops_geom()
    e = L.SCALES[len(name) % 3]
    a, b = _accum_case(row, len(name))
    x = row.batch(L.to_float(a, e)).to(DEV)
    wt_buf = torch.empty(k * d + 1, device=DEV)
    wt = wt_buf[row.wt_off:row.wt_off + k * d].view(k, d)
    wt.copy_(L.to_float(b, e))
    rbar_buf, rbar_flat = _guarded(k * d, row.rbar_off)
    p = accum_plan(x.data_ptr(), geom, wt.data_ptr(), k, rbar_flat.data_ptr())
    _assert_plan(p, row.expect, row.check, name)
    if p["path"] != "scan":
        assert p["n_chunks"] == (n + p["S"] - 1) // p["S"]
    bmu = U.segment_bmu(n, k, p["S"] if p["S"] > 0 else 8, seed=len(name))
    U.check_accum_bound(a, b, bmu, k, "scan" if p["path"] == "scan" else "sorted", p["vec"], p["S"])
    ad, bd, bmu_d = a.to(DEV), b.to(DEV), bmu.to(DEV)
    rbar_i, xbar_i, counts_i, sse_i = U.accum_reference(ad, bd, bmu_d, k)
    rbar, counts, sse = ops.accumulate(x, geom, bmu_d, wt, k, want_counts=True, want_sse=True,
                                       out=rbar_flat.view(k, d))
    torch.cuda.synchronize()
    assert _guard_ok(rbar_buf, k * d, row.rbar_off), f"{name}: guard band written"
    bad = int((rbar.double() != L.to_float(rbar_i, e, torch.float64)).sum())
    assert bad == 0, f"{name}: {bad} Rbar elements differ"
    assert torch.equal(counts, counts_i)
    sse_want = float(L.to_float(torch.tensor([sse_i]), 2 * e, torch.float64))
    assert float(sse) == sse_want, f"{name}: sse {float(sse)} != {sse_want}"
    rbar = rbar.clone()
    # plain-sum mode (the autograd backward)
    xbar, _, _ = ops.accumulate(x, geom, bmu_d, None, k, out=rbar_flat.view(k, d))
    assert torch.equal(xbar.double(), L.to_float(xbar_i, e, torch.float64)), f"{name}: plain sums"
    # packed form: [Rbar | sse_hi, sse_lo, n / 4096, n % 4096]
    packed = ops.accumulate_packed(x, geom, bmu_d, wt, k)
    assert torch.equal(packed[:k * d].view(k, d), rbar)
    assert torch.equal(packed[k * d:].cpu(), U.packed_tail(sse_want, n))


def test_accumulate_rows_reach_every_path_width_and_chunk():
    seen = set()
    for name, row in AROWS.items():
        x_ptr, wt_ptr, rbar_ptr = 1 << 20, (1 << 20) + 4 * row.wt_off, (1 << 20) + 4 * row.rbar_off
        p = accum_plan(x_ptr, row.ops_geom(), wt_ptr, row.k, rbar_ptr)
        _assert_plan(p, row.expect, row.check, name)
        seen.add((p["path"], p["vec"]))
        seen.add(("S", p["S"]))
        if p["path"] == "counting":
            seen.add(("cs_per > 2048", p["cs_per"] > 2048))
        if p["path"] == "radix":
            seen.add(("radix", row.k > 16384, row.n > 1 << 22))
        if row.geom[0] == "nchw":
            seen.add(("pW", row.geom[3]))
        seen.add(("misaligned", p["path"] == "scan", row.wt_off, row.rbar_off))
    want = {("scan", 4), ("scan", 2), ("scan", 1), ("counting", 2), ("counting", 1), ("radix", 4), ("radix", 1),
            ("S", 8), ("S", 16), ("S", 32), ("S", 64), ("cs_per > 2048", True), ("cs_per > 2048", False),
            ("radix", True, False), ("radix", False, True), ("pW", 2), ("pW", 3), ("pW", 4),
            ("misaligned", True, 1, 0), ("misaligned", True, 0, 1), ("misaligned", False, 1, 0),
            ("misaligned", False, 0, 1)}
    assert want <= seen, f"unreached: {want - seen}"


# =========================================== one-kernel step =======================================================
# (D, R, h, images): K = (R - 1) s + 7 units (ceil(K / s) = R rows per CTA), h = "max" for the widest band the staged
# rows allow, images of side `side`
SIDE = {16: 24, 32: 32, 64: 20, 128: 16, 256: 24}
GEOM = {16: (4, 2), 32: (2, 4), 64: (4, 4), 128: (8, 4), 256: (4, 8)}
SROWS = {
    "d16_h0": (16, 7, 0, 5),
    "d16_hmax": (16, 14, "max", 5),
    "d32_slot0_n2048": (32, 11, 30, 32),
    "d32_slot1_hmax": (32, 21, "max", 3),
    "d64_slot0": (64, 7, 0, 9),
    "d64_slot1_hmax": (64, 28, "max", 7),
    "d128_slot0_hmax": (128, 4, "max", 11),
    "d128_slot1": (128, 11, 0, 5),
    "d128_slot2_hmax": (128, 28, "max", 3),
    "d256_slot0": (256, 2, 0, 3),
    "d256_slot1": (256, 7, 10, 5),
    "d256_slot2_hmax": (256, 32, "max", 1),
}


def _srow(name):
    d, r, h, n_img = SROWS[name]
    s = _sms()
    k = (r - 1) * s + 7
    c, p = GEOM[d]
    side = SIDE[d]
    if h == "max":
        h = min((32768 // d - r) // 2, 2048, k)
    rng = range_for_h(k, h)
    return d, k, h, rng, (n_img, c, side, side, p, p)


def _composed_step(x, geom, w, m, v, t, rng, bmu, lr):
    """the step from the separate kernels: scalar filter (4-byte offset out), scan accumulation, the scalar filter of
    Rbar with scale fl32(2 / numel), adam_step_dev"""
    k, d = w.shape
    wt_buf = torch.empty(k * d + 1, device=DEV)
    wt = wt_buf[1:].view(k, d)
    ops.neighbourhood_filter(w, rng, out=wt, tensor_cores=False)
    rbar, _, sse = ops.accumulate(x, geom, bmu, wt, k, want_sse=True)
    g_buf = torch.empty(k * d + 1, device=DEV)
    g = g_buf[1:].view(k, d)
    ops.neighbourhood_filter(rbar, rng, scale=2.0 / x.numel(), out=g, tensor_cores=False)
    ops.adam_step_dev(w, m, v, g.clone(), lr, t)
    return float(sse)


@pytest.mark.parametrize("arm", ["lattice", "tanh"])
@pytest.mark.parametrize("name", list(SROWS))
def test_one_kernel_step_is_bit_identical_to_the_scalar_composition(name, arm):
    d, k, h, rng, geom = _srow(name)
    n = ops.n_patches_of(geom)
    p = step_plan(n, d, k, rng)
    assert p is not None and p["h"] == h, f"{name}: plan {p}"
    assert p["R"] == SROWS[name][1]
    c, ph = GEOM[d]
    side = SIDE[d]
    g = torch.Generator().manual_seed(k + d)
    if arm == "lattice":
        a, b = L.lattice_ints(n, d, k, "narrow", seed=k + d)
        L.check_bound(a, b)
        rows = L.to_float(a, 0)
        w0 = L.to_float(b, 0)
    else:
        rows = torch.tanh(torch.randn(n, d, generator=g))
        w0 = 0.5 * torch.tanh(torch.randn(k, d, generator=g))
    x = L.unpatchify(rows, c, ph, ph, side // ph, side // ph).to(DEV)
    w1, w2 = w0.clone().to(DEV), w0.clone().to(DEV)
    m1, v1 = torch.zeros_like(w1), torch.zeros_like(w1)
    m2, v2 = torch.zeros_like(w1), torch.zeros_like(w1)
    t1 = torch.zeros(1, dtype=torch.int64, device=DEV)
    t2 = torch.zeros(1, dtype=torch.int64, device=DEV)
    lr = 1e-2
    for step in range(3):
        r = rng * 0.5 ** step
        loss, bmu = ops.step_small(x, geom, w1, m1, v1, r, lr, t1)
        if step == 0 and arm == "lattice":
            ref, _ = L.fp64_bmu(rows.to(DEV), w0.to(DEV))
            assert torch.equal(bmu, ref), f"{name}: {int((bmu != ref).sum())} BMUs differ from the fp64 argmin"
        sse = _composed_step(x, geom, w2, m2, v2, t2, r, bmu, lr)
        tag = f"{name} {arm} step {step}"
        assert torch.equal(w1, w2), f"{tag}: W differs ({int((w1 != w2).sum())} elements)"
        assert torch.equal(m1, m2) and torch.equal(v1, v2), f"{tag}: moments differ"
        assert int(t1[0]) == int(t2[0]) == step + 1
        numel = x.numel()
        if step == 0 and arm == "lattice" and h == 0:
            # W~ = W: every residual is an integer, and the squared error of every CTA stays below 2^24
            res = (b[bmu.cpu()] - a)
            sse_exact = int((res * res).sum())
            assert sse_exact < 1 << 24
            assert float(loss) == sse_exact * (1.0 / numel), f"{tag}: loss {float(loss)} vs {sse_exact / numel}"
            assert sse == float(sse_exact)
        else:
            assert abs(float(loss) - sse / numel) <= 2e-6 * abs(sse / numel), f"{tag}: loss"


def test_step_rows_reach_every_instantiation():
    """(D, RBCAP slot) pairs the one-kernel step can run on this part, from the hook, against the rows"""
    s = _sms()
    reach = set()
    for d in (16, 32, 64, 128, 256):
        for r in range(1, 40):
            p = step_plan(64, d, (r - 1) * s + 7, 0.01)
            if p is not None:
                reach.add((d, p["slot"]))
    rows = set()
    for name in SROWS:
        d, k, h, rng, geom = _srow(name)
        p = step_plan(ops.n_patches_of(geom), d, k, rng)
        rows.add((d, p["slot"]))
    assert reach == rows, f"unreached: {reach - rows}"
    assert len(reach) >= 11 if s == 148 else len(reach) > 0
    # the rows' own edges: h = 0 and the widest staged band, n = 2048 and n % 64 != 0, K % R != 0 and K % 64 != 0
    edges = set()
    for name in SROWS:
        d, k, h, rng, geom = _srow(name)
        n = ops.n_patches_of(geom)
        p = step_plan(n, d, k, rng)
        edges.add(("h = 0", h == 0))
        edges.add(("widest band", (p["R"] + 2 * (h + 1)) * d > 32768 or h == k))
        edges.add(("n = 2048", n == 2048))
        edges.add(("n % 64", n % 64 != 0))
        assert k % p["R"] != 0 and k % 64 != 0, name
    assert all((e, True) in edges for e in ("h = 0", "widest band", "n = 2048", "n % 64")), edges
