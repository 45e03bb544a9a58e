"""Every BMU kernel regime against an exact fp64 argmin, at its edge shapes, with zero tolerance.

Which kernel runs depends on n, D, K, the SM count and the element type (csrc/som_bmu.cu, som_bmu_tc.cu and the
planners of som_bmu_tc_l.cu / som_bmu_tc_l16.cu / som_bmu_tc_s.cu).  Each row of ROWS names a regime; the row first
asserts through som_debug_bmu_plan that its shape reaches it on this part, then runs every variant that covers the
shape on exact-lattice inputs (tests/_lattice.py): each must return the lowest-index fp64 argmin and the exact reduced
distance, bit for bit.  L16 rows repeat the narrow lattice as fp16 and bf16 batches on the native kernel.  A row also
checks the guard bands around every output and the workspace, the staging copy, a 64-bit unit offset, a 3-way uneven
unit-shard merge, and real-valued (tanh) data against fp64 with the usual parity rule.  The last test asserts that the
rows together still reach every kernel instantiation and mode, so the matrix cannot shrink silently."""
import ctypes
from dataclasses import dataclass

import pytest
import torch

from somcb import _lib, ops
from _helpers import assert_bmu_parity
import _lattice as L

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

FIELDS = ("family", "arith", "cg", "merged", "mode", "S", "fb_per_split", "U", "chunk_rows", "NT", "DB", "Rr",
          "mtiles")                                        # csrc/som_common.cuh: PlanField
FAMILY = {0: "FFMA", 1: "S", 2: "L16", 3: "L"}
MODE = {0: "splitk", 1: "resident", 2: "streamed"}
ELEMS = (torch.float32, torch.float16, torch.bfloat16)
AUTO, FFMA, TC3X, TC_TF32, TC_F16 = (ops.SOM_BMU_AUTO, ops.SOM_BMU_FFMA, ops.SOM_BMU_TC3X, ops.SOM_BMU_TC_TF32,
                                     ops.SOM_BMU_TC_F16)


def plan(n, d, k, variant=AUTO):
    """The plan som_debug_bmu_plan reports (dict, family / mode as names), or None where the variant has no kernel."""
    fn = _lib.load().som_debug_bmu_plan
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int64),
                   ctypes.c_int]
    out = (ctypes.c_int64 * len(FIELDS))()
    if fn(n, d, k, variant, out, len(FIELDS)) != 0:
        return None
    p = dict(zip(FIELDS, list(out)))
    p["family"] = FAMILY[p["family"]]
    p["mode"] = MODE.get(p["mode"], None)
    return p


@dataclass
class Row:
    geom: tuple            # ("nchw", C, pH, pW, gH, gW, n_img) or ("flat", n, D)
    k: int
    variant: int
    expect: dict           # plan fields the row is about
    check: object = None   # extra predicate on the plan (the row's edge: odd tiles, ragged splits, chunks)

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
        """(n, D) patch rows -> the batch this row's geometry reads them from"""
        g = self.geom
        if g[0] == "flat":
            return rows.contiguous()
        _, c, ph, pw, gh, gw, _ = g
        return L.unpatchify(rows, c, ph, pw, gh, gw)


def _odd_ragged(p):
    return p["mtiles"] % 2 == 1


# Shapes follow the SM count `s` of the part (148 on a B200); the comments give the values at 148.
ROWS = {
    # D <= 16 below 4096 patches: FFMA (n = 3000, pW = 2)
    "ffma_d16": lambda s: Row(("nchw", 4, 2, 2, 5, 5, 120), 4096, AUTO, {"family": "FFMA"}),
    # K * D < 16 384: FFMA at any size (flat, D = 2048, K = 7)
    "ffma_tiny_codebook": lambda s: Row(("flat", 500, 2048), 7, AUTO, {"family": "FFMA"}),
    # config S, TF32, fewer resident tiles than R = 4 (5000 patches), ragged K
    "s_tf32_partial_rr": lambda s: Row(("nchw", 4, 2, 2, 5, 5, 200), 4093, AUTO, {"family": "S", "arith": 0},
                                       lambda p: p["Rr"] < 4),
    # config S, FP16 from 65 536 patches, ragged tail (65 616 = 512 * 128 + 80), pW = 3
    "s_fp16_ragged": lambda s: Row(("nchw", 1, 4, 3, 3, 4, 5468), 3000, AUTO, {"family": "S", "arith": 1},
                                   lambda p: p["mtiles"] * 128 != 65616),
    # config S, FP16 forced on a small flat batch of D = 3
    "s_fp16_forced": lambda s: Row(("flat", 300, 3), 20000, TC_F16, {"family": "S", "arith": 1}),
    # L16: one wave of tiles (s + 1, the last half full), D = 20 (a partial 16-wide k-step), single CTAs, merged ring
    "l16_one_wave": lambda s: Row(("nchw", 5, 2, 2, 8, 8, 2 * s + 1), 1100, AUTO,
                                  {"family": "L16", "cg": 1, "merged": 1, "DB": 1}),
    # L16: CTA pairs on an odd, ragged tile count (2 s + 1 tiles, the last one half full), D = 128 (C = 8, P = 4)
    "l16_pairs_odd_tiles": lambda s: Row(("nchw", 8, 4, 4, 8, 8, 4 * s + 1), 4096, AUTO,
                                         {"family": "L16", "cg": 2, "merged": 1, "DB": 2}, _odd_ragged),
    # L16: DB = 3 (four slots), pairs, 2 s + 5 tiles with a ragged last one, ragged K, pW = 3
    "l16_db3_pairs": lambda s: Row(("nchw", 16, 4, 3, 4, 8, 8 * s + 19), 2000, AUTO,
                                   {"family": "L16", "cg": 2, "merged": 0, "DB": 3}, _odd_ragged),
    # L16 forced: 379 patches = 3 tiles -> the second CTA of the last pair has no rows; D = 200 (D % 16 = 8), flat
    "l16_forced_empty_peer": lambda s: Row(("flat", 3 * 128 - 5, 200), 1000, TC_F16,
                                           {"family": "L16", "cg": 2, "merged": 0, "DB": 4, "mtiles": 3}),
    # L16 forced: one tile, four slots on a single CTA, D = 256
    "l16_four_slots_single": lambda s: Row(("nchw", 64, 2, 2, 5, 5, 4), 1024, TC_F16,
                                           {"family": "L16", "cg": 1, "merged": 0, "DB": 4}),
    # L16: K > 32 768 (separate codebook-scale kernel), ragged K (40 000 = 156.25 tiles)
    "l16_big_k": lambda s: Row(("nchw", 4, 4, 4, 8, 8, 2 * (s + 12)), 40000, AUTO,
                               {"family": "L16", "cg": 1, "merged": 1, "NT": 157}),
    # L16: pairs, merged, D = 96 with pW = 1 (scalar builder loads)
    "l16_pairs_d96": lambda s: Row(("nchw", 24, 4, 1, 8, 32, s + 2), 16384, AUTO,
                                   {"family": "L16", "cg": 2, "merged": 1, "DB": 2}),
    # 3xTF32 resident-A with unit splits, the last split shorter
    "l_resident_unit_split": lambda s: Row(("nchw", 4, 4, 4, 5, 5, 80), 5000, AUTO,
                                           {"family": "L", "mode": "resident", "cg": 1},
                                           lambda p: p["U"] > 1 and p["NT"] % p["U"] != 0),
    # 3xTF32 resident-A with CTA pairs (NT = 3: no FP16-split kernel under the rule), odd ragged tiles, D = 48 flat
    "l_resident_pairs": lambda s: Row(("flat", (2 * s + 4) * 128 + 9, 48), 700, AUTO,
                                      {"family": "L", "mode": "resident", "cg": 2, "U": 1, "NT": 3}, _odd_ragged),
    # 3xTF32 resident-A, single CTAs, D = 36 (pW = 3, a 4-feature last block)
    "l_resident_single": lambda s: Row(("nchw", 4, 3, 3, 10, 10, 100), 1500, AUTO,
                                       {"family": "L", "mode": "resident", "cg": 1, "U": 1, "S": 1}),
    # 3xTF32 streamed, one chunk, unit splits
    "l_streamed_one_chunk": lambda s: Row(("nchw", 10, 4, 4, 5, 5, 40), 4000, AUTO,
                                          {"family": "L", "mode": "streamed", "S": 1},
                                          lambda p: p["U"] > 1 and p["chunk_rows"] >= 1000),
    # 3xTF32 streamed over several pre-split chunks (the last ragged), CTA pairs, odd tiles, D = 320 with pW = 2
    "l_streamed_chunks": lambda s: Row(("nchw", 40, 4, 2, 8, 16, 2 * s + 5), 2048, AUTO,
                                       {"family": "L", "mode": "streamed", "cg": 2, "U": 1},
                                       lambda p: (p["chunk_rows"] < (2 * s + 5) * 128
                                                  and ((2 * s + 5) * 128) % p["chunk_rows"] != 0 and _odd_ragged(p))),
    # 3xTF32 split-K at the C3 shape (4096 patches, D = 4096, K = 512), pW = 2
    "l_splitk_c3": lambda s: Row(("nchw", 1024, 2, 2, 8, 8, 64), 512, AUTO, {"family": "L", "mode": "splitk"},
                                 lambda p: p["S"] > 1),
    # 3xTF32 split-K, D = 1102 flat: 35 blocks in splits of 9, 9, 9, 8, a 14-feature last block, pair-wise loads
    "l_splitk_partial_block": lambda s: Row(("flat", 200, 1102), 777, AUTO,
                                            {"family": "L", "mode": "splitk", "DB": 35},
                                            lambda p: p["S"] > 1 and 35 % p["fb_per_split"] != 0),
    # 3xTF32 split-K at D = 8192 (eight splits on 148 SMs)
    "l_splitk_d8192": lambda s: Row(("nchw", 2048, 2, 2, 4, 4, 4), 300, AUTO, {"family": "L", "mode": "splitk"},
                                    lambda p: p["S"] > 1),
    # the 256 MB cap on the partial-distance buffer: no feature split, streamed with unit splits, pW = 1
    "l_splitk_cap": lambda s: Row(("nchw", 128, 4, 1, 4, 16, s), 32768, AUTO,
                                  {"family": "L", "mode": "streamed", "S": 1}, lambda p: p["U"] > 1),
}


def _row(name):
    return ROWS[name](ops.device_info()[0])


def _assert_plan(row, p, what=""):
    assert p is not None, f"{what}: no kernel"
    for f, v in row.expect.items():
        assert p[f] == v, f"{what}: plan {f} = {p[f]}, expected {v} ({p})"
    if row.check is not None:
        assert row.check(p), f"{what}: plan misses the row's edge: {p}"


def _variants(row):
    """FFMA, the tensor-core dispatch, 3xTF32 forced, and the FP16 split where a kernel of it covers the shape."""
    vs = [FFMA]
    if plan(row.n, row.d, row.k, TC3X) is not None:
        vs += [TC3X, TC_TF32]
        if plan(row.n, row.d, row.k, TC_F16) is not None:
            vs.append(TC_F16)
    if row.variant not in vs and row.variant != AUTO:
        vs.append(row.variant)
    return vs


def _lattice(row, kind, seed):
    a, b = L.lattice_ints(row.n, row.d, row.k, kind, seed)
    try:
        L.check_bound(a, b)
    except AssertionError:
        return None
    e = L.SCALES[seed % 3]
    rows = L.to_float(a, e)
    return row.batch(rows).to(DEV), rows.to(DEV), L.to_float(b, e).to(DEV)


def _guarded_call(row, x, w, cn, variant):
    """The raw C-ABI with idx, rd, the staging copy and the workspace inside sentinel-filled buffers."""
    lib = _lib.load()
    n, d, k = row.n, row.d, row.k
    guard = 4096
    st = torch.cuda.current_stream().cuda_stream
    ws_bytes = lib.som_bmu_workspace_bytes(n, d, k, variant)
    ws_big = torch.full((ws_bytes + 2 * guard + 256,), 0x5A, dtype=torch.uint8, device=DEV)
    ws_ptr = (ws_big.data_ptr() + guard + 255) // 256 * 256
    off = ws_ptr - ws_big.data_ptr()
    idx_big = torch.full((n + 2 * 512,), -777, dtype=torch.int64, device=DEV)
    rd_big = torch.full((n + 2 * 512,), -777.0, dtype=torch.float32, device=DEV)
    can_stage = bool(lib.som_bmu_can_stage(n, d, k, variant))
    stage_big = torch.full((n * d + 2 * 1024,), -777.0, dtype=torch.float32, device=DEV) if can_stage else None
    rc = lib.som_bmu_stage_nchw_f32(x.data_ptr(), *row.ops_geom(), w.data_ptr(), cn.data_ptr(), k, 0,
                                    idx_big.data_ptr() + 512 * 8, rd_big.data_ptr() + 512 * 4,
                                    stage_big.data_ptr() + 1024 * 4 if can_stage else None,
                                    ws_ptr if ws_bytes else None, ws_bytes, variant, st)
    assert rc == 0, lib.som_last_error()
    torch.cuda.synchronize()
    assert bool((idx_big[:512] == -777).all()) and bool((idx_big[512 + n:] == -777).all()), "idx guard band"
    assert bool((rd_big[:512] == -777.0).all()) and bool((rd_big[512 + n:] == -777.0).all()), "rd guard band"
    assert bool((ws_big[:off] == 0x5A).all()) and bool((ws_big[off + ws_bytes:] == 0x5A).all()), "workspace guard"
    stage = None
    if can_stage:
        assert bool((stage_big[:1024] == -777.0).all()) and bool((stage_big[1024 + n * d:] == -777.0).all())
        stage = stage_big[1024:1024 + n * d].reshape(n, d)
    return idx_big[512:512 + n], rd_big[512:512 + n], stage


@pytest.mark.parametrize("name", list(ROWS))
def test_regime_is_exact_on_the_lattice(name):
    row = _row(name)
    geom = row.ops_geom()
    _assert_plan(row, plan(row.n, row.d, row.k, row.variant), name)
    ran = 0
    for kind, seed in (("narrow", 1), ("wide", 2)):
        case = _lattice(row, kind, seed + len(name))
        if case is None:
            assert kind == "wide", "the narrow lattice must fit the bound at every shape"
            continue
        x, flat, w = case
        ref, ref_rd = L.fp64_bmu(flat, w)
        if kind == "narrow":
            # the 16-bit and guarded runs below use this case only: its answers must depend on x
            assert L.zero_unit_share(flat, w, ref) <= L.MAX_ZERO_SHARE, f"{name}: degenerate narrow lattice"
        cn = ops.prepare_codebook(w)
        for v in _variants(row):
            idx, rd = ops.bmu(x, geom, w, cn, want_rd=True, variant=v)
            bad = int((idx != ref).sum())
            assert bad == 0, f"{name} {kind} variant {v}: {bad} of {row.n} indices differ from the fp64 argmin"
            assert torch.equal(rd.double(), ref_rd), (
                f"{name} {kind} variant {v}: rd differs ({int((rd.double() != ref_rd).sum())} rows)")
            ran += 1
        if kind != "narrow":
            continue
        if plan(row.n, row.d, row.k, row.variant)["family"] == "L16":
            for dt in (torch.float16, torch.bfloat16):
                assert ops.bmu_f16_native(geom, row.k, row.variant)
                idx, rd = ops.bmu(x.to(dt), geom, w, cn, want_rd=True, variant=row.variant)
                assert torch.equal(idx, ref) and torch.equal(rd.double(), ref_rd), f"{name} {dt}"
        # guard bands and the staging copy, on the row's own dispatch
        v = row.variant
        idx, rd, stage = _guarded_call(row, x, w, cn, v)
        assert torch.equal(idx, ref) and torch.equal(rd.double(), ref_rd), f"{name}: guarded call"
        if stage is not None:
            assert torch.equal(stage, flat), f"{name}: staging copy != patchify(x)"
        # a 64-bit unit offset comes back exactly
        off = 3 << 31
        idx = ops.bmu(x, geom, w, cn, unit_offset=off, variant=v)
        assert torch.equal(idx, ref + off), f"{name}: unit_offset"
        # a 3-way uneven unit-shard split (each shard may land in another regime) merged == the unsharded answer
        k = row.k
        cuts = [0, k // 7 + 1, k // 7 + 1 + k // 2, k]
        rds, idxs = [], []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            i, r = ops.bmu(x, geom, w[lo:hi].contiguous(), unit_offset=lo, want_rd=True)
            rds.append(r)
            idxs.append(i)
        m_idx, m_rd = ops.merge_candidates(torch.stack(rds), torch.stack(idxs))
        assert torch.equal(m_idx, ref) and torch.equal(m_rd.double(), ref_rd), f"{name}: shard merge"
    assert ran >= 2


@pytest.mark.parametrize("name", list(ROWS))
def test_regime_on_real_valued_data(name):
    """tanh data against a codebook of noisy data rows: the fp64 argmin with the parity rule of _helpers.  The noise
    keeps BMU distances within an order of magnitude of ||c||: an fp32 rd resolves distances only to ~2^-24 ||c||^2, so
    a codebook much closer to its data than that holds near ties no fp32 kernel can order to 1e-6 (seen with FFMA at
    D = 512, K = 32 768 and noise 0.05, where rows drawn twice from the data compete)."""
    row = _row(name)
    g = torch.Generator(device=DEV).manual_seed(row.n + row.k)
    flat = torch.tanh(torch.randn(row.n, row.d, generator=g, device=DEV))
    pick = torch.randint(0, row.n, (row.k,), generator=g, device=DEV)
    w = (flat[pick] + 0.25 * torch.randn(row.k, row.d, generator=g, device=DEV)).contiguous()
    x = row.batch(flat)
    ref, _ = L.fp64_bmu(flat, w)
    flat_c, w_c, ref_c = flat.cpu(), w.cpu(), ref.cpu()
    for v in _variants(row):
        idx = ops.bmu(x, row.ops_geom(), w, variant=v)
        n_bad = assert_bmu_parity(idx, ref_c, flat_c, w_c)
        assert n_bad <= max(1, row.n // 20000), f"{name} variant {v}: {n_bad} mismatches"


@pytest.mark.parametrize("p,k,n_f,rng", [(4, 1024, 8, 512), (2, 512, 4, 256), (8, 300, 16, 32), (4, 4096, 8, 512),
                                         (4, 1024, 32, 100)])
def test_one_kernel_step_bmu_is_exact_on_the_lattice(p, k, n_f, rng):
    """The BMU phase of som_step_small_f32 (the first shape is BASELINE config 1) on the narrow lattice."""
    pd, d = (p, p), 4 * p * p
    geom = ops.geometry((n_f, 4, 32, 32), pd)
    assert ops.step_small_supported(geom, k, rng)
    n = ops.n_patches_of(geom)
    a, b = L.lattice_ints(n, d, k, "narrow", seed=p * k)
    L.check_bound(a, b)
    rows, w = L.to_float(a, 0).to(DEV), L.to_float(b, 0).to(DEV)
    ref, _ = L.fp64_bmu(rows, w)
    assert L.zero_unit_share(rows, w, ref) <= L.MAX_ZERO_SHARE
    x = L.unpatchify(rows, 4, p, p, 32 // p, 32 // p)
    wt = w.clone()
    m, v = torch.zeros_like(wt), torch.zeros_like(wt)
    steps = torch.zeros(2, dtype=torch.int64, device=DEV)
    _, idx = ops.step_small(x, geom, wt, m, v, rng, 1e-4, steps)
    assert torch.equal(idx, ref), f"{int((idx != ref).sum())} of {n} BMUs differ from the fp64 argmin"


def test_rows_reach_every_instantiation_and_mode():
    """The table above, read through the planners on this part: all 12 FP16-split instantiations and every listed
    3xTF32 / config-S / FFMA plan.  Merged ring x CTA pair come from the planner.  The element-type axis does not enter
    any planner: every L16 row is asserted to read 16-bit batches natively (som_bmu_f16_native), and
    test_regime_is_exact_on_the_lattice runs each such row as fp32, fp16 and bf16, so each row reaches one
    (merged, cg) instantiation for all three element types."""
    sms = ops.device_info()[0]
    assert sms % 2 == 0, "CTA pairs need an even SM count"
    l16, seen = set(), set()
    for name in ROWS:
        row = ROWS[name](sms)
        p = plan(row.n, row.d, row.k, row.variant)
        _assert_plan(row, p, name)
        if p["family"] == "L16":
            assert ops.bmu_f16_native(row.ops_geom(), row.k, row.variant), name
            l16.update((t, p["merged"], p["cg"]) for t in ELEMS)
        if p["family"] == "L":
            seen.add(("L", p["mode"], p["cg"], p["S"] > 1, p["U"] > 1,
                      p["mode"] == "streamed" and p["chunk_rows"] < row.n))
        if p["family"] == "S":
            seen.add(("S", p["arith"], row.variant == TC_F16))
        if p["family"] == "FFMA":
            seen.add(("FFMA", row.d <= 16))
    assert l16 == {(t, m, c) for t in ELEMS for m in (0, 1) for c in (1, 2)}, sorted(map(str, l16))
    want = {("L", "splitk", 1, True, False, False),              # split-K
            ("L", "resident", 1, False, True, False),            # resident-A, unit splits
            ("L", "resident", 2, False, False, False),           # resident-A, CTA pairs
            ("L", "resident", 1, False, False, False),           # resident-A, single CTAs
            ("L", "streamed", 1, False, True, False),            # streamed, one chunk, unit splits
            ("L", "streamed", 2, False, False, True),            # streamed, several chunks, CTA pairs
            ("S", 0, False), ("S", 1, False), ("S", 1, True),    # config S: TF32, FP16 by the rule, FP16 forced
            ("FFMA", True), ("FFMA", False)}
    assert want <= seen, f"unreached: {want - seen}"
