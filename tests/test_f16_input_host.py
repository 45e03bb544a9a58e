"""fp16 feature maps on the host side: a numpy emulation of the FP16-split kernel's row scale (csrc/som_bmu_tc_l16.cu)
on binary16 input with the per-tile "lo is non-zero" flag, and the version-2 (fp16) feature-map shards.

The emulation pins the claim the skipped A_lo x B_hi product group rests on: where the flag is clear every lo operand
is exactly zero, so the two-product sum equals the three-product sum, whatever the rows hold."""
import json
import os
import struct

import numpy as np
import pytest

from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
from _helpers import flat_patches

F32, F16 = np.float32, np.float16


def _codebook_scales(w):
    """(s_c, exponent of t_c) as scales_from_max_norm derives them from max ||c||^2"""
    mn = np.float32((w.astype(F32) ** 2).sum(1).max())
    en = int((mn.view(np.uint32) >> 23) & 0xFF)
    e = g = 0
    if mn > 0 and en not in (0, 0xFF):
        e2 = en - 127
        e = max(-60, min(60, 7 - (e2 >> 1)))
        g = max(-60, min(60, 14 - (e2 + e)))
    return F32(2.0 ** e), g


def _row_scale(v, tc_exp):
    """s_p of the builders for fp32 rows v (n, D): max |s_p x| in [64, 128) unless a_p = s_p / t_c leaves FP16"""
    mx = np.fmax.reduce(np.abs(v), axis=1, initial=F32(0))          # fmaxf drops NaN
    eb = ((mx.view(np.uint32) >> 23) & 0xFF).astype(np.int64)
    ep = 133 - eb
    ep[~(mx > 0) | (eb == 0xFF)] = 0
    ka = ep - tc_exp
    far = ka < -24
    ka = np.minimum(ka, 15)
    es = np.clip(np.where(far, ep, ka + tc_exp), -120, 120)
    return np.ldexp(F32(1), es).astype(F32)


def _emulate(x16, w):
    """Per 128-row tile and 64-feature block: (flag, three-product sum, two-product sum) of the patch-unit products,
    exactly as the kernel forms hi / lo from the upcast fp16 rows (products exact, sums in fp64)."""
    v = x16.astype(F32)
    sc, tc_exp = _codebook_scales(w)
    with np.errstate(invalid="ignore", over="ignore"):
        s = v * _row_scale(v, tc_exp)[:, None]                      # exact: power-of-two scale
        h = s.astype(F16).astype(F32)
        lo = s - h
        ah, al = h.astype(F16), lo.astype(F16)
        b = F32(-2) * sc * w.astype(F32)
        bh = b.astype(F16)
        bl = (b - bh.astype(F32)).astype(F16)
    out = []
    for r0 in range(0, v.shape[0], 128):
        for f0 in range(0, v.shape[1], 64):
            rs, fs = slice(r0, r0 + 128), slice(f0, f0 + 64)
            flag = bool((lo[rs, fs] != 0).any() | np.isnan(lo[rs, fs]).any())
            a_h, a_l = ah[rs, fs].astype(np.float64), al[rs, fs].astype(np.float64)
            b_h, b_l = bh[:, fs].astype(np.float64), bl[:, fs].astype(np.float64)
            with np.errstate(invalid="ignore", over="ignore"):
                two = a_h @ b_h.T + a_h @ b_l.T
                three = a_h @ b_h.T + a_l @ b_h.T + a_h @ b_l.T
            if not flag:
                assert not np.any(al[rs, fs].astype(np.float64)), "flag clear but a lo operand is non-zero"
            out.append((flag, three, two))
    return out


def _special_rows(d):
    """One row of each kind the scale rule treats differently (fp16 values)."""
    rng = np.random.default_rng(3)
    rows = [np.tanh(rng.standard_normal(d))]
    for mag in (1e-6, 1e-3, 1.0, 100.0, 127.9, 128.0, 1e3, 6e4):
        rows.append(rng.uniform(-mag, mag, d))
    sub = np.float16(2.0 ** -24) * rng.integers(-1023, 1024, d)      # fp16 subnormals
    rows.append(sub)
    rows.append(np.where(rng.random(d) < 0.5, 65504.0, -65504.0))
    wide = rng.uniform(-1, 1, d)
    wide[0], wide[1] = 6e4, 2.0 ** -24                                # large max, tiny entries: lo of the tiny ones
    rows.append(wide)
    rows.append(np.zeros(d))
    r = np.tanh(rng.standard_normal(d)); r[5] = np.nan
    rows.append(r)
    r = np.tanh(rng.standard_normal(d)); r[7] = np.inf
    rows.append(r)
    r = np.tanh(rng.standard_normal(d)); r[9] = -np.inf
    rows.append(r)
    return np.stack(rows).astype(F16)


@pytest.mark.parametrize("d", [32, 64, 256])
def test_tanh_tiles_take_the_two_product_path(d):
    pd = {32: (4, 2), 64: (4, 4), 256: (8, 8)}[d]
    x = flat_patches(synthetic_fmaps(4, 11), pd).numpy().astype(F16)[:512]
    w = trained_like_codebook(512, pd, 7).numpy()
    for flag, three, two in _emulate(x, w):
        assert not flag, "a tile of tanh-range fp16 rows keeps the third product"
        assert np.array_equal(three, two)


@pytest.mark.parametrize("mixed", [False, True])
def test_flag_clear_means_exactly_zero_lo(mixed):
    d = 64
    special = _special_rows(d)
    tanh = flat_patches(synthetic_fmaps(1, 2), (4, 4)).numpy().astype(F16)
    w = trained_like_codebook(512, (4, 4), 7).numpy()
    if mixed:
        x = np.concatenate([tanh[:128 - len(special)], special])      # one tile mixing every kind of row
    else:
        x = np.concatenate([np.repeat(r[None], 128, 0) for r in special])   # one tile per kind
    res = _emulate(x, w)
    flags = [f for f, _, _ in res]
    for flag, three, two in res:
        if not flag:
            assert np.array_equal(three, two)
    if mixed:
        assert flags == [True], "the non-finite / wide rows must keep the tile's third product"
    else:
        kinds = ["tanh", 1e-6, 1e-3, 1.0, 100.0, 127.9, 128.0, 1e3, 6e4, "sub", "65504", "wide", "zero",
                 "nan", "inf", "-inf"]
        by_kind = dict(zip(kinds, flags))
        for k in ("tanh", 1e-6, 1e-3, 1.0, 100.0, 127.9, "sub", "zero"):
            assert not by_kind[k], f"{k} rows should be exact in FP16 after the row scale"
        for k in ("wide", "nan", "inf", "-inf"):
            assert by_kind[k], f"{k} rows must keep the third product"


# ---- fp16 shards -------------------------------------------------------------------------------------------------

def test_shard_v1_is_byte_identical_and_v2_round_trips(tmp_path):
    from somcb import fmap_shards as fs
    x = synthetic_fmaps(5, 1).numpy()
    p1 = str(tmp_path / "a.shard")
    fs.write_shard(p1, x)
    head = b"SOMFMAP1" + struct.pack("<IIIIQ", 1, 4, 32, 32, 5)
    want = head + b"\0" * (64 - len(head)) + x.astype(np.float32).tobytes()
    assert open(p1, "rb").read() == want
    assert fs.read_header(p1) == (4, 32, 32, 5) and fs.shard_dtype(p1) == np.float32

    p2 = str(tmp_path / "b.shard")
    fs.write_shard(p2, x, dtype=np.float16)
    raw = open(p2, "rb").read()
    assert struct.unpack("<I", raw[8:12])[0] == 2 and struct.unpack("<I", raw[32:36])[0] == 1
    assert len(raw) == 64 + x.size * 2
    assert fs.read_header(p2) == (4, 32, 32, 5) and fs.shard_dtype(p2) == np.float16
    r = fs.ShardReader([p2], batch_fmaps=2, pin=False)
    got = np.concatenate([t.numpy().copy() for _, _, t in r.batches()])     # staging slots are reused
    assert got.dtype == np.float16 and np.array_equal(got, x.astype(np.float16))
    assert np.array_equal(r.read_all().numpy(), x.astype(np.float16))

    with pytest.raises(ValueError, match="dtype"):
        fs.ShardReader([p1, p2], pin=False)
    with pytest.raises(ValueError):
        fs.write_shard(str(tmp_path / "c.shard"), x, dtype=np.float64)
    os.truncate(p2, len(raw) - 2)                                     # the size check counts 2 bytes a value
    with pytest.raises(ValueError, match="size"):
        fs.read_header(p2)


def test_convert_reference_dataset_to_fp16(tmp_path):
    from somcb import fmap_shards as fs
    x = synthetic_fmaps(3, 4).numpy().astype(np.float64)
    db = {"_default": {}}
    for i in range(3):
        p = str(tmp_path / f"f{i}.npy")
        np.save(p, x[i])
        db["_default"][str(i + 1)] = {"fmap_path": p, "image_path": f"img{i}.png"}
    with open(tmp_path / "db.json", "w") as f:
        json.dump(db, f)
    shards = fs.convert_reference_dataset(str(tmp_path / "db.json"), str(tmp_path / "out"), fmaps_per_shard=2,
                                          dtype=np.float16)
    assert len(shards) == 2 and all(fs.shard_dtype(s) == np.float16 for s in shards)
    got = fs.ShardReader(shards, pin=False).read_all().numpy()
    assert np.array_equal(got, x.astype(np.float16))                  # one rounding from the stored values
    assert os.path.exists(tmp_path / "out" / "index.json")
