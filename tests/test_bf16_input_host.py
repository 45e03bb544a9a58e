"""bf16 feature maps on the host side: the FP16-split kernel's row scale and per-tile "lo is non-zero" flag
(csrc/som_bmu_tc_l16.cu) on bfloat16 input, with the numpy emulation of test_f16_input_host.py, and the bfloat16
(version-2, code 2) feature-map shards.

bf16 has an 8-bit significand but fp32's exponent range.  After the power-of-two row scale (max |s_p x| in [64, 128))
an element is exact in FP16 when its lowest significand bit sits on FP16's 2^-24 grid (an element within about 2^-23
of its row's largest magnitude always does) and the scaled value is below FP16's overflow.  Where a tile's flag is
clear every lo operand is exactly zero, so the two-product sum equals the three-product sum; tiles that fail the
test keep the third product."""
import json
import os
import struct

import numpy as np
import pytest
import torch

from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
from _helpers import flat_patches
from test_f16_input_host import _codebook_scales, _emulate, _row_scale

F32 = np.float32


def _bf16(a):
    """float32 array of the bfloat16 values nearest to ``a`` (torch's round-to-nearest-even)."""
    return torch.from_numpy(np.ascontiguousarray(a, dtype=F32)).to(torch.bfloat16).float().numpy()


def _bf16_bits(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=F32)).to(torch.bfloat16).view(torch.int16).numpy() \
        .view(np.uint16)


def _exact_in_fp16(s):
    """Whether each scaled value is an FP16 value: finite, below FP16's overflow, lowest set bit at 2^-24 or above."""
    out = np.isfinite(s) & (np.abs(s) < 65520)
    f, e = np.frexp(np.where(out, s, 0).astype(np.float64))     # s = f 2^e, |f| in [0.5, 1)
    m = (np.abs(f) * 2.0 ** 24).astype(np.int64)                  # the 24-bit significand as an integer
    lowbit = e - 24 + np.log2(np.maximum(m & -m, 1))
    return out & ((s == 0) | (lowbit >= -24))


def _predicted_flags(x, w):
    """The flag per 128-row tile and 64-feature block as the exactness rule predicts it (one row scale per row)."""
    _, tc_exp = _codebook_scales(w)
    with np.errstate(invalid="ignore", over="ignore"):
        s = x * _row_scale(x, tc_exp)[:, None]
    bad = ~_exact_in_fp16(s)
    return [bool(bad[r0:r0 + 128, f0:f0 + 64].any()) for r0 in range(0, x.shape[0], 128)
            for f0 in range(0, x.shape[1], 64)]


def _odd(rng, lo_exp, hi_exp, d):
    """bf16 values with the lowest significand bit set, magnitudes in [2^lo_exp, 2^hi_exp): never exact in FP16 below
    the 2^-24 grid."""
    e = rng.integers(lo_exp, hi_exp, d)
    m = 128 + 2 * rng.integers(0, 64, d) + 1                     # 8-bit significand, odd
    return np.where(rng.random(d) < 0.5, 1.0, -1.0) * m * np.ldexp(1.0, e - 7)


# row kind -> whether its tile keeps the third product (row max 0.9: row scale 2^7)
KINDS = {"tanh": False, "near": False, "below": True, "sub": True, "clamp": True, 1e-6: False, 1e-3: False,
         1.0: False, 100.0: False, 1e30: False, 3.38e38: False, "zero": False, "nan": True, "inf": True, "-inf": True}


def _special_rows(d):
    """One row of each kind in KINDS (fp32 arrays holding bf16 values)."""
    rng = np.random.default_rng(5)
    rows = {"tanh": np.tanh(rng.standard_normal(d))}
    near = rng.uniform(1.0, 16.0, d) * 2.0 ** -24 * np.where(rng.random(d) < 0.5, 1, -1)
    near[0] = 0.9                                                   # within 2^-23.9 of the max: still exact
    rows["near"] = near
    below = np.tanh(rng.standard_normal(d))
    below[0] = 0.9
    below[1:9] = _odd(rng, -30, -25, 8)                            # lowest bits under 2^-24 after the x128 scale
    rows["below"] = below
    rows["sub"] = _odd(rng, -133, -127, d)                         # bf16 subnormals (below 2^-126)
    # max 2^-30: a_p = s_p / t_c would leave FP16, so the row scale is lowered; elements 2^-10 under the max, exact
    # with the full scale, then fall below the 2^-24 grid
    clamp = _odd(rng, -40, -37, d)
    clamp[0] = 2.0 ** -30
    rows["clamp"] = clamp
    for mag in (1e-6, 1e-3, 1.0, 100.0, 1e30, 3.38e38):             # 1e-6: clamped too, but still exact
        rows[mag] = rng.uniform(-mag, mag, d)
    rows["zero"] = np.zeros(d)
    for k, v in (("nan", np.nan), ("inf", np.inf), ("-inf", -np.inf)):
        r = np.tanh(rng.standard_normal(d))
        r[5] = v
        rows[k] = r
    assert list(rows) == list(KINDS)
    out = _bf16(np.stack(list(rows.values())))
    assert np.isfinite(out[:-3]).all()                              # bf16 rounding made no inf of 3.38e38
    return out


@pytest.mark.parametrize("d", [32, 64, 256])
def test_tanh_tiles_take_the_two_product_path(d):
    pd = {32: (4, 2), 64: (4, 4), 256: (8, 8)}[d]
    x = _bf16(flat_patches(synthetic_fmaps(4, 11), pd).numpy()[:512])
    w = trained_like_codebook(512, pd, 7).numpy()
    for flag, three, two in _emulate(x, w):
        assert not flag, "a tile of tanh-range bf16 rows keeps the third product"
        assert np.array_equal(three, two)


def test_special_tiles_set_the_flag_as_predicted():
    d = 64
    special = _special_rows(d)
    w = trained_like_codebook(512, (4, 4), 7).numpy()
    x = np.concatenate([np.repeat(r[None], 128, 0) for r in special])      # one tile per kind
    res = _emulate(x, w)
    flags = [f for f, _, _ in res]
    assert flags == _predicted_flags(x, w)
    assert dict(zip(KINDS, flags)) == KINDS
    for flag, three, two in res:
        if not flag:
            assert np.array_equal(three, two)


def test_flag_clear_means_exactly_zero_lo_in_mixed_tiles():
    # _emulate asserts that every lo operand of a tile with a clear flag is zero
    d = 64
    special = _special_rows(d)
    tanh = _bf16(flat_patches(synthetic_fmaps(2, 2), (4, 4)).numpy())
    w = trained_like_codebook(512, (4, 4), 7).numpy()
    clean = [k for k, keep in KINDS.items() if not keep]
    rows = {k: special[i] for i, k in enumerate(KINDS)}
    x_clear = np.concatenate([tanh[:128 - len(clean)], np.stack([rows[k] for k in clean])])
    x_kept = np.concatenate([tanh[:127], rows["below"][None]])
    for x, want in ((x_clear, False), (x_kept, True)):
        res = _emulate(x, w)
        assert [f for f, _, _ in res] == [want] == _predicted_flags(x, w)
        if not want:
            assert np.array_equal(res[0][1], res[0][2])


# ---- bf16 shards -------------------------------------------------------------------------------------------------

def test_bf16_shard_round_trips_bit_patterns(tmp_path):
    from somcb import fmap_shards as fs
    x = synthetic_fmaps(5, 1).numpy()
    p = str(tmp_path / "a.shard")
    assert fs.write_shard(p, x, dtype=torch.bfloat16) == 5
    raw = open(p, "rb").read()
    head = b"SOMFMAP1" + struct.pack("<IIIIQI", 2, 4, 32, 32, 5, 2)
    assert raw[:64] == head + b"\0" * (64 - len(head))
    assert raw[64:] == _bf16_bits(x).tobytes() and len(raw) == 64 + x.size * 2
    assert fs.read_header(p) == (4, 32, 32, 5) and fs.shard_torch_dtype(p) == torch.bfloat16
    with pytest.raises(ValueError, match="shard_torch_dtype"):
        fs.shard_dtype(p)

    r = fs.ShardReader([p], batch_fmaps=2, pin=False)
    assert r.torch_dtype == torch.bfloat16 and r.dtype is None
    parts = [t.clone() for _, _, t in r.batches()]                   # staging slots are reused
    assert all(t.dtype == torch.bfloat16 for t in parts)
    got = torch.cat(parts)
    assert np.array_equal(got.view(torch.int16).numpy().view(np.uint16), _bf16_bits(x))
    assert torch.equal(r.read_all().view(torch.int16), got.view(torch.int16))

    # every bit pattern (NaN payloads and -0 included) of a bf16 tensor is stored as it is
    bits = torch.arange(1 << 16, dtype=torch.int32).to(torch.int16).view(torch.bfloat16).reshape(1, 1, 256, 256)
    q = str(tmp_path / "all.shard")
    fs.write_shard(q, bits, dtype=torch.bfloat16)
    assert open(q, "rb").read()[64:] == bits.view(torch.int16).numpy().tobytes()
    assert torch.equal(fs.ShardReader(q, pin=False).read_all().view(torch.int16), bits.view(torch.int16))

    os.truncate(p, len(raw) - 2)                                     # the size check counts 2 bytes a value
    with pytest.raises(ValueError, match="size"):
        fs.read_header(p)


def test_bf16_and_fp16_shards_do_not_mix(tmp_path):
    from somcb import fmap_shards as fs
    x = synthetic_fmaps(2, 3).numpy()
    p16, pb = str(tmp_path / "h.shard"), str(tmp_path / "b.shard")
    fs.write_shard(p16, x, dtype=np.float16)
    fs.write_shard(pb, x, dtype=torch.bfloat16)
    assert fs.shard_dtype(p16) == np.float16 and fs.shard_torch_dtype(p16) == torch.float16
    for paths in ([p16, pb], [pb, p16]):
        with pytest.raises(ValueError, match="dtype"):
            fs.ShardReader(paths, pin=False)
    with pytest.raises(ValueError):
        fs.write_shard(str(tmp_path / "c.shard"), x, dtype=torch.float64)


def test_convert_reference_dataset_to_bf16(tmp_path):
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
                                          dtype=torch.bfloat16)
    assert len(shards) == 2 and all(fs.shard_torch_dtype(s) == torch.bfloat16 for s in shards)
    got = fs.ShardReader(shards, pin=False).read_all()
    assert got.dtype == torch.bfloat16
    # the reference's .float(), then one rounding to nearest even
    assert np.array_equal(got.view(torch.int16).numpy().view(np.uint16), _bf16_bits(x.astype(F32)))
