"""Host-side logic on CPU: drop-in API surface, checkpoint layout, geometry, loud failure
without CUDA, and the SomTrainer orchestration driven by the CPU test double."""
import pytest
import torch

import oracle
import somcb
from somcb import ops
from _helpers import (CASES, assert_close_norm, assert_weights_parity, fp64_truth_step, golden_rows, load_case,
                      load_golden)
import _oracle_ops


def test_constructor_attributes_and_state_dict_match_reference_layout():
    cb = somcb.Codebook(patch_dim=(4, 4), image_dim=(32, 32), image_channel=4,
                        num_embeddings=1024, init_neighbour_range=512)
    assert cb.embedding_dim == 64 and cb.num_embeddings == 1024
    assert cb.patch_dim == (4, 4) and cb.image_dim == (32, 32) and cb.neighbourhood_range == 512
    assert isinstance(cb.codebook, torch.nn.Embedding)
    assert list(cb.state_dict().keys()) == ["codebook.weight"]
    params = list(cb.parameters())
    assert len(params) == 1 and params[0].shape == (1024, 64) and params[0].dtype == torch.float32
    assert float(params[0].detach().abs().max()) <= 1.0 / 1024          # U(-1/K, 1/K) init


def test_same_seed_same_init_as_oracle_class():
    torch.manual_seed(0)
    a = somcb.Codebook(num_embeddings=64)
    torch.manual_seed(0)
    b = oracle.OracleCodebook(num_embeddings=64)
    assert torch.equal(a.codebook.weight, b.codebook.weight)


def test_decrease_neighbourhood_semantics():
    cb = somcb.Codebook(num_embeddings=8, init_neighbour_range=3)
    cb.decrease_neighbourhood(steps=5)            # `steps` is validated but otherwise ignored
    assert cb.neighbourhood_range == 2
    cb.decrease_neighbourhood()
    assert cb.neighbourhood_range == 1
    cb.decrease_neighbourhood()
    assert cb.neighbourhood_range == 1.0 and isinstance(cb.neighbourhood_range, float)
    with pytest.raises(Exception, match="Invalid value for steps"):
        cb.decrease_neighbourhood(steps=0)


def test_loads_reference_checkpoint(capsys):
    ck = load_golden("reference_checkpoint.pt")
    cb = somcb.Codebook(patch_dim=ck["patch_dim"], image_dim=ck["image_dim"], image_channel=ck["image_C"],
                        num_embeddings=ck["num_embeddings"], init_neighbour_range=ck["neighbourhood_range"])
    cb.custom_load_state_dict(ck["checkpoint"])
    assert torch.equal(cb.codebook.weight.detach(), ck["checkpoint"]["codebook.weight"])
    # unknown / mismatched keys are skipped with the reference's messages
    cb.custom_load_state_dict({"nope": torch.zeros(1), "codebook.weight": torch.zeros(2, 2)})
    out = capsys.readouterr().out
    assert "No Layer found: nope, skipping" in out and "Skipped: codebook.weight" in out
    cb.custom_load_state_dict({"nope": torch.zeros(1)}, ignore_msgs=True)
    assert capsys.readouterr().out == ""


def test_cpu_compute_fails_loudly():
    cb = somcb.Codebook(patch_dim=(4, 4), num_embeddings=16)
    x = torch.zeros(1, 4, 32, 32)
    with pytest.raises(RuntimeError, match="CUDA only"):
        cb.get_patches_bmu(x)
    with pytest.raises(RuntimeError, match="CUDA only"):
        cb(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.prepare_codebook(torch.zeros(4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.neighbourhood_filter(torch.zeros(4, 4), 2)


def test_geometry_helpers():
    g = ops.geometry((8, 4, 32, 32), (4, 4))
    assert g == (8, 4, 32, 32, 4, 4) and ops.n_patches_of(g) == 512 and ops.dim_of(g) == 64
    f = ops.flat_geometry(100, 48)
    assert ops.n_patches_of(f) == 100 and ops.dim_of(f) == 48
    with pytest.raises(ValueError):
        ops.geometry((1, 4, 30, 32), (4, 4))


def test_patchify_matches_oracle():
    x = torch.randn(3, 5, 12, 8)
    assert torch.equal(somcb.patchify(x, (3, 2)), oracle.patchify(x, (3, 2)))
    p = somcb.patchify(x, (3, 2))
    assert torch.equal(somcb.unpatchify(p, (12, 8), (3, 2)), x)


def test_shard_arithmetic():
    for total, world in ((262144, 8), (10, 3), (7, 8)):
        spans = [somcb.shard_bounds(total, world, r) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
        sizes = [b - a for a, b in spans]
        assert max(sizes) - min(sizes) <= 1
    x = torch.arange(8).reshape(8, 1, 1, 1)
    assert somcb.split_batch(x, 4, 2).flatten().tolist() == [4, 5]
    # ragged (and empty) shares are allowed: the step all-reduces the patch count
    assert [somcb.split_batch(x, 3, r).shape[0] for r in range(3)] == [3, 3, 2]
    assert [somcb.split_batch(x[:2], 4, r).shape[0] for r in range(4)] == [1, 1, 0, 0]


@pytest.mark.parametrize("name", CASES)
def test_trainer_orchestration_matches_reference_step(name):
    """SomTrainer (factorised step) with the CPU test double reproduces the reference's
    weight_after_step / loss; on the GPU the same class runs with the CUDA ops."""
    rec = load_case(name)
    cb = somcb.Codebook(patch_dim=rec["patch_dim"], image_dim=rec["image_dim"],
                        image_channel=rec["channels"], num_embeddings=rec["weight"].shape[0],
                        init_neighbour_range=rec["neighbourhood_range"])
    with torch.no_grad():
        cb.codebook.weight.copy_(rec["weight"])
    tr = somcb.SomTrainer(cb, lr=1e-4, neighbourhood_step=10 ** 9, ops=_oracle_ops)
    loss = tr.step(rec["x"], bmu=rec["bmu"])
    assert_close_norm(loss, rec["loss"], 1e-6, "loss")
    w_truth, _, _ = fp64_truth_step(rec)
    w, w_truth, w_ref = golden_rows(rec, "weight_after_step", cb.codebook.weight.detach(), w_truth)
    assert_weights_parity(w, w_ref, w_truth)
    assert tr.global_steps == 1 and tr.t == 1


def test_trainer_schedule_bookkeeping():
    rec = load_case("range_floor")
    cb = somcb.Codebook(patch_dim=rec["patch_dim"], image_dim=rec["image_dim"],
                        image_channel=rec["channels"], num_embeddings=64, init_neighbour_range=3)
    tr = somcb.SomTrainer(cb, lr=1e-3, neighbourhood_step=2, lr_step=3, ops=_oracle_ops)
    lrs, ranges = [], []
    for _ in range(8):
        tr.step(rec["x"])
        lrs.append(tr.lr)
        ranges.append(cb.neighbourhood_range)
    # lr halves when global_steps % 3 == 0 and > 0, checked BEFORE the increment (steps 3, 6)
    assert lrs == [1e-3, 1e-3, 1e-3, 5e-4, 5e-4, 5e-4, 2.5e-4, 2.5e-4]
    # range decreases when the incremented counter hits a multiple of 2; floors at float 1.0
    assert ranges == [3, 2, 2, 1, 1, 1.0, 1.0, 1.0]
    ck = tr.checkpoint_dict(image_channel=rec["channels"])
    assert set(ck) == {"patch_dim", "image_dim", "image_C", "num_embeddings", "neighbourhood_range",
                       "global_steps", "checkpoint"}
    assert ck["global_steps"] == 8 and list(ck["checkpoint"]) == ["codebook.weight"]


def test_fmap_shards_round_trip_from_reference_layout(tmp_path):
    """The reference's on-disk dataset (generate_fmap_dataset.py:42-72: one .npy per fmap, <=1000 per
    folder, TinyDB json) -> packed shards -> ShardReader batches: values, order and image paths."""
    import json
    import numpy as np
    import torch
    from somcb import fmap_shards as fs
    rng = np.random.default_rng(3)
    src = tmp_path / "ref"
    docs, maps = {}, []
    for i in range(37):
        folder = src / str(i // 10)                       # the reference's folder roll-over
        folder.mkdir(parents=True, exist_ok=True)
        fmap = np.tanh(rng.standard_normal((4, 8, 8))).astype(np.float32)
        path = folder / str(i)
        with open(path, "wb") as f:
            np.save(f, fmap, allow_pickle=False)
        maps.append(fmap)
        docs[str(i + 1)] = {"fmap_path": str(path), "image_path": f"img_{i}.jpg"}
    db = src / "all_dataset.json"
    db.write_text(json.dumps({"_default": docs}))
    shards = fs.convert_reference_dataset(str(db), str(tmp_path / "packed"), fmaps_per_shard=16)
    assert len(shards) == 3 and [fs.read_header(s)[3] for s in shards] == [16, 16, 5]
    reader = fs.ShardReader(shards, batch_fmaps=7, pin=False)
    assert len(reader) == 37 and reader.shape == (4, 8, 8)
    ref = torch.from_numpy(np.stack(maps))
    assert torch.equal(reader.read_all(), ref)
    seen = 0
    for lo, hi, t in reader.batches():
        assert lo == seen and torch.equal(t, ref[lo:hi]) and t.dtype == torch.float32
        seen = hi
    assert seen == 37
    idx = json.loads((tmp_path / "packed" / "index.json").read_text())
    assert idx["entries"][20] == {"i": 20, "shard": 1, "row": 4, "image_path": "img_20.jpg"}
    import pytest
    (tmp_path / "empty.json").write_text(json.dumps({"_default": {}}))
    with pytest.raises(Exception, match="No data found"):
        fs.reference_entries(str(tmp_path / "empty.json"))
    bad = tmp_path / "bad.shard"
    bad.write_bytes(b"x" * 100)
    with pytest.raises(ValueError):
        fs.read_header(str(bad))


def test_numa_binding_is_a_noop_without_topology():
    """No CUDA device / no sysfs topology: bind_host_to_gpu_node returns None and leaves the affinity alone."""
    import os
    before = os.sched_getaffinity(0)
    assert somcb.bind_host_to_gpu_node() is None
    assert somcb.bind_host_to_gpu_node("cuda:0") is None
    assert os.sched_getaffinity(0) == before
