"""Save and resume of the fused trainers on CPU (kernels replaced by the test double tests/_oracle_ops.py): a run split
by checkpoint_dict(C, with_state=True) -> torch.save -> torch.load -> resume into a new Codebook and trainer is
bit-identical to the run that was not interrupted, also when the split falls just before an lr halving or a
neighbourhood decrement; a checkpoint without the trainer state resumes as the reference does; the reference's loader
reads a with-state file silently; a mismatched state is refused without a partial load; a state saved by two
data-parallel ranks (gloo) resumes on one process and the other way round."""
import io
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle
import somcb
import _oracle_ops
from _helpers import assert_close_norm
from oracle.step_oracle import synthetic_fmaps, trained_like_codebook

HERE = os.path.dirname(os.path.abspath(__file__))
PD, K, C, N_F = (4, 4), 256, 4, 4            # 4 feature maps of 4 x 32 x 32: 256 patches of D = 64 per step
LR = 1e-3


def _cb(w0=None, rng=K // 2):
    cb = somcb.Codebook(patch_dim=PD, image_dim=(32, 32), image_channel=C, num_embeddings=K, init_neighbour_range=rng)
    with torch.no_grad():
        cb.codebook.weight.copy_(trained_like_codebook(K, PD, 7) if w0 is None else w0)
    return cb


def _batch(step):
    return synthetic_fmaps(N_F, 300 + step)


def _trainer(cls=somcb.SomTrainer, **kw):
    return cls(_cb(), lr=LR, ops=_oracle_ops, **kw)


def _run(tr, steps, first=0, split=None):
    """Losses of steps [first, first + steps); ``split(x)`` gives the batch this trainer sees of the global batch x."""
    out = []
    for s in range(first, first + steps):
        x = _batch(s)
        out.append(tr.step(x if split is None else split(x)).clone())
    return torch.stack(out)


def _save_load(ck):
    buf = io.BytesIO()
    torch.save(ck, buf)
    buf.seek(0)
    return torch.load(buf)                   # weights_only (the default): the with-state file needs nothing more


def _state_of(tr):
    return {"w": tr.cb.codebook.weight.detach().clone(), "m": tr.m.clone(), "v": tr.v.clone(),
            "t_dev": tr.t_dev.clone(), "t": tr.t, "lr": tr.lr, "global_steps": tr.global_steps,
            "range": tr.cb.neighbourhood_range, "betas": tuple(tr.betas), "eps": tr.eps}


def _assert_same_state(a, b):
    for key in ("w", "m", "v", "t_dev"):
        assert torch.equal(a[key], b[key]), key
    for key in ("t", "lr", "global_steps", "range", "betas", "eps"):
        assert a[key] == b[key] and type(a[key]) is type(b[key]), (key, a[key], b[key])


@pytest.mark.parametrize("lr_step,neighbourhood_step,n", [
    (3, 10 ** 9, 3),          # the first step after the split halves lr (global_steps == lr_step before its increment)
    (10 ** 5, 4, 3),          # the first step after the split decrements the neighbourhood range
    (10 ** 5, 10 ** 9, 4),    # neither
])
def test_split_run_equals_straight_run(lr_step, neighbourhood_step, n):
    kw = dict(neighbourhood_step=neighbourhood_step, lr_step=lr_step)
    straight = _trainer(**kw)
    want = _run(straight, 2 * n)

    first = _trainer(**kw)
    _run(first, n)
    lr_at_split, range_at_split = first.lr, first.cb.neighbourhood_range
    ck = _save_load(first.checkpoint_dict(C, with_state=True))
    del first
    second = somcb.SomTrainer(_cb(torch.zeros(K, 64)), lr=0.5, neighbourhood_step=1, ops=_oracle_ops)
    second.resume(ck)
    assert second.t == n and int(second.t_dev[0]) == n
    got = _run(second, n, first=n)

    assert torch.equal(got, want[n:])
    _assert_same_state(_state_of(second), _state_of(straight))
    assert second.lr_step == lr_step and second.neighbourhood_step == neighbourhood_step
    if lr_step == n:
        assert lr_at_split == LR and straight.lr == LR / 2
    if neighbourhood_step == n + 1:
        assert straight.cb.neighbourhood_range == range_at_split - 1


def test_checkpoint_without_state_resumes_as_the_reference_does():
    """The reference's layout: moments and step count at zero, global_steps and range from the file; the continuation
    equals a trainer built the reference's way from that file (rebuild, custom_load_state_dict, global_steps)."""
    first = _trainer(neighbourhood_step=2)
    _run(first, 3)
    ck = _save_load(first.checkpoint_dict(C))
    assert "trainer" not in ck
    tr = _trainer(neighbourhood_step=2)
    _run(tr, 1)                              # a trainer that has moments of its own: resume resets them
    tr.resume(ck)
    assert tr.t == 0 and int(tr.t_dev[0]) == 0 and int(tr.t_dev[1]) == 0
    assert not tr.m.any() and not tr.v.any()
    assert tr.global_steps == 3 and tr.cb.neighbourhood_range == ck["neighbourhood_range"] == K // 2 - 1
    assert torch.equal(tr.cb.codebook.weight.detach(), ck["checkpoint"]["codebook.weight"])

    cb = somcb.Codebook(patch_dim=ck["patch_dim"], image_dim=ck["image_dim"], image_channel=ck["image_C"],
                        num_embeddings=ck["num_embeddings"], init_neighbour_range=ck["neighbourhood_range"])
    cb.custom_load_state_dict(ck["checkpoint"])
    ref = somcb.SomTrainer(cb, lr=LR, neighbourhood_step=2, global_steps=ck["global_steps"], ops=_oracle_ops)
    assert torch.equal(_run(tr, 3, first=3), _run(ref, 3, first=3))
    _assert_same_state(_state_of(tr), _state_of(ref))


def test_with_state_checkpoint_keeps_the_reference_keys_and_loads_in_the_reference(capsys):
    tr = _trainer(neighbourhood_step=2)
    _run(tr, 3)
    plain = tr.checkpoint_dict(C)
    full = tr.checkpoint_dict(C, with_state=True)
    assert list(plain) == ["patch_dim", "image_dim", "image_C", "num_embeddings", "neighbourhood_range",
                           "global_steps", "checkpoint"]
    assert list(full) == list(plain) + ["trainer"]
    assert set(full["trainer"]) == set(somcb.SomTrainer.STATE_KEYS)
    a, b = io.BytesIO(), io.BytesIO()
    torch.save(plain, a)
    torch.save({key: full[key] for key in plain}, b)
    assert a.getvalue() == b.getvalue()                 # every reference key byte-identical

    ck = _save_load(full)
    ocb = oracle.OracleCodebook(patch_dim=ck["patch_dim"], image_dim=ck["image_dim"], image_channel=ck["image_C"],
                                num_embeddings=ck["num_embeddings"], init_neighbour_range=ck["neighbourhood_range"])
    ocb.custom_load_state_dict(ck["checkpoint"])
    assert capsys.readouterr().out == ""
    assert torch.equal(ocb.codebook.weight.detach(), tr.cb.codebook.weight.detach())
    assert ck["global_steps"] == 3


def _bad_states(good):
    wrong_k = dict(good, num_embeddings=K + 1, m=torch.zeros(K + 1, 64), v=torch.zeros(K + 1, 64))
    wrong_d = dict(good, embedding_dim=48, m=torch.zeros(K, 48), v=torch.zeros(K, 48))
    wrong_m = dict(good, m=torch.zeros(K, 48))
    wrong_v = dict(good, v=torch.zeros(K - 1, 64))
    missing = {key: val for key, val in good.items() if key != "t_dev"}
    return [wrong_k, wrong_d, wrong_m, wrong_v, missing]


def test_mismatched_state_raises_and_leaves_the_trainer_unchanged():
    donor = _trainer(neighbourhood_step=2)
    _run(donor, 2)
    good = donor.state_dict()
    tr = _trainer(neighbourhood_step=3, lr_step=2)
    _run(tr, 3)
    before = _state_of(tr)
    for bad in _bad_states(good):
        with pytest.raises(ValueError):
            tr.load_state_dict(bad)
        with pytest.raises(ValueError):
            tr.resume(dict(donor.checkpoint_dict(C), trainer=bad))
        _assert_same_state(_state_of(tr), before)
    ck = donor.checkpoint_dict(C, with_state=True)
    ck["checkpoint"] = {"codebook.weight": torch.zeros(K, 48)}
    with pytest.raises(ValueError, match="shape"):
        tr.resume(ck)
    _assert_same_state(_state_of(tr), before)
    tr.load_state_dict(good)                 # the same trainer takes a matching state
    _assert_same_state({**_state_of(tr), "w": before["w"]}, {**_state_of(donor), "w": before["w"]})


def test_betas_and_eps_come_from_the_state():
    donor = somcb.SomTrainer(_cb(), lr=LR, neighbourhood_step=5, betas=(0.9, 0.99), eps=1e-6, ops=_oracle_ops)
    _run(donor, 2)
    ck = _save_load(donor.checkpoint_dict(C, with_state=True))
    tr = _trainer(neighbourhood_step=5)
    tr.resume(ck)
    assert tr.betas == (0.9, 0.99) and tr.eps == 1e-6
    assert torch.equal(_run(tr, 2, first=2), _run(donor, 2, first=2))


# ---- data parallel under gloo (world size 2) ----------------------------------------------------------------------
DP_KW = dict(neighbourhood_step=4, lr_step=3)
DP_N = 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    for p in (HERE, os.path.dirname(HERE),
              os.path.join(os.path.dirname(HERE), "quantized-autoregression-image-generator_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.set_num_threads(2)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        _dp_resume_body(rank, world, out_dir)
    finally:
        dist.destroy_process_group()


def _dp_resume_body(rank, world, out_dir):
    """(a) DP_N steps at world size 2, then save; (b) resume at world size 2 from the one-process checkpoint the test
    wrote, and DP_N more steps."""
    def split(x):
        return somcb.split_batch(x, world, rank).contiguous()

    tr = _trainer(somcb.DataParallelSom, **DP_KW)
    assert tr.world_size == world and tr.reduce_fn is not None
    _run(tr, DP_N, split=split)
    torch.save(tr.checkpoint_dict(C, with_state=True), os.path.join(out_dir, f"ck_dp_{rank}.pt"))

    tr = somcb.DataParallelSom(_cb(torch.zeros(K, 64)), lr=0.5, neighbourhood_step=1, ops=_oracle_ops)
    tr.resume(torch.load(os.path.join(out_dir, "ck_single.pt")))
    losses = _run(tr, DP_N, first=DP_N, split=split)
    torch.save({"w": tr.cb.codebook.weight.detach().clone(), "loss": losses, "state": tr.state_dict()},
               os.path.join(out_dir, f"resumed_dp_{rank}.pt"))


def test_data_parallel_state_resumes_at_another_world_size(tmp_path):
    straight = _trainer(**DP_KW)
    want = _run(straight, 2 * DP_N)
    single = _trainer(**DP_KW)
    _run(single, DP_N)
    torch.save(single.checkpoint_dict(C, with_state=True), tmp_path / "ck_single.pt")

    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)

    # saved at world size 2: both ranks wrote the same state; resumed on one process
    ck0, ck1 = torch.load(tmp_path / "ck_dp_0.pt"), torch.load(tmp_path / "ck_dp_1.pt")
    for key, val in ck0["trainer"].items():
        same = torch.equal(val, ck1["trainer"][key]) if torch.is_tensor(val) else val == ck1["trainer"][key]
        assert same, key
    assert torch.equal(ck0["checkpoint"]["codebook.weight"], ck1["checkpoint"]["codebook.weight"])
    tr = _trainer(neighbourhood_step=1)
    tr.resume(ck0)
    got = _run(tr, DP_N, first=DP_N)
    assert_close_norm(got, want[DP_N:], 1e-6, "losses resumed from a world-size-2 state")
    assert_close_norm(tr.cb.codebook.weight.detach(), straight.cb.codebook.weight.detach(), 1e-6,
                      "weights resumed from a world-size-2 state")
    assert (tr.t, tr.lr, tr.global_steps, tr.cb.neighbourhood_range) == \
        (straight.t, straight.lr, straight.global_steps, straight.cb.neighbourhood_range)

    # saved on one process: resumed at world size 2
    r0, r1 = torch.load(tmp_path / "resumed_dp_0.pt"), torch.load(tmp_path / "resumed_dp_1.pt")
    assert torch.equal(r0["w"], r1["w"]) and torch.equal(r0["loss"], r1["loss"]), "replicas diverged"
    assert_close_norm(r0["loss"], want[DP_N:], 1e-6, "losses resumed at world size 2")
    assert_close_norm(r0["w"], straight.cb.codebook.weight.detach(), 1e-6, "weights resumed at world size 2")
    st = r0["state"]
    assert (st["t"], st["t_dev"], st["lr"], st["global_steps"], st["neighbourhood_range"]) == \
        (straight.t, int(straight.t_dev[0]), straight.lr, straight.global_steps, straight.cb.neighbourhood_range)
