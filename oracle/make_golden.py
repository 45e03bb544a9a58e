"""Generate tests/golden/*.pt by running the UNMODIFIED reference module.

Run in the build container only (needs /root/reference):

    python oracle/make_golden.py

Imports ``models.Codebook`` / ``models.layers`` from /root/reference (read-only), feeds
them the seeded synthetic inputs of SURVEY.md §8d and stores inputs + outputs as small
torch files.  The GPU box has no /root/reference; tests there read only these files.
TEST INFRASTRUCTURE (see oracle/__init__.py).
"""
import os
import sys

import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("SOM_REFERENCE_PATH", "/root/reference")
sys.path.insert(0, ROOT)

from oracle.step_oracle import synthetic_fmaps, trained_like_codebook  # noqa: E402


def _ref_modules():
    sys.path.insert(0, REF)
    from models.Codebook import Codebook  # type: ignore
    from models import layers  # type: ignore
    sys.path.pop(0)
    return Codebook, layers


def _build(Codebook, weight, patch_dim, image_dim, channels, rng):
    cb = Codebook(patch_dim=patch_dim, image_dim=image_dim, image_channel=channels,
                  num_embeddings=weight.shape[0], init_neighbour_range=rng)
    with torch.no_grad():
        cb.codebook.weight.copy_(weight)
    return cb


# reference outputs that are stored as a sample of their rows when a record would not fit GOLDEN_BYTES
CASE_OUTPUTS = ("patches", "quant_gauss", "quant_hard", "forward_gauss", "quant_image", "grad", "weight_after_step")
GOLDEN_BYTES = 900_000


def keep_sampled_rows(rec, names, seed=0):
    """Fit a record under GOLDEN_BYTES of tensor data.  Inputs and small outputs stay whole; each output in ``names``
    (a tensor, or a dict of same-shaped tensors) keeps a fixed, seeded sample of the rows of t.reshape(-1, t.shape[-1]),
    as many as fit beside the rest.  The rows go to rec["sampled_rows"][name], the full shape to rec["shapes"][name]
    (tests/_helpers.golden_rows compares on those rows)."""
    def parts(v):
        return list(v.values()) if isinstance(v, dict) else [v]

    def nbytes(v):
        return sum(t.numel() * t.element_size() for t in parts(v) if isinstance(t, torch.Tensor))
    fixed = sum(nbytes(v) for k, v in rec.items() if k not in names and isinstance(v, (torch.Tensor, dict)))
    frac = (GOLDEN_BYTES - fixed) / sum(nbytes(rec[n]) for n in names)
    if frac >= 1.0:
        return rec
    rec = dict(rec, sampled_rows={}, shapes={})
    for n in names:
        shape = tuple(parts(rec[n])[0].shape)
        n_rows = parts(rec[n])[0].numel() // shape[-1]
        rows = torch.randperm(n_rows, generator=torch.Generator().manual_seed(seed))[:max(1, int(n_rows * frac))]
        rows = rows.sort().values

        def pick(t):
            return t.reshape(-1, shape[-1])[rows].clone()
        rec[n] = {k: pick(t) for k, t in rec[n].items()} if isinstance(rec[n], dict) else pick(rec[n])
        rec["sampled_rows"][n], rec["shapes"][n] = rows, shape
    return rec


def fresh_weight(k, d, seed=0):
    """The reference init U(-1/K, 1/K) (models/Codebook.py:44-46) under a fixed seed."""
    torch.manual_seed(seed)
    return torch.empty(k, d).uniform_(-1 / k, 1 / k)


CASES = [
    # name, batch, C, H, W, (pH,pW), K, range, init
    ("c1_fresh", 8, 4, 32, 32, (4, 4), 1024, 512, "fresh"),
    ("c1_trained", 8, 4, 32, 32, (4, 4), 1024, 512, "trained"),
    ("c2_trained", 4, 4, 32, 32, (2, 2), 4096, 2048, "trained"),
    ("c2_fresh", 2, 4, 32, 32, (2, 2), 4096, 2048, "fresh"),
    ("c3_shape_small", 24, 4, 16, 16, (16, 16), 128, 64, "trained"),
    ("c5_shape_small", 4, 4, 32, 32, (8, 8), 512, 256, "trained"),
    ("odd_geom", 5, 3, 8, 12, (2, 3), 37, 5, "trained"),
    ("range_floor", 3, 4, 16, 16, (4, 4), 64, 1.0, "trained"),
]


def main():
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    Codebook, layers = _ref_modules()
    torch.set_num_threads(8)

    # ---- BMU, quantise (both branches), forward, one training step ---------------------
    for name, b, c, h, w, pd, k, rng, init in CASES:
        d = c * pd[0] * pd[1]
        x = synthetic_fmaps(b, 123, c, h, w)
        wt = fresh_weight(k, d) if init == "fresh" else trained_like_codebook(k, pd, 7, c, h, w)
        cb = _build(Codebook, wt, pd, (h, w), c, rng)
        rec = {"x": x, "weight": wt.clone(), "patch_dim": pd, "image_dim": (h, w),
               "channels": c, "neighbourhood_range": rng}
        with torch.no_grad():
            rec["bmu"] = cb.get_patches_bmu(x)
            rec["bmu_reshaped"] = cb.get_patches_bmu(x, reshape=True)
            rec["patches"] = layers.patchify(x, pd).clone()
            rec["quant_gauss"] = cb.get_quantized_patches(x, use_gaussian=True).clone()
            rec["quant_hard"] = cb.get_quantized_patches(x, use_gaussian=False).clone()
            rec["forward_gauss"] = cb(x).clone()
            rec["quant_image"] = cb.get_quantized_image(rec["bmu_reshaped"]).clone()
        # one literal training step (train_codebook.py:183-186, 227-242)
        opt = torch.optim.Adam(cb.parameters(), lr=1e-4, betas=(0.5, 0.999))
        opt.zero_grad()
        q = cb(x, use_gaussian=True)
        loss = F.mse_loss(q, x)
        loss.backward()
        rec["grad"] = cb.codebook.weight.grad.clone()
        opt.step()
        rec["loss"] = loss.detach().clone()
        rec["weight_after_step"] = cb.codebook.weight.detach().clone()
        torch.save(keep_sampled_rows(rec, CASE_OUTPUTS), os.path.join(out_dir, f"case_{name}.pt"))
        print(name, "patches", rec["bmu"].numel(), "loss", float(loss.detach()))

    # ---- tie-break: duplicated rows must resolve to the lowest index --------------------
    pd = (4, 4)
    x = synthetic_fmaps(4, 321)
    wt = trained_like_codebook(64, pd, 11)
    wt = torch.cat([wt, wt[:32], wt], dim=0).contiguous()      # rows 64..95 and 96..159 duplicate
    cb = _build(Codebook, wt, pd, (32, 32), 4, 80)
    with torch.no_grad():
        bmu = cb.get_patches_bmu(x)
    torch.save({"x": x, "weight": wt, "patch_dim": pd, "image_dim": (32, 32), "channels": 4,
                "bmu": bmu}, os.path.join(out_dir, "case_ties.pt"))
    print("ties: max idx", int(bmu.max()))

    # ---- 100 free-running steps from a trained-like init (BASELINE config 1 shape) ------
    pd, k, rng = (4, 4), 1024, 512
    wt = trained_like_codebook(k, pd, 7)
    cb = _build(Codebook, wt, pd, (32, 32), 4, rng)
    opt = torch.optim.Adam(cb.parameters(), lr=1e-4, betas=(0.5, 0.999))
    losses, snaps, ranges = [], {}, []
    global_steps, neighbourhood_step = 0, 20
    for step in range(100):
        x = synthetic_fmaps(8, 123 + step)
        cb.train()
        opt.zero_grad()
        loss = F.mse_loss(cb(x, use_gaussian=True), x)
        loss.backward()
        opt.step()
        losses.append(float(loss))
        global_steps += 1
        if global_steps % neighbourhood_step == 0:
            cb.decrease_neighbourhood(steps=1)
        ranges.append(cb.neighbourhood_range)
        if step + 1 in (1, 10, 50, 100):
            snaps[step + 1] = cb.codebook.weight.detach().clone()
    torch.save(keep_sampled_rows({"weight0": wt, "patch_dim": pd, "image_dim": (32, 32), "channels": 4,
                                  "range0": rng, "lr": 1e-4, "neighbourhood_step": neighbourhood_step,
                                  "losses": torch.tensor(losses, dtype=torch.float64), "ranges": ranges,
                                  "weights": snaps}, ("weights",)),
               os.path.join(out_dir, "run_c1_trained_100.pt"))
    print("100-step run: loss", losses[0], "->", losses[-1], "range", ranges[-1])

    # ---- histogram + prune (prune_codebook.py:129-162) ----------------------------------
    pd, k = (4, 4), 256
    wt = trained_like_codebook(k, pd, 5)
    cb = _build(Codebook, wt, pd, (32, 32), 4, 128)
    total = {i: 0 for i in range(k)}
    batches = [synthetic_fmaps(8, 900 + i) for i in range(3)]
    with torch.no_grad():
        for fm in batches:
            cb.eval()
            for j in cb.get_patches_bmu(fm).tolist():
                total[j] += 1
    thr = 6
    good = [i for i, cnt in total.items() if cnt >= thr]
    new_cb = Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4,
                      num_embeddings=len(good), init_neighbour_range=128)
    with torch.no_grad():
        new_cb.codebook.weight.copy_(cb.codebook.weight[good])
    torch.save({"weight": wt, "patch_dim": pd, "image_dim": (32, 32), "channels": 4,
                "seeds": [900, 901, 902], "batch": 8, "threshold": thr,
                "counts": torch.tensor([total[i] for i in range(k)], dtype=torch.int64),
                "good": torch.tensor(good, dtype=torch.int64),
                "pruned_state_dict": new_cb.state_dict()},
               os.path.join(out_dir, "prune_case.pt"))
    print("prune: kept", len(good), "of", k)

    # ---- checkpoint layout (train_codebook.py:271-278) ----------------------------------
    ck = {"patch_dim": pd, "image_dim": (32, 32), "image_C": 4, "num_embeddings": k,
          "neighbourhood_range": 128, "global_steps": 17, "checkpoint": cb.state_dict()}
    torch.save(ck, os.path.join(out_dir, "reference_checkpoint.pt"))

    # ---- dual-codebook token assembly (train_quantized_transformer.py:407-455) -----------
    # The script cannot be imported here (tinydb is not installed), so its OWN lines are read from
    # the reference tree at generation time, dedented and executed on reference Codebook modules:
    # the golden outputs come from the reference's code, which is never copied into this repository.
    import textwrap
    with open(os.path.join(REF, "train_quantized_transformer.py")) as f:
        src_lines = f.read().splitlines()
    snippet = textwrap.dedent("\n".join(src_lines[406:455]))         # lines 407-455 of the training loop
    assert "lr_codebook.get_patches_bmu" in snippet and "hr_target = hr_target.to(device)" in snippet
    xt = synthetic_fmaps(6, 777)
    lr_w = trained_like_codebook(96, (8, 8), 31)
    hr_w = trained_like_codebook(160, (4, 4), 32)
    rec = {"x": xt, "lr_weight": lr_w, "hr_weight": hr_w, "lr_patch": (8, 8), "hr_patch": (4, 4),
           "image_dim": (32, 32), "channels": 4}
    for base in (True, False):
        env = {"torch": torch, "device": torch.device("cpu"), "feature_map": xt, "train_base_model": base,
               "lr_codebook": _build(Codebook, lr_w, (8, 8), (32, 32), 4, 48),
               "hr_codebook": _build(Codebook, hr_w, (4, 4), (32, 32), 4, 80),
               "lr_num_embeddings": 96, "hr_num_embeddings": 160}
        exec(compile(snippet, "train_quantized_transformer.py[407:455]", "exec"), env)
        tag = "base" if base else "cond"
        rec[f"hr_input_{tag}"] = env["hr_input"].clone()
        rec[f"hr_target_{tag}"] = env["hr_target"].clone()
        rec[f"lr_input_{tag}"] = None if env["lr_input"] is None else env["lr_input"].clone()
    torch.save(rec, os.path.join(out_dir, "tokens_case.pt"))
    print("tokens:", tuple(rec["hr_input_base"].shape), tuple(rec["hr_input_cond"].shape))
    print("done ->", out_dir)


if __name__ == "__main__":
    main()
