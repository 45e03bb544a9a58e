"""The oracle restatement against outputs of the UNMODIFIED reference (tests/golden, generated
by oracle/make_golden.py in the build container).  CPU only."""
import pytest
import torch

import oracle
from oracle.step_oracle import (AdamState, closed_form_step, factorised_grad, histogram_prune,
                                make_oracle_codebook, make_reference_optimizer, reference_step,
                                synthetic_fmaps, trained_like_codebook)
from _helpers import (CASES, assert_bmu_parity, assert_close_norm, flat_patches, golden_rows, load_case,
                      load_golden)


def _cb(rec):
    return make_oracle_codebook(rec["weight"], rec["patch_dim"], rec["image_dim"], rec["channels"],
                                rec["neighbourhood_range"])


@pytest.mark.parametrize("name", CASES)
def test_oracle_forward_matches_reference(name):
    rec = load_case(name)
    cb = _cb(rec)
    x = rec["x"]
    flat = flat_patches(x, rec["patch_dim"])
    with torch.no_grad():
        patches = oracle.patchify(x, rec["patch_dim"])
        assert torch.equal(*golden_rows(rec, "patches", patches))
        assert torch.equal(oracle.unpatchify(patches, rec["image_dim"], rec["patch_dim"]), x)
        bmu = cb.get_patches_bmu(x)
        # same torch build -> normally bit-identical; a different BLAS thread count may move a
        # near-tie, which the parity rule still bounds
        assert_bmu_parity(bmu, rec["bmu"], flat, rec["weight"])
        assert cb.get_patches_bmu(x, reshape=True).shape == rec["bmu_reshaped"].shape
        if torch.equal(bmu, rec["bmu"]):
            assert_close_norm(*golden_rows(rec, "quant_gauss", cb.get_quantized_patches(x, True)), 1e-6, "quant_gauss")
            assert torch.equal(*golden_rows(rec, "quant_hard", cb.get_quantized_patches(x, False)))
            assert_close_norm(*golden_rows(rec, "forward_gauss", cb(x)), 1e-6, "forward")
            assert torch.equal(*golden_rows(rec, "quant_image", cb.get_quantized_image(rec["bmu_reshaped"])))


@pytest.mark.parametrize("name", CASES)
def test_oracle_step_matches_reference(name):
    rec = load_case(name)
    cb = _cb(rec)
    opt = make_reference_optimizer(cb, 1e-4)
    loss = reference_step(cb, opt, rec["x"])
    assert_close_norm(loss, rec["loss"], 1e-6, "loss")
    assert_close_norm(*golden_rows(rec, "grad", cb.codebook.weight.grad), 1e-6, "grad")
    assert_close_norm(*golden_rows(rec, "weight_after_step", cb.codebook.weight.detach()), 1e-6, "weight")


@pytest.mark.parametrize("name", CASES)
def test_closed_form_and_factorised_match_reference(name):
    rec = load_case(name)
    w = rec["weight"].clone()
    st = AdamState.zeros_like(w)
    loss, bmu, grad = closed_form_step(w, st, rec["x"], rec["patch_dim"], rec["neighbourhood_range"],
                                       1e-4, bmu=rec["bmu"])
    assert_close_norm(*golden_rows(rec, "grad", grad), 2e-6, "closed-form grad")
    assert_close_norm(*golden_rows(rec, "weight_after_step", w), 1e-6, "closed-form weight")
    assert_close_norm(loss, rec["loss"], 1e-6, "closed-form loss")
    flat = flat_patches(rec["x"], rec["patch_dim"])
    _, _, counts, sse, g = factorised_grad(rec["weight"], flat, rec["bmu"], rec["neighbourhood_range"],
                                           rec["x"].numel())
    assert int(counts.sum()) == flat.shape[0]
    assert_close_norm(*golden_rows(rec, "grad", g), 2e-6, "factorised grad")
    assert_close_norm(sse / rec["x"].numel(), rec["loss"], 1e-6, "factorised loss")


def test_oracle_ties_lowest_index():
    rec = load_golden("case_ties.pt")
    cb = make_oracle_codebook(rec["weight"], rec["patch_dim"], rec["image_dim"], rec["channels"], 80)
    with torch.no_grad():
        bmu = cb.get_patches_bmu(rec["x"])
    assert torch.equal(bmu, rec["bmu"])
    assert int(bmu.max()) < 64          # rows 64.. are duplicates of rows 0..63


def test_oracle_free_run_100_steps():
    run = load_golden("run_c1_trained_100.pt")
    cb = make_oracle_codebook(run["weight0"], run["patch_dim"], run["image_dim"], run["channels"],
                              run["range0"])
    opt = make_reference_optimizer(cb, run["lr"])
    gs = 0
    for step in range(100):
        loss = reference_step(cb, opt, synthetic_fmaps(8, 123 + step))
        assert abs(float(loss) - float(run["losses"][step])) <= 1e-5 * abs(float(run["losses"][step]))
        gs += 1
        if gs % run["neighbourhood_step"] == 0:
            cb.decrease_neighbourhood(steps=1)
        assert cb.neighbourhood_range == run["ranges"][step]
        if step + 1 in run["weights"]:
            w, snaps = golden_rows(run, "weights", cb.codebook.weight.detach())
            assert_close_norm(w, snaps[step + 1], 1e-5, f"weights@{step + 1}")


def test_oracle_prune_matches_reference():
    rec = load_golden("prune_case.pt")
    cb = make_oracle_codebook(rec["weight"], rec["patch_dim"], rec["image_dim"], rec["channels"], 128)
    batches = [synthetic_fmaps(rec["batch"], s) for s in rec["seeds"]]
    with torch.no_grad():
        counts, good, rows = histogram_prune(cb, batches, rec["threshold"])
    assert counts == rec["counts"].tolist()
    assert good == rec["good"].tolist()
    assert torch.equal(rows, rec["pruned_state_dict"]["codebook.weight"])


def test_synthetic_inputs_are_seed_stable():
    rec = load_case("c1_trained")
    assert torch.equal(synthetic_fmaps(8, 123), rec["x"])
    assert torch.equal(trained_like_codebook(1024, (4, 4), 7), rec["weight"])


def test_band_half_width_values():
    # SURVEY.md 0.7: range 512 -> 152, 8192 -> 608, 1 -> 6
    assert oracle.band_half_width(512) == 152
    assert oracle.band_half_width(8192) == 608
    assert oracle.band_half_width(1) == 6


def test_token_assembly_oracle_shapes_and_tokens():
    """The tokeniser restatement (train_quantized_transformer.py:411-455): shapes, shift, <start>/<end>."""
    from oracle import tokenize_pair_oracle
    from oracle.step_oracle import make_oracle_codebook, synthetic_fmaps, trained_like_codebook
    x = synthetic_fmaps(3, 5)
    lr = make_oracle_codebook(trained_like_codebook(50, (8, 8), 1), (8, 8), (32, 32), 4, 25)
    hr = make_oracle_codebook(trained_like_codebook(70, (4, 4), 2), (4, 4), (32, 32), 4, 35)
    hi, ht, li = tokenize_pair_oracle(lr, hr, x, True)
    assert hi.shape == (3, 16 + 64) and ht.shape == (3, 65) and li is None
    assert int(hi[:, :16].max()) < 50 and int(hi[:, 16:].min()) >= 50 and bool((ht[:, -1] == 70).all())
    assert torch.equal(hi[:, 16:] - 50, ht[:, :-1])
    hi2, ht2, li2 = tokenize_pair_oracle(lr, hr, x, False)
    assert hi2.shape == (3, 65) and bool((hi2[:, 0] == 70).all()) and torch.equal(hi2[:, 1:], ht2[:, :-1])
    assert torch.equal(li2, hi[:, :16]) and torch.equal(ht, ht2)


def test_token_assembly_oracle_matches_reference_golden():
    """tokens_case.pt holds the outputs of the reference script's own lines 407-455."""
    from oracle import tokenize_pair_oracle
    from oracle.step_oracle import make_oracle_codebook
    from _helpers import load_golden
    rec = load_golden("tokens_case.pt")
    lr = make_oracle_codebook(rec["lr_weight"], rec["lr_patch"], rec["image_dim"], rec["channels"], 48)
    hr = make_oracle_codebook(rec["hr_weight"], rec["hr_patch"], rec["image_dim"], rec["channels"], 80)
    for base, tag in ((True, "base"), (False, "cond")):
        hi, ht, li = tokenize_pair_oracle(lr, hr, rec["x"], base)
        assert torch.equal(hi, rec[f"hr_input_{tag}"]) and torch.equal(ht, rec[f"hr_target_{tag}"])
        if rec[f"lr_input_{tag}"] is None:
            assert li is None
        else:
            assert torch.equal(li, rec[f"lr_input_{tag}"])
