"""Shared test helpers: golden loading and the parity rules of SURVEY.md 8c."""
import os

import torch

from oracle import distance_fp64, patchify

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ["c1_fresh", "c1_trained", "c2_trained", "c2_fresh", "c3_shape_small", "c5_shape_small",
         "odd_geom", "range_floor"]
BMU_EPS = 1e-6      # north-star: relative fp64 distance gap allowed between our pick and the oracle's
W_TOL = 1e-5        # north-star: norm-relative weight tolerance


def load_case(name):
    return torch.load(os.path.join(GOLDEN, f"case_{name}.pt"), weights_only=True)


def load_golden(fname):
    return torch.load(os.path.join(GOLDEN, fname), weights_only=True)


def golden_rows(rec, name, *got):
    """The given tensors, each shaped like the reference output ``name``, and that stored output, on the rows the
    golden file keeps: a large output is stored as a fixed, seeded sample of the rows of t.reshape(-1, t.shape[-1])
    (oracle/make_golden.keep_sampled_rows), a small one whole.  Returns (*got, want)."""
    rows = rec.get("sampled_rows", {}).get(name)
    if rows is None:
        return (*got, rec[name])
    out = []
    for t in got:
        assert tuple(t.shape) == tuple(rec["shapes"][name]), f"{name}: shape {tuple(t.shape)}"
        out.append(t.reshape(-1, t.shape[-1])[rows.to(t.device)])
    return (*out, rec[name])


def flat_patches(x, patch_dim):
    p = patchify(x, patch_dim)
    return p.reshape(-1, p.shape[-1])


def assert_bmu_parity(idx_new, idx_ref, flat, weight, eps=BMU_EPS):
    """Indices equal, or our pick within eps (relative, fp64 direct distance) of the oracle's."""
    idx_new = idx_new.cpu().reshape(-1)
    idx_ref = idx_ref.cpu().reshape(-1)
    assert idx_new.shape == idx_ref.shape
    bad = torch.nonzero(idx_new != idx_ref).flatten()
    if bad.numel() == 0:
        return 0
    d_new = distance_fp64(flat[bad], weight, idx_new[bad])
    d_ref = distance_fp64(flat[bad], weight, idx_ref[bad])
    gap = (d_new - d_ref).abs()
    ok = gap <= eps * d_ref
    assert bool(ok.all()), (f"{int((~ok).sum())} of {idx_new.numel()} BMU picks are worse than the "
                            f"oracle's by more than {eps} relative (max {float((gap / d_ref).max()):.3e})")
    return int(bad.numel())


def rel_fro(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def rel_max(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def assert_close_norm(a, b, tol=W_TOL, what="tensor"):
    f, m = rel_fro(a, b), rel_max(a, b)
    assert f <= tol and m <= tol, f"{what}: rel_fro={f:.3e} rel_max={m:.3e} > {tol}"


def fp64_truth_step(rec, lr=1e-4):
    """Exact-arithmetic (fp64) teacher-forced step from a golden case: (W', grad, loss)."""
    from oracle.step_oracle import AdamState, closed_form_step
    w = rec["weight"].double().clone()
    st = AdamState.zeros_like(w)
    loss, _, grad = closed_form_step(w, st, rec["x"].double(), rec["patch_dim"],
                                     rec["neighbourhood_range"], lr, bmu=rec["bmu"])
    return w, grad, loss


def assert_weights_parity(w_new, w_ref, w_truth, tol=W_TOL, what="weights"):
    """North-star bound (1e-5 norm-relative) on the Frobenius norm always.  On the max norm the
    bound is 1e-5 too, EXCEPT where the reference itself is further than that from exact
    arithmetic: at the reference's fresh U(-1/K, 1/K) init the first Adam step is
    lr * g / (|g| + 1e-8), which amplifies fp32 rounding of near-zero gradient entries, and the
    reference's own W' is 6e-5..9e-5 (max-relative) away from the fp64 result.  There we require
    to be as close to the fp64 truth as the reference is (x3 slack for summation order)."""
    f = rel_fro(w_new, w_ref)
    assert f <= tol, f"{what}: rel_fro={f:.3e} > {tol}"
    m = rel_max(w_new, w_ref)
    ref_err = rel_max(w_ref, w_truth)
    new_err = rel_max(w_new, w_truth)
    assert m <= tol or new_err <= max(tol, 3.0 * ref_err), (
        f"{what}: rel_max vs reference {m:.3e}; vs fp64 truth ours {new_err:.3e}, reference {ref_err:.3e}")
