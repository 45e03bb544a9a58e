"""The optimizer half of the training step, exactly: every Adam entry point, the packed tail, the loss and the step
counters against the correctly rounded emulation of csrc/som_step_rules.cuh in tests/_adam_exact.py.

Every row runs several consecutive steps and compares W, m and v bit for bit (a NaN matches any NaN: IEEE fixes where a
NaN appears, not its payload) and the device step counters exactly:

* entry points: som_adam_f32 (scalars on the host), som_adam_devstep_f32 and som_adam_dp_f32 (step count, and for the
  latter the gradient scale and the loss, on the device), also replayed from captured CUDA graphs;
* shapes: n = 1, 3, 4, 5, 4k + 3 (the scalar tail loop after the 16-byte body), each of W, m, v, g one float off 16-byte
  alignment (the scalar path for every element), and more elements than one wave of blocks (the grid-stride loop wraps,
  over a thousand blocks meet at the data-parallel kernel's arrival counter);
* rules: b1 = 0.5 (the lerp's `end - diff (1 - w)` branch) and 0.9 (`fma(w, diff, start)`), t = 1 and t = 10^6 (b^t
  underflows), eps = 0, zero / subnormal / underflowing / overflowing / infinite / NaN gradients;
* the data-parallel tail: hand-built reduced tails of 8 ranks with up to 2^31 - 1 patches each, D = 3, 64 and 4096;
* the composed step at h = 0 on the integer lattice (the filter is the identity), through the separate kernels and the
  one-kernel step, against exact argmin, exact Rbar and the emulation: this also runs the packed tail the accumulation
  writes;
* SomTrainer's schedule: which step first sees a halved lr, eager and graph-replayed.

torch.optim.Adam is compared with a per-element bound only: torch's CUDA kernels divide by a CPU scalar through its
reciprocal and may contract differently, so bit equality with torch is not part of the contract."""
import math

import pytest
import torch

import somcb
from somcb import ops
import _adam_exact as E
import _lattice as L
import _update_exact as U

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EPS = 1e-8


def _sms():
    return ops.device_info()[0]


def _blocks(n):
    """the grid of the Adam kernels (csrc/som_core.cu: grid_for(n, 256 * 4, 8))"""
    return max(1, min((n + 1023) // 1024, _sms() * 8))


def mismatches(got, want):
    """elements whose fp32 bits differ (any NaN matches any NaN)"""
    g = got.detach().cpu().reshape(-1)
    w = want.reshape(-1)
    eq = (g.view(torch.int32) == w.view(torch.int32)) | (torch.isnan(g) & torch.isnan(w))
    return int((~eq).sum())


def _assert_state(tag, dev, emu):
    for name, got, want in zip("mvw", dev, emu):
        bad = mismatches(got, want)
        assert bad == 0, f"{tag}: {bad} of {want.numel()} elements of {name} differ from the emulation"


def _state(n, seed):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(n, generator=g)
    m = torch.randn(n, generator=g) * 0.1
    v = torch.rand(n, generator=g) * 1e-2 + 1e-6
    return w, m, v


def _grad(n, seed):
    g = torch.Generator().manual_seed(seed)
    mag = 10.0 ** torch.randint(-4, 2, (n,), generator=g).double()
    return (torch.randn(n, generator=g).double() * mag).float()


def _buffers(w, m, v, off):
    """device copies of w, m, v and a gradient buffer, each either 16-byte aligned or one float off (off: the names)"""
    n = w.numel()
    out = []
    for name, src in (("w", w), ("m", m), ("v", v), ("g", torch.zeros(n))):
        k = 1 if name in off else 0
        buf = torch.empty(n + 4, device=DEV)
        view = buf[k:k + n]
        view.copy_(src)
        out.append(view)
    return out


class Entry:
    """one Adam entry point, its device step count and its emulation"""

    def __init__(self, kind, lr, betas, eps, t0, d=64, tail=None):
        self.kind, self.lr, self.betas, self.eps = kind, lr, betas, eps
        self.t = t0                                                     # completed steps
        self.sd = torch.tensor([t0, 0], dtype=torch.int64, device=DEV)
        self.d = d
        self.tail = tail if tail is not None else E.pack_tail(1234.5, 4099)
        self.tail_dev = self.tail.to(DEV)
        self.loss = torch.full((1,), -1.0, dtype=torch.float64, device=DEV)

    def run(self, w, m, v, g):
        b = self.betas
        if self.kind == "host":
            ops.adam_step(w, m, v, g, self.lr, self.t + 1, betas=b, eps=self.eps)
        elif self.kind == "dev":
            ops.adam_step_dev(w, m, v, g, self.lr, self.sd, betas=b, eps=self.eps)
        else:
            ops.adam_step_dp(w, m, v, g, self.d, self.lr, self.sd, self.tail_dev, loss_out=self.loss, betas=b,
                             eps=self.eps)

    def emulate(self, g, m, v, w):
        a = E.adam_scalars(self.lr, self.betas[0], self.betas[1], self.eps, self.t + 1)
        gscale = E.tail_totals(self.tail, self.d)[1] if self.kind == "dp" else None
        self.t += 1
        return E.adam_update(a, g, m, v, w, gscale=gscale)

    def check_counters(self, tag):
        torch.cuda.synchronize()
        if self.kind == "host":
            return
        assert int(self.sd[0]) == self.t, f"{tag}: steps_done[0] = {int(self.sd[0])}, expected {self.t}"
        assert int(self.sd[1]) == 0, f"{tag}: steps_done[1] = {int(self.sd[1])} after the call"
        if self.kind == "dp":
            numel = E.tail_totals(self.tail, self.d)[0]
            assert float(self.loss) == E.tail_loss(self.tail, numel), f"{tag}: loss"


def _run_row(tag, entry, n, off=(), seed=0, steps=E.STEPS):
    w, m, v = _state(n, seed)
    wd, md, vd, gd = _buffers(w, m, v, off)
    emu = (m, v, w)
    for s in range(steps):
        g = _grad(n, seed + 101 * (s + 1))
        gd.copy_(g)
        entry.run(wd, md, vd, gd)
        emu = entry.emulate(g, *emu)
        entry.check_counters(f"{tag} step {s}")
        _assert_state(f"{tag} step {s}", (md, vd, wd), emu)
    return wd


ENTRIES = ("host", "dev", "dp")
SHAPES = {"n1": (1, ()), "n3": (3, ()), "n4": (4, ()), "n5": (5, ()), "n4099": (4099, ()),
          "w_off": (1027, ("w",)), "m_off": (1027, ("m",)), "v_off": (1027, ("v",)), "g_off": (1027, ("g",)),
          "grid_wraps": ("wrap", ())}


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind", ENTRIES)
def test_adam_entry_points_are_exact_at_every_shape_and_alignment(kind, shape):
    n, off = SHAPES[shape]
    if n == "wrap":
        n = _sms() * 8 * 1024 * 2 + 7                  # two and a bit passes of the grid-stride loop
        assert _blocks(n) > 1000 and n > _blocks(n) * 1024
    entry = Entry(kind, E.LR, (0.5, 0.999), EPS, 0)
    _run_row(f"{kind} {shape}", entry, n, off, seed=n)


RULES = {"b1_0.5_t1": ((0.5, 0.999), 0, EPS), "b1_0.9_t1": ((0.9, 0.999), 0, EPS),
         "b1_0.5_t_large": ((0.5, 0.999), E.T_LARGE - 1, EPS), "b1_0.9_t_large": ((0.9, 0.999), E.T_LARGE - 1, EPS),
         "eps_0": ((0.5, 0.999), 0, 0.0)}


@pytest.mark.parametrize("rule", list(RULES))
@pytest.mark.parametrize("kind", ENTRIES)
def test_adam_entry_points_are_exact_for_every_rule(kind, rule):
    betas, t0, eps = RULES[rule]
    entry = Entry(kind, E.LR, betas, eps, t0)
    _run_row(f"{kind} {rule}", entry, 4099, ("g",) if kind == "dp" else (), seed=7)


# special gradients and what the emulation makes of them with m finite and v > 0 (b1 = 0.5 | 0.9)
SPECIAL = {
    "+0": (0.0, "finite"),
    "-0": (-0.0, "finite"),
    "+subnormal": (1e-40, "finite"),
    "-subnormal": (-3e-42, "finite"),
    "square underflows": (1e-30, "v = fl32(v b2)"),
    "square overflows": (1e25, "v = inf, W unchanged"),
    "+inf": (math.inf, "m = NaN | +inf, v = inf, W = NaN"),
    "-inf": (-math.inf, "m = NaN | -inf, v = inf, W = NaN"),
    "NaN": (math.nan, "m, v, W = NaN"),
}


def _check_special_class(name, b1, g, m0, v0, w0, m, v, w, b2):
    fin = all(bool(torch.isfinite(x).all()) for x in (m, v, w))
    if SPECIAL[name][1] == "finite":
        assert fin
    elif name == "square underflows":
        assert fin and torch.equal(v, E.fmul(v0, b2))
    elif name == "square overflows":
        assert bool(torch.isinf(v).all()) and torch.equal(w, w0)
    elif name in ("+inf", "-inf"):
        want_m = torch.full_like(m, g) if b1 == 0.9 else torch.full_like(m, math.nan)
        assert mismatches(m, want_m) == 0 and bool(torch.isinf(v).all()) and bool(torch.isnan(w).all())
    else:
        assert all(bool(torch.isnan(x).all()) for x in (m, v, w))


@pytest.mark.parametrize("b1", [0.5, 0.9])
@pytest.mark.parametrize("kind", ENTRIES)
def test_special_gradients_follow_the_emulation(kind, b1):
    """each special value on 7 elements (5 in the 16-byte body, 2 in the scalar tail); the data-parallel entry gets a
    tail with gscale = 1 (one patch of D = 2) so the values reach the rule unchanged"""
    per = 7
    names = list(SPECIAL)
    n = per * len(names)
    g = torch.tensor([SPECIAL[nm][0] for nm in names for _ in range(per)], dtype=torch.float32)
    w, m, v = _state(n, 3)
    entry = Entry(kind, E.LR, (b1, 0.999), EPS, 0, d=2, tail=E.pack_tail(8.0, 1))
    assert E.tail_totals(entry.tail, 2)[1] == 1.0
    wd, md, vd, gd = _buffers(w, m, v, ())
    gd.copy_(g)
    entry.run(wd, md, vd, gd)
    em, ev, ew = entry.emulate(g, m, v, w)
    entry.check_counters(f"{kind} b1={b1} special")
    _assert_state(f"{kind} b1={b1} special", (md, vd, wd), (em, ev, ew))
    b2 = E.adam_scalars(E.LR, b1, 0.999, EPS, 1).b2
    for i, nm in enumerate(names):
        sl = slice(i * per, (i + 1) * per)
        _check_special_class(nm, b1, SPECIAL[nm][0], m[sl], v[sl], w[sl], em[sl], ev[sl], ew[sl], b2)


def _tail_of_ranks(counts, seed):
    """the fp32 sum, rank by rank, of the packed tails of ranks with these patch counts and random squared errors"""
    g = torch.Generator().manual_seed(seed)
    acc = torch.zeros(4, dtype=torch.float32)
    for n in counts:
        acc = acc + E.pack_tail(float(torch.rand(1, generator=g, dtype=torch.float64)) * 1e12 * (n > 0), n)
    return acc


TAILS = {"8x2^30": [2 ** 30] * 8, "8x(2^30-1)": [2 ** 30 - 1] * 8, "ragged": [2 ** 31 - 1, 0, 5, 4096, 2 ** 20 + 3]}


@pytest.mark.parametrize("tail", list(TAILS))
@pytest.mark.parametrize("d", [3, 64, 4096])
def test_dp_reads_gradient_scale_and_loss_from_large_reduced_tails(d, tail):
    counts = TAILS[tail]
    t = _tail_of_ranks(counts, d)
    assert E.tail_count(t[2], t[3]) == sum(counts)
    assert float(t[2]) >= 2 ** 18 or tail == "ragged"
    entry = Entry("dp", E.LR, (0.5, 0.999), EPS, 0, d=d, tail=t)
    _run_row(f"dp D={d} {tail}", entry, 4099, seed=d)


def test_dp_and_devstep_with_no_weights_still_count_the_step():
    """n = 0 through the C-ABI (torch gives a zero-element tensor a null data pointer, which the entry points refuse):
    the step count advances; som_adam_dp_f32 does not write loss_out then (include/somcb.h)"""
    lib = somcb._lib.load()
    buf = torch.zeros(8, device=DEV)
    p = buf.data_ptr()
    sd = torch.tensor([41, 0], dtype=torch.int64, device=DEV)
    loss = torch.full((1,), -7.0, dtype=torch.float64, device=DEV)
    tail = E.pack_tail(100.0, 10).to(DEV)
    st = torch.cuda.current_stream().cuda_stream
    somcb._lib.check("som_adam_dp_f32", lib.som_adam_dp_f32(p, p, p, p, 0, 4, E.LR, 0.5, 0.999, EPS, sd.data_ptr(),
                                                            tail.data_ptr(), loss.data_ptr(), st))
    somcb._lib.check("som_adam_devstep_f32", lib.som_adam_devstep_f32(p, p, p, p, 0, E.LR, 0.5, 0.999, EPS,
                                                                      sd.data_ptr(), st))
    somcb._lib.check("som_adam_f32", lib.som_adam_f32(p, p, p, p, 0, E.LR, 0.5, 0.999, EPS, 1, st))
    torch.cuda.synchronize()
    assert sd.tolist() == [43, 0]
    assert float(loss) == -7.0, "loss_out written by the n = 0 data-parallel step"
    assert bool((buf == 0).all())


@pytest.mark.parametrize("kind", ["dev", "dp"])
def test_graph_replays_use_the_next_step_count(kind):
    """one captured graph of adam_step_dev / adam_step_dp replayed 5 times after an eager step: each replay uses
    t + 1 and advances the count once; the arrival word stays 0 (n spans more than 1000 blocks)"""
    n = 1001 * 1024 + 3
    assert _blocks(n) > 1000
    w, m, v = _state(n, 17)
    wd, md, vd, gd = _buffers(w, m, v, ())
    entry = Entry(kind, E.LR, (0.5, 0.999), EPS, 0)
    emu = (m, v, w)
    g = _grad(n, 18)
    gd.copy_(g)
    entry.run(wd, md, vd, gd)                           # eager: one-time launch set-up happens outside the capture
    emu = entry.emulate(g, *emu)
    entry.check_counters(f"{kind} eager")
    _assert_state(f"{kind} eager", (md, vd, wd), emu)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        entry.run(wd, md, vd, gd)
    torch.cuda.synchronize()
    assert int(entry.sd[0]) == 1, "capture ran the step"
    for r in range(5):
        g = _grad(n, 19 + r)
        gd.copy_(g)
        graph.replay()
        emu = entry.emulate(g, *emu)
        entry.check_counters(f"{kind} replay {r}")
        _assert_state(f"{kind} replay {r}", (md, vd, wd), emu)
    assert entry.t == 6


# ================================ the composed step at h = 0 on the integer lattice ==================================
def test_composed_step_at_h0_is_exact_on_the_lattice():
    """bmu -> accumulate_packed -> filter -> adam_step_dp, and step_small, at a range whose band has h = 0 (the filter
    is the identity: w(0) = 1 exactly), on lattice data with exact BMUs: both equal exact argmin, exact Rbar,
    G = fl32(fl32(2 / numel) Rbar) and the emulated Adam.  Three steps in a row carry m, v and the step count; each step
    starts from a fresh lattice codebook (an Adam step leaves the lattice, and the exact chain needs it)."""
    k, d, n = 1024, 64, 2048
    rng = 0.01
    geom = ops.flat_geometry(n, d)
    assert ops.filter_half_width(k, rng) == 0 and ops.step_small_supported(geom, k, rng)
    numel = n * d
    gscale = E._f32(2.0 / numel)
    m = torch.zeros(k, d)
    v = torch.zeros(k, d)
    w_dp, w_sm = torch.empty(k, d, device=DEV), torch.empty(k, d, device=DEV)
    m_dp, v_dp, m_sm, v_sm = (torch.zeros(k, d, device=DEV) for _ in range(4))
    sd_dp = torch.zeros(2, dtype=torch.int64, device=DEV)
    sd_sm = torch.zeros(2, dtype=torch.int64, device=DEV)
    for s in range(3):
        tag = f"step {s}"
        a, b = L.lattice_ints(n, d, k, "narrow", seed=100 + s)
        L.check_bound(a, b)
        rows, w0 = L.to_float(a, 0), L.to_float(b, 0)
        bmu_ref, _ = L.fp64_bmu(rows, w0)
        rbar_i, _, _, sse_i = U.accum_reference(a, b, bmu_ref, k)
        # every fp32 partial sum (of Rbar per unit, of the squared error per CTA) is an integer below 2^24
        assert sse_i < 1 << 24 and int((b[bmu_ref] - a).abs().sum()) < 1 << 24
        rbar = rbar_i.to(torch.float32)
        em, ev, ew = E.adam_update(E.adam_scalars(E.COMPOSED_LR, 0.5, 0.999, EPS, s + 1), rbar, m, v, w0,
                                   gscale=gscale)
        x = rows.contiguous().to(DEV)
        w_dp.copy_(w0)
        w_sm.copy_(w0)
        # the separate kernels
        bmu = ops.bmu(x, geom, w_dp)
        assert torch.equal(bmu.cpu(), bmu_ref), f"{tag}: {int((bmu.cpu() != bmu_ref).sum())} BMUs differ"
        wt = ops.neighbourhood_filter(w_dp, rng)
        assert torch.equal(wt, w_dp), f"{tag}: the h = 0 filter is not the identity"
        packed = ops.accumulate_packed(x, geom, bmu, wt, k)
        tail = packed[k * d:].cpu()
        assert torch.equal(tail, E.pack_tail(float(sse_i), n)), f"{tag}: packed tail {tail.tolist()}"
        assert torch.equal(packed[:k * d].view(k, d).cpu(), rbar), f"{tag}: Rbar"
        grad = ops.neighbourhood_filter(packed[:k * d].view(k, d), rng, scale=1.0)
        loss = ops.adam_step_dp(w_dp, m_dp, v_dp, grad, d, E.COMPOSED_LR, sd_dp, packed[k * d:])
        _assert_state(f"{tag} separate kernels", (m_dp, v_dp, w_dp), (em, ev, ew))
        assert float(loss) == E.tail_loss(tail, float(numel)) == sse_i / numel
        # the one-kernel step
        loss_sm, bmu_sm = ops.step_small(x, geom, w_sm, m_sm, v_sm, rng, E.COMPOSED_LR, sd_sm)
        assert torch.equal(bmu_sm.cpu(), bmu_ref), f"{tag}: one-kernel BMUs"
        _assert_state(f"{tag} one-kernel step", (m_sm, v_sm, w_sm), (em, ev, ew))
        assert float(loss_sm) == sse_i * (1.0 / numel)
        assert sd_dp.tolist() == [s + 1, 0] and int(sd_sm[0]) == s + 1
        m, v = em, ev


# ========================================== the trainer's schedule ====================================================
@pytest.mark.parametrize("graph", [False, True])
def test_trainer_schedule_applies_each_steps_lr_and_count(graph):
    """SomTrainer on the separate kernels, lr_step = 2, neighbourhood_step = 3, 7 steps.  train_codebook.py halves lr
    after the step at which global_steps (before its increment) is a positive multiple of lr_step, so steps 1-3 use lr,
    4-5 lr / 2, 6-7 lr / 4 (1-based), and the range drops after steps 3 and 6.  Each step's G comes from the library's
    own kernels on the trainer's state just before the step; W, m, v, t, t_dev, lr and the loss must match the emulation
    with that step's lr and t."""
    from oracle.step_oracle import synthetic_fmaps, trained_like_codebook
    pd, k = (4, 4), 2048
    lr0 = E.TRAINER_LR
    cb = somcb.Codebook(patch_dim=pd, image_dim=(32, 32), image_channel=4, num_embeddings=k,
                        init_neighbour_range=k // 8)
    with torch.no_grad():
        cb.codebook.weight.copy_(trained_like_codebook(k, pd, 5))
    cb = cb.to(DEV)
    tr = somcb.SomTrainer(cb, lr=lr0, neighbourhood_step=3, lr_step=2, use_cuda_graph=graph,
                          small_step_kernel=False)
    d = cb.embedding_dim
    lrs = [lr0, lr0, lr0, lr0 / 2, lr0 / 2, lr0 / 4, lr0 / 4]
    ranges = [k // 8] * 3 + [k // 8 - 1] * 3 + [k // 8 - 2]
    m, v = torch.zeros(k, d), torch.zeros(k, d)
    for s in range(E.TRAINER_STEPS):
        x = synthetic_fmaps(64, 700 + s).to(DEV)                # 4096 patches
        w = cb.codebook.weight.data
        rng = cb.neighbourhood_range
        assert rng == ranges[s] and tr.lr == lrs[s], f"step {s}: range {rng}, lr {tr.lr}"
        geom = ops.geometry(x.shape, pd)
        wt = ops.neighbourhood_filter(w, rng)
        # the search and accumulation as the step runs them (through the search's staging copy where it writes one)
        npat = ops.n_patches_of(geom)
        stage = torch.empty(npat, d, device=DEV) if ops.bmu_can_stage(geom, k, cb.bmu_variant) else None
        bmu = ops.bmu(x, geom, w, ops.prepare_codebook(w), variant=cb.bmu_variant, stage=stage)
        x_acc, geom_acc = (stage, ops.flat_geometry(npat, d)) if stage is not None else (x, geom)
        packed = ops.accumulate_packed(x_acc, geom_acc, bmu, wt, k)
        grad = ops.neighbourhood_filter(packed[:k * d].view(k, d), rng, scale=1.0).cpu()
        tail = packed[k * d:].cpu()
        numel, gscale = E.tail_totals(tail, d)
        assert numel == x.numel()
        w0 = w.cpu()
        em, ev, ew = E.adam_update(E.adam_scalars(lrs[s], 0.5, 0.999, EPS, s + 1), grad, m, v, w0, gscale=gscale)
        loss = tr.step(x)
        torch.cuda.synchronize()
        tag = f"graph={graph} step {s}"
        _assert_state(tag, (tr.m, tr.v, cb.codebook.weight.data), (em, ev, ew))
        assert float(loss) == E.tail_loss(tail, numel), f"{tag}: loss"
        assert tr.t == s + 1 and tr.t_dev.tolist() == [s + 1, 0], f"{tag}: t {tr.t}, t_dev {tr.t_dev.tolist()}"
        m, v = em, ev
    assert tr.lr == lr0 / 8
    if graph:
        assert len(tr._graphs) >= 3


# ============================================== against torch.optim.Adam =============================================
@pytest.mark.parametrize("device", ["cpu", DEV])
@pytest.mark.parametrize("b1", [0.5, 0.9])
def test_adam_kernel_is_within_a_per_element_bound_of_torch_adam(device, b1):
    """som_adam_f32 against torch.optim.Adam(foreach=False), one step at a time from the kernel's own state:
    |W_kernel - W_torch| <= 2 ulp(W_torch) + 8 u |W_torch - W_before| (u = 2^-24) for every element"""
    n = 4099
    w, _, _ = _state(n, 31)
    wd, md, vd, gd = _buffers(w, torch.zeros(n), torch.zeros(n), ())             # torch's moments start at zero
    p = torch.nn.Parameter(w.clone().to(device))
    opt = torch.optim.Adam([p], lr=E.LR, betas=(b1, 0.999), eps=EPS, foreach=False)
    for t in range(1, E.STEPS + 1):
        g = _grad(n, 40 + t)
        with torch.no_grad():
            p.copy_(wd)
            if t > 1:
                opt.state[p]["exp_avg"].copy_(md)
                opt.state[p]["exp_avg_sq"].copy_(vd)
        before = wd.detach().cpu().double()
        p.grad = g.to(device)
        opt.step()
        gd.copy_(g)
        ops.adam_step(wd, md, vd, gd, E.LR, t, betas=(b1, 0.999), eps=EPS)
        wt = p.detach().cpu().double()
        wk = wd.cpu().double()
        a32 = wt.float().abs()
        ulp = (torch.nextafter(a32, torch.tensor(math.inf)) - a32).double()
        bound = 2 * ulp + 8 * 2.0 ** -24 * (wt - before).abs()
        excess = (wk - wt).abs() - bound
        assert bool((excess <= 0).all()), f"{device} b1={b1} t={t}: {int((excess > 0).sum())} elements beyond the bound"
