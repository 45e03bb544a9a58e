"""Fused SOM training step, hit histogram and pruning -- the fast path next to the drop-in.

``SomTrainer.step`` performs exactly the arithmetic of one iteration of
/root/reference/train_codebook.py:225-249 + :300-304 (forward with use_gaussian=True, mse_loss,
backward, Adam(betas=(0.5, 0.999)).step, lr halving, neighbourhood decrease), but through the
factorised form of SURVEY.md A.3, never materialising the quantised batch or the N x K Gaussian:

    W~   = T @ W                                   som_filter_ws_f32
    bmu  = argmin_j ||x - W_j||                    som_bmu_nchw_f32
    [Rbar | sse, n] = segsum_bmu(W~[bmu] - x)      som_accumulate_packed_nchw_f32
           (data parallel: ONE all-reduce of that packed buffer here; ragged shares allowed)
    G~   = T @ Rbar                                som_filter_ws_f32 (scale 1)
    Adam(W, (2 / numel) G~), loss = sse / numel    som_adam_dp_f32   (numel from the reduced tail, on the device)

Nothing in the step needs the host: the Adam step count, the global batch size and the loss live in
device memory, so the whole step -- the NCCL all-reduce included -- is captured into a CUDA graph and
replayed (``use_cuda_graph``).  The drop-in ``Codebook`` + torch autograd + torch.optim.Adam path
produces the same update; the tests check both against the reference's outputs.
"""
import torch

from . import ops as _default_ops


class SomTrainer:
    MAX_GRAPHS = 8

    def __init__(self, codebook, lr, neighbourhood_step, lr_step=100000, global_steps=0,
                 betas=(0.5, 0.999), eps=1e-8, ops=None, reduce_fn=None, world_size=1,
                 use_cuda_graph=False, check_nan=False, small_step_kernel=True, overlap_filter=True):
        """``codebook``: a somcb.Codebook on a CUDA device.  ``reduce_fn(packed)`` sums the packed
        accumulator buffer in place across data-parallel ranks (None: single device).

        ``use_cuda_graph``: the step is ~20 launches; small batches (BASELINE config 1: 512 patches per
        step) and strong-scaled data-parallel shards are bound by them, not by the kernels.  With this
        flag the step is captured once per (batch shape, neighbourhood range, lr) into a CUDA graph and
        replayed: the batch is copied into a static buffer first.  ``use_cuda_graph="alias"`` captures on
        the caller's own input buffer instead (one graph per distinct buffer address, at most MAX_GRAPHS
        kept): for loops that refill a few device staging buffers.  The first step always runs eagerly
        (one-time kernel attribute set-up and NCCL communicator creation must not happen during capture).

        ``check_nan``: the reference's ``NaN encountered during training`` guard (train_codebook.py:237-238);
        it reads the loss back, i.e. one host synchronisation per step, so it is off by default.

        ``overlap_filter``: W~ = T @ W is only needed by the accumulation, the search reads W -- so the filter runs on
        a side stream beside norms, operand split and the start of the search (fork / join with stream waits, also
        inside a captured graph) instead of in front of them.  Measured on B200 (graph-replayed C4 step, one GPU,
        alternating A/B inside one process, tools/overlap_ab.py): 1.282 -> 1.259 ms at 262 144 patches, -7.7 us at
        131 072 (an N = 8 rank's share), equal within the run-to-run noise at 1 048 576.  False keeps one stream."""
        self.cb = codebook
        self.lr = float(lr)
        self.neighbourhood_step = int(neighbourhood_step)
        self.lr_step = int(lr_step)
        self.global_steps = int(global_steps)
        self.betas = betas
        self.eps = eps
        self.ops = ops or _default_ops
        self.reduce_fn = reduce_fn
        self.world_size = int(world_size)
        self.check_nan = bool(check_nan)
        self.small_step_kernel = bool(small_step_kernel)    # False: always the separate kernels (tests, A/B)
        self.overlap_filter = bool(overlap_filter)
        self._side = None                                   # side stream of the W~ filter
        self._wt_side = None                                # its output (kept: written on one stream, read on another)
        w = codebook.codebook.weight
        # the reference does not checkpoint Adam state: a resume restarts the moments at zero
        self.m = torch.zeros_like(w, requires_grad=False)
        self.v = torch.zeros_like(w, requires_grad=False)
        self.t = 0
        # Adam's step count lives on the device (the captured graph and the eager path share it): [count, scratch]
        self.t_dev = torch.zeros(2, dtype=torch.int64, device=w.device)
        self.packed = torch.empty(w.numel() + 4, dtype=torch.float32, device=w.device)
        self.last_bmu = None
        self.use_cuda_graph = bool(use_cuda_graph)
        self._graph_alias = use_cuda_graph == "alias"
        self._graphs = {}             # key -> (CUDAGraph, x_static, loss_static)

    @torch.no_grad()
    def step(self, feature_map, bmu=None):
        """One training step on a (local) batch; returns the loss as a 0-dim float64 device
        tensor (global mean squared error, as F.mse_loss over the global batch).  Under ``use_cuda_graph`` the
        tensor is the captured graph's own output buffer: read it (``float(loss)``, ``.clone()``) before the same
        graph is replayed again."""
        if self.use_cuda_graph and bmu is None and self.t >= 1 and feature_map.is_cuda:
            loss = self._graph_step(feature_map)
        else:
            loss = self._eager_step(feature_map, bmu)
        if self.check_nan and bool(torch.isnan(loss)):
            raise Exception("NaN encountered during training")
        return loss

    def _graph_step(self, feature_map):
        cb = self.cb
        # an fp16 / bf16 batch keeps its dtype in the static buffer (half the bytes to copy); anything else is copied as
        # fp32
        dtype = feature_map.dtype if feature_map.dtype in _default_ops.HALF_DTYPES else torch.float32
        alias = self._graph_alias and feature_map.is_contiguous() and feature_map.dtype == dtype
        key = (tuple(feature_map.shape), dtype, float(cb.neighbourhood_range), float(self.lr),
               feature_map.data_ptr() if alias else 0)
        entry = self._graphs.get(key)
        if entry is None:
            if len(self._graphs) >= self.MAX_GRAPHS:
                self._graphs.pop(next(iter(self._graphs)))
            x_static = feature_map if alias else \
                torch.empty(feature_map.shape, dtype=dtype, device=feature_map.device)
            graph = torch.cuda.CUDAGraph()
            torch.cuda.synchronize(feature_map.device)
            # thread_local: the NCCL watchdog thread may touch the CUDA API while we capture
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                loss_static = self._device_step(x_static, None)
            entry = (graph, x_static, loss_static)
            self._graphs[key] = entry
        graph, x_static, loss_static = entry
        if x_static is not feature_map:
            x_static.copy_(feature_map)
        graph.replay()
        self.t += 1
        self.last_bmu = None
        self._bookkeeping()
        # the graph's own loss buffer (overwritten by the next replay of THIS graph): no copy kernel per step
        return loss_static.reshape(())

    def _bookkeeping(self):
        # schedule bookkeeping, in the reference's order (train_codebook.py:247-249, 300-304)
        if self.global_steps % self.lr_step == 0 and self.global_steps > 0:
            self.lr = self.lr * 0.5
        self.global_steps += 1
        if self.global_steps % self.neighbourhood_step == 0:
            self.cb.decrease_neighbourhood(steps=1)

    def _eager_step(self, feature_map, bmu=None):
        loss = self._device_step(feature_map, bmu)
        self.t += 1
        self._bookkeeping()
        return loss.reshape(())

    def _device_step(self, feature_map, bmu):
        """Enqueue one step on the current stream (eagerly or under graph capture); returns the (1,) float64
        device tensor the loss is written to."""
        ops = self.ops
        cb = self.cb
        w = cb.codebook.weight.data
        x, geom = cb._input(feature_map, require_cuda=getattr(ops, 'REQUIRES_CUDA', True), allow_half=True)
        k, d = cb.num_embeddings, cb.embedding_dim
        rng = cb.neighbourhood_range
        kd = k * d

        small = (bmu is None and self.reduce_fn is None and self.small_step_kernel
                 and cb.bmu_variant == ops.SOM_BMU_AUTO and getattr(ops, "step_small_supported", None) is not None
                 and ops.step_small_supported(geom, k, rng))
        x = self._half_input(x, geom, staged=bmu is None and not small)
        if small:
            # small problems (BASELINE config 1): the whole step is ONE cooperative kernel, a launch costs more than
            # any of the step's kernels at this size
            loss, self.last_bmu = ops.step_small(x, geom, w, self.m, self.v, rng, self.lr, self.t_dev,
                                                 betas=self.betas, eps=self.eps)
            return loss

        wt, side = self._fork_filter(w, rng)
        x_acc, geom_acc = x, geom
        if bmu is None:
            bmu, x_acc, geom_acc = self._search(x, geom, w)
        self._join_filter(side)
        packed = self.packed
        ops.accumulate_packed(x_acc, geom_acc, bmu, wt, k, packed=packed)
        if self.reduce_fn is not None:
            # ONE collective per step: Rbar, the squared error (float pair) and the patch count travel together
            self.reduce_fn(packed)
        grad = ops.neighbourhood_filter(packed[:kd].view(k, d), rng, scale=1.0)
        loss = ops.adam_step_dp(w, self.m, self.v, grad, d, self.lr, self.t_dev, packed[kd:], betas=self.betas,
                                eps=self.eps)
        self.last_bmu = bmu
        return loss

    def _fork_filter(self, w, rng):
        """W~ = T @ W (models/Codebook.py:112-130 forward).  The search that follows does not read it, so on a CUDA
        device it is enqueued on a side stream that forks from the current one; ``_join_filter`` makes the current
        stream wait for it before the accumulation.  Returns (W~, side stream or None)."""
        ops = self.ops
        if not (self.overlap_filter and w.is_cuda):
            return ops.neighbourhood_filter(w, rng), None
        cur = torch.cuda.current_stream(w.device)
        if self._side is None:
            self._side = torch.cuda.Stream(device=w.device)
        if self._wt_side is None or self._wt_side.shape != w.shape or self._wt_side.device != w.device:
            self._wt_side = torch.empty_like(w)
        self._side.wait_stream(cur)
        with torch.cuda.stream(self._side):
            ops.neighbourhood_filter(w, rng, out=self._wt_side)
        return self._wt_side, self._side

    @staticmethod
    def _join_filter(side):
        if side is not None:
            torch.cuda.current_stream(side.device).wait_stream(side)

    def _can_stage(self, geom):
        ops, cb = self.ops, self.cb
        can = getattr(ops, "bmu_can_stage", None)
        return can is not None and ops.n_patches_of(geom) > 0 and can(geom, cb.num_embeddings, cb.bmu_variant)

    def _half_input(self, x, geom, staged):
        """An fp16 / bf16 batch keeps its dtype only where the step's search reads it itself and writes the fp32 staging
        rows that the accumulation reads (``staged``: the step searches with the separate kernels; the staging kernel is
        the one that reads 16-bit values).  Otherwise it is upcast once, exactly, and that copy feeds every kernel of
        the step."""
        if x.dtype not in _default_ops.HALF_DTYPES or (staged and self._can_stage(geom)):
            return x
        return self.ops.upcast_bf16(x) if x.dtype == torch.bfloat16 else self.ops.upcast_f16(x)

    def _search(self, x, geom, w):
        """BMU search of the step.  Where the kernel can emit it, also the patch-major staging copy of the patch rows:
        the segmented gather of the update then reads one contiguous row per patch (returns the buffer and geometry
        the accumulation should read: the staging rows, or x itself)."""
        ops, cb = self.ops, self.cb
        cn = ops.prepare_codebook(w)
        if self._can_stage(geom):
            npat, d = ops.n_patches_of(geom), ops.dim_of(geom)
            stage = torch.empty(npat, d, dtype=torch.float32, device=x.device)
            bmu = ops.bmu(x, geom, w, cn, variant=cb.bmu_variant, stage=stage)
            return bmu, stage, ops.flat_geometry(npat, d)
        return ops.bmu(x, geom, w, cn, variant=cb.bmu_variant), x, geom

    def checkpoint_dict(self, image_channel):
        """The reference's checkpoint layout (train_codebook.py:271-278)."""
        cb = self.cb
        return {"patch_dim": cb.patch_dim, "image_dim": cb.image_dim, "image_C": image_channel,
                "num_embeddings": cb.num_embeddings, "neighbourhood_range": cb.neighbourhood_range,
                "global_steps": self.global_steps, "checkpoint": cb.state_dict()}


@torch.no_grad()
def bmu_histogram(codebook, batches, counts=None, ops=None):
    """Hit counts over an iterable of feature-map batches (prune_codebook.py:129-142), kept on
    the device: one BMU launch + one histogram launch per batch, no host round trip."""
    ops = ops or _default_ops
    for fmap in batches:
        idx = codebook.get_patches_bmu(fmap)
        counts = ops.histogram(idx, codebook.num_embeddings, counts)
    if counts is None:
        raise ValueError("bmu_histogram: no batches")
    return counts


@torch.no_grad()
def prune_codebook(codebook, counts, prune_threshold, image_channel=None, global_steps=0, ops=None):
    """Keep units with count >= threshold in ascending index order and build the smaller
    codebook + the reference's checkpoint dict (prune_codebook.py:144-178).  The pruned codebook keeps the weights'
    dtype (fp32, or fp16 / bf16 for a 16-bit codebook)."""
    from .codebook import Codebook
    ops = ops or _default_ops
    keep = torch.nonzero(counts >= prune_threshold).flatten().to(torch.int64)
    rows = ops.gather_rows(codebook.codebook.weight.data, keep)
    if image_channel is None:
        image_channel = codebook.embedding_dim // (codebook.patch_dim[0] * codebook.patch_dim[1])
    new_cb = Codebook(patch_dim=codebook.patch_dim, image_dim=codebook.image_dim,
                      image_channel=image_channel, num_embeddings=int(keep.numel()),
                      init_neighbour_range=codebook.neighbourhood_range).to(device=rows.device, dtype=rows.dtype)
    new_cb.codebook.weight.data.copy_(rows)
    ck = {"patch_dim": codebook.patch_dim, "image_dim": codebook.image_dim, "image_C": image_channel,
          "num_embeddings": int(keep.numel()), "neighbourhood_range": codebook.neighbourhood_range,
          "global_steps": global_steps, "checkpoint": new_cb.state_dict()}
    return new_cb, keep, ck
