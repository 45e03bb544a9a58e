"""Multi-GPU SOM codebook: one process per GPU, torch.distributed (NCCL over NVLink) as plumbing.

Two shardings (SURVEY.md 8e):

* patch-sharded data parallel (``DataParallelSom``): every rank holds the full codebook and Adam
  state, takes about 1/R of the step's feature maps (shares may be ragged), runs BMU + per-unit
  accumulation locally, then ONE all-reduce(sum) of the packed [Rbar (K*D fp32) | SSE (2 fp32) |
  patch count (2 fp32)] buffer; filter + Adam are replicated, so replicas stay bit-identical (the
  all-reduce returns identical bits everywhere).  The whole step, collective included, is captured
  in a CUDA graph (``use_cuda_graph``).
  BMU-only / histogram workloads need no exchange beyond a final all-reduce of K int64 counts.
* unit-sharded search (``sharded_bmu``): rank r owns units [lo_r, hi_r); patches are replicated;
  each rank returns (reduced distance, global index) candidates from the same kernels as the
  unsharded path, ONE all-gather of a packed 12 B/patch/rank record block, then som_merge_candidates
  (smaller distance, tie -> smaller global index == the single-device first-minimum rule).  The
  kernel plan (split arithmetic, unit / feature splits) depends on the shard's shape, so picks may
  differ from the unsharded search between candidates closer than the 1e-6 near-tie rule.

``ops`` is injectable so the host logic (sharding arithmetic, collective wiring) is testable
under gloo on CPU with a test double; the default is the CUDA library, which raises on CPU.
"""
import torch
import torch.distributed as dist

from . import ops as _default_ops
from .trainer import SomTrainer


def shard_bounds(total, world_size, rank):
    """Contiguous near-equal shard [lo, hi) of ``total`` items for ``rank``."""
    base, rem = divmod(int(total), int(world_size))
    lo = rank * base + min(rank, rem)
    hi = lo + base + (1 if rank < rem else 0)
    return lo, hi


def split_batch(feature_map, world_size, rank):
    """Contiguous near-equal slice of the batch dimension for ``rank``.  Shares may be ragged (and empty when there
    are fewer feature maps than ranks): the step all-reduces the patch count next to the accumulators."""
    lo, hi = shard_bounds(feature_map.shape[0], world_size, rank)
    return feature_map[lo:hi]


class PeerMemory:
    """Symmetric (peer-mapped + NVSwitch-multicast) device allocations of one process group.  torch's symmetric-memory
    allocator is the plumbing (allocation, handle exchange, multicast binding); the kernels that use the addresses
    are libsomcb's (som_peer_*)."""

    def __init__(self, group, device):
        import torch.distributed._symmetric_memory as symm_mem
        self._sm = symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.device = device
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self._keep = []
        sig = self.alloc(_default_ops.peer_signal_bytes() // 4, torch.int32)
        sig[0].zero_()
        torch.cuda.synchronize(device)
        dist.barrier(group=group)
        self.signal_ptrs = sig[2]

    def alloc(self, numel, dtype=torch.float32):
        """Returns (local tensor, multicast address or 0, list of peer addresses)."""
        t = self._sm.empty(int(numel), dtype=dtype, device=self.device)
        hdl = self._sm.rendezvous(t, self.group)
        mc = int(hdl.multicast_ptr) if hdl.has_multicast_support else 0
        self._keep.append((t, hdl))
        return t, mc, [int(p) for p in hdl.buffer_ptrs]

    @staticmethod
    def available(device):
        try:
            import torch.distributed._symmetric_memory  # noqa: F401
        except Exception:  # noqa: BLE001
            return False
        return torch.cuda.is_available() and torch.cuda.get_device_capability(device)[0] >= 9


class DataParallelSom(SomTrainer):
    """SomTrainer whose accumulators are summed across the process group once per step.

    ``tail`` selects what follows the local accumulation:

    * ``"nccl"``: ONE ``all_reduce`` of the packed buffer, then every rank runs both filters and Adam on the whole
      codebook (replicated);
    * ``"peer"``: the sharded tail over NVLink / NVSwitch multicast memory (csrc/som_peer.cu).  Rank r owns units
      [lo_r, hi_r): it pulls the in-switch-reduced accumulator rows of its slice plus the filter's halo
      (``som_peer_reduce_rows_f32``: the reduce-scatter half, with overlap), filters them, runs Adam on its rows and
      stores the new rows into every rank's codebook (``som_peer_adam_slice_f32``: the all-gather fused into the
      update); ``W~ = T @ W`` is computed by every rank for the whole codebook (``wt="full"``, default) or per slice
      and multicast the same way (``wt="slice"``).  Of the non-shrinking part of a strong-scaled step (two
      whole-codebook filters, Adam, a 4 MB all-reduce) the gradient filter, Adam and the reduction become 1/R-sized.  Falls back to one in-switch all-reduce (``som_peer_allreduce_f32``) + replicated tail when
      the halo makes slicing pointless (slice + halo >= 3/4 of the units);
    * ``"auto"`` (default): ``"peer"`` when symmetric memory with multicast is available, else ``"nccl"``.

    Replicas stay bit-identical in every mode: a row is computed once, by its owner, and multicast."""

    def __init__(self, codebook, lr, neighbourhood_step, group=None, tail="auto", wt="full", **kw):
        self.group = group
        # peer tail: "full" (default) lets every rank compute W~ = T @ W for the whole codebook itself; "slice" computes
        # it per slice and multicasts the rows, which costs one more cross-rank barrier per step (measured at 8 ranks:
        # 0.781 ms per step against 0.749 ms with "full" -- the slice filter saves 17 us, the barrier costs more)
        self.wt_mode = wt
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        super().__init__(codebook, lr, neighbourhood_step, world_size=world,
                         reduce_fn=self._allreduce if world > 1 else None, **kw)
        self.tail = "nccl"
        self.peer = None
        w = codebook.codebook.weight
        want_peer = tail in ("auto", "peer") and world > 1 and w.is_cuda and self.ops is _default_ops
        if want_peer and codebook.embedding_dim % 4 == 0 and PeerMemory.available(w.device):
            try:
                self._setup_peer(w.device)
            except Exception:  # noqa: BLE001
                if tail == "peer":
                    raise
                self.peer = None
        if tail == "peer" and self.peer is None and world > 1:
            raise RuntimeError("DataParallelSom(tail='peer'): NVSwitch multicast symmetric memory is not available")

    def _setup_peer(self, device):
        cb = self.cb
        k, d = cb.num_embeddings, cb.embedding_dim
        pm = PeerMemory(self.group, device)
        packed, mc_packed, peer_packed = pm.alloc(k * d + 4)
        w_sym, mc_w, _ = pm.alloc(k * d)
        wt_sym, mc_wt, _ = pm.alloc(k * d)
        if not (mc_packed and mc_w and mc_wt):
            raise RuntimeError("no multicast support")
        with torch.no_grad():
            w_sym.copy_(cb.codebook.weight.data.reshape(-1))
            cb.codebook.weight.data = w_sym.view(k, d)       # the parameter now lives in peer-mapped memory
        self.packed = packed
        self.peer = pm
        self._mc = {"packed": mc_packed, "w": mc_w, "wt": mc_wt}
        self._peer_packed = peer_packed
        self._wt = wt_sym.view(k, d)
        self._tail_local = torch.empty(4, dtype=torch.float32, device=device)
        self.tail = "peer"
        torch.cuda.synchronize(device)
        dist.barrier(group=self.group)

    def _allreduce(self, packed):
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=self.group)

    def _slices(self, h):
        """(lo, hi, g0, g1) of this rank, the largest slice and the largest slice + halo of any rank."""
        k = self.cb.num_embeddings
        pm = self.peer
        spans = [shard_bounds(k, pm.world, r) for r in range(pm.world)]
        halo = [(max(0, lo - h), min(k, hi + h)) if hi > lo else (lo, lo) for lo, hi in spans]
        lo, hi = spans[pm.rank]
        g0, g1 = halo[pm.rank]
        return lo, hi, g0, g1, max(b - a for a, b in spans), max(b - a for a, b in halo)

    def _device_step(self, feature_map, bmu):
        if self.peer is None:
            return super()._device_step(feature_map, bmu)
        ops, cb, pm = self.ops, self.cb, self.peer
        w = cb.codebook.weight.data
        x, geom = cb._input(feature_map, allow_half=True)
        x = self._half_input(x, geom, staged=bmu is None)
        k, d = cb.num_embeddings, cb.embedding_dim
        rng = cb.neighbourhood_range
        kd = k * d
        lo, hi, g0, g1, max_own, max_halo = self._slices(ops.filter_half_width(k, rng))
        sig, rank, world = pm.signal_ptrs, pm.rank, pm.world
        sliced = 4 * max_halo <= 3 * k
        if sliced and self.wt_mode == "slice":
            # W~ rows of the own slice from W[g0:g1] (complete on every rank: the previous step ended with the barrier
            # of the weight broadcast), multicast into every rank's W~
            if hi > lo:
                wth = ops.neighbourhood_filter(w[g0:g1], rng)
                src = wth[lo - g0:hi - g0]
            else:
                src = self._tail_local[0:0]                  # no rows of its own: takes part in the barrier only
            ops.peer_bcast_rows(src, self._mc["wt"] + lo * d * 4, max_own * d, rank, world, sig, 0)
            wt, side = self._wt, None
        else:
            wt, side = self._fork_filter(w, rng)             # beside norms / operand split / the start of the search
        x_acc, geom_acc = x, geom
        if bmu is None:
            bmu, x_acc, geom_acc = self._search(x, geom, w)
        self._join_filter(side)
        ops.accumulate_packed(x_acc, geom_acc, bmu, wt, k, packed=self.packed)
        if sliced:
            rsum = torch.empty(max(1, max_halo), d, dtype=torch.float32, device=w.device)
            if hi > lo:
                # reduce-scatter fused into the filter's read: G rows = T @ (sum over ranks of Rbar rows [g0, g1))
                gh = torch.empty(g1 - g0, d, dtype=torch.float32, device=w.device)
                ops.peer_reduce_filter_rows(self._mc["packed"], self._peer_packed, k, d, g0, g1, max_halo, rng, rsum, gh,
                                            self._tail_local, rank, world, sig, 1)
                g_rows = gh[lo - g0:hi - g0]
            else:
                ops.peer_reduce_rows(self._mc["packed"], self._peer_packed, k, d, g0, g1, max_halo, rsum,
                                     self._tail_local, rank, world, sig, 1)
                g_rows = self._tail_local[0:0]
            loss = ops.peer_adam_slice(w[lo:hi], self._mc["w"] + lo * d * 4, self.m.data[lo:hi], self.v.data[lo:hi],
                                       g_rows, max_own * d, d, self.lr, self.t_dev, self._tail_local, rank, world,
                                       sig, 2, betas=self.betas, eps=self.eps)
        else:
            ops.peer_allreduce(self._mc["packed"], kd + 4, rank, world, sig, 1, w.device,
                               peer_ptrs=self._peer_packed, tail_out=self._tail_local)
            grad = ops.neighbourhood_filter(self.packed[:kd].view(k, d), rng, scale=1.0)
            loss = ops.adam_step_dp(w, self.m, self.v, grad, d, self.lr, self.t_dev, self._tail_local,
                                    betas=self.betas, eps=self.eps)
        self.last_bmu = bmu
        return loss

    def broadcast_weights(self, src=0):
        """Make every replica start from rank ``src``'s codebook."""
        dist.broadcast(self.cb.codebook.weight.data, src=src, group=self.group)


@torch.no_grad()
def sharded_bmu(x, geom, weight_shard, unit_offset, group=None, ops=None, c_norm2=None):
    """Unit-sharded BMU.  ``weight_shard``: this rank's rows [unit_offset, unit_offset + K_r).
    ``x`` is the same on every rank.  Returns the global indices (n_patches,) on every rank."""
    ops = ops or _default_ops
    idx, rd = ops.bmu(x, geom, weight_shard, c_norm2, unit_offset=unit_offset, want_rd=True)
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return idx
    n = idx.numel()
    # ONE all-gather of a packed 12-byte-per-patch record block [idx (n int64) | rd (n fp32)] per rank
    send = torch.empty(3 * n, dtype=torch.int32, device=idx.device)
    send[:2 * n].view(torch.int64).copy_(idx)
    send[2 * n:].view(torch.float32).copy_(rd)
    recv = torch.empty(world * 3 * n, dtype=torch.int32, device=idx.device)
    dist.all_gather_into_tensor(recv, send, group=group)      # rank-major: row r = rank r
    recv = recv.view(world, 3 * n)
    all_idx = recv[:, :2 * n].contiguous().view(torch.int64)
    all_rd = recv[:, 2 * n:].contiguous().view(torch.float32)
    merged, _ = ops.merge_candidates(all_rd.view(world, n), all_idx.view(world, n))
    return merged


@torch.no_grad()
def sharded_histogram(idx, lo, hi, counts=None, ops=None):
    """Counts of this rank's own unit range [lo, hi) from replicated merged indices: no reduction
    is needed afterwards -- the global histogram is the concatenation over ranks."""
    ops = ops or _default_ops
    return ops.histogram(idx - lo, hi - lo, counts)


@torch.no_grad()
def allreduce_counts(counts, group=None):
    """Patch-sharded histogram: sum the K int64 counts across ranks."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    return counts
