"""Host-buffer tokeniser: the end-to-end BMU path with HOST inputs and outputs.

Models what train_quantized_transformer.py:404-421 / prune_codebook.py:133-138 do per batch
(feature maps arrive in host memory, ``.to(device)``, get_patches_bmu, indices come back), as a
three-stage pipeline over pinned buffers: H2D copy of chunk i+1 and D2H copy of chunk i-1 overlap
the BMU kernel of chunk i on separate streams, ordered by events.
"""
import os

import torch

from . import ops as _ops


def bind_host_to_gpu_node(device=None):
    """Pin the calling process to the CPUs of the NUMA node the GPU hangs off, so that pinned staging buffers
    allocated afterwards (first touch) live in that node's memory and host<->device copies do not cross sockets.
    With one process per GPU on an 8-GPU box the per-GPU copy rate otherwise drops when several ranks stage out of
    the other socket's memory.  Returns the node number, or None when the topology is not exposed (single-node
    hosts, containers without sysfs): then nothing is changed."""
    try:
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        props = torch.cuda.get_device_properties(dev)
        bdf = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except (OSError, ValueError, AttributeError, RuntimeError):
        return None


class HostTokenizer:
    def __init__(self, codebook, chunk_fmaps=4096, depth=3):
        self.cb = codebook
        self.chunk = int(chunk_fmaps)
        self.depth = int(depth)
        w = codebook.codebook.weight
        if not w.is_cuda:
            raise RuntimeError("HostTokenizer needs the codebook on a CUDA device (no CPU fallback)")
        self.device = w.device
        self._bufs = None
        self.done = None

    def _alloc(self, c, h, w, seq, dtype):
        key = (c, h, w, seq, dtype)
        if self._bufs is not None and self._bufs[0] == key:
            return self._bufs[1]
        dev = self.device
        slots = []
        for _ in range(self.depth):
            slots.append({
                "x": torch.empty(self.chunk, c, h, w, dtype=dtype, device=dev),
                "idx": torch.empty(self.chunk * seq, dtype=torch.int64, device=dev),
                "h2d": torch.cuda.Event(), "comp": torch.cuda.Event(), "d2h": torch.cuda.Event(),
            })
        streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
        self._bufs = (key, (slots, streams))
        return self._bufs[1]

    @torch.no_grad()
    def tokenize(self, fmaps_host, out_host=None, sync=True):
        """fmaps_host: (N, C, H, W) fp32, fp16 or bf16 host tensor (pinned for async copies; a 16-bit batch is copied
        as it is, half the bytes, and searched as if it were ``fmaps_host.float()``).  Returns the (N, Seq) int64 host tensor of BMU indices (``out_host`` if given, pinned otherwise).

        With ``sync=True`` (default) the call returns only after the last device-to-host copy has landed and the
        last host-to-device copy has been read: the returned indices are valid and ``fmaps_host`` may be refilled.
        With ``sync=False`` the copies may still be in flight on return; wait on ``self.done`` (a CUDA event covering
        both copy streams) -- ``self.done.synchronize()`` -- before touching either host buffer."""
        cb = self.cb
        n, c, h, w = fmaps_host.shape
        geom1 = _ops.geometry((1, c, h, w), cb.patch_dim)
        seq = _ops.n_patches_of(geom1)
        if out_host is None:
            out_host = torch.empty(n, seq, dtype=torch.int64, pin_memory=True)
        dtype = fmaps_host.dtype if fmaps_host.dtype in _ops.HALF_DTYPES else torch.float32
        slots, (s_in, s_out) = self._alloc(c, h, w, seq, dtype)
        compute = torch.cuda.current_stream(self.device)
        weight = cb.codebook.weight.detach()
        norms = cb._norms()
        start = torch.cuda.Event()
        start.record(compute)
        s_in.wait_event(start)
        s_out.wait_event(start)
        n_chunks = (n + self.chunk - 1) // self.chunk
        for i in range(n_chunks):
            sl = slots[i % self.depth]
            lo, hi = i * self.chunk, min(n, (i + 1) * self.chunk)
            m = hi - lo
            if i >= self.depth:
                s_in.wait_event(sl["comp"])          # x slot consumed by chunk i - depth
            with torch.cuda.stream(s_in):
                sl["x"][:m].copy_(fmaps_host[lo:hi], non_blocking=True)
                sl["h2d"].record(s_in)
            compute.wait_event(sl["h2d"])
            if i >= self.depth:
                compute.wait_event(sl["d2h"])        # idx slot drained by chunk i - depth
            geom = _ops.geometry((m, c, h, w), cb.patch_dim)
            _ops.bmu(sl["x"][:m], geom, weight, norms, variant=cb.bmu_variant, out=sl["idx"][:m * seq])
            sl["comp"].record(compute)
            s_out.wait_event(sl["comp"])
            with torch.cuda.stream(s_out):
                out_host[lo:hi].view(-1).copy_(sl["idx"][:m * seq], non_blocking=True)
                sl["d2h"].record(s_out)
        compute.wait_stream(s_out)
        compute.wait_stream(s_in)
        self.done = torch.cuda.Event()
        self.done.record(compute)
        if sync:
            # wait_stream only orders GPU streams; the HOST must not read out_host (or refill fmaps_host) earlier
            self.done.synchronize()
        return out_host


class PendingLoss:
    """Loss of an enqueued step: a pinned host scalar that becomes valid when ``event`` has completed."""

    def __init__(self, host, event):
        self.host, self.event = host, event

    def item(self):
        self.event.synchronize()
        return float(self.host)


class HostTrainer:
    """SOM training from HOST batches: what the loop of train_codebook.py:216-249 does per step (the DataLoader's
    batch arrives in host memory, ``.to(device)``, step, ``loss.item()``), as a pipeline over ``depth`` device staging
    buffers: the host-to-device copy of batch i+1 runs on a copy stream while step i computes, the step itself is
    the trainer's CUDA graph captured on the staging buffer (``use_cuda_graph="alias"``), and the loss comes back
    through a pinned scalar.  ``trainer`` is a SomTrainer / DataParallelSom; under data parallelism every rank
    feeds its own share."""

    def __init__(self, trainer, depth=2):
        self.tr = trainer
        self.depth = int(depth)
        w = trainer.cb.codebook.weight
        if not w.is_cuda:
            raise RuntimeError("HostTrainer needs the codebook on a CUDA device (no CPU fallback)")
        self.device = w.device
        self._slots = None
        self._i = 0
        self._copy = torch.cuda.Stream(self.device)

    def _alloc(self, shape, dtype):
        key = (tuple(shape), dtype)
        if self._slots is not None and self._slots[0] == key:
            return self._slots[1]
        slots = [{"x": torch.empty(shape, dtype=dtype, device=self.device),
                  "loss": torch.empty((), dtype=torch.float64, pin_memory=True),
                  "h2d": torch.cuda.Event(), "done": None} for _ in range(self.depth)]
        self._slots = (key, slots)
        return slots

    @torch.no_grad()
    def step(self, fmaps_host):
        """Enqueue copy + step for one (local) host batch (pinned for asynchronous copies; fp16 / bf16 batches are
        staged as they are and trained on as if they were ``fmaps_host.float()``); returns a PendingLoss.
        ``fmaps_host`` may be refilled once ``h2d_done()`` of this call has completed (or after the loss is read)."""
        slots = self._alloc(fmaps_host.shape,
                            fmaps_host.dtype if fmaps_host.dtype in _ops.HALF_DTYPES else torch.float32)
        sl = slots[self._i % self.depth]
        self._i += 1
        compute = torch.cuda.current_stream(self.device)
        if sl["done"] is not None:
            self._copy.wait_event(sl["done"])         # the step that last read this staging buffer
        else:
            self._copy.wait_stream(compute)
        with torch.cuda.stream(self._copy):
            sl["x"].copy_(fmaps_host, non_blocking=True)
            sl["h2d"].record(self._copy)
        compute.wait_event(sl["h2d"])
        loss = self.tr.step(sl["x"])
        sl["loss"].copy_(loss, non_blocking=True)
        done = torch.cuda.Event()
        done.record(compute)
        sl["done"] = done
        self.last_h2d = sl["h2d"]
        return PendingLoss(sl["loss"], done)

    def h2d_done(self):
        """Event after which the host batch of the LAST step() call has been read completely."""
        return self.last_h2d
