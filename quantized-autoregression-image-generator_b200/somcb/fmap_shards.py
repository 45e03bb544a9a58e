"""Packed feature-map shards: the data format either side of the BMU path (SURVEY.md 8f rank 3).

The reference stores one ``.npy`` per feature map, at most 1000 per folder, indexed by a TinyDB
JSON file (``generate_fmap_dataset.py:42-72``), and reads them back one ``np.load`` at a time in
DataLoader workers (``dataset_loader/feature_map_dataset.py:22-42``).  At 1e8-1e9 patches/s that
reader, not the GPU, bounds tokenisation and pruning.  This module packs the same data into a few
large, memory-mappable shards and streams them into pinned batches:

    shard file  = 64-byte header | n * C*H*W values, C-contiguous (the reference's layout)
    header v1   = b"SOMFMAP1" | u32 version = 1 | u32 C | u32 H | u32 W | u64 n | zero padding to 64 bytes
                  (float32 values, the reference's dtype)
    header v2   = the same with version = 2 and a u32 dtype code at byte 32 (1 = float16, 2 = bfloat16): half
                  the bytes to read and to copy to the device; the searches treat the values as what they are (as
                  ``.float()``).  bfloat16 values are stored as their raw 16-bit patterns (numpy has no bfloat16:
                  they are read through ``np.uint16`` and handed out as ``torch.bfloat16`` tensors)

* ``convert_reference_dataset`` reads the reference layout (TinyDB json -> ``fmap_path`` entries, in
  document order) and writes shards; ``image_path`` is kept in a side ``index.json``.
* ``ShardReader`` memory-maps shards and yields ``(lo, hi, pinned_tensor_view)`` batches that feed
  ``HostTokenizer.tokenize`` / ``bmu_histogram`` directly.  Pure host code: numpy + torch pinned memory.
"""
import json
import os
import struct

import numpy as np
import torch

MAGIC = b"SOMFMAP1"
HEADER_BYTES = 64
VERSION = 1                       # float32 shards
VERSION_DTYPE = 2                 # shards of another dtype: u32 code at byte 32
DTYPE_CODES = {1: torch.float16, 2: torch.bfloat16}
# how the values of each dtype are stored and memory-mapped
_STORAGE = {torch.float32: np.dtype(np.float32), torch.float16: np.dtype(np.float16),
            torch.bfloat16: np.dtype(np.uint16)}
_FROM_NUMPY = {np.dtype(np.float32): torch.float32, np.dtype(np.float16): torch.float16}


def _shard_dtype(dtype):
    """The torch dtype of a shard dtype given as a torch dtype or as anything ``np.dtype`` takes."""
    t = dtype if isinstance(dtype, torch.dtype) else None
    if t is None:
        try:
            t = _FROM_NUMPY.get(np.dtype(dtype))
        except TypeError:
            pass
    if t not in _STORAGE:
        raise ValueError(f"shards hold float32, float16 or bfloat16 values, not {dtype}")
    return t


def _header(c, h, w, n, dtype):
    if dtype == torch.float32:
        head = MAGIC + struct.pack("<IIIIQ", VERSION, c, h, w, n)
    else:
        code = next(k for k, v in DTYPE_CODES.items() if v == dtype)
        head = MAGIC + struct.pack("<IIIIQI", VERSION_DTYPE, c, h, w, n, code)
    return head + b"\0" * (HEADER_BYTES - len(head))


def _read_header(path):
    with open(path, "rb") as f:
        head = f.read(HEADER_BYTES)
    if len(head) != HEADER_BYTES or head[:8] != MAGIC:
        raise ValueError(f"{path}: not a feature-map shard")
    version, c, h, w, n = struct.unpack("<IIIIQ", head[8:32])
    if version == VERSION:
        dtype = torch.float32
    elif version == VERSION_DTYPE:
        (code,) = struct.unpack("<I", head[32:36])
        if code not in DTYPE_CODES:
            raise ValueError(f"{path}: unknown dtype code {code}")
        dtype = DTYPE_CODES[code]
    else:
        raise ValueError(f"{path}: shard version {version}, expected {VERSION} or {VERSION_DTYPE}")
    expect = HEADER_BYTES + n * c * h * w * _STORAGE[dtype].itemsize
    if os.path.getsize(path) != expect:
        raise ValueError(f"{path}: size {os.path.getsize(path)} != {expect} implied by the header")
    return c, h, w, n, dtype


def read_header(path):
    """(C, H, W, n) of a shard of either version."""
    return _read_header(path)[:4]


def shard_torch_dtype(path):
    """torch dtype of a shard's values: float32, float16 or bfloat16."""
    return _read_header(path)[4]


def shard_dtype(path):
    """numpy dtype of a shard's values (float32 for version 1, or float16).  numpy has no bfloat16: a bfloat16 shard
    raises ``ValueError`` (ask ``shard_torch_dtype``)."""
    dtype = shard_torch_dtype(path)
    if dtype == torch.bfloat16:
        raise ValueError(f"{path}: a bfloat16 shard has no numpy dtype; use shard_torch_dtype")
    return _STORAGE[dtype]


def _numpy_view(t):
    """numpy view of a CPU tensor's storage (the raw 16-bit patterns for bfloat16)."""
    return t.view(torch.int16).numpy().view(np.uint16) if t.dtype == torch.bfloat16 else t.numpy()


def _bf16_bits(fmaps):
    """bfloat16 bit patterns of ``fmaps``: a bfloat16 tensor as it is, anything else rounded from float32 to nearest
    even (torch's conversion)."""
    if isinstance(fmaps, torch.Tensor) and fmaps.dtype == torch.bfloat16:
        t = fmaps.detach().cpu()
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(fmaps), dtype=np.float32)).to(torch.bfloat16)
    return _numpy_view(t.contiguous())


def write_shard(path, fmaps, dtype=np.float32):
    """fmaps: (n, C, H, W) array-like, stored as ``dtype`` (float32: version 1; float16 or torch.bfloat16: version 2).
    float16 values are rounded to nearest by numpy's conversion; bfloat16 values are the float32 values rounded to
    nearest even by torch's (a bfloat16 tensor is stored as it is).  Returns n."""
    dtype = _shard_dtype(dtype)
    if dtype == torch.bfloat16:
        arr = _bf16_bits(fmaps)
    else:
        arr = np.ascontiguousarray(np.asarray(fmaps), dtype=_STORAGE[dtype])
    if arr.ndim != 4:
        raise ValueError("write_shard expects (n, C, H, W)")
    n, c, h, w = arr.shape
    with open(path, "wb") as f:
        f.write(_header(c, h, w, n, dtype))
        f.write(arr.tobytes(order="C"))
    return n


def reference_entries(db_json_path):
    """The documents of the reference's TinyDB file in document-id order (generate_fmap_dataset.py
    :62-72 inserts them in file_index order).  TinyDB's on-disk form is
    {"_default": {"1": {...}, "2": {...}}}; no tinydb import is needed to read it."""
    with open(db_json_path, "r") as f:
        db = json.load(f)
    table = db.get("_default", db)
    if not isinstance(table, dict) or len(table) == 0:
        raise Exception("No data found.")          # same message as feature_map_dataset.py:29
    return [table[k] for k in sorted(table, key=lambda s: int(s))]


def convert_reference_dataset(db_json_path, out_dir, fmaps_per_shard=65536, path_root=None, dtype=np.float32):
    """Pack the reference's per-file dataset into shards of ``dtype`` (float32, float16 or torch.bfloat16, see
    ``write_shard``).
    ``path_root`` re-bases relative ``fmap_path`` entries.  Returns the list of shard paths; writes ``index.json``
    beside them."""
    dtype = _shard_dtype(dtype)
    # bfloat16: the reference's .float() first, then one rounding in write_shard
    load_as = np.float32 if dtype == torch.bfloat16 else _STORAGE[dtype]
    entries = reference_entries(db_json_path)
    os.makedirs(out_dir, exist_ok=True)
    shards, index, batch = [], [], []

    def flush():
        if not batch:
            return
        path = os.path.join(out_dir, f"fmaps_{len(shards):05d}.shard")
        write_shard(path, np.stack(batch), dtype=dtype)
        shards.append(path)
        batch.clear()

    for i, doc in enumerate(entries):
        p = doc["fmap_path"]
        if path_root is not None and not os.path.isabs(p):
            p = os.path.join(path_root, p)
        with open(p, "rb") as f:
            fmap = np.load(f, allow_pickle=False)           # as feature_map_dataset.py:38-39
        batch.append(np.asarray(fmap, dtype=load_as))       # .float() of :42 (float16: one rounding)
        index.append({"i": i, "shard": len(shards), "row": len(batch) - 1,
                      "image_path": doc.get("image_path")})
        if len(batch) == fmaps_per_shard:
            flush()
    flush()
    with open(os.path.join(out_dir, "index.json"), "w") as f:
        json.dump({"shards": [os.path.basename(s) for s in shards], "entries": index}, f)
    return shards


class ShardReader:
    """Sequential reader over shards: memory-mapped, double-buffered pinned staging."""

    def __init__(self, shard_paths, batch_fmaps=4096, pin=True, depth=2):
        if isinstance(shard_paths, str):
            shard_paths = [shard_paths]
        if len(shard_paths) == 0:
            raise Exception("No data found.")
        self.paths = list(shard_paths)
        self.shape = None
        self.torch_dtype = None       # dtype of every shard (batches come in it)
        self.counts = []
        for p in self.paths:
            c, h, w, n, dt = _read_header(p)
            if self.shape is None:
                self.shape, self.torch_dtype = (c, h, w), dt
            elif self.shape != (c, h, w):
                raise ValueError(f"{p}: shape {(c, h, w)} differs from {self.shape}")
            elif self.torch_dtype != dt:
                raise ValueError(f"{p}: dtype {dt} differs from {self.torch_dtype}")
            self.counts.append(n)
        # numpy dtype of the shards' values (None for bfloat16, which numpy lacks)
        self.dtype = None if self.torch_dtype == torch.bfloat16 else _STORAGE[self.torch_dtype]
        self.batch = int(batch_fmaps)
        self.pin = bool(pin) and torch.cuda.is_available()
        self.depth = int(depth)
        self._bufs = None
        self._busy = {}               # staging slot -> CUDA event of the last asynchronous consumer
        self._last_slot = None

    def mark_in_flight(self, event):
        """Tell the reader that the batch yielded LAST is still being read asynchronously (e.g. by a non-blocking
        host-to-device copy); ``event`` is a ``torch.cuda.Event`` recorded after that work.  The staging slot is not
        refilled before the event has completed.  Consumers that finish with a batch before asking for the next one
        (``HostTokenizer.tokenize(..., sync=True)``) need not call this."""
        if self._last_slot is not None:
            self._busy[self._last_slot] = event

    def __len__(self):
        return sum(self.counts)

    def _map(self, i):
        c, h, w = self.shape
        return np.memmap(self.paths[i], dtype=_STORAGE[self.torch_dtype], mode="r", offset=HEADER_BYTES,
                         shape=(self.counts[i], c, h, w))

    def read_all(self):
        """All feature maps as one (N, C, H, W) tensor of the shards' dtype (pinned when CUDA is present)."""
        c, h, w = self.shape
        out = torch.empty(len(self), c, h, w, dtype=self.torch_dtype, pin_memory=self.pin)
        lo = 0
        for i, n in enumerate(self.counts):
            _numpy_view(out[lo:lo + n])[...] = self._map(i)
            lo += n
        return out

    def batches(self):
        """Yields (lo, hi, tensor) with tensor a (hi - lo, C, H, W) view (shards' dtype) of a staging buffer
        that stays valid until ``depth`` further batches have been produced."""
        c, h, w = self.shape
        if self._bufs is None:
            self._bufs = [torch.empty(self.batch, c, h, w, dtype=self.torch_dtype, pin_memory=self.pin)
                          for _ in range(self.depth)]
        k, lo = 0, 0
        for i, n in enumerate(self.counts):
            mm = self._map(i)
            for a in range(0, n, self.batch):
                b = min(n, a + self.batch)
                slot = k % self.depth
                ev = self._busy.pop(slot, None)
                if ev is not None:
                    ev.synchronize()              # an earlier DMA out of this pinned slot is still pending
                buf = self._bufs[slot]
                _numpy_view(buf[:b - a])[...] = mm[a:b]
                self._last_slot = slot
                yield lo + a, lo + b, buf[:b - a]
                k += 1
            lo += n
