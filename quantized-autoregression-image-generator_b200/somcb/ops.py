"""Tensor-level wrappers over the C-ABI (include/somcb.h).

PyTorch is plumbing here: it owns device memory (outputs and workspaces are torch tensors from
the caching allocator, so they are stream-ordered and never freed under a running kernel) and
the current CUDA stream.  All arithmetic happens inside libsomcb.  Every function raises on
CPU tensors -- there is no fallback path.
"""
import torch

from . import _lib
from ._lib import SOM_BMU_AUTO, SOM_BMU_FFMA, SOM_BMU_TC3X, SOM_BMU_TC_TF32, SOM_BMU_TC_F16, check  # noqa: F401


REQUIRES_CUDA = True


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _req(t, dtype, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name}: somcb kernels need a CUDA tensor (got {t.device}); "
                           "there is no CPU fallback")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    return t


def _workspace(nbytes, device):
    if nbytes == 0:
        return None, 0
    ws = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
    return ws, int(nbytes)


def geometry(x_shape, patch_dim):
    """(n_img, C, H, W, pH, pW) for an NCHW batch; validates divisibility like the C side."""
    n, c, h, w = (int(v) for v in x_shape)
    p_h, p_w = (int(v) for v in patch_dim)
    if h % p_h or w % p_w:
        raise ValueError(f"image {h}x{w} is not divisible by patch {p_h}x{p_w}")
    return n, c, h, w, p_h, p_w


def flat_geometry(n_rows, dim):
    """A pre-flattened (n, D) row matrix seen as n one-patch images (include/somcb.h)."""
    return int(n_rows), 1, 1, int(dim), 1, int(dim)


def n_patches_of(geom):
    n, c, h, w, p_h, p_w = geom
    return n * (h // p_h) * (w // p_w)


def dim_of(geom):
    n, c, h, w, p_h, p_w = geom
    return c * p_h * p_w


def device_info():
    import ctypes
    sm, major, minor = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    lib = _lib.load()
    check("som_device_info", lib.som_device_info(ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor)))
    return sm.value, major.value, minor.value


# 16-bit codebook dtypes and their C dtype codes (include/somcb.h: w_dtype; also the feature-map shards' codes)
_W16_CODES = {torch.float16: 1, torch.bfloat16: 2}


def _req_weight(weight):
    """A codebook: fp32, or fp16 / bf16 (inference only: the search, decoding and row compaction)."""
    if isinstance(weight, torch.Tensor) and weight.dtype in _W16_CODES:
        return _req(weight, weight.dtype, "weight")
    return _req(weight, torch.float32, "weight")


def prepare_codebook(weight, out=None):
    """c_norm2[j] = ||W_j||^2  (K0).  A 16-bit ``weight`` gives the norms of ``weight.float()`` bit for bit."""
    lib = _lib.load()
    w = _req_weight(weight)
    k, d = w.shape
    if out is None:
        out = torch.empty(k, dtype=torch.float32, device=w.device)
    with torch.cuda.device(w.device):
        if w.dtype in _W16_CODES:
            check("som_prepare_codebook_w16",
                  lib.som_prepare_codebook_w16(_ptr(w), _W16_CODES[w.dtype], k, d, _ptr(out), _stream(w)))
        else:
            check("som_prepare_codebook_f32",
                  lib.som_prepare_codebook_f32(_ptr(w), k, d, _ptr(out), _stream(w)))
    return out


def bmu_can_stage(geom, num_units, variant=SOM_BMU_AUTO):
    """Whether the BMU kernel for this shape can also emit the patch-major staging copy (``bmu(stage=...)``)."""
    return bool(_lib.load().som_bmu_can_stage(n_patches_of(geom), dim_of(geom), int(num_units), int(variant)))


def bmu_f16_native(geom, num_units, variant=SOM_BMU_AUTO):
    """Whether the BMU kernel for this shape reads a 16-bit batch (fp16 or bf16: the same kernel) itself (otherwise
    ``bmu`` upcasts it first)."""
    return bool(_lib.load().som_bmu_f16_native(n_patches_of(geom), dim_of(geom), int(num_units), int(variant)))


# 16-bit feature-map dtypes: the C entry points of the exact fp32 copy and of the native search
_HALF_ENTRIES = {torch.float16: ("som_convert_f16_f32", "som_bmu_stage_nchw_f16"),
                 torch.bfloat16: ("som_convert_bf16_f32", "som_bmu_stage_nchw_bf16")}
HALF_DTYPES = tuple(_HALF_ENTRIES)          # the feature-map dtypes the search takes besides fp32


def _upcast(x, out, dtype):
    lib = _lib.load()
    x = _req(x, dtype, "x")
    if out is None:
        out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    out = _req(out, torch.float32, "out")
    if out.numel() != x.numel():
        raise ValueError("out must hold as many elements as x")
    entry = _HALF_ENTRIES[dtype][0]
    with torch.cuda.device(x.device):
        check(entry, getattr(lib, entry)(_ptr(x), x.numel(), _ptr(out), _stream(x)))
    return out


def upcast_f16(x, out=None):
    """Exact fp32 copy of a contiguous fp16 CUDA tensor (som_convert_f16_f32); ``out``: optional fp32 destination of
    the same number of elements."""
    return _upcast(x, out, torch.float16)


def upcast_bf16(x, out=None):
    """Exact fp32 copy of a contiguous bf16 CUDA tensor (som_convert_bf16_f32); ``out``: optional fp32 destination of
    the same number of elements."""
    return _upcast(x, out, torch.bfloat16)


def bmu(x, geom, weight, c_norm2=None, unit_offset=0, want_rd=False, variant=SOM_BMU_AUTO,
        out=None, stage=None):
    """K1.  x: fp32, fp16 or bf16 contiguous buffer described by ``geom``.  Returns idx (n_patches,) int64
    [and the reduced distance rd (n_patches,) fp32 when ``want_rd``].  ``stage``: optional (n_patches, D) fp32
    tensor that receives the patch-major copy of the patch rows (only where ``bmu_can_stage``).

    A 16-bit ``x`` gives exactly the results of the same call on ``x.float()``: the FP16-split kernel reads it
    directly where ``bmu_f16_native`` says so, other shapes search an fp32 copy made by ``upcast_f16`` /
    ``upcast_bf16``.  Likewise a 16-bit (fp16 / bf16) ``weight`` gives exactly the results of ``weight.float()``
    (som_bmu_w16_nchw); it takes no ``stage``, which only the training step reads."""
    lib = _lib.load()
    w = _req_weight(weight)
    k, d = w.shape
    if w.dtype in _W16_CODES and stage is not None:
        raise ValueError("bmu: stage is not available with a 16-bit codebook (training needs fp32 weights)")
    if isinstance(x, torch.Tensor) and x.dtype in _HALF_ENTRIES:
        x = _req(x, x.dtype, "x")
        if not bmu_f16_native(geom, k, variant):
            return bmu(_upcast(x, None, x.dtype), geom, w, c_norm2, unit_offset, want_rd, variant, out, stage)
        entry = _HALF_ENTRIES[x.dtype][1]
    else:
        x = _req(x, torch.float32, "x")
        entry = "som_bmu_stage_nchw_f32"
    if d != dim_of(geom):
        raise ValueError(f"codebook dim {d} != patch dim {dim_of(geom)}")
    npat = n_patches_of(geom)
    if x.numel() != geom[0] * geom[1] * geom[2] * geom[3]:
        raise ValueError("x does not match the geometry")
    if c_norm2 is None:
        c_norm2 = prepare_codebook(w)
    c_norm2 = _req(c_norm2, torch.float32, "c_norm2")
    if out is None:
        out = torch.empty(npat, dtype=torch.int64, device=x.device)
    rd = torch.empty(npat, dtype=torch.float32, device=x.device) if want_rd else None
    if stage is not None:
        stage = _req(stage, torch.float32, "stage")
        if stage.numel() != npat * d:
            raise ValueError("stage must hold n_patches x D floats")
    with torch.cuda.device(x.device):
        if w.dtype in _W16_CODES:
            x_code = _W16_CODES.get(x.dtype, 0)
            ws, ws_bytes = _workspace(lib.som_bmu_w16_workspace_bytes(npat, d, k, variant), x.device)
            check("som_bmu_w16_nchw",
                  lib.som_bmu_w16_nchw(_ptr(x), x_code, *geom, _ptr(w), _W16_CODES[w.dtype], _ptr(c_norm2), k,
                                       int(unit_offset), _ptr(out), _ptr(rd), _ptr(ws), ws_bytes, variant, _stream(x)))
            return (out, rd) if want_rd else out
        ws, ws_bytes = _workspace(lib.som_bmu_workspace_bytes(npat, d, k, variant), x.device)
        check(entry, getattr(lib, entry)(_ptr(x), *geom, _ptr(w), _ptr(c_norm2), k, int(unit_offset),
                                         _ptr(out), _ptr(rd), _ptr(stage), _ptr(ws), ws_bytes, variant, _stream(x)))
    return (out, rd) if want_rd else out


def merge_candidates(rd, idx):
    """K1b.  rd, idx: (R, n).  Returns (idx (n,), rd (n,))."""
    lib = _lib.load()
    rd = _req(rd, torch.float32, "rd")
    idx = _req(idx, torch.int64, "idx")
    r, n = rd.shape
    out_idx = torch.empty(n, dtype=torch.int64, device=rd.device)
    out_rd = torch.empty(n, dtype=torch.float32, device=rd.device)
    with torch.cuda.device(rd.device):
        check("som_merge_candidates",
              lib.som_merge_candidates(_ptr(rd), _ptr(idx), r, n, _ptr(out_idx), _ptr(out_rd), _stream(rd)))
    return out_idx, out_rd


def histogram(idx, num_units, counts=None):
    """K5.  counts[j] += #{idx == j}; creates a zeroed int64 counts when not given."""
    lib = _lib.load()
    idx = _req(idx, torch.int64, "idx")
    if counts is None:
        counts = torch.zeros(num_units, dtype=torch.int64, device=idx.device)
    counts = _req(counts, torch.int64, "counts")
    with torch.cuda.device(idx.device):
        check("som_histogram_i64",
              lib.som_histogram_i64(_ptr(idx), idx.numel(), int(num_units), _ptr(counts), _stream(idx)))
    return counts


def neighbourhood_filter(inp, neighbourhood_range, scale=1.0, out=None, tensor_cores=True):
    """K3.  out = scale * T @ inp along the unit axis.  ``tensor_cores=False`` forces the FFMA kernel
    (the library picks by shape otherwise: tcgen05 for K >= 256 and D >= 48)."""
    lib = _lib.load()
    inp = _req(inp, torch.float32, "inp")
    k, d = inp.shape
    if out is None:
        out = torch.empty_like(inp)
    out = _req(out, torch.float32, "out")
    with torch.cuda.device(inp.device):
        if not tensor_cores:
            check("som_filter_f32",
                  lib.som_filter_f32(_ptr(inp), _ptr(out), k, d, float(neighbourhood_range), float(scale),
                                     _stream(inp)))
            return out
        ws, ws_bytes = _workspace(lib.som_filter_workspace_bytes(k, d, float(neighbourhood_range)), inp.device)
        check("som_filter_ws_f32",
              lib.som_filter_ws_f32(_ptr(inp), _ptr(out), k, d, float(neighbourhood_range), float(scale),
                                    _ptr(ws), ws_bytes, _stream(inp)))
    return out


def accumulate(x, geom, bmu_idx, table, num_units, want_counts=False, want_sse=False, out=None):
    """K2.  Returns (Rbar (K, D), counts or None, sse (1,) float64 or None)."""
    lib = _lib.load()
    x = _req(x, torch.float32, "x")
    bmu_idx = _req(bmu_idx, torch.int64, "bmu")
    d = dim_of(geom)
    npat = n_patches_of(geom)
    if bmu_idx.numel() != npat:
        raise ValueError("bmu does not match the geometry")
    if table is not None:
        table = _req(table, torch.float32, "table")
    if out is None:
        out = torch.empty(num_units, d, dtype=torch.float32, device=x.device)
    counts = torch.empty(num_units, dtype=torch.int64, device=x.device) if want_counts else None
    sse = torch.empty(1, dtype=torch.float64, device=x.device) if want_sse else None
    with torch.cuda.device(x.device):
        ws, ws_bytes = _workspace(lib.som_accumulate_workspace_bytes(npat, d, int(num_units)), x.device)
        check("som_accumulate_nchw_f32",
              lib.som_accumulate_nchw_f32(_ptr(x), *geom, _ptr(bmu_idx), _ptr(table), int(num_units),
                                          _ptr(out), _ptr(counts), _ptr(sse), _ptr(ws), ws_bytes,
                                          _stream(x)))
    return out, counts, sse


def accumulate_packed(x, geom, bmu_idx, table, num_units, packed=None, ws=None):
    """K2, data-parallel form.  ``packed``: (K*D + 4,) fp32 = [Rbar | sse_hi, sse_lo, n/4096, n%4096] (see
    include/somcb.h); allocated when not given.  ``ws``: optional caller-kept workspace (uint8)."""
    lib = _lib.load()
    x = _req(x, torch.float32, "x")
    bmu_idx = _req(bmu_idx, torch.int64, "bmu")
    table = _req(table, torch.float32, "table")
    d = dim_of(geom)
    npat = n_patches_of(geom)
    if bmu_idx.numel() != npat:
        raise ValueError("bmu does not match the geometry")
    if packed is None:
        packed = torch.empty(num_units * d + 4, dtype=torch.float32, device=x.device)
    packed = _req(packed, torch.float32, "packed")
    if packed.numel() != num_units * d + 4:
        raise ValueError("packed must hold K*D + 4 floats")
    with torch.cuda.device(x.device):
        need = lib.som_accumulate_workspace_bytes(npat, d, int(num_units))
        if ws is None or ws.numel() < need:
            ws, _ = _workspace(need, x.device)
        check("som_accumulate_packed_nchw_f32",
              lib.som_accumulate_packed_nchw_f32(_ptr(x), *geom, _ptr(bmu_idx), _ptr(table), int(num_units),
                                                 _ptr(packed), _ptr(ws), ws.numel(), _stream(x)))
    return packed


def adam_step_dp(weight, m, v, grad, dim, lr, steps_done, tail, loss_out=None, betas=(0.5, 0.999), eps=1e-8):
    """K4, data-parallel tail: ``grad`` unscaled (T @ Rbar_global), ``tail`` the all-reduced 4-float tail of
    ``accumulate_packed``; scales by 2 / numel on the device, writes the loss, increments ``steps_done[0]``
    (``steps_done``: two int64, [completed steps, scratch word kept at zero])."""
    lib = _lib.load()
    for t, nm in ((weight, "weight"), (m, "m"), (v, "v"), (grad, "grad"), (tail, "tail")):
        _req(t, torch.float32, nm)
    _req(steps_done, torch.int64, "steps_done")
    if steps_done.numel() < 2:
        raise ValueError("steps_done must hold two int64: [completed steps, scratch]")
    if loss_out is None:
        loss_out = torch.empty(1, dtype=torch.float64, device=weight.device)
    _req(loss_out, torch.float64, "loss_out")
    with torch.cuda.device(weight.device):
        check("som_adam_dp_f32",
              lib.som_adam_dp_f32(_ptr(weight), _ptr(m), _ptr(v), _ptr(grad), weight.numel(), int(dim), float(lr),
                                  float(betas[0]), float(betas[1]), float(eps), _ptr(steps_done), _ptr(tail),
                                  _ptr(loss_out), _stream(weight)))
    return loss_out


def quantize(idx, table, geom, out=None):
    """Gather + fused unpatchify: returns the buffer described by ``geom`` in the table's dtype (fp32, or fp16 / bf16:
    the 16-bit values are copied exactly)."""
    lib = _lib.load()
    idx = _req(idx, torch.int64, "idx")
    table = _req_weight(table)
    k, d = table.shape
    if d != dim_of(geom) or idx.numel() != n_patches_of(geom):
        raise ValueError("idx/table do not match the geometry")
    n, c, h, w, _, _ = geom
    if out is None:
        out = torch.empty(n, c, h, w, dtype=table.dtype, device=table.device)
    entry = "som_quantize_nchw_b16" if table.dtype in _W16_CODES else "som_quantize_nchw_f32"
    with torch.cuda.device(table.device):
        check(entry, getattr(lib, entry)(_ptr(idx), _ptr(table), k, *geom, _ptr(out), _stream(table)))
    return out


def adam_step(weight, m, v, grad, lr, step, betas=(0.5, 0.999), eps=1e-8):
    """K4, in place on weight/m/v.  ``step`` is the 1-based count after increment."""
    lib = _lib.load()
    for t, nm in ((weight, "weight"), (m, "m"), (v, "v"), (grad, "grad")):
        _req(t, torch.float32, nm)
    with torch.cuda.device(weight.device):
        check("som_adam_f32",
              lib.som_adam_f32(_ptr(weight), _ptr(m), _ptr(v), _ptr(grad), weight.numel(), float(lr),
                               float(betas[0]), float(betas[1]), float(eps), int(step), _stream(weight)))
    return weight


def adam_step_dev(weight, m, v, grad, lr, steps_done, betas=(0.5, 0.999), eps=1e-8):
    """K4 with the step count in device memory (``steps_done``: int64 tensor of one element, the
    number of completed steps); increments it on the stream.  Used under CUDA-graph capture."""
    lib = _lib.load()
    for t, nm in ((weight, "weight"), (m, "m"), (v, "v"), (grad, "grad")):
        _req(t, torch.float32, nm)
    _req(steps_done, torch.int64, "steps_done")
    with torch.cuda.device(weight.device):
        check("som_adam_devstep_f32",
              lib.som_adam_devstep_f32(_ptr(weight), _ptr(m), _ptr(v), _ptr(grad), weight.numel(), float(lr),
                                       float(betas[0]), float(betas[1]), float(eps), _ptr(steps_done),
                                       _stream(weight)))
    return weight


def step_small_supported(geom, num_units, neighbourhood_range):
    """Whether the one-kernel training step covers this shape (include/somcb.h, som_step_small_f32)."""
    return _lib.load().som_step_small_workspace_bytes(n_patches_of(geom), dim_of(geom), int(num_units),
                                                      float(neighbourhood_range)) > 0


def step_small(x, geom, weight, m, v, neighbourhood_range, lr, steps_done, betas=(0.5, 0.999), eps=1e-8,
               want_bmu=True, loss_out=None):
    """The whole training step in one cooperative kernel (small problems).  Returns (loss (1,) float64, bmu or None)."""
    lib = _lib.load()
    x = _req(x, torch.float32, "x")
    for t, nm in ((weight, "weight"), (m, "m"), (v, "v")):
        _req(t, torch.float32, nm)
    _req(steps_done, torch.int64, "steps_done")
    k, d = weight.shape
    npat = n_patches_of(geom)
    if loss_out is None:
        loss_out = torch.empty(1, dtype=torch.float64, device=x.device)
    bmu_out = torch.empty(npat, dtype=torch.int64, device=x.device) if want_bmu else None
    with torch.cuda.device(x.device):
        ws, ws_bytes = _workspace(lib.som_step_small_workspace_bytes(npat, d, k, float(neighbourhood_range)), x.device)
        check("som_step_small_f32",
              lib.som_step_small_f32(_ptr(x), *geom, _ptr(weight), _ptr(m), _ptr(v), k, float(neighbourhood_range),
                                     float(lr), float(betas[0]), float(betas[1]), float(eps), _ptr(steps_done),
                                     _ptr(bmu_out), _ptr(loss_out), _ptr(ws), ws_bytes, _stream(x)))
    return loss_out, bmu_out


def gather_rows(weight, keep):
    """out[r] = weight[keep[r]] in the weight's dtype (fp32, fp16 or bf16)."""
    lib = _lib.load()
    w = _req_weight(weight)
    keep = _req(keep, torch.int64, "keep")
    out = torch.empty(keep.numel(), w.shape[1], dtype=w.dtype, device=w.device)
    entry = "som_gather_rows_b16" if w.dtype in _W16_CODES else "som_gather_rows_f32"
    with torch.cuda.device(w.device):
        check(entry, getattr(lib, entry)(_ptr(w), w.shape[1], _ptr(keep), keep.numel(), _ptr(out), _stream(w)))
    return out


def assemble_tokens(lr_idx, hr_idx, lr_num_embeddings, hr_num_embeddings, base_model):
    """Token tensors of train_quantized_transformer.py:411-455 from the two (n, Seq) BMU index
    tensors in one launch.  Returns (hr_input, hr_target)."""
    lib = _lib.load()
    hr_idx = _req(hr_idx, torch.int64, "hr_idx")
    n, hr_seq = hr_idx.shape
    lr_seq = 0
    if lr_idx is not None:
        lr_idx = _req(lr_idx, torch.int64, "lr_idx")
        if lr_idx.shape[0] != n:
            raise ValueError("lr_idx and hr_idx disagree on the batch size")
        lr_seq = lr_idx.shape[1]
    in_w = lr_seq + hr_seq if base_model else 1 + hr_seq
    hr_input = torch.empty(n, in_w, dtype=torch.int64, device=hr_idx.device)
    hr_target = torch.empty(n, hr_seq + 1, dtype=torch.int64, device=hr_idx.device)
    with torch.cuda.device(hr_idx.device):
        check("som_assemble_tokens_i64",
              lib.som_assemble_tokens_i64(_ptr(lr_idx), _ptr(hr_idx), n, lr_seq, hr_seq,
                                          int(lr_num_embeddings), int(hr_num_embeddings),
                                          1 if base_model else 0, _ptr(hr_input), _ptr(hr_target),
                                          _stream(hr_idx)))
    return hr_input, hr_target


# ---- data-parallel tail over NVLink / NVSwitch peer memory (include/somcb.h, som_peer_*) -----------------------
def filter_half_width(num_units, neighbourhood_range):
    return int(_lib.load().som_filter_half_width(int(num_units), float(neighbourhood_range)))


def peer_signal_bytes():
    return int(_lib.load().som_peer_signal_bytes())


def _pads(signal_ptrs):
    import ctypes
    return (ctypes.c_void_p * len(signal_ptrs))(*[int(p) for p in signal_ptrs])


def peer_allreduce(mc_ptr, n, rank, world, signal_ptrs, channel, device, peer_ptrs=None, tail_out=None):
    """In-place all-reduce(sum) of ``n`` floats at the multicast address ``mc_ptr`` (every rank calls it).  With
    ``peer_ptrs`` / ``tail_out`` (the buffer's peer addresses and a separate local 4-float tensor) the buffer is a packed
    accumulator buffer whose 4-float tail is summed exactly into ``tail_out``."""
    lib = _lib.load()
    with torch.cuda.device(device):
        check("som_peer_allreduce_f32",
              lib.som_peer_allreduce_f32(int(mc_ptr), int(n), _pads(peer_ptrs) if peer_ptrs is not None else None,
                                         _ptr(tail_out), int(rank), int(world), _pads(signal_ptrs), int(channel),
                                         torch.cuda.current_stream(device).cuda_stream))


def peer_reduce_rows(mc_packed, peer_ptrs, num_units, dim, row0, row1, max_rows, out_rows, out_tail, rank, world,
                     signal_ptrs, channel):
    lib = _lib.load()
    out_rows = _req(out_rows, torch.float32, "out_rows")
    out_tail = _req(out_tail, torch.float32, "out_tail")
    with torch.cuda.device(out_rows.device):
        check("som_peer_reduce_rows_f32",
              lib.som_peer_reduce_rows_f32(int(mc_packed), _pads(peer_ptrs), int(num_units), int(dim), int(row0),
                                           int(row1), int(max_rows),
                                           _ptr(out_rows), _ptr(out_tail), int(rank), int(world), _pads(signal_ptrs),
                                           int(channel), _stream(out_rows)))


def peer_reduce_filter_rows(mc_packed, peer_ptrs, num_units, dim, row0, row1, max_rows, neighbourhood_range, rows_scratch,
                            out_rows, out_tail, rank, world, signal_ptrs, channel, scale=1.0):
    """Reduce-scatter fused into the filter: out_rows = scale * T @ (sum over ranks of accumulator rows [row0, row1))."""
    lib = _lib.load()
    rows = int(row1) - int(row0)
    rows_scratch = _req(rows_scratch, torch.float32, "rows_scratch")
    out_rows = _req(out_rows, torch.float32, "out_rows")
    out_tail = _req(out_tail, torch.float32, "out_tail")
    if rows_scratch.numel() < int(max_rows) * int(dim) or out_rows.numel() < rows * int(dim):
        raise ValueError("rows_scratch must hold max_rows x D floats and out_rows (row1 - row0) x D")
    with torch.cuda.device(out_rows.device):
        ws, ws_bytes = _workspace(lib.som_filter_workspace_bytes(rows, int(dim), float(neighbourhood_range)),
                                  out_rows.device)
        check("som_peer_reduce_filter_rows_f32",
              lib.som_peer_reduce_filter_rows_f32(int(mc_packed), _pads(peer_ptrs), int(num_units), int(dim), int(row0),
                                                  int(row1), int(max_rows), float(neighbourhood_range), float(scale),
                                                  _ptr(rows_scratch), _ptr(out_rows), _ptr(out_tail), int(rank),
                                                  int(world), _pads(signal_ptrs), int(channel), _ptr(ws), ws_bytes,
                                                  _stream(out_rows)))
    return out_rows


def peer_bcast_rows(src_rows, mc_dst, max_n, rank, world, signal_ptrs, channel):
    lib = _lib.load()
    src_rows = _req(src_rows, torch.float32, "src_rows")
    with torch.cuda.device(src_rows.device):
        check("som_peer_bcast_rows_f32",
              lib.som_peer_bcast_rows_f32(_ptr(src_rows), int(mc_dst), src_rows.numel(), int(max_n), int(rank),
                                          int(world), _pads(signal_ptrs), int(channel), _stream(src_rows)))


def peer_adam_slice(w_rows, mc_w_rows, m_rows, v_rows, g_rows, max_n, dim, lr, steps_done, tail, rank, world,
                    signal_ptrs, channel, loss_out=None, betas=(0.5, 0.999), eps=1e-8):
    lib = _lib.load()
    for t, nm in ((w_rows, "w_rows"), (m_rows, "m_rows"), (v_rows, "v_rows"), (g_rows, "g_rows"), (tail, "tail")):
        _req(t, torch.float32, nm)
    _req(steps_done, torch.int64, "steps_done")
    if steps_done.numel() < 2:
        raise ValueError("steps_done must hold two int64: [completed steps, scratch]")
    if loss_out is None:
        loss_out = torch.empty(1, dtype=torch.float64, device=w_rows.device)
    with torch.cuda.device(w_rows.device):
        check("som_peer_adam_slice_f32",
              lib.som_peer_adam_slice_f32(_ptr(w_rows), int(mc_w_rows), _ptr(m_rows), _ptr(v_rows), _ptr(g_rows),
                                          w_rows.numel(), int(max_n), int(dim), float(lr), float(betas[0]),
                                          float(betas[1]), float(eps), _ptr(steps_done), _ptr(tail), _ptr(loss_out),
                                          int(rank), int(world), _pads(signal_ptrs), int(channel), _stream(w_rows)))
    return loss_out
