"""Drop-in replacement for the reference's ``Codebook`` (models/Codebook.py:18-164).

Same constructor, attributes (``neighbourhood_range``, ``patch_dim``, ``image_dim``,
``embedding_dim``, ``num_embeddings``, ``codebook`` = nn.Embedding), methods, error behaviour
(plain ``Exception`` with the reference's messages) and ``state_dict`` ({"codebook.weight"}
only), so train_codebook.py, prune_codebook.py and the tokenisation calls of
train_quantized_transformer.py run unchanged.  The arithmetic runs in libsomcb:

  get_patches_bmu        -> som_bmu_nchw_f32                 (models/Codebook.py:77-99; also fp16 and bf16
                                                              feature maps, as if given x.float())
  get_quantized_patches  -> som_filter_f32 + som_quantize    (:102-135, S = onehot(bmu) @ T)
  forward                -> the same with fused unpatchify    (:156-164)
  backward (autograd)    -> som_accumulate_nchw_f32 + som_filter_f32
  get_quantized_image    -> som_quantize_nchw_f32             (:138-154)

After ``cb.half()`` or ``cb.to(torch.bfloat16)`` the inference methods keep working -- ``get_patches_bmu`` (results as
for the fp32 module on ``weight.float()``) and ``get_quantized_image`` (detached output in the weight's dtype, as
``nn.Embedding`` gives) -- and so do ``bmu_histogram``, ``prune_codebook`` and the tokenisers; ``forward`` and
``get_quantized_patches`` (the training / autograd path) need fp32 weights.

There is no CPU path: CPU inputs raise.
"""
import torch
import torch.nn as nn

from . import ops


class _FilterFn(torch.autograd.Function):
    """W~ = T @ W along the unit axis; T is symmetric, so backward is the same filter."""

    @staticmethod
    def forward(ctx, weight, neighbourhood_range):
        ctx.neighbourhood_range = float(neighbourhood_range)
        return ops.neighbourhood_filter(weight.detach().contiguous(), neighbourhood_range)

    @staticmethod
    def backward(ctx, grad_out):
        return ops.neighbourhood_filter(grad_out.contiguous(), ctx.neighbourhood_range), None


class _GatherFn(torch.autograd.Function):
    """out = table[idx] laid out per ``geom``; backward is the per-unit segmented sum."""

    @staticmethod
    def forward(ctx, table, idx, geom, out_shape):
        ctx.save_for_backward(idx)
        ctx.geom = geom
        ctx.num_units = table.shape[0]
        out = ops.quantize(idx, table.detach().contiguous(), geom)
        return out.view(out_shape)

    @staticmethod
    def backward(ctx, grad_out):
        (idx,) = ctx.saved_tensors
        g = grad_out.contiguous()
        rbar, _, _ = ops.accumulate(g, ctx.geom, idx, None, ctx.num_units)
        return rbar, None, None, None


class Codebook(nn.Module):
    def __init__(self, patch_dim=(2, 2), image_dim=(32, 32), image_channel=4,
                 num_embeddings=512, init_neighbour_range=256):
        super().__init__()
        # reference check (models/Codebook.py:27-28) kept verbatim in behaviour: the `and`
        # makes it unreachable, so no value is ever rejected here.
        if init_neighbour_range > num_embeddings and init_neighbour_range < 1:
            raise Exception("Invalid value for init_neighbour_range.")
        self.neighbourhood_range = init_neighbour_range
        self.patch_dim = patch_dim
        self.image_dim = image_dim
        patch_h, patch_w = self.patch_dim
        self.embedding_dim = image_channel * patch_h * patch_w
        self.num_embeddings = num_embeddings
        self.codebook = nn.Embedding(self.num_embeddings, self.embedding_dim)
        self.codebook.weight.data.uniform_(-1 / self.num_embeddings, 1 / self.num_embeddings)
        self._norm_cache = None       # unused (kept so that code which reset the former ||c||^2 cache keeps working)
        self.bmu_variant = ops.SOM_BMU_AUTO

    # ---- reference API --------------------------------------------------------------------
    def custom_load_state_dict(self, state_dict, ignore_msgs=False):
        own_state = self.state_dict()
        for name, param in state_dict.items():
            if name not in own_state:
                if not ignore_msgs:
                    print(f"No Layer found: {name}, skipping")
                continue
            if own_state[name].shape != param.data.shape:
                if not ignore_msgs:
                    print(f"Skipped: {name}")
                continue
            if isinstance(param, torch.nn.parameter.Parameter):
                param = param.data
            own_state[name].copy_(param)

    def decrease_neighbourhood(self, steps=1):
        if steps < 1:
            raise Exception("Invalid value for steps, should be > 1.")
        min_value = 1.0
        self.neighbourhood_range = min_value if self.neighbourhood_range <= 1 \
            else self.neighbourhood_range - 1

    def get_patches_bmu(self, x, reshape=False):
        x, geom = self._input(x, allow_half=True)
        idx = ops.bmu(x, geom, self._weight(), self._norms(), variant=self.bmu_variant)
        if reshape:
            # explicit Seq, not -1: an empty batch gives (0, Seq) as the reference does
            idx = idx.reshape(x.shape[0], (geom[2] // geom[4]) * (geom[3] // geom[5]))
        return idx

    def get_quantized_patches(self, x, use_gaussian=True):
        self._require_fp32_weights("get_quantized_patches")
        x, geom = self._input(x)
        idx = ops.bmu(x, geom, self._weight(), self._norms(), variant=self.bmu_variant)
        n_patches = idx.numel()
        flat = ops.flat_geometry(n_patches, self.embedding_dim)
        table = self._table(use_gaussian)
        return _GatherFn.apply(table, idx, flat, (x.shape[0], -1, self.embedding_dim))

    def get_quantized_image(self, indices, unpatchify_input=True):
        """Codebook rows of ``indices`` (N, Seq), unpatchified to (N, C, H, W) or as (N, Seq, D).  With fp16 / bf16
        weights the result is in that dtype and detached (no autograd through a 16-bit codebook)."""
        n, seq = indices.shape
        idx = self._indices(indices)
        w = self.codebook.weight
        gather = _GatherFn.apply
        if w.dtype in ops.HALF_DTYPES:
            w = w.detach()

            def gather(table, i, geom, shape):
                return ops.quantize(i, table, geom).view(shape)
        if unpatchify_input:
            c = self.embedding_dim // (self.patch_dim[0] * self.patch_dim[1])
            geom = ops.geometry((n, c, self.image_dim[0], self.image_dim[1]), self.patch_dim)
            if ops.n_patches_of(geom) != idx.numel():
                raise Exception("indices do not match image_dim / patch_dim.")
            return gather(w, idx, geom, (n, c, self.image_dim[0], self.image_dim[1]))
        flat = ops.flat_geometry(idx.numel(), self.embedding_dim)
        return gather(w, idx, flat, (n, seq, self.embedding_dim))

    def forward(self, x, use_gaussian=True):
        self._require_fp32_weights("forward")
        x, geom = self._input(x)
        idx = ops.bmu(x, geom, self._weight(), self._norms(), variant=self.bmu_variant)
        table = self._table(use_gaussian)
        return _GatherFn.apply(table, idx, geom, tuple(x.shape))

    # ---- helpers ---------------------------------------------------------------------------
    def _require_fp32_weights(self, what):
        dt = self.codebook.weight.dtype
        if dt != torch.float32:
            raise TypeError(f"Codebook.{what}: the training / autograd path needs float32 weights, the codebook holds "
                            f"{dt} (16-bit codebooks support get_patches_bmu and get_quantized_image)")

    def _weight(self):
        return self.codebook.weight.detach()

    def _table(self, use_gaussian):
        if use_gaussian:
            return _FilterFn.apply(self.codebook.weight, self.neighbourhood_range)
        return self.codebook.weight

    def _norms(self):
        # ||c||^2 is recomputed on every call (one 2-3 us kernel): a cache keyed on the parameter's version counter
        # goes stale silently whenever the weights are written through ``weight.data``, raw pointers, a collective
        # or this library's own Adam kernels, and stale norms mean wrong BMUs
        return ops.prepare_codebook(self.codebook.weight.detach())

    def _input(self, x, require_cuda=True, allow_half=False):
        """(contiguous x, geometry).  fp32 only, except where ``allow_half``: the search and the fast-path trainer
        also take fp16 and bf16 feature maps (results as on ``x.float()``); the autograd path does not."""
        if x.dim() != 4:
            raise Exception("Expected a (N, C, H, W) feature map.")
        w = self.codebook.weight
        if require_cuda and not (x.is_cuda and w.is_cuda):
            raise RuntimeError("somcb.Codebook runs on CUDA only (B200, sm_100a); move the module "
                               "and its input to the GPU -- there is no CPU fallback")
        if x.device != w.device:
            raise RuntimeError(f"input on {x.device} but codebook on {w.device}")
        if x.dtype != torch.float32 and not (allow_half and x.dtype in ops.HALF_DTYPES):
            raise TypeError(f"expected float32 feature maps, got {x.dtype}")
        x = x.detach().contiguous()
        geom = ops.geometry(x.shape, self.patch_dim)
        if ops.dim_of(geom) != self.embedding_dim:
            raise Exception("Input channels/patch size do not match the codebook embedding_dim.")
        return x, geom

    def _indices(self, indices):
        if not indices.is_cuda:
            raise RuntimeError("somcb.Codebook runs on CUDA only; indices must be a CUDA tensor")
        return indices.reshape(-1).to(torch.int64).contiguous()
