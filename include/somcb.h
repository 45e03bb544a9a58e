/*
 * somcb.h -- C-ABI of libsomcb.so: the B200 (sm_100a) SOM-codebook hot path.
 *
 * The reference (Vinmwaura/Quantized-Autoregression-Image-Generator) is pure Python and has no
 * FFI of its own; its boundary for this path is the class models/Codebook.py::Codebook.  Every
 * entry point below names the reference lines it replaces.  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated;
 *   - `stream` is a cudaStream_t passed as void*; every call only ENQUEUES work on it (no host
 *     synchronisation inside), so host scalars are passed by value, results stay on the device;
 *   - the library never allocates, frees or retains device memory: inputs, outputs and
 *     workspaces are caller-owned (size a workspace with the matching *_workspace_bytes call);
 *   - return 0 on success, a negative SOM_E_* code for argument/shape/workspace errors, a
 *     positive cudaError_t for a failed launch; som_last_error() gives the thread-local text;
 *   - patch geometry (n_img, C, H, Wd, pH, pW) describes an fp32 contiguous NCHW batch that is
 *     cut into (H/pH)*(Wd/pW) patches per image, patch s = ph*(Wd/pW)+pw, feature
 *     d = c*pH*pW + i*pW + j  <->  x[n, c, ph*pH+i, pw*pW+j]   (models/layers.py:8-34).
 *     A pre-flattened (n, D) row matrix is the geometry (n, 1, 1, D, 1, D);
 *   - a zero count (n_img == 0 / n == 0) is a successful no-op and is the only case in which the
 *     per-item input/output pointers may be NULL (torch gives zero-element tensors a null
 *     data pointer); the reference returns empty tensors there (models/Codebook.py:77-99);
 *   - non-finite input: a patch that holds a NaN gets unit 0 of the searched range, as
 *     torch.argmin over the reference's all-NaN distance row does; a patch that holds +-inf gets
 *     some in-range index (the reference's pick there is an accident of its sgemm's inf - inf);
 *     other patches are unaffected.
 */
#ifndef SOMCB_H_
#define SOMCB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOM_ABI_VERSION 2

#if defined(__GNUC__)
#define SOM_API __attribute__((visibility("default")))
#else
#define SOM_API
#endif

/* error codes */
#define SOM_OK               0
#define SOM_E_BADARG        -1   /* null pointer, non-positive size, misaligned buffer          */
#define SOM_E_SHAPE         -2   /* H % pH != 0, K too large for the variant, ...               */
#define SOM_E_WORKSPACE     -3   /* workspace smaller than *_workspace_bytes says               */
#define SOM_E_UNSUPPORTED   -4   /* variant not available for this shape / device               */

/* BMU kernel variants (static rule in som_bmu_pick_variant; no runtime autotuner) */
#define SOM_BMU_AUTO         0
#define SOM_BMU_FFMA         1   /* fp32 FFMA register-tiled kernel, any shape                  */
#define SOM_BMU_TC3X         2   /* tcgen05, error-compensated hi/lo split (3 products), TMEM argmin.  The split
                                  * arithmetic follows a static rule on the shape (som_bmu_split_mode): kind::tf32
                                  * 3xTF32, or -- large batches: D <= 16 from 65 536 patches, 16 < D <= 256 from one
                                  * full wave of 128-patch tiles -- a kind::f16 FP16 hi/lo split with exact
                                  * power-of-two scaling (same 11+11-bit operand precision, fp32 accumulation)       */
#define SOM_BMU_TC_TF32      3   /* SOM_BMU_TC3X with the 3xTF32 arithmetic at every size                            */
#define SOM_BMU_TC_F16       4   /* SOM_BMU_TC3X with the FP16 split at every size (SOM_E_UNSUPPORTED when no FP16
                                  * kernel covers the shape: D > 256 or fewer than 513 units); near-tie picks may
                                  * differ between the arithmetics within the 1e-6 relative distance rule            */

SOM_API int         som_version(void);
SOM_API const char* som_last_error(void);
/* Number of kernel launches this library has enqueued in this process (telemetry for bench.py;
 * a cub radix sort counts as one). */
SOM_API uint64_t    som_launch_count(void);
/* SM count and compute capability of the current device (host pointers). */
SOM_API int         som_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- K0: per-weights-version precompute -------------------------------------------------
 * c_norm2[j] = ||W[j]||^2 (fp32).  Replaces the [W, 1, ||W||^2] operand torch.cdist builds
 * on every call (models/Codebook.py:86-88). */
SOM_API int som_prepare_codebook_f32(const float* W, int K, int D, float* c_norm2, void* stream);

/* ---- K1: Best-Matching-Unit search ------------------------------------------------------
 * Replaces Codebook.get_patches_bmu (models/Codebook.py:77-99): patchify + torch.cdist +
 * argmin, first index on ties.  The (N*Seq) x K distance matrix is never materialised.
 *   out_idx[p]  = unit_offset + argmin_j ( ||W_j||^2 - 2 x_p . W_j )        (int64)
 *   out_rd[p]   = that minimum "reduced distance" (= d^2 - ||x_p||^2), or NULL
 * unit_offset / out_rd serve the unit-sharded mode (som_merge_candidates).              */
SOM_API size_t som_bmu_workspace_bytes(int64_t n_patches, int D, int K, int variant);
SOM_API int    som_bmu_pick_variant(int64_t n_patches, int D, int K);
/* Split arithmetic the static rule picks for this shape: 1 = FP16 hi/lo (kind::f16), 0 = 3xTF32, -1 = not a
 * tensor-core shape (FFMA variant).  Host-only, no device work.                                              */
SOM_API int    som_bmu_split_mode(int64_t n_patches, int D, int K);
SOM_API int som_bmu_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                     const float* W, const float* c_norm2, int K, int64_t unit_offset,
                     int64_t* out_idx, float* out_rd,
                     void* ws, size_t ws_bytes, int variant, void* stream);

/* The same search that ALSO writes stage_rows, a patch-major (n_patches, D) fp32 copy of the patch rows -- the
 * (N, Seq, D) tensor patchify materialises in models/layers.py:8-34, here a by-product of the kernel that holds
 * every row in registers anyway.  The training step's segmented gather (som_accumulate_*_nchw_f32 on the geometry
 * (n_patches, 1, 1, D, 1, D)) then reads ONE contiguous row per patch instead of pH*C pieces of pW floats, which
 * in NCHW cost a whole DRAM burst each.  Only the FP16-split kernel of 16 < D <= 256 emits it: ask
 * som_bmu_can_stage (host-only) first; SOM_E_UNSUPPORTED otherwise.  stage_rows == NULL: som_bmu_nchw_f32.     */
SOM_API int som_bmu_can_stage(int64_t n_patches, int D, int K, int variant);
SOM_API int som_bmu_stage_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                           const float* W, const float* c_norm2, int K, int64_t unit_offset,
                           int64_t* out_idx, float* out_rd, float* stage_rows,
                           void* ws, size_t ws_bytes, int variant, void* stream);

/* ---- K1 on 16-bit feature maps (binary16 and bfloat16) ---------------------------------------------------
 * A 16-bit batch means the data ARE those values: every result equals the fp32 call on x.float().
 * som_bmu_stage_nchw_f16 / _bf16 are som_bmu_stage_nchw_f32 on a contiguous NCHW batch of IEEE half / bfloat16 bit
 * patterns (2-byte aligned); stage_rows (fp32, may be NULL) is patchify(x.float()).  Only the FP16-split kernel of
 * 16 < D <= 256 reads 16-bit values itself -- ask som_bmu_f16_native (host-only) first: it answers for BOTH formats,
 * the kernel being the same; SOM_E_UNSUPPORTED where it says 0.  There a tile whose patch rows are exact in FP16
 * after the row scale skips the A_lo x B_hi product group (9 instead of 13 MMAs per tile at D = 64).  fp16 rows
 * always are unless the row scale was clamped; a bf16 element is when it lies within about 2^-23 of its row's
 * largest magnitude (tanh-range latents: almost every tile), so a bf16 tile may keep the third product where an fp16
 * tile would not -- the result is exact either way.  Other shapes: convert with som_convert_f16_f32 /
 * som_convert_bf16_f32 and call the fp32 entry points.  Same workspace as som_bmu_workspace_bytes.              */
SOM_API int som_bmu_f16_native(int64_t n_patches, int D, int K, int variant);
SOM_API int som_bmu_stage_nchw_f16(const void* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                   const float* W, const float* c_norm2, int K, int64_t unit_offset,
                                   int64_t* out_idx, float* out_rd, float* stage_rows,
                                   void* ws, size_t ws_bytes, int variant, void* stream);
SOM_API int som_bmu_stage_nchw_bf16(const void* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                    const float* W, const float* c_norm2, int K, int64_t unit_offset,
                                    int64_t* out_idx, float* out_rd, float* stage_rows,
                                    void* ws, size_t ws_bytes, int variant, void* stream);
/* out[i] = (float)in[i] for n binary16 / bfloat16 values (exact); in 2-byte, out 4-byte aligned.             */
SOM_API int som_convert_f16_f32(const void* in, int64_t n, float* out, void* stream);
SOM_API int som_convert_bf16_f32(const void* in, int64_t n, float* out, void* stream);

/* Same search on pre-flattened patch rows: `patches` is (n, D) row-major fp32 (what patchify +
 * reshape produce in models/Codebook.py:83-84).  Equivalent to som_bmu_nchw_f32 with the rows seen
 * as n one-patch images (n_img = n, C = 1, H = 1, W = D, pH = 1, pW = D).                       */
SOM_API int som_bmu_flat_f32(const float* patches, int64_t n, int D,
                     const float* W, const float* c_norm2, int K, int64_t unit_offset,
                     int64_t* out_idx, float* out_rd,
                     void* ws, size_t ws_bytes, int variant, void* stream);

/* ---- K0 / K1 with 16-bit codebooks (binary16 and bfloat16 weights; inference only) ---------------------------
 * A 16-bit codebook means the weights ARE those values: every result equals the fp32 call on W.float() -- indices,
 * reduced distances, unit_offset, NaN rows and ties included, for every variant.  w_dtype: 1 = binary16, 2 = bfloat16
 * (the dtype codes of the feature-map shards); x_dtype: 0 = fp32, 1 = binary16, 2 = bfloat16.  W is K x D row-major,
 * 2-byte aligned.
 * som_prepare_codebook_w16: c_norm2 bit-identical to som_prepare_codebook_f32 on W.float() (same summation order). */
SOM_API int    som_prepare_codebook_w16(const void* W, int w_dtype, int K, int D, float* c_norm2, void* stream);
/* som_bmu_w16_nchw is som_bmu_nchw_f32 (x fp32) or som_bmu_stage_nchw_f16 / _bf16 without stage_rows (x 16-bit; like
 * them SOM_E_UNSUPPORTED where som_bmu_f16_native says 0 -- pass the batch's fp32 copy then).  The workspace
 * (som_bmu_w16_workspace_bytes) holds the fp32 search's workspace, an exact fp32 copy of W made on every call (the
 * weights may have changed since the last one, as for c_norm2) and one flag bit per (256-unit tile, 64-feature block).
 * The FP16-split kernel (16 < D <= 256) splits -2 s_c c into FP16 hi + lo; where every lo of a tile's block is zero it
 * skips that block's B_lo load and its A_hi x B_lo product group (17 instead of 33 MMAs per tile at D = 256 when the
 * batch is 16-bit too).  The dropped products are exact zeros, so the result does not depend on the skip:
 *   binary16 : every finite lo is zero whenever s_c >= 1, i.e. whenever the largest unit norm is below 256 (a
 *              tanh-range codebook has ||c|| <= sqrt(D) <= 16);
 *   bfloat16 : lo is zero for an element within about 2^-23 of the largest |s_c c| of the codebook (the rule of bf16
 *              patch rows); units far below the largest, subnormals, inf and NaN keep the product.
 * The other kernels search the fp32 copy unchanged.                                                              */
SOM_API size_t som_bmu_w16_workspace_bytes(int64_t n_patches, int D, int K, int variant);
SOM_API int    som_bmu_w16_nchw(const void* x, int x_dtype, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                const void* W, int w_dtype, const float* c_norm2, int K, int64_t unit_offset,
                                int64_t* out_idx, float* out_rd, void* ws, size_t ws_bytes, int variant, void* stream);

/* ---- K1b: merge per-shard candidates (new; multi-GPU unit-sharded search) ---------------
 * rd, idx are (R, n) row-major; picks the smaller rd, ties -> the smaller global index,
 * which reproduces the single-device first-minimum rule when shards are index-ordered.   */
SOM_API int som_merge_candidates(const float* rd, const int64_t* idx, int R, int64_t n,
                         int64_t* out_idx, float* out_rd, void* stream);

/* ---- K5: BMU hit histogram --------------------------------------------------------------
 * counts[j] += #{p : idx[p] == j}.  Replaces the Python dict loop of
 * prune_codebook.py:129-142.  Indices outside [0, K) are ignored.                        */
SOM_API int som_histogram_i64(const int64_t* idx, int64_t n, int K, int64_t* counts, void* stream);

/* ---- K3: Gaussian neighbourhood filter along the unit axis ------------------------------
 * out = scale * T @ in,  T[a,j] = expf(-( float((j-a)^2) / float(two_var) )),
 * two_var = 2 * -(neighbourhood_range / (2 ln 0.1))   (models/Codebook.py:112-130).
 * T is exactly banded in fp32, so this is the dense S @ W of the reference after the
 * factorisation S = onehot(bmu) @ T (SURVEY.md A.3).  `in` and `out` are K x D, distinct. */
SOM_API int som_filter_f32(const float* in, float* out, int K, int D, double neighbourhood_range,
                   float scale, void* stream);

/* The same filter with a caller-owned workspace: for K >= 256 units and rows of >= 48 features it runs as a
 * banded-Toeplitz GEMM on the tensor cores (tcgen05 kind::tf32, fp32-faithful 3xTF32; the workspace holds the
 * transposed hi | lo split of `in`), otherwise -- or with ws == NULL -- it is som_filter_f32.  Replaces the dense
 * S @ W (models/Codebook.py:128-130) and its autograd transpose like som_filter_f32.
 * som_filter_workspace_bytes returns 0 when the shape takes the FFMA kernel.                               */
SOM_API size_t som_filter_workspace_bytes(int K, int D, double neighbourhood_range);
/* Band half-width h of T for this range: the largest |j - a| whose fp32 weight is non-zero (at most K - 1).  Row a
 * of the output depends on input rows [a - h, a + h] only, which is what lets a rank filter a slice of units from
 * the slice plus an h-row halo (host-only, no device work).                                                   */
SOM_API int    som_filter_half_width(int K, double neighbourhood_range);
SOM_API int som_filter_ws_f32(const float* in, float* out, int K, int D, double neighbourhood_range,
                      float scale, void* ws, size_t ws_bytes, void* stream);

/* ---- K2: per-unit accumulation (segmented by BMU, deterministic, no float atomics) ------
 *   Wt != NULL:  Rbar[a] = sum_{p: bmu[p]==a} (Wt[a] - x_p),  sse = sum_p ||Wt[bmu_p]-x_p||^2
 *   Wt == NULL:  Rbar[a] = sum_{p: bmu[p]==a} x_p             (autograd backward of the gather)
 * Replaces the S^T @ grad half of autograd for models/Codebook.py:128-130 together with
 * F.mse_loss (train_codebook.py:233-240).  Rbar (K x D) is fully overwritten.  counts (K,
 * int64) and sse (1, double) may be NULL; both are overwritten, not accumulated.         */
SOM_API size_t som_accumulate_workspace_bytes(int64_t n_patches, int D, int K);
SOM_API int som_accumulate_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                            const int64_t* bmu, const float* Wt, int K,
                            float* Rbar, int64_t* counts, double* sse,
                            void* ws, size_t ws_bytes, void* stream);

/* Data-parallel form of K2 (train_codebook.py:225-249 sharded over ranks; the reference has no counterpart):
 * `packed` holds K*D + 4 floats = [ Rbar | sse_hi, sse_lo, n/4096, n%4096 ] -- the fp64 squared error as a float
 * pair and the LOCAL patch count n as two exactly representable floats -- so that ONE fp32 all-reduce(sum) of the
 * buffer carries the accumulators, the loss numerator and the global batch size (ragged shares allowed; an empty
 * share, n_img == 0, zero-fills).  Wt must not be NULL.  Same workspace as som_accumulate_nchw_f32.        */
SOM_API int som_accumulate_packed_nchw_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                   const int64_t* bmu, const float* Wt, int K,
                                   float* packed, void* ws, size_t ws_bytes, void* stream);

/* Autograd backward of the quantise gather (drop-in path): Rbar[a] = sum_{p: bmu[p]==a} patchify(grad_out)[p]
 * -- the segment sum the reference's S^T @ grad reduces to after S = onehot(bmu) @ T; follow it
 * with som_filter_f32(scale = 1) to obtain grad_W (autograd of models/Codebook.py:128-130).
 * Same workspace as som_accumulate_nchw_f32 (this is that kernel with Wt = NULL).             */
SOM_API int som_backward_nchw_f32(const float* grad_out, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                          const int64_t* bmu, int K, float* Rbar, void* ws, size_t ws_bytes, void* stream);

/* ---- quantise: gather rows by BMU, fused unpatchify -------------------------------------
 * out[n, c, ph*pH+i, pw*pW+j] = table[idx[n*Seq+s]][d].  With table = T@W this is the
 * Gaussian branch of get_quantized_patches + unpatchify (models/Codebook.py:128-134,
 * 156-164); with table = W it is the hard branch (:132) and get_quantized_image
 * (:138-154).  Indices must be in [0, K).                                                */
SOM_API int som_quantize_nchw_f32(const int64_t* idx, const float* table, int K,
                          int64_t n_img, int C, int H, int Wd, int pH, int pW,
                          float* out, void* stream);
/* The same gather of 16-bit values (binary16, bfloat16 or any other 2-byte format: the bit patterns are copied
 * exactly); table and out 2-byte aligned.  Decodes a 16-bit codebook in its own dtype.                          */
SOM_API int som_quantize_nchw_b16(const int64_t* idx, const void* table, int K,
                                  int64_t n_img, int C, int H, int Wd, int pH, int pW,
                                  void* out, void* stream);

/* ---- K4: Adam on the codebook (fast-path trainer; the drop-in leaves it to torch) -------
 * torch.optim.Adam(betas=(b1,b2), eps) single-tensor rule, no weight decay / amsgrad
 * (train_codebook.py:183-186, 242).  `step` is the 1-based step count after increment.   */
SOM_API int som_adam_f32(float* W, float* m, float* v, const float* g, int64_t n,
                 double lr, double b1, double b2, double eps, int64_t step, void* stream);

/* Same update with the step count kept in DEVICE memory (for CUDA-graph replay of the training
 * step): uses t = *steps_done + 1, then increments *steps_done on the stream.               */
SOM_API int som_adam_devstep_f32(float* W, float* m, float* v, const float* g, int64_t n,
                         double lr, double b1, double b2, double eps, int64_t* steps_done, void* stream);

/* Data-parallel tail of the step: `g` is the UNSCALED gradient T @ Rbar_global (som_filter_ws_f32 with scale 1 on
 * the all-reduced accumulators) and `tail` the all-reduced 4-float tail of som_accumulate_packed_nchw_f32.  Applies
 * g * (float)(2 / numel), numel = D * n_global (F.mse_loss's mean, train_codebook.py:233-235) and the Adam rule of
 * som_adam_devstep_f32; writes loss = sse / numel to loss_out (device double, may be NULL) -- except at n == 0,
 * where only the step count advances and loss_out is left as it was.  Everything the host
 * would have to wait for stays on the device, so the whole step can be captured in a CUDA graph.
 * steps_done points to TWO int64: [0] the number of completed steps (t = steps_done[0] + 1 is used, then it is
 * incremented by the kernel itself), [1] a scratch word the kernel uses as its block-arrival counter: zero it once,
 * the kernel leaves it at zero.                                                                               */
SOM_API int som_adam_dp_f32(float* W, float* m, float* v, const float* g, int64_t n, int D,
                    double lr, double b1, double b2, double eps, int64_t* steps_done,
                    const float* tail, double* loss_out, void* stream);

/* ---- one-kernel training step for small problems (BASELINE config 1: 512 patches, K = 1024, D = 64) --------
 * The whole iteration of train_codebook.py:225-249 (forward with the Gaussian neighbourhood, mse_loss, backward,
 * Adam(b1, b2, eps); models/Codebook.py:77-135) as ONE cooperative kernel with three grid barriers: W~ = T @ W,
 * BMU (fp32 FFMA, first minimum on ties), per-unit residual sums in ascending patch order, G = (2/numel) T @ Rbar,
 * Adam in place on W / m / v, loss = mean squared error to loss_out (device double, may be NULL), BMU indices to
 * bmu_out (n_patches int64, may be NULL).  Covered shapes: n_patches <= 2048, D in {16, 32, 64, 128, 256},
 * K <= 32 * SMs, <= 16 * SMs patches, band half-width <= 2048: som_step_small_workspace_bytes returns 0 otherwise
 * (and the call SOM_E_UNSUPPORTED) -- use the separate kernels then.  steps_done: two int64 as for som_adam_dp_f32
 * ([0] is read as the completed-step count and incremented; [1] is not touched).                              */
SOM_API size_t som_step_small_workspace_bytes(int64_t n_patches, int D, int K, double neighbourhood_range);
SOM_API int som_step_small_f32(const float* x, int64_t n_img, int C, int H, int Wd, int pH, int pW,
                       float* W, float* m, float* v, int K, double neighbourhood_range,
                       double lr, double b1, double b2, double eps, int64_t* steps_done,
                       int64_t* bmu_out, double* loss_out, void* ws, size_t ws_bytes, void* stream);

/* ---- data-parallel tail over NVLink / NVSwitch peer memory (new; multi-GPU only) -------------------------
 * Replaces, across ranks, "all-reduce the accumulators, then every rank filters and updates the whole codebook"
 * (train_codebook.py:240-242 + models/Codebook.py:112-130 have no multi-GPU form in the reference).  Pointers
 * named mc_* are NVSwitch MULTICAST addresses of caller-owned symmetric allocations (the same offset in the same
 * allocation on every rank); `signal_pads` is a HOST array of `world` device pointers, entry r = rank r's flag
 * area (som_peer_signal_bytes() bytes, zero-filled once, peer-mapped) as seen from THIS rank.  Every call must be
 * made by all ranks in the same order with the same `channel` (0..3); the flags reset themselves, so the calls can
 * be replayed from a CUDA graph (the max_* arguments are kept for ABI stability and ignored).  One barrier costs
 * `world` remote atomics: the last block of a kernel to arrive runs the exchange for its grid, and a kernel that
 * must see the peers' earlier work is preceded by a one-block barrier kernel.  A peer that never arrives makes the
 * kernel trap after ~4 s instead of hanging.                                                                  */
SOM_API size_t som_peer_signal_bytes(void);
/* In-place all-reduce(sum) of n floats (n % 4 == 0): rank r reduces quads [r*n/4/world, ...) in the switch
 * (multimem.ld_reduce) and stores them to every rank (multimem.st).  With peer_bufs (HOST array of the buffer's
 * `world` peer addresses) and tail_out (a LOCAL 4-float buffer, 16-byte aligned, not part of the buffer) the buffer
 * is a packed accumulator buffer: its last 4 floats are the tail of som_accumulate_packed_nchw_f32; they stay as
 * they are on every rank and are summed EXACTLY into tail_out instead -- every rank reads the R tails through the
 * peer addresses and adds them in rank order, the squared error in fp64 (the patch count must be exact).
 * Both NULL: plain data, all n floats reduced in the switch.                                                  */
SOM_API int som_peer_allreduce_f32(void* mc_buf, int64_t n, void* const* peer_bufs, float* tail_out, int rank,
                           int world, void* const* signal_pads, int channel, void* stream);
/* Rows [row0, row1) of the K x D accumulator matrix at mc_packed (layout of som_accumulate_packed_nchw_f32),
 * reduced over the ranks into LOCAL out_rows, and the reduced 4-float tail into LOCAL out_tail: the
 * reduce-scatter half of the all-reduce for a rank that owns a slice of units plus the filter's halo.
 * max_rows = the largest row1 - row0 of any rank.  Waits until every rank's accumulators are complete.  The tail
 * is summed exactly through peer_packed (HOST array of the buffer's peer addresses), as in som_peer_allreduce_f32. */
SOM_API int som_peer_reduce_rows_f32(const void* mc_packed, void* const* peer_packed, int K, int D, int row0,
                             int row1, int max_rows, float* out_rows, float* out_tail, int rank, int world,
                             void* const* signal_pads, int channel, void* stream);
/* The same reduction FUSED into its consumer: out_rows (row1 - row0 x D) = scale * T @ (sum over the ranks of rows
 * [row0, row1)), T the neighbourhood matrix of a (row1 - row0)-unit codebook as in som_filter_ws_f32 (ws / ws_bytes:
 * som_filter_workspace_bytes(row1 - row0, D, range)).  The filter's pre-pass reads the rows through the multicast
 * address with the in-switch add, so no reduced copy exists in between; out_tail as above.  Shapes the tensor-core
 * filter does not take run som_peer_reduce_rows_f32 into rows_scratch (max_rows x D floats) + som_filter_ws_f32.
 * row0 < row1 (a rank that owns no rows calls som_peer_reduce_rows_f32 with row0 == row1).  Replaces, across ranks,
 * loss.backward()'s S^T @ dL/dW~ (models/Codebook.py:128-130) after the ranks' accumulators exist.              */
SOM_API int som_peer_reduce_filter_rows_f32(const void* mc_packed, void* const* peer_packed, int K, int D, int row0,
                             int row1, int max_rows, double neighbourhood_range, float scale, float* rows_scratch,
                             float* out_rows, float* out_tail, int rank, int world, void* const* signal_pads,
                             int channel, void* ws, size_t ws_bytes, void* stream);
/* n floats of local src_rows stored to mc_dst_rows on every rank, then a barrier over the ranks: when the call
 * has completed on a rank, every rank's rows have landed in its copy.  max_n = the largest n of any rank.      */
SOM_API int som_peer_bcast_rows_f32(const float* src_rows, void* mc_dst_rows, int64_t n, int64_t max_n, int rank,
                            int world, void* const* signal_pads, int channel, void* stream);
/* som_adam_dp_f32 on the n weights of this rank's rows (all pointers address the slice; W_rows is this rank's
 * local copy, read) with the updated rows stored to mc_W_rows on EVERY rank -- the all-gather fused into the
 * update -- then the barrier over the ranks.  steps_done: two int64 as for som_adam_dp_f32.                   */
SOM_API int som_peer_adam_slice_f32(const float* W_rows, void* mc_W_rows, float* m_rows, float* v_rows,
                            const float* g_rows, int64_t n, int64_t max_n, int D, double lr, double b1,
                            double b2, double eps, int64_t* steps_done, const float* tail, double* loss_out,
                            int rank, int world, void* const* signal_pads, int channel, void* stream);

/* ---- row compaction for pruning ----------------------------------------------------------
 * out[r] = W[keep[r]] for r < n_keep (prune_codebook.py:161-162).                        */
SOM_API int som_gather_rows_f32(const float* W, int D, const int64_t* keep, int64_t n_keep,
                        float* out, void* stream);
/* The same for 16-bit rows (bit patterns copied exactly, 2-byte aligned): pruning a 16-bit codebook.            */
SOM_API int som_gather_rows_b16(const void* W, int D, const int64_t* keep, int64_t n_keep,
                                void* out, void* stream);

/* ---- dual-codebook token assembly (tokenisation call site of the Transformer trainer) ----
 * Replaces the index arithmetic of train_quantized_transformer.py:411-455 after the two
 * get_patches_bmu calls: lr_idx (n, lr_seq) and hr_idx (n, hr_seq) are the UNSHIFTED BMU
 * indices of the low- / high-resolution codebooks of the same feature maps.
 *   base_model != 0 : hr_input (n, lr_seq + hr_seq) = [ lr_idx | hr_idx + lr_K ]   (:425-431)
 *   base_model == 0 : hr_input (n, 1 + hr_seq)      = [ hr_K   | hr_idx ]          (:436-441)
 *   always          : hr_target (n, hr_seq + 1)     = [ hr_idx | hr_K ]            (:449-454)
 * hr_K (= hr_num_embeddings) is the reference's <start>/<end> token.                       */
SOM_API int som_assemble_tokens_i64(const int64_t* lr_idx, const int64_t* hr_idx, int64_t n,
                            int lr_seq, int hr_seq, int64_t lr_K, int64_t hr_K, int base_model,
                            int64_t* hr_input, int64_t* hr_target, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SOMCB_H_ */
