/* nerf_pl_b200 — C ABI of the B200-native volumetric-rendering hot path of kwea123/nerf_pl.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Every entry point
 * cites the reference interface it replaces (paths relative to the reference repository).
 * All pointers are DEVICE pointers unless the name ends in `_host`.  `stream` is a
 * cudaStream_t passed as void* (NULL = legacy default stream).  Functions never allocate or
 * free caller-visible memory and never throw.
 *
 * Return value: 0 = ok; negative = invalid argument (NERFB200_E*); positive = cudaError_t.
 * nerfb200_last_error() returns a thread-local, human-readable description of the last
 * non-zero return on this thread.
 */
#ifndef NERF_PL_B200_H_
#define NERF_PL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NERFB200_ABI_VERSION 3

#define NERFB200_EINVAL (-1)      /* bad argument value / null pointer            */
#define NERFB200_EUNSUPPORTED (-2) /* shape outside what the fused kernel supports */
#define NERFB200_EDEVICE (-3)     /* device is not sm_100 / kernel image missing   */

int nerfb200_abi_version(void);
const char* nerfb200_last_error(void);

/* ---- weights --------------------------------------------------------------------------
 * Replaces: the implicit use of the 12 nn.Linear parameter tensors by NeRF.forward
 * (models/nerf.py:61-81, 83-124).  `params` are the 24 fp32 device tensors of one NeRF in
 * state_dict order: xyz_encoding_{1..8}.0.{weight,bias}, xyz_encoding_final.{weight,bias},
 * dir_encoding.0.{weight,bias}, sigma.{weight,bias}, rgb.0.{weight,bias}; weights are
 * (out,in) row-major as torch stores them.  Produces the fp16/fp32 image the kernels stream
 * (nerfb200_packed_bytes() bytes, 1024-byte aligned): the forward slices, the fp32 constants and
 * the transposed 16-bit slices of the backward chain kernel. */
size_t nerfb200_packed_bytes(void);
int nerfb200_pack_weights(const float* const params[24], void* packed, void* stream);
/* Both networks of a render (coarse, fine) in ONE launch: what a training step does after every optimiser update. */
int nerfb200_pack_weights_pair(const float* const params_a[24], void* packed_a, const float* const params_b[24],
                               void* packed_b, void* stream);

/* ---- render_rays -----------------------------------------------------------------------
 * Replaces: models/rendering.py:58-244 render_rays(models, embeddings, rays, N_samples,
 * use_disp, perturb, noise_std, N_importance, chunk, white_back, test_time) including the
 * inner inference() closure (:91-172), sample_pdf (:14-55), the torchsearchsorted call
 * (:42) and the torch.sort merge (:229).  `chunk` has no equivalent (nothing is chunked).
 *
 * rays: (n_rays, 8) fp32 rows [o(3) d(3) near far], row stride `ray_stride` floats.
 * Random inputs are supplied by the caller so a seeded torch stream can be reproduced:
 *   perturb_rand (n_rays,N_samples) U[0,1)  — required iff perturb > 0     (:203)
 *   noise_coarse (n_rays,N_samples) N(0,1)  — required iff noise_std > 0   (:152)
 *   u_rand       (n_rays,N_importance) U[0,1) — required iff perturb > 0 and N_importance > 0 (:39)
 *   noise_fine   (n_rays,N_samples+N_importance) N(0,1) — iff noise_std > 0 and N_importance > 0
 * Outputs (result-dict keys, :209-221, :240-242); fp32:
 *   rgb_coarse (n,3), depth_coarse (n) — written unless test_time; may be NULL if test_time
 *   opacity_coarse (n); rgb_fine (n,3), depth_fine (n), opacity_fine (n) iff N_importance > 0
 * Optional outputs (NULL to skip): z_fine (n, N_samples+N_importance) merged sorted depths,
 *   weights_coarse (n,N_samples), weights_fine (n,N_samples+N_importance).
 * Supported shapes: N_samples in {32, 64, 128}; N_importance a multiple of 32 (0 = coarse only);
 * N_samples + N_importance <= 192 (the reference defaults 64 + 128 and the README recipes 64 + 64 included).
 * `status` is a device int32 the kernel sets non-zero on a device-side fault.  It may be NULL:
 * then a per-device internal word (mapped pinned host memory) is used; the library reads it
 * without synchronising at the START of every later call on that device and returns
 * NERFB200_EDEVICE once if an earlier kernel reported a fault (nerfb200_check_status() does the
 * same check on demand, e.g. after a stream synchronise).  The *_host entry always checks the
 * word of its own launch before returning. */
typedef struct nerfb200_render_args {
  const float* rays;
  int64_t n_rays;
  int64_t ray_stride;
  const void* packed_coarse;
  const void* packed_fine; /* NULL iff n_importance == 0 */
  int32_t n_samples;
  int32_t n_importance;
  int32_t use_disp;
  float perturb;
  float noise_std;
  int32_t white_back;
  int32_t test_time;
  const float* perturb_rand;
  const float* noise_coarse;
  const float* u_rand;
  const float* noise_fine;
  float* rgb_coarse;
  float* depth_coarse;
  float* opacity_coarse;
  float* rgb_fine;
  float* depth_fine;
  float* opacity_fine;
  float* z_fine;
  float* weights_coarse;
  float* weights_fine;
  int32_t* status;
  int32_t max_ctas; /* 0 = one CTA per SM */
  /* Optional: the (stratified) coarse depths (n, N_samples) (models/rendering.py:189-204). */
  float* z_coarse;
  /* Training mode (NULL = inference; requires test_time == 0): a device workspace of
   * nerfb200_train_workspace_bytes() bytes, initialised once with nerfb200_train_workspace_init().
   * The same fused launch then also stores, per sample, what nerfb200_render_backward needs: the
   * encoded input and the outputs of xyz_encoding_1..8 (fp16), the ReLU sign bits, the output of
   * dir_encoding, raw sigma, rgb and the depths of both passes. */
  void* train_workspace;
  /* Fused loss epilogue (replaces losses.py:9-14 MSELoss.forward and metrics.py:4-13 psnr on the
   * rendered batch; all NULL = off): target (n,3) -> loss_out[4] (device) = {mse(rgb_coarse),
   * mse(rgb_fine) or 0, their sum (= MSELoss), psnr of the finest pass}.  Needs train_workspace
   * (it holds the per-CTA partial sums; the reduction order is fixed, so the result is
   * deterministic). */
  const float* target;
  float* loss_out;
  /* Uniform random inputs drawn INSIDE the kernel (rng_in_kernel != 0): perturb_rand / u_rand may then be NULL and
   * are ignored; element (ray r, index i) of stream s (0 = perturb_rand, 1 = u_rand) is word i & 3 of
   * Philox4x32-10(counter = {r, i >> 2, s, 0}, key = {rng_seed lo, hi}) mapped to [0,1) as (x >> 8) * 2^-24 -
   * counter-based, so the numbers do not depend on the launch shape and a host replica reproduces them
   * (tests/philox.py).  The reference draws these with torch.rand from the global generator
   * (models/rendering.py:203, :39); the tensor inputs remain the way to replay a seeded torch stream.  The Gaussian
   * noise inputs (noise_std > 0) are always tensors. */
  uint64_t rng_seed;
  int32_t rng_in_kernel;
} nerfb200_render_args;

int nerfb200_render_rays(const nerfb200_render_args* args, void* stream);

/* ---- training step: backward of render_rays -------------------------------------------------
 * Replaces: loss.backward() of train.py:103-117 through models/rendering.py:143-170 (quadrature)
 * and models/nerf.py:100-124 (both MLPs); no gradient flows through the fine-depth sampling
 * (models/rendering.py:225-227 .detach()) nor into the rays.
 *
 * Protocol: (1) nerfb200_render_rays(args with train_workspace set, test_time = 0);
 * (2) nerfb200_render_backward with the SAME render args (rays, random inputs, flags, packed
 * images, outputs) and either the upstream gradients of the result tensors (g_*, any may be
 * NULL = zero) or `target` (the fused MSE seed dL/drgb = 2 (rgb - target) / (3 n) * *loss_grad for
 * both passes, added to g_rgb_* if those are given).  Writes the gradients of the 24 parameter
 * tensors of each network (state_dict order and shapes, fp32; `params_*` are the live fp32
 * parameters).  grads_fine / params_fine are ignored when n_importance == 0.
 * All kernels are hand-written sm_100a code on `stream`: compositing backward, rgb head,
 * tcgen05 dgrad chain, tcgen05 split-K wgrad, partial reduction, unfolding of the packed
 * final.dir layer. */
size_t nerfb200_train_workspace_bytes(int64_t n_rays, int32_t n_samples, int32_t n_importance);
/* One-time set-up of a workspace for (n_rays, n_samples, n_importance): zeroes the padding rows,
 * counters and uploads the wgrad job table.  Synchronous with respect to `stream`. */
int nerfb200_train_workspace_init(void* workspace, size_t bytes, int64_t n_rays, int32_t n_samples,
                                  int32_t n_importance, void* stream);
/* fp16 gradient elements that the last nerfb200_render_backward on this workspace stored at the fp16
 * limit (clipped by the saturating conversion) or as NaN, for the coarse and the fine pass: out[2] on
 * the host.  0 unless a batch defeats the per-layer scale selection (DESIGN.md section 3); the weight
 * gradients of a step with a non-zero count are inexact.  Synchronises `stream`. */
int nerfb200_train_saturation(const void* workspace, int64_t n_rays, int32_t n_samples, int32_t n_importance,
                              uint32_t* out, void* stream);
typedef struct nerfb200_backward_args {
  const nerfb200_render_args* render;   /* as passed to the forward call */
  const float* const* params_coarse;    /* 24 device pointers */
  const float* const* params_fine;
  const float* g_rgb_coarse;            /* (n,3) */
  const float* g_depth_coarse;          /* (n)   */
  const float* g_opacity_coarse;        /* (n)   */
  const float* g_rgb_fine;
  const float* g_depth_fine;
  const float* g_opacity_fine;
  const float* target;                  /* (n,3) or NULL */
  const float* loss_grad;               /* device scalar or NULL (= 1) */
  float* const* grads_coarse;           /* 24 device pointers, shapes of params_coarse */
  float* const* grads_fine;
} nerfb200_backward_args;
int nerfb200_render_backward(const nerfb200_backward_args* args, void* stream);

/* ---- optimiser step ("next" row: the caller of the backward) ---------------------------------
 * Replaces: torch.optim.Adam.step() as the reference configures it (utils/__init__.py:16-18:
 * Adam(lr, eps, weight_decay), betas (0.9, 0.999), no amsgrad; train.py:77-82) for up to 64 fp32
 * tensors in one launch.  `step` is the 1-based count of this update (bias correction). */
int nerfb200_adam_step(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                       float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2, float eps,
                       float weight_decay, int64_t step, void* stream);

/* Same call with HOST buffers; returns with the requested outputs readable on the host (synchronises `stream`).
 * The packed weight images stay device-resident.  This is the end-to-end entry the reference's eval.py loop
 * (eval.py:117-123 `.cuda()` ... `.cpu()`) maps to.
 *   - every buffer page-locked and mapped (cudaHostAlloc / cudaHostRegister, torch pin_memory()): the kernel reads
 *     the rays and writes the results over PCIe itself; the call is launch + synchronise, no staging copies;
 *   - otherwise (pageable memory): rays and the random inputs that are non-NULL and not already device memory are
 *     staged with cudaMemcpyAsync, results are copied back the same way.
 * Random inputs may be device pointers in both cases (drawn on the device by the caller). */
int nerfb200_render_rays_host(const nerfb200_render_args* host_args, void* stream);

/* ---- NeRF.forward ------------------------------------------------------------------------
 * Replaces: models/nerf.py:83-124 NeRF.forward(x, sigma_only).  x: (n, x_stride) fp32 rows of
 * embedded xyz (63) followed, unless sigma_only, by the embedded direction (27).
 * out: (n,4) [r,g,b,sigma] or (n,1) sigma. */
int nerfb200_nerf_forward(const float* x, int64_t n, int64_t x_stride, const void* packed,
                          int32_t sigma_only, float* out, void* stream);

/* ---- dense sigma query ("next" row: mesh extraction) -------------------------------------
 * Replaces: extract_color_mesh.py:127-140 (embedding_xyz + embedding_dir + cat + nerf(...)[:, -1]
 * per chunk): raw positions xyz (n, xyz_stride >= 3) -> raw sigma (n); the positional encoding is
 * computed in the kernel, the direction does not enter sigma (models/nerf.py:112). */
int nerfb200_query_sigma(const float* xyz, int64_t n, int64_t xyz_stride, const void* packed, float* sigma,
                         void* stream);

/* ---- loss / metric epilogue ("next" row) -------------------------------------------------
 * Replaces: losses.py:9-14 MSELoss.forward and metrics.py:4-13 psnr on the rendered batch.
 * rgb_coarse / rgb_fine: (n_rays,3), either may be NULL; target (n_rays,3).
 * out4 (device): [mse_coarse, mse_fine, mse_coarse + mse_fine, psnr of the finest pass]. */
int nerfb200_mse_psnr(const float* rgb_coarse, const float* rgb_fine, const float* target, int64_t n_rays,
                      float* out4, void* stream);

/* ---- Embedding.forward -------------------------------------------------------------------
 * Replaces: models/nerf.py:21-38.  x: (n,3) -> out: (n, 3 + 6*n_freqs). */
int nerfb200_embed(const float* x, int64_t n, int32_t n_freqs, float* out, void* stream);

/* ---- searchsorted ------------------------------------------------------------------------
 * Replaces: torchsearchsorted/src/torchsearchsorted/searchsorted.py:20-53 and
 * src/cuda/searchsorted_cuda_kernel.cu:83-142.  a: (nrow_a, ncol_a) sorted rows,
 * v: (nrow_v, ncol_v); nrow_a == nrow_v or one of them is 1 (broadcast).
 * out: (max(nrow_a,nrow_v), ncol_v) int64.  side_right: 0 = 'left', 1 = 'right'. */
int nerfb200_searchsorted(const float* a, const float* v, int64_t* out, int64_t nrow_a,
                          int64_t nrow_v, int32_t ncol_a, int32_t ncol_v, int32_t side_right,
                          void* stream);

/* ---- sample_pdf --------------------------------------------------------------------------
 * Replaces: models/rendering.py:14-55 with the random/deterministic u supplied by the caller.
 * bins (n_rays, n_weights+1), weights (n_rays, n_weights), u (n_rays, n_u) -> out (n_rays, n_u). */
int nerfb200_sample_pdf(const float* bins, const float* weights, const float* u, int64_t n_rays,
                        int32_t n_weights, int32_t n_u, float* out, void* stream);

/* ---- volume rendering quadrature ---------------------------------------------------------
 * Replaces: models/rendering.py:143-170 (inside inference()).  sigmas (n,S), rgbs (n,S,3) or
 * NULL (weights_only), z_vals (n,S), dirs (n,3), noise (n,S) or NULL.  S % 32 == 0, S <= 192.
 * weights (n,S) may be NULL; rgb (n,3) / depth (n) ignored when rgbs is NULL; opacity (n). */
int nerfb200_composite(const float* sigmas, const float* rgbs, const float* z_vals,
                       const float* dirs, const float* noise, float noise_std, int32_t white_back,
                       int64_t n_rays, int32_t n_samples, float* weights, float* rgb, float* depth,
                       float* opacity, void* stream);

/* ---- ray generation ("next" row: the caller side of the path) ----------------------------
 * Replaces: datasets/ray_utils.py:5-94 get_ray_directions + get_rays (+ get_ndc_rays as
 * datasets/llff.py:236-241 applies it when ndc != 0: near plane 1.0, near/far columns 0/1) and
 * the torch.cat of datasets/blender.py:97-102.  c2w_host: 12 HOST floats, row-major (3,4).
 * rays: (H*W, 8) device rows [o(3) d(3) near far], pixel order row-major (j, i). */
int nerfb200_generate_rays(int32_t H, int32_t W, float focal, const float c2w_host[12], float near, float far,
                           int32_t ndc, float* rays, void* stream);

/* Replaces: eval.py:126-128 (clip(img,0,1)*255).astype(uint8) on the rendered image, on device. */
int nerfb200_to_uint8(const float* src, int64_t n, uint8_t* dst, void* stream);

/* ---- diagnostics -------------------------------------------------------------------------
 * Number of kernels this library has launched on the calling process so far (all entry
 * points).  bench.py reports the delta as `gpu_launches`. */
int64_t nerfb200_launch_count(void);
/* Returns NERFB200_EDEVICE (and clears the flag) if a kernel launched by an earlier call on the
 * current device reported a device-side fault through the internal status word; 0 otherwise.
 * Does not synchronise: call it after synchronising the stream to cover the latest launch. */
int nerfb200_check_status(void);
/* Device properties the launcher uses: SM count of the current device (0 if none). */
int nerfb200_sm_count(void);

#ifdef __cplusplus
}
#endif
#endif /* NERF_PL_B200_H_ */
