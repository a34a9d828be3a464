/* nrnerf_b200 -- C ABI of the B200-native NR-NeRF render hot path (libnrnerf_b200.so).
 *
 * Plain C: raw device pointers, sizes, a cudaStream_t passed as void*.  No torch types, no C++
 * types, no exceptions.  Every function returns 0 on success or a negative NRN_E_* code; the
 * message is available from nrn_last_error() (thread-local).  All work is enqueued on the given
 * stream; nothing synchronises except nrn_device_error().
 *
 * The reference (facebookresearch/nonrigid_nerf) has no FFI layer: its boundary for this path is a
 * set of Python callables.  Each entry point below names the reference function(s) it replaces
 * (paths relative to the reference checkout); INTEGRATION.md shows the ctypes binding.
 */
#ifndef NRNERF_B200_H
#define NRNERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRN_ABI_VERSION 2

#define NRN_OK 0
#define NRN_E_INVALID (-1)   /* bad argument / unsupported configuration */
#define NRN_E_CUDA (-2)      /* CUDA runtime error (see nrn_last_error) */
#define NRN_E_DEVICE (-3)    /* device-side protocol error recorded by a kernel */

int nrn_abi_version(void);
const char* nrn_last_error(void);

/* Synchronises the current device, reads and clears the device-side error word written by the
 * fused kernels (0 = ok; non-zero = id of the mbarrier wait that timed out). */
int nrn_device_error(int* code_out);

/* ---- weight packing -------------------------------------------------------------------------
 * fp32 nn.Linear tensors in the reference's checkpoint layout ([out][in] row-major) -> fp16 UMMA
 * operand images.  Replaces nothing in the reference (derived data); sources are
 * NeRF.pts_linears / output_linear (run_nerf_helpers.py:218-238) and ray_bending.network /
 * rigidity_network (run_nerf_helpers.py:411-482). */
size_t nrn_packed_nerf_bytes(void);
size_t nrn_packed_bender_bytes(void);
/* w[0..7] = pts_linears.i.weight, w[8] = output_linear.weight; b likewise. input_ch = 63. */
int nrn_pack_nerf(const float* const* w, const float* const* b, int input_ch, int out_ch, void* packed,
                  void* stream);
int nrn_pack_bender(const float* const* net_w /*5*/, const float* const* net_b /*4*/,
                    const float* const* rig_w /*3*/, const float* const* rig_b /*3*/, int latent_size,
                    void* packed, void* stream);

/* ---- ray generation: get_rays / get_rays_np (run_nerf_helpers.py:588-622) on the device -----------------------------
 * c2w [3][4] row-major, intrinsics = (focal_x, focal_y, center_x, center_y); rays_o / rays_d [H*W][3] in the [H, W, 3]
 * order of the reference.  Bit-identical to the reference's float32 arithmetic. */
int nrn_get_rays(const float* c2w, const float* intrinsics, int height, int width, float* rays_o, float* rays_d, void* stream);
/* rays [n][8] = (o, d, near, far) as render() assembles them before batchify_rays (train.py:388-398), scalar near / far. */
int nrn_pack_rays(const float* rays_o, const float* rays_d, float near, float far, int n_rays, float* rays, void* stream);
/* A training batch computed on demand instead of gathered from the host table of every ray of every image
 * (train.py:1498-1517, :1546-1564): pix [n][3] int64 = (image, x, y) as in batch_pixel_indices; poses [n_images][3][4];
 * intrinsics [n_views][4]; image_to_view [n_images] int32 or NULL (single view); images [n_images][H][W][3] fp32 or NULL
 * (then target may be NULL). */
int nrn_ray_batch(const int64_t* pix, int n, const float* poses, const float* intrinsics, const int32_t* image_to_view,
                  const float* images, int height, int width, float* rays_o, float* rays_d, float* target, void* stream);
/* ---- free-viewpoint post-processing, free_viewpoint_rendering.py:623-629: per ray the index of the sample whose
 * accumulated visibility weight is closest to 0.5 (first minimum).  weights [n][n_samples] -> index [n] int64. */
int nrn_median_visibility_index(const float* weights, int n_rays, int n_samples, int64_t* index, void* stream);

/* ---- coarse depth sampling: render_rays, train.py:847-869 ------------------------------------
 * rays [n][8] = (o, d, near, far); t_rand [n][S] uniform randoms or NULL (perturb == 0). */
int nrn_sample_coarse(const float* rays, const float* t_rand, int n_rays, int n_samples, int lindisp,
                      float* z_vals, void* stream);

/* ---- fused field evaluation: run_network (train.py:57-105) + NeRF.forward
 * (run_nerf_helpers.py:240-314) + ray_bending.forward (:507-584) + Embedder.embed (:149-150) --- */
typedef struct NrnFieldArgs {
  const float* rays;          /* [n_rays][8] (o, d, near, far) */
  const float* z_vals;        /* [n_rays][n_samples] */
  const float* points;        /* point mode (NeRF.forward(x), run_nerf_helpers.py:240): rays = z_vals = NULL,
                                 n_samples = 1, n_rays = number of points; xyz = points[i*points_stride + 0..2] */
  int64_t points_stride;
  const float* latents;       /* [n_rays][32], NULL when bender_packed is NULL */
  int64_t latent_stride;      /* floats between consecutive rays' latents (0 = broadcast one row) */
  int32_t n_rays;
  int32_t n_samples;
  const void* nerf_packed;    /* nrn_pack_nerf output */
  const void* bender_packed;  /* nrn_pack_bender output or NULL (canonical rendering, ray_bender=(None,)) */
  int32_t out_ch;             /* 4 or 5 (output_linear rows) */
  int32_t use_cutoff;  float rigidity_cutoff;   /* ray_bending.rigidity_test_time_cutoff */
  int32_t use_scaling; float scaling;           /* ray_bending.test_time_scaling */
  int32_t use_removal; float removal_threshold; /* NeRF.test_time_nonrigid_object_removal_threshold */
  float* raw;                 /* out [n_rays][n_samples][out_ch] */
  float* initial_input_pts;   /* out [P][3] or NULL  (details of detailed_output=True) */
  float* input_pts;           /* out [P][3] or NULL */
  float* unmasked_offsets;    /* out [P][3] or NULL */
  float* masked_offsets;      /* out [P][3] or NULL */
  float* rigidity_mask;       /* out [P]    or NULL */
  void* stash;                /* training only: activation stash of nrn_stash_bytes() bytes, else NULL */
  void* stream;
} NrnFieldArgs;
int nrn_field_forward(const NrnFieldArgs* args);

/* ---- compositing: raw2outputs (train.py:724-789), optionally fused with sample_pdf
 * (run_nerf_helpers.py:651-698), the sort of train.py:920 and z_std of train.py:959 ------------ */
typedef struct NrnCompositeArgs {
  const float* raw;           /* [n][S][C] */
  const float* z_vals;        /* [n][S] */
  const float* rays_d;        /* ray directions, row stride rays_d_stride floats */
  int32_t rays_d_stride;
  const float* noise;         /* [n][S] sigma noise already multiplied by raw_noise_std, or NULL */
  int32_t n_rays, n_samples, channels, white_bkgd;
  float* rgb_map;             /* out [n][3] */
  float* disp_map;            /* out [n] */
  float* acc_map;             /* out [n] */
  float* depth_map;           /* out [n] or NULL */
  float* weights;             /* out [n][S] or NULL */
  float* alpha;               /* out [n][S] or NULL */
  int32_t n_importance;       /* 0 = composite only */
  const float* u;             /* [n][n_importance] or NULL (deterministic linspace, perturb == 0) */
  float* z_vals_out;          /* out [n][S + n_importance] sorted union */
  float* z_std;               /* out [n] or NULL */
  void* stream;
} NrnCompositeArgs;
int nrn_composite(const NrnCompositeArgs* args);

/* stand-alone sample_pdf (run_nerf_helpers.py:651-698): bins [n][nbins], weights [n][nbins-1] */
int nrn_sample_pdf(const float* bins, const float* weights, const float* u, int n, int nbins, int n_samples,
                   float* samples, void* stream);

/* ---- backward of raw2outputs w.r.t. raw (what torch.autograd derives for train.py:724-789) ---- */
typedef struct NrnCompositeBwdArgs {
  const float* raw; const float* z_vals; const float* rays_d; int32_t rays_d_stride; const float* noise;
  int32_t n_rays, n_samples, channels, white_bkgd;
  const float* d_rgb_map;     /* [n][3] */
  const float* d_acc_map;     /* [n] or NULL */
  float* d_raw;               /* out [n][S][C] */
  void* stream;
} NrnCompositeBwdArgs;
int nrn_composite_backward(const NrnCompositeBwdArgs* args);

/* ---- backward of the fused field (what torch.autograd derives for NeRF.forward +
 * ray_bending.forward, run_nerf_helpers.py:240-314 / :507-584; SURVEY.md appendix C):
 * DGRAD chain + WGRAD + deterministic split reduction.  Needs the stash written by
 * nrn_field_forward (ray mode) and, with a bender, that call's unmasked_offsets / rigidity_mask. */
size_t nrn_stash_bytes(int n_rays, int n_samples);
size_t nrn_grad_stash_bytes(int n_rays, int n_samples);
size_t nrn_wgrad_scratch_bytes(void);
int nrn_nerf_grad_floats(int out_ch);   /* flat order: W0 b0 W1 b1 ... W7 b7 Wout bout (reference shapes) */
int nrn_bender_grad_floats(void);       /* flat order: network.0.w .0.b .1.w .1.b .2.w .2.b .3.w .3.b .4.w,
                                           rigidity_network.0.w .0.b .1.w .1.b .2.w .2.b */
typedef struct NrnFieldBwdArgs {
  int32_t n_rays, n_samples, out_ch;
  const float* d_raw;             /* [n_rays][n_samples][out_ch] upstream gradient */
  const void* stash;              /* from the forward call */
  void* grad_stash;               /* workspace, nrn_grad_stash_bytes() */
  float* wgrad_scratch;           /* workspace, nrn_wgrad_scratch_bytes() */
  const void* nerf_packed;
  const void* bender_packed;      /* or NULL */
  const float* unmasked_offsets;  /* [P][3] forward output (bender only) */
  const float* rigidity_mask;     /* [P]    forward output (bender only) */
  const float* d_unmasked_offsets;/* [P][3] upstream gradient (offsets regulariser) or NULL */
  const float* d_rigidity_mask;   /* [P]    upstream gradient (rigidity regulariser) or NULL */
  int32_t use_cutoff;  float rigidity_cutoff;
  int32_t use_scaling; float scaling;
  float* nerf_grad;               /* out, nrn_nerf_grad_floats(out_ch) floats, overwritten */
  float* bender_grad;             /* out, nrn_bender_grad_floats() floats, overwritten (or NULL) */
  float* d_latents;               /* out [n_rays][32], overwritten (or NULL without bender) */
  void* stream;
  /* Gradients written where PyTorch keeps them (SURVEY.md 8b "gradient buffers that alias param.grad"):
   * nerf_grad_head, if not NULL, receives the output_linear part (Wout bout) instead of the tail of nerf_grad -- in
   * module.parameters() order the dead views_linears sit between pts_linears and output_linear; accumulate_* != 0
   * adds to the destination instead of overwriting it (what autograd's AccumulateGrad would do). */
  float* nerf_grad_head;
  int32_t accumulate_nerf, accumulate_bender;
} NrnFieldBwdArgs;
int nrn_field_backward(const NrnFieldBwdArgs* args);

/* ---- divergence regulariser of the offset field on the coarse samples: compute_divergence_loss /
 * divergence_approx (run_nerf_helpers.py:22-116) as driven by train.py:245-286, forward and backward
 * in closed form (no double backward).  Needs the coarse pass's activation stash. ---------------- */
size_t nrn_div_stash_bytes(int n_rays, int n_samples);
size_t nrn_div_grad_stash_bytes(int n_rays, int n_samples);
typedef struct NrnDivArgs {
  int32_t n_rays, n_samples;
  const void* stash;               /* activation stash of the coarse nrn_field_forward call */
  const float* e;                  /* [P][3] probe vectors ~ N(0, I) (torch.randn_like, run_nerf_helpers.py:110) */
  const float* unmasked_offsets;   /* [P][3] coarse pass output */
  const float* rigidity_mask;      /* [P]    coarse pass output */
  const float* weights;            /* [P]    1 - exp(-relu(opacity_alpha)), detached (train.py:267) ... */
  int32_t weights_are_opacity_alpha; /* ... or, if 1, opacity_alpha itself: the kernels apply 1 - exp(-relu(.)) */
  const float* const* net_w;       /* 5: ray_bending.network.i.weight (fp32, reference layout) */
  const float* const* rig_w;       /* 3: ray_bending.rigidity_network.i.weight */
  void* tangent_stash;             /* nrn_div_stash_bytes(): written by forward, read by backward */
  float* d; float* alpha; float* beta; float* tau_c;   /* [P] each: written by forward, read by backward */
  float* loss;                     /* forward out [n_rays]: mean over the ray's samples of weights * d^2 */
  /* backward only */
  const float* G;                  /* [P] dL/dd = g_ray * 2 * weights * d / n_samples, or NULL with g_ray / G_workspace: */
  const float* g_ray;              /* [n_rays] upstream gradient of `loss`; G is then computed into G_workspace [P] */
  float* G_workspace;
  void* adjoint_stash;             /* workspace, nrn_div_grad_stash_bytes() */
  float* wgrad_scratch;            /* workspace, nrn_wgrad_scratch_bytes() */
  float* d_unmasked_offsets;       /* out [P][3] gradient w.r.t. the coarse unmasked offsets */
  float* d_rigidity_mask;          /* out [P]    gradient w.r.t. the coarse rigidity mask */
  float* bender_grad;              /* out, nrn_bender_grad_floats(): weight gradients of the tangent chain */
  void* stream;
  int32_t accumulate_bender;       /* != 0: add to bender_grad instead of overwriting it */
} NrnDivArgs;
int nrn_divergence_forward(const NrnDivArgs* args);
int nrn_divergence_backward(const NrnDivArgs* args);

/* ---- per-ray training loss of training_wrapper_class.forward (train.py:208-242): image terms (fine +
 * coarse) and the offsets / rigidity regulariser on the coarse samples, with the gradients per unit
 * upstream gradient written in the same pass (the loss is linear in dL/dloss[ray]). ----------------- */
typedef struct NrnRayLossArgs {
  int32_t n_rays, n_samples;
  const float* rgb;                /* [n][3] rgb_map */
  const float* rgb0;               /* [n][3] coarse rgb_map or NULL */
  const float* target;             /* [n][3] */
  const float* weights;            /* [n][S] coarse visibility weights (detached) or NULL */
  const float* unmasked_offsets;   /* [n][S][3] or NULL: no offsets term */
  const float* rigidity_mask;      /* [n][S] */
  float lam_offsets;               /* offsets_loss_weight (times the schedule, unless sched_step is given) */
  float lam_rigidity;              /* rigidity_loss_weight */
  float* loss;                     /* out [n] */
  float* u_rgb; float* u_rgb0;     /* out [n][3]: d loss / d rgb, d loss / d rgb0 */
  float* u_unmasked_offsets;       /* out [n][S][3] */
  float* u_rigidity_mask;          /* out [n][S] */
  void* stream;
  /* Regulariser schedule (1/100)^(1 - global_step / N_iters) of train.py:229 / :281 evaluated on the device: sched_step is a
   * device scalar holding global_step (NULL: the caller folded the schedule into the weights), so that a captured CUDA graph
   * follows the schedule.  divergence [n] (or NULL) is the per-ray divergence regulariser (nrn_divergence_forward), added as
   * lam_divergence * schedule * divergence; u_divergence [n] receives d loss / d divergence. */
  const float* sched_step;
  float sched_n_iters;
  const float* divergence;
  float lam_divergence;
  float* u_divergence;
} NrnRayLossArgs;
int nrn_ray_loss(const NrnRayLossArgs* args);
/* out[i] = g[i / per_row] * unit[i] */
int nrn_scale_rows(const float* g, const float* unit, float* out, int64_t n, int per_row, void* stream);
/* Backward of nrn_ray_loss in ONE launch: every out_k[i] = g[ray of i] * unit_k[i] for the (up to five) unit-gradient arrays
 * nrn_ray_loss wrote (NULL pairs are skipped): rgb [n][3], rgb0 [n][3], unmasked_offsets [n][S][3], rigidity_mask [n][S],
 * divergence [n]. */
typedef struct NrnRayLossBwdArgs {
  int32_t n_rays, n_samples;
  const float* g;                  /* [n] upstream gradient of the per-ray loss */
  const float* u_rgb; const float* u_rgb0; const float* u_unmasked_offsets; const float* u_rigidity_mask; const float* u_divergence;
  float* d_rgb; float* d_rgb0; float* d_unmasked_offsets; float* d_rigidity_mask; float* d_divergence;
  void* stream;
} NrnRayLossBwdArgs;
int nrn_ray_loss_backward(const NrnRayLossBwdArgs* args);

/* ---- optimizer step: replaces torch.optim.Adam(params=grad_vars, lr, betas=(0.9, 0.999)) of train.py:656-658 and its
 * optimizer.step() at train.py:1608.  All trainable tensors live in one flat fp32 buffer (the host side makes the
 * nn.Parameters views into it); `blocks` (device, int32 x 4 per entry: tensor index, first element inside the tensor,
 * element count <= 2048, offset inside the flat buffers) maps CUDA blocks to tensors; `grad_ptrs` (device, one
 * const float* per tensor, NULL = parameter without gradient, skipped like torch does) is where autograd left each
 * gradient.  lr (scalar) and step (one int64 per tensor, as torch counts steps per parameter) live on the device
 * (CUDA-graph replay); the call increments the step of every tensor that has a gradient, then applies
 * m += (g-m)(1-b1); v = b2 v + (1-b2) g^2; p -= lr/(1-b1^t) m / (sqrt(v)/sqrt(1-b2^t) + eps). */
typedef struct NrnAdamArgs {
  void* params;            /* float [total] */
  void* exp_avg;           /* float [total] */
  void* exp_avg_sq;        /* float [total] */
  const void* grad_ptrs;   /* device array of n_tensors pointers */
  const void* blocks;      /* device array of n_blocks x 4 int32 */
  int n_tensors, n_blocks;
  const void* lr;          /* device float */
  void* step;              /* device int64 [n_tensors] */
  float beta1, beta2, eps;
  void* stream;
} NrnAdamArgs;
int nrn_adam_step(const NrnAdamArgs* args);

/* ---- multi-GPU: gradient all-reduce fused into the optimizer step over NVLink peer memory.  Replaces the gradient
 * reduction torch.nn.DataParallel performs on GPU 0 (train.py:290-297; backward of the scatter at :1566-1577) plus the
 * optimizer.step() at :1608, for one process per GPU on one node.  Every rank allocates a window
 *   [ 1024 B flags | 2 x slot_floats floats (double-buffered row slots) | arena_floats floats (gradient arena) ]
 * with nrn_peer_alloc, publishes its 64-byte CUDA IPC handle to the other ranks (any side channel: the host side uses
 * torch.distributed.all_gather_object), maps theirs with nrn_peer_open, and points every parameter's .grad into its own
 * window's arena.  nrn_peer_reduce_adam then sums the ranks' arenas in rank order while reading them over NVLink and applies
 * Adam (same arithmetic as nrn_adam_step; grad_ptrs is ignored, gradients come from the arenas at the blocks' flat
 * offsets); afterwards the arena holds the reduced gradient.  nrn_peer_gather_rows all-gathers n_per_rank floats per rank
 * (the per-ray losses the caller logs) through the slots.  All launches are plain kernels on `stream` (CUDA-graph
 * capturable); a peer that never arrives becomes device error 901/902/903 (nrn_device_error), not a hang. */
size_t nrn_peer_window_bytes(int64_t arena_floats, int64_t slot_floats);
int nrn_peer_alloc(size_t bytes, void** dev_ptr, void* ipc_handle_64bytes);
int nrn_peer_open(const void* ipc_handle_64bytes, void** dev_ptr);
int nrn_peer_close(void* dev_ptr);
int nrn_peer_free(void* dev_ptr);
typedef struct NrnPeerCtx {
  void* window[8];          /* all ranks' windows as mapped into this process; window[rank] = own allocation */
  int32_t world, rank;
  int64_t arena_floats, slot_floats;
  void* state;              /* device, 16 bytes, zero-initialised once: 3 epoch counters + block counter */
  float* reduced;           /* device workspace, arena_floats floats */
} NrnPeerCtx;
int nrn_peer_reduce_adam(const NrnPeerCtx* ctx, const NrnAdamArgs* adam);
int nrn_peer_gather_rows(const NrnPeerCtx* ctx, const float* local, int n_per_rank, float* out, void* stream);

/* ---- optional per-kernel timing (measurement aid for bench.py) ---------------------------------
 * While enabled, every launch of the kernel kinds below is bracketed by CUDA events recorded on the
 * launch stream.  kinds: 0 field forward, 1 field DGRAD, 2 WGRAD (+reduce), 3 composite(+resample),
 * 4 composite backward, 5 divergence regulariser.  nrn_timing_read synchronises the recorded events and returns per-kind sums.
 * The events live until the process ends, so a graph captured while timing was on may be replayed after it is turned off. */
int nrn_timing_enable(int on);
int nrn_timing_read(double* ms_sum, int* counts, int n_kinds);

#ifdef __cplusplus
}
#endif
#endif /* NRNERF_B200_H */
