// extern "C" boundary of libnrnerf_b200.so (declarations: include/nrnerf_b200.h).
// Argument validation, launch, error reporting.  No exceptions cross this file.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include "../../include/nrnerf_b200.h"
#include "nrn_common.cuh"
#include "pack.cuh"
#include "ray_ops.cuh"
#include "wgrad.cuh"
#include "div.cuh"
#include "loss.cuh"
#include "adam.cuh"
#include "peer.cuh"

namespace nrn {
cudaError_t launch_field_fwd(const FieldFwdParams& p, bool has_bender, int num_sms, cudaStream_t stream);
cudaError_t launch_field_bwd(const FieldBwdParams& p, bool has_bender, int num_sms, cudaStream_t stream);
}

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  return fail(NRN_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

constexpr int kMaxDevices = 64;
struct DeviceState {
  int* err_word = nullptr;   // [0] error word, [1] loss-scale source (float) of the running backward
  int num_sms = 0;
};
DeviceState g_dev[kMaxDevices];

int device_state(DeviceState** out) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  if (dev < 0 || dev >= kMaxDevices) return fail(NRN_E_INVALID, "device index %d out of range", dev);
  DeviceState& s = g_dev[dev];
  if (!s.err_word) {
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
    if (prop.major != 10) return fail(NRN_E_INVALID, "nrnerf_b200 needs an sm_100 GPU, found sm_%d%d", prop.major, prop.minor);
    s.num_sms = prop.multiProcessorCount;
    if (const char* g = getenv("NRN_GRID")) { const int v = atoi(g); if (v > 0 && v < s.num_sms) s.num_sms = v; }   // developer experiments
    e = cudaMalloc(&s.err_word, 4 * sizeof(int));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(err word)");
    e = cudaMemset(s.err_word, 0, 4 * sizeof(int));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemset(err word)");
  }
  *out = &s;
  return NRN_OK;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- optional per-kernel timing: CUDA events recorded on the launch stream around each kernel ----
struct TimedLaunch {
  cudaEvent_t a, b;
  int kind;
};
bool g_timing = false;
TimedLaunch g_timed[4096];
int g_timed_n = 0;
struct ScopedTimer {
  int idx = -1;
  cudaStream_t st;
  ScopedTimer(int kind, cudaStream_t s) : st(s) {
    if (!g_timing || g_timed_n >= 4096) return;
    TimedLaunch& t = g_timed[g_timed_n];
    if ((!t.a && cudaEventCreate(&t.a) != cudaSuccess) || (!t.b && cudaEventCreate(&t.b) != cudaSuccess)) return;
    t.kind = kind;
    idx = g_timed_n++;
    record(t.a);
  }
  ~ScopedTimer() {
    if (idx >= 0) record(g_timed[idx].b);
  }
  // inside a CUDA-graph capture the records become external event-record nodes: every replay of the graph
  // re-stamps them, and the elapsed time of the last replay can be read afterwards
  void record(cudaEvent_t ev) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cs);
    cudaEventRecordWithFlags(ev, st, cs == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault);
  }
};

}  // namespace

extern "C" {

int nrn_abi_version(void) { return NRN_ABI_VERSION; }
const char* nrn_last_error(void) { return g_err; }

int nrn_device_error(int* code_out) {
  DeviceState* ds;
  int rc = device_state(&ds);
  if (rc) return rc;
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceSynchronize");
  int code = 0;
  e = cudaMemcpy(&code, ds->err_word, sizeof(int), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(err word)");
  if (code) cudaMemset(ds->err_word, 0, sizeof(int));
  if (code_out) *code_out = code;
  if (code) return fail(NRN_E_DEVICE, "device-side protocol error: wait id %d timed out", code);
  return NRN_OK;
}

size_t nrn_packed_nerf_bytes(void) { return nrn::kNerfPackedBytes; }
size_t nrn_packed_bender_bytes(void) { return nrn::kBendPackedBytes; }

int nrn_pack_nerf(const float* const* w, const float* const* b, int input_ch, int out_ch, void* packed, void* stream) {
  if (!w || !b || !packed) return fail(NRN_E_INVALID, "nrn_pack_nerf: null argument");
  if (input_ch < 1 || input_ch > 63) return fail(NRN_E_INVALID, "nrn_pack_nerf: input_ch=%d unsupported (1..63; multires=10 gives 63)", input_ch);
  if (out_ch < 4 || out_ch > 16) return fail(NRN_E_INVALID, "nrn_pack_nerf: out_ch=%d unsupported", out_ch);
  if (!aligned16(packed)) return fail(NRN_E_INVALID, "nrn_pack_nerf: packed buffer must be 16-byte aligned");
  nrn::NerfSrc src;
  for (int i = 0; i < 9; ++i) {
    if (!w[i] || !b[i]) return fail(NRN_E_INVALID, "nrn_pack_nerf: null layer %d", i);
    src.w[i] = w[i];
    src.b[i] = b[i];
  }
  cudaError_t e = nrn::launch_pack_nerf(src, input_ch, out_ch, packed, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "pack_nerf_kernel");
}

int nrn_pack_bender(const float* const* net_w, const float* const* net_b, const float* const* rig_w,
                    const float* const* rig_b, int latent_size, void* packed, void* stream) {
  if (!net_w || !net_b || !rig_w || !rig_b || !packed) return fail(NRN_E_INVALID, "nrn_pack_bender: null argument");
  if (latent_size != nrn::kLatent) return fail(NRN_E_INVALID, "nrn_pack_bender: ray_bending_latent_size=%d unsupported (32)", latent_size);
  if (!aligned16(packed)) return fail(NRN_E_INVALID, "nrn_pack_bender: packed buffer must be 16-byte aligned");
  nrn::BenderSrc src;
  for (int i = 0; i < 5; ++i) src.net_w[i] = net_w[i];
  for (int i = 0; i < 4; ++i) src.net_b[i] = net_b[i];
  for (int i = 0; i < 3; ++i) { src.rig_w[i] = rig_w[i]; src.rig_b[i] = rig_b[i]; }
  cudaError_t e = nrn::launch_pack_bender(src, packed, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "pack_bender_kernel");
}

int nrn_sample_coarse(const float* rays, const float* t_rand, int n_rays, int n_samples, int lindisp, float* z_vals,
                      void* stream) {
  if (n_rays < 0 || n_samples < 1) return fail(NRN_E_INVALID, "nrn_sample_coarse: bad sizes n=%d S=%d", n_rays, n_samples);
  if (n_rays == 0) return NRN_OK;
  if (!rays || !z_vals) return fail(NRN_E_INVALID, "nrn_sample_coarse: null argument");
  cudaError_t e = nrn::launch_sample_coarse(rays, t_rand, n_rays, n_samples, lindisp, z_vals, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "sample_coarse_kernel");
}

int nrn_get_rays(const float* c2w, const float* K, int H, int W, float* rays_o, float* rays_d, void* stream) {
  if (H < 0 || W < 0) return fail(NRN_E_INVALID, "nrn_get_rays: bad sizes");
  if (H == 0 || W == 0) return NRN_OK;
  if (!c2w || !K || !rays_o || !rays_d) return fail(NRN_E_INVALID, "nrn_get_rays: null argument");
  const cudaError_t e = nrn::launch_get_rays(c2w, K, H, W, rays_o, rays_d, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "get_rays_kernel");
}

int nrn_pack_rays(const float* rays_o, const float* rays_d, float near, float far, int n_rays, float* rays, void* stream) {
  if (n_rays < 0) return fail(NRN_E_INVALID, "nrn_pack_rays: bad size");
  if (n_rays == 0) return NRN_OK;
  if (!rays_o || !rays_d || !rays) return fail(NRN_E_INVALID, "nrn_pack_rays: null argument");
  const cudaError_t e = nrn::launch_pack_rays(rays_o, rays_d, near, far, n_rays, rays, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "pack_rays_kernel");
}

int nrn_ray_batch(const int64_t* pix, int n, const float* poses, const float* K, const int32_t* image_to_view, const float* images,
                  int H, int W, float* rays_o, float* rays_d, float* target, void* stream) {
  if (n < 0 || H < 1 || W < 1) return fail(NRN_E_INVALID, "nrn_ray_batch: bad sizes");
  if (n == 0) return NRN_OK;
  if (!pix || !poses || !K || !rays_o || !rays_d || (images && !target)) return fail(NRN_E_INVALID, "nrn_ray_batch: null argument");
  static_assert(sizeof(long long) == sizeof(int64_t), "int64");
  const cudaError_t e = nrn::launch_ray_batch(reinterpret_cast<const long long*>(pix), n, poses, K, image_to_view, images, H, W, rays_o, rays_d,
                                              target, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "ray_batch_kernel");
}

int nrn_median_visibility_index(const float* weights, int n_rays, int n_samples, int64_t* index, void* stream) {
  if (n_rays < 0 || n_samples < 1) return fail(NRN_E_INVALID, "nrn_median_visibility_index: bad sizes");
  if (n_rays == 0) return NRN_OK;
  if (!weights || !index) return fail(NRN_E_INVALID, "nrn_median_visibility_index: null argument");
  const cudaError_t e = nrn::launch_median_index(weights, n_rays, n_samples, reinterpret_cast<long long*>(index), static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "median_index_kernel");
}

int nrn_field_forward(const NrnFieldArgs* a) {
  if (!a) return fail(NRN_E_INVALID, "nrn_field_forward: null args");
  if (a->n_rays < 0 || a->n_samples < 1) return fail(NRN_E_INVALID, "nrn_field_forward: bad sizes n=%d S=%d", a->n_rays, a->n_samples);
  if (a->n_rays == 0) return NRN_OK;
  if (!a->nerf_packed || !a->raw) return fail(NRN_E_INVALID, "nrn_field_forward: null argument");
  if (a->points) {
    if (a->n_samples != 1 || a->points_stride < 3) return fail(NRN_E_INVALID, "nrn_field_forward: point mode needs n_samples=1, stride>=3");
  } else if (!a->rays || !a->z_vals) {
    return fail(NRN_E_INVALID, "nrn_field_forward: null rays / z_vals");
  }
  if (a->bender_packed && !a->latents) return fail(NRN_E_INVALID, "nrn_field_forward: bender given without latents");
  if (a->out_ch < 4 || a->out_ch > 5) return fail(NRN_E_INVALID, "nrn_field_forward: out_ch=%d unsupported (4 or 5)", a->out_ch);
  if (!aligned16(a->nerf_packed) || (a->bender_packed && !aligned16(a->bender_packed)))
    return fail(NRN_E_INVALID, "nrn_field_forward: packed weights must be 16-byte aligned");
  DeviceState* ds;
  int rc = device_state(&ds);
  if (rc) return rc;
  nrn::FieldFwdParams p{};
  p.rays = a->rays; p.z_vals = a->z_vals; p.pts = a->points; p.pts_stride = a->points_stride; p.latents = a->latents; p.latent_stride = a->latent_stride;
  p.n_rays = a->n_rays; p.S = a->n_samples;
  p.P = static_cast<long long>(a->n_rays) * a->n_samples;
  const long long tiles = (p.P + nrn::kTileM - 1) / nrn::kTileM;
  if (tiles > 0x7fffffffLL) return fail(NRN_E_INVALID, "nrn_field_forward: too many points");
  p.n_tiles = static_cast<int>(tiles);
  const uint8_t* np = static_cast<const uint8_t*>(a->nerf_packed);
  p.nerf_w = np; p.nerf_bias = reinterpret_cast<const float*>(np + nrn::kNerfWBytes);
  if (a->bender_packed) {
    const uint8_t* bp = static_cast<const uint8_t*>(a->bender_packed);
    p.bend_w = bp; p.bend_bias = reinterpret_cast<const float*>(bp + nrn::kBendWBytes);
  }
  p.cutoff = a->rigidity_cutoff; p.use_cutoff = a->use_cutoff;
  p.scaling = a->scaling; p.use_scaling = a->use_scaling;
  p.removal = a->removal_threshold; p.use_removal = a->use_removal;
  p.out_ch = a->out_ch;
  p.raw = a->raw; p.d_init = a->initial_input_pts; p.d_bent = a->input_pts; p.d_unmasked = a->unmasked_offsets;
  p.d_masked = a->masked_offsets; p.d_rigid = a->rigidity_mask;
  p.stash = static_cast<uint8_t*>(a->stash);
  { const char* dm = getenv("NRN_DEBUG_MODE"); p.debug_mode = dm ? atoi(dm) : 0; }
  if (a->stash && a->points) return fail(NRN_E_INVALID, "nrn_field_forward: the training stash needs ray mode");
  p.err = ds->err_word;
  cudaError_t e;
  {
    ScopedTimer tm(0, static_cast<cudaStream_t>(a->stream));
    e = nrn::launch_field_fwd(p, a->bender_packed != nullptr, ds->num_sms, static_cast<cudaStream_t>(a->stream));
  }
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "field_fwd_kernel");
}

int nrn_composite(const NrnCompositeArgs* a) {
  if (!a) return fail(NRN_E_INVALID, "nrn_composite: null args");
  if (a->n_rays < 0 || a->n_samples < 1 || a->channels < 4) return fail(NRN_E_INVALID, "nrn_composite: bad sizes");
  if (a->n_rays == 0) return NRN_OK;
  if (!a->raw || !a->z_vals || !a->rays_d || !a->rgb_map || !a->disp_map || !a->acc_map) return fail(NRN_E_INVALID, "nrn_composite: null argument");
  if (a->n_importance < 0) return fail(NRN_E_INVALID, "nrn_composite: n_importance < 0");
  if (a->n_importance > 0 && (!a->z_vals_out || a->n_samples < 3)) return fail(NRN_E_INVALID, "nrn_composite: resampling needs z_vals_out and >= 3 samples");
  if (4 * a->n_samples + a->n_importance > 12000) return fail(NRN_E_INVALID, "nrn_composite: too many samples per ray");
  nrn::CompositeParams p{};
  p.raw = a->raw; p.z = a->z_vals; p.rays_d = a->rays_d; p.rays_d_stride = a->rays_d_stride; p.noise = a->noise;
  p.n = a->n_rays; p.S = a->n_samples; p.C = a->channels; p.white_bkgd = a->white_bkgd;
  p.rgb = a->rgb_map; p.disp = a->disp_map; p.acc = a->acc_map; p.depth = a->depth_map; p.weights = a->weights; p.alpha = a->alpha;
  p.n_imp = a->n_importance; p.u = a->u; p.z_out = a->z_vals_out; p.z_std = a->z_std;
  cudaError_t e; { ScopedTimer tm(3, static_cast<cudaStream_t>(a->stream)); e = nrn::launch_composite(p, static_cast<cudaStream_t>(a->stream)); }
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "composite_kernel");
}

int nrn_sample_pdf(const float* bins, const float* weights, const float* u, int n, int nbins, int n_samples, float* samples,
                   void* stream) {
  if (n < 0 || nbins < 2 || n_samples < 1 || nbins > 4000) return fail(NRN_E_INVALID, "nrn_sample_pdf: bad sizes");
  if (n == 0) return NRN_OK;
  if (!bins || !weights || !samples) return fail(NRN_E_INVALID, "nrn_sample_pdf: null argument");
  cudaError_t e = nrn::launch_sample_pdf(bins, weights, u, n, nbins, n_samples, samples, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "sample_pdf_kernel");
}

int nrn_composite_backward(const NrnCompositeBwdArgs* a) {
  if (!a) return fail(NRN_E_INVALID, "nrn_composite_backward: null args");
  if (a->n_rays < 0 || a->n_samples < 1 || a->channels < 4 || a->n_samples > 12000) return fail(NRN_E_INVALID, "nrn_composite_backward: bad sizes");
  if (a->n_rays == 0) return NRN_OK;
  if (!a->raw || !a->z_vals || !a->rays_d || !a->d_rgb_map || !a->d_raw) return fail(NRN_E_INVALID, "nrn_composite_backward: null argument");
  nrn::CompositeBwdParams p{};
  p.raw = a->raw; p.z = a->z_vals; p.rays_d = a->rays_d; p.rays_d_stride = a->rays_d_stride; p.noise = a->noise;
  p.n = a->n_rays; p.S = a->n_samples; p.C = a->channels; p.white_bkgd = a->white_bkgd;
  p.d_rgb = a->d_rgb_map; p.d_acc = a->d_acc_map; p.d_raw = a->d_raw;
  cudaError_t e; { ScopedTimer tm(4, static_cast<cudaStream_t>(a->stream)); e = nrn::launch_composite_bwd(p, static_cast<cudaStream_t>(a->stream)); }
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "composite_bwd_kernel");
}

static long long even_tiles(int n_rays, int n_samples) {
  const long long P = static_cast<long long>(n_rays) * n_samples;
  const long long tiles = (P + nrn::kTileM - 1) / nrn::kTileM;
  return (tiles + 1) & ~1LL;   // the kernels work on tile pairs (two slots per CTA)
}
size_t nrn_stash_bytes(int n_rays, int n_samples) { return static_cast<size_t>(even_tiles(n_rays, n_samples)) * nrn::kStashTileBytes; }
size_t nrn_grad_stash_bytes(int n_rays, int n_samples) { return static_cast<size_t>(even_tiles(n_rays, n_samples)) * nrn::kGradTileBytes; }
size_t nrn_wgrad_scratch_bytes(void) { return static_cast<size_t>(nrn::kWgMaxCtas) * nrn::kWgScratchFloats * sizeof(float); }
int nrn_nerf_grad_floats(int out_ch) { return 256 * 63 + 256 + 6 * (65536 + 256) + 256 * 319 + 256 + out_ch * 257; }
int nrn_bender_grad_floats(void) { return 16193; }

int nrn_field_backward(const NrnFieldBwdArgs* a) {
  if (!a) return fail(NRN_E_INVALID, "nrn_field_backward: null args");
  if (a->n_rays < 0 || a->n_samples < 1) return fail(NRN_E_INVALID, "nrn_field_backward: bad sizes");
  if (a->out_ch < 4 || a->out_ch > 5) return fail(NRN_E_INVALID, "nrn_field_backward: out_ch=%d unsupported", a->out_ch);
  if (!a->nerf_packed || !a->nerf_grad) return fail(NRN_E_INVALID, "nrn_field_backward: null argument");
  const bool bend = a->bender_packed != nullptr;
  if (bend && (!a->unmasked_offsets || !a->rigidity_mask || !a->bender_grad || !a->d_latents))
    return fail(NRN_E_INVALID, "nrn_field_backward: bender needs unmasked_offsets, rigidity_mask, bender_grad, d_latents");
  DeviceState* ds;
  int rc = device_state(&ds);
  if (rc) return rc;
  if (ds->num_sms + 16 > nrn::kWgMaxCtas) return fail(NRN_E_INVALID, "nrn_field_backward: %d SMs exceed the scratch layout", ds->num_sms);
  cudaStream_t st = static_cast<cudaStream_t>(a->stream);
  const int nerf_n = nrn_nerf_grad_floats(a->out_ch);
  const int bend_n = bend ? nrn_bender_grad_floats() : 0;
  cudaError_t e;
  if (bend) {
    e = cudaMemsetAsync(a->d_latents, 0, sizeof(float) * static_cast<size_t>(a->n_rays) * nrn::kLatent, st);
    if (e != cudaSuccess) return cuda_fail(e, "memset d_latents");
  }
  if (a->n_rays == 0) {   // an empty shard contributes zero gradients
    e = cudaSuccess;
    if (!a->accumulate_nerf) {
      const int head_n = a->nerf_grad_head ? a->out_ch * 257 : 0;
      e = cudaMemsetAsync(a->nerf_grad, 0, sizeof(float) * (nerf_n - head_n), st);
      if (e == cudaSuccess && head_n) e = cudaMemsetAsync(a->nerf_grad_head, 0, sizeof(float) * head_n, st);
    }
    if (e == cudaSuccess && bend && !a->accumulate_bender) e = cudaMemsetAsync(a->bender_grad, 0, sizeof(float) * bend_n, st);
    return e == cudaSuccess ? NRN_OK : cuda_fail(e, "memset grads");
  }
  if (!a->d_raw || !a->stash || !a->grad_stash || !a->wgrad_scratch) return fail(NRN_E_INVALID, "nrn_field_backward: null argument");
  float* amax = reinterpret_cast<float*>(ds->err_word + 1);
  nrn::FieldBwdParams p{};
  p.P = static_cast<long long>(a->n_rays) * a->n_samples;
  p.n_tiles = static_cast<int>((p.P + nrn::kTileM - 1) / nrn::kTileM);
  p.S = a->n_samples; p.n_rays = a->n_rays; p.out_ch = a->out_ch;
  p.d_raw = a->d_raw; p.amax = amax;
  p.stash = static_cast<const uint8_t*>(a->stash); p.gstash = static_cast<uint8_t*>(a->grad_stash);
  p.nerf_wT = static_cast<const uint8_t*>(a->nerf_packed) + nrn::kNerfTOffset;
  if (bend) p.bend_wT = static_cast<const uint8_t*>(a->bender_packed) + nrn::kBendTOffset;
  p.unmasked = a->unmasked_offsets; p.rigidity = a->rigidity_mask;
  p.d_unmasked_up = a->d_unmasked_offsets; p.d_rigid_up = a->d_rigidity_mask;
  p.cutoff = a->rigidity_cutoff; p.use_cutoff = a->use_cutoff; p.scaling = a->scaling; p.use_scaling = a->use_scaling;
  p.d_latents = a->d_latents; p.err = ds->err_word;
  e = nrn::launch_absmax(a->d_raw, p.P * a->out_ch, amax, st);
  // the regularisers' upstream gradients share the fp16 loss scale: they take part in the maximum, otherwise a large
  // offsets_loss_weight saturates them (or, with a vanishing data term, lets them underflow)
  if (e == cudaSuccess && bend && p.d_unmasked_up) e = nrn::launch_absmax(p.d_unmasked_up, p.P * 3, amax, st, true);
  if (e == cudaSuccess && bend && p.d_rigid_up) e = nrn::launch_absmax(p.d_rigid_up, p.P, amax, st, true);
  if (e != cudaSuccess) return cuda_fail(e, "absmax_kernel");
  { ScopedTimer tm(1, st); e = nrn::launch_field_bwd(p, bend, ds->num_sms, st); }
  if (e != cudaSuccess) return cuda_fail(e, "field_bwd_kernel");
  nrn::WgradParams w{};
  w.stash = p.stash; w.gstash = p.gstash; w.scratch = a->wgrad_scratch; w.amax = amax; w.n_tiles = p.n_tiles; w.err = ds->err_word;
  const nrn::WgradDst dst{a->nerf_grad, a->nerf_grad_head, a->bender_grad, nerf_n, bend_n, a->accumulate_nerf, a->accumulate_bender};
  { ScopedTimer tm(2, st); e = nrn::launch_wgrad(w, bend, ds->num_sms, dst, a->out_ch, st); }
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "wgrad_kernel");
}

static long long point_tiles(int n_rays, int n_samples) {
  return (static_cast<long long>(n_rays) * n_samples + nrn::kTileM - 1) / nrn::kTileM;
}
size_t nrn_div_stash_bytes(int n_rays, int n_samples) { return static_cast<size_t>(point_tiles(n_rays, n_samples)) * nrn::kTanTileBytes; }
size_t nrn_div_grad_stash_bytes(int n_rays, int n_samples) { return static_cast<size_t>(point_tiles(n_rays, n_samples)) * nrn::kAdjTileBytes; }

static int fill_div(const NrnDivArgs* a, nrn::DivParams& p, const char* who) {
  if (!a) return fail(NRN_E_INVALID, "%s: null args", who);
  if (a->n_rays < 0 || a->n_samples < 1) return fail(NRN_E_INVALID, "%s: bad sizes", who);
  if (!a->stash || !a->e || !a->unmasked_offsets || !a->rigidity_mask || !a->weights || !a->net_w || !a->rig_w || !a->tangent_stash ||
      !a->d || !a->alpha || !a->beta || !a->tau_c)
    return fail(NRN_E_INVALID, "%s: null argument", who);
  p.P = static_cast<long long>(a->n_rays) * a->n_samples;
  p.S = a->n_samples; p.n_rays = a->n_rays;
  p.stash = static_cast<const uint8_t*>(a->stash);
  p.e = a->e; p.unmasked = a->unmasked_offsets; p.rigidity = a->rigidity_mask; p.w = a->weights; p.w_is_alpha = a->weights_are_opacity_alpha != 0;
  for (int i = 0; i < 5; ++i) { if (!a->net_w[i]) return fail(NRN_E_INVALID, "%s: null weight", who); p.net_w[i] = a->net_w[i]; }
  for (int i = 0; i < 3; ++i) { if (!a->rig_w[i]) return fail(NRN_E_INVALID, "%s: null weight", who); p.rig_w[i] = a->rig_w[i]; }
  p.tan = static_cast<uint8_t*>(a->tangent_stash);
  p.d = a->d; p.adot = a->alpha; p.beta = a->beta; p.tauc = a->tau_c;
  return NRN_OK;
}

int nrn_divergence_forward(const NrnDivArgs* a) {
  nrn::DivParams p{};
  int rc = fill_div(a, p, "nrn_divergence_forward");
  if (rc) return rc;
  if (!a->loss) return fail(NRN_E_INVALID, "nrn_divergence_forward: null loss");
  cudaStream_t st = static_cast<cudaStream_t>(a->stream);
  cudaError_t e = cudaMemsetAsync(a->loss, 0, sizeof(float) * static_cast<size_t>(a->n_rays), st);
  if (e != cudaSuccess) return cuda_fail(e, "memset loss");
  p.loss = a->loss;
  { ScopedTimer tm(5, st); e = nrn::launch_div_fwd(p, st); }
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "div_fwd_kernel");
}

int nrn_divergence_backward(const NrnDivArgs* a) {
  nrn::DivParams p{};
  int rc = fill_div(a, p, "nrn_divergence_backward");
  if (rc) return rc;
  if ((!a->G && !(a->g_ray && a->G_workspace)) || !a->adjoint_stash || !a->wgrad_scratch || !a->d_unmasked_offsets || !a->d_rigidity_mask ||
      !a->bender_grad)
    return fail(NRN_E_INVALID, "nrn_divergence_backward: null argument");
  DeviceState* ds;
  rc = device_state(&ds);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(a->stream);
  float* amax = reinterpret_cast<float*>(ds->err_word + 2);
  p.G = a->G ? a->G : a->G_workspace; p.amax = amax; p.adj = static_cast<uint8_t*>(a->adjoint_stash);
  p.d_unmasked = a->d_unmasked_offsets; p.d_rigid = a->d_rigidity_mask;
  cudaError_t e = a->G ? nrn::launch_absmax(a->G, p.P, amax, st) : nrn::launch_div_G(p, a->g_ray, a->G_workspace, amax, st);
  if (e != cudaSuccess) return cuda_fail(e, "absmax_kernel");
  { ScopedTimer tm(5, st); e = nrn::launch_div_bwd(p, st); }
  if (e != cudaSuccess) return cuda_fail(e, "div_bwd_kernel");
  nrn::WgradParams w{};
  w.stash = p.tan; w.gstash = p.adj; w.scratch = a->wgrad_scratch; w.amax = amax; w.compact = 1;
  w.n_tiles = static_cast<int>((p.P + nrn::kTileM - 1) / nrn::kTileM); w.err = ds->err_word;
  const nrn::WgradDst dst{nullptr, nullptr, a->bender_grad, 0, nrn_bender_grad_floats(), 0, a->accumulate_bender};
  { ScopedTimer tm(2, st); e = nrn::launch_wgrad(w, true, ds->num_sms, dst, 5, st); }
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "wgrad_kernel (divergence)");
}

int nrn_ray_loss(const NrnRayLossArgs* a) {
  if (!a) return fail(NRN_E_INVALID, "nrn_ray_loss: null args");
  if (a->n_rays < 0 || a->n_samples < 1) return fail(NRN_E_INVALID, "nrn_ray_loss: bad sizes");
  if (a->n_rays == 0) return NRN_OK;
  if (!a->rgb || !a->target || !a->loss || !a->u_rgb || (a->rgb0 && !a->u_rgb0)) return fail(NRN_E_INVALID, "nrn_ray_loss: null argument");
  if (a->unmasked_offsets && (!a->weights || !a->rigidity_mask || !a->u_unmasked_offsets || !a->u_rigidity_mask))
    return fail(NRN_E_INVALID, "nrn_ray_loss: the offsets term needs weights, rigidity_mask and both gradient outputs");
  if (a->divergence && !a->u_divergence) return fail(NRN_E_INVALID, "nrn_ray_loss: the divergence term needs u_divergence");
  if (a->sched_step && !(a->sched_n_iters > 0.f)) return fail(NRN_E_INVALID, "nrn_ray_loss: sched_n_iters must be positive");
  nrn::RayLossParams p{};
  p.n = a->n_rays; p.S = a->n_samples;
  p.rgb = a->rgb; p.rgb0 = a->rgb0; p.target = a->target; p.w = a->weights; p.off = a->unmasked_offsets; p.rig = a->rigidity_mask;
  p.lam_o = a->lam_offsets; p.lam_r = a->lam_rigidity;
  p.sched_step = a->sched_step; p.sched_n_iters = a->sched_n_iters; p.div = a->divergence; p.lam_div = a->lam_divergence; p.u_div = a->u_divergence;
  p.loss = a->loss; p.u_rgb = a->u_rgb; p.u_rgb0 = a->u_rgb0; p.u_off = a->u_unmasked_offsets; p.u_rig = a->u_rigidity_mask;
  cudaError_t e = nrn::launch_ray_loss(p, static_cast<cudaStream_t>(a->stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "ray_loss_kernel");
}

int nrn_ray_loss_backward(const NrnRayLossBwdArgs* a) {
  if (!a) return fail(NRN_E_INVALID, "nrn_ray_loss_backward: null args");
  if (a->n_rays < 0 || a->n_samples < 1) return fail(NRN_E_INVALID, "nrn_ray_loss_backward: bad sizes");
  if (a->n_rays == 0) return NRN_OK;
  if (!a->g) return fail(NRN_E_INVALID, "nrn_ray_loss_backward: null upstream gradient");
  nrn::RayLossBwdParams p{};
  p.n = a->n_rays; p.S = a->n_samples; p.g = a->g;
  const float* u[5] = {a->u_rgb, a->u_rgb0, a->u_unmasked_offsets, a->u_rigidity_mask, a->u_divergence};
  float* d[5] = {a->d_rgb, a->d_rgb0, a->d_unmasked_offsets, a->d_rigidity_mask, a->d_divergence};
  for (int k = 0; k < 5; ++k) {
    if ((u[k] == nullptr) != (d[k] == nullptr)) return fail(NRN_E_INVALID, "nrn_ray_loss_backward: unit / output pair %d half given", k);
    p.u[k] = u[k]; p.d[k] = d[k];
  }
  const cudaError_t e = nrn::launch_ray_loss_bwd(p, static_cast<cudaStream_t>(a->stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "ray_loss_bwd_kernel");
}

int nrn_scale_rows(const float* g, const float* unit, float* out, int64_t n, int per_row, void* stream) {
  if (n < 0 || per_row < 1) return fail(NRN_E_INVALID, "nrn_scale_rows: bad sizes");
  if (n == 0) return NRN_OK;
  if (!g || !unit || !out) return fail(NRN_E_INVALID, "nrn_scale_rows: null argument");
  cudaError_t e = nrn::launch_ray_loss_scale(g, unit, out, n, per_row, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "ray_loss_scale_kernel");
}

static int fill_adam(const NrnAdamArgs* a, nrn::AdamParams& p, const char* who, bool need_grads);
int nrn_adam_step(const NrnAdamArgs* a) {
  nrn::AdamParams p{};
  const int rc = fill_adam(a, p, "nrn_adam_step", true);
  if (rc) return rc;
  const cudaError_t e = nrn::launch_adam(p, a->n_tensors, a->n_blocks, static_cast<cudaStream_t>(a->stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "adam_kernel");
}

static int fill_adam(const NrnAdamArgs* a, nrn::AdamParams& p, const char* who, bool need_grads) {
  if (!a) return fail(NRN_E_INVALID, "%s: null args", who);
  if (a->n_blocks < 0 || a->n_tensors < 0) return fail(NRN_E_INVALID, "%s: n_tensors = %d, n_blocks = %d", who, a->n_tensors, a->n_blocks);
  if (!a->params || !a->exp_avg || !a->exp_avg_sq || (need_grads && !a->grad_ptrs) || !a->blocks || !a->lr || !a->step)
    return fail(NRN_E_INVALID, "%s: null buffer", who);
  if (!(a->beta1 >= 0.f && a->beta1 < 1.f && a->beta2 >= 0.f && a->beta2 < 1.f && a->eps >= 0.f))
    return fail(NRN_E_INVALID, "%s: betas / eps out of range", who);
  p.params = static_cast<float*>(a->params); p.exp_avg = static_cast<float*>(a->exp_avg); p.exp_avg_sq = static_cast<float*>(a->exp_avg_sq);
  p.grads = static_cast<const float* const*>(a->grad_ptrs); p.blocks = static_cast<const nrn::AdamBlock*>(a->blocks);
  p.lr = static_cast<const float*>(a->lr); p.step = static_cast<long long*>(a->step);
  p.beta1 = a->beta1; p.beta2 = a->beta2; p.eps = a->eps;
  return NRN_OK;
}

size_t nrn_peer_window_bytes(int64_t arena_floats, int64_t slot_floats) {
  if (arena_floats < 0 || slot_floats < 0) return 0;
  const size_t slot_bytes = (static_cast<size_t>(slot_floats) * 4 + 255) / 256 * 256;
  return nrn::kPeerFlagBytes + 2 * slot_bytes + (static_cast<size_t>(arena_floats) * 4 + 255) / 256 * 256;
}

int nrn_peer_alloc(size_t bytes, void** dev_ptr, void* ipc_handle) {
  if (!dev_ptr || !ipc_handle || bytes < nrn::kPeerFlagBytes) return fail(NRN_E_INVALID, "nrn_peer_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(peer window)");
  e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return cuda_fail(e, "cudaIpcGetMemHandle"); }
  memcpy(ipc_handle, &h, sizeof(h));
  *dev_ptr = p;
  return NRN_OK;
}

int nrn_peer_open(const void* ipc_handle, void** dev_ptr) {
  if (!ipc_handle || !dev_ptr) return fail(NRN_E_INVALID, "nrn_peer_open: null argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle, sizeof(h));
  void* p = nullptr;
  const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return cuda_fail(e, "cudaIpcOpenMemHandle (peer-to-peer access between the GPUs of this node is required)");
  *dev_ptr = p;
  return NRN_OK;
}

int nrn_peer_close(void* dev_ptr) {
  if (!dev_ptr) return NRN_OK;
  const cudaError_t e = cudaIpcCloseMemHandle(dev_ptr);
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "cudaIpcCloseMemHandle");
}

int nrn_peer_free(void* dev_ptr) {
  if (!dev_ptr) return NRN_OK;
  const cudaError_t e = cudaFree(dev_ptr);
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "cudaFree(peer window)");
}

static int fill_peer(const NrnPeerCtx* c, nrn::PeerCtx& p, const char* who) {
  if (!c) return fail(NRN_E_INVALID, "%s: null context", who);
  if (c->world < 1 || c->world > nrn::kPeerMaxRanks || c->rank < 0 || c->rank >= c->world)
    return fail(NRN_E_INVALID, "%s: world = %d, rank = %d (at most %d ranks of one node)", who, c->world, c->rank, nrn::kPeerMaxRanks);
  if (!c->state || c->arena_floats < 0 || c->slot_floats < 0) return fail(NRN_E_INVALID, "%s: bad context", who);
  for (int r = 0; r < c->world; ++r) {
    if (!c->window[r]) return fail(NRN_E_INVALID, "%s: window of rank %d not mapped", who, r);
    p.window[r] = static_cast<uint8_t*>(c->window[r]);
  }
  p.world = c->world; p.rank = c->rank;
  p.slot_off = nrn::kPeerFlagBytes;
  p.slot_bytes = (static_cast<size_t>(c->slot_floats) * 4 + 255) / 256 * 256;
  p.arena_off = p.slot_off + 2 * p.slot_bytes;
  return NRN_OK;
}

int nrn_peer_reduce_adam(const NrnPeerCtx* c, const NrnAdamArgs* a) {
  nrn::PeerCtx pc{};
  int rc = fill_peer(c, pc, "nrn_peer_reduce_adam");
  if (rc) return rc;
  nrn::AdamParams p{};
  rc = fill_adam(a, p, "nrn_peer_reduce_adam", false);
  if (rc) return rc;
  if (!c->reduced) return fail(NRN_E_INVALID, "nrn_peer_reduce_adam: null workspace");
  DeviceState* ds;
  rc = device_state(&ds);
  if (rc) return rc;
  uint32_t* state = static_cast<uint32_t*>(c->state);
  const cudaError_t e = nrn::launch_peer_reduce_adam(pc, p, a->n_tensors, a->n_blocks, c->arena_floats, state, c->reduced, state + 3,
                                                     ds->err_word, static_cast<cudaStream_t>(a->stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "peer_adam_kernel");
}

int nrn_peer_gather_rows(const NrnPeerCtx* c, const float* local, int n_per_rank, float* out, void* stream) {
  nrn::PeerCtx pc{};
  int rc = fill_peer(c, pc, "nrn_peer_gather_rows");
  if (rc) return rc;
  if (n_per_rank < 0 || n_per_rank > c->slot_floats) return fail(NRN_E_INVALID, "nrn_peer_gather_rows: %d floats per rank exceed the slot (%lld)", n_per_rank, (long long)c->slot_floats);
  if (n_per_rank == 0) return NRN_OK;
  if (!local || !out) return fail(NRN_E_INVALID, "nrn_peer_gather_rows: null argument");
  DeviceState* ds;
  rc = device_state(&ds);
  if (rc) return rc;
  const cudaError_t e = nrn::launch_peer_gather(pc, static_cast<uint32_t*>(c->state), local, n_per_rank, out, ds->err_word, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? NRN_OK : cuda_fail(e, "peer_collect_kernel");
}

int nrn_timing_enable(int on) {
  // the events are reused, never destroyed: a graph captured while timing was on holds event-record nodes naming them,
  // and replaying it after they were destroyed makes cudaGraphLaunch read freed memory
  g_timed_n = 0;
  g_timing = on != 0;
  return NRN_OK;
}

int nrn_timing_read(double* ms_sum, int* counts, int n_kinds) {
  if (!ms_sum || !counts || n_kinds < 1) return fail(NRN_E_INVALID, "nrn_timing_read: bad arguments");
  for (int k = 0; k < n_kinds; ++k) { ms_sum[k] = 0.0; counts[k] = 0; }
  for (int i = 0; i < g_timed_n; ++i) {
    cudaError_t e = cudaEventSynchronize(g_timed[i].b);
    if (e != cudaSuccess) return cuda_fail(e, "cudaEventSynchronize");
    float ms = 0.f;
    e = cudaEventElapsedTime(&ms, g_timed[i].a, g_timed[i].b);
    if (e != cudaSuccess) return cuda_fail(e, "cudaEventElapsedTime");
    if (g_timed[i].kind < n_kinds) { ms_sum[g_timed[i].kind] += ms; counts[g_timed[i].kind] += 1; }
  }
  return NRN_OK;
}

}  // extern "C"
