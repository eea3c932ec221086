// C ABI of libnerf_pl_b200.so (declarations + reference citations: include/nerf_pl_b200.h).
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/nerf_pl_b200.h"
#include "aux_kernels.cuh"
#include "bwd_kernels.cuh"
#ifdef NERFB200_DIAG
#include "../../include/nerf_pl_b200_diag.h"
#include "diag_kernels.cuh"
#endif

using namespace nerfb200;

namespace {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, const char* detail = "") {
  std::snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}
int cuda_fail(cudaError_t e, const char* where) {
  std::snprintf(g_err, sizeof(g_err), "%s: %s (%s)", where, cudaGetErrorString(e), cudaGetErrorName(e));
  return static_cast<int>(e);
}
#define CUDA_TRY(expr, where)                          \
  do {                                                 \
    cudaError_t e_ = (expr);                           \
    if (e_ != cudaSuccess) return cuda_fail(e_, where); \
  } while (0)

struct DeviceInfo {
  int sm_count = 0;
  int cc_major = 0;
  bool attrs_set = false;
  bool diag_attrs_set = false;
  int* status = nullptr;        // device view of the mapped status word below
  volatile int* status_host = nullptr;   // pinned, mapped: the kernels write it, the host polls it without a sync
  long long* timeline = nullptr;
};

// Experiment switches are read ONCE per process (NERFB200_FLAGS: bit 1 = device timeline in
// -DNERFB200_TIMELINE builds; NERFB200_MAX_CTAS: cap on the persistent grid).  Unset in production.
struct EnvSwitches {
  unsigned flags = 0;
  int max_ctas = 0;
  int wg_plan = 1;        // wgrad plan: 0 = contiguous equal-byte shares, 1 = whole CTAs per GEMM, chunks interleaved
  int wg_copy = 32768;    // bytes per bulk copy of a wgrad operand chunk
  unsigned wg_exp = 0;    // wgrad timing experiments: bit 0 = no MMAs, bit 1 = no CUDA-core reductions
  int no_zero_copy = 0;   // host entry: always stage through device memory (A/B of the mapped-memory fast path)
  EnvSwitches() {
    if (const char* v = std::getenv("NERFB200_NO_ZERO_COPY")) no_zero_copy = std::atoi(v);
    if (const char* v = std::getenv("NERFB200_WG_EXP")) wg_exp = static_cast<unsigned>(std::atoi(v));
    if (const char* v = std::getenv("NERFB200_WG_PLAN")) wg_plan = std::atoi(v);
    if (const char* v = std::getenv("NERFB200_WG_COPY")) wg_copy = std::atoi(v);
    if (const char* f = std::getenv("NERFB200_FLAGS")) flags = static_cast<unsigned>(std::strtoul(f, nullptr, 0));
    if (const char* mc = std::getenv("NERFB200_MAX_CTAS")) max_ctas = std::atoi(mc);
  }
};
const EnvSwitches& env_switches() {
  static const EnvSwitches e;
  return e;
}
std::mutex g_mu;
DeviceInfo g_dev[64];

int device_info(DeviceInfo** out) {
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev), "cudaGetDevice");
  if (dev < 0 || dev >= 64) return fail(NERFB200_EDEVICE, "device ordinal out of range%s");
  std::lock_guard<std::mutex> lk(g_mu);
  DeviceInfo& d = g_dev[dev];
  if (d.sm_count == 0) {
    CUDA_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev), "attr sm");
    CUDA_TRY(cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev), "attr cc");
  }
  if (d.cc_major != 10) return fail(NERFB200_EDEVICE, "nerf_pl_b200 needs an sm_100 (B200) device%s");
  if (!d.attrs_set) {
    CUDA_TRY(cudaFuncSetAttribute(render_rays_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(kSmemTotal)), "smem attr render");
    CUDA_TRY(cudaFuncSetAttribute(render_rays_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(kSmemTotal)), "smem attr render(save)");
    CUDA_TRY(cudaFuncSetAttribute(mlp_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(kSmemTotal)), "smem attr mlp");
    CUDA_TRY(cudaFuncSetAttribute(chain_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(kChSmemTotal)), "smem attr chain");
    CUDA_TRY(cudaFuncSetAttribute(chain_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(kChSmemTotal)), "smem attr chain (probe)");
    CUDA_TRY(cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(kWgSmemTotal)), "smem attr wgrad");
    int* hs = nullptr;
    CUDA_TRY(cudaHostAlloc(&hs, sizeof(int), cudaHostAllocMapped), "status alloc");
    *hs = 0;
    CUDA_TRY(cudaHostGetDevicePointer(&d.status, hs, 0), "status device pointer");
    d.status_host = hs;
    d.attrs_set = true;
  }
  *out = &d;
  return 0;
}

// A kernel of an EARLIER call on this device reported a device-side fault (misaligned shared
// memory, code 101) through the internal status word: surface it on this call and clear it.
// (The word lives in mapped pinned host memory, so this is a plain host read, no synchronisation;
// callers that want the fault of THIS call pass their own `status` word or call
// nerfb200_check_status() after synchronising.)
int check_sticky_status(DeviceInfo* d) {
  if (d->status_host == nullptr) return 0;
  const int st = *d->status_host;
  if (st == 0) return 0;
  *d->status_host = 0;
  std::snprintf(g_err, sizeof(g_err), "an earlier nerf_pl_b200 kernel reported device status %d", st);
  return NERFB200_EDEVICE;
}

int check_render_shapes(const nerfb200_render_args* a) {
  if (a == nullptr) return fail(NERFB200_EINVAL, "args is NULL%s");
  if (a->n_rays < 0) return fail(NERFB200_EINVAL, "n_rays < 0%s");
  if (a->n_samples != 32 && a->n_samples != 64 && a->n_samples != 128)
    return fail(NERFB200_EUNSUPPORTED, "N_samples must be 32, 64 or 128%s");
  if (a->n_importance < 0 || (a->n_importance % 32) != 0)
    return fail(NERFB200_EUNSUPPORTED, "N_importance must be a multiple of 32%s");
  if (a->n_samples + a->n_importance > kMaxSf)
    return fail(NERFB200_EUNSUPPORTED, "N_samples + N_importance must be <= 192%s");
  if (a->n_rays == 0) return 0;
  if (!a->rays || !a->packed_coarse) return fail(NERFB200_EINVAL, "rays / packed_coarse is NULL%s");
  if (a->ray_stride < 8) return fail(NERFB200_EINVAL, "ray_stride < 8%s");
  if (!a->opacity_coarse) return fail(NERFB200_EINVAL, "opacity_coarse is NULL%s");
  if (!a->test_time && (!a->rgb_coarse || !a->depth_coarse))
    return fail(NERFB200_EINVAL, "rgb_coarse / depth_coarse is NULL with test_time=0%s");
  if (a->n_importance > 0) {
    if (!a->packed_fine) return fail(NERFB200_EINVAL, "packed_fine is NULL with N_importance>0%s");
    if (!a->rgb_fine || !a->depth_fine || !a->opacity_fine)
      return fail(NERFB200_EINVAL, "fine outputs are NULL with N_importance>0%s");
  }
  if (a->perturb > 0.f && !a->rng_in_kernel) {
    if (!a->perturb_rand) return fail(NERFB200_EINVAL, "perturb>0 needs perturb_rand%s");
    if (a->n_importance > 0 && !a->u_rand) return fail(NERFB200_EINVAL, "perturb>0 needs u_rand%s");
  }
  if (a->noise_std > 0.f) {
    if (!a->noise_coarse) return fail(NERFB200_EINVAL, "noise_std>0 needs noise_coarse%s");
    if (a->n_importance > 0 && !a->noise_fine) return fail(NERFB200_EINVAL, "noise_std>0 needs noise_fine%s");
  }
  if ((reinterpret_cast<uintptr_t>(a->packed_coarse) & 15) ||
      (reinterpret_cast<uintptr_t>(a->packed_fine) & 15))
    return fail(NERFB200_EINVAL, "packed images must be 16-byte aligned%s");
  return 0;
}


// ------------------------------------------------------------------ training workspace layout
// One device buffer per (n_rays, N_samples, N_importance); the layout is a pure function of those
// numbers and the SM count, recomputed on every call (no state kept in the library).
struct WgJobPlan { int ps, kind, split, n_split; };
enum { kJ1 = 0, kJ2, kJ3, kJ4, kJ5a, kJ5b, kJ6, kJ7, kJ8, kJ9, kNumJobKinds };
constexpr int kWgSlotFloats = 256 * 256 + 256;           // partial of one piece: out (transposed), bias
constexpr int kMaxWgJobs = 1024;
constexpr int kMaxWgCtas = 512;
struct TrainLayout {
  PassBufs pass[2];
  int n_pass, n_rays;
  WgradJob* jobs_dev;             // pieces, in (pass, layer, chunk) order
  int* cta_first_dev;             // [n_cta + 1]: CTA b works on pieces [cta_first[b], cta_first[b + 1])
  int n_jobs, n_cta;
  int n_split[2][kNumJobKinds];   // pieces of each (pass, layer)
  int first_job[2][kNumJobKinds];
  float* wg_part;                 // [n_jobs][kWgSlotFloats]
  int head_grid;                  // blocks of head_bwd_kernel (both passes in one launch)
  float* head_part[2];            // [head_grid][kHeadPartFloats] per pass
  float* raysum[2];               // (n_rays, 128) per-ray sums of dd
  float* direnc;                  // (n_rays, 28) embedded directions
  float* dir_part[2];             // [kDirSlices][128][27]
  float* gWp[2];                  // (128,256)
  float* gbp[2];                  // (128)
  float* lscale;                  // [2][kLevels] per-pass, per-level gradient scales
  float* linv;                    // [2][kLevels] their inverses
  unsigned* lamax;                // [2][kLevels] probe statistics
  unsigned* amax;                 // [2][2] max |d sigma|, |d rgb_pre| per pass
  unsigned* tile_amax[2];         // [n_pad / 128][2] the same maxima per 128-sample tile
  float* wnorm;                   // [2][2] weight norms of the level-0 bound
  unsigned* saturated;            // [2] fp16 gradient elements the last backward's chain clipped
  float* loss_part;               // [max CTAs][2]
  unsigned* loss_counter;
  size_t bytes;
};

struct TrainLayout;
void plan_wgrad(TrainLayout* L, int n_cta, WgradJob* jobs, int* cta_first);

void job_shape(int kind, int* a_fb, int* b_fb) {
  *a_fb = (kind == kJ9) ? 2 : 4;
  *b_fb = (kind == kJ1 || kind == kJ5a) ? 1 : 4;
}

void make_train_layout(TrainLayout* L, uint8_t* base, int64_t n_rays, int n_samples, int n_importance, int sm_count) {
  size_t off = 0;
  auto take = [&](size_t bytes) -> uint8_t* {
    uint8_t* ptr = base ? base + off : nullptr;
    off += (bytes + 1023) & ~static_cast<size_t>(1023);
    return ptr;
  };
  L->n_pass = n_importance > 0 ? 2 : 1;
  L->n_rays = static_cast<int>(n_rays);
  std::memset(L->pass, 0, sizeof(L->pass));
  for (int ps = 0; ps < L->n_pass; ++ps) {
    PassBufs& b = L->pass[ps];
    b.S = ps ? n_samples + n_importance : n_samples;
    b.n = n_rays * b.S;
    b.n_pad = (b.n + 127) / 128 * 128;
    const size_t np = static_cast<size_t>(b.n_pad);
    b.enc = take(np * 128);
    b.act = take(np * 512 * 8);
    b.mask = reinterpret_cast<uint2*>(take(np * 32 * 8));
    b.d = take(np * 256);
    b.sigma = reinterpret_cast<float*>(take(np * 4));
    b.rgb = reinterpret_cast<float*>(take(np * 12));
    b.z = reinterpret_cast<float*>(take(static_cast<size_t>(b.n) * 4));
    b.dsigma = reinterpret_cast<float*>(take(np * 4));
    b.dprergb = reinterpret_cast<float*>(take(np * 12));
    b.dd = take(np * 256);
    b.dpre = take(np * 512 * 8);
  }
  // wgrad plan: the concatenation of all (pass, layer) GEMMs, measured in 8 KiB blocks streamed, is cut
  // into one equal share per SM; a share boundary inside a GEMM splits it into two pieces
  plan_wgrad(L, sm_count > 0 ? sm_count : 148, nullptr, nullptr);
  L->jobs_dev = reinterpret_cast<WgradJob*>(take(sizeof(WgradJob) * kMaxWgJobs));
  L->cta_first_dev = reinterpret_cast<int*>(take(sizeof(int) * (kMaxWgCtas + 1)));
  L->wg_part = reinterpret_cast<float*>(take(static_cast<size_t>(L->n_jobs) * kWgSlotFloats * 4));
  L->head_grid = static_cast<int>((L->n_pass * n_rays + kHeadWarps - 1) / kHeadWarps);
  L->direnc = reinterpret_cast<float*>(take(static_cast<size_t>(n_rays) * 28 * 4));
  for (int ps = 0; ps < 2; ++ps) {
    L->head_part[ps] = reinterpret_cast<float*>(take(static_cast<size_t>(L->head_grid) * kHeadPartFloats * 4));
    L->raysum[ps] = reinterpret_cast<float*>(take(static_cast<size_t>(n_rays) * 128 * 4));
    L->dir_part[ps] = reinterpret_cast<float*>(take(static_cast<size_t>(kDirSlices) * 128 * 27 * 4));
    L->gWp[ps] = reinterpret_cast<float*>(take(128 * 256 * 4));
    L->gbp[ps] = reinterpret_cast<float*>(take(128 * 4));
  }
  L->lscale = reinterpret_cast<float*>(take(2 * kLevels * 4));
  L->linv = reinterpret_cast<float*>(take(2 * kLevels * 4));
  L->lamax = reinterpret_cast<unsigned*>(take(2 * kLevels * 4));
  L->amax = reinterpret_cast<unsigned*>(take(16));
  for (int ps = 0; ps < 2; ++ps)
    L->tile_amax[ps] = ps < L->n_pass ? reinterpret_cast<unsigned*>(take(static_cast<size_t>(L->pass[ps].n_pad / 128) * 8)) : nullptr;
  L->wnorm = reinterpret_cast<float*>(take(16));
  L->saturated = reinterpret_cast<unsigned*>(take(8));
  L->loss_part = reinterpret_cast<float*>(take(1024 * 2 * 4));
  L->loss_counter = reinterpret_cast<unsigned*>(take(16));
  L->bytes = off;
}

// The wgrad plan of a layout: piece counts per (pass, layer) (always), and when `jobs` / `cta_first` are
// given the host image of the piece table and of the per-CTA piece ranges.
void job_operands(const TrainLayout& L, int ps, int k, const uint8_t** A, const uint8_t** B) {
  const PassBufs& b = L.pass[ps];
  const size_t lay = static_cast<size_t>(b.n_pad) * 512;
  switch (k) {
    case kJ1: *A = b.dpre; *B = b.enc; break;
    case kJ5a: *A = b.dpre + 4 * lay; *B = b.enc; break;
    case kJ5b: *A = b.dpre + 4 * lay; *B = b.act + 3 * lay; break;
    case kJ9: *A = b.dd; *B = b.act + 7 * lay; break;
    default: {
      const int l = (k <= kJ4) ? k + 1 : k;            // kJ2..kJ4 -> layers 2..4, kJ6..kJ8 -> layers 6..8
      *A = b.dpre + static_cast<size_t>(l - 1) * lay;
      *B = b.act + static_cast<size_t>(l - 2) * lay;
    }
  }
}

void fill_piece(TrainLayout* L, WgradJob* jobs, int piece, int ps, int k, long long c0, long long c1, int step) {
  if (!jobs) return;
  int a_fb, b_fb;
  job_shape(k, &a_fb, &b_fb);
  const uint8_t *A = nullptr, *B = nullptr;
  job_operands(*L, ps, k, &A, &B);
  WgradJob& j = jobs[piece];
  float* slot = L->wg_part + static_cast<size_t>(piece) * kWgSlotFloats;
  j.a = A; j.b = B; j.a_fb = a_fb; j.b_fb = b_fb;
  j.chunk0 = static_cast<int>(c0);
  j.chunk1 = static_cast<int>(c1);
  j.chunk_step = step;
  j.out = slot;
  j.bias_out = (k == kJ5b) ? nullptr : slot + 256 * 256;
}

void plan_wgrad(TrainLayout* L, int n_cta, WgradJob* jobs, int* cta_first) {
  if (n_cta > kMaxWgCtas) n_cta = kMaxWgCtas;
  long long total = 0;
  long long work[2][kNumJobKinds];
  for (int ps = 0; ps < L->n_pass; ++ps)
    for (int k = 0; k < kNumJobKinds; ++k) {
      int a_fb, b_fb;
      job_shape(k, &a_fb, &b_fb);
      work[ps][k] = (L->pass[ps].n_pad / 64) * (a_fb + b_fb);
      total += work[ps][k];
    }
  const int n_kinds = L->n_pass * kNumJobKinds;
  if (env_switches().wg_plan == 1 && n_cta >= n_kinds) {
    // ---- plan 1: whole CTAs per GEMM (largest-remainder apportionment of the SMs by bytes streamed); the
    // CTAs of one GEMM take its chunks round-robin, so together they read ONE moving window of each operand
    int n_of[2][kNumJobKinds];
    double frac[2][kNumJobKinds];
    int used = 0;
    for (int ps = 0; ps < L->n_pass; ++ps)
      for (int k = 0; k < kNumJobKinds; ++k) {
        const double share = static_cast<double>(work[ps][k]) * n_cta / static_cast<double>(total);
        int n = static_cast<int>(share);
        if (n < 1) n = 1;
        n_of[ps][k] = n;
        frac[ps][k] = share - n;
        used += n;
      }
    while (used < n_cta) {          // hand the remaining SMs to the GEMMs with the most work per CTA
      int bp = 0, bk = 0;
      double best = -1;
      for (int ps = 0; ps < L->n_pass; ++ps)
        for (int k = 0; k < kNumJobKinds; ++k) {
          const double load = static_cast<double>(work[ps][k]) / n_of[ps][k];
          if (load > best) { best = load; bp = ps; bk = k; }
        }
      ++n_of[bp][bk];
      ++used;
    }
    (void)frac;
    int piece = 0;
    for (int ps = 0; ps < L->n_pass; ++ps)
      for (int k = 0; k < kNumJobKinds; ++k) {
        const long long chunks = L->pass[ps].n_pad / 64;
        int g = n_of[ps][k];
        if (g > chunks) g = static_cast<int>(chunks);
        L->first_job[ps][k] = piece;
        for (int j = 0; j < g; ++j) {
          fill_piece(L, jobs, piece, ps, k, j, chunks, g);
          if (cta_first) cta_first[piece] = piece;
          ++piece;
        }
        L->n_split[ps][k] = g;
      }
    if (cta_first) cta_first[piece] = piece;
    L->n_jobs = piece;
    L->n_cta = piece;
    return;
  }
  // ---- plan 0: the concatenation of all GEMMs cut into one equal-byte share per SM
  int cta = 0, piece = 0;
  long long done = 0;                                  // units handed out so far
  if (cta_first) cta_first[0] = 0;
  for (int ps = 0; ps < L->n_pass; ++ps)
    for (int k = 0; k < kNumJobKinds; ++k) {
      int a_fb, b_fb;
      job_shape(k, &a_fb, &b_fb);
      const long long unit = a_fb + b_fb, chunks = L->pass[ps].n_pad / 64;
      L->first_job[ps][k] = piece;
      long long c = 0;
      while (c < chunks) {
        const long long end = total * (cta + 1) / n_cta;
        long long take_chunks = (end - done + unit - 1) / unit;       // chunks until this CTA's share is full
        if (take_chunks < 1) take_chunks = 1;
        if (take_chunks > chunks - c) take_chunks = chunks - c;
        fill_piece(L, jobs, piece, ps, k, c, c + take_chunks, 1);
        ++piece;
        c += take_chunks;
        done += take_chunks * unit;
        while (cta < n_cta - 1 && done >= total * (cta + 1) / n_cta) {
          ++cta;
          if (cta_first) cta_first[cta] = piece;
        }
      }
      L->n_split[ps][k] = piece - L->first_job[ps][k];
    }
  if (cta_first) {
    for (int i = cta + 1; i <= n_cta; ++i) cta_first[i] = piece;
  }
  L->n_jobs = piece;
  L->n_cta = n_cta;
}

// grow-only device arena for the *_host entry
struct Arena {
  uint8_t* base = nullptr;
  size_t cap = 0;
  size_t off = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return 0;
    if (base) cudaFree(base);
    base = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&base, bytes);
    if (e != cudaSuccess) return cuda_fail(e, "arena cudaMalloc");
    cap = bytes;
    return 0;
  }
  void* take(size_t bytes) {
    void* p = base + off;
    off += (bytes + 255) & ~static_cast<size_t>(255);
    return p;
  }
};
Arena g_arena[64];
std::mutex g_host_call_mu;
std::mutex g_arena_mu;   // separate from g_mu: the host entry calls nerfb200_render_rays (device_info locks g_mu)

}  // namespace

extern "C" {

int nerfb200_abi_version(void) { return NERFB200_ABI_VERSION; }
const char* nerfb200_last_error(void) { return g_err; }
size_t nerfb200_packed_bytes(void) { return kPackedBytes; }
int64_t nerfb200_launch_count(void) { return g_launches.load(); }

int nerfb200_sm_count(void) {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  return n;
}

static int fill_pack_params(PackParams* pp, const float* const params[24], void* packed) {
  if (!params || !packed) return fail(NERFB200_EINVAL, "pack_weights: NULL argument%s");
  if (reinterpret_cast<uintptr_t>(packed) & 15) return fail(NERFB200_EINVAL, "packed must be 16-byte aligned%s");
  for (int i = 0; i < kNumParams; ++i) {
    if (!params[i]) return fail(NERFB200_EINVAL, "pack_weights: NULL parameter tensor%s");
    pp->p[i] = params[i];
  }
  pp->out = static_cast<uint8_t*>(packed);
  pp->bwd_bf16 = kBwdBf16 ? 1 : 0;
  return 0;
}

static int launch_pack(const PackParams2& pp2, int n_nets, void* stream) {
  const long long total = kHalfRegionBytes / 2 + kF32Count + static_cast<long long>(kNumSlicesBwd) * 256 * 64;
  const int threads = 256;
  const int blocks = static_cast<int>((total + threads - 1) / threads);
  pack_weights_kernel<<<dim3(blocks, n_nets), threads, 0, static_cast<cudaStream_t>(stream)>>>(pp2);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "pack_weights launch");
  return 0;
}

int nerfb200_pack_weights(const float* const params[24], void* packed, void* stream) {
  PackParams2 pp2;
  int rc = fill_pack_params(&pp2.net[0], params, packed);
  if (rc) return rc;
  pp2.net[1] = pp2.net[0];
  return launch_pack(pp2, 1, stream);
}

int nerfb200_pack_weights_pair(const float* const params_a[24], void* packed_a, const float* const params_b[24],
                               void* packed_b, void* stream) {
  PackParams2 pp2;
  int rc = fill_pack_params(&pp2.net[0], params_a, packed_a);
  if (rc) return rc;
  rc = fill_pack_params(&pp2.net[1], params_b, packed_b);
  if (rc) return rc;
  return launch_pack(pp2, 2, stream);
}

int nerfb200_render_rays(const nerfb200_render_args* a, void* stream) {
  int rc = check_render_shapes(a);
  if (rc) return rc;
  if (a->n_rays == 0) return 0;
  if (a->n_rays > 0x7fffffff) return fail(NERFB200_EINVAL, "n_rays too large%s");
  DeviceInfo* d = nullptr;
  rc = device_info(&d);
  if (rc) return rc;
  if (!a->status && (rc = check_sticky_status(d)) != 0) return rc;
  RenderParams p;
  p.rays = a->rays;
  p.ray_stride = a->ray_stride;
  p.n_rays = static_cast<int>(a->n_rays);
  p.net_coarse = static_cast<const uint8_t*>(a->packed_coarse);
  p.net_fine = static_cast<const uint8_t*>(a->packed_fine);
  p.n_samples = a->n_samples;
  p.n_importance = a->n_importance;
  p.use_disp = a->use_disp;
  p.perturb = a->perturb;
  p.noise_std = a->noise_std;
  p.white_back = a->white_back;
  p.test_time = a->test_time;
  p.perturb_rand = a->perturb_rand;
  p.noise_coarse = a->noise_coarse;
  p.noise_fine = a->noise_fine;
  p.u_rand = a->u_rand;
  p.rgb_coarse = a->rgb_coarse;
  p.depth_coarse = a->depth_coarse;
  p.opacity_coarse = a->opacity_coarse;
  p.rgb_fine = a->rgb_fine;
  p.depth_fine = a->depth_fine;
  p.opacity_fine = a->opacity_fine;
  p.z_fine = a->z_fine;
  p.weights_coarse = a->weights_coarse;
  p.weights_fine = a->weights_fine;
  p.status = a->status ? a->status : d->status;
  p.z_coarse = a->z_coarse;
  p.rng_seed = a->rng_seed;
  p.rng_in_kernel = a->rng_in_kernel;
  p.train = 0;
  p.target = nullptr; p.loss_part = nullptr; p.loss_out = nullptr; p.loss_counter = nullptr;
  std::memset(p.tr, 0, sizeof(p.tr));
  const bool save = a->train_workspace != nullptr;
  if (save && a->test_time) return fail(NERFB200_EINVAL, "train_workspace needs test_time = 0%s");
  if ((a->target != nullptr) != (a->loss_out != nullptr)) return fail(NERFB200_EINVAL, "target and loss_out go together%s");
  if (a->target && !save) return fail(NERFB200_EINVAL, "the fused loss epilogue needs train_workspace%s");
  if (save) {
    TrainLayout L;
    make_train_layout(&L, static_cast<uint8_t*>(a->train_workspace), a->n_rays, a->n_samples, a->n_importance, d->sm_count);
    p.train = 1;
    p.tr[0] = L.pass[0];
    p.tr[1] = L.pass[1];
    if (!p.z_coarse) p.z_coarse = L.pass[0].z;
    else return fail(NERFB200_EINVAL, "z_coarse is owned by the workspace in training mode%s");
    if (a->n_importance > 0) {
      if (p.z_fine) return fail(NERFB200_EINVAL, "z_fine is owned by the workspace in training mode%s");
      p.z_fine = L.pass[1].z;
    }
    if (a->target) {
      p.target = a->target;
      p.loss_out = a->loss_out;
      p.loss_part = L.loss_part;
      p.loss_counter = L.loss_counter;
    }
  }
  p.flags = env_switches().flags;
  p.timeline = nullptr;
#ifdef NERFB200_TIMELINE
  if (p.flags & 2u) {
    if (!d->timeline) {
      CUDA_TRY(cudaMalloc(&d->timeline, 3 * kTlMax * 2 * sizeof(long long)), "timeline alloc");
    }
    CUDA_TRY(cudaMemsetAsync(d->timeline, 0, 3 * kTlMax * 2 * sizeof(long long), static_cast<cudaStream_t>(stream)), "timeline memset");
    p.timeline = d->timeline;
  }
#endif
  const int n_groups = (p.n_rays + 1) / 2;     // two rays share the coarse tile
  int ctas = d->sm_count;
  if (a->max_ctas > 0 && a->max_ctas < ctas) ctas = a->max_ctas;
  if (env_switches().max_ctas > 0 && env_switches().max_ctas < ctas) ctas = env_switches().max_ctas;
  if (n_groups < ctas) ctas = n_groups;
  if (save)
    render_rays_kernel<true><<<ctas, kRenderThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(p);
  else
    render_rays_kernel<false><<<ctas, kRenderThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(p);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "render_rays launch");
  return 0;
}

int nerfb200_render_rays_host(const nerfb200_render_args* h, void* stream_v) {
  int rc = check_render_shapes(h);
  if (rc) return rc;
  if (h->n_rays == 0) return 0;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  if (h->train_workspace || h->target || h->z_coarse)
    return fail(NERFB200_EINVAL, "render_rays_host: train_workspace / target / z_coarse are device-only%s");
  {
    // Fast path: every host buffer is page-locked and mapped into the device's address space (cudaHostAlloc /
    // cudaHostRegister; torch's pin_memory()).  The kernel then reads the rays and writes the <= 40 B of results
    // per ray straight over PCIe - no staging copies, no copy-engine round trips (each small cudaMemcpyAsync
    // costs ~8 us of latency on the stream; the bytes that cross the bus are the same) - and the call is
    // "launch + synchronise".  Random inputs may be device tensors (drawn there by the caller) or mapped too.
    bool all_mapped = true;
    auto mapped = [&](const void* p, const void** dp) -> bool {
      *dp = nullptr;
      if (!p) return true;
      cudaPointerAttributes attr;
      if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
      if ((attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) &&
          attr.devicePointer != nullptr) {
        *dp = attr.devicePointer;
        return true;
      }
      return false;
    };
    nerfb200_render_args a = *h;
    const void* dp = nullptr;
#define NERFB200_MAP(field, type)                                          \
    all_mapped = all_mapped && mapped(h->field, &dp);                      \
    a.field = static_cast<type>(const_cast<void*>(dp));
    NERFB200_MAP(rays, const float*)
    NERFB200_MAP(perturb_rand, const float*)
    NERFB200_MAP(noise_coarse, const float*)
    NERFB200_MAP(u_rand, const float*)
    NERFB200_MAP(noise_fine, const float*)
    NERFB200_MAP(rgb_coarse, float*)
    NERFB200_MAP(depth_coarse, float*)
    NERFB200_MAP(opacity_coarse, float*)
    NERFB200_MAP(rgb_fine, float*)
    NERFB200_MAP(depth_fine, float*)
    NERFB200_MAP(opacity_fine, float*)
    NERFB200_MAP(z_fine, float*)
    NERFB200_MAP(weights_coarse, float*)
    NERFB200_MAP(weights_fine, float*)
#undef NERFB200_MAP
    if (all_mapped && !env_switches().no_zero_copy) {
      int dev0 = 0;
      CUDA_TRY(cudaGetDevice(&dev0), "cudaGetDevice");
      static int* host_status[64] = {nullptr};
      {
        std::lock_guard<std::mutex> lk(g_arena_mu);
        if (!host_status[dev0])
          CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&host_status[dev0]), 256, cudaHostAllocMapped | cudaHostAllocPortable),
                   "status cudaHostAlloc");
      }
      // one in-flight host call per device at a time shares the status word: serialise
      std::lock_guard<std::mutex> lk(g_host_call_mu);
      volatile int* hs = host_status[dev0];
      *hs = 0;
      int* dstatus = nullptr;
      CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&dstatus), host_status[dev0], 0), "status device pointer");
      a.status = dstatus;
      rc = nerfb200_render_rays(&a, stream);
      if (rc) return rc;
      CUDA_TRY(cudaStreamSynchronize(stream), "render_rays_host sync");
      const int hstatus = *hs;
      if (hstatus != 0) {
        std::snprintf(g_err, sizeof(g_err), "render kernel reported device status %d", hstatus);
        return NERFB200_EDEVICE;
      }
      if (h->status) *h->status = 0;
      return 0;
    }
  }
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev), "cudaGetDevice");
  const size_t n = static_cast<size_t>(h->n_rays);
  const size_t Sc = h->n_samples, K = h->n_importance, Sf = Sc + K;
  const size_t fl = sizeof(float);
  // rays + 4 random inputs + 8 float outputs (+3 optional) + status, each rounded to 256 B
  size_t need = 16 * 256 + n * fl * (8 + Sc + Sc + K + Sf + 3 + 1 + 1 + 3 + 1 + 1 + Sf + Sc + Sf) + 256;
  Arena& ar = g_arena[dev];
  std::lock_guard<std::mutex> lk(g_arena_mu);
  rc = ar.reserve(need);
  if (rc) return rc;
  ar.off = 0;
  nerfb200_render_args a = *h;
  a.ray_stride = 8;
  auto up = [&](const float* src, size_t count, size_t src_stride, size_t width) -> const float* {
    if (!src) return nullptr;
    if (src_stride == width) {
      // random inputs may already live on the device (drawn there by the caller): use them in place
      cudaPointerAttributes attr;
      if (cudaPointerGetAttributes(&attr, src) == cudaSuccess && attr.type == cudaMemoryTypeDevice) return src;
      (void)cudaGetLastError();
    }
    float* dst = static_cast<float*>(ar.take(count * fl));
    if (src_stride == width) {
      cudaMemcpyAsync(dst, src, count * fl, cudaMemcpyHostToDevice, stream);
    } else {
      cudaMemcpy2DAsync(dst, width * fl, src, src_stride * fl, width * fl, count / width,
                        cudaMemcpyHostToDevice, stream);
    }
    return dst;
  };
  a.rays = up(h->rays, n * 8, static_cast<size_t>(h->ray_stride), 8);
  a.perturb_rand = up(h->perturb_rand, n * Sc, Sc, Sc);
  a.noise_coarse = up(h->noise_coarse, n * Sc, Sc, Sc);
  a.u_rand = up(h->u_rand, n * K, K, K);
  a.noise_fine = up(h->noise_fine, n * Sf, Sf, Sf);
  auto dn = [&](float* hostp, size_t count) -> float* {
    return hostp ? static_cast<float*>(ar.take(count * fl)) : nullptr;
  };
  a.rgb_coarse = dn(h->rgb_coarse, n * 3);
  a.depth_coarse = dn(h->depth_coarse, n);
  a.opacity_coarse = dn(h->opacity_coarse, n);
  a.rgb_fine = dn(h->rgb_fine, n * 3);
  a.depth_fine = dn(h->depth_fine, n);
  a.opacity_fine = dn(h->opacity_fine, n);
  a.z_fine = dn(h->z_fine, n * Sf);
  a.weights_coarse = dn(h->weights_coarse, n * Sc);
  a.weights_fine = dn(h->weights_fine, n * Sf);
  int* dstatus = static_cast<int*>(ar.take(sizeof(int)));
  CUDA_TRY(cudaMemsetAsync(dstatus, 0, sizeof(int), stream), "status memset");
  a.status = dstatus;
  rc = nerfb200_render_rays(&a, stream);
  if (rc) return rc;
  auto back = [&](float* hostp, const float* devp, size_t count) {
    if (hostp) cudaMemcpyAsync(hostp, devp, count * fl, cudaMemcpyDeviceToHost, stream);
  };
  back(h->rgb_coarse, a.rgb_coarse, n * 3);
  back(h->depth_coarse, a.depth_coarse, n);
  back(h->opacity_coarse, a.opacity_coarse, n);
  back(h->rgb_fine, a.rgb_fine, n * 3);
  back(h->depth_fine, a.depth_fine, n);
  back(h->opacity_fine, a.opacity_fine, n);
  back(h->z_fine, a.z_fine, n * Sf);
  back(h->weights_coarse, a.weights_coarse, n * Sc);
  back(h->weights_fine, a.weights_fine, n * Sf);
  int hstatus = 0;
  CUDA_TRY(cudaMemcpyAsync(&hstatus, dstatus, sizeof(int), cudaMemcpyDeviceToHost, stream), "status copy");
  CUDA_TRY(cudaStreamSynchronize(stream), "render_rays_host sync");
  if (hstatus != 0) {
    std::snprintf(g_err, sizeof(g_err), "render kernel reported device status %d", hstatus);
    return NERFB200_EDEVICE;
  }
  if (h->status) *h->status = hstatus;
  return 0;
}

int nerfb200_nerf_forward(const float* x, int64_t n, int64_t x_stride, const void* packed,
                          int32_t sigma_only, float* out, void* stream) {
  if (n < 0) return fail(NERFB200_EINVAL, "nerf_forward: n < 0%s");
  if (n == 0) return 0;
  if (!x || !packed || !out) return fail(NERFB200_EINVAL, "nerf_forward: NULL argument%s");
  if (x_stride < (sigma_only ? kEncXyz : kEncXyz + kEncDir))
    return fail(NERFB200_EINVAL, "nerf_forward: x_stride too small for the input width%s");
  if (!sigma_only && (reinterpret_cast<uintptr_t>(out) & 15))
    return fail(NERFB200_EINVAL, "nerf_forward: out must be 16-byte aligned%s");
  DeviceInfo* d = nullptr;
  int rc = device_info(&d);
  if (rc) return rc;
  if ((rc = check_sticky_status(d)) != 0) return rc;
  MlpParams p;
  p.raw_xyz = 0;
  p.x = x; p.x_stride = x_stride; p.n = n;
  p.net = static_cast<const uint8_t*>(packed);
  p.sigma_only = sigma_only;
  p.out = out;
  p.status = d->status;
  const long long tiles = (n + 127) / 128;
  const int ctas = static_cast<int>(tiles < d->sm_count ? tiles : d->sm_count);
  mlp_forward_kernel<<<ctas, kThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(p);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "nerf_forward launch");
  return 0;
}

int nerfb200_query_sigma(const float* xyz, int64_t n, int64_t xyz_stride, const void* packed, float* sigma,
                         void* stream) {
  if (n < 0) return fail(NERFB200_EINVAL, "query_sigma: n < 0%s");
  if (n == 0) return 0;
  if (!xyz || !packed || !sigma) return fail(NERFB200_EINVAL, "query_sigma: NULL argument%s");
  if (xyz_stride < 3) return fail(NERFB200_EINVAL, "query_sigma: xyz_stride < 3%s");
  DeviceInfo* d = nullptr;
  int rc = device_info(&d);
  if (rc) return rc;
  if ((rc = check_sticky_status(d)) != 0) return rc;
  MlpParams p;
  p.raw_xyz = 1;
  p.x = xyz; p.x_stride = xyz_stride; p.n = n;
  p.net = static_cast<const uint8_t*>(packed);
  p.sigma_only = 1;
  p.out = sigma;
  p.status = d->status;
  const long long tiles = (n + 127) / 128;
  const int ctas = static_cast<int>(tiles < d->sm_count ? tiles : d->sm_count);
  mlp_forward_kernel<<<ctas, kThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(p);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "query_sigma launch");
  return 0;
}

int nerfb200_mse_psnr(const float* rgb_coarse, const float* rgb_fine, const float* target, int64_t n_rays,
                      float* out4, void* stream) {
  if (n_rays <= 0) return fail(NERFB200_EINVAL, "mse_psnr: n_rays <= 0%s");
  if ((!rgb_coarse && !rgb_fine) || !target || !out4) return fail(NERFB200_EINVAL, "mse_psnr: NULL argument%s");
  mse_psnr_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(rgb_coarse, rgb_fine, target, n_rays * 3, out4);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "mse_psnr launch");
  return 0;
}

int nerfb200_embed(const float* x, int64_t n, int32_t n_freqs, float* out, void* stream) {
  if (n < 0 || n_freqs < 0 || n_freqs > 16) return fail(NERFB200_EINVAL, "embed: bad n / n_freqs%s");
  if (n == 0) return 0;
  if (!x || !out) return fail(NERFB200_EINVAL, "embed: NULL argument%s");
  const long long total = n * (3 + 6 * n_freqs);
  const int threads = 256;
  long long blocks = (total + threads - 1) / threads;
  if (blocks > 148 * 16) blocks = 148 * 16;
  embed_kernel<<<static_cast<int>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(x, n, n_freqs, out);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "embed launch");
  return 0;
}

int nerfb200_searchsorted(const float* a, const float* v, int64_t* out, int64_t nrow_a,
                          int64_t nrow_v, int32_t ncol_a, int32_t ncol_v, int32_t side_right,
                          void* stream) {
  if (nrow_a < 0 || nrow_v < 0 || ncol_a < 0 || ncol_v < 0)
    return fail(NERFB200_EINVAL, "searchsorted: negative size%s");
  // searchsorted.py:26-29: same number of rows, or one of them has a single row
  if (nrow_a != nrow_v && nrow_a != 1 && nrow_v != 1)
    return fail(NERFB200_EINVAL, "searchsorted: a and v need the same number of rows, or 1 row%s");
  const long long nrow = nrow_a > nrow_v ? nrow_a : nrow_v;
  const long long total = nrow * ncol_v;
  if (total == 0) return 0;
  if (!a && ncol_a > 0) return fail(NERFB200_EINVAL, "searchsorted: a is NULL%s");
  if (!v || !out) return fail(NERFB200_EINVAL, "searchsorted: NULL argument%s");
  const int threads = 256;
  long long blocks = (total + threads - 1) / threads;
  if (blocks > 148 * 16) blocks = 148 * 16;
  searchsorted_kernel<<<static_cast<int>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(
      a, v, reinterpret_cast<long long*>(out), nrow_a, nrow_v, ncol_a, ncol_v, side_right);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "searchsorted launch");
  return 0;
}

int nerfb200_sample_pdf(const float* bins, const float* weights, const float* u, int64_t n_rays,
                        int32_t n_weights, int32_t n_u, float* out, void* stream) {
  if (n_rays < 0 || n_weights < 1 || n_u < 0 || n_weights > 4096)
    return fail(NERFB200_EINVAL, "sample_pdf: bad sizes%s");
  if (n_rays == 0 || n_u == 0) return 0;
  if (!bins || !weights || !u || !out) return fail(NERFB200_EINVAL, "sample_pdf: NULL argument%s");
  const int wpb = 4;
  const size_t sh = wpb * (n_weights + 1) * sizeof(float);
  long long blocks = (n_rays + wpb - 1) / wpb;
  if (blocks > 148 * 8) blocks = 148 * 8;
  sample_pdf_kernel<<<static_cast<int>(blocks), wpb * 32, sh, static_cast<cudaStream_t>(stream)>>>(
      bins, weights, u, n_rays, n_weights, n_u, out);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "sample_pdf launch");
  return 0;
}

int nerfb200_composite(const float* sigmas, const float* rgbs, const float* z_vals,
                       const float* dirs, const float* noise, float noise_std, int32_t white_back,
                       int64_t n_rays, int32_t S, float* weights, float* rgb, float* depth,
                       float* opacity, void* stream) {
  if (n_rays < 0) return fail(NERFB200_EINVAL, "composite: n_rays < 0%s");
  if (S <= 0 || (S % 32) != 0 || S > kMaxSf) return fail(NERFB200_EUNSUPPORTED, "composite: S must be a multiple of 32, <= 192%s");
  if (n_rays == 0) return 0;
  if (!sigmas || !z_vals || !dirs || !opacity) return fail(NERFB200_EINVAL, "composite: NULL argument%s");
  if (rgbs && (!rgb || !depth)) return fail(NERFB200_EINVAL, "composite: rgb/depth outputs NULL%s");
  const int wpb = 4;
  const size_t sh = wpb * 6 * S * sizeof(float);
  long long blocks = (n_rays + wpb - 1) / wpb;
  if (blocks > 148 * 8) blocks = 148 * 8;
  composite_kernel<<<static_cast<int>(blocks), wpb * 32, sh, static_cast<cudaStream_t>(stream)>>>(
      sigmas, rgbs, z_vals, dirs, noise, noise_std, white_back, n_rays, S, weights, rgb, depth, opacity);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "composite launch");
  return 0;
}

int nerfb200_generate_rays(int32_t H, int32_t W, float focal, const float c2w_host[12], float near, float far,
                           int32_t ndc, float* rays, void* stream) {
  if (H <= 0 || W <= 0 || !(focal > 0.f)) return fail(NERFB200_EINVAL, "generate_rays: bad H / W / focal%s");
  if (!c2w_host || !rays) return fail(NERFB200_EINVAL, "generate_rays: NULL argument%s");
  if (reinterpret_cast<uintptr_t>(rays) & 15) return fail(NERFB200_EINVAL, "generate_rays: rays must be 16-byte aligned%s");
  RayGenParams p;
  p.H = H; p.W = W; p.focal = focal; p.near = near; p.far = far; p.ndc = ndc; p.rays = rays;
  for (int i = 0; i < 12; ++i) p.c2w[i] = c2w_host[i];
  const long long total = static_cast<long long>(H) * W;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  generate_rays_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "generate_rays launch");
  return 0;
}

int nerfb200_to_uint8(const float* src, int64_t n, uint8_t* dst, void* stream) {
  if (n < 0) return fail(NERFB200_EINVAL, "to_uint8: n < 0%s");
  if (n == 0) return 0;
  if (!src || !dst) return fail(NERFB200_EINVAL, "to_uint8: NULL argument%s");
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  to_uint8_kernel<<<static_cast<int>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, n, dst);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "to_uint8 launch");
  return 0;
}

size_t nerfb200_train_workspace_bytes(int64_t n_rays, int32_t n_samples, int32_t n_importance) {
  if (n_rays <= 0 || n_samples <= 0 || n_importance < 0) return 0;
  TrainLayout L;
  make_train_layout(&L, nullptr, n_rays, n_samples, n_importance, nerfb200_sm_count());
  return L.bytes;
}

int nerfb200_train_workspace_init(void* workspace, size_t bytes, int64_t n_rays, int32_t n_samples,
                                  int32_t n_importance, void* stream_v) {
  if (!workspace || n_rays <= 0) return fail(NERFB200_EINVAL, "train_workspace_init: bad argument%s");
  if (reinterpret_cast<uintptr_t>(workspace) & 1023) return fail(NERFB200_EINVAL, "train workspace must be 1024-byte aligned%s");
  DeviceInfo* d = nullptr;
  int rc = device_info(&d);
  if (rc) return rc;
  TrainLayout L;
  make_train_layout(&L, static_cast<uint8_t*>(workspace), n_rays, n_samples, n_importance, d->sm_count);
  if (bytes < L.bytes) return fail(NERFB200_EINVAL, "train workspace too small%s");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  // padding rows of the operand arrays must be zero (never written afterwards), counters zero
  CUDA_TRY(cudaMemsetAsync(workspace, 0, L.bytes, stream), "workspace memset");
  std::vector<WgradJob> jobs(kMaxWgJobs);
  std::vector<int> cta_first(kMaxWgCtas + 1, 0);
  std::memset(jobs.data(), 0, sizeof(WgradJob) * kMaxWgJobs);
  plan_wgrad(&L, d->sm_count, jobs.data(), cta_first.data());
  CUDA_TRY(cudaMemcpyAsync(L.jobs_dev, jobs.data(), sizeof(WgradJob) * kMaxWgJobs, cudaMemcpyHostToDevice, stream),
           "job table upload");
  CUDA_TRY(cudaMemcpyAsync(L.cta_first_dev, cta_first.data(), sizeof(int) * (kMaxWgCtas + 1), cudaMemcpyHostToDevice, stream),
           "cta table upload");
  CUDA_TRY(cudaStreamSynchronize(stream), "workspace init sync");
  return 0;
}

int nerfb200_render_backward(const nerfb200_backward_args* b, void* stream_v) {
  if (!b || !b->render) return fail(NERFB200_EINVAL, "render_backward: NULL argument%s");
  const nerfb200_render_args* a = b->render;
  int rc = check_render_shapes(a);
  if (rc) return rc;
  if (a->n_rays == 0) return 0;
  if (!a->train_workspace || a->test_time) return fail(NERFB200_EINVAL, "render_backward needs the forward's train_workspace, test_time = 0%s");
  const bool fine = a->n_importance > 0;
  if (!b->params_coarse || !b->grads_coarse || (fine && (!b->params_fine || !b->grads_fine)))
    return fail(NERFB200_EINVAL, "render_backward: params / grads tables are NULL%s");
  for (int i = 0; i < kNumParams; ++i)
    if (!b->params_coarse[i] || !b->grads_coarse[i] || (fine && (!b->params_fine[i] || !b->grads_fine[i])))
      return fail(NERFB200_EINVAL, "render_backward: NULL parameter / gradient tensor%s");
  DeviceInfo* d = nullptr;
  rc = device_info(&d);
  if (rc) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  TrainLayout L;
  make_train_layout(&L, static_cast<uint8_t*>(a->train_workspace), a->n_rays, a->n_samples, a->n_importance, d->sm_count);
  const float* const* params[2] = {b->params_coarse, b->params_fine};
  float* const* grads[2] = {b->grads_coarse, b->grads_fine};
  const float* g_rgb[2] = {b->g_rgb_coarse, b->g_rgb_fine};
  const float* g_depth[2] = {b->g_depth_coarse, b->g_depth_fine};
  const float* g_opac[2] = {b->g_opacity_coarse, b->g_opacity_fine};
  const float* rgb_out[2] = {a->rgb_coarse, a->rgb_fine};
  const float* noise[2] = {a->noise_coarse, a->noise_fine};

  // 1. compositing backward -> per-sample d sigma / d rgb_pre
  for (int ps = 0; ps < L.n_pass; ++ps) {
    CompBwdParams cp;
    cp.n_rays = L.n_rays; cp.S = L.pass[ps].S; cp.n_pad = L.pass[ps].n_pad;
    cp.z = L.pass[ps].z; cp.sigma = L.pass[ps].sigma; cp.rgb = L.pass[ps].rgb;
    cp.rays = a->rays; cp.ray_stride = a->ray_stride;
    cp.noise = a->noise_std > 0.f ? noise[ps] : nullptr;
    cp.noise_std = a->noise_std; cp.white_back = a->white_back;
    cp.g_rgb = g_rgb[ps]; cp.g_depth = g_depth[ps]; cp.g_opac = g_opac[ps];
    cp.rgb_out = rgb_out[ps]; cp.target = b->target; cp.loss_grad = b->loss_grad;
    cp.dsigma = L.pass[ps].dsigma; cp.dprergb = L.pass[ps].dprergb;
    cp.amax_bits = L.amax + 2 * ps;
    cp.tile_amax = L.tile_amax[ps];
    composite_bwd_kernel<<<(L.n_rays + 3) / 4, 128, 0, stream>>>(cp);
    g_launches++;
  }
  ScaleParams sp;
  sp.n_pass = L.n_pass; sp.phase = 0;
  sp.amax = L.amax; sp.lamax = L.lamax; sp.lscale = L.lscale; sp.linv = L.linv;
  sp.wnorm = L.wnorm; sp.saturated = L.saturated;
  for (int ps = 0; ps < 2; ++ps) {
    const int q = ps < L.n_pass ? ps : 0;
    sp.w_rgb[ps] = params[q][22];
    sp.w_sigma[ps] = params[q][20];
  }
  bwd_scale_kernel<<<1, 128, 0, stream>>>(sp);
  g_launches++;
  // 2. rgb head, ReLU of the direction layer (both passes in one launch), direction part of gW_dir
  {
    HeadBwdParams hp;
    hp.n_rays = L.n_rays; hp.n_pass = L.n_pass;
    hp.pass[0] = L.pass[0]; hp.pass[1] = L.pass[1];
    hp.w_rgb[0] = params[0][22]; hp.w_rgb[1] = fine ? params[1][22] : params[0][22];
    hp.lscale = L.lscale;
    hp.rays = a->rays; hp.ray_stride = a->ray_stride;
    hp.raysum[0] = L.raysum[0]; hp.raysum[1] = L.raysum[1];
    hp.direnc = L.direnc;
    hp.part[0] = L.head_part[0]; hp.part[1] = L.head_part[1];
    head_bwd_kernel<<<L.head_grid, kHeadWarps * 32, 0, stream>>>(hp);
    g_launches++;
    DirGradParams dp;
    dp.n_rays = L.n_rays;
    dp.raysum[0] = L.raysum[0]; dp.raysum[1] = L.raysum[1];
    dp.direnc = L.direnc;
    dp.part[0] = L.dir_part[0]; dp.part[1] = L.dir_part[1];
    dir_grad_kernel<<<dim3(kDirSlices, L.n_pass), 128, 0, stream>>>(dp);
    g_launches++;
  }
  // 3. dgrad chain (tcgen05): a probe pass over one tile per SM (the largest of its stride class) measures the
  //    per-layer growth factors that pick the per-layer scales, then the real pass
  {
    ChainParams cp;
    cp.n_pass = L.n_pass;
    cp.pass[0] = L.pass[0]; cp.pass[1] = L.pass[1];
    cp.net[0] = static_cast<const uint8_t*>(a->packed_coarse);
    cp.net[1] = static_cast<const uint8_t*>(a->packed_fine);
    cp.lscale = L.lscale;
    cp.lamax = L.lamax;
    cp.status = d->status;
    const long long t0 = L.pass[0].n_pad / 128, t1 = fine ? L.pass[1].n_pad / 128 : 0;
    cp.pass_tiles[0] = t0; cp.pass_tiles[1] = t1;
    cp.tile_amax[0] = L.tile_amax[0]; cp.tile_amax[1] = L.tile_amax[1];
    cp.wnorm = L.wnorm;
    cp.saturated = L.saturated;
    if (!kBwdBf16) {
      const long long half = (d->sm_count + 1) / 2;
      cp.tiles[0] = fine ? (t0 < half ? t0 : half) : (t0 < d->sm_count ? t0 : d->sm_count);
      cp.tiles[1] = fine ? (t1 < half ? t1 : half) : 0;
      const int pc = static_cast<int>(cp.tiles[0] + cp.tiles[1]);
      chain_bwd_kernel<true><<<pc, kThreads, kChSmemTotal, stream>>>(cp);
      g_launches++;
      sp.phase = 1;
      bwd_scale_kernel<<<1, 128, 0, stream>>>(sp);
      g_launches++;
    }
    cp.tiles[0] = t0;
    cp.tiles[1] = t1;
    const long long total = t0 + t1;
    const int ctas = static_cast<int>(total < d->sm_count ? total : d->sm_count);
    chain_bwd_kernel<false><<<ctas, kThreads, kChSmemTotal, stream>>>(cp);
    g_launches++;
  }
  // 4. split-K wgrad (tcgen05)
  wgrad_kernel<<<L.n_cta, kWgThreads, kWgSmemTotal, stream>>>(L.jobs_dev, L.cta_first_dev,
                                                               static_cast<uint32_t>(env_switches().wg_copy),
                                                               env_switches().wg_exp, d->status);
  g_launches++;
  // 5. partial sums -> gradient tensors (fixed order), 6. unfold W'
  ReduceTable tab;
  tab.n = 0;
  auto add = [&](const float* part, long long stride, int n_split, float* out, const float* mul, int rows, int cols,
                 int part_ld, int out_ld, int out_col0, int transposed = 0) {
    ReduceItem& it = tab.it[tab.n++];
    it.part = part; it.split_stride = stride; it.n_split = n_split; it.out = out; it.mul = mul;
    it.rows = rows; it.cols = cols; it.part_ld = part_ld; it.out_ld = out_ld; it.out_col0 = out_col0;
    it.transposed = transposed;
    it.by_warp = (n_split >= 128 && rows * cols <= 4096) ? 1 : 0;
  };
  for (int ps = 0; ps < L.n_pass; ++ps) {
    const float* linv = L.linv + ps * kLevels;       // level v: 0 = dd, v = 1..8 = dpre_{9-v}
    auto slot = [&](int kind) { return L.wg_part + static_cast<size_t>(L.first_job[ps][kind]) * kWgSlotFloats; };
    auto ns = [&](int kind) { return L.n_split[ps][kind]; };
    float* const* g = grads[ps];
    add(slot(kJ1), kWgSlotFloats, ns(kJ1), g[0], linv + 8, 256, 63, 256, 63, 0, 1);
    add(slot(kJ1) + 65536, kWgSlotFloats, ns(kJ1), g[1], linv + 8, 1, 256, 256, 256, 0);
    const int hidden[6] = {kJ2, kJ3, kJ4, kJ6, kJ7, kJ8};
    const int layer[6] = {2, 3, 4, 6, 7, 8};
    for (int i = 0; i < 6; ++i) {
      const float* inv = linv + (9 - layer[i]);
      add(slot(hidden[i]), kWgSlotFloats, ns(hidden[i]), g[2 * (layer[i] - 1)], inv, 256, 256, 256, 256, 0, 1);
      add(slot(hidden[i]) + 65536, kWgSlotFloats, ns(hidden[i]), g[2 * (layer[i] - 1) + 1], inv, 1, 256, 256, 256, 0);
    }
    add(slot(kJ5a), kWgSlotFloats, ns(kJ5a), g[8], linv + 4, 256, 63, 256, 319, 0, 1);
    add(slot(kJ5b), kWgSlotFloats, ns(kJ5b), g[8], linv + 4, 256, 256, 256, 319, 63, 1);
    add(slot(kJ5a) + 65536, kWgSlotFloats, ns(kJ5a), g[9], linv + 4, 1, 256, 256, 256, 0);
    add(slot(kJ9), kWgSlotFloats, ns(kJ9), L.gWp[ps], linv, 128, 256, 128, 256, 0, 1);
    add(slot(kJ9) + 65536, kWgSlotFloats, ns(kJ9), L.gbp[ps], linv, 1, 128, 128, 128, 0);
    add(L.head_part[ps] + kHeadPartSigW, kHeadPartFloats, L.head_grid, g[20], nullptr, 1, 256, 256, 256, 0);
    add(L.head_part[ps] + kHeadPartSigB, kHeadPartFloats, L.head_grid, g[21], nullptr, 1, 1, 1, 1, 0);
    add(L.head_part[ps] + kHeadPartRgbW, kHeadPartFloats, L.head_grid, g[22], nullptr, 1, 384, 384, 384, 0);
    add(L.head_part[ps] + kHeadPartRgbB, kHeadPartFloats, L.head_grid, g[23], nullptr, 1, 3, 3, 3, 0);
    add(L.dir_part[ps], 128 * 27, kDirSlices, g[18], nullptr, 128, 27, 27, 283, 256);
  }
  wgrad_reduce_kernel<<<dim3(64, tab.n), 256, 0, stream>>>(tab);   // latency-bound: 64 blocks per item (16 measured 40 us)
  g_launches++;
  UnfoldParams up;
  for (int ps = 0; ps < 2; ++ps) {
    const int q = ps < L.n_pass ? ps : 0;
    up.gWp[ps] = L.gWp[q]; up.gbp[ps] = L.gbp[q];
    up.Wf[ps] = params[q][16]; up.bf[ps] = params[q][17]; up.Wd[ps] = params[q][18];
    up.gWd[ps] = grads[q][18]; up.gbd[ps] = grads[q][19]; up.gWf[ps] = grads[q][16]; up.gbf[ps] = grads[q][17];
  }
  // warps: one per gWd output (128 x 256), then one thread per gWf / gbf output
  unfold_kernel<<<dim3((128 * 256 + (256 * 256 + 256 + 31) / 32 + 7) / 8, L.n_pass), 256, 0, stream>>>(up);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "render_backward launches");
  return 0;
}

int nerfb200_train_saturation(const void* workspace, int64_t n_rays, int32_t n_samples, int32_t n_importance,
                              uint32_t* out, void* stream_v) {
  if (!workspace || !out || n_rays <= 0 || n_samples <= 0 || n_importance < 0)
    return fail(NERFB200_EINVAL, "train_saturation: bad argument%s");
  DeviceInfo* d = nullptr;
  int rc = device_info(&d);
  if (rc) return rc;
  TrainLayout L;
  make_train_layout(&L, static_cast<uint8_t*>(const_cast<void*>(workspace)), n_rays, n_samples, n_importance, d->sm_count);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CUDA_TRY(cudaMemcpyAsync(out, L.saturated, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream), "saturation copy");
  CUDA_TRY(cudaStreamSynchronize(stream), "saturation sync");
  if (L.n_pass < 2) out[1] = 0;
  return 0;
}

int nerfb200_adam_step(int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                       float* const* exp_avg_sq, const int64_t* numel, float lr, float beta1, float beta2, float eps,
                       float weight_decay, int64_t step, void* stream) {
  if (n_tensors < 0 || n_tensors > kAdamMaxTensors) return fail(NERFB200_EINVAL, "adam_step: at most 64 tensors per call%s");
  if (n_tensors == 0) return 0;
  if (!params || !grads || !exp_avg || !exp_avg_sq || !numel || step < 1)
    return fail(NERFB200_EINVAL, "adam_step: NULL argument / step < 1%s");
  AdamParams a;
  a.n_tensors = n_tensors;
  int blocks = 0;
  for (int i = 0; i < n_tensors; ++i) {
    if (!params[i] || !grads[i] || !exp_avg[i] || !exp_avg_sq[i] || numel[i] < 0 || numel[i] > 0x7fffffff)
      return fail(NERFB200_EINVAL, "adam_step: NULL tensor / bad size%s");
    a.p[i] = params[i]; a.g[i] = grads[i]; a.m[i] = exp_avg[i]; a.v[i] = exp_avg_sq[i];
    a.numel[i] = static_cast<int>(numel[i]);
    a.block0[i] = blocks;
    blocks += static_cast<int>((numel[i] + 1023) / 1024);
  }
  a.block0[n_tensors] = blocks;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay;
  a.bias1 = 1.f - std::pow(beta1, static_cast<float>(step));
  a.bias2_sqrt = std::sqrt(1.f - std::pow(beta2, static_cast<float>(step)));
  if (blocks == 0) return 0;
  adam_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "adam_step launch");
  return 0;
}

int nerfb200_check_status(void) {
  DeviceInfo* d = nullptr;
  int rc = device_info(&d);
  if (rc) return rc;
  return check_sticky_status(d);
}

#ifdef NERFB200_DIAG
// ---------------------------------------------------------------------------- diagnostics build
static int diag_attrs(DeviceInfo* di) {
  if (di->diag_attrs_set) return 0;
  CUDA_TRY(cudaFuncSetAttribute(gemm_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                static_cast<int>(kSmemTotal)), "smem attr probe");
  CUDA_TRY(cudaFuncSetAttribute(gemm_mn_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                static_cast<int>(kSmemTotal)), "smem attr mn probe");
  CUDA_TRY(cudaFuncSetAttribute(mma_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                static_cast<int>(kSmemTotal)), "smem attr bench");
  CUDA_TRY(cudaFuncSetAttribute(mma_contention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                static_cast<int>(kSmemTotal)), "smem attr contention");
  di->diag_attrs_set = true;
  return 0;
}

int nerfb200_debug_gemm_mn(const float* a, const float* b, int32_t lbo, int32_t sbo, int32_t fmt, float* d, void* stream) {
  if (!a || !b || !d) return fail(NERFB200_EINVAL, "debug_gemm_mn: NULL argument%s");
  DeviceInfo* di = nullptr;
  int rc = device_info(&di);
  if (rc) return rc;
  if ((rc = diag_attrs(di)) != 0) return rc;
  gemm_mn_probe_kernel<<<1, kThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(
      a, b, static_cast<uint32_t>(lbo), static_cast<uint32_t>(sbo), static_cast<uint32_t>(fmt), d, di->status);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "debug_gemm_mn launch");
  return 0;
}

int nerfb200_debug_timeline(int64_t* host_out, int64_t n_values) {
  DeviceInfo* di = nullptr;
  int rc = device_info(&di);
  if (rc) return rc;
  if (!di->timeline || !host_out) return fail(NERFB200_EINVAL, "debug_timeline: no timeline recorded%s");
  const int64_t cap = 3 * kTlMax * 2;
  CUDA_TRY(cudaDeviceSynchronize(), "timeline sync");
  CUDA_TRY(cudaMemcpy(host_out, di->timeline, sizeof(long long) * (n_values < cap ? n_values : cap),
                      cudaMemcpyDeviceToHost), "timeline copy");
  return 0;
}

int nerfb200_debug_mma_bench(int64_t* out_dev, int32_t n_ctas, int32_t reps, void* stream) {
  if (!out_dev || n_ctas < 1 || reps < 1) return fail(NERFB200_EINVAL, "debug_mma_bench: bad argument%s");
  DeviceInfo* di = nullptr;
  int rc = device_info(&di);
  if (rc) return rc;
  if ((rc = diag_attrs(di)) != 0) return rc;
  mma_bench_kernel<<<n_ctas, kThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<long long*>(out_dev), reps, di->status);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "debug_mma_bench launch");
  return 0;
}

int nerfb200_debug_mma_contention(int64_t* out_dev, int32_t n_ctas, int32_t reps, int32_t bg, int32_t variant,
                                  void* stream) {
  if (!out_dev || n_ctas < 1 || reps < 1) return fail(NERFB200_EINVAL, "debug_mma_contention: bad argument%s");
  DeviceInfo* di = nullptr;
  int rc = device_info(&di);
  if (rc) return rc;
  if ((rc = diag_attrs(di)) != 0) return rc;
  if (bg < 0) {     // issue-pattern benchmark: variant = mode, -bg - 1 = arg
    const int arg = -bg - 1;
    long long* o = reinterpret_cast<long long*>(out_dev);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define NERFB200_ISSUE_CASE(M)                                                                      \
  case M:                                                                                           \
    CUDA_TRY(cudaFuncSetAttribute(mma_issue_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                  static_cast<int>(kSmemTotal)), "smem attr issue");                \
    mma_issue_kernel<M><<<n_ctas, kThreads, kSmemTotal, st>>>(o, reps, arg, di->status);            \
    break;
    switch (variant) {
      NERFB200_ISSUE_CASE(0) NERFB200_ISSUE_CASE(1) NERFB200_ISSUE_CASE(2) NERFB200_ISSUE_CASE(3)
      NERFB200_ISSUE_CASE(4) NERFB200_ISSUE_CASE(5) NERFB200_ISSUE_CASE(6) NERFB200_ISSUE_CASE(7)
      NERFB200_ISSUE_CASE(8)
      default: return fail(NERFB200_EINVAL, "debug_mma_contention: bad issue mode%s");
    }
#undef NERFB200_ISSUE_CASE
  } else {
    mma_contention_kernel<<<n_ctas, kThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<long long*>(out_dev), reps, bg, variant, di->status);
  }
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "debug_mma_contention launch");
  return 0;
}

int nerfb200_debug_gemm(const float* a, const void* packed, int32_t slice, int32_t mode, float* d,
                        void* stream) {
  if (!a || !packed || !d) return fail(NERFB200_EINVAL, "debug_gemm: NULL argument%s");
  if (slice < 0 || slice >= kNumSlices256 + kNumSlices128) return fail(NERFB200_EINVAL, "debug_gemm: bad slice%s");
  DeviceInfo* di = nullptr;
  int rc = device_info(&di);
  if (rc) return rc;
  if ((rc = diag_attrs(di)) != 0) return rc;
  gemm_probe_kernel<<<1, kThreads, kSmemTotal, static_cast<cudaStream_t>(stream)>>>(
      a, static_cast<const uint8_t*>(packed), slice, mode, d, di->status);
  g_launches++;
  CUDA_TRY(cudaGetLastError(), "debug_gemm launch");
  return 0;
}

#endif  // NERFB200_DIAG

}  // extern "C"
