// libmbe.so -- C ABI (include/mbe.h) over the sm_100a kernels in mbe_step.cuh.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <initializer_list>
#include <memory>
#include <new>
#include <string>
#include <vector>

#include "../../include/mbe.h"
#include "mbe_step.cuh"
#include "mbe_step_spec.cuh"
#include "mbe_step_big.cuh"
#include "mbe_step_upt.cuh"
#include "mbe_step_tpe.cuh"
#include "mbe_render.cuh"
#include "mbe_evolve.cuh"
#include "mbe_map.cuh"

namespace {

thread_local std::string g_err;

int fail(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}

#define MBE_CUDA(expr)                                                                     \
  do {                                                                                     \
    cudaError_t e_ = (expr);                                                               \
    if (e_ != cudaSuccess) return fail("%s failed: %s", #expr, cudaGetErrorString(e_));    \
  } while (0)

// Makes the handle's device current for the duration of a call and restores the caller's device
// afterwards (a process may drive several devices / handles from one thread).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device) {
      err = cudaSetDevice(device);
      switched = err == cudaSuccess;
    }
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

#define MBE_ON_DEVICE(dev)                                                                          \
  DeviceGuard guard_(dev);                                                                          \
  if (guard_.err != cudaSuccess) return fail("cudaSetDevice(%d): %s", dev, cudaGetErrorString(guard_.err))

// One step-kernel launch: the kernel instance and everything launch() needs to run it.
struct StepKernel {
  void (*fn)(mbe::StepArgs) = nullptr;
  const char* name = "";     // what mbe_step_kernel_name reports
  int threads = 0, epb = 0;  // CTA size and envs per CTA (grid = ceil(E / epb))
  size_t smem = 0;           // dynamic shared memory per CTA
  bool pdl = false;          // launched with programmatic stream serialization
  bool whole_warps = false;  // thread per env: takes only E % 32 == 0 and 16-byte aligned buffers
  bool prefetch = false;     // prefetches state slices pf_dist CTAs ahead into L2
  int pf_dist = 0;           // (prefetch) set at create from the kernel's occupancy
  bool bound_ok = true;      // (whole_warps) the bound buffers are aligned; set by mbe_bind
};

}  // namespace

struct mbe_env {
  mbe_config cfg;
  mbe_buffers bufs;
  bool bound = false;
  mbe::StepArgs args;
  std::vector<void*> luts;  // device tables owned by the handle
  int64_t launches = 0;
  // general: the generic or the block-per-env kernel, which serves every op.  steps: the whole-step
  // kernels of this shape in priority order (see pick).  episode: the fused rollout (fn == nullptr: none).
  StepKernel general, episode;
  std::vector<StepKernel> steps;
  uint32_t bound_xy[mbe::kMapMaxB] = {};  // a shared layout as mbe_bind read it (int16 pairs), for layout maps
  bool prefetch_ok = false;  // the prefetched streams (pos, wp, conn, actions) are 16-byte aligned
  // mbe_step_host pipeline: second stream + fork/join events (created on first use)
  cudaStream_t host_stream = nullptr;
  cudaEvent_t host_fork = nullptr, host_join = nullptr;

  template <class F>
  void each_kernel(F f) {
    f(general);
    for (StepKernel& k : steps) f(k);
    if (episode.fn) f(episode);
  }
};

namespace {

// wide shapes and the schedulers other than ResourceFair run on the block-per-env kernel alone
bool block_per_env(const mbe_config& c) {
  return c.num_ues > 32 || c.num_bs > 32 || c.scheduler != MBE_SCHED_RESOURCE_FAIR;
}

bool aligned16(std::initializer_list<const void*> ptrs) {
  uintptr_t all = 0;
  for (const void* p : ptrs) all |= (uintptr_t)p;
  return (all & 15) == 0;
}

// Copies count host elements into a new device table that the handle owns (freed by mbe_destroy).
template <class T>
cudaError_t upload(mbe_env* env, const T* src, size_t count, T*& dst) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, count * sizeof(T));
  if (e != cudaSuccess) return e;
  env->luts.push_back(p);
  dst = static_cast<T*>(p);
  return cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice);
}

// The kernel that runs a launch of E envs: the first whole-step kernel that accepts it, else the
// general one (reset, observe, the split phases and the debug SNR output only exist there).  A window
// that is not a whole number of 32-env warps passes over the thread-per-env kernel to the warp-segment
// kernel, which handles ragged tails.
const StepKernel& pick(const mbe_env* env, int op, int phases, int E, bool dbg_snr) {
  if (op == mbe::OP_STEP && phases == MBE_PHASE_ALL && !dbg_snr)
    for (const StepKernel& k : env->steps)
      if (k.bound_ok && (!k.whole_warps || E % 32 == 0)) return k;
  return env->general;
}

// Launches k over the a.E envs of a on stream.
int run(mbe_env* env, const StepKernel& k, mbe::StepArgs a, void* stream) {
  a.epb = k.epb;  // envs per CTA of this mapping (bounds and size of the obs bulk store)
  a.pf_dist = env->prefetch_ok ? k.pf_dist : 0;
  cudaLaunchConfig_t lc = {};
  lc.gridDim = dim3((a.E + k.epb - 1) / k.epb);
  lc.blockDim = dim3(k.threads);
  lc.dynamicSmemBytes = k.smem;
  lc.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute pdl;
  pdl.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  pdl.val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = &pdl;
  lc.numAttrs = k.pdl ? 1 : 0;
  MBE_CUDA(cudaLaunchKernelEx(&lc, k.fn, a));
  env->launches += 1;
  return 0;
}

// One compiled whole-step or fused-episode instance, the handles it serves (mode, handler: any in FORK mode,
// U, B, BS layout, several BS classes or one) and its launch record, read from the kernel's header.
// k.whole_warps also limits it to E % 32 == 0 and a map of at most 2048 x 2048 (packed nearest-BS key).
struct Instance {
  int mode, handler, U, B;
  bool per_env, multi_class;
  bool episode;  // the fused episode of mbe_rollout, else a whole step
  StepKernel k;
};

// Programmatic dependent launch (the next step's CTAs become resident while this grid drains and
// prefetch their state slices into L2 before the dependency wait).  Measured on B200
// (profiles/README.md): 3-7% (graph replay) to 10% (plain launches) faster for the medium GYM
// kernels, 14% for the small shape, neutral for the large one, 2% slower for the FORK kernels (no
// prefetch there) -> on for the GYM step kernels only.
template <int MODE, int HANDLER, int U, int B, bool PER_ENV, bool MC>
constexpr Instance spec() {
  using L = mbe::SpecLayout<MODE, HANDLER, U, B, PER_ENV>;
  return {MODE, HANDLER, U, B, PER_ENV, MC, false,
          {mbe::step_spec_kernel<MODE, HANDLER, U, B, PER_ENV, MC>, "step_spec_kernel", mbe::kThreads, L::EPB, L::BYTES,
           /*pdl=*/MODE == MBE_MODE_GYM, /*whole_warps=*/false, /*prefetch=*/true}};
}
template <int HANDLER, int U, int B, int K>
constexpr Instance upt() {
  using L = mbe::UptLayout<HANDLER, U, B, K>;
  return {MBE_MODE_GYM, HANDLER, U, B, false, false, false,
          {mbe::step_upt_kernel<HANDLER, U, B, K>, "step_upt_kernel", mbe::kUptThreads, L::EPB, L::BYTES,
           /*pdl=*/true, /*whole_warps=*/false, /*prefetch=*/true}};
}
template <int U, int B, bool ROLLOUT, bool SHARED>
constexpr Instance tpe() {
  return {MBE_MODE_FORK, 0, U, B, !SHARED, false, ROLLOUT,
          {mbe::step_tpe_fork_kernel<U, B, ROLLOUT, SHARED>, "step_tpe_fork_kernel", mbe::kTpeThreads,
           mbe::kTpeEnvsPerCta, sizeof(mbe::TpeSmem<U, B, ROLLOUT>), /*pdl=*/false, /*whole_warps=*/true}};
}

// Every compiled instance.  A handle's whole-step kernels are the matching step rows in this order,
// which is their priority (see pick): thread per env, UEs per thread, warp segment.  Shapes: the
// scenario sizes of BASELINE.json (small 5 x 3, medium 15 x 4, large 30 x 13) and the fork's MComCustom
// (7 UEs, <= 10 random BSs per env).
constexpr Instance kInstances[] = {
    // thread per env <U, B, fused episode, shared layout>: MComCustom's FORK step and fused episode.  The
    // scenario shapes in FORK mode have the fused episode only; their single step stays on the warp-segment
    // kernel.  A fused 30 x 13 episode (one env per lane walking 30 x 13 pairs in scalar code at 208
    // registers) took 1.43 ms per 20-step episode of 65,536 envs against 0.83 ms for 20 launches of the
    // warp-segment kernel (profiles/r02_j_fork_rollout.txt); the small and medium shapes win 7.1x and 1.8x.
    tpe<7, 10, false, false>(), tpe<7, 10, true, false>(), tpe<5, 3, true, true>(), tpe<15, 4, true, true>(),
    // UEs per thread <handler, U, B, K>: the shared 15 x 4 GYM layout with one BS class, which therefore
    // has no one-class warp-segment instance (small 5 x 3 with K = 1 and large 30 x 13 with K = 10 were
    // measured slower than one thread per UE)
    upt<0, 15, 4, 5>(), upt<1, 15, 4, 5>(),
    // warp segment <mode, handler, U, B, per-env layout, several BS classes>
    spec<1, 0, 5, 3, false, false>(), spec<1, 1, 5, 3, false, false>(), spec<1, 0, 5, 3, false, true>(),
    spec<1, 1, 5, 3, false, true>(), spec<1, 0, 15, 4, false, true>(), spec<1, 1, 15, 4, false, true>(),
    spec<1, 0, 30, 13, false, false>(), spec<1, 1, 30, 13, false, false>(), spec<1, 0, 30, 13, false, true>(),
    spec<1, 1, 30, 13, false, true>(), spec<1, 0, 7, 10, true, false>(), spec<1, 1, 7, 10, true, false>(),
    spec<0, 0, 5, 3, false, false>(), spec<0, 0, 5, 3, false, true>(), spec<0, 0, 15, 4, false, false>(),
    spec<0, 0, 15, 4, false, true>(), spec<0, 0, 30, 13, false, false>(), spec<0, 0, 30, 13, false, true>(),
    spec<0, 0, 7, 10, true, false>(),
};

// mbe_step_host starts its env windows at multiples of kAlign envs: a multiple of 32 (16-byte aligned
// slices) and of every instance's envs per CTA.  The generic kernel's 4 * floor(32 / U) envs per CTA need
// not divide it (40 at U = 3): a window is a launch of its own, so only its last CTA may be partial.
constexpr int kAlign = 384;
static_assert([] {
  for (const Instance& r : kInstances)
    if (kAlign % r.k.epb) return false;
  return kAlign % 32 == 0;
}(), "kAlign must be a multiple of 32 and of every instance's envs per CTA");

}  // namespace

extern "C" {

int mbe_abi_version(void) { return MBE_ABI_VERSION; }

const char* mbe_build_info(void) {
#define MBE_STR2(x) #x
#define MBE_STR(x) MBE_STR2(x)
  return "libmbe abi " MBE_STR(MBE_ABI_VERSION) " | sm_100a | built " __DATE__ " " __TIME__;
}

int mbe_struct_size(int which) {
  switch (which) {
    case 0: return (int)sizeof(mbe_config);
    case 1: return (int)sizeof(mbe_buffers);
    case 2: return (int)sizeof(mbe_link_class);
    case 3: return (int)sizeof(mbe_ue_class);
    case 4: return (int)sizeof(mbe_rollout_out);
    case 5: return (int)sizeof(mbe_render_style);
    case 6: return (int)sizeof(mbe_evolve_params);
    case 7: return (int)sizeof(mbe_map_params);
    default: return -1;
  }
}

const char* mbe_last_error(void) { return g_err.c_str(); }

int mbe_create(const mbe_config* cfg, mbe_env** out) {
  if (!cfg || !out) return fail("mbe_create: null argument");
  *out = nullptr;
  if (cfg->abi_version != MBE_ABI_VERSION)
    return fail("mbe_create: abi_version %d, library is %d", cfg->abi_version, MBE_ABI_VERSION);
  if (cfg->num_envs <= 0) return fail("mbe_create: num_envs must be > 0");
  if (cfg->num_ues <= 0 || cfg->num_ues > mbe::kBigMaxI * mbe::kBigThreads)
    return fail("mbe_create: num_ues=%d out of range (1..%d)", cfg->num_ues, mbe::kBigMaxI * mbe::kBigThreads);
  if (cfg->num_bs <= 0 || cfg->num_bs > mbe::kBigMaxB)
    return fail("mbe_create: num_bs=%d out of range (1..%d)", cfg->num_bs, mbe::kBigMaxB);
  if (cfg->mode != MBE_MODE_FORK && cfg->mode != MBE_MODE_GYM) return fail("mbe_create: bad mode %d", cfg->mode);
  if (cfg->handler != MBE_HANDLER_CENTRAL && cfg->handler != MBE_HANDLER_MA)
    return fail("mbe_create: bad handler %d", cfg->handler);
  if (cfg->scheduler != MBE_SCHED_RESOURCE_FAIR && cfg->scheduler != MBE_SCHED_PROPORTIONAL_FAIR &&
      cfg->scheduler != MBE_SCHED_RATE_FAIR)
    return fail("mbe_create: scheduler %d not available", cfg->scheduler);
  const int nuc = cfg->num_ue_classes > 1 ? cfg->num_ue_classes : 1;
  if (nuc > MBE_MAX_UE_CLASSES) return fail("mbe_create: num_ue_classes=%d out of range", cfg->num_ue_classes);
  if (nuc > 1 && !cfg->ue_class) return fail("mbe_create: num_ue_classes > 1 needs ue_class");
  if (cfg->num_classes < 1 || cfg->num_classes * nuc > MBE_MAX_CLASSES)
    return fail("mbe_create: %d BS classes x %d UE classes exceed %d link classes", cfg->num_classes, nuc,
                MBE_MAX_CLASSES);
  const int nlink = cfg->num_classes * nuc;
  if (!(cfg->width > 0 && cfg->width <= 32767 && cfg->height > 0 && cfg->height <= 32767))
    return fail("mbe_create: map %gx%g does not fit int16 coordinates", cfg->width, cfg->height);
  if (cfg->ep_time <= 0) return fail("mbe_create: ep_time must be > 0");
  if (cfg->bs_random_max > 0 &&
      (cfg->bs_layout != MBE_BS_PER_ENV || cfg->bs_random_min < 1 || cfg->bs_random_max > cfg->num_bs ||
       cfg->bs_random_min > cfg->bs_random_max))
    return fail("mbe_create: random BS layouts need bs_layout=PER_ENV and 1 <= min <= max <= num_bs");
  if (!(cfg->util_upper > cfg->util_lower) || !(cfg->util_w3 > 0) || cfg->util_w3 == 1.0)
    return fail("mbe_create: bad utility parameters");
  for (int c = 0; c < nlink; ++c) {
    if (cfg->classes[c].d2max >= 0 && !cfg->classes[c].rate_lut)
      return fail("mbe_create: link class %d has no rate_lut", c);
    if (cfg->classes[c].log2snr_lut && cfg->classes[c].log2snr_len <= 0)
      return fail("mbe_create: link class %d: log2snr_lut needs log2snr_len > 0", c);
  }
  if (nuc > 1)
    for (int u = 0; u < cfg->num_ues; ++u)
      if (cfg->ue_class[u] >= nuc) return fail("mbe_create: ue_class[%d]=%d >= num_ue_classes", u, cfg->ue_class[u]);

  if (cfg->env_offset < 0 || cfg->env_offset + (int64_t)cfg->num_envs > (int64_t)0xffffffffll)
    return fail("mbe_create: env_offset + num_envs must stay below 2^32 (global env ids are 32-bit Philox counter words)");
  const int M = cfg->num_trajectories;
  if (M < 0) return fail("mbe_create: num_trajectories=%d must be >= 0", M);
  if (M >= 2) {
    if (!(cfg->flags & MBE_FLAG_SHARED_TRAJECTORY))
      return fail("mbe_create: num_trajectories=%d needs MBE_FLAG_SHARED_TRAJECTORY", M);
    if (M & (M - 1)) return fail("mbe_create: num_trajectories=%d must be a power of two", M);
    if (M > cfg->num_envs) return fail("mbe_create: num_trajectories=%d exceeds num_envs=%d", M, cfg->num_envs);
    if (cfg->num_envs % M)
      return fail("mbe_create: num_envs=%d must be a multiple of num_trajectories=%d", cfg->num_envs, M);
    if (cfg->env_offset % M)
      return fail("mbe_create: env_offset=%lld must be a multiple of num_trajectories=%d",
                  (long long)cfg->env_offset, M);
  }
  MBE_ON_DEVICE(cfg->device);
  mbe_env* env = new (std::nothrow) mbe_env();
  if (!env) return fail("mbe_create: out of host memory");
  std::unique_ptr<mbe_env, void (*)(mbe_env*)> owned(env, mbe_destroy);  // released on success only
  env->cfg = *cfg;
  std::memset(&env->bufs, 0, sizeof env->bufs);
  mbe::StepArgs& a = env->args;
  std::memset(&a, 0, sizeof a);
  a.E = cfg->num_envs;
  a.U = cfg->num_ues;
  a.B = cfg->num_bs;
  const bool gym = cfg->mode == MBE_MODE_GYM, ma = cfg->handler == MBE_HANDLER_MA;
  const bool big = block_per_env(*cfg);
  a.scheduler = cfg->scheduler;
  a.F = gym ? (ma ? 4 * a.B + 1 : 2 * a.B + 1) : 0;
  a.epw = big ? 1 : mbe::envs_per_warp(a.U);  // the generic kernel's warp-segment mapping
  a.epb = big ? 1 : mbe::segment_envs_per_cta(a.U);
  a.env_offset = (unsigned)cfg->env_offset;
  // shared trajectories: env g follows trajectory g & (M - 1), so M = 0 or 1 keeps trajectory 0 for all
  a.traj_gid_mask = (cfg->flags & MBE_FLAG_SHARED_TRAJECTORY) ? (M >= 2 ? (unsigned)(M - 1) : 0u) : 0xffffffffu;
  a.ep_time = cfg->ep_time;
  a.autoreset = cfg->autoreset;
  a.reset_rng_episode = cfg->reset_rng_episode;
  a.bs_per_env = cfg->bs_layout == MBE_BS_PER_ENV;
  a.bs_rand_min = cfg->bs_random_min;
  a.bs_rand_max = cfg->bs_random_max;
  a.seed_lo = (unsigned)(cfg->seed & 0xffffffffu);
  a.seed_hi = (unsigned)(cfg->seed >> 32);
  a.width = cfg->width;
  a.height = cfg->height;
  a.wh_int = (cfg->width == std::floor(cfg->width) && cfg->height == std::floor(cfg->height)) ? 1 : 0;
  a.wh_int_w = (int)cfg->width;
  a.wh_int_h = (int)cfg->height;
  for (int c = 0; c < nuc; ++c) {
    const double vel = nuc > 1 ? cfg->ue_classes[c].velocity : cfg->velocity;
    mbe::MoveDev& m = a.mv[c];
    m.velocity = vel;
    m.velocity_f = (float)vel;
    m.tie_eps = (float)(vel * 1e-6 + 1e-6);
    m.move_d2max = nuc > 1 ? cfg->ue_classes[c].move_d2max : cfg->move_d2max;
    // is an axis-aligned step exactly +-velocity in the reference's FP64 chain (movement.py:58-59)?
    volatile double v = vel;
    int ok = 1;
    const int dmax = (int)std::max(cfg->width, cfg->height) + 1;
    for (int d = 1; d <= dmax && ok; ++d) {
      volatile double prod = v * (double)d;
      volatile double q = prod / (double)d;
      if (q != v) ok = 0;
    }
    m.axis_exact = ok;
  }
  a.util_c = (float)(cfg->util_w1 * std::log(2.0) / std::log(cfg->util_w3));
  a.util_w2 = (float)cfg->util_w2;
  a.util_lo = (float)cfg->util_lower;
  a.util_hi = (float)cfg->util_upper;
  a.util_scale = (float)(2.0 / (cfg->util_upper - cfg->util_lower));
  a.inv_U = 1.0f / (float)a.U;
  a.n_classes = cfg->num_classes;
  a.n_ue_classes = nuc;
  bool any_ltab = false;
  for (int c = 0; c < nlink; ++c) {
    const mbe_link_class& h = cfg->classes[c];
    mbe::ClassDev& d = a.cls[c];
    d.l0_hi = (float)h.l0;
    d.l0_lo = (float)(h.l0 - (double)d.l0_hi);
    d.k_hi = (float)h.k;
    d.k_lo = (float)(h.k - (double)d.k_hi);
    d.l_zero = (float)h.l_zero;
    d.d2max = h.d2max;
    d.stride = h.d2max + 1;
    d.lutn = nullptr;
    d.lut0 = nullptr;
    d.ltab = nullptr;
    d.ltab_len = 0;
    if (h.log2snr_lut) {  // log2 snr per d2 (loss not affine in log-distance)
      float* pt = nullptr;
      if (cudaError_t e = upload(env, h.log2snr_lut, (size_t)h.log2snr_len, pt))
        return fail("mbe_create: log2snr_lut upload failed: %s", cudaGetErrorString(e));
      d.ltab = pt;
      d.ltab_len = h.log2snr_len;
      any_ltab = true;
    }
    if (h.d2max >= 0) {  // the raw table, for the block-per-env kernel
      double* p0 = nullptr;
      if (cudaError_t e = upload(env, h.rate_lut, (size_t)d.stride, p0))
        return fail("mbe_create: rate_lut upload failed: %s", cudaGetErrorString(e));
      d.lut0 = p0;
    }
    if (h.d2max >= 0 && !big) {
      // device table: [0] = 0.0, then rows n = 1..U of round(rate_lut[d2] / n, 2) in FP64
      // (schedules.py:20-22, base.py:435); kernels index it as lutn[n*stride + d2]
      const int rows = a.U;
      std::vector<double> tab((size_t)rows * d.stride + 1);
      tab[0] = 0.0;
      for (int n = 1; n <= rows; ++n)
        for (int i = 0; i < d.stride; ++i) {
          volatile double share = h.rate_lut[i] / (double)n;
          volatile double scaled = share * 100.0;
          tab[1 + (size_t)(n - 1) * d.stride + i] = std::nearbyint(scaled) / 100.0;
        }
      double* p = nullptr;
      if (cudaError_t e = upload(env, tab.data(), tab.size(), p))
        return fail("mbe_create: rate table upload failed: %s", cudaGetErrorString(e));
      d.lutn = p + 1 - d.stride;  // biased: row n starts at lutn + n*stride, lutn[stride-1] == 0.0
    }
  }
  if (cfg->bs_class) {
    for (int b = 0; b < cfg->num_bs; ++b)
      if (cfg->bs_class[b] >= cfg->num_classes)
        return fail("mbe_create: bs_class[%d]=%d >= num_classes", b, cfg->bs_class[b]);
    uint8_t* p = nullptr;
    if (cudaError_t e = upload(env, cfg->bs_class, (size_t)cfg->num_bs, p))
      return fail("mbe_create: bs_class upload failed: %s", cudaGetErrorString(e));
    a.bs_class = p;
  }
  if (nuc > 1) {
    uint8_t* p = nullptr;
    if (cudaError_t e = upload(env, cfg->ue_class, (size_t)cfg->num_ues, p))
      return fail("mbe_create: ue_class upload failed: %s", cudaGetErrorString(e));
    a.ue_class = p;
  }
  for (int b = 0; b < mbe::kMaxSlots; ++b) {
    const int c = (cfg->bs_class && b < cfg->num_bs) ? cfg->bs_class[b] : 0;
    const mbe::ClassDev& d = a.cls[c * nuc];  // (the slot table serves the one-UE-class kernels)
    mbe::SlotDev& sl = a.slot[b];
    sl.x = sl.y = 0;  // coordinates of a shared layout arrive with mbe_bind (host copy of bs_xy)
    sl.d2max = d.d2max;
    sl.stride = d.stride;
    sl.k = d.k_hi;
    sl.l0 = d.l0_hi;
    sl.xf = sl.yf = 0.0f;
    sl.lutn = d.lutn;
  }
  // the specialised kernels assume one UE class, log2 snr affine in log-distance and squared
  // distances exact in FP32; the warp-segment ones take per-BS classes (folded per slot), the
  // UEs-per-thread and thread-per-env ones a single class
  const bool d2_exact =
      std::floor(cfg->width) * std::floor(cfg->width) + std::floor(cfg->height) * std::floor(cfg->height) < 16777216.0;
  const bool spec_ok = nuc == 1 && !any_ltab && d2_exact;
  if (big && !d2_exact)
    return fail("mbe_create: the block-per-env kernel (wide shapes, ProportionalFair / RateFair) needs a map whose "
                "squared diagonal is below 2^24 (distances are exact FP32 integers)");
  const size_t smem = big ? 0 : mbe::smem_bytes(gym, ma, a.epb, a.U, a.B, a.F, a.bs_per_env);
  if (smem > 200 * 1024) return fail("mbe_create: needs %zu bytes of shared memory per block", smem);
  if (big) {
    // UEs per thread held in registers: 2 (64 registers, 4 CTAs per SM) up to 512 UEs, else 4 (80 registers,
    // 3 CTAs per SM).  With the observation rows leaving as aligned bulk tiles the 2-UEs-per-thread instance
    // is the faster one where both fit: 802 vs 920 us per 16,384-env synthetic step
    // (profiles/r02_zb_variants.txt); while the rows were direct 4-byte stores it was the slower one
    // (1105 vs 1046 us, r02_q): more resident CTAs only meant more contention on misaligned sectors
    const bool two = a.U <= 2 * mbe::kBigThreads;
    auto fn = gym ? (ma ? (two ? mbe::step_big_kernel<1, 1, 2> : mbe::step_big_kernel<1, 1, 4>)
                        : (two ? mbe::step_big_kernel<1, 0, 2> : mbe::step_big_kernel<1, 0, 4>))
                  : (two ? mbe::step_big_kernel<0, 0, 2> : mbe::step_big_kernel<0, 0, 4>);
    env->general = StepKernel{fn, "step_big_kernel", mbe::kBigThreads, 1,
                              two ? mbe::big_smem_bytes<2>() : mbe::big_smem_bytes<4>()};
  } else {
    auto fn = gym ? (ma ? mbe::step_kernel<1, 1> : mbe::step_kernel<1, 0>) : mbe::step_kernel<0, 0>;
    env->general = StepKernel{fn, "step_kernel", mbe::kThreads, a.epb, smem};
  }
  if (!big && spec_ok && !(cfg->flags & MBE_FLAG_GENERIC_KERNEL)) {
    const bool whole_warps = a.E % 32 == 0 && cfg->width <= 2048 && cfg->height <= 2048;
    for (const Instance& r : kInstances)
      if (r.mode == cfg->mode && (!gym || r.handler == cfg->handler) && r.U == a.U && r.B == a.B &&
          r.per_env == (a.bs_per_env != 0) && r.multi_class == (cfg->num_classes > 1) &&
          (!r.k.whole_warps || whole_warps)) {
        if (r.episode)
          env->episode = r.k;
        else
          env->steps.push_back(r.k);
      }
  }
  // L2 prefetch distance: 0.75 waves of resident CTAs (measured best of 0.25 .. 2 waves on B200,
  // profiles/README.md)
  int sms = 0;
  cudaError_t e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
  env->each_kernel([&](StepKernel& k) {
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute((const void*)k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem);
    if (!k.prefetch) return;
    int per_sm = 0;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k.fn, k.threads, k.smem);
    k.pf_dist = per_sm * sms * 3 / 4;
  });
  if (e != cudaSuccess)
    return fail("mbe_create: cudaFuncSetAttribute(%zu B smem): %s", smem, cudaGetErrorString(e));
  *out = owned.release();
  return 0;
}

void mbe_destroy(mbe_env* env) {
  if (!env) return;
  for (void* p : env->luts) cudaFree(p);
  if (env->host_stream) cudaStreamDestroy(env->host_stream);
  if (env->host_fork) cudaEventDestroy(env->host_fork);
  if (env->host_join) cudaEventDestroy(env->host_join);
  delete env;
}

int mbe_bind(mbe_env* env, const mbe_buffers* b) {
  if (!env || !b) return fail("mbe_bind: null argument");
  MBE_ON_DEVICE(env->cfg.device);
  const bool gym = env->cfg.mode == MBE_MODE_GYM;
  if (!b->pos || !b->wp || !b->t || !b->episode || !b->bs_xy || !b->utility || !b->done)
    return fail("mbe_bind: pos, wp, t, episode, bs_xy, utility and done are required");
  if (gym && (!b->conn || !b->actions || !b->obs || !b->reward))
    return fail("mbe_bind: GYM mode needs conn, actions, obs and reward");
  if (!gym && !b->assoc) return fail("mbe_bind: FORK mode needs assoc");
  if (env->cfg.bs_random_max > 0 && !b->nbs) return fail("mbe_bind: random BS layouts need nbs");
  if (b->inj_wp && (!b->wp_cnt || b->inj_k <= 0)) return fail("mbe_bind: inj_wp needs wp_cnt and inj_k > 0");
  if (((uintptr_t)b->pos | (uintptr_t)b->wp | (uintptr_t)b->bs_xy | (uintptr_t)b->inj_wp) & 3)
    return fail("mbe_bind: int16 pair buffers must be 4-byte aligned");
  if (b->metrics && ((uintptr_t)b->metrics & 15)) return fail("mbe_bind: metrics must be 16-byte aligned");
  if (b->rate && ((uintptr_t)b->rate & 7)) return fail("mbe_bind: rate must be 8-byte aligned");
  env->bufs = *b;
  mbe::StepArgs& a = env->args;
  a.pos = reinterpret_cast<uint32_t*>(b->pos);
  a.wp = reinterpret_cast<uint32_t*>(b->wp);
  a.t = b->t;
  a.episode = b->episode;
  a.bs_xy = reinterpret_cast<uint32_t*>(b->bs_xy);
  a.nbs = b->nbs;
  a.conn = b->conn;
  a.assoc = b->assoc;
  a.actions = b->actions;
  a.rate = b->rate;
  a.utility = b->utility;
  a.obs = b->obs;
  a.reward = b->reward;
  a.done = b->done;
  a.metrics = b->metrics;
  a.dbg_snr = b->dbg_snr;
  a.inj_wp = reinterpret_cast<const uint32_t*>(b->inj_wp);
  a.wp_cnt = b->wp_cnt;
  a.inj_k = b->inj_k;
  a.obs_bulk_ok = b->obs && (((uintptr_t)b->obs & 15) == 0);
  // the thread-per-env kernels move their streams by bulk async copies, which need 16-byte aligned global
  // addresses; with a per-env layout they also read its BS table and nbs
  const bool tpe_ok =
      a.bs_per_env ? aligned16({b->pos, b->wp, b->t, b->episode, b->bs_xy, b->nbs, b->assoc, b->rate, b->utility,
                                b->done, b->metrics}) && b->nbs != nullptr
                   : aligned16({b->pos, b->wp, b->t, b->episode, b->assoc, b->rate, b->utility, b->done, b->metrics});
  env->each_kernel([&](StepKernel& k) { k.bound_ok = !k.whole_warps || tpe_ok; });
  env->prefetch_ok = aligned16({b->pos, b->wp, b->conn, b->actions});
  if (!a.bs_per_env) {
    // a shared layout is constant for the life of the binding: fold the coordinates into the
    // kernel parameters (constant bank) for the specialised kernels
    int16_t xy[2 * mbe::kBigMaxB];
    MBE_CUDA(cudaMemcpy(xy, b->bs_xy, sizeof(int16_t) * 2 * a.B, cudaMemcpyDeviceToHost));
    for (int i = 0; i < a.B && i < mbe::kMaxSlots; ++i) {
      a.slot[i].x = xy[2 * i];
      a.slot[i].y = xy[2 * i + 1];
      a.slot[i].xf = (float)xy[2 * i];
      a.slot[i].yf = (float)xy[2 * i + 1];
    }
    for (int i = 0; i < a.B; ++i) env->bound_xy[i] = (uint16_t)xy[2 * i] | ((uint32_t)(uint16_t)xy[2 * i + 1] << 16);
  }
  env->bound = true;
  return 0;
}

// Restricts the launch arguments to the env window [first, first + count): every stream is
// env-major, so a window is a pointer shift; Philox counters keep using the global env id.
static void shift_window(mbe::StepArgs& a, bool ma, size_t first, int count) {
  const size_t U = a.U, MW = (a.B + 31) >> 5;
  auto adv = [&](auto*& p, size_t n) {
    if (p) p += n;
  };
  adv(a.pos, first * U);
  adv(a.wp, first * U);
  adv(a.t, first);
  adv(a.episode, first);
  if (a.bs_per_env) adv(a.bs_xy, first * a.B);
  adv(a.nbs, first);
  adv(a.conn, first * U * MW);
  adv(a.assoc, first * U);
  adv(a.actions, first * U);
  adv(a.rate, first * U);
  adv(a.utility, first * U);
  adv(a.obs, first * U * a.F);
  adv(a.reward, ma ? first * U : first);
  adv(a.done, first);
  adv(a.metrics, first * 4);
  adv(a.dbg_snr, first * U * a.B);
  adv(a.inj_wp, first * U * (size_t)a.inj_k);
  adv(a.wp_cnt, first * U);
  a.env_offset += (unsigned)first;
  a.E = count;
}

// window_count == 0: all envs; otherwise the full step of envs [window_first, +window_count)
// (window_first a multiple of 32 keeps every bulk-copy address 16-byte aligned)
static int launch(mbe_env* env, int op, int phases, const uint8_t* mask, void* stream, size_t window_first = 0,
                  int window_count = 0) {
  if (!env) return fail("null handle");
  if (!env->bound) return fail("mbe_bind has not been called");
  MBE_ON_DEVICE(env->cfg.device);
  mbe::StepArgs a = env->args;
  a.op = op;
  a.phases = phases;
  a.reset_mask = mask;
  if (window_count > 0)
    shift_window(a, env->cfg.handler == MBE_HANDLER_MA && env->cfg.mode == MBE_MODE_GYM, window_first, window_count);
  return run(env, pick(env, op, phases, a.E, a.dbg_snr != nullptr), a, stream);
}

int mbe_reset(mbe_env* env, const uint8_t* env_mask, void* stream) {
  return launch(env, mbe::OP_RESET, 0, env_mask, stream);
}

int mbe_step(mbe_env* env, void* stream) { return launch(env, mbe::OP_STEP, MBE_PHASE_ALL, nullptr, stream); }

int mbe_step_window(mbe_env* env, int first_env, int num_envs, void* stream) {
  if (!env) return fail("null handle");
  if (first_env < 0 || num_envs <= 0 || (long long)first_env + num_envs > env->cfg.num_envs)
    return fail("mbe_step_window: window [%d, +%d) outside 0..%d", first_env, num_envs, env->cfg.num_envs);
  if (first_env % 32) return fail("mbe_step_window: first_env must be a multiple of 32 (16-byte aligned slices)");
  return launch(env, mbe::OP_STEP, MBE_PHASE_ALL, nullptr, stream, (size_t)first_env, num_envs);
}

int mbe_stage(mbe_env* env, int phase_mask, void* stream) {
  if (phase_mask <= 0 || phase_mask > MBE_PHASE_ALL) return fail("mbe_stage: bad phase mask %d", phase_mask);
  return launch(env, mbe::OP_STEP, phase_mask, nullptr, stream);
}

int mbe_observe(mbe_env* env, void* stream) {
  if (env && env->cfg.mode != MBE_MODE_GYM) return fail("mbe_observe: GYM mode only");
  return launch(env, mbe::OP_OBSERVE, 0, nullptr, stream);
}

int mbe_channel(mbe_env* env, float* out_snr, uint32_t* out_elig, void* stream) {
  if (!env) return fail("null handle");
  if (!env->bound) return fail("mbe_bind has not been called");
  MBE_ON_DEVICE(env->cfg.device);
  const mbe::StepArgs& a = env->args;
  if (out_elig && a.B > 32) return fail("mbe_channel: the connectable bitmask output needs num_bs <= 32");
  const size_t total = (size_t)a.E * a.U;
  const int grid = (int)((total + mbe::kThreads - 1) / mbe::kThreads);
  const size_t smem = 4 * (size_t)(a.bs_per_env ? (mbe::kThreads / a.U + 2) * a.B : a.B) + a.B + 16;
  mbe::channel_kernel<<<grid, mbe::kThreads, smem, static_cast<cudaStream_t>(stream)>>>(a, out_snr, out_elig);
  MBE_CUDA(cudaGetLastError());
  env->launches += 1;
  return 0;
}

int mbe_accumulate_qoe(mbe_env* env, float* acc, float threshold, void* stream) {
  if (!env || !acc) return fail("mbe_accumulate_qoe: null argument");
  if (!env->bound) return fail("mbe_bind has not been called");
  if ((uintptr_t)acc & 15) return fail("mbe_accumulate_qoe: acc must be 16-byte aligned");
  MBE_ON_DEVICE(env->cfg.device);
  const mbe::StepArgs& a = env->args;
  const int per_blk = mbe::kThreads / 32;
  mbe::qoe_accumulate_kernel<<<(a.E + per_blk - 1) / per_blk, mbe::kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      a.utility, reinterpret_cast<float4*>(acc), a.E, a.U, threshold);
  MBE_CUDA(cudaGetLastError());
  env->launches += 1;
  return 0;
}

int mbe_rollout(mbe_env* env, int steps, float* qoe_acc, float threshold, const mbe_rollout_out* out, void* stream) {
  if (!env) return fail("null handle");
  if (!env->bound) return fail("mbe_bind has not been called");
  if (env->cfg.mode != MBE_MODE_FORK) return fail("mbe_rollout: FORK mode only (a GYM step needs fresh actions)");
  if (steps <= 0) return fail("mbe_rollout: steps must be positive");
  if ((uintptr_t)qoe_acc & 15) return fail("mbe_rollout: qoe_acc must be 16-byte aligned");
  MBE_ON_DEVICE(env->cfg.device);
  const mbe_rollout_out none = {};
  const mbe_rollout_out& o = out ? *out : none;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const mbe::StepArgs& a0 = env->args;
  const size_t EU = (size_t)a0.E * a0.U;
  if (env->episode.fn && env->episode.bound_ok && !a0.dbg_snr && aligned16({o.pos, o.wp, o.assoc, o.rate, o.utility}) &&
      (o.rate == nullptr || a0.rate)) {
    // fused episode: one launch, state read and written once
    mbe::StepArgs a = a0;
    a.op = mbe::OP_STEP;
    a.phases = MBE_PHASE_ALL;
    a.reset_mask = nullptr;
    a.ro_steps = steps;
    a.qoe_thr = threshold;
    a.qoe_acc = reinterpret_cast<float4*>(qoe_acc);
    a.ro_pos = reinterpret_cast<uint32_t*>(o.pos);
    a.ro_wp = reinterpret_cast<uint32_t*>(o.wp);
    a.ro_assoc = o.assoc;
    a.ro_rate = o.rate;
    a.ro_util = o.utility;
    return run(env, env->episode, a, stream);
  }
  // other shapes: the same episode as a sequence of step launches
  if ((o.pos || o.wp) && env->cfg.autoreset)
    return fail("mbe_rollout: per-step positions with autoreset need the fused kernel (MComCustom's 7 UEs x 10 BS slots "
                "or a scenario shape, num_envs a multiple of 32)");
  if (o.rate && !a0.rate) return fail("mbe_rollout: a rate series needs the rate buffer bound");
  for (int s = 0; s < steps; ++s) {
    if (int rc = launch(env, mbe::OP_STEP, MBE_PHASE_ALL, nullptr, stream)) return rc;
    if (qoe_acc)
      if (int rc = mbe_accumulate_qoe(env, qoe_acc, threshold, stream)) return rc;
    if (o.pos) MBE_CUDA(cudaMemcpyAsync(o.pos + 2 * EU * s, a0.pos, EU * 4, cudaMemcpyDeviceToDevice, st));
    if (o.wp) MBE_CUDA(cudaMemcpyAsync(o.wp + 2 * EU * s, a0.wp, EU * 4, cudaMemcpyDeviceToDevice, st));
    if (o.assoc) MBE_CUDA(cudaMemcpyAsync(o.assoc + EU * s, a0.assoc, EU * 4, cudaMemcpyDeviceToDevice, st));
    if (o.rate) MBE_CUDA(cudaMemcpyAsync(o.rate + EU * s, a0.rate, EU * 8, cudaMemcpyDeviceToDevice, st));
    if (o.utility) MBE_CUDA(cudaMemcpyAsync(o.utility + EU * s, a0.utility, EU * 4, cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

int mbe_render(mbe_env* env, const int32_t* env_ids, int n, const mbe_rollout_out* series, int steps,
               const mbe_render_style* style, uint8_t* out, void* stream) {
  if (!env || !style || !out) return fail("mbe_render: null argument");
  if (!env->bound) return fail("mbe_bind has not been called");
  const int H = style->height, W = style->width;
  if (H < 8 || H > 4096 || W < 8 || W > 4096 || W % 4)
    return fail("mbe_render: frame %d x %d out of range (8..4096 each, width a multiple of 4)", H, W);
  const int lim = MBE_RENDER_MAX_STYLE_PX;
  if (style->ue_radius < 0 || style->ue_radius > lim || style->bs_half < 0 || style->bs_half > lim ||
      style->line_width < 0 || style->line_width > lim)
    return fail("mbe_render: ue_radius, bs_half and line_width must be in 0..%d pixels", lim);
  if (n < 1) return fail("mbe_render: n must be positive");
  if (steps < 1) return fail("mbe_render: steps must be positive");
  if (steps > 1 && !series) return fail("mbe_render: steps > 1 needs a series");
  const bool gym = env->cfg.mode == MBE_MODE_GYM;
  if (series && gym) return fail("mbe_render: series are FORK-mode only (there is no connection series in GYM mode)");
  if (series && (!series->pos || !series->assoc || !series->utility))
    return fail("mbe_render: a series needs pos, assoc and utility");
  if ((uintptr_t)out & 3) return fail("mbe_render: out must be 4-byte aligned");
  const mbe::StepArgs& s = env->args;
  const int Wm = (int)env->cfg.width, Hm = (int)env->cfg.height;
  if (Wm < 1 || Hm < 1) return fail("mbe_render: the map must be at least 1 x 1 in integer units");
  mbe::RenderArgs a = {};
  a.pos = series ? reinterpret_cast<const uint32_t*>(series->pos) : s.pos;
  a.conn = s.conn;
  a.assoc = series ? series->assoc : s.assoc;
  a.utility = series ? series->utility : s.utility;
  a.bs_xy = s.bs_xy;
  a.nbs = s.nbs;
  a.bs_class = s.bs_class;
  a.env_ids = env_ids;
  a.out = out;
  a.step_eu = series ? (long long)s.E * s.U : 0;
  a.E = s.E, a.U = s.U, a.B = s.B, a.MW = (s.B + 31) >> 5, a.n = n, a.gym = gym, a.bs_per_env = s.bs_per_env;
  a.Wm = Wm, a.Hm = Hm;
  const int nuc = s.n_ue_classes;
  for (int c = 0; c < env->cfg.num_classes; ++c) a.cov_d2max[c] = env->cfg.classes[c * nuc].d2max;
  a.band_rows = std::min(H, std::max(4, (mbe::kRenderBandPixels / W) & ~3));
  a.bands = (H + a.band_rows - 1) / a.band_rows;
  a.seg_cap = mbe::kRenderSegUes * s.B;
  const long long blocks = (long long)steps * n * a.bands;
  if (blocks > 0x7fffffffll) return fail("mbe_render: %lld CTAs exceed one launch", blocks);
  const size_t smem = mbe::render_smem_layout(s.U, W, a.band_rows, a.seg_cap).total;
  MBE_ON_DEVICE(env->cfg.device);
  MBE_CUDA(cudaFuncSetAttribute((const void*)mbe::render_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mbe::render_kernel<<<(unsigned)blocks, mbe::kRenderThreads, smem, static_cast<cudaStream_t>(stream)>>>(a, *style);
  MBE_CUDA(cudaGetLastError());
  env->launches += 1;
  return 0;
}

namespace {
bool ranges_overlap(const void* a, size_t na, const void* b, size_t nb) {
  if (!a || !b) return false;
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return x < y + nb && y < x + na;
}
}  // namespace

int mbe_evolve_layouts(mbe_env* env, const float* fitness, const int16_t* parent_xy, const int32_t* parent_nbs,
                       const int32_t* elite_ids, int n_elite, const mbe_evolve_params* p, int16_t* child_xy,
                       int32_t* child_nbs, void* stream) {
  if (!env) return fail("null handle");
  if (!fitness || !parent_xy || !parent_nbs || !p || !child_xy || !child_nbs)
    return fail("mbe_evolve_layouts: null argument");
  const mbe_config& cfg = env->cfg;
  if (cfg.bs_layout != MBE_BS_PER_ENV || cfg.bs_random_max <= 0)
    return fail("mbe_evolve_layouts: needs random per-env BS layouts (bs_layout=PER_ENV, bs_random_max > 0)");
  // with M >= 2 trajectories per layout the population is the L = num_envs / M layouts (mbe.h)
  const int M = cfg.num_trajectories >= 2 ? cfg.num_trajectories : 1;
  const int E = cfg.num_envs / M, B = cfg.num_bs;
  if (n_elite < 0 || n_elite > E) return fail("mbe_evolve_layouts: n_elite=%d outside 0..%d", n_elite, E);
  if (n_elite > 0 && !elite_ids) return fail("mbe_evolve_layouts: n_elite > 0 needs elite_ids");
  if (p->tournament < 1 || p->tournament > 4)
    return fail("mbe_evolve_layouts: tournament=%d outside 1..4", p->tournament);
  if (p->step < 0 || p->step > 32767) return fail("mbe_evolve_layouts: step=%d outside 0..32767", p->step);
  const double probs[4] = {p->p_cross, p->p_move, p->p_add, p->p_del};
  for (double q : probs)
    if (!std::isfinite(q) || q < 0.0 || q > 1.0)
      return fail("mbe_evolve_layouts: probability %g is not in [0, 1]", q);
  const size_t xy_bytes = (size_t)E * B * 4, nbs_bytes = (size_t)E * 4;
  const void* inputs[4] = {fitness, parent_xy, parent_nbs, elite_ids};
  const size_t in_bytes[4] = {nbs_bytes, xy_bytes, nbs_bytes, (size_t)n_elite * 4};
  for (int i = 0; i < 4; ++i)
    if (ranges_overlap(child_xy, xy_bytes, inputs[i], in_bytes[i]) ||
        ranges_overlap(child_nbs, nbs_bytes, inputs[i], in_bytes[i]))
      return fail("mbe_evolve_layouts: child buffers overlap an input");
  if (ranges_overlap(child_xy, xy_bytes, child_nbs, nbs_bytes))
    return fail("mbe_evolve_layouts: child_xy and child_nbs overlap");
  if (((uintptr_t)fitness | (uintptr_t)parent_xy | (uintptr_t)parent_nbs | (uintptr_t)elite_ids |
       (uintptr_t)child_xy | (uintptr_t)child_nbs) & 3)
    return fail("mbe_evolve_layouts: buffers must be 4-byte aligned");
  const mbe::StepArgs& s = env->args;
  mbe::EvolveArgs a = {};
  a.fitness = fitness;
  a.parent = reinterpret_cast<const uint32_t*>(parent_xy);
  a.parent_nbs = parent_nbs;
  a.elite_ids = elite_ids;
  a.child = reinterpret_cast<uint32_t*>(child_xy);
  a.child_nbs = child_nbs;
  a.E = E, a.B = B, a.K = n_elite, a.T = p->tournament, a.step = p->step;
  a.nmin = cfg.bs_random_min, a.nmax = std::min(cfg.bs_random_max, B);
  a.env_offset = s.env_offset / (unsigned)M, a.generation = p->generation;
  a.seed_lo = (unsigned)(p->seed & 0xffffffffu), a.seed_hi = (unsigned)(p->seed >> 32);
  a.XM = (int)std::ceil(cfg.width) - 1, a.YM = (int)std::ceil(cfg.height) - 1;
  a.wh_int = s.wh_int, a.wh_int_w = s.wh_int_w, a.wh_int_h = s.wh_int_h;
  a.width = cfg.width, a.height = cfg.height;
  a.p_cross = p->p_cross, a.p_move = p->p_move, a.p_add = p->p_add, a.p_del = p->p_del;
  const size_t smem = (size_t)mbe::kEvolveThreads * B * 4;
  MBE_ON_DEVICE(cfg.device);
  mbe::evolve_kernel<<<(unsigned)((E + mbe::kEvolveThreads - 1) / mbe::kEvolveThreads), mbe::kEvolveThreads, smem,
                       static_cast<cudaStream_t>(stream)>>>(a);
  MBE_CUDA(cudaGetLastError());
  env->launches += 1;
  return 0;
}

int mbe_layout_map(mbe_env* env, const int32_t* env_ids, int n, const mbe_map_params* p, int64_t* stats,
                   int32_t* area, uint8_t* coverage, int8_t* serving, int8_t* qoe, void* stream) {
  static_assert(mbe::kMapMaxB == mbe::kBigMaxB, "a layout map stages every BS slot of a handle");
  if (!env) return fail("mbe_layout_map: null handle");
  if (!env->bound) return fail("mbe_bind has not been called");
  if (!p) return fail("mbe_layout_map: null params");
  const mbe::StepArgs& s = env->args;
  if (n < 0) return fail("mbe_layout_map: n=%d must be >= 0", n);
  if (p->stride < 1) return fail("mbe_layout_map: stride=%d must be >= 1", p->stride);
  if (p->load < 1) return fail("mbe_layout_map: load=%d must be >= 1", p->load);
  if (p->ue_class < 0 || p->ue_class >= s.n_ue_classes)
    return fail("mbe_layout_map: ue_class=%d outside 0..%d", p->ue_class, s.n_ue_classes - 1);
  if (!std::isfinite(p->threshold)) return fail("mbe_layout_map: threshold must be finite");
  if ((uintptr_t)stats & 7) return fail("mbe_layout_map: stats must be 8-byte aligned");
  if ((uintptr_t)area & 3) return fail("mbe_layout_map: area must be 4-byte aligned");
  if (n == 0) return 0;
  const mbe_config& cfg = env->cfg;
  mbe::MapArgs m = {};
  m.bs_xy = s.bs_per_env ? s.bs_xy : nullptr;
  m.nbs = s.nbs;
  m.env_ids = env_ids;
  m.bs_class = s.bs_class;
  m.stats = reinterpret_cast<long long*>(stats);
  m.area = area;
  m.coverage = coverage;
  m.serving = serving;
  m.qoe = qoe;
  m.E = s.E, m.B = s.B, m.n = n, m.s = p->stride;
  const int XM = (int)std::ceil(cfg.width) - 1, YM = (int)std::ceil(cfg.height) - 1;
  m.GX = XM / p->stride + 1;
  const int GY = YM / p->stride + 1;
  m.G = m.GX * GY;  // <= 32767^2
  m.bands = (m.G + mbe::kMapPoints - 1) / mbe::kMapPoints;
  if ((long long)n * m.bands > 0x7fffffffll) return fail("mbe_layout_map: %lld CTAs exceed one launch", (long long)n * m.bands);
  // a cent k is low iff float32(k / 100) < float32(threshold); float32(k / 100) increases with k
  m.k_low = 101;
  for (int k = 100; k >= -100; --k)
    if ((float)((double)k / 100.0) >= p->threshold) m.k_low = k;
  m.vec = m.G % 4 == 0 && (((uintptr_t)coverage | (uintptr_t)serving | (uintptr_t)qoe) & 3) == 0;
  m.n_classes = cfg.num_classes;
  m.load = (double)p->load;
  long long tab = 0;
  for (int c = 0; c < cfg.num_classes; ++c) {
    m.link[c] = c * s.n_ue_classes + p->ue_class;
    m.d2max[c] = s.cls[m.link[c]].d2max;
    m.off[c] = (int)tab;
    if (m.d2max[c] >= 0) tab += (long long)m.d2max[c] + 1;
    if (tab > 0x7fffffffll) return fail("mbe_layout_map: cent table of %lld entries is too large", tab);
  }
  m.tab_len = (int)tab;
  std::memcpy(m.xy, env->bound_xy, sizeof m.xy);
  MBE_ON_DEVICE(cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (m.tab_len > 0) MBE_CUDA(cudaMallocAsync((void**)&m.cent, (size_t)m.tab_len, st));
  const long long prep = std::max({(long long)m.tab_len, stats ? (long long)n * mbe::kMapStats : 0ll,
                                   area ? (long long)n * m.B : 0ll});
  int rc = 0;
  if (prep > 0) {
    mbe::map_prep_kernel<<<(unsigned)((prep + mbe::kMapThreads - 1) / mbe::kMapThreads), mbe::kMapThreads, 0, st>>>(
        s, m);
    env->launches += 1;
    if (cudaError_t e = cudaGetLastError()) rc = fail("mbe_layout_map: map_prep_kernel: %s", cudaGetErrorString(e));
  }
  if (rc == 0) {
    mbe::map_kernel<<<(unsigned)(n * m.bands), mbe::kMapThreads, 0, st>>>(m);
    env->launches += 1;
    if (cudaError_t e = cudaGetLastError()) rc = fail("mbe_layout_map: map_kernel: %s", cudaGetErrorString(e));
  }
  if (m.cent) MBE_CUDA(cudaFreeAsync(m.cent, st));
  return rc;
}

int64_t mbe_launch_count(const mbe_env* env) { return env ? env->launches : 0; }

const char* mbe_step_kernel_name(const mbe_env* env) {
  if (!env) return "";
  return pick(env, mbe::OP_STEP, MBE_PHASE_ALL, env->cfg.num_envs, env->args.dbg_snr != nullptr).name;
}

int mbe_step_host(mbe_env* env, const int32_t* actions_host, float* obs_host, float* reward_host,
                  uint8_t* done_host, void* stream) {
  if (!env) return fail("null handle");
  if (!env->bound) return fail("mbe_bind has not been called");
  MBE_ON_DEVICE(env->cfg.device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const mbe::StepArgs& a = env->args;
  const bool gym = env->cfg.mode == MBE_MODE_GYM, ma = env->cfg.handler == MBE_HANDLER_MA;
  if (!gym && (actions_host || obs_host || reward_host))
    return fail("mbe_step_host: actions, obs and reward only exist in GYM mode");
  // Env windows on two streams: the action upload and the step of window c+1 overlap the result
  // download of window c (PCIe is full duplex).  With observations the call is bound by their
  // download: plain FP32 rows by DMA straight into obs_host (48 GB/s on the B200 box, no host thread
  // touches them).  A compact wire format (a third fewer bytes, expanded into obs_host by host threads)
  // measured 0.52-0.70x this DMA path on the 16-vCPU B200 box (profiles/README.md): the host must still
  // write the FP32 rows.
  const int want = obs_host ? 4 : 1;
  int windows = std::min(want, std::max(1, a.E / (block_per_env(env->cfg) ? kAlign : 8 * kAlign)));
  const int per = ((a.E + windows - 1) / windows + kAlign - 1) / kAlign * kAlign;
  windows = (a.E + per - 1) / per;
  if (windows > 1 && !env->host_stream) {
    MBE_CUDA(cudaStreamCreateWithFlags(&env->host_stream, cudaStreamNonBlocking));
    MBE_CUDA(cudaEventCreateWithFlags(&env->host_fork, cudaEventDisableTiming));
    MBE_CUDA(cudaEventCreateWithFlags(&env->host_join, cudaEventDisableTiming));
  }
  if (windows > 1) {  // the side stream starts after everything already queued on the caller's stream
    MBE_CUDA(cudaEventRecord(env->host_fork, st));
    MBE_CUDA(cudaStreamWaitEvent(env->host_stream, env->host_fork, 0));
  }
  const size_t U = a.U;
  for (int w = 0, first = 0; first < a.E; ++w, first += per) {
    const int count = std::min(per, a.E - first);
    cudaStream_t s = (w & 1) ? env->host_stream : st;
    const size_t fu = (size_t)first * U, cu = (size_t)count * U;
    if (actions_host)
      MBE_CUDA(cudaMemcpyAsync(const_cast<int32_t*>(env->bufs.actions) + fu, actions_host + fu, cu * 4,
                               cudaMemcpyHostToDevice, s));
    if (int rc = (windows > 1 ? launch(env, mbe::OP_STEP, MBE_PHASE_ALL, nullptr, s, (size_t)first, count)
                              : launch(env, mbe::OP_STEP, MBE_PHASE_ALL, nullptr, s)))
      return rc;
    if (obs_host)
      MBE_CUDA(cudaMemcpyAsync(obs_host + fu * a.F, env->bufs.obs + fu * a.F, cu * a.F * 4, cudaMemcpyDeviceToHost, s));
    if (reward_host) {
      const size_t f = ma ? fu : (size_t)first, c = ma ? cu : (size_t)count;
      MBE_CUDA(cudaMemcpyAsync(reward_host + f, env->bufs.reward + f, c * 4, cudaMemcpyDeviceToHost, s));
    }
    if (done_host)
      MBE_CUDA(cudaMemcpyAsync(done_host + first, env->bufs.done + first, (size_t)count, cudaMemcpyDeviceToHost, s));
  }
  if (windows > 1) {
    MBE_CUDA(cudaEventRecord(env->host_join, env->host_stream));
    MBE_CUDA(cudaStreamWaitEvent(st, env->host_join, 0));
  }
  MBE_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"
