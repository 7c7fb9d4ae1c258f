// Device-side building blocks of the batched MComCore.step (sm_100a).
// Reference semantics are cited per function (paths relative to the reference repo).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mbe {

constexpr int kWarpsPerBlock = 4;
constexpr int kThreads = kWarpsPerBlock * 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxSlots = 32;

// Envs per warp when an env takes `lanes` adjacent lanes of it (the lanes past the last env idle).
__host__ __device__ constexpr int envs_per_warp(int lanes) { return 32 / lanes; }
// Envs per CTA of the warp-segment mapping (generic and specialised kernels): U lanes per env,
// kWarpsPerBlock warps per CTA.
__host__ __device__ constexpr int segment_envs_per_cta(int U) { return envs_per_warp(U) * kWarpsPerBlock; }

enum Op : int { OP_STEP = 0, OP_RESET = 1, OP_OBSERVE = 2 };
enum Purpose : unsigned { P_WAYPOINT = 0, P_INITPOS = 1, P_BSLAYOUT = 2 };

// One link class (include/mbe.h mbe_link_class: a BS parameter set x a UE parameter set) as the
// kernels see it.  Link class of the pair (b, u) = bs_class[b] * n_ue_classes + ue_class[u].
struct ClassDev {
  float l0_hi, l0_lo;  // log2 snr at d2 = 1, split hi+lo (channel kernel keeps ~2^-30 of it)
  float k_hi, k_lo;    // slope per log2(d2)
  float l_zero;        // log2 snr at d2 == 0
  int d2max;           // connectable iff d2 <= d2max
  int stride;          // d2max + 1
  int ltab_len;
  // lutn[n*stride + d2] = round(rate_lut[d2] / n, 2) for n >= 1: Channel.datarate
  // (channels.py:78-83) split over n UEs (schedules.py:20-22) and rounded like base.py:435, all
  // in FP64.  Row n = 0 does not exist: the pointer is biased so that lutn[stride - 1] is a
  // 0.0 entry placed just before row 1 (an unconnected link adds exactly nothing).
  const double* lutn;
  const double* lut0;  // rate_lut[d2] itself (un-split, un-rounded) for the block-per-env kernel
  const float* ltab;   // log2 snr per d2 for losses that are not affine in log-distance, else nullptr
};

// Movement parameters of one UE class (include/mbe.h mbe_ue_class), folded on the host.
struct MoveDev {
  double velocity;
  float velocity_f, tie_eps;  // FP32 fast path of the movement and its fallback band
  int axis_exact;             // (velocity*d)/|d| == +-velocity in FP64 for every |d| on the map
  int move_d2max;             // largest integer d2 with sqrt(d2) <= velocity (movement.py:54)
};

constexpr int kMaxLinkClasses = 16;
constexpr int kMaxUeClasses = 8;

// One BS slot of a shared layout with its class folded in: every field becomes a constant-bank
// operand once the specialised kernels unroll their loops over b.
struct SlotDev {
  int x, y, d2max, stride;
  float k, l0, xf, yf;  // xf, yf: the same coordinates as floats (exact)
  const double* lutn;
};

struct StepArgs {
  // geometry of the launch
  int E, U, B, F;
  int epw;  // envs per warp
  int epb;  // envs per block
  int op, phases;
  unsigned env_offset;
  unsigned traj_gid_mask;  // 0xffffffff, or 0 when all envs share the UE trajectories
  // scenario
  int ep_time, autoreset, reset_rng_episode, bs_per_env, bs_rand_min, bs_rand_max;
  unsigned seed_lo, seed_hi;
  double width, height;
  int wh_int, wh_int_w, wh_int_h;  // width and height are integers (the usual case): integer draws
  MoveDev mv[kMaxUeClasses];       // [0] is the only one when all UEs are alike
  // utility: u = clip(util_c * log2(w2 + r), lo, hi); scaled = (u - lo) * util_scale - 1
  float util_c, util_w2, util_lo, util_hi, util_scale;
  float inv_U;  // 1/U for the per-env means
  int n_classes;     // BS classes
  int n_ue_classes;  // UE classes (>= 1)
  int scheduler;  // 0 ResourceFair; 1 ProportionalFair, 2 RateFair (block-per-env kernel only)
  ClassDev cls[kMaxLinkClasses];  // [bs class * n_ue_classes + ue class]
  SlotDev slot[kMaxSlots];
  const uint8_t* bs_class;  // device [B] or nullptr
  const uint8_t* ue_class;  // device [U] or nullptr (all UEs class 0)
  // bound buffers (see include/mbe.h)
  uint32_t* pos;
  uint32_t* wp;
  int32_t* t;
  int32_t* episode;
  uint32_t* bs_xy;
  int32_t* nbs;
  uint32_t* conn;
  int32_t* assoc;
  const int32_t* actions;
  double* rate;
  float* utility;
  float* obs;
  float* reward;
  uint8_t* done;
  float* metrics;
  float* dbg_snr;
  const uint32_t* inj_wp;
  int32_t* wp_cnt;
  int inj_k;
  const uint8_t* reset_mask;
  int obs_bulk_ok;  // obs base is 16B aligned -> whole-block TMA bulk store allowed
  int pf_dist;      // L2 prefetch distance in CTAs (0 = off; needs 16B aligned pos/wp/conn/actions)
  // fused episode (mbe_rollout, FORK thread-per-env kernel): steps per launch, score statistics,
  // optional per-step series [T,E,U]
  int ro_steps;
  float qoe_thr;
  float4* qoe_acc;
  uint32_t* ro_pos;
  uint32_t* ro_wp;
  int32_t* ro_assoc;
  double* ro_rate;
  float* ro_util;
};

// L2 prefetch (cp.async.bulk.prefetch.L2) of the per-UE state slices of the CTA that runs
// a.pf_dist CTAs after this one -- about 0.75 waves of resident CTAs, so the slices are in L2
// when that CTA starts and its first loads do not pay HBM latency.  CTAs of the first a.pf_dist
// (nobody runs ahead of them) prefetch their own slices: called before griddepcontrol.wait, that
// overlaps the drain of the previous grid under programmatic dependent launch (a prefetch returns
// nothing to the SM and L2 is the point of coherence, so it may run ahead of the dependency).
// One thread, 2 (FORK) or 4 (GYM) instructions per slice set; slices are EPB*U words, whole CTAs only.
template <int EPB, int U, bool GYM>
__device__ __forceinline__ void prefetch_slices(const StepArgs& a, size_t cta) {
  constexpr uint32_t bytes = EPB * U * 4;
  const size_t off = cta * EPB * U;
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.pos + off), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.wp + off), "r"(bytes) : "memory");
  if (GYM) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.conn + off), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.actions + off), "r"(bytes) : "memory");
  }
}

template <int EPB, int U, bool GYM>
__device__ __forceinline__ void prefetch_ahead(const StepArgs& a) {
  if constexpr ((EPB * U) % 4 == 0) {
    if (a.pf_dist > 0 && threadIdx.x == 0) {
      const size_t ahead = (size_t)blockIdx.x + (size_t)a.pf_dist;
      if ((int)blockIdx.x < a.pf_dist && ((size_t)blockIdx.x + 1) * EPB <= (size_t)a.E)
        prefetch_slices<EPB, U, GYM>(a, blockIdx.x);
      if ((ahead + 1) * EPB <= (size_t)a.E) prefetch_slices<EPB, U, GYM>(a, ahead);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011): counter-based replacement for the shared PCG64 stream
// behind RandomWaypointMovement (movement.py:16-18,44-47,64-72).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  constexpr unsigned M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    unsigned hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    unsigned hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}

// x = int(u0 * W), y = int(u1 * H) with u = r * 2^-32 in FP64: the counter-based analogue of
// int(rng.uniform(0, W)) (movement.py:45-46, 69-70).  Counter = (env gid, ue, t, purpose+4*salt).
__device__ __forceinline__ void philox_point(const StepArgs& a, unsigned gid, unsigned ue, unsigned t,
                                          unsigned purpose, unsigned salt, int& x, int& y) {
  // UE trajectories (waypoints, initial positions) can be shared by all envs -- the fork's dataset:
  // movement reset_rng_episode=True gives every epoch the same UE trajectory (base.py:130-134) and
  // only the BS layout differs; layouts always use the env's own id
  if (purpose != P_BSLAYOUT) gid &= a.traj_gid_mask;
  uint4 r = philox4x32_10(make_uint4(gid, ue, t, purpose + 4u * salt), make_uint2(a.seed_lo, a.seed_hi));
  if (a.wh_int) {  // integer map size: floor(r * 2^-32 * W) is exactly the high word of r * W
    x = (int)__umulhi(r.x, (unsigned)a.wh_int_w);
    y = (int)__umulhi(r.y, (unsigned)a.wh_int_h);
  } else {
    x = (int)((double)r.x * 0x1p-32 * a.width);
    y = (int)((double)r.y * 0x1p-32 * a.height);
  }
}

__device__ __forceinline__ int philox_bs_count(const StepArgs& a, unsigned gid, unsigned salt) {
  uint4 r = philox4x32_10(make_uint4(gid, 0xFFFFu, 0xFFFFu, P_BSLAYOUT + 4u * salt),
                          make_uint2(a.seed_lo, a.seed_hi));
  return a.bs_rand_min + (int)((double)r.x * 0x1p-32 * (double)(a.bs_rand_max - a.bs_rand_min + 1));
}

// raw SFU ops (flush-to-zero: one MUFU each, no denormal fix-up code around them)
__device__ __forceinline__ float lg2_sfu(float v) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ float ex2_sfu(float v) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

__device__ __forceinline__ uint32_t pack_xy(int x, int y) {
  return ((uint32_t)x & 0xffffu) | ((uint32_t)y << 16);
}
__device__ __forceinline__ void unpack_xy(uint32_t p, int& x, int& y) {
  x = (int)(int16_t)(p & 0xffffu);
  y = (int)(p) >> 16;
}

// The waypoint a UE without one gets (movement.py:44-47): the next injected one when a replay
// table is bound (tests replaying reference trajectories), else a Philox draw.
__device__ __forceinline__ void next_waypoint(const StepArgs& a, unsigned gid, unsigned ue, size_t idx, int t_e,
                                              int epi, bool valid, int& wx, int& wy) {
  if (a.inj_wp) {
    if (valid) {
      const int k = a.wp_cnt[idx];
      unpack_xy(a.inj_wp[idx * a.inj_k + min(k, a.inj_k - 1)], wx, wy);
      a.wp_cnt[idx] = k + 1;
    } else {
      wx = wy = 0;
    }
  } else {
    philox_point(a, gid, ue, (unsigned)t_e, P_WAYPOINT, a.reset_rng_episode ? 0u : (unsigned)epi, wx, wy);
  }
}

// ---------------------------------------------------------------------------------------
// RandomWaypointMovement.move once the waypoint exists (movement.py:49-62).
// Reference arithmetic (FP64): pos + (velocity * v) / norm(v), np.round (half-even), astype(int).
// "norm <= velocity" is the integer test d2 <= move_d2max (host-folded, exact).
// The step t = velocity*d/norm is first taken in FP32 (SFU rsqrt, |error| < 4e-7*velocity);
// only when t lies within tie_eps of a rounding tie is the reference's FP64 chain replayed, so
// the integer result is always the reference's.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void move_slow(const MoveDev& m, int& x, int& y, int dx, int dy, int d2) {
  double norm = sqrt((double)d2);
  x = (int)rint((double)x + (m.velocity * (double)dx) / norm);
  y = (int)rint((double)y + (m.velocity * (double)dy) / norm);
}

__device__ __forceinline__ bool move_ue(const MoveDev& m, int& x, int& y, int wx, int wy) {
  int dx = wx - x, dy = wy - y;
  int d2 = dx * dx + dy * dy;
  if (d2 <= m.move_d2max) {
    x = wx;
    y = wy;
    return true;  // arrived: snap and pop the waypoint (movement.py:54-56)
  }
  float s = m.velocity_f * rsqrtf((float)d2);
  float tx = (float)dx * s, ty = (float)dy * s;
  float rx = rintf(tx), ry = rintf(ty);
  float worst = fmaxf(fabsf(tx - rx), fabsf(ty - ry));  // distance to the nearest integer, <= 0.5
  if (worst > 0.5f - m.tie_eps) {
    if (m.axis_exact && (dx == 0 || dy == 0)) {
      // axis-aligned (frequent: integer snapping lines UEs up with their waypoint): the FP64
      // step is exactly +-velocity (host-verified), so only the final rint needs FP64
      if (dx != 0) x = (int)rint((double)x + (dx > 0 ? m.velocity : -m.velocity));
      if (dy != 0) y = (int)rint((double)y + (dy > 0 ? m.velocity : -m.velocity));
    } else {
      move_slow(m, x, y, dx, dy, d2);
    }
  } else {
    x += (int)rx;
    y += (int)ry;
  }
  return false;
}

// log2 of the SNR (channels.py:24-27 + 132-146 folded): l0 - k*log2(d2); SFU lg2 on FP32.  Losses
// that are not affine in log-distance come as a table over d2 (Channel.fold).
__device__ __forceinline__ float log2_snr(const ClassDev& c, int d2) {
  if (c.ltab) return c.ltab[min(d2, c.ltab_len - 1)];
  if (d2 == 0) return c.l_zero;
  float lg = lg2_sfu((float)d2);
  float l = fmaf(-c.k_hi, lg, c.l0_hi);
  return fmaf(-c.k_lo, lg, l) + c.l0_lo;
}

// single-float form used for the observation ratios snr/max snr (error < 2e-6 relative).
// d2f is the squared distance in FP32 (exact below 2^24); d = 0 is the reference's EPSILON
// (channels.py:8): log10(0 + 1e-16) <=> d2 = 1e-32.
__device__ __forceinline__ float log2_snr_obs_f(float k, float l0, float d2f) {
  return fmaf(-k, lg2_sfu(fmaxf(d2f, 1e-32f)), l0);
}
// the same for any link class (runtime-shape kernels)
__device__ __forceinline__ float log2_snr_obs(const ClassDev& c, int d2) {
  if (c.ltab) return c.ltab[min(d2, c.ltab_len - 1)];
  return log2_snr_obs_f(c.k_hi, c.l0_hi, (float)d2);
}

// BoundedLogUtility.calculateUtility + scaleUtility (utilities.py:44-55); SFU lg2
// (absolute error 2^-22 near 1, relative 2^-22 elsewhere).
__device__ __forceinline__ float scaled_utility(const StepArgs& a, double rate) {
  float u = a.util_c * lg2_sfu(a.util_w2 + (float)rate);
  u = fminf(fmaxf(u, a.util_lo), a.util_hi);
  u = fmaf(u - a.util_lo, a.util_scale, -1.0f);
  return (rate <= 0.0) ? -1.0f : u;  // rate <= 0 -> lower bound -> scaled -1
}

// The two-decimal QoE value behind the layout score (base.py:269 stores round(qoe, 2)), shared by
// qoe_accumulate_kernel and the fused episode so that both keep agreeing bit for bit (include/mbe.h
// mbe_accumulate_qoe): the cent k is the exact half-even rounding of u * 100 and the value is
// float32(k / 100).  u * 100 rounded to FP32 lands exactly on a half for some u whose exact product
// lies off it (u = float32(0.015) = 0.01499999966 gives 1.5); the FMA residual of that product is exact
// and says on which side.  k * 0.01f is not float32(k / 100) for 60 of the 201 cents (10 * 0.01f =
// 0.099999994f < 0.1f); one correction with the exact residual k - 100 * q0 gives the correctly rounded
// quotient for every |k| <= 100.  __fmul_rn keeps the products from being contracted into FMAs.
__device__ __forceinline__ float qoe_cent_value(float u) {
  const float p = __fmul_rn(u, 100.0f);
  float k = rintf(p);
  if (fabsf(p - k) == 0.5f) {
    const float e = fmaf(u, 100.0f, -p);
    if (e != 0.0f) k = p + copysignf(0.5f, e);
  }
  const float q0 = __fmul_rn(k, 0.01f);
  return fmaf(fmaf(-q0, 100.0f, k), 0.01f, q0);
}

// The cent k itself, as an integer: the same exact half-even rounding of u * 100 as qoe_cent_value
// (layout maps, mbe_map.cuh, tabulate it per squared distance).
__device__ __forceinline__ int qoe_cent(float u) {
  const float p = __fmul_rn(u, 100.0f);
  float k = rintf(p);
  if (fabsf(p - k) == 0.5f) {
    const float e = fmaf(u, 100.0f, -p);
    if (e != 0.0f) k = p + copysignf(0.5f, e);
  }
  return (int)k;
}

// mean over the connected UEs (metrics.py:18-21): 0 when nobody is connected
__device__ __forceinline__ float mean_or_zero(float sum, float n) { return n > 0.0f ? __fdividef(sum, n) : 0.0f; }

// Sum over the lanes of one env (contiguous segment of U lanes inside the warp), result
// broadcast to every lane of the segment.  Fixed tree order => deterministic.
__device__ __forceinline__ float seg_sum(float v, int u, int U, int lane) {
  for (int off = 1; off < U; off <<= 1) {
    float o = __shfl_down_sync(kFull, v, off);
    if (u + off < U) v += o;
  }
  return __shfl_sync(kFull, v, lane - u);
}

// Same tree without the final broadcast: only the env's first lane (u == 0) holds the sum.
template <int U>
__device__ __forceinline__ float seg_sum_head(float v, int u) {
#pragma unroll
  for (int off = 1; off < U; off <<= 1) {
    float o = __shfl_down_sync(kFull, v, off);
    if (u + off < U) v += o;
  }
  return v;
}

// (Re)initialise one env: MComCore.reset + MComCustom.reset (base.py:172-209, custom.py:40-62).
// `sel` is uniform over the lanes of an env; every lane of the warp must call (syncwarp inside).
__device__ __forceinline__ void reinit_env(const StepArgs& a, bool sel, unsigned gid, int u, size_t idx, int env,
                                        uint32_t* sbs_env, int& epi, int& t_e, uint32_t& conn, int& x, int& y,
                                        int& wx, int& wy, int& nb, bool& fresh) {
  if (sel) {
    epi += 1;
    t_e = 0;
    conn = 0;
    wx = wy = -1;
    philox_point(a, gid, (unsigned)u, 0u, P_INITPOS, a.reset_rng_episode ? 0u : (unsigned)epi, x, y);
    if (a.inj_wp) a.wp_cnt[idx] = 0;
    if (a.bs_rand_max > 0 && a.bs_per_env) {  // generate_base_stations (custom.py:68-77)
      nb = philox_bs_count(a, gid, (unsigned)epi);
      for (int b = u; b < a.B; b += a.U) {
        int bx = 0, by = 0;
        if (b < nb) philox_point(a, gid, (unsigned)b, 0u, P_BSLAYOUT, (unsigned)epi, bx, by);
        uint32_t p = pack_xy(bx, by);
        sbs_env[b] = p;
        a.bs_xy[(size_t)env * a.B + b] = p;
      }
      if (u == 0 && a.nbs) a.nbs[env] = nb;
    }
    if (u == 0) a.episode[env] = epi;
    fresh = true;
  }
  __syncwarp();
}

// the observation block of a CTA leaves shared memory: one bulk async copy (TMA) when the
// block is whole and aligned, else a predicated cooperative copy
template <int THREADS = kThreads>
__device__ __forceinline__ void store_obs_block(const StepArgs& a, const float* sobs, int env_base, int tid,
                                                bool whole) {
  // fast path: a full block (epb*U*F*4 bytes is a multiple of 16 by construction) leaves as one
  // bulk copy issued by thread 0; nobody else computes an address
  if (whole && a.obs_bulk_ok && env_base + a.epb <= a.E) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      const uint32_t bytes = (uint32_t)(a.epb * a.U * a.F) * 4u;
      float* gdst = a.obs + (size_t)env_base * (size_t)(a.U * a.F);
      uint32_t saddr = (uint32_t)__cvta_generic_to_shared(sobs);
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(saddr), "r"(bytes)
                   : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    return;
  }
  const int envs_here = min(a.epb, a.E - env_base);
  const size_t words = (size_t)envs_here * a.U * a.F;
  float* gdst = a.obs + (size_t)env_base * a.U * a.F;
  __syncthreads();
  for (size_t i = tid; i < words; i += THREADS) {
    int e = env_base + (int)(i / ((size_t)a.U * a.F));
    if (whole || a.reset_mask[e] != 0) gdst[i] = sobs[i];
  }
}

}  // namespace mbe
