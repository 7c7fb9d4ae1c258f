// "Thread per env" fused FORK step (the reference's real step, base.py:230-296) for per-env BS
// layouts (MComCustom: 7 UEs, up to 10 random BSs per env): a CTA is ONE warp and owns 32
// consecutive envs; lane e walks the U UEs and B BS slots of its env in scalar code -- no ballots,
// no match, no shuffles, no idle lanes, and the per-env work (clock, metrics, BS table) is paid
// once per env instead of once per UE.  The FORK step has no observation, so an env needs only
// ~200 bytes of shared memory and occupancy is not limited by it (the same mapping for the GYM
// step was occupancy-bound by its 1 KB/env observation staging, profiles/README.md).
// Every global stream of the 32 envs is one contiguous slice: all HBM traffic is bulk async
// copies (TMA) -- 6 loads tracked by an mbarrier, 8-11 stores.
// Sums replay the association order of the warp-segment kernels' shuffle tree, so all outputs are
// bit-identical to them.
// ROLLOUT = true is the fused episode (mbe_rollout): the same step repeated a.ro_steps times with the
// state staying in shared memory / registers between steps -- state is read once and written once
// per launch; optional per-step outputs (positions after the move, association, rate, QoE:
// the series behind base.py:298-404's dumps) leave as bulk stores [T,E,U], and the QoE statistics
// of the layout score (qoe_accumulate_kernel, mbe_step.cuh) accumulate in registers.
// SHARED = true is the same kernel for a layout shared by all envs (the scenario shapes in FORK mode):
// the BS terms come from the kernel parameters, there is no per-env BS table to load, regenerate or store.
// Preconditions (dispatcher): FORK mode, per-env layout (or SHARED), one BS class, E % 32 == 0, exact-FP32
// map no larger than 2048 x 2048 (the packed nearest-BS key must not overflow), no debug SNR buffer, all stream
// bases 16-byte aligned, nbs bound.
#pragma once
#include "mbe_device.cuh"
#include <type_traits>

namespace mbe {

template <int U, int B>
struct TpeForkSmem {
  alignas(16) uint32_t pos[32 * U];
  alignas(16) uint32_t wp[32 * U];
  alignas(16) uint32_t bs[32 * B];
  alignas(16) int32_t nbs[32];
  alignas(16) int32_t t[32];
  alignas(16) int32_t epi[32];
  alignas(16) int32_t assoc[32 * U];
  alignas(16) double rate[32 * U];
  alignas(16) float util[32 * U];
  alignas(16) float metrics[32 * 4];
  alignas(16) uint8_t done[32];
  alignas(8) uint64_t bar;
};

template <int U, int B>
struct TpeRolloutSmem : TpeForkSmem<U, B> {
  alignas(16) uint32_t pos_out[32 * U];  // positions after the move (the reset below overwrites pos)
  alignas(16) uint32_t wp_out[32 * U];   // waypoints after the move ((-1,-1): arrived this step, movement.py:54-56)
};

// the dynamic shared memory of an instance
template <int U, int B, bool ROLLOUT>
using TpeSmem = typename std::conditional<ROLLOUT, TpeRolloutSmem<U, B>, TpeForkSmem<U, B>>::type;

// a CTA is one warp and owns as many consecutive envs, one per lane
constexpr int kTpeThreads = 32;
constexpr int kTpeEnvsPerCta = kTpeThreads;

// the lane-strided accumulation + shfl_down tree of qoe_accumulate_kernel (mbe_step.cuh) for one env
// on a thread-local array: lane 0's result after off = 16, 8, 4, 2, 1 with zeros in lanes >= U.
// Adding those zeros only ever turns a -0 into +0, which no later sum can see, so they are skipped.
template <int U>
__device__ __forceinline__ float tree32_sum(const float (&q)[U]) {
  constexpr int P = U <= 1 ? 1 : U <= 2 ? 2 : U <= 4 ? 4 : U <= 8 ? 8 : U <= 16 ? 16 : 32;
  float v[P];
#pragma unroll
  for (int i = 0; i < P; ++i) v[i] = i < U ? q[i] : 0.0f;
#pragma unroll
  for (int off = P / 2; off > 0; off >>= 1) {
#pragma unroll
    for (int i = 0; i < off; ++i)
      if (i + off < U) v[i] += v[i + off];
  }
  return v[0];
}

// the shuffle tree of seg_sum / seg_sum_head (mbe_device.cuh) replayed on a thread-local array:
// v[u] += v[u+off] for off = 1, 2, 4, ... where every lane reads pre-step values
template <int U>
__device__ __forceinline__ float tree_sum(float (&v)[U]) {
#pragma unroll
  for (int off = 1; off < U; off <<= 1) {
#pragma unroll
    for (int u = 0; u + off < U; ++u) v[u] += v[u + off];  // ascending u: v[u+off] is still the old value
  }
  return v[0];
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = (uint32_t)__cvta_generic_to_shared(bar);
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void bulk_load(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(sdst)),
               "l"(gsrc), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"((uint32_t)__cvta_generic_to_shared(ssrc)), "r"(bytes)
               : "memory");
}

// resident one-warp CTAs per SM the register allocation is held to (step / fused episode)
constexpr int kTpeBlocks = 20;
constexpr int kTpeRolloutBlocks = 16;

// |connections(b)| of one env, 4 bits per BS in one 64-bit word
template <int U, int B>
struct TpeCounts {
  static_assert(U <= 15 && B <= 16, "a count must fit 4 bits and all BSs one word");
  unsigned long long w;
  __device__ __forceinline__ void clear() { w = 0ull; }
  __device__ __forceinline__ void add(int b) { w += 1ull << (4 * b); }
  __device__ __forceinline__ unsigned get(int b) const { return (unsigned)(w >> (4 * b)) & 15u; }
};

template <int U, int B, bool ROLLOUT = false, bool SHARED = false>
__global__ void __launch_bounds__(kTpeThreads, ROLLOUT ? kTpeRolloutBlocks : kTpeBlocks) step_tpe_fork_kernel(const __grid_constant__ StepArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using S = TpeSmem<U, B, ROLLOUT>;
  static_assert(B <= 16, "the nearest-BS key keeps the BS index in 4 bits");
  static_assert(U <= 32, "the QoE tree replays a 32-lane reduction");
  S& s = *reinterpret_cast<S*>(smem_raw);
  const int lane = threadIdx.x;
  const size_t e0 = (size_t)blockIdx.x * kTpeEnvsPerCta;  // first env of this warp
  const int env = (int)e0 + lane;
  const unsigned gid = a.env_offset + (unsigned)env;
  const SlotDev& C0 = a.slot[0];  // the single BS class

  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // ---- state slices of the 32 envs -> shared memory (bulk async copies) ----
  constexpr uint32_t EU = 32 * U * 4, EB = 32 * B * 4, EE = 32 * 4;
  if (lane == 0) {
    mbar_init(&s.bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_expect_tx(&s.bar, 2 * EU + (SHARED ? 0u : EB + EE) + 2 * EE);
    bulk_load(s.pos, a.pos + e0 * U, EU, &s.bar);
    bulk_load(s.wp, a.wp + e0 * U, EU, &s.bar);
    if (!SHARED) {
      bulk_load(s.bs, a.bs_xy + e0 * B, EB, &s.bar);
      bulk_load(s.nbs, a.nbs + e0, EE, &s.bar);
    }
    bulk_load(s.t, a.t + e0, EE, &s.bar);
    bulk_load(s.epi, a.episode + e0, EE, &s.bar);
  }
  __syncwarp();
  mbar_wait(&s.bar, 0);

  uint32_t* my_pos = s.pos + lane * U;
  uint32_t* my_wp = s.wp + lane * U;
  uint32_t* my_bs = s.bs + lane * B;
  int t_e = s.t[lane], epi = s.epi[lane], nb = SHARED ? B : s.nbs[lane];

  float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  if (ROLLOUT && a.qoe_acc) acc = a.qoe_acc[env];
  const int steps = ROLLOUT ? a.ro_steps : 1;
  const bool ro_out = ROLLOUT && (a.ro_pos || a.ro_wp || a.ro_assoc || a.ro_rate || a.ro_util);
#pragma unroll 1
  for (int step = 0; step < steps; ++step) {
  if (ro_out && step > 0) {  // the previous step's bulk stores must have read their staging
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
  }
  // Per-BS terms of key(u, b) = 16 * d2(u, b) + b = cb + mx * x + my * y + 16 * (x^2 + y^2): two
  // multiply-adds and a min per UE x BS pair; the UE's own term is added after the min.
  // Absent slots (b >= nb) are parked far outside the map: they can never be the nearest BS.
  int cb[B], mx[B], my[B];
#pragma unroll
  for (int b = 0; b < B; ++b) {
    int bx, by;
    if (SHARED) {
      bx = a.slot[b].x, by = a.slot[b].y;
    } else {
      unpack_xy(my_bs[b], bx, by);
      if (b >= nb) bx = by = -6000;  // 2*(6000+2048)^2 << 4 still fits int32; > any d2max on such a map
    }
    cb[b] = ((bx * bx + by * by) << 4) | b;
    mx[b] = -32 * bx;
    my[b] = -32 * by;
  }

  // ---- waypoint draws first (movement.py:44-47): a lane that needs k new waypoints loops k times,
  // so the warp pays max-over-lanes draws (usually 1-3) instead of one per UE slot ----
  unsigned need = 0;
#pragma unroll
  for (int u = 0; u < U; ++u) need |= ((my_wp[u] >> 15) & 1u) << u;  // x < 0: no waypoint
  while (need) {
    const int u = __ffs((int)need) - 1;
    need &= need - 1;
    int wx, wy;
    next_waypoint(a, gid, (unsigned)u, (size_t)env * U + u, t_e, epi, true, wx, wy);
    my_wp[u] = pack_xy(wx, wy);
  }

  // ---- move (movement.py:42-62), then nearest connectable BS (base.py:236-241) ----
  int best[U], bestd2[U];
  TpeCounts<U, B> packed;  // |connections(b)|
  packed.clear();
#pragma unroll
  for (int u = 0; u < U; ++u) {
    int x, y, wx, wy;
    unpack_xy(my_pos[u], x, y);
    unpack_xy(my_wp[u], wx, wy);
    if (move_ue(a.mv[0], x, y, wx, wy)) wx = wy = -1;
    my_pos[u] = pack_xy(x, y);
    my_wp[u] = pack_xy(wx, wy);
    if constexpr (ROLLOUT) {
      s.pos_out[lane * U + u] = my_pos[u];
      s.wp_out[lane * U + u] = my_wp[u];
    }
    // nearest BS = min over (d2 << 4 | b): lowest b wins a distance tie like Python's min
    // (base.py:240); with a single BS class it is connectable iff its d2 <= d2max (base.py:212-214)
    int key = 0x7fffffff;
#pragma unroll
    for (int b = 0; b < B; ++b) key = min(key, cb[b] + mx[b] * x + my[b] * y);
    key += (x * x + y * y) << 4;
    const int bd = key >> 4;
    const int bb = (bd <= C0.d2max) ? (key & 15) : -1;
    best[u] = bb;
    bestd2[u] = bd;
    if (bb >= 0) packed.add(bb);
  }

  // ---- ResourceFair split + rounding (schedules.py:20-22, base.py:435), utility (253-258) ----
  const double* lut = C0.lutn;
  const unsigned stride = (unsigned)C0.stride;
  float uv[U], rv[U];
  int nconn = 0;
#pragma unroll
  for (int u = 0; u < U; ++u) {
    double rate = 0.0;
    if (best[u] >= 0) {
      const unsigned n = packed.get(best[u]);
      rate = lut[n * stride + (unsigned)bestd2[u]];
      nconn += 1;
    }
    const float util = scaled_utility(a, rate);
    s.assoc[lane * U + u] = best[u];
    s.rate[lane * U + u] = rate;
    s.util[lane * U + u] = util;
    uv[u] = util;
    rv[u] = (float)rate;
  }
  {
    const float usum = tree_sum<U>(uv), rsum = tree_sum<U>(rv);
    const float nc = (float)nconn;
    reinterpret_cast<float4*>(s.metrics)[lane] = make_float4(nc, nc, usum * a.inv_U, mean_or_zero(rsum, nc));
  }
  if (ROLLOUT && a.qoe_acc) {  // this step's two-decimal QoE values (base.py:269) into the score statistics
    float q1[U], q2[U], ql[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const float q = qoe_cent_value(s.util[lane * U + u]);
      q1[u] = q;
      q2[u] = fmaf(q, q, 0.0f);
      ql[u] = (q < a.qoe_thr) ? 1.0f : 0.0f;
    }
    acc = make_float4(acc.x + tree32_sum<U>(q1), acc.y + tree32_sum<U>(q2), acc.z + tree32_sum<U>(ql), acc.w + (float)U);
  }

  // ---- clock, same-step autoreset (base.py:280-291, 407-409; 172-209; custom.py:40-77) ----
  t_e += 1;
  const bool done = t_e >= a.ep_time;
  s.done[lane] = done ? 1 : 0;
  if (done && a.autoreset) {
    epi += 1;
    t_e = 0;
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
      int x, y;
      philox_point(a, gid, (unsigned)u, 0u, P_INITPOS, a.reset_rng_episode ? 0u : (unsigned)epi, x, y);
      my_pos[u] = pack_xy(x, y);
      my_wp[u] = pack_xy(-1, -1);
      if (a.inj_wp) a.wp_cnt[(size_t)env * U + u] = 0;
    }
    if (!SHARED && a.bs_rand_max > 0) {  // generate_base_stations (custom.py:68-77)
      nb = philox_bs_count(a, gid, (unsigned)epi);
#pragma unroll 1
      for (int b = 0; b < B; ++b) {
        int x = 0, y = 0;
        if (b < nb) philox_point(a, gid, (unsigned)b, 0u, P_BSLAYOUT, (unsigned)epi, x, y);
        my_bs[b] = pack_xy(x, y);
      }
    }
  }
  s.t[lane] = t_e;
  s.epi[lane] = epi;
  if (!SHARED) s.nbs[lane] = nb;

  if constexpr (ROLLOUT) if (ro_out) {  // per-step series [T,E,U]
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
      const size_t off = ((size_t)step * a.E + e0) * U;
      if (a.ro_pos) bulk_store(a.ro_pos + off, s.pos_out, EU);
      if (a.ro_wp) bulk_store(a.ro_wp + off, s.wp_out, EU);
      if (a.ro_assoc) bulk_store(a.ro_assoc + off, s.assoc, EU);
      if (a.ro_rate) bulk_store(a.ro_rate + off, s.rate, 2 * EU);
      if (a.ro_util) bulk_store(a.ro_util + off, s.util, EU);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  }
  }  // steps
  if (ROLLOUT && a.qoe_acc) a.qoe_acc[env] = acc;

  // ---- everything leaves as bulk async stores ----
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();
  if (lane == 0) {
    bulk_store(a.pos + e0 * U, s.pos, EU);
    bulk_store(a.wp + e0 * U, s.wp, EU);
    bulk_store(a.assoc + e0 * U, s.assoc, EU);
    if (a.rate) bulk_store(a.rate + e0 * U, s.rate, 2 * EU);
    bulk_store(a.utility + e0 * U, s.util, EU);
    if (a.metrics) bulk_store(a.metrics + e0 * 4, s.metrics, 4 * EE);
    bulk_store(a.done + e0, s.done, 32);
    bulk_store(a.t + e0, s.t, EE);
    bulk_store(a.episode + e0, s.epi, EE);
    if (!SHARED && a.bs_rand_max > 0) {
      bulk_store(a.bs_xy + e0 * B, s.bs, EB);
      bulk_store(a.nbs + e0, s.nbs, EE);
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  }
}

}  // namespace mbe
