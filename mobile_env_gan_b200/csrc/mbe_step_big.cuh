// Block-per-env fused step kernel for the wide shapes (32 < U <= 1024 UEs or 32 < B <= 64 BS
// slots, e.g. the synthetic 64 x 512 scale-up) and for the ProportionalFair / RateFair schedulers:
// one CTA of 256 threads owns one env.
//
// Two mappings inside the CTA:
//   * per-UE work (movement, connectivity, association / action, split, utility): a thread owns up
//     to 4 UEs in registers, the BS table and the per-BS accumulators live in shared memory.  Per-BS
//     counts / proportional-fair totals / multi-agent BS utilities are integer (fixed-point)
//     shared-memory atomics, so every result is independent of the order threads arrive in;
//   * the observation writer is ROW-PARALLEL: a warp walks its share of the UE rows and its lanes
//     are the BS columns (lane = b and b + 32, coordinates and per-BS values in registers), so the
//     row maximum of log2 snr is one warp reduction (redux.sync.max.f32) and every store instruction
//     writes 128 contiguous bytes of one observation row straight from registers -- no staging tile,
//     no transposition.  (Round 1 produced lane-per-row tiles in shared memory and transposed them:
//     three passes over a padded tile, 2x the instructions; profiles/README.md.)
// Same arithmetic helpers as the warp-segment kernels (mbe_device.cuh).
#pragma once
#include <type_traits>
#include "mbe_device.cuh"

namespace mbe {

constexpr int kBigThreads = 256;
constexpr int kBigWarps = kBigThreads / 32;
constexpr int kBigMaxI = 4;     // UEs per thread  => U <= 1024
constexpr int kBigMaxB = 64;    // BS slots        => two 32-bit mask words
constexpr int kBigMinBlocks = 3;  // resident CTAs per SM at 4 UEs per thread (one more at 2)
// per-warp shared-memory tile of whole observation rows on their way out (floats): 8 rows of the 64-BS
// central shape (8 x 129), 4 of the multi-agent one (4 x 257); 16-byte multiple
constexpr int kBigTileFloats = 1056;

template <int MAXU>
struct BigSmemT {
  float2 bsf[kBigMaxB];  // BS coordinates as floats (integers, exact)
  int cnt[kBigMaxB];
  unsigned long long pf_tot[kBigMaxB];
  long long bsu_acc[kBigMaxB];
  float bsu[kBigMaxB];
  uint8_t cls[kBigMaxB];
  float red_f[3][kBigWarps];
  int red_i[2][kBigWarps];
  float usum, rsum;
  int csum, ncon;
  // inputs of the observation rows, published by the threads that own the UEs
  float2 pxy[MAXU];   // position after the move
  uint2 cw[MAXU];     // connection mask words
  float ut[MAXU];     // own-utility column
  uint8_t ucls[MAXU]; // UE class
};

// dynamic shared memory of the kernel: the struct above sized for MAXI UEs per thread, then (128-byte
// aligned) one row tile per warp
template <int MAXI>
__host__ __device__ constexpr size_t big_tile_offset() {
  return (sizeof(BigSmemT<MAXI * kBigThreads>) + 127) & ~(size_t)127;
}
template <int MAXI>
__host__ __device__ constexpr size_t big_smem_bytes() {
  return big_tile_offset<MAXI>() + (size_t)kBigTileFloats * 4 * kBigWarps;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(kFull, v, off);
  return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(kFull, v, off);
  return v;
}
// warp-wide float maximum in one instruction (sm_100a: CREDUX.MAX.F32)
__device__ __forceinline__ float warp_max_f32(float v) {
  float r;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}

// one link's share of its BS (schedules.py:20-22 / proportional fair), rounded like base.py:435
__device__ __forceinline__ double link_share(const StepArgs& a, const ClassDev& c, int d2, int n,
                                             unsigned long long pf_tot) {
  const double raw = c.lut0[d2];  // Channel.datarate (channels.py:78-83), FP64 table
  double share;
  if (a.scheduler == 1) {
    const double tot = __ll2double_rn((long long)pf_tot) * (1.0 / 1048576.0);
    share = (raw * raw) / tot;
  } else if (a.scheduler == 2) {  // RateFair: the same 1 / sum(1/r) for every UE of the BS
    const double tot = __ll2double_rn((long long)pf_tot) * 0x1p-50;
    share = 1.0 / tot;
  } else {
    share = raw / (double)n;
  }
  return rint(share * 100.0) / 100.0;
}

// MAXI = UEs per thread held in registers (U <= MAXI * 256): 2 covers the synthetic 512-UE shape with 64
// registers and 4 resident CTAs per SM, 4 (U <= 1024) needs 80 registers / 3 CTAs
template <int MODE, int HANDLER, int MAXI = kBigMaxI>
__global__ void __launch_bounds__(kBigThreads, MAXI <= 2 ? kBigMinBlocks + 1 : kBigMinBlocks) step_big_kernel(const __grid_constant__ StepArgs a) {
  constexpr int kBigMaxI = MAXI;  // shadows the namespace constant inside this kernel
  constexpr bool GYM = (MODE == 1);
  constexpr bool MA = (HANDLER == 1);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using BigSmem = BigSmemT<MAXI * kBigThreads>;
  BigSmem& s = *reinterpret_cast<BigSmem*>(smem_raw);
  const int U = a.U, B = a.B, F = a.F, MW = (B + 31) >> 5;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int env = blockIdx.x;
  const unsigned gid = a.env_offset + (unsigned)env;
  const int op = a.op;
  int ph = a.phases;
  if (op == OP_RESET || op == OP_OBSERVE) ph = GYM ? 8 : 0;
  // the env's outputs are (re)written by this launch (per env = per CTA: uniform)
  if (op == OP_RESET && a.reset_mask != nullptr && a.reset_mask[env] == 0) return;

  // ---- P0: env scalars, BS table, accumulators ----
  int t_e = a.t[env], epi = a.episode[env];
  int nb = a.nbs ? a.nbs[env] : B;
  if (tid < B) {
    int bx, by;
    unpack_xy(a.bs_per_env ? a.bs_xy[(size_t)env * B + tid] : a.bs_xy[tid], bx, by);
    s.bsf[tid] = make_float2((float)bx, (float)by);
    s.cls[tid] = a.bs_class ? a.bs_class[tid] : (uint8_t)0;
    s.cnt[tid] = 0;
    s.pf_tot[tid] = 0ull;
    s.bsu_acc[tid] = 0ll;
    s.bsu[tid] = -1.0f;
  }
  __syncthreads();

  // ---- per-UE registers ----
  int x[kBigMaxI], y[kBigMaxI], wx[kBigMaxI], wy[kBigMaxI];
  uint32_t c0[kBigMaxI], c1[kBigMaxI], e0[kBigMaxI], e1[kBigMaxI];
  float util[kBigMaxI];
  int best[kBigMaxI];
  int ucls[kBigMaxI];
#pragma unroll
  for (int i = 0; i < kBigMaxI; ++i) {
    const int u = tid + i * kBigThreads;
    x[i] = y[i] = 0;
    wx[i] = wy[i] = -1;
    c0[i] = c1[i] = e0[i] = e1[i] = 0;
    util[i] = -1.0f;
    best[i] = -1;
    ucls[i] = 0;
    if (u < U) {
      const size_t idx = (size_t)env * U + u;
      unpack_xy(a.pos[idx], x[i], y[i]);
      unpack_xy(a.wp[idx], wx[i], wy[i]);
      if (GYM) {
        c0[i] = a.conn[idx * MW];
        if (MW > 1) c1[i] = a.conn[idx * MW + 1];
      }
      // link class of (b, this UE) = bs_class[b] * n_ue_classes + ue_class[u] (entities.py:6-57)
      if (a.ue_class) ucls[i] = (int)a.ue_class[u];
    }
  }
  bool done = false, fresh = false, util_known = false;
  const bool one_class = a.n_classes == 1 && a.n_ue_classes == 1;
  const int nuc = a.n_ue_classes;
  auto link = [&](int i, int b) -> const ClassDev& { return a.cls[(int)s.cls[b] * nuc + ucls[i]]; };
  const float d2max0f = (float)a.cls[0].d2max;  // exact: below 2^24

  // squared distance UE -- BS b in FP32: coordinates are integers below 2^15, so every product and
  // the sum are exact (whenever the map's squared diagonal is below 2^24; mbe_create checks it)
  auto d2f_to = [&](float xf, float yf, int b) {
    const float2 q = s.bsf[b];
    const float dx = xf - q.x, dy = yf - q.y;
    return fmaf(dx, dx, dy * dy);
  };
  auto d2_to = [&](int i, int b) { return (int)d2f_to((float)x[i], (float)y[i], b); };
  auto has_bit = [&](uint32_t lo, uint32_t hi, int b) { return (((b < 32) ? (lo >> b) : (hi >> (b - 32))) & 1u) != 0; };

  auto phase_move = [&]() {
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      if (wx[i] < 0) next_waypoint(a, gid, (unsigned)u, (size_t)env * U + u, t_e, epi, true, wx[i], wy[i]);
      if (move_ue(a.mv[ucls[i]], x[i], y[i], wx[i], wy[i])) wx[i] = wy[i] = -1;
    }
  };

  // block-wide sums in a fixed order (warp tree, then warp partials in ascending order)
  auto block_sums = [&](float fu, float fr, int ic, int in) {
    fu = warp_sum(fu);
    fr = warp_sum(fr);
    ic = warp_sum_i(ic);
    in = warp_sum_i(in);
    if (lane == 0) {
      s.red_f[0][warp] = fu;
      s.red_f[1][warp] = fr;
      s.red_i[0][warp] = ic;
      s.red_i[1][warp] = in;
    }
    __syncthreads();
    if (tid == 0) {
      float su = 0.0f, sr = 0.0f;
      int sc = 0, sn = 0;
      for (int w = 0; w < kBigWarps; ++w) {
        su += s.red_f[0][w];
        sr += s.red_f[1][w];
        sc += s.red_i[0][w];
        sn += s.red_i[1][w];
      }
      s.usum = su;
      s.rsum = sr;
      s.csum = sc;
      s.ncon = sn;
    }
    __syncthreads();
  };

  // allStationUtilities (base.py:438-447) from the connection masks and utilities in registers:
  // 2^-32 fixed-point sums, so the mean does not depend on the order the threads arrive in
  auto bs_utilities = [&]() {
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      const long long q = __double2ll_rn((double)util[i] * 4294967296.0);
      for (int w = 0; w < 2; ++w) {
        uint32_t m = w ? c1[i] : c0[i];
        while (m) {
          const int b = (__ffs(m) - 1) + 32 * w;
          m &= m - 1;
          atomicAdd((unsigned long long*)&s.bsu_acc[b], (unsigned long long)q);
        }
      }
    }
    __syncthreads();
    if (tid < B)
      s.bsu[tid] = s.cnt[tid] ? (float)(__ll2double_rn(s.bsu_acc[tid]) * (1.0 / 4294967296.0) / (double)s.cnt[tid])
                              : -1.0f;
    __syncthreads();
  };

  auto reinit_all = [&]() {
    // MComCore.reset + MComCustom.reset for this env (base.py:172-209, custom.py:40-62)
    epi += 1;
    t_e = 0;
    fresh = true;
    if (a.bs_rand_max > 0 && a.bs_per_env) {
      nb = philox_bs_count(a, gid, (unsigned)epi);
      __syncthreads();
      if (tid < B) {
        int bx = 0, by = 0;
        if (tid < nb) philox_point(a, gid, (unsigned)tid, 0u, P_BSLAYOUT, (unsigned)epi, bx, by);
        s.bsf[tid] = make_float2((float)bx, (float)by);
        a.bs_xy[(size_t)env * B + tid] = pack_xy(bx, by);
      }
      if (tid == 0 && a.nbs) a.nbs[env] = nb;
    }
    __syncthreads();
    if (tid < B) {
      s.cnt[tid] = 0;
      s.bsu[tid] = -1.0f;
    }
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      c0[i] = c1[i] = 0;
      wx[i] = wy[i] = -1;
      philox_point(a, gid, (unsigned)u, 0u, P_INITPOS, a.reset_rng_episode ? 0u : (unsigned)epi, x[i], y[i]);
      if (a.inj_wp) a.wp_cnt[(size_t)env * U + u] = 0;
    }
    __syncthreads();
  };

  // ---- PRE: connectivity, association / action, per-BS accumulators, split, utility ----
  auto phase_pre = [&]() {
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      const size_t idx = (size_t)env * U + u;
      const float xf = (float)x[i], yf = (float)y[i];
      float bestf = 3.0e38f;
      int act = 0;
      if (GYM) act = a.actions[idx];
      if (GYM && !MA && !a.dbg_snr) {
        // The central handler only ever asks "is BS b connectable" for the BSs the UE is connected to
        // (update_connections, base.py:221-227) and for the BS its action names: test those few pairs
        // instead of all B (the multi-agent reward and the FORK association need every pair).  Only
        // the tested bits of e0 / e1 are meaningful afterwards, and only those are read below.
        const int ab = (act > 0 && act <= nb) ? act - 1 : -1;
        for (int w = 0; w < 2; ++w) {
          uint32_t m = (w ? c1[i] : c0[i]) | ((ab >= 32 * w && ab < 32 * w + 32) ? 1u << (ab & 31) : 0u);
          uint32_t ew = 0;
          while (m) {
            const int bl = __ffs(m) - 1, b = bl + 32 * w;
            m &= m - 1;
            if (d2f_to(xf, yf, b) <= (one_class ? d2max0f : (float)link(i, b).d2max)) ew |= 1u << bl;
          }
          if (w) e1[i] = ew; else e0[i] = ew;
        }
      } else
      for (int w = 0; w < 2; ++w) {  // one 32-bit mask word at a time (no per-BS word select)
        uint32_t ew = 0;
        const int b_lo = 32 * w, b_hi = min(nb, 32 * w + 32);
#pragma unroll 4
        for (int b = b_lo; b < b_hi; ++b) {
          const float d2f = d2f_to(xf, yf, b);
          if (d2f <= (one_class ? d2max0f : (float)link(i, b).d2max)) {  // check_connectivity (base.py:212-214)
            ew |= 1u << (b - b_lo);
            if (!GYM && d2f < bestf) {  // nearest connectable BS, first minimum (base.py:240)
              best[i] = b;
              bestf = d2f;
            }
          }
        }
        if (w) e1[i] = ew; else e0[i] = ew;
      }
      if (GYM) {
        c0[i] &= e0[i];  // update_connections (base.py:221-227)
        c1[i] &= e1[i];
        if (act > 0 && act <= nb) {  // NOOP_ACTION = 0 (base.py:29)
          const int b = act - 1;
          uint32_t& cw = (b < 32) ? c0[i] : c1[i];
          const uint32_t ew = (b < 32) ? e0[i] : e1[i];
          const uint32_t bit = 1u << (b & 31);
          cw = (cw & bit) ? (cw & ~bit) : (cw | (ew & bit));
        }
      } else {
        c0[i] = c1[i] = 0;
        if (best[i] >= 0) {
          if (best[i] < 32) c0[i] = 1u << best[i]; else c1[i] = 1u << (best[i] - 32);
        }
      }
      for (int w = 0; w < 2; ++w) {
        uint32_t m = w ? c1[i] : c0[i];
        while (m) {
          const int b = (__ffs(m) - 1) + 32 * w;
          m &= m - 1;
          atomicAdd(&s.cnt[b], 1);
          if (a.scheduler == 1) {
            const double raw = link(i, b).lut0[d2_to(i, b)];
            atomicAdd(&s.pf_tot[b], (unsigned long long)__double2ll_rn(raw * 1048576.0));
          } else if (a.scheduler == 2) {
            const double raw = link(i, b).lut0[d2_to(i, b)];
            atomicAdd(&s.pf_tot[b], (unsigned long long)__double2ll_rn(0x1p50 / raw));
          }
        }
      }
      if (a.dbg_snr)
        for (int b = 0; b < B; ++b)
          a.dbg_snr[idx * B + b] = (b < nb) ? ex2_sfu(log2_snr(link(i, b), d2_to(i, b))) : 0.0f;
    }
    __syncthreads();

    // split, rounding, utility (base.py:421-435, 413-418, 253-258)
    float fu = 0.0f, fr = 0.0f;
    int ic = 0, in = 0;
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      const size_t idx = (size_t)env * U + u;
      double r = 0.0;
      for (int w = 0; w < 2; ++w) {
        uint32_t m = w ? c1[i] : c0[i];
        while (m) {  // ascending bs order = the reference's bs-major accumulation
          const int b = (__ffs(m) - 1) + 32 * w;
          m &= m - 1;
          r += link_share(a, link(i, b), d2_to(i, b), s.cnt[b], s.pf_tot[b]);
        }
      }
      util[i] = scaled_utility(a, r);
      if (a.rate) a.rate[idx] = r;
      a.utility[idx] = util[i];
      if (!GYM) a.assoc[idx] = best[i];
      fu += util[i];
      fr += (float)r;
      ic += __popc(c0[i]) + __popc(c1[i]);
      in += (c0[i] | c1[i]) ? 1 : 0;
    }
    util_known = true;
    block_sums(fu, fr, ic, in);
    if (GYM && MA) {
      bs_utilities();
#pragma unroll
      for (int i = 0; i < kBigMaxI; ++i) {
        const int u = tid + i * kBigThreads;
        if (u >= U) continue;
        float nu = 0.0f;
        int ncnt = 0;
        for (int b = 0; b < nb; ++b)
          if (has_bit(e0[i], e1[i], b)) {  // available_connections (base.py:216-218)
            nu += s.bsu[b];
            ncnt += s.cnt[b];
          }
        a.reward[(size_t)env * U + u] = (nu + util[i]) / (float)(ncnt + 1);
      }
    }
    if (tid == 0) {
      if (GYM && !MA) a.reward[env] = s.usum * a.inv_U;  // mean utility (metrics.py:25-28)
      if (a.metrics) {
        const float nc = (float)s.ncon;
        reinterpret_cast<float4*>(a.metrics)[env] =
            make_float4((float)s.csum, nc, s.usum * a.inv_U, mean_or_zero(s.rsum, nc));
      }
    }
  };

  // ---- CLOCK (base.py:280-291, 407-409) ----
  auto phase_clock = [&]() {
    t_e += 1;
    done = t_e >= a.ep_time;
    if (tid == 0) a.done[env] = done ? 1 : 0;
    if (done) {
      __syncthreads();
#pragma unroll
      for (int i = 0; i < kBigMaxI; ++i) c0[i] = c1[i] = 0;  // everyone leaves at ep_time
      if (tid < B) {
        s.cnt[tid] = 0;
        s.bsu[tid] = -1.0f;
      }
      if (a.autoreset) reinit_all();
      else __syncthreads();
    }
  };

  // ---- POST: observation rows (GYM), row-parallel: warp = row, lanes = BS columns ----
  auto phase_post = [&]() {
    if (!GYM) return;
    if (!(ph & 4)) done = !fresh && (t_e >= a.ep_time);  // CLOCK ran in an earlier launch: the clock tells
    const bool is_fresh = fresh || (t_e == 0);
    if (!util_known) {
#pragma unroll
      for (int i = 0; i < kBigMaxI; ++i) {
        const int u = tid + i * kBigThreads;
        if (u < U) util[i] = a.utility[(size_t)env * U + u];
      }
      if (MA && !is_fresh && !done) {  // split phases / mbe_observe: rebuild the per-BS statistics
        __syncthreads();
        if (tid < B) {
          s.cnt[tid] = 0;
          s.bsu_acc[tid] = 0ll;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < kBigMaxI; ++i) {
          if (tid + i * kBigThreads >= U) continue;
          for (int w = 0; w < 2; ++w) {
            uint32_t m = w ? c1[i] : c0[i];
            while (m) {
              atomicAdd(&s.cnt[(__ffs(m) - 1) + 32 * w], 1);
              m &= m - 1;
            }
          }
        }
        __syncthreads();
        bs_utilities();
      }
    }
    if (MA && (is_fresh || done)) {  // nobody is connected in a fresh / finished episode
      __syncthreads();
      if (tid < B) {
        s.cnt[tid] = 0;
        s.bsu[tid] = -1.0f;
      }
    }
    // publish what the rows need
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      s.pxy[u] = make_float2((float)x[i], (float)y[i]);
      s.cw[u] = (is_fresh || done) ? make_uint2(0u, 0u) : make_uint2(c0[i], c1[i]);
      s.ut[u] = is_fresh ? -1.0f : util[i];
      s.ucls[u] = (uint8_t)ucls[i];
    }
    __syncthreads();

    // Rows leave through shared memory: a warp fills a tile of TR whole rows (a multiple of 4 rows is a
    // multiple of 16 bytes; with U % 4 == 0 every tile is also 16-byte aligned in global memory) and sends
    // it as ONE bulk async copy.  The rows are 4F bytes with F odd, so direct 128-byte segment stores from
    // registers start at every 4-byte phase of a 32-byte sector: profiles/row_store_bench.cu measures
    // 3.5 TB/s for that pattern against 7.1-7.3 TB/s for the same rows as aligned bulk tiles.  Shapes
    // whose rows cannot be tiled that way (U % 4 != 0, unaligned obs) keep the direct stores.
    const bool tiled = a.obs_bulk_ok && (U % 4 == 0) && F <= kBigTileFloats / 4;
    const int rpw = tiled ? (((U + kBigWarps - 1) / kBigWarps + 3) & ~3) : (U + kBigWarps - 1) / kBigWarps;
    const int r0 = min(U, warp * rpw), r1 = min(U, r0 + rpw);  // rows of this warp (contiguous)
    const int TR = tiled ? min(16, (kBigTileFloats / F) & ~3) : max(1, r1 - r0);
    float* const tile = reinterpret_cast<float*>(smem_raw + big_tile_offset<MAXI>()) + (size_t)warp * kBigTileFloats;
    float* obase = a.obs + (size_t)env * U * F;
    if (done && !fresh) {  // inactive UEs observe zeros
      for (size_t e = (size_t)r0 * F + lane; e < (size_t)r1 * F; e += 32) obase[e] = 0.0f;
      return;
    }
    const int b0 = lane, b1 = lane + 32;
    const bool h0 = b0 < B, h1 = b1 < B;    // the column exists
    const bool v0 = b0 < nb, v1 = b1 < nb;  // the BS slot is live
    const float2 q0 = h0 ? s.bsf[b0] : make_float2(0.0f, 0.0f), q1 = h1 ? s.bsf[b1] : make_float2(0.0f, 0.0f);
    const int cb0 = h0 ? (int)s.cls[b0] * nuc : 0, cb1 = h1 ? (int)s.cls[b1] * nuc : 0;
    const float kk = a.cls[0].k_hi, l0c = a.cls[0].l0_hi;
    float bsu0 = -1.0f, bsu1 = -1.0f;
    int cn0 = 0, cn1 = 0;
    if (MA) {
      if (h0) { bsu0 = s.bsu[b0]; cn0 = s.cnt[b0]; }
      if (h1) { bsu1 = s.bsu[b1]; cn1 = s.cnt[b1]; }
    }
    // FULL = both column groups exist for every lane (B == 64, the synthetic scale-up) and one link
    // class: no column predicates, the row's stores are one base pointer plus immediates
    // rows [u_lo, u_hi) into `dst` (row u_lo first, stride F): the global block or a shared-memory tile
    auto rows = [&](auto full_tag, int u_lo, int u_hi, float* dst, bool with_util) {
      constexpr bool FULL = decltype(full_tag)::value;
      const int BB = FULL ? 64 : B;
#pragma unroll 2
      for (int u = u_lo; u < u_hi; ++u) {
        const float2 p = s.pxy[u];
        const uint2 cw = s.cw[u];
        float* row = dst + (size_t)(u - u_lo) * F;
        // log2 snr of this lane's two BSs (d = 0 is the reference's EPSILON, channels.py:8: the 1e-32
        // vanishes in the rounding of every d2 >= 1)
        float dx = p.x - q0.x, dy = p.y - q0.y;
        const float d2f0 = fmaf(dx, dx, fmaf(dy, dy, 1e-32f));
        dx = p.x - q1.x, dy = p.y - q1.y;
        const float d2f1 = fmaf(dx, dx, fmaf(dy, dy, 1e-32f));
        float l0v, l1v, m0, m1;  // log2 snr, connectable range
        if (FULL || one_class) {
          l0v = fmaf(-kk, lg2_sfu(d2f0), l0c);
          l1v = fmaf(-kk, lg2_sfu(d2f1), l0c);
          m0 = m1 = d2max0f;
        } else {
          const int uc = (int)s.ucls[u];
          const ClassDev& k0 = a.cls[cb0 + uc];
          const ClassDev& k1 = a.cls[cb1 + uc];
          l0v = k0.ltab ? k0.ltab[min((int)d2f0, k0.ltab_len - 1)] : fmaf(-k0.k_hi, lg2_sfu(d2f0), k0.l0_hi);
          l1v = k1.ltab ? k1.ltab[min((int)d2f1, k1.ltab_len - 1)] : fmaf(-k1.k_hi, lg2_sfu(d2f1), k1.l0_hi);
          m0 = (float)k0.d2max;
          m1 = (float)k1.d2max;
        }
        if (!v0) l0v = -INFINITY;
        if (!v1) l1v = -INFINITY;
        const float lmax = warp_max_f32(fmaxf(l0v, l1v));
        // the connection bit of this lane's column as 0.0f / 1.0f: (bit ? ~0 : 0) & bits(1.0f)
        const float one0 = __uint_as_float((uint32_t)((int32_t)(cw.x << (31 - lane)) >> 31) & 0x3f800000u);
        const float one1 = __uint_as_float((uint32_t)((int32_t)(cw.y << (31 - lane)) >> 31) & 0x3f800000u);
        if (FULL || h0) {
          row[b0] = one0;
          row[BB + b0] = ex2_sfu(l0v - lmax);  // snr / max snr (a dead slot: ex2(-inf) = 0)
        }
        if (FULL || h1) {
          row[b1] = one1;
          row[BB + b1] = ex2_sfu(l1v - lmax);
        }
        if (MA) {
          const bool ok0 = v0 && d2f0 <= m0, ok1 = v1 && d2f1 <= m1;  // available_connections (base.py:216-218)
          const int tot = __reduce_add_sync(kFull, (ok0 ? cn0 : 0) + (ok1 ? cn1 : 0));
          const float inv = 1.0f / fmaxf(1.0f, (float)tot);
          if (FULL || h0) {
            row[2 * BB + 1 + b0] = ok0 ? bsu0 : -1.0f;
            row[3 * BB + 1 + b0] = ok0 ? (float)cn0 * inv : 0.0f;
          }
          if (FULL || h1) {
            row[2 * BB + 1 + b1] = ok1 ? bsu1 : -1.0f;
            row[3 * BB + 1 + b1] = ok1 ? (float)cn1 * inv : 0.0f;
          }
        }
      }
      // the utility column (one element per row, stride F): up to 32 rows per store instruction
      // instead of a predicated single-lane store in every row
      if (with_util)
        for (int u = u_lo + lane; u < u_hi; u += 32) dst[(size_t)(u - u_lo) * F + 2 * B] = s.ut[u];
    };
    const bool full = B == 64 && one_class;
    if (!tiled) {
      if (full) rows(std::true_type{}, r0, r1, obase + (size_t)r0 * F, true);
      else rows(std::false_type{}, r0, r1, obase + (size_t)r0 * F, true);
      return;
    }
    for (int t0 = r0; t0 < r1; t0 += TR) {
      const int t1 = min(r1, t0 + TR);
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the previous tile has been read
      __syncwarp();
      if (full) rows(std::true_type{}, t0, t1, tile, true);
      else rows(std::false_type{}, t0, t1, tile, true);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(obase + (size_t)t0 * F),
                     "r"((uint32_t)__cvta_generic_to_shared(tile)), "r"((uint32_t)((t1 - t0) * F) * 4u)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  };

  // ================= run =================
  if (op == OP_RESET) {
    reinit_all();
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      const size_t idx = (size_t)env * U + u;
      util[i] = -1.0f;
      a.utility[idx] = -1.0f;
      if (a.rate) a.rate[idx] = 0.0;
      if (!GYM) a.assoc[idx] = -1;
      if (GYM && MA) a.reward[idx] = 0.0f;
    }
    util_known = true;
    if (tid == 0) {
      a.done[env] = 0;
      if (GYM && !MA) a.reward[env] = 0.0f;
    }
    phase_post();
  } else if (op == OP_OBSERVE) {
    phase_post();
  } else if (!GYM) {
    if (ph & 1) phase_move();  // FORK moves first (base.py:232-233)
    if (ph & 2) phase_pre();
    if (ph & 4) phase_clock();
  } else {
    if (ph & 2) phase_pre();
    if (ph & 1) phase_move();
    if (ph & 4) phase_clock();
    if (ph & 8) phase_post();
  }

  // ---- store state ----
  if (op != OP_OBSERVE) {
#pragma unroll
    for (int i = 0; i < kBigMaxI; ++i) {
      const int u = tid + i * kBigThreads;
      if (u >= U) continue;
      const size_t idx = (size_t)env * U + u;
      a.pos[idx] = pack_xy(x[i], y[i]);
      a.wp[idx] = pack_xy(wx[i], wy[i]);
      if (GYM) {
        a.conn[idx * MW] = c0[i];
        if (MW > 1) a.conn[idx * MW + 1] = c1[i];
      }
    }
    if (tid == 0) {
      if ((ph & 4) || op == OP_RESET) a.t[env] = t_e;
      if (fresh) a.episode[env] = epi;
    }
  }
}

}  // namespace mbe
