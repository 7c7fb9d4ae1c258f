// "UEs per thread" fused GYM step for shared layouts with one BS class: an env is a group of K
// adjacent lanes and every lane owns UPT = U / K UEs (u = k, k+K, k+2K, ...), so the per-thread
// prologue, constant loads, per-env reductions and per-env stores are amortised over UPT UEs
// instead of one.  floor(32/K) envs per warp, 4 warps per CTA; loads stay direct (K consecutive
// words per env per instruction), the observation block is staged in shared memory and leaves as
// one bulk async copy like in the warp-segment kernels (mbe_step_spec.cuh).
//   medium (U=15, B=4): K=5, 3 UEs per lane, 6 envs per warp (30 lanes busy)
//   large  (U=30, B=13): K=10, 3 UEs per lane, 3 envs per warp (central handler)
// Per-BS connection counts are packed 8 bits per BS into words and summed over the K lanes with K
// shuffles; float sums are (local sum in UE order) then (lane 0..K-1 in order): a fixed order, but a
// different association than the 15-lane shuffle tree of the other kernels (last-ulp differences
// in reward / mean metrics only; everything discrete and the FP64 rates are identical).
#pragma once
#include "mbe_device.cuh"

namespace mbe {

// resident CTAs per SM x 2 (register budget), tuned on B200: 7 for both handlers (72 registers, no
// forced cap; 8 = 64 registers was best before the L2 prefetch, 3.5% slower with it)
constexpr int kUptBlocks = 7;
// warps per CTA of this mapping: 2 measured best (finer CTA granularity; 1 would break the 16-byte
// size rule of the observation bulk store for U=15)
constexpr int kUptWarps = 2;
constexpr int kUptThreads = 32 * kUptWarps;

// Envs per CTA of an instance and its dynamic shared memory, the observation staging block.
template <int HANDLER, int U, int B, int K>
struct UptLayout {
  static constexpr int EPW = envs_per_warp(K);
  static constexpr int EPB = EPW * kUptWarps;
  static constexpr int F = (HANDLER == 1 ? 4 : 2) * B + 1;
  static constexpr size_t BYTES = ((size_t)EPB * U * F * 4 + 15) & ~(size_t)15;
};

template <int HANDLER, int U, int B, int K>
__global__ void __launch_bounds__(kUptThreads, kUptBlocks * 4 / kUptWarps) step_upt_kernel(const __grid_constant__ StepArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  static_assert(U % K == 0, "U must be a multiple of K");
  using L = UptLayout<HANDLER, U, B, K>;
  constexpr bool MA = (HANDLER == 1);
  constexpr int UPT = U / K;
  constexpr int EPW = L::EPW;
  constexpr int EPB = L::EPB;
  constexpr int F = L::F;
  constexpr int NW = (B + 3) / 4;  // packed count words (8 bits per BS)
  float* s_obs = reinterpret_cast<float*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  prefetch_ahead<EPB, U, true>(a);
  asm volatile("griddepcontrol.wait;" ::: "memory");

  int g = lane / K;
  int k = lane - g * K;
  const bool in_group = g < EPW;
  if (!in_group) {
    g = EPW;
    k = 0;
  }
  const int base = min(g * K, 31);  // first lane of the env's group
  const int env_base = blockIdx.x * EPB;
  const int env_in_blk = warp * EPW + g;
  const int env = env_base + env_in_blk;
  const bool valid = in_group && env < a.E;
  const int env_ld = valid ? env : 0;
  const unsigned gid = a.env_offset + (unsigned)env;
  const SlotDev& C0 = a.slot[0];

  // ---- load state ----
  unsigned idx[UPT];
  uint32_t pos_in[UPT], wp_in[UPT], conn[UPT], conn_in[UPT];
  int act[UPT];
#pragma unroll
  for (int j = 0; j < UPT; ++j) {
    idx[j] = (unsigned)env_ld * U + (unsigned)(k + K * j);
    pos_in[j] = a.pos[idx[j]];
    wp_in[j] = a.wp[idx[j]];
    conn[j] = valid ? a.conn[idx[j]] : 0u;
    act[j] = valid ? a.actions[idx[j]] : 0;
  }
  int t_e = a.t[env_ld];
  int epi = a.episode[env_ld];
  int x[UPT], y[UPT], wx[UPT], wy[UPT];
#pragma unroll
  for (int j = 0; j < UPT; ++j) {
    unpack_xy(pos_in[j], x[j], y[j]);
    unpack_xy(wp_in[j], wx[j], wy[j]);
    conn_in[j] = conn[j];
  }

  // ---- pass 1: update_connections + actions (base.py:221-227, :29), packed per-BS counts ----
  uint32_t elig[UPT];
  int d2pre[UPT][B];
  uint32_t packed[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) packed[w] = 0;
#pragma unroll
  for (int j = 0; j < UPT; ++j) {
    elig[j] = 0;
#pragma unroll
    for (int b = 0; b < B; ++b) {
      const int dx = x[j] - a.slot[b].x, dy = y[j] - a.slot[b].y;
      d2pre[j][b] = dx * dx + dy * dy;
      elig[j] |= (d2pre[j][b] <= C0.d2max) ? (1u << b) : 0u;  // check_connectivity (base.py:212-214)
    }
    conn[j] &= elig[j];
    {  // toggle BS act-1: disconnect when connected, else connect when connectable (one XOR)
      const uint32_t bit = ((unsigned)(act[j] - 1) < (unsigned)B) ? (1u << (act[j] - 1)) : 0u;
      conn[j] ^= bit & (conn[j] | elig[j]);
    }
    // 4 connection bits -> 4 byte counters: bit i lands on bit 8i of (nibble * 0x204081), no collisions
#pragma unroll
    for (int w = 0; w < NW; ++w) packed[w] += (((conn[j] >> (4 * w)) & 0xfu) * 0x00204081u) & 0x01010101u;
  }
  uint32_t tot[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    tot[w] = 0;
#pragma unroll
    for (int i = 0; i < K; ++i) tot[w] += __shfl_sync(kFull, packed[w], min(base + i, 31));
  }
  int cnt[B];
  int csum = 0;
#pragma unroll
  for (int b = 0; b < B; ++b) {
    cnt[b] = (tot[b >> 2] >> (8 * (b & 3))) & 0xff;
    csum += cnt[b];
  }

  // ---- pass 2: split + rounding (base.py:421-435, 413-418), utility (253-258) ----
  const double* lut = C0.lutn;
  const unsigned stride = (unsigned)C0.stride;
  double rate[UPT];
  float util[UPT];
  float lu = 0.0f, lr = 0.0f;
  int ln = 0;
#pragma unroll
  for (int j = 0; j < UPT; ++j) {
    double r = 0.0;
#pragma unroll
    for (int b = 0; b < B; ++b) {
      // the rate table through the read-only path: measured -2.3% (multi-agent), neutral (central)
      if (MA) {  // measured: predicated gathers win with the multi-agent register budget ...
        if ((conn[j] >> b) & 1u) r += __ldg(lut + ((unsigned)cnt[b] * stride + (unsigned)d2pre[j][b]));
      } else {   // ... unconditional ones (unconnected -> the table's 0.0 entry) for the central handler
        const unsigned off = (unsigned)cnt[b] * stride + (unsigned)d2pre[j][b];
        r += __ldg(lut + (((conn[j] >> b) & 1u) ? off : stride - 1u));
      }
    }
    rate[j] = r;
    util[j] = scaled_utility(a, r);
    lu += valid ? util[j] : 0.0f;
    lr += (float)r;
    ln += conn[j] ? 1 : 0;
  }
  float usum = 0.0f, rsum = 0.0f;
  int nconn = 0;
#pragma unroll
  for (int i = 0; i < K; ++i) {  // lanes of the env in order: fixed association
    const int src = min(base + i, 31);
    usum += __shfl_sync(kFull, lu, src);
    rsum += __shfl_sync(kFull, lr, src);
    nconn += __shfl_sync(kFull, ln, src);
  }
  float bsu[B];
  if (MA) {  // allStationUtilities (base.py:438-447)
#pragma unroll
    for (int b = 0; b < B; ++b) {
      float part = 0.0f;
#pragma unroll
      for (int j = 0; j < UPT; ++j) part += ((conn[j] >> b) & 1u) ? util[j] : 0.0f;
      float sum = 0.0f;
#pragma unroll
      for (int i = 0; i < K; ++i) sum += __shfl_sync(kFull, part, min(base + i, 31));
      bsu[b] = cnt[b] ? sum / (float)cnt[b] : -1.0f;
    }
  }
  if (valid) {
#pragma unroll
    for (int j = 0; j < UPT; ++j) {
      if (a.rate) a.rate[idx[j]] = rate[j];
      a.utility[idx[j]] = util[j];
      if (MA) {
        float nu = 0.0f;
        int ncnt = 0;
#pragma unroll
        for (int b = 0; b < B; ++b)
          if ((elig[j] >> b) & 1u) {  // available_connections (base.py:216-218)
            nu += bsu[b];
            ncnt += cnt[b];
          }
        a.reward[idx[j]] = (nu + util[j]) / (float)(ncnt + 1);
      }
    }
    if (k == 0) {
      if (!MA) a.reward[env] = usum * a.inv_U;  // mean utility (metrics.py:25-28)
      if (a.metrics) {
        const float nc = (float)nconn;
        reinterpret_cast<float4*>(a.metrics)[env] = make_float4((float)csum, nc, usum * a.inv_U, mean_or_zero(rsum, nc));
      }
    }
  }

  // ---- move (movement.py:42-62) ----
  // (Issuing the rate gathers before the move, to hide their L2 latency behind it, was measured and
  // rejected, profiles/r02_h_variants.txt: the 24 registers of gathered doubles held across the
  // movement code spill at the 72-register budget, 18.2 vs 16.3 us per medium-central step, and a
  // 6-CTA budget loses as much in occupancy, 18.6 us.)
#pragma unroll
  for (int j = 0; j < UPT; ++j) {
    if (wx[j] < 0) next_waypoint(a, gid, (unsigned)(k + K * j), idx[j], t_e, epi, valid, wx[j], wy[j]);
    if (move_ue(a.mv[0], x[j], y[j], wx[j], wy[j])) wx[j] = wy[j] = -1;
  }

  // ---- clock, departures, same-step autoreset (base.py:280-291, 407-409; 172-209) ----
  t_e += 1;
  const bool done = valid && (t_e >= a.ep_time);
  const bool fresh = done && a.autoreset;
  if (valid && k == 0) a.done[env] = done ? 1 : 0;
  if (done) {
#pragma unroll
    for (int j = 0; j < UPT; ++j) conn[j] = 0;
#pragma unroll
    for (int b = 0; b < B; ++b) {
      cnt[b] = 0;
      if (MA) bsu[b] = -1.0f;
    }
  }
  if (fresh) {
    epi += 1;
    t_e = 0;
#pragma unroll
    for (int j = 0; j < UPT; ++j) {
      wx[j] = wy[j] = -1;
      philox_point(a, gid, (unsigned)(k + K * j), 0u, P_INITPOS, a.reset_rng_episode ? 0u : (unsigned)epi, x[j], y[j]);
      if (a.inj_wp) a.wp_cnt[idx[j]] = 0;
    }
    if (k == 0) a.episode[env] = epi;
  }

  // ---- observation of the new state into the staging block ----
  if (valid) {
#pragma unroll
    for (int j = 0; j < UPT; ++j) {
      float* row = s_obs + ((unsigned)env_in_blk * U + (unsigned)(k + K * j)) * F;
      if (done && !fresh) {  // inactive UEs observe zeros
#pragma unroll
        for (int f = 0; f < F; ++f) row[f] = 0.0f;
        continue;
      }
      float l[B];
      float lmax = -INFINITY;
      uint32_t elig2 = 0;
      const float xf = (float)x[j], yf = (float)y[j];
#pragma unroll
      for (int b = 0; b < B; ++b) {
        const float dx = xf - a.slot[b].xf, dy = yf - a.slot[b].yf;
        // exact: integers below 2^24; the 1e-32 (d = 0 is the reference's EPSILON, channels.py:8) vanishes
        // in the rounding of every d2 >= 1
        const float d2f = fmaf(dx, dx, fmaf(dy, dy, 1e-32f));
        l[b] = fmaf(-C0.k, lg2_sfu(d2f), C0.l0);
        lmax = fmaxf(lmax, l[b]);
        if (MA && d2f <= (float)C0.d2max) elig2 |= 1u << b;  // (d2max + 1e-32 rounds to d2max)
      }
#pragma unroll
      for (int b = 0; b < B; ++b) {
        row[b] = ((conn[j] >> b) & 1u) ? 1.0f : 0.0f;
        row[B + b] = ex2_sfu(l[b] - lmax);  // snr / max snr
      }
      row[2 * B] = fresh ? -1.0f : util[j];
      if (MA) {
        float c[B];
        float tsum = 0.0f;
#pragma unroll
        for (int b = 0; b < B; ++b) {
          const bool ok = (elig2 >> b) & 1u;
          c[b] = ok ? (float)cnt[b] : 0.0f;
          row[2 * B + 1 + b] = ok ? bsu[b] : -1.0f;
          tsum += c[b];
        }
        const float inv = 1.0f / fmaxf(1.0f, tsum);
#pragma unroll
        for (int b = 0; b < B; ++b) row[3 * B + 1 + b] = c[b] * inv;
      }
    }
  }

  // ---- store state (only what changed) ----
  if (valid) {
#pragma unroll
    for (int j = 0; j < UPT; ++j) {
      const uint32_t p = pack_xy(x[j], y[j]), w = pack_xy(wx[j], wy[j]);
      if (p != pos_in[j]) a.pos[idx[j]] = p;
      if (w != wp_in[j]) a.wp[idx[j]] = w;
      if (conn[j] != conn_in[j]) a.conn[idx[j]] = conn[j];
    }
    if (k == 0) a.t[env] = t_e;
  }
  store_obs_block<kUptThreads>(a, s_obs, env_base, tid, true);
}

}  // namespace mbe
