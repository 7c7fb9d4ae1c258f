// Fused step kernel, "warp-segment" mapping (U <= 32, B <= 32):
//   one thread per (env, UE); the U lanes of an env are a contiguous segment of a warp,
//   floor(32/U) envs per warp, 4 warps per block.  Global index of a lane = env*U + ue, so
//   every [E,U] stream is read/written fully coalesced; per-env reductions are warp
//   ballots / match / segmented shuffles; the observation block [envs of the CTA, U, F] is
//   staged in shared memory and leaves with ONE bulk async copy (TMA, UBLKCP in SASS).
#pragma once
#include "mbe_device.cuh"

namespace mbe {

struct Smem {
  float* obs;      // [epb*U*F]           (GYM)
  uint32_t* bs;    // [B] or [epb*B]      packed int16 x,y
  float* bsu;      // [epb*B] mean utility of the BS's UEs (allStationUtilities, base.py:438-447)
  int* bsn;        // [epb*B] |connections(bs)|
  uint8_t* cls;    // [B]
};

// Size of step_kernel's shared-memory carve-up for epb envs per CTA.  The kernel carves inline: through a
// layout function shared with this one its three instances compile to different code (register order).
__host__ __device__ inline size_t smem_bytes(int mode_gym, int handler_ma, int epb, int U, int B, int F,
                                            int bs_per_env) {
  size_t n = 0;
  if (mode_gym) n += (size_t)epb * U * F * 4;
  n = (n + 15) & ~(size_t)15;
  n += (size_t)(bs_per_env ? epb * B : B) * 4;
  if (mode_gym && handler_ma) n += (size_t)epb * B * 8;
  n += (size_t)B;
  return (n + 15) & ~(size_t)15;
}

template <int MODE, int HANDLER>
__global__ void __launch_bounds__(kThreads) step_kernel(const __grid_constant__ StepArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr bool GYM = (MODE == 1);
  constexpr bool MA = (HANDLER == 1);
  const int U = a.U, B = a.B, F = a.F;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // ---- shared memory carve-up ----
  Smem s;
  {
    size_t off = 0;
    s.obs = reinterpret_cast<float*>(smem_raw);
    if (GYM) off += (size_t)a.epb * U * F * 4;
    off = (off + 15) & ~(size_t)15;
    s.bs = reinterpret_cast<uint32_t*>(smem_raw + off);
    off += (size_t)(a.bs_per_env ? a.epb * B : B) * 4;
    s.bsu = reinterpret_cast<float*>(smem_raw + off);
    s.bsn = reinterpret_cast<int*>(smem_raw + off + (size_t)a.epb * B * 4);
    if (GYM && MA) off += (size_t)a.epb * B * 8;
    s.cls = smem_raw + off;
  }

  const int env_base = blockIdx.x * a.epb;
  // ---- stage the BS table (coalesced) ----
  if (a.bs_per_env) {
    const int n = min(a.epb, a.E - env_base) * B;
    const uint32_t* g = a.bs_xy + (size_t)env_base * B;
    for (int i = tid; i < n; i += kThreads) s.bs[i] = g[i];
  } else {
    for (int i = tid; i < B; i += kThreads) s.bs[i] = a.bs_xy[i];
  }
  for (int i = tid; i < B; i += kThreads) s.cls[i] = a.bs_class ? a.bs_class[i] : (uint8_t)0;
  __syncthreads();

  // ---- lane -> (env, ue) ----
  int seg = lane / U;
  int u = lane - seg * U;
  if (seg >= a.epw) {
    seg = a.epw;
    u = lane - a.epw * U;
  }
  const int env_in_blk = warp * a.epw + seg;
  const int env = env_base + env_in_blk;
  bool valid = (seg < a.epw) && (env < a.E);
  const unsigned segmask = valid ? (((U == 32) ? kFull : ((1u << U) - 1u)) << (seg * U)) : 0u;
  const size_t idx = (size_t)env * U + u;
  const unsigned gid = a.env_offset + (unsigned)env;
  const uint32_t* bs_tab = a.bs_per_env ? (s.bs + (size_t)min(env_in_blk, a.epb - 1) * B) : s.bs;
  // link class of (b, this UE) = bs_class[b] * n_ue_classes + ue_class[u] (entities.py:6-57)
  const int ucls = a.ue_class ? (int)a.ue_class[min(u, U - 1)] : 0;
  const int nuc = a.n_ue_classes;
  auto link = [&](int b) -> const ClassDev& { return a.cls[(int)s.cls[b] * nuc + ucls]; };
  const MoveDev& mv = a.mv[ucls];

  const int op = a.op;
  int ph = a.phases;
  bool touched = valid;  // this env's outputs are (re)written by this launch
  if (op == OP_RESET) {
    touched = valid && (a.reset_mask == nullptr || a.reset_mask[env] != 0);
    ph = GYM ? 8 : 0;
  } else if (op == OP_OBSERVE) {
    ph = GYM ? 8 : 0;
  }

  // ---- load state ----
  int x = 0, y = 0, wx = -1, wy = -1, t_e = 0, epi = 0, nb = B;
  uint32_t conn = 0;
  float util = -1.0f;
  if (valid) {
    unpack_xy(a.pos[idx], x, y);
    unpack_xy(a.wp[idx], wx, wy);
    t_e = a.t[env];
    epi = a.episode[env];
    if (a.nbs) nb = a.nbs[env];
    if (GYM) conn = a.conn[idx];
  }
  const uint32_t pos_in = pack_xy(x, y), wp_in = pack_xy(wx, wy), conn_in = conn;
  bool util_known = false;  // util computed in this launch
  bool done = false;
  bool fresh = false;       // env was re-initialised in this launch

  auto d2_to = [&](int b) {
    int bx, by;
    unpack_xy(bs_tab[b], bx, by);
    int dx = x - bx, dy = y - by;
    return dx * dx + dy * dy;
  };

  // per-BS statistics of the env into shared memory (MA only); all lanes of the warp call it
  auto bs_stats = [&](uint32_t cmask, float uval) {
    if (GYM && MA) {
      for (int b = 0; b < B; ++b) {
        bool bit = valid && ((cmask >> b) & 1u);
        unsigned m = __ballot_sync(kFull, bit) & segmask;
        float sum = seg_sum(bit ? uval : 0.0f, u, U, lane);
        if (valid && u == 0) {
          int n = __popc(m);
          s.bsn[env_in_blk * B + b] = n;
          s.bsu[env_in_blk * B + b] = n ? sum / (float)n : -1.0f;
        }
      }
      __syncwarp();
    }
  };

  // ---- MOVE: RandomWaypointMovement.move (movement.py:42-62) ----
  auto phase_move = [&]() {
    if (!valid) return;
    if (wx < 0) {  // no waypoint: draw one (movement.py:44-47)
      if (a.inj_wp) {
        int k = a.wp_cnt[idx];
        unpack_xy(a.inj_wp[idx * a.inj_k + min(k, a.inj_k - 1)], wx, wy);
        a.wp_cnt[idx] = k + 1;
      } else {
        philox_point(a, gid, (unsigned)u, (unsigned)t_e, P_WAYPOINT, a.reset_rng_episode ? 0u : (unsigned)epi,
                     wx, wy);
      }
    }
    if (move_ue(mv, x, y, wx, wy)) wx = wy = -1;
  };

  // ---- PRE (FORK): nearest connectable BS, ResourceFair split, utility (base.py:236-258) ----
  auto phase_pre_fork = [&]() {
    int best = -1, bestd2 = 0x7fffffff;
    if (valid) {
      for (int b = 0; b < nb; ++b) {
        int d2 = d2_to(b);
        if (d2 <= link(b).d2max && d2 < bestd2) {  // strict <: first minimum wins (base.py:240)
          best = b;
          bestd2 = d2;
        }
      }
    }
    // UEs of the same env attached to the same BS
    unsigned peers = __match_any_sync(kFull, (valid && best >= 0) ? (seg * 64 + best) : (0x10000 + lane));
    double rate = 0.0;
    if (valid && best >= 0) {
      int n = __popc(peers);
      const ClassDev& c = link(best);
      rate = c.lutn[(size_t)n * c.stride + bestd2];  // schedules.py:20-22, base.py:435
    }
    util = scaled_utility(a, rate);
    util_known = true;
    unsigned cm = __ballot_sync(kFull, valid && best >= 0) & segmask;
    float usum = seg_sum(valid ? util : 0.0f, u, U, lane);
    float rsum = seg_sum((float)rate, u, U, lane);
    if (valid) {
      a.assoc[idx] = best;
      if (a.rate) a.rate[idx] = rate;
      a.utility[idx] = util;
      if (a.metrics && u == 0) {
        float nc = (float)__popc(cm);
        reinterpret_cast<float4*>(a.metrics)[env] = make_float4(nc, nc, usum * a.inv_U, mean_or_zero(rsum, nc));
      }
      if (a.dbg_snr) {
        for (int b = 0; b < B; ++b)
          a.dbg_snr[idx * B + b] = (b < nb) ? ex2_sfu(log2_snr(link(b), d2_to(b))) : 0.0f;
      }
    }
  };

  // ---- PRE (GYM): update_connections, apply action, split, utility, reward ----
  uint32_t elig_pre = 0;
  auto phase_pre_gym = [&]() {
    if (valid) {
      for (int b = 0; b < nb; ++b)
        if (d2_to(b) <= link(b).d2max) elig_pre |= 1u << b;  // check_connectivity (base.py:212-214)
      conn &= elig_pre;  // update_connections (base.py:221-227)
      int act = a.actions[idx];
      if (act > 0 && act <= nb) {  // NOOP_ACTION = 0 (base.py:29)
        uint32_t bit = 1u << (act - 1);
        if (conn & bit) conn &= ~bit;
        else if (elig_pre & bit) conn |= bit;
      }
    }
    double rate = 0.0;
    for (int b = 0; b < B; ++b) {
      bool bit = (conn >> b) & 1u;
      unsigned m = __ballot_sync(kFull, bit) & segmask;
      if (bit) {  // allocateDataRate2User (base.py:421-435), bs-major accumulation (413-418)
        int n = __popc(m);
        const ClassDev& c = link(b);
        rate += c.lutn[(size_t)n * c.stride + d2_to(b)];
      }
    }
    util = scaled_utility(a, rate);
    util_known = true;
    float usum = seg_sum(valid ? util : 0.0f, u, U, lane);
    if (valid) {
      if (a.rate) a.rate[idx] = rate;
      a.utility[idx] = util;
    }
    if (MA) {
      bs_stats(conn, util);
      if (valid) {
        float nu = 0.0f;
        int ncnt = 0;
        for (int b = 0; b < nb; ++b)
          if ((elig_pre >> b) & 1u) {  // available_connections (base.py:216-218)
            nu += s.bsu[env_in_blk * B + b];
            ncnt += s.bsn[env_in_blk * B + b];
          }
        a.reward[idx] = (nu + util) / (float)(ncnt + 1);
      }
    } else if (valid && u == 0) {
      a.reward[env] = usum * a.inv_U;  // mean utility (metrics.py:25-28)
    }
    if (a.metrics) {
      unsigned cm = __ballot_sync(kFull, valid && conn != 0) & segmask;
      float csum = seg_sum((float)__popc(conn), u, U, lane);
      float rsum = seg_sum((float)rate, u, U, lane);
      if (valid && u == 0) {
        float nc = (float)__popc(cm);
        reinterpret_cast<float4*>(a.metrics)[env] = make_float4(csum, nc, usum * a.inv_U, mean_or_zero(rsum, nc));
      }
    }
    if (valid && a.dbg_snr) {
      for (int b = 0; b < B; ++b)
        a.dbg_snr[idx * B + b] = (b < nb) ? ex2_sfu(log2_snr(link(b), d2_to(b))) : 0.0f;
    }
  };

  auto reinit = [&](bool sel) {
    reinit_env(a, sel, gid, u, idx, env, a.bs_per_env ? s.bs + (size_t)min(env_in_blk, a.epb - 1) * B : nullptr, epi,
               t_e, conn, x, y, wx, wy, nb, fresh);
  };

  // ---- CLOCK: time += 1, departures, done (base.py:280-291, 407-409) ----
  auto phase_clock = [&]() {
    t_e += 1;
    done = valid && (t_e >= a.ep_time);
    if (done) conn = 0;  // everyone leaves at ep_time (arrival.py:32-36, base.py:283-285)
    if (valid && u == 0) a.done[env] = done ? 1 : 0;
    reinit(done && a.autoreset);
  };

  // ---- POST: observation of the (new) state into the staging block ----
  auto phase_post = [&]() {
    if (!GYM) return;
    if (!util_known && valid) util = a.utility[idx];
    // when CLOCK ran in an earlier launch (split phases, mbe_observe) the clock tells
    if (!(ph & 4)) done = valid && !fresh && (t_e >= a.ep_time);
    const bool is_fresh = fresh || (t_e == 0);
    if (MA) {
      // warp-collective: every lane takes part as soon as one env of the warp needs fresh
      // statistics; recomputing for the others reproduces the PRE values (same conn, util)
      const bool need = valid && (is_fresh || !util_known || done);
      if (__any_sync(kFull, need)) bs_stats((is_fresh || done) ? 0u : conn, util);
    }
    float* row = s.obs + ((size_t)env_in_blk * U + u) * F;
    if (!valid) return;
    if (done && !fresh) {  // inactive UEs observe zeros
      for (int f = 0; f < F; ++f) row[f] = 0.0f;
      return;
    }
    float lmax = -INFINITY;
    uint32_t elig = 0;
    for (int b = 0; b < nb; ++b) {
      const ClassDev& c = link(b);
      int d2 = d2_to(b);
      float l = log2_snr_obs(c, d2);
      row[B + b] = l;
      lmax = fmaxf(lmax, l);
      if (d2 <= c.d2max) elig |= 1u << b;
    }
    for (int b = 0; b < B; ++b) {
      row[b] = ((conn >> b) & 1u) ? 1.0f : 0.0f;
      row[B + b] = (b < nb) ? ex2_sfu(row[B + b] - lmax) : 0.0f;  // snr / max snr
    }
    row[2 * B] = is_fresh ? -1.0f : util;
    if (MA) {
      float tot = 0.0f;
      for (int b = 0; b < B; ++b) {
        bool ok = (elig >> b) & 1u;
        float n = ok ? (float)s.bsn[env_in_blk * B + b] : 0.0f;
        row[2 * B + 1 + b] = ok ? s.bsu[env_in_blk * B + b] : -1.0f;
        row[3 * B + 1 + b] = n;
        tot += n;
      }
      float inv = 1.0f / fmaxf(1.0f, tot);
      for (int b = 0; b < B; ++b) row[3 * B + 1 + b] *= inv;
    }
  };

  // ================= run =================
  if (op == OP_RESET) {
    reinit(touched);
    if (touched) {
      util = -1.0f;
      a.utility[idx] = -1.0f;
      if (u == 0) {
        a.done[env] = 0;
        if (GYM && !MA) a.reward[env] = 0.0f;
      }
      if (GYM && MA) a.reward[idx] = 0.0f;
      if (!GYM) a.assoc[idx] = -1;
      if (a.rate) a.rate[idx] = 0.0;
    }
    phase_post();
  } else if (op == OP_OBSERVE) {
    phase_post();
  } else if (!GYM) {
    if (ph & 1) phase_move();
    if (ph & 2) phase_pre_fork();
    if (ph & 4) phase_clock();
  } else {
    if (ph & 2) phase_pre_gym();
    if (ph & 1) phase_move();
    if (ph & 4) phase_clock();
    if (ph & 8) phase_post();
  }

  // ---- store state (only what changed) ----
  if (touched && op != OP_OBSERVE) {
    uint32_t p = pack_xy(x, y), w = pack_xy(wx, wy);
    if (p != pos_in) a.pos[idx] = p;
    if (w != wp_in) a.wp[idx] = w;
    if (GYM && (conn != conn_in || op == OP_RESET)) a.conn[idx] = conn;
    if (u == 0) {
      if ((ph & 4) || op == OP_RESET) a.t[env] = t_e;
    }
  }

  // ---- observation block leaves shared memory ----
  if (GYM && (ph & 8)) store_obs_block(a, s.obs, env_base, tid, op != OP_RESET || a.reset_mask == nullptr);
}

// Channel.calculateSNR for every pair (channels.py:24-27): thread per (env, ue), BS table in
// shared memory, lg2/ex2 on the SFU.  Used for per-stage parity and the SFU-pipe profile.
__global__ void __launch_bounds__(kThreads) channel_kernel(const __grid_constant__ StepArgs a, float* out_snr,
                                                           uint32_t* out_elig) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int U = a.U, B = a.B;
  const int per_blk = kThreads;  // (env,ue) pairs per block
  const size_t first = (size_t)blockIdx.x * per_blk;
  const size_t total = (size_t)a.E * U;
  uint32_t* sbs = reinterpret_cast<uint32_t*>(smem_raw);
  uint8_t* scls = smem_raw + 4 * (size_t)(a.bs_per_env ? (per_blk / U + 2) * B : B);
  const int e0 = (int)(first / U);
  if (a.bs_per_env) {
    const int e1 = (int)min((first + per_blk - 1) / U, (size_t)a.E - 1);
    const int n = (e1 - e0 + 1) * B;
    for (int i = threadIdx.x; i < n; i += kThreads) sbs[i] = a.bs_xy[(size_t)e0 * B + i];
  } else {
    for (int i = threadIdx.x; i < B; i += kThreads) sbs[i] = a.bs_xy[i];
  }
  for (int i = threadIdx.x; i < B; i += kThreads) scls[i] = a.bs_class ? a.bs_class[i] : (uint8_t)0;
  __syncthreads();
  const size_t idx = first + threadIdx.x;
  if (idx >= total) return;
  const int env = (int)(idx / U);
  const uint32_t* tab = a.bs_per_env ? sbs + (size_t)(env - e0) * B : sbs;
  int x, y;
  unpack_xy(a.pos[idx], x, y);
  const int nb = a.nbs ? a.nbs[env] : B;
  uint32_t elig = 0;
  for (int b = 0; b < B; ++b) {
    float snr = 0.0f;
    if (b < nb) {
      int bx, by;
      unpack_xy(tab[b], bx, by);
      int dx = x - bx, dy = y - by, d2 = dx * dx + dy * dy;
      const ClassDev& c = a.cls[(int)scls[b] * a.n_ue_classes + (a.ue_class ? (int)a.ue_class[idx % U] : 0)];
      snr = ex2_sfu(log2_snr(c, d2));
      if (d2 <= c.d2max) elig |= 1u << b;
    }
    if (out_snr) out_snr[idx * B + b] = snr;
  }
  if (out_elig) out_elig[idx] = elig;
}

// Episode statistics of the per-UE QoE behind the fork's layout score (chooseBaseStation.ipynb
// cell 5 `qoeValue`: mean - 0.1*var - 10*P(qoe < threshold) over all two-decimal QoE values of an
// epoch, as stored by base.py:269).  One warp per env adds this step's U values to acc[env] =
// (sum q, sum q^2, #q < threshold, #values); a fixed lane-strided order keeps it deterministic.
// q is qoe_cent_value (mbe_device.cuh): float32(k / 100) of the exact half-even cent k.
__global__ void __launch_bounds__(kThreads) qoe_accumulate_kernel(const float* __restrict__ utility, float4* acc, int E,
                                                                  int U, float threshold) {
  const int env = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (env >= E) return;
  float s1 = 0.0f, s2 = 0.0f, neg = 0.0f;
  for (int u = lane; u < U; u += 32) {
    const float q = qoe_cent_value(utility[(size_t)env * U + u]);  // round(qoe, 2)
    s1 += q;
    s2 = fmaf(q, q, s2);
    neg += (q < threshold) ? 1.0f : 0.0f;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s1 += __shfl_down_sync(kFull, s1, off);
    s2 += __shfl_down_sync(kFull, s2, off);
    neg += __shfl_down_sync(kFull, neg, off);
  }
  if (lane == 0) {
    float4 a = acc[env];
    acc[env] = make_float4(a.x + s1, a.y + s2, a.z + neg, a.w + (float)U);
  }
}

}  // namespace mbe
