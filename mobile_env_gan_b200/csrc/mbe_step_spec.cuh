// Specialised fused step kernels: U (UEs) and B (BS slots) are template constants, so every
// loop over b unrolls, BS coordinates of a shared layout are constant-bank operands (no
// shared-memory table, no unpacking) and the per-pair values stay in registers.
// Same warp-segment mapping and the same arithmetic helpers as the generic kernel
// (mbe_step.cuh), which remains the path for reset / observe / split phases and for shapes
// without an instantiation.  Only the whole fused step (OP_STEP, all phases) runs here.
// Preconditions checked by the dispatcher (mbe.cu): one BS class, width^2+height^2 < 2^24
// (squared distances are exact in FP32), no debug SNR output bound.
#pragma once
#include "mbe_device.cuh"

namespace mbe {

// Resident CTAs (128 threads) per SM the register allocation is held to, tuned per kernel on B200
// (profiles/README.md): the small central shapes run at full occupancy with 32 registers (10..16 CTAs
// measure the same within noise), the multi-agent and wide shapes need more registers for their
// per-BS arrays (large central 9 CTAs = 56 registers, large multi-agent 8 = 64).
constexpr int spec_min_blocks(int mode, int handler, int B) {
  return B <= 4 ? (handler == 1 ? 12 : 16) : B <= 10 ? (mode == 0 ? 11 : 10) : (handler == 1 ? 8 : 9);
}

// Envs per CTA of an instance and its dynamic shared memory: the observation staging block (GYM) at 0,
// then the per-env BS table (PER_ENV), then the multi-agent BS utilities and counts (GYM, multi-agent).
// The host sizes the launch with EPB and BYTES, the kernel carves its shared memory with the offsets.
template <int MODE, int HANDLER, int U, int B, bool PER_ENV>
struct SpecLayout {
  static constexpr int EPB = segment_envs_per_cta(U);
  static constexpr int F = MODE == 1 ? (HANDLER == 1 ? 4 : 2) * B + 1 : 0;
  static constexpr size_t BS = ((size_t)EPB * U * F * 4 + 15) & ~(size_t)15;
  static constexpr size_t BSU = BS + (PER_ENV ? (size_t)EPB * B * 4 : 0);
  static constexpr size_t BSN = BSU + (size_t)EPB * B * 4;
  static constexpr size_t BYTES = ((MODE == 1 && HANDLER == 1 ? BSN + (size_t)EPB * B * 4 : BSU) + 15) & ~(size_t)15;
};

// Shared / staged memory one chunk of envs (the envs of one CTA iteration) works on.
struct ChunkMem {
  float* obs;      // [EPB*U*F] observation staging block
  uint32_t* bs;    // [EPB*B] per-env BS table (PER_ENV)
  float* bsu;      // [EPB*B] multi-agent BS utilities
  int* bsn;        // [EPB*B] multi-agent BS connection counts
};

// One fused step of the EPB envs starting at env_base, state straight from global memory.  The
// observation block is left in m.obs; the caller stores it.  (Written inline in the kernel, the same
// body compiles differently: the compiler then bounds threadIdx.x by the launch bounds and allocates
// registers of the multi-agent instances anew, one of them with a spill.)
template <int MODE, int HANDLER, int U, int B, bool PER_ENV, bool MC = false>
__device__ __forceinline__ void step_chunk(const StepArgs& a, const int env_base, const ChunkMem& m) {
  constexpr bool GYM = (MODE == 1);
  constexpr bool MA = (HANDLER == 1);
  using L = SpecLayout<MODE, HANDLER, U, B, PER_ENV>;
  constexpr int EPW = envs_per_warp(U);
  constexpr int EPB = L::EPB;
  constexpr int F = L::F;
  constexpr unsigned SEG = (U == 32) ? kFull : ((1u << U) - 1u);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* s_obs = m.obs;
  uint32_t* s_bs = m.bs;
  float* s_bsu = m.bsu;
  int* s_bsn = m.bsn;

  int seg = lane / U;
  int u = lane - seg * U;
  if (seg >= EPW) {
    seg = EPW;
    u = lane - EPW * U;
  }
  const int env_in_blk = warp * EPW + seg;
  const int env = env_base + env_in_blk;
  const bool valid = (seg < EPW) && (env < a.E);
  const unsigned segmask = valid ? (SEG << (seg * U)) : 0u;
  // idle lanes (32 - EPW*U per warp, and the tail of the last block) run the same code on a
  // clamped index and only their stores are predicated off
  const int env_ld = valid ? env : 0;
  const unsigned idx = (unsigned)env_ld * U + (valid ? u : 0);
  const unsigned gid = a.env_offset + (unsigned)env;
  uint32_t* bs_env = PER_ENV ? s_bs + (size_t)min(env_in_blk, EPB - 1) * B : nullptr;
  // the slot's class constants.  MC: the BSs of a shared layout differ in bw/freq/tx/height
  // (entities.py:6-29) -- every slot has its own folded class, constant-bank operands once the loops
  // over b unroll; otherwise all slots share slot 0's (one register set)
  auto SL = [&](int b) -> const SlotDev& { return a.slot[MC ? b : 0]; };

  // ---- load state (all loads issued before any use) ----
  const uint32_t pos_in = a.pos[idx];
  const uint32_t wp_in = a.wp[idx];
  uint32_t conn = 0;
  int act = 0;
  if (GYM) {
    conn = a.conn[idx];
    act = a.actions[idx];
  }
  int t_e = a.t[env_ld];
  int epi = a.episode[env_ld];
  int nb = B;
  if (PER_ENV && a.nbs) nb = a.nbs[env_ld];
  int x, y, wx, wy;
  unpack_xy(pos_in, x, y);
  unpack_xy(wp_in, wx, wy);
  if (!valid) {
    conn = 0;
    act = 0;
  }
  const uint32_t conn_in = conn;
  bool done = false, fresh = false;
  float util = -1.0f;

  auto bs_xy_of = [&](int b, int& bx, int& by) {
    if (PER_ENV) {
      unpack_xy(bs_env[b], bx, by);
    } else {
      bx = a.slot[b].x;
      by = a.slot[b].y;
    }
  };
  auto d2_to = [&](int b) {
    int bx, by;
    bs_xy_of(b, bx, by);
    int dx = x - bx, dy = y - by;
    return dx * dx + dy * dy;
  };

  auto phase_move = [&]() {
    if (wx < 0) next_waypoint(a, gid, (unsigned)u, idx, t_e, epi, valid, wx, wy);  // movement.py:44-47
    if (move_ue(a.mv[0], x, y, wx, wy)) wx = wy = -1;
  };

  auto phase_clock = [&]() {
    t_e += 1;
    done = valid && (t_e >= a.ep_time);
    if (done) conn = 0;  // everyone leaves at ep_time (arrival.py:32-36, base.py:283-285)
    if (valid && u == 0) a.done[env] = done ? 1 : 0;
    if (__any_sync(kFull, done && a.autoreset))
      reinit_env(a, done && a.autoreset, gid, u, idx, env, bs_env, epi, t_e, conn, x, y, wx, wy, nb, fresh);
  };

  if (!GYM) {
    // ================= FORK: move -> associate -> split -> utility (base.py:230-296) =================
    phase_move();
    int best = -1, bestd2 = 0x7fffffff;
#pragma unroll
    for (int b = 0; b < B; ++b) {
      int d2 = d2_to(b);
      bool ok = (d2 <= SL(b).d2max) && (d2 < bestd2);  // strict <: first minimum wins (base.py:240)
      if (PER_ENV) ok = ok && (b < nb);
      if (ok) {
        best = b;
        bestd2 = d2;
      }
    }
    const bool has = valid && best >= 0;
    unsigned peers = __match_any_sync(kFull, has ? (seg * 64 + best) : (0x10000 + lane));
    double rate = 0.0;
    if (has) {
      const SlotDev& sb = SL(best);
      rate = sb.lutn[(unsigned)__popc(peers) * (unsigned)sb.stride + (unsigned)bestd2];
    }
    util = scaled_utility(a, rate);
    if (valid) {
      a.assoc[idx] = best;
      if (a.rate) a.rate[idx] = rate;
      a.utility[idx] = util;
    }
    if (a.metrics) {
      unsigned cm = __ballot_sync(kFull, has) & segmask;
      float usum = seg_sum_head<U>(valid ? util : 0.0f, u);
      float rsum = seg_sum_head<U>((float)rate, u);
      if (valid && u == 0) {
        float nc = (float)__popc(cm);
        reinterpret_cast<float4*>(a.metrics)[env] = make_float4(nc, nc, usum * a.inv_U, mean_or_zero(rsum, nc));
      }
    }
    phase_clock();
  } else {
    // ================= GYM: actions -> split -> utility -> reward -> move -> obs =================
    uint32_t elig = 0;
    int d2pre[B];
#pragma unroll
    for (int b = 0; b < B; ++b) {
      d2pre[b] = d2_to(b);
      bool ok = d2pre[b] <= SL(b).d2max;  // check_connectivity (base.py:212-214)
      if (PER_ENV) ok = ok && (b < nb);
      elig |= ok ? (1u << b) : 0u;
    }
    conn &= elig;  // update_connections (base.py:221-227)
    if (act > 0 && act <= nb) {  // NOOP_ACTION = 0 (base.py:29)
      uint32_t bit = 1u << (act - 1);
      conn = (conn & bit) ? (conn & ~bit) : (conn | (elig & bit));
    }
    // |connections(b)| for every BS of the env, then allocateDataRate2User (base.py:421-435):
    // the link's share comes from the pre-rounded table, bs-major accumulation (413-418); an
    // unconnected slot reads the table's 0.0 entry, so the loads need no predication
    int cnt[B];
    int csum_i = 0;
#pragma unroll
    for (int b = 0; b < B; ++b) {
      if constexpr (EPW == 1)  // the env is the whole warp (idle lanes hold conn = 0): one warp-wide integer add
        cnt[b] = (int)__reduce_add_sync(kFull, (conn >> b) & 1u);
      else
        cnt[b] = __popc(__ballot_sync(kFull, (conn >> b) & 1u) & segmask);
      csum_i += cnt[b];
    }
    double rate = 0.0;
#pragma unroll
    for (int b = 0; b < B; ++b) {
      const unsigned stride = (unsigned)SL(b).stride;
      unsigned off = (unsigned)cnt[b] * stride + (unsigned)d2pre[b];
      rate += SL(b).lutn[((conn >> b) & 1u) ? off : stride - 1u];
    }
    util = scaled_utility(a, rate);
    float usum = seg_sum_head<U>(valid ? util : 0.0f, u);
    if (valid) {
      if (a.rate) a.rate[idx] = rate;
      a.utility[idx] = util;
    }
    if (MA) {
#pragma unroll
      for (int b = 0; b < B; ++b) {
        bool bit = (conn >> b) & 1u;
        float sum = seg_sum_head<U>(bit ? util : 0.0f, u);
        if (valid && u == 0) {
          int n = cnt[b];
          s_bsn[env_in_blk * B + b] = n;
          s_bsu[env_in_blk * B + b] = n ? sum / (float)n : -1.0f;
        }
      }
      __syncwarp();
      if (valid) {
        float nu = 0.0f;
        int ncnt = 0;
#pragma unroll
        for (int b = 0; b < B; ++b)
          if ((elig >> b) & 1u) {  // available_connections (base.py:216-218)
            nu += s_bsu[env_in_blk * B + b];
            ncnt += s_bsn[env_in_blk * B + b];
          }
        a.reward[idx] = (nu + util) / (float)(ncnt + 1);
      }
    } else if (valid && u == 0) {
      a.reward[env] = usum * a.inv_U;  // mean utility (metrics.py:25-28)
    }
    if (a.metrics) {
      unsigned cm = __ballot_sync(kFull, conn != 0) & segmask;
      float csum = (float)csum_i;
      float rsum = seg_sum_head<U>((float)rate, u);
      if (valid && u == 0) {
        float nc = (float)__popc(cm);
        reinterpret_cast<float4*>(a.metrics)[env] = make_float4(csum, nc, usum * a.inv_U, mean_or_zero(rsum, nc));
      }
    }

    phase_move();
    phase_clock();

    // ---- observation of the new state ----
    if (MA) {
      // statistics change only for envs that ended (connections dropped / fresh episode)
      if (__any_sync(kFull, done)) {
        if (done && u == 0) {
#pragma unroll
          for (int b = 0; b < B; ++b) {
            s_bsn[env_in_blk * B + b] = 0;
            s_bsu[env_in_blk * B + b] = -1.0f;
          }
        }
        __syncwarp();
      }
    }
    if (valid) {
      float* row = s_obs + ((unsigned)env_in_blk * U + u) * F;
      if (done && !fresh) {  // inactive UEs observe zeros
#pragma unroll
        for (int f = 0; f < F; ++f) row[f] = 0.0f;
      } else {
        float l[B];
        float lmax = -INFINITY;
        uint32_t elig2 = 0;
        const float xf = (float)x, yf = (float)y;
#pragma unroll
        for (int b = 0; b < B; ++b) {
          float bxf, byf;
          if (PER_ENV) {
            int bx, by;
            unpack_xy(bs_env[b], bx, by);
            bxf = (float)bx;
            byf = (float)by;
          } else {
            bxf = a.slot[b].xf;
            byf = a.slot[b].yf;
          }
          float dx = xf - bxf, dy = yf - byf;
          float d2f = fmaf(dx, dx, dy * dy);  // exact: integers below 2^24
          l[b] = log2_snr_obs_f(SL(b).k, SL(b).l0, d2f);
          bool live = !PER_ENV || (b < nb);
          if (!live) l[b] = -INFINITY;
          lmax = fmaxf(lmax, l[b]);
          if (MA && live && d2f <= (float)SL(b).d2max) elig2 |= 1u << b;
        }
#pragma unroll
        for (int b = 0; b < B; ++b) {
          row[b] = ((conn >> b) & 1u) ? 1.0f : 0.0f;
          row[B + b] = ex2_sfu(l[b] - lmax);  // snr / max snr
        }
        row[2 * B] = fresh ? -1.0f : util;
        if (MA) {
          float cnt[B];
          float tot = 0.0f;
#pragma unroll
          for (int b = 0; b < B; ++b) {
            bool ok = (elig2 >> b) & 1u;
            cnt[b] = ok ? (float)s_bsn[env_in_blk * B + b] : 0.0f;
            row[2 * B + 1 + b] = ok ? s_bsu[env_in_blk * B + b] : -1.0f;
            tot += cnt[b];
          }
          float inv = 1.0f / fmaxf(1.0f, tot);
#pragma unroll
          for (int b = 0; b < B; ++b) row[3 * B + 1 + b] = cnt[b] * inv;
        }
      }
    }
  }

  // ---- store state (only what changed) ----
  if (valid) {
    uint32_t p = pack_xy(x, y), w = pack_xy(wx, wy);
    if (p != pos_in) a.pos[idx] = p;
    if (w != wp_in) a.wp[idx] = w;
    if (GYM && conn != conn_in) a.conn[idx] = conn;
    if (u == 0) {
      a.t[env] = t_e;
    }
  }
}

// ---- one chunk per CTA (works for any E) ----
template <int MODE, int HANDLER, int U, int B, bool PER_ENV, bool MC = false>
__global__ void __launch_bounds__(kThreads, spec_min_blocks(MODE, HANDLER, B)) step_spec_kernel(const __grid_constant__ StepArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr bool GYM = (MODE == 1);
  using L = SpecLayout<MODE, HANDLER, U, B, PER_ENV>;
  constexpr int EPB = L::EPB;
  // Programmatic dependent launch: let the next launch in the stream become resident while this
  // grid drains, and (as the dependent) wait for the previous grid's memory before touching state.
  // Both are no-ops when the launch does not carry the attribute.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  prefetch_ahead<EPB, U, GYM>(a);
  asm volatile("griddepcontrol.wait;" ::: "memory");
  ChunkMem m = {};
  m.obs = reinterpret_cast<float*>(smem_raw);
  m.bs = reinterpret_cast<uint32_t*>(smem_raw + L::BS);
  m.bsu = reinterpret_cast<float*>(smem_raw + L::BSU);
  m.bsn = reinterpret_cast<int*>(smem_raw + L::BSN);
  const int env_base = blockIdx.x * EPB;
  if (PER_ENV) {
    const int n = min(EPB, a.E - env_base) * B;
    const uint32_t* g = a.bs_xy + (size_t)env_base * B;
    for (int i = threadIdx.x; i < n; i += kThreads) m.bs[i] = g[i];
    __syncthreads();
  }
  step_chunk<MODE, HANDLER, U, B, PER_ENV, MC>(a, env_base, m);
  if (GYM) store_obs_block(a, m.obs, env_base, threadIdx.x, true);
}

}  // namespace mbe
