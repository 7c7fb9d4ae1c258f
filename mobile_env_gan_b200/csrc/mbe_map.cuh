// Layout maps (DESIGN.md section 10.2): at every point of a stride-s grid over the map, per env, the number of
// connectable BSs, the BS the FORK association rule picks and the QoE cent of a UE served there, plus the
// map-wide integer statistics of the layout.  Integer arithmetic and byte gathers only, so
// oracle/map_ref.py reproduces every output exactly.
//
// Two launches.  map_prep_kernel tabulates the cent per (BS class, d2 <= d2max) with the step kernels'
// device helpers and zeroes the statistics rows.  map_kernel runs one CTA per (output row, band of
// kMapPoints consecutive grid points): the env's connectable live BSs sit in shared memory, each thread
// takes 4 consecutive points per pass and writes one 4-byte word per map, the statistics are reduced per
// warp with shuffles and leave with one 64-bit atomic per statistic per CTA.
#pragma once
#include "mbe_device.cuh"
#include "../../include/mbe.h"

namespace mbe {

constexpr int kMapThreads = 256;
constexpr int kMapQuads = 4;                             // passes of 4 points per thread
constexpr int kMapPoints = kMapThreads * 4 * kMapQuads;  // grid points per CTA
constexpr int kMapMaxB = 64;
constexpr int kMapStats = 6;  // points, covered, overlap, sum k, sum k^2, low

struct MapArgs {
  const uint32_t* bs_xy;    // per-env layouts [E,B] (int16 pairs), nullptr: the shared layout xy below
  const int32_t* nbs;       // [E] or nullptr
  const int32_t* env_ids;   // [n] or nullptr (envs 0..n-1)
  const uint8_t* bs_class;  // [B] or nullptr (all class 0)
  int8_t* cent;             // cent table: BS class c at cent + off[c], d2 = 0..d2max[c]
  long long* stats;         // [n, kMapStats] or nullptr
  int32_t* area;            // [n, B] or nullptr
  uint8_t* coverage;        // [n, G] or nullptr
  int8_t* serving;          // [n, G] or nullptr
  int8_t* qoe;              // [n, G] or nullptr
  int E, B, n, s, GX, G, bands;
  int k_low;     // a cent k is low QoE iff k < k_low
  int vec;       // G % 4 == 0 and the maps are 4-byte aligned: one word per 4 points
  int n_classes; // BS classes
  int tab_len;   // entries of the cent table
  double load;   // UEs sharing the serving BS
  int d2max[MBE_MAX_CLASSES];  // per BS class: d2max of the link class (BS class, UE class), -1 never
  int off[MBE_MAX_CLASSES];    // per BS class: its first entry in the cent table
  int link[MBE_MAX_CLASSES];   // per BS class: its link class with the map's UE class
  uint32_t xy[kMapMaxB];       // shared layout: the coordinates mbe_bind captured
};

// Cent of a UE at squared distance d2 from a BS of class c that it shares with load - 1 others: the rate
// round(rate_lut[d2] / load, 2) in FP64 as mbe_create folds lutn, then scaled_utility and qoe_cent.
__global__ void __launch_bounds__(kMapThreads) map_prep_kernel(const __grid_constant__ StepArgs a,
                                                               const __grid_constant__ MapArgs m) {
  const long long i = (long long)blockIdx.x * kMapThreads + threadIdx.x;
  if (i < m.tab_len) {
    int c = 0;
    for (int t = 0; t < m.n_classes; ++t)
      if (m.d2max[t] >= 0 && i >= m.off[t] && i - m.off[t] <= m.d2max[t]) c = t;
    const int d2 = (int)(i - m.off[c]);
    const double share = __ddiv_rn(a.cls[m.link[c]].lut0[d2], m.load);
    const double rate = __ddiv_rn(rint(__dmul_rn(share, 100.0)), 100.0);
    m.cent[i] = (int8_t)qoe_cent(scaled_utility(a, rate));
  }
  if (m.stats && i < (long long)m.n * kMapStats) m.stats[i] = 0;
  if (m.area && i < (long long)m.n * m.B) m.area[i] = 0;
}

__device__ __forceinline__ int map_warp_sum(int v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
  return v;
}

__global__ void __launch_bounds__(kMapThreads) map_kernel(const __grid_constant__ MapArgs m) {
  __shared__ int4 sbs[kMapMaxB];  // x, y, d2max, cent-table offset of the connectable live BSs, in slot order
  __shared__ int sslot[kMapMaxB];
  __shared__ int sarea[kMapMaxB];
  __shared__ long long sred[kMapThreads / 32][kMapStats - 1];
  __shared__ int s_nl;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int k = (int)(blockIdx.x / (unsigned)m.bands), band = (int)(blockIdx.x - (unsigned)k * m.bands);
  const int e = m.env_ids ? m.env_ids[k] : k;
  const bool valid = e >= 0 && e < m.E;  // an id out of range gives an empty map and zero statistics
  const int nb = !valid ? 0 : (m.nbs ? min(max(m.nbs[e], 0), m.B) : m.B);
  if (warp == 0) {
    int cnt = 0;
    for (int b0 = 0; b0 < m.B; b0 += 32) {
      const int b = b0 + lane;
      const int c = b < nb ? (m.bs_class ? (int)m.bs_class[b] : 0) : 0;
      const bool keep = b < nb && m.d2max[c] >= 0;
      const unsigned bal = __ballot_sync(kFull, keep);
      if (keep) {
        const int o = cnt + __popc(bal & ((1u << lane) - 1u));
        int x, y;
        unpack_xy(m.bs_xy ? m.bs_xy[(size_t)e * m.B + b] : m.xy[b], x, y);
        sbs[o] = make_int4(x, y, m.d2max[c], m.off[c]);
        sslot[o] = b;
      }
      cnt += __popc(bal);
    }
    if (lane == 0) s_nl = cnt;
  }
  for (int b = tid; b < m.B; b += kMapThreads) sarea[b] = 0;
  __syncthreads();
  const int nl = s_nl;

  const int p_begin = band * kMapPoints, p_end = min(m.G, p_begin + kMapPoints);
  const size_t row = (size_t)k * m.G;
  int n_cov = 0, n_ovl = 0, sum_k = 0, sum_k2 = 0, n_low = 0;
  int run_b = -1, run_n = 0;  // serving slot of the last points, and how many (area, flushed on change)
  for (int q = 0; q < kMapQuads; ++q) {
    const int p0 = p_begin + 4 * (q * kMapThreads + tid);
    if (p0 >= p_end) break;
    int j = p0 / m.GX, i = p0 - j * m.GX;
    int xs[4], ys[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      xs[t] = i * m.s;
      ys[t] = j * m.s;
      if (++i == m.GX) i = 0, ++j;
    }
    // d2 <= d2max as dx^2 <= d2max and dy^2 <= d2max - dx^2: every term is exact in unsigned 32-bit
    // arithmetic (|dx|, |dy| < 2^16, d2max < 2^31), and a connectable d2 is below 2^31
    unsigned best_d2[4] = {~0u, ~0u, ~0u, ~0u};
    int best[4] = {-1, -1, -1, -1}, cov[4] = {0, 0, 0, 0};
    for (int t = 0; t < nl; ++t) {
      const int4 b = sbs[t];
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const unsigned dx = (unsigned)(xs[p] - b.x), dy = (unsigned)(ys[p] - b.y);
        const unsigned dxx = dx * dx, dyy = dy * dy;
        const bool in = dxx <= (unsigned)b.z && dyy <= (unsigned)b.z - dxx;
        const unsigned d2 = dxx + dyy;
        cov[p] += in;
        if (in && d2 < best_d2[p]) {  // strict <: the lowest slot of the nearest ones (FORK association)
          best_d2[p] = d2;
          best[p] = t;
        }
      }
    }
    uint32_t wc = 0, ws = 0, wq = 0;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const bool on = p0 + p < p_end;
      int slot = -1, kq = valid ? -100 : -128;  // no server: rate 0, utility -1
      if (best[p] >= 0) {
        slot = sslot[best[p]];
        kq = m.cent[sbs[best[p]].w + best_d2[p]];
      }
      wc |= (uint32_t)min(cov[p], 255) << (8 * p);
      ws |= (uint32_t)(uint8_t)slot << (8 * p);
      wq |= (uint32_t)(uint8_t)kq << (8 * p);
      if (on && valid) {
        n_cov += cov[p] >= 1;
        n_ovl += cov[p] >= 2;
        sum_k += kq;
        sum_k2 += kq * kq;
        n_low += kq < m.k_low;
        if (slot != run_b) {
          if (run_n) atomicAdd(&sarea[run_b], run_n);
          run_b = slot, run_n = 0;
        }
        run_n += slot >= 0;
      }
    }
    const size_t o = row + p0;
    if (m.vec && p0 + 3 < p_end) {
      if (m.coverage) *reinterpret_cast<uint32_t*>(m.coverage + o) = wc;
      if (m.serving) *reinterpret_cast<uint32_t*>(m.serving + o) = ws;
      if (m.qoe) *reinterpret_cast<uint32_t*>(m.qoe + o) = wq;
    } else {
      for (int p = 0; p < 4 && p0 + p < p_end; ++p) {
        if (m.coverage) m.coverage[o + p] = (uint8_t)(wc >> (8 * p));
        if (m.serving) m.serving[o + p] = (int8_t)(ws >> (8 * p));
        if (m.qoe) m.qoe[o + p] = (int8_t)(wq >> (8 * p));
      }
    }
  }
  if (!valid) return;  // (uniform over the CTA)
  if (run_n) atomicAdd(&sarea[run_b], run_n);
  if (m.stats) {
    const int v[kMapStats - 1] = {map_warp_sum(n_cov), map_warp_sum(n_ovl), map_warp_sum(sum_k), map_warp_sum(sum_k2),
                                  map_warp_sum(n_low)};
    if (lane == 0)
      for (int i = 0; i < kMapStats - 1; ++i) sred[warp][i] = v[i];
  }
  __syncthreads();
  if (m.stats && tid < kMapStats) {
    long long v = p_end - p_begin;
    if (tid > 0) {
      v = 0;
      for (int w = 0; w < kMapThreads / 32; ++w) v += sred[w][tid - 1];
    }
    if (v) atomicAdd(reinterpret_cast<unsigned long long*>(m.stats + (size_t)k * kMapStats + tid), (unsigned long long)v);
  }
  if (m.area)
    for (int b = tid; b < m.B; b += kMapThreads)
      if (sarea[b]) atomicAdd(m.area + (size_t)k * m.B + b, sarea[b]);
}

}  // namespace mbe
