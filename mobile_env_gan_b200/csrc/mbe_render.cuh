// Map-panel frames of env states (DESIGN.md section 9): coverage, connection lines, BS squares, UE discs,
// painted with integer geometry only, so oracle/render_ref.py reproduces every byte.
//
// One CTA paints one band of `band_rows` full-width rows of one frame.  The band's palette indices live in
// shared memory while the layers are painted in painter's order; the last pass turns them into RGB and
// every warp stores its 32 quads (4 pixels = 12 bytes each) as 24 coalesced 16-byte words.  Entities are
// staged per CTA and culled to the band (rows), and each warp skips the entities whose bounding box
// misses its 128 pixels before the per-pixel tests.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>

#include "../../include/mbe.h"

namespace mbe {

constexpr int kRenderThreads = 256;
constexpr int kRenderWarps = kRenderThreads / 32;
constexpr int kRenderMaxBs = 64;              // two connection words per UE
constexpr int kRenderBandPixels = 4096;       // target pixels per CTA (rows are a multiple of 4)
constexpr int kRenderSegUes = 32;             // UEs whose lines are staged per pass (one per lane of warp 0)
enum { RP_BACKGROUND = 0, RP_COVERAGE = 1, RP_BS = 4, RP_UNCONNECTED = 5, RP_RAMP = 6 };

struct RenderArgs {
  const uint32_t* pos;      // int16 pairs, [E,U] (+ step * step_eu)
  const uint32_t* conn;     // GYM [E,U,MW]
  const int32_t* assoc;     // FORK [E,U] (+ step * step_eu)
  const float* utility;     // [E,U] (+ step * step_eu)
  const uint32_t* bs_xy;    // int16 pairs, [B] or [E,B]
  const int32_t* nbs;       // [E] or nullptr
  const uint8_t* bs_class;  // [B] or nullptr (all class 0)
  const int32_t* env_ids;   // [n] or nullptr
  uint8_t* out;             // [steps, n, H, W, 3]
  long long step_eu;        // E * U for a series, 0 for the bound state
  int E, U, B, MW, n, gym, bs_per_env;
  int Wm, Hm;               // int(width), int(height) of the map
  int band_rows, bands, seg_cap;
  int cov_d2max[MBE_MAX_CLASSES];  // per BS class: d2max of the link class (BS class, UE class 0)
};

struct RenderSeg {
  short ax, ay, dx, dy;  // UE pixel, BS pixel - UE pixel
  int len2;              // |B - A|^2
  int kmax;              // largest k with 4 k^2 <= w^2 len2: inside the projection, hit iff |cross| <= kmax
};

// floor division for a positive divisor (entity coordinates are int16 and may in principle be negative)
__device__ __forceinline__ int render_fdiv(int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

__device__ __forceinline__ int render_clamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// utility ramp index: clamp(floor((u + 1) * 128), 0, 255) in FP32, add rounded on its own (no FMA)
__device__ __forceinline__ int render_ramp(float u) {
  const float v = floorf(__fmul_rn(__fadd_rn(u, 1.0f), 128.0f));
  return v >= 255.0f ? 255 : (v > 0.0f ? (int)v : 0);
}

// shared-memory carve-up; the host sizes the launch with the same function
struct RenderSmem {
  size_t pal, bs, cov, ue_xy, ue_col, ue_mask, disc, seg, seg_col, xs, idx, xbuf, total;
};
__host__ __device__ inline RenderSmem render_smem_layout(int U, int W, int band_rows, int seg_cap) {
  auto up = [](size_t v) { return (v + 15) & ~(size_t)15; };
  RenderSmem s;
  size_t o = 0;
  s.pal = o;     o = up(o + 4 * MBE_RENDER_PALETTE);
  s.bs = o;      o = up(o + 8 * kRenderMaxBs);        // short4 (map x, map y, pixel x, pixel y)
  s.cov = o;     o = up(o + 8 * kRenderMaxBs);        // int2 (d2max, floor(sqrt(d2max)))
  s.ue_xy = o;   o = up(o + 4 * (size_t)U);           // short2 pixel position
  s.ue_col = o;  o = up(o + 2 * (size_t)U);           // palette index
  s.ue_mask = o; o = up(o + 8 * (size_t)U);           // live connection bits, two words
  s.disc = o;    o = up(o + 2 * (size_t)U);           // UEs whose disc meets the band
  s.seg = o;     o = up(o + sizeof(RenderSeg) * (size_t)seg_cap);
  s.seg_col = o; o = up(o + 2 * (size_t)seg_cap);
  s.xs = o;      o = up(o + 2 * (size_t)W);           // map x sampled by each pixel column
  s.idx = o;     o = up(o + 2 * (size_t)band_rows * W);
  s.xbuf = o;    o = up(o + 384 * (size_t)kRenderWarps);
  s.total = o;
  return s;
}

// pixel box of the 32 quads [q0, q0 + 32) of a band (clipped to nq): warp-uniform culling
struct RenderBox {
  int r_lo, r_hi, c_lo, c_hi;
};
__device__ __forceinline__ RenderBox render_box(int q0, int nq, int wq, int r0) {
  const int q1 = min(q0 + 31, nq - 1);
  RenderBox b;
  b.r_lo = r0 + q0 / wq;
  b.r_hi = r0 + q1 / wq;
  b.c_lo = b.r_lo == b.r_hi ? (q0 % wq) * 4 : 0;
  b.c_hi = b.r_lo == b.r_hi ? (q1 % wq) * 4 + 3 : wq * 4 - 1;
  return b;
}

__global__ void __launch_bounds__(kRenderThreads) render_kernel(RenderArgs a, mbe_render_style st) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int H = st.height, W = st.width, wq = W >> 2;
  const RenderSmem L = render_smem_layout(a.U, W, a.band_rows, a.seg_cap);
  uint32_t* pal = reinterpret_cast<uint32_t*>(smem + L.pal);
  short4* bsd = reinterpret_cast<short4*>(smem + L.bs);
  int2* cov = reinterpret_cast<int2*>(smem + L.cov);
  short2* ue_xy = reinterpret_cast<short2*>(smem + L.ue_xy);
  uint16_t* ue_col = reinterpret_cast<uint16_t*>(smem + L.ue_col);
  uint2* ue_mask = reinterpret_cast<uint2*>(smem + L.ue_mask);
  uint16_t* disc = reinterpret_cast<uint16_t*>(smem + L.disc);
  RenderSeg* seg = reinterpret_cast<RenderSeg*>(smem + L.seg);
  uint16_t* seg_col = reinterpret_cast<uint16_t*>(smem + L.seg_col);
  int16_t* xs_tab = reinterpret_cast<int16_t*>(smem + L.xs);
  uint16_t* idx = reinterpret_cast<uint16_t*>(smem + L.idx);
  __shared__ int s_ndisc, s_nseg;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long frame = blockIdx.x / a.bands;
  const int band = (int)(blockIdx.x - frame * a.bands);
  const int k = (int)(frame % a.n), step = (int)(frame / a.n);
  const int e = a.env_ids ? a.env_ids[k] : k;
  const bool valid = e >= 0 && e < a.E;  // an id out of range paints the background only
  const int r0 = band * a.band_rows, rows = min(a.band_rows, H - r0);
  const int nq = rows * wq;
  const int nb = !valid ? 0 : (a.nbs ? render_clamp(a.nbs[e], 0, a.B) : a.B);
  const int R = st.ue_radius, S = st.bs_half, Wl = st.line_width;
  const int lm = (Wl + 1) >> 1;  // line half-width, rounded up: bounding-box margin

  // ---- staging: palette, map x per column, BSs, UEs ----
  for (int i = tid; i < MBE_RENDER_PALETTE; i += kRenderThreads)
    pal[i] = st.palette[i][0] | ((uint32_t)st.palette[i][1] << 8) | ((uint32_t)st.palette[i][2] << 16);
  for (int j = tid; j < W; j += kRenderThreads) xs_tab[j] = (int16_t)(((2 * j + 1) * a.Wm) / (2 * W));
  if (tid < nb) {
    const uint32_t xy = a.bs_xy[(a.bs_per_env ? (size_t)e * a.B : 0) + tid];
    const int bx = (int16_t)(xy & 0xffffu), by = (int16_t)(xy >> 16);
    const int cx = render_clamp(render_fdiv(bx * W, a.Wm), 0, W - 1);
    const int cy = render_clamp(H - 1 - render_fdiv(by * H, a.Hm), 0, H - 1);
    bsd[tid] = make_short4((short)bx, (short)by, (short)cx, (short)cy);
    const int d2 = a.cov_d2max[a.bs_class ? a.bs_class[tid] : 0];
    int rad = d2 < 0 ? -1 : (int)sqrtf((float)d2);
    while (rad >= 0 && rad * rad > d2) --rad;
    while (d2 >= 0 && (rad + 1) * (rad + 1) <= d2) ++rad;
    cov[tid] = make_int2(d2, rad);
  }
  const size_t eu = valid ? (size_t)step * a.step_eu + (size_t)e * a.U : 0;
  for (int u = tid; u < (valid ? a.U : 0); u += kRenderThreads) {
    const uint32_t xy = a.pos[eu + u];
    const int x = (int16_t)(xy & 0xffffu), y = (int16_t)(xy >> 16);
    uint2 m = make_uint2(0u, 0u);
    if (a.gym) {
      const uint32_t* c = a.conn + ((size_t)e * a.U + u) * a.MW;
      m.x = c[0];
      if (a.MW > 1) m.y = c[1];
    } else {
      const int b = a.assoc[eu + u];
      if (b >= 0 && b < 32) m.x = 1u << b;
      else if (b >= 32 && b < 64) m.y = 1u << (b - 32);
    }
    // only live slots are drawn or count as a connection
    m.x &= nb >= 32 ? 0xffffffffu : ((1u << nb) - 1u);
    m.y &= nb >= 64 ? 0xffffffffu : (nb <= 32 ? 0u : ((1u << (nb - 32)) - 1u));
    ue_xy[u] = make_short2((short)render_clamp(render_fdiv(x * W, a.Wm), 0, W - 1),
                           (short)render_clamp(H - 1 - render_fdiv(y * H, a.Hm), 0, H - 1));
    ue_mask[u] = m;
    ue_col[u] = (uint16_t)((m.x | m.y) ? RP_RAMP + render_ramp(a.utility[eu + u]) : RP_UNCONNECTED);
  }
  __syncthreads();
  // discs that meet the band, in UE order (warp 0, ballot compaction)
  if (warp == 0) {
    int cnt = 0;
    for (int u0 = 0; u0 < (valid ? a.U : 0); u0 += 32) {
      const int u = u0 + lane;
      const bool hit = u < a.U && ue_xy[u].y + R >= r0 && ue_xy[u].y - R < r0 + rows;
      const unsigned bal = __ballot_sync(kFull, hit);
      if (hit) disc[cnt + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)u;
      cnt += __popc(bal);
    }
    if (lane == 0) s_ndisc = cnt;
  }

  // ---- layers 1 + 2: background and coverage counts ----
  for (int q0 = warp * 32; q0 < nq; q0 += kRenderWarps * 32) {
    const RenderBox bx = render_box(q0, nq, wq, r0);
    const int ys_lo = ((2 * (H - 1 - bx.r_hi) + 1) * a.Hm) / (2 * H);
    const int ys_hi = ((2 * (H - 1 - bx.r_lo) + 1) * a.Hm) / (2 * H);
    const int xs_lo = xs_tab[bx.c_lo], xs_hi = xs_tab[bx.c_hi];
    const int q = q0 + lane;
    const bool on = q < nq;
    const int i = r0 + (on ? q / wq : 0), j0 = (on ? q % wq : 0) * 4;
    const int ys = ((2 * (H - 1 - i) + 1) * a.Hm) / (2 * H);
    int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int b = 0; b < nb; ++b) {
      const int2 cv = cov[b];
      const short4 p = bsd[b];
      if (cv.y < 0 || p.x + cv.y < xs_lo || p.x - cv.y > xs_hi || p.y + cv.y < ys_lo || p.y - cv.y > ys_hi) continue;
      const int dy = ys - p.y;
      if (dy > cv.y || -dy > cv.y) continue;
      // |dx| < 2^16, so dx^2 is exact in unsigned 32-bit arithmetic; rem >= 0 because |dy| <= rad
      const unsigned rem = (unsigned)(cv.x - dy * dy);
      unsigned dx = (unsigned)(xs_tab[j0] - p.x);     c0 += dx * dx <= rem;
      dx = (unsigned)(xs_tab[j0 + 1] - p.x);          c1 += dx * dx <= rem;
      dx = (unsigned)(xs_tab[j0 + 2] - p.x);          c2 += dx * dx <= rem;
      dx = (unsigned)(xs_tab[j0 + 3] - p.x);          c3 += dx * dx <= rem;
    }
    if (on) {
      const uint32_t lo = min(c0, 3) | ((uint32_t)min(c1, 3) << 16), hi = min(c2, 3) | ((uint32_t)min(c3, 3) << 16);
      reinterpret_cast<uint2*>(idx)[q] = make_uint2(lo, hi);  // tint index = count (0 = background)
    }
  }
  __syncthreads();

  // ---- layer 3: connection lines, 32 UEs per pass (UE order, then BS order) ----
  const int e2 = (Wl * Wl) >> 2;  // endpoint test: 4 d^2 <= w^2  <=>  d^2 <= floor(w^2 / 4)
  for (int u0 = 0; u0 < (valid ? a.U : 0); u0 += kRenderSegUes) {
    if (warp == 0) {
      const int u = u0 + lane;
      uint2 m = u < a.U ? ue_mask[u] : make_uint2(0u, 0u);
      short2 p = u < a.U ? ue_xy[u] : make_short2(0, 0);
      // count this lane's segments whose box meets the band, then write them in (UE, BS) order
      int mine = 0;
      for (int w = 0; w < 2; ++w)
        for (uint32_t bits = w ? m.y : m.x; bits; bits &= bits - 1) {
          const short4 q = bsd[w * 32 + __ffs(bits) - 1];
          mine += min(p.y, q.w) - lm < r0 + rows && max(p.y, q.w) + lm >= r0;
        }
      int incl = mine;
      for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(kFull, incl, d);
        if (lane >= d) incl += v;
      }
      int o = incl - mine;
      for (int w = 0; w < 2; ++w)
        for (uint32_t bits = w ? m.y : m.x; bits; bits &= bits - 1) {
          const short4 q = bsd[w * 32 + __ffs(bits) - 1];
          if (!(min(p.y, q.w) - lm < r0 + rows && max(p.y, q.w) + lm >= r0)) continue;
          RenderSeg s;
          s.ax = p.x, s.ay = p.y, s.dx = (short)(q.z - p.x), s.dy = (short)(q.w - p.y);
          s.len2 = s.dx * s.dx + s.dy * s.dy;
          const long long rhs = (long long)Wl * Wl * s.len2;  // 4 k^2 <= rhs
          long long kk = (long long)sqrt((double)rhs * 0.25);
          while (kk > 0 && 4 * kk * kk > rhs) --kk;
          while (4 * (kk + 1) * (kk + 1) <= rhs) ++kk;
          s.kmax = (int)kk;
          seg[o] = s;
          seg_col[o] = ue_col[u];
          ++o;
        }
      if (lane == 31) s_nseg = incl;
    }
    __syncthreads();
    const int ns = s_nseg;
    if (ns > 0) {
      for (int q0 = warp * 32; q0 < nq; q0 += kRenderWarps * 32) {
        const RenderBox bx = render_box(q0, nq, wq, r0);
        const int q = q0 + lane;
        const bool on = q < nq;
        const int i = r0 + (on ? q / wq : 0), j0 = (on ? q % wq : 0) * 4;
        uint2 cur = on ? reinterpret_cast<uint2*>(idx)[q] : make_uint2(0u, 0u);
        uint32_t c[4] = {cur.x & 0xffffu, cur.x >> 16, cur.y & 0xffffu, cur.y >> 16};
        bool any = false;
        for (int t = 0; t < ns; ++t) {
          const RenderSeg s = seg[t];
          const int bxe = s.ax + s.dx, bye = s.ay + s.dy;
          if (min(s.ax, bxe) - lm > bx.c_hi || max(s.ax, bxe) + lm < bx.c_lo || min(s.ay, bye) - lm > bx.r_hi ||
              max(s.ay, bye) + lm < bx.r_lo)
            continue;
          const int ry = i - s.ay;
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            const int rx = j0 + p - s.ax;
            const int tt = s.dx * rx + s.dy * ry;
            bool hit;
            if (tt <= 0) {
              hit = rx * rx + ry * ry <= e2;
            } else if (tt >= s.len2) {
              const int ux = rx - s.dx, uy = ry - s.dy;
              hit = ux * ux + uy * uy <= e2;
            } else {
              const int cr = s.dx * ry - s.dy * rx;
              hit = (cr < 0 ? -cr : cr) <= s.kmax;
            }
            if (hit) c[p] = seg_col[t], any = true;
          }
        }
        if (on && any) reinterpret_cast<uint2*>(idx)[q] = make_uint2(c[0] | (c[1] << 16), c[2] | (c[3] << 16));
      }
    }
    __syncthreads();
  }

  // ---- layers 4 + 5 (BS squares, UE discs), palette lookup, coalesced store ----
  const int ndisc = s_ndisc;
  uint32_t* xb = reinterpret_cast<uint32_t*>(smem + L.xbuf) + warp * 96;
  uint8_t* fout = a.out + (size_t)frame * H * W * 3;
  for (int q0 = warp * 32; q0 < nq; q0 += kRenderWarps * 32) {
    const RenderBox bx = render_box(q0, nq, wq, r0);
    const int q = q0 + lane;
    const bool on = q < nq;
    const int i = r0 + (on ? q / wq : 0), j0 = (on ? q % wq : 0) * 4;
    uint2 cur = on ? reinterpret_cast<uint2*>(idx)[q] : make_uint2(0u, 0u);
    uint32_t c[4] = {cur.x & 0xffffu, cur.x >> 16, cur.y & 0xffffu, cur.y >> 16};
    for (int b = 0; b < nb; ++b) {
      const short4 p = bsd[b];
      if (p.z + S < bx.c_lo || p.z - S > bx.c_hi || p.w + S < bx.r_lo || p.w - S > bx.r_hi) continue;
      const int dy = i - p.w;
      if (dy > S || -dy > S) continue;
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const int dx = j0 + k4 - p.z;
        if (dx <= S && -dx <= S) c[k4] = RP_BS;
      }
    }
    for (int t = 0; t < ndisc; ++t) {
      const int u = disc[t];
      const short2 p = ue_xy[u];
      if (p.x + R < bx.c_lo || p.x - R > bx.c_hi || p.y + R < bx.r_lo || p.y - R > bx.r_hi) continue;
      const int dy = i - p.y, rem = R * R - dy * dy;
      if (rem < 0) continue;
      const uint32_t col = ue_col[u];
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const int dx = j0 + k4 - p.x;
        if (dx * dx <= rem) c[k4] = col;
      }
    }
    // 4 pixels = 12 bytes = 3 words, staged per warp, then stored as 16-byte words where aligned
    const uint32_t p0 = pal[c[0]], p1 = pal[c[1]], p2 = pal[c[2]], p3 = pal[c[3]];
    xb[3 * lane] = p0 | (p1 << 24);
    xb[3 * lane + 1] = (p1 >> 8) | (p2 << 16);
    xb[3 * lane + 2] = (p2 >> 16) | (p3 << 8);
    __syncwarp();
    const int nquads = min(32, nq - q0);
    uint8_t* dst = fout + ((size_t)r0 * wq + q0) * 12;
    const int words = nquads * 3;
    if ((((uintptr_t)dst) & 15) == 0 && (words & 3) == 0) {
      if (lane < (words >> 2))
        reinterpret_cast<uint4*>(dst)[lane] = reinterpret_cast<const uint4*>(xb)[lane];
    } else {
      for (int w = lane; w < words; w += 32) reinterpret_cast<uint32_t*>(dst)[w] = xb[w];
    }
    __syncwarp();
  }
}

}  // namespace mbe
