// One generation of a genetic search over per-env BS layouts (DESIGN.md section 10): tournament
// selection, uniform slot crossover, bounded per-slot moves, add / delete of one BS, elites copied.
// Every decision is integer or FP64 arithmetic on Philox words, so oracle/evolve_ref.py reproduces
// every child bit for bit.
//
// One thread breeds one child.  Its row (B int16 pairs) is gathered from the parents (L2-resident at
// the sizes this runs at) into the CTA's shared block of child rows; the block, contiguous in the
// output, then leaves with coalesced 4-byte stores instead of one strided B-word row per thread.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mbe.h"
#include "mbe_device.cuh"

namespace mbe {

constexpr int kEvolveThreads = 128;
constexpr unsigned P_EVOLVE = 3u;  // Philox purpose word: reset draws use purpose + 4 * salt, purpose 0..2

struct EvolveArgs {
  const float* fitness;     // [E]
  const uint32_t* parent;   // int16 pairs [E,B]
  const int32_t* parent_nbs;  // [E]
  const int32_t* elite_ids;   // [K] or nullptr
  uint32_t* child;          // int16 pairs [E,B]
  int32_t* child_nbs;       // [E]
  int E, B, K, T, step, nmin, nmax;
  unsigned env_offset, generation, seed_lo, seed_hi;
  int XM, YM;               // inclusive coordinate range [0, XM] x [0, YM]
  int wh_int, wh_int_w, wh_int_h;  // new points: exactly philox_point's draw
  double width, height;
  double p_cross, p_move, p_add, p_del;
};

__device__ __forceinline__ bool evolve_coin(unsigned r, double p) { return (double)r * 0x1p-32 < p; }

// T candidates drawn with replacement from the words of one block; NaN fitness counts as -inf and
// a tie goes to the smaller index
__device__ __forceinline__ int evolve_tournament(const EvolveArgs& a, uint4 r) {
  const unsigned w[4] = {r.x, r.y, r.z, r.w};
  int best = (int)__umulhi(w[0], (unsigned)a.E);
  float bf = __ldg(a.fitness + best);
  if (bf != bf) bf = -INFINITY;
#pragma unroll
  for (int j = 1; j < 4; ++j) {
    if (j < a.T) {
      const int c = (int)__umulhi(w[j], (unsigned)a.E);
      float f = __ldg(a.fitness + c);
      if (f != f) f = -INFINITY;
      if (f > bf || (f == bf && c < best)) best = c, bf = f;
    }
  }
  return best;
}

__device__ __forceinline__ int evolve_clamp(int v, int hi) { return v < 0 ? 0 : (v > hi ? hi : v); }

__global__ void __launch_bounds__(kEvolveThreads) evolve_kernel(const EvolveArgs a) {
  extern __shared__ uint32_t srow[];  // [kEvolveThreads][B]
  const int tid = threadIdx.x, B = a.B;
  const int c0 = blockIdx.x * kEvolveThreads, c = c0 + tid;
  uint32_t* row = srow + tid * B;
  if (c < a.E) {
    const unsigned G = a.env_offset + (unsigned)c;
    const uint2 key = make_uint2(a.seed_lo, a.seed_hi);
    auto draw = [&](unsigned k) { return philox4x32_10(make_uint4(G, a.generation, k, P_EVOLVE), key); };
    const int elite = c < a.K ? __ldg(a.elite_ids + c) : -1;
    int n;
    if (elite >= 0 && elite < a.E) {  // verbatim copy, dead slots included
      const uint32_t* src = a.parent + (size_t)elite * B;
      for (int i = 0; i < B; ++i) row[i] = __ldg(src + i);
      n = __ldg(a.parent_nbs + elite);
    } else {
      const int p1 = evolve_tournament(a, draw(0u));
      const uint4 r2 = draw(2u);
      const bool cross = evolve_coin(r2.x, a.p_cross);
      const int p2 = cross ? evolve_tournament(a, draw(1u)) : p1;
      n = min(max(__ldg(a.parent_nbs + p1), 0), B);
      const int n2 = __ldg(a.parent_nbs + p2);
      const uint32_t* s1 = a.parent + (size_t)p1 * B;
      const uint32_t* s2 = a.parent + (size_t)p2 * B;
      const int span = 2 * a.step + 1;
      for (int i = 0; i < n; ++i) {
        const uint4 r = draw(4u + (unsigned)i);
        uint32_t v = __ldg((cross && i < n2 && (r.x >> 31)) ? s2 + i : s1 + i);
        if (evolve_coin(r.y, a.p_move)) {
          int x, y;
          unpack_xy(v, x, y);
          x = evolve_clamp(x + (int)__umulhi(r.z, (unsigned)span) - a.step, a.XM);
          y = evolve_clamp(y + (int)__umulhi(r.w, (unsigned)span) - a.step, a.YM);
          v = pack_xy(x, y);
        }
        row[i] = v;
      }
      if (evolve_coin(r2.y, a.p_add) && n < a.nmax) {
        const uint4 r = draw(3u);
        int x, y;
        if (a.wh_int) {
          x = (int)__umulhi(r.x, (unsigned)a.wh_int_w);
          y = (int)__umulhi(r.y, (unsigned)a.wh_int_h);
        } else {
          x = (int)((double)r.x * 0x1p-32 * a.width);
          y = (int)((double)r.y * 0x1p-32 * a.height);
        }
        row[n++] = pack_xy(x, y);
      } else if (evolve_coin(r2.z, a.p_del) && n > a.nmin) {
        row[__umulhi(r2.w, (unsigned)n)] = row[n - 1];
        --n;
      }
      for (int i = n; i < B; ++i) row[i] = 0u;
    }
    a.child_nbs[c] = n;
  }
  __syncthreads();
  // the CTA's child rows are one contiguous range of the output
  const int words = min(kEvolveThreads, a.E - c0) * B;
  uint32_t* dst = a.child + (size_t)c0 * B;
  for (int w = tid; w < words; w += kEvolveThreads) dst[w] = srow[w];
}

}  // namespace mbe
