// radix_select.cuh -- exact order statistics of a float row by radix select, shared by psis_kernel (loo.cu) and
// market_quantile_kernel (markets.cu): order-preserving keys, warp-aggregated histogram adds, the block-wide search
// for the bin that holds a rank, and the strided row walk.  A select takes three passes over the row: a histogram of
// the top 11 key bits, then of the next 11 bits within the chosen top bin, then of the last 10 bits.
#pragma once
#include "common.cuh"

namespace bplx {
namespace radix {

constexpr int kBins = 2048;  // radix digits of 11, 11 and 10 bits

// order-preserving keys: ascending key <=> ascending float
__device__ __forceinline__ uint32_t f2key(float v) {
  const uint32_t u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// For every r < MAXR in the bit mask `which`: the bin of hist[0, nb) that holds the element of 1-based rank rank[r]
// goes to bin[r], and rank[r] becomes the rank inside that bin.  rank, bin and wsum ([NT / 32]) are shared memory;
// every thread of the block calls this.
template <int NT, int MAXR>
__device__ void find_bins(const uint32_t* hist, int nb, uint32_t which, uint32_t* rank, uint32_t* bin, uint32_t* wsum) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = nb / NT;
  uint32_t local = 0;
  for (int b = 0; b < per; b++) local += hist[tid * per + b];
  uint32_t incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  uint32_t before = 0;
  for (int w = 0; w < warp; w++) before += wsum[w];
  const uint32_t excl = before + incl - local;
  uint32_t rr[MAXR];
#pragma unroll
  for (int r = 0; r < MAXR; r++) rr[r] = (which >> r) & 1u ? rank[r] : 0u;
  __syncthreads();
#pragma unroll
  for (int r = 0; r < MAXR; r++) {
    if (rr[r] > excl && rr[r] <= excl + local) {
      uint32_t c = excl;
      for (int b = 0; b < per; b++) {
        const uint32_t hb = hist[tid * per + b];
        if (rr[r] <= c + hb) {
          bin[r] = tid * per + b;
          rank[r] = rr[r] - c;
          break;
        }
        c += hb;
      }
    }
  }
  __syncthreads();
}

// hist[bin] += 1, one shared-memory atomic per distinct bin of the warp (the values of a row crowd into a few top-bit
// bins: plain atomics would serialise on them)
__device__ __forceinline__ void hist_add(uint32_t* hist, uint32_t bin) {
  const uint32_t peers = __match_any_sync(__activemask(), bin);
  if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], (uint32_t)__popc(peers));
}

// fn(value) for every entry of the row; four independent loads in flight per thread
template <int NT, class Fn>
__device__ __forceinline__ void for_row(const float* __restrict__ row, int S, Fn&& fn) {
  for (int i0 = threadIdx.x; i0 < S; i0 += 4 * NT) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int i = i0 + u * NT;
      v[u] = i < S ? __ldg(row + i) : 0.0f;
    }
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (i0 + u * NT < S) fn(v[u]);
  }
}

}  // namespace radix
}  // namespace bplx
