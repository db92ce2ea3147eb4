// sample_score.cuh -- the per-draw score sampler (DESIGN §3c) shared by the simulation kernels (simulate.cu) and the
// posterior predictive kernel (ppc.cu), with the Philox block of a fixed word address and the 1/k constant it reads.
// Each translation unit that includes this header has its own copy of c_sim_inv_k and uploads it once with
// upload_sim_constants() before its first launch.
#pragma once
#include <curand_kernel.h>
#include <float.h>

#include "common.cuh"

namespace bplx {

namespace {

__constant__ float c_sim_inv_k[64];  // 1 / k (k >= 1)

// one fixture of one simulation; false when the rates or the normaliser are unusable
__device__ __forceinline__ bool sample_score(float lh, float la, float c, float uh, float ua, int G, int& hg, int& ag) {
  if (!(isfinite(lh) && isfinite(la))) return false;
  const float t00 = fmaxf(1.0f - (c * lh) * la, 0.0f), t01 = fmaxf(fmaf(c, lh, 1.0f), 0.0f);
  const float t10 = fmaxf(fmaf(c, la, 1.0f), 0.0f), t11 = fmaxf(1.0f - c, 0.0f);
  // un-normalised pmfs p_i = lh^i / i!, q_j = la^j / j!: P2 = sum_{i >= 2} p_i, Q2 = sum_{j >= 2} q_j
  float p = lh, q = la, P2 = 0.0f, Q2 = 0.0f;
  for (int k = 2; k <= G; k++) {
    p *= lh * c_sim_inv_k[k];
    q *= la * c_sim_inv_k[k];
    P2 += p;
    Q2 += q;
  }
  const float Q = 1.0f + la + Q2;          // row mass / p_i for i >= 2
  const float r0 = t00 + t01 * la + Q2;    // row mass of i = 0 (p_0 = 1)
  const float r1 = t10 + t11 * la + Q2;    // row mass / p_1 of i = 1
  const float Z = r0 + lh * r1 + P2 * Q;
  if (!(Z > 0.0f && Z <= FLT_MAX)) return false;
  // home goals: the smallest i whose cumulative row mass reaches u_h Z
  float target = uh * Z, cum = r0;
  int i = -1, last = -1;
  if (r0 > 0.0f) {
    last = 0;
    if (cum >= target) i = 0;
  }
  if (i < 0) {
    const float m1 = lh * r1;
    cum += m1;
    if (m1 > 0.0f) {
      last = 1;
      if (cum >= target) i = 1;
    }
  }
  if (i < 0) {
    float pk = lh;
    for (int k = 2; k <= G; k++) {
      pk *= lh * c_sim_inv_k[k];
      const float m = pk * Q;
      cum += m;
      if (m > 0.0f) {
        last = k;
        if (cum >= target) {
          i = k;
          break;
        }
      }
    }
  }
  if (i < 0) i = last;
  // away goals within row i: the smallest j whose cumulative weight reaches u_a m(i) (p_i cancels)
  const float w0 = i == 0 ? t00 : i == 1 ? t10 : 1.0f;
  const float w1 = (i == 0 ? t01 : i == 1 ? t11 : 1.0f) * la;
  const float mrow = i == 0 ? r0 : i == 1 ? r1 : Q;
  target = ua * mrow;
  cum = w0;
  int j = -1;
  last = -1;
  if (w0 > 0.0f) {
    last = 0;
    if (cum >= target) j = 0;
  }
  if (j < 0) {
    cum += w1;
    if (w1 > 0.0f) {
      last = 1;
      if (cum >= target) j = 1;
    }
  }
  if (j < 0) {
    float qk = la;
    for (int k = 2; k <= G; k++) {
      qk *= la * c_sim_inv_k[k];
      cum += qk;
      if (qk > 0.0f) {
        last = k;
        if (cum >= target) {
          j = k;
          break;
        }
      }
    }
  }
  if (j < 0) j = last;
  hg = i;
  ag = j;
  return true;
}

// words 4b .. 4b + 3 of the Philox sequence of simulation n (curand_init(seed, n, 0) followed by curand()) without a
// state: one Philox4x32_10 block
__device__ __forceinline__ uint4 philox_block(unsigned long long seed, unsigned long long n, unsigned b) {
  return curand_Philox4x32_10(make_uint4(b, 0u, (unsigned)n, (unsigned)(n >> 32)),
                              make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
}

// c_sim_inv_k of this translation unit, uploaded once
int upload_sim_constants() {
  static bool done = false;
  if (done) return BPLX_OK;
  float inv[64];
  for (int k = 0; k < 64; k++) inv[k] = k ? (float)(1.0 / k) : 0.0f;
  BPLX_CUDA(cudaMemcpyToSymbol(c_sim_inv_k, inv, sizeof inv));
  done = true;
  return BPLX_OK;
}

}  // namespace

}  // namespace bplx
