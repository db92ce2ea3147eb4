// dynamic_predict.cu -- the dynamic model's gameweeks after the fit, drawn from its own generative process.
//
// Definition (the same text in include/bplx.h, oracle/dynamic_predict.py, DESIGN §3h and the docstrings):
//   for each draw s and each gameweek j = G .. G + h - 1 in order, fresh sites from their priors
//   (the dynamic model's, as its fit samples them): mean_home_attack, mean_home_defence ~ N(0.1, 0.2); mean_away_attack,
//   mean_away_defence ~ N(-0.1, 0.2); the six std_* ~ HalfNormal(1); per team u ~ Beta(2, 4), rho = 2u - 1,
//   za ~ N(0, 1), zd = rho za + sqrt(1 - rho^2) eps with eps ~ N(0, 1), and the four *_decentered ~ N(0, 1).  Then
//   attack[j] = attack[j - 1] + za std_attack[j] (defence likewise with zd) and effect[j] = mean[j] + std[j] dec[j] (not
//   cumulative).
//
// Random numbers: Philox4_32_10 under the key seed ^ BPLX_FORECAST_KEY, subsequence first_draw + s; counter block b
// holds words 4b .. 4b + 3.  Gameweek k = j - G uses blocks k (3 + 3T) + 0 .. 2 for the draw and k (3 + 3T) + 3 + 3t +
// 0 .. 2 for team t (word map in include/bplx.h).  Every variate has a fixed address: the forecast does not depend on
// the launch geometry or on how the draws are cut into ranges.
//
// Kernel: one thread per (draw, team), whole draws per CTA, the gameweeks walked in order with attack / defence in
// registers.  Per gameweek the thread of team 0 draws the draw's ten scalars into shared memory (drawn once, read by
// every team of the draw).  Beta(2, 4) is the 2nd smallest of 5 uniforms: exact, no rejection loop.
#include "dynamic_predict.h"

#include <curand_kernel.h>

namespace bplx {

namespace {

__device__ __forceinline__ uint4 forecast_block(unsigned long long key, unsigned long long n, unsigned b) {
  return curand_Philox4x32_10(make_uint4(b, 0u, (unsigned)n, (unsigned)(n >> 32)),
                              make_uint2((unsigned)key, (unsigned)(key >> 32)));
}

__global__ void __launch_bounds__(kForecastThreads) dynamic_forecast_kernel(const __grid_constant__ ForecastParams fp) {
  // per draw of the CTA: mean_ha, mean_aa, mean_hd, mean_ad, std_ha, std_aa, std_hd, std_ad, std_attack, std_defence
  __shared__ float s_hyper[kForecastThreads][10];
  const int T = fp.T;
  const int ld = threadIdx.x / T, t = threadIdx.x - ld * T;
  const int s = blockIdx.x * fp.draws_per_cta + ld;
  const bool live = ld < fp.draws_per_cta && s < fp.S;
  const unsigned long long n = (unsigned long long)(fp.first_draw + s);
  const unsigned per_gw = 3u + 3u * (unsigned)T;
  float att = 0.0f, def = 0.0f;
  if (live) {
    att = fp.attack[(size_t)s * T + t];
    def = fp.defence[(size_t)s * T + t];
  }
  for (int k = 0; k < fp.h; k++) {
    const unsigned b0 = (unsigned)k * per_gw;
    if (live && t == 0) {
      float* hp = s_hyper[ld];
      const uint4 w0 = forecast_block(fp.key, n, b0), w1 = forecast_block(fp.key, n, b0 + 1),
                  w2 = forecast_block(fp.key, n, b0 + 2);
      float2 z = _curand_box_muller(w0.x, w0.y);
      hp[0] = fmaf(0.2f, z.x, 0.1f);   // mean_home_attack
      hp[1] = fmaf(0.2f, z.y, -0.1f);  // mean_away_attack
      z = _curand_box_muller(w0.z, w0.w);
      hp[2] = fmaf(0.2f, z.x, 0.1f);   // mean_home_defence
      hp[3] = fmaf(0.2f, z.y, -0.1f);  // mean_away_defence
      z = _curand_box_muller(w1.x, w1.y);
      hp[4] = fabsf(z.x);  // std_home_attack
      hp[5] = fabsf(z.y);  // std_away_attack
      z = _curand_box_muller(w1.z, w1.w);
      hp[6] = fabsf(z.x);  // std_home_defence
      hp[7] = fabsf(z.y);  // std_away_defence
      z = _curand_box_muller(w2.x, w2.y);
      hp[8] = fabsf(z.x);  // std_attack
      hp[9] = fabsf(z.y);  // std_defence
    }
    __syncthreads();
    if (live) {
      const float* hp = s_hyper[ld];
      const unsigned bt = b0 + 3u + 3u * (unsigned)t;
      const uint4 w0 = forecast_block(fp.key, n, bt), w1 = forecast_block(fp.key, n, bt + 1),
                  w2 = forecast_block(fp.key, n, bt + 2);
      // u ~ Beta(2, 4): the 2nd smallest of the 5 uniforms of words 0 .. 4
      float lo = _curand_uniform(w0.x), u2 = 2.0f;
      const float rest[4] = {_curand_uniform(w0.y), _curand_uniform(w0.z), _curand_uniform(w0.w), _curand_uniform(w1.x)};
#pragma unroll
      for (int i = 0; i < 4; i++) {
        u2 = fminf(u2, fmaxf(lo, rest[i]));
        lo = fminf(lo, rest[i]);
      }
      const float rho = 2.0f * u2 - 1.0f;
      const float2 ze = _curand_box_muller(w1.z, w1.w);  // (za, eps); word 5 is unused
      const float zd = fmaf(rho, ze.x, sqrtf(1.0f - rho * rho) * ze.y);
      att = fmaf(ze.x, hp[8], att);
      def = fmaf(zd, hp[9], def);
      const float2 da = _curand_box_muller(w2.x, w2.y), dd = _curand_box_muller(w2.z, w2.w);
      const size_t o = ((size_t)k * fp.S + s) * T + t;
      fp.out[0][o] = att;
      fp.out[1][o] = def;
      fp.out[2][o] = fmaf(hp[4], da.x, hp[0]);  // home_attack
      fp.out[3][o] = fmaf(hp[5], da.y, hp[1]);  // away_attack
      fp.out[4][o] = fmaf(hp[6], dd.x, hp[2]);  // home_defence
      fp.out[5][o] = fmaf(hp[7], dd.y, hp[3]);  // away_defence
    }
    __syncthreads();  // s_hyper is rewritten for the next gameweek
  }
}

}  // namespace

int launch_dynamic_forecast(ForecastParams& fp, cudaStream_t stream) {
  fp.draws_per_cta = kForecastThreads / fp.T;
  const int threads = fp.draws_per_cta * fp.T;
  const unsigned ctas = (unsigned)((fp.S + fp.draws_per_cta - 1) / fp.draws_per_cta);
  dynamic_forecast_kernel<<<ctas, threads, 0, stream>>>(fp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
