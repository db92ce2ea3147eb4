// loo.cu -- pointwise log-likelihood of observed scores over the posterior draws, and PSIS-LOO.
//
//   ll[s, m] = log Pois(yh; lh) + log Pois(ya; la) + log tau(yh, ya; lh, la, corr_coef_s)
//
// with the rates of the predict path (score_grid.cu, oracle/predict.py::expected_goals): neutral venues and
// confederations included, no clip of the rates, tau clamped at 0 (bpl/_util.py:62-68) so a match can give -inf, and no
// match weights.  exp(ll) averaged over s is what predict_score_proba returns for that match.
//
//   pointwise  K3's skeleton: the same pre-pass (score_grid_tables: e^(log-rate halves) per (sample, team)), the same
//              TMA ring of sample-row stages, one thread per match.  Per (sample, match): 2-4 LDS.64, two logf, one logf
//              of tau on the four low-score cells; -lgamma(yh+1) - lgamma(ya+1) is a per-thread constant.  The thread
//              writes its stage's samples to its row of the match-major [M, ld] matrix as 16-byte stores (full sectors,
//              no transpose) and keeps the running max, sum exp(ll - max), sum ll and sum ll^2 (float64).  Few matches:
//              the samples are split over CTAs (up to 64 splits, planned from S alone); a finalize kernel combines the
//              splits in a fixed order.
//              pointwise_kernel<true>: matches grouped by gameweek over a gameweek-major table ([G'][S] rows); each CTA
//              takes up to 256 matches of ONE gameweek (a host-built descriptor) and streams only that gameweek's rows.
//   psis       one CTA per match (row of the matrix), ArviZ's _psislw / _gpdfit:
//              (1) min ll, non-finite check and the histogram of the top 11 key bits in one pass; (2) two more radix
//              passes (11 + 10 bits) select the (Mt+1)-th smallest ll = the (Mt+1)-th largest log-ratio x = -ll;
//              (3) one pass sums the body (x <= x_cut) in float64 and gathers the tail keys into shared memory;
//              (4) bitonic sort of the tail, generalised-Pareto fit, smoothing and the two log-sum-exps in float64.
//              The row is read four times; after the first pass it is served from L2 (one row per CTA).
#include "loo.h"
#include "radix_select.cuh"

#include <float.h>
#include <math.h>

namespace bplx {

// ---- pointwise kernel ------------------------------------------------------------------------------------------------
// SEG: matches grouped by gameweek, one gameweek per CTA (its descriptor pp.seg[blockIdx.x]); the CTA streams that
// gameweek's S rows of the gameweek-major table.  Otherwise 256 consecutive matches per CTA over the S rows.
template <bool SEG>
__global__ void __launch_bounds__(kPwThreads, 3) pointwise_kernel(const __grid_constant__ PointwiseParams pp) {
  const GridParams& gp = pp.gp;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* const buf0 = reinterpret_cast<float*>(smem_raw + 128);
  const uint32_t bar0 = smem_u32(smem_raw);
  const int tid = threadIdx.x;
  const RowLayout L = row_layout(gp.T, gp.Cf, gp.ntab);
  int f_raw, f_end;
  const float* table = gp.table;
  if (SEG) {
    const int4 d = pp.seg[blockIdx.x];
    f_raw = d.y + tid;
    f_end = d.y + d.z;
    table += (size_t)d.x * gp.S * gp.row_floats;
  } else {
    f_raw = blockIdx.x * kPwThreads + tid;
    f_end = gp.F;
  }
  const bool live = f_raw < f_end;
  const int f = min(f_raw, f_end - 1);
  const int split = blockIdx.y;
  const int s_begin = split * gp.samples_per_split;
  const int s_end = min(gp.S, s_begin + gp.samples_per_split);
  const int NS = gp.ns_stage;
  const uint32_t row_bytes = (uint32_t)gp.row_floats * 4u, stage_floats = (uint32_t)NS * gp.row_floats;

  const int h = gp.home[f], a = gp.away[f];
  const bool wc = gp.model == BPLX_NEUTRAL_WC;
  const bool neutral = gp.ntab == 3 && gp.nv && gp.nv[f];
  const FixtureOffsets off = fixture_offsets(L, h, a, neutral, wc, wc ? gp.hconf[f] : 0, wc ? gp.aconf[f] : 0);
  const int offC = L.C;
  const int yh = pp.hg[f], ya = pp.ag[f];
  const float fyh = (float)yh, fya = (float)ya;
  const float cst = (float)(-lgamma(yh + 1.0) - lgamma(ya + 1.0));  // once per match, not per sample
  // tau cell: 1 = (0, 0), 2 = (0, 1), 3 = (1, 0), 4 = (1, 1), 0 = tau is 1
  const int cell = yh > 1 || ya > 1 ? 0 : 1 + 2 * yh + ya;
  float* const out = (pp.ll && live) ? pp.ll + (size_t)f * pp.ld : nullptr;

  float mx = -INFINITY;
  double se = 0.0, s1 = 0.0, s2 = 0.0;

  const int nst = (s_end - s_begin + NS - 1) / NS;
  auto issue = [&](int st) {
    const int s0 = s_begin + st * NS;
    const uint32_t bytes = (uint32_t)min(NS, s_end - s0) * row_bytes;
    const uint32_t slot = (uint32_t)st % kPwStages;
    mbar_arrive_expect_tx(bar0 + 8 * slot, bytes);
    tma_load_1d(smem_u32(buf0 + slot * stage_floats), table + (size_t)s0 * gp.row_floats, bytes, bar0 + 8 * slot);
  };
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kPwStages; s++) mbar_init(bar0 + 8 * s, 1);
    fence_mbar_init();
    fence_proxy_async();
    for (int st = 0; st < kPwStages && st < nst; st++) issue(st);
  }
  __syncthreads();

  auto loglik = [&](const float* row) -> float {
    const float2 lam = fixture_rates(row, off, neutral, wc);
    const float lh = lam.x, la = lam.y;
    float ll = fmaf(fyh, logf(lh), fmaf(fya, logf(la), cst - lh - la));
    if (cell) {
      const float c = row[offC];
      const float t = cell == 1 ? 1.0f - (c * lh) * la : cell == 2 ? fmaf(c, lh, 1.0f) : cell == 3 ? fmaf(c, la, 1.0f) : 1.0f - c;
      ll += logf(fmaxf(t, 0.0f));
    }
    return ll;
  };
  // running max / sum exp(ll - max) / sum ll / sum ll^2.  exp(ll - max) in float with the rounding error of ll - max
  // carried (two-sum), accumulated in float64; a NaN propagates, -inf adds nothing
  auto update = [&](float x) {
    s1 += (double)x;
    s2 = fma((double)x, (double)x, s2);
    if (x > mx) {
      se = se * exp((double)mx - (double)x) + 1.0;
      mx = x;
    } else if (x != -INFINITY) {
      const float d = x - mx, bb = d - x, err = (x - (d - bb)) + (-mx - bb);
      const float e = expf(d);
      se += (double)fmaf(e, err, e);
    }
  };

  for (int st = 0; st < nst; st++) {
    const float* cur = buf0 + (st % kPwStages) * stage_floats;
    mbar_wait(bar0 + 8 * (st % kPwStages), (st / kPwStages) & 1);
    const int s0 = s_begin + st * NS;
    const int ns = min(NS, s_end - s0);
#pragma unroll 1
    for (int j0 = 0; j0 < ns; j0 += 4) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        v[u] = 0.0f;
        if (j0 + u < ns) {
          v[u] = loglik(cur + (j0 + u) * gp.row_floats);
          update(v[u]);
        }
      }
      if (out) {
        if (pp.vec && j0 + 4 <= ns) {
          __stcs(reinterpret_cast<float4*>(out + s0 + j0), make_float4(v[0], v[1], v[2], v[3]));
        } else {
#pragma unroll
          for (int u = 0; u < 4; u++)
            if (j0 + u < ns) __stcs(out + s0 + j0 + u, v[u]);
        }
      }
    }
    __syncthreads();  // every thread is done with this buffer: refill it
    if (tid == 0 && st + kPwStages < nst) issue(st + kPwStages);
  }
  if (live) {
    double* p = pp.partial + ((size_t)split * gp.F + f) * 4;
    p[0] = (double)mx;
    p[1] = se;
    p[2] = s1;
    p[3] = s2;
  }
}

// combines the sample splits in split order (deterministic): stats[m] = (max ll, sum exp(ll - max), sum ll, sum ll^2)
__global__ void pointwise_finalize(const __grid_constant__ PointwiseParams pp) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  const int M = pp.gp.F;
  if (m >= M) return;
  double mx = -INFINITY;
  for (int k = 0; k < pp.gp.nsplit; k++) mx = fmax(mx, pp.partial[((size_t)k * M + m) * 4]);
  double se = 0.0, s1 = 0.0, s2 = 0.0;
  for (int k = 0; k < pp.gp.nsplit; k++) {
    const double* p = pp.partial + ((size_t)k * M + m) * 4;
    if (p[0] != -INFINITY || isnan(p[1])) se += p[1] * exp(p[0] - mx);
    s1 += p[2];
    s2 += p[3];
  }
  double* o = pp.stats + (size_t)m * 4;
  o[0] = mx;
  o[1] = se;
  o[2] = s1;
  o[3] = s2;
}

size_t pointwise_plan(PointwiseParams* pp, const char** err) {
  GridParams* gp = &pp->gp;
  const size_t table_bytes = table_layout(gp);
  const size_t row_bytes = (size_t)gp->row_floats * 4;
  if (row_bytes > (size_t)kPwStageBytes) {
    if (err) *err = "pointwise log-likelihood: a sample row (teams x tables) does not fit one stage buffer: too many teams";
    return 0;
  }
  int ns = (int)((size_t)kPwStageBytes / row_bytes);
  ns = ns > kGridStageMax ? kGridStageMax : ns;
  gp->ns_stage = ns >= 4 ? ns / 4 * 4 : ns;  // a multiple of 4: every stage starts on a 16-byte boundary of a matrix row
  // The sample splits depend on S and the row layout only, never on M: the statistics of a match are then the same
  // bits whichever other matches share the call (callers may cut the matches into ranges).  Up to 64 splits of at
  // least four stages each: enough CTAs for a 380-match season, and 64 x M x 32 bytes of partial sums at most.
  int best = gp->S / (4 * gp->ns_stage);
  best = best < 1 ? 1 : (best > 64 ? 64 : best);
  int sps = (gp->S + best - 1) / best;
  sps = (sps + gp->ns_stage - 1) / gp->ns_stage * gp->ns_stage;
  gp->nsplit = (gp->S + sps - 1) / sps;
  gp->samples_per_split = sps;
  return table_bytes + (size_t)gp->nsplit * gp->F * 4 * sizeof(double);
}

int launch_pointwise(PointwiseParams& pp, cudaStream_t stream) {
  GridParams& gp = pp.gp;
  pp.vec = pp.ll && pp.ld % 4 == 0 && gp.ns_stage % 4 == 0 && (reinterpret_cast<uintptr_t>(pp.ll) & 15u) == 0;
  int rc = launch_score_grid_tables(gp, stream);
  if (rc != BPLX_OK) return rc;
  const size_t smem = 128 + (size_t)kPwStages * gp.ns_stage * gp.row_floats * 4;
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    BPLX_CUDA(cudaFuncSetAttribute(pointwise_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  dim3 grid((gp.F + kPwThreads - 1) / kPwThreads, gp.nsplit);
  pointwise_kernel<false><<<grid, kPwThreads, smem, stream>>>(pp);
  BPLX_CUDA(cudaGetLastError());
  pointwise_finalize<<<(gp.F + 255) / 256, 256, 0, stream>>>(pp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(2);
  return BPLX_OK;
}

int launch_pointwise_segmented(PointwiseParams& pp, int ngw, cudaStream_t stream) {
  GridParams& gp = pp.gp;
  pp.vec = pp.ll && pp.ld % 4 == 0 && gp.ns_stage % 4 == 0 && (reinterpret_cast<uintptr_t>(pp.ll) & 15u) == 0;
  GridParams all = gp;  // the pre-pass builds every gameweek's rows in one launch: (gameweek, draw) is a pseudo-draw
  all.S = ngw * gp.S;
  int rc = launch_score_grid_tables(all, stream);
  if (rc != BPLX_OK) return rc;
  const size_t smem = 128 + (size_t)kPwStages * gp.ns_stage * gp.row_floats * 4;
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    BPLX_CUDA(cudaFuncSetAttribute(pointwise_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  dim3 grid(pp.nseg, gp.nsplit);
  pointwise_kernel<true><<<grid, kPwThreads, smem, stream>>>(pp);
  BPLX_CUDA(cudaGetLastError());
  pointwise_finalize<<<(gp.F + 255) / 256, 256, 0, stream>>>(pp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(2);
  return BPLX_OK;
}

// ---- PSIS kernel -----------------------------------------------------------------------------------------------------
namespace {

using radix::f2key;
using radix::hist_add;
using radix::key2f;
using radix::kBins;
constexpr int kPsisWarps = kPsisThreads / 32;
constexpr int kMaxCand = 32 + 30 + 128;  // GPD candidates: 30 + floor(sqrt(n)), n <= kPsisTailMax
constexpr double kLogTiny = -708.3964185322641;  // log(DBL_MIN), ArviZ's cutoffmin

struct PsisShared {
  double red[kPsisWarps + 1];
  double b[kMaxCand], k[kMaxCand], L[kMaxCand], w[kMaxCand];
  double bhat;
  float wmin[kPsisWarps];
  uint32_t wsum[kPsisWarps];
  uint32_t bin, rank, cnt;
};

// fixed-order block sum (deterministic)
__device__ double block_sum(double v, PsisShared& sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) sh.red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = lane < kPsisWarps ? sh.red[lane] : 0.0;
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sh.red[kPsisWarps] = v;
  }
  __syncthreads();
  const double r = sh.red[kPsisWarps];
  __syncthreads();
  return r;
}

}  // namespace

__global__ void __launch_bounds__(kPsisThreads) psis_kernel(const __grid_constant__ PsisParams pp) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  double* const zs = reinterpret_cast<double*>(smem_dyn);  // [cap]  sorted exp(x_tail) - exp(x_cut)
  uint32_t* const hist = reinterpret_cast<uint32_t*>(zs + pp.cap);  // [kBins]
  uint32_t* const keys = hist + kBins;  // [cap]  tail keys
  __shared__ PsisShared sh;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int m = blockIdx.x, S = pp.S;
  const float* row = pp.ll + (size_t)m * pp.ld;

  for (int i = tid; i < kBins; i += kPsisThreads) hist[i] = 0;
  if (tid == 0) sh.cnt = 0;
  __syncthreads();

  // (1) min ll (= -max x), non-finite entries, histogram of the top 11 key bits
  float mn = INFINITY;
  int bad = 0;
  radix::for_row<kPsisThreads>(row, S, [&](float v) {
    bad |= !isfinite(v);
    mn = fminf(mn, v);
    hist_add(hist, f2key(v) >> 21);
  });
#pragma unroll
  for (int o = 16; o; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
  if (lane == 0) sh.wmin[warp] = mn;
  if (__syncthreads_or(bad)) {
    if (tid == 0) {
      pp.elpd[m] = __longlong_as_double(0x7ff8000000000000ll);
      pp.khat[m] = INFINITY;
    }
    return;
  }
  mn = sh.wmin[0];
  for (int w = 1; w < kPsisWarps; w++) mn = fminf(mn, sh.wmin[w]);
  const double xmax = -(double)mn;

  // (2) x_(Mt+1), the (Mt+1)-th largest x = the (Mt+1)-th smallest ll: radix select on the keys
  double x_cut = kLogTiny;
  if (pp.Mt + 1 <= S) {
    if (tid == 0) sh.rank = (uint32_t)pp.Mt + 1;
    __syncthreads();
    radix::find_bins<kPsisThreads, 1>(hist, kBins, 1u, &sh.rank, &sh.bin, sh.wsum);
    uint32_t prefix = sh.bin << 21;
    for (int i = tid; i < kBins; i += kPsisThreads) hist[i] = 0;
    __syncthreads();
    radix::for_row<kPsisThreads>(row, S, [&](float v) {
      const uint32_t k = f2key(v);
      if ((k >> 21) == (prefix >> 21)) hist_add(hist, (k >> 10) & 2047u);
    });
    __syncthreads();
    radix::find_bins<kPsisThreads, 1>(hist, kBins, 1u, &sh.rank, &sh.bin, sh.wsum);
    prefix |= sh.bin << 10;
    for (int i = tid; i < kBins; i += kPsisThreads) hist[i] = 0;
    __syncthreads();
    radix::for_row<kPsisThreads>(row, S, [&](float v) {
      const uint32_t k = f2key(v);
      if ((k >> 10) == (prefix >> 10)) hist_add(hist, k & 1023u);
    });
    __syncthreads();
    radix::find_bins<kPsisThreads, 1>(hist, 1024, 1u, &sh.rank, &sh.bin, sh.wsum);
    prefix |= sh.bin;
    x_cut = fmax(-(double)key2f(prefix) - xmax, kLogTiny);
  }
  const double exp_cut = exp(x_cut);

  // (3) body sums (x <= x_cut) and the tail gather.  For the body, lw + ll = x + ll is -xmax up to rounding: the sum of
  // exp(x + ll + xmax) takes 1 + d + d^2/2 for the tiny d instead of a float64 exp
  double b1 = 0.0, b2 = 0.0;
  radix::for_row<kPsisThreads>(row, S, [&](float v) {
    const double x = -(double)v - xmax;
    if (x > x_cut) {
      const uint32_t pos = atomicAdd(&sh.cnt, 1u);
      if (pos < (uint32_t)pp.cap) keys[pos] = f2key(v);
    } else {
      b1 += exp(x);
      const double d = (x + (double)v) + xmax;
      b2 += fabs(d) < 1e-5 ? 1.0 + d * (1.0 + 0.5 * d) : exp(d);
    }
  });
  b1 = block_sum(b1, sh);
  b2 = block_sum(b2, sh);
  const int n = (int)min(sh.cnt, (uint32_t)pp.cap);

  // (4) sort the tail by ascending x (descending key; tied values are equal, so their order does not matter)
  int P = 1;
  while (P < n) P <<= 1;
  for (int i = n + tid; i < P; i += kPsisThreads) keys[i] = 0u;
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < P; i += kPsisThreads) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const uint32_t a = keys[i], b = keys[ixj];
          if ((i & k) == 0 ? a < b : a > b) {
            keys[i] = b;
            keys[ixj] = a;
          }
        }
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < n; i += kPsisThreads) zs[i] = exp(-(double)key2f(keys[i]) - xmax) - exp_cut;
  __syncthreads();

  // generalised Pareto fit (Zhang & Stephens 2009 with ArviZ's weak prior on k)
  double khat = INFINITY, sigma = 0.0;
  if (n > 4) {
    const int mc = 30 + (int)sqrt((double)n);
    const double q3 = 3.0 * zs[(int)(n / 4.0 + 0.5) - 1];
    const double binv = 1.0 / zs[n - 1];
    for (int j = tid; j < mc; j += kPsisThreads) sh.b[j] = (1.0 - sqrt((double)mc / ((j + 1) - 0.5))) / q3 + binv;
    __syncthreads();
    for (int j = warp; j < mc; j += kPsisWarps) {
      const double bj = sh.b[j];
      double acc = 0.0;
      for (int i = lane; i < n; i += 32) acc += log1p(-bj * zs[i]);
#pragma unroll
      for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) sh.k[j] = acc / n;
    }
    __syncthreads();
    for (int j = tid; j < mc; j += kPsisThreads) sh.L[j] = n * (log(-(sh.b[j] / sh.k[j])) - sh.k[j] - 1.0);
    __syncthreads();
    for (int j = tid; j < mc; j += kPsisThreads) {
      double s = 0.0;
      for (int i = 0; i < mc; i++) s += exp(sh.L[i] - sh.L[j]);
      sh.w[j] = 1.0 / s;
    }
    __syncthreads();
    if (tid == 0) {  // drop negligible weights, normalise, posterior mean of b
      double ws = 0.0, bh = 0.0;
      for (int j = 0; j < mc; j++)
        if (sh.w[j] >= 10.0 * DBL_EPSILON) ws += sh.w[j];
      for (int j = 0; j < mc; j++)
        if (sh.w[j] >= 10.0 * DBL_EPSILON) bh += sh.b[j] * (sh.w[j] / ws);
      sh.bhat = bh;
    }
    __syncthreads();
    const double bh = sh.bhat;
    double kk = 0.0;
    for (int i = tid; i < n; i += kPsisThreads) kk += log1p(-bh * zs[i]);
    kk = block_sum(kk, sh) / n;
    sigma = -kk / bh;
    khat = (n * kk + 10.0 * 0.5) / (n + 10.0);
  }
  // smoothing: the i-th smallest tail value becomes log(GPD quantile at (i + 0.5) / n + exp(x_cut)), truncated at 0
  const bool smooth = n > 4 && isfinite(khat);
  double t1 = 0.0, t2 = 0.0;
  for (int i = tid; i < n; i += kPsisThreads) {
    const double llv = (double)key2f(keys[i]);
    double v = -llv - xmax;
    if (smooth) {
      const double p = (i + 0.5) / n;
      double g = fabs(khat) < DBL_EPSILON ? -log1p(-p) : expm1(-khat * log1p(-p)) / khat;
      g = sigma > 0.0 ? g * sigma : __longlong_as_double(0x7ff8000000000000ll);
      v = log(g + exp_cut);
      if (v > 0.0) v = 0.0;
    }
    t1 += exp(v);
    t2 += exp(v + llv + xmax);
  }
  t1 = block_sum(t1, sh);
  t2 = block_sum(t2, sh);
  if (tid == 0) {
    // lw = x' - log(sum exp x');  elpd_loo_m = log sum exp(lw + ll) = log sum exp(x' + ll + xmax) - xmax - log sum exp x'
    pp.elpd[m] = log(b2 + t2) - xmax - log(b1 + t1);
    pp.khat[m] = khat;
  }
}

int psis_tail_length(int S, double r_eff) {
  const double t = fmin(0.2 * S, 3.0 * sqrt(S / r_eff));
  return (int)ceil(t);
}

int launch_psis(const PsisParams& pp, cudaStream_t stream) {
  const size_t smem = (size_t)pp.cap * (sizeof(double) + sizeof(uint32_t)) + kBins * sizeof(uint32_t);
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    BPLX_CUDA(cudaFuncSetAttribute(psis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  psis_kernel<<<pp.M, kPsisThreads, smem, stream>>>(pp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
