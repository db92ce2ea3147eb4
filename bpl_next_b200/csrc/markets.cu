// markets.cu -- forecast uncertainty: per-draw market probabilities (outcome, both teams to score, total-goals and
// goal-margin lines, the rates) and exact posterior quantiles of any row-major float matrix.
//
//   draws      pointwise_kernel's skeleton (loo.cu): score_grid_tables tabulates e^(log-rate halves) per (draw, team), a
//              ring of TMA stages of draw rows feeds one thread per fixture, and the draws are cut into splits planned
//              from S alone, combined by market_finalize in split order.  A CTA computes kMdChunk of the K rows.  The
//              grid is never formed: P_s(i, j) = p_i q_j off the four low cells, so every row is a sum over i of p_i
//              times a prefix or suffix sum of q (or q_i itself for the draw row), plus p_i q_j (tau - 1) on the low
//              cells it covers: O(G) per row and draw.  The per-thread prefix / suffix sums live in shared memory,
//              [k][thread], read at a warp-uniform k (the lines are the same for every fixture).  pmfs by the
//              normalised recurrence p_k = p_{k-1} lambda / k: nothing overflows for max_goals <= 63.  Each thread
//              writes its stage's draws to its rows of the [F K, ld] matrix as 16-byte streaming stores and keeps
//              float64 sums of p - p0 and (p - p0)^2 per row, p0 the split's first value (a row that barely varies
//              keeps its sd); market_finalize merges the splits' counts, means and squared deviations.
//   quantiles  one CTA per row, psis_kernel's radix select (radix_select.cuh) for up to 16 ranks at once: a histogram
//              of the top 11 key bits (and the odds exceedances) in pass 1; pass 2 histograms the next 11 bits of the
//              values in each distinct selected top bin (a byte table maps a top bin to its histogram); pass 3 the last
//              10 bits of each distinct 22-bit prefix.  The row is read three times for any number of levels.
#include "markets.h"
#include "radix_select.cuh"

#include <math.h>

namespace bplx {

namespace {

__constant__ float c_md_inv_k[64];  // 1 / k (k >= 1)

int upload_market_constants() {
  static bool done = false;
  if (done) return BPLX_OK;
  float inv[64];
  for (int k = 0; k < 64; k++) inv[k] = k ? (float)(1.0 / k) : 0.0f;
  BPLX_CUDA(cudaMemcpyToSymbol(c_md_inv_k, inv, sizeof inv));
  done = true;
  return BPLX_OK;
}

// bytes of the per-thread prefix / suffix sums: two arrays of G + 3 floats (k = -1 .. G + 1) per thread
size_t sums_bytes(int g) { return (size_t)2 * (g + 2) * kMdThreads * sizeof(float); }

}  // namespace

// ---- draws kernel ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMdThreads, 2) market_draws_kernel(const __grid_constant__ MarketParams mp) {
  const GridParams& gp = mp.gp;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* const buf0 = reinterpret_cast<float*>(smem_raw + 128);
  const uint32_t bar0 = smem_u32(smem_raw);
  const int tid = threadIdx.x;
  const RowLayout L = row_layout(gp.T, gp.Cf, gp.ntab);
  const int f_raw = blockIdx.x * kMdThreads + tid;
  const bool live = f_raw < gp.F;
  const int f = min(f_raw, gp.F - 1);
  const int r0 = blockIdx.y * kMdChunk;
  const int nr = min(kMdChunk, mp.K - r0);
  const int split = blockIdx.z;
  const int s_begin = split * gp.samples_per_split;
  const int s_end = min(gp.S, s_begin + gp.samples_per_split);
  const int NS = gp.ns_stage;
  const int G = gp.g - 1;
  const uint32_t row_bytes = (uint32_t)gp.row_floats * 4u, stage_floats = (uint32_t)NS * gp.row_floats;
  // this thread's prefix sums Xc[k] = sum_{j <= k} q_j and suffix sums Xs[k] = sum_{j >= k} q_j at [(k + 1) * kMdThreads]
  // for k = -1 .. G + 1 (Xc: 0 below, the total above; Xs: the total below, 0 above)
  float* const Xc = buf0 + kMdStages * stage_floats + tid;
  float* const Xs = Xc + (G + 3) * kMdThreads;

  const int h = gp.home[f], a = gp.away[f];
  const bool wc = gp.model == BPLX_NEUTRAL_WC;
  const bool neutral = gp.ntab == 3 && gp.nv && gp.nv[f];
  const FixtureOffsets off = fixture_offsets(L, h, a, neutral, wc, wc ? gp.hconf[f] : 0, wc ? gp.aconf[f] : 0);
  const int offC = L.C;
  float* const out = (mp.draws && live) ? mp.draws + ((size_t)f * mp.K + r0) * mp.ld : nullptr;

  // per row: sum (p - p0) and sum (p - p0)^2 with p0 the split's first value, so that rows that barely vary keep their sd
  double s1[kMdChunk], s2[kMdChunk];
  float shift[kMdChunk];
#pragma unroll
  for (int r = 0; r < kMdChunk; r++) s1[r] = s2[r] = 0.0, shift[r] = 0.0f;
  int bad = 0;

  const int nst = (s_end - s_begin + NS - 1) / NS;
  auto issue = [&](int st) {
    const int s0 = s_begin + st * NS;
    const uint32_t bytes = (uint32_t)min(NS, s_end - s0) * row_bytes;
    const uint32_t slot = (uint32_t)st % kMdStages;
    mbar_arrive_expect_tx(bar0 + 8 * slot, bytes);
    tma_load_1d(smem_u32(buf0 + slot * stage_floats), gp.table + (size_t)s0 * gp.row_floats, bytes, bar0 + 8 * slot);
  };
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kMdStages; s++) mbar_init(bar0 + 8 * s, 1);
    fence_mbar_init();
    fence_proxy_async();
    for (int st = 0; st < kMdStages && st < nst; st++) issue(st);
  }
  __syncthreads();

  // the chunk's rows of one draw
  auto market = [&](const float* row, float (&v)[kMdChunk]) {
    const float2 lam = fixture_rates(row, off, neutral, wc);
    const float lh = lam.x, la = lam.y;
    const bool ok = isfinite(lh) && isfinite(la);
    bad += !ok;
    const float c = row[offC];
    const float p0 = expf(-lh), q0 = expf(-la);
    float q = q0, sc = 0.0f;
    Xc[0] = 0.0f;
    for (int k = 0; k <= G; k++) {
      if (k) q *= la * c_md_inv_k[k];
      sc += q;
      Xc[(k + 1) * kMdThreads] = sc;
      Xs[(k + 1) * kMdThreads] = q;
    }
    Xc[(G + 2) * kMdThreads] = sc;
    Xs[(G + 2) * kMdThreads] = 0.0f;
    float ss = 0.0f;
    for (int k = G; k >= 0; k--) {
      ss += Xs[(k + 1) * kMdThreads];
      Xs[(k + 1) * kMdThreads] = ss;
    }
    Xs[0] = ss;
    float acc[kMdChunk];
#pragma unroll
    for (int r = 0; r < kMdChunk; r++) acc[r] = 0.0f;
    float p = p0, qd = q0;
    for (int i = 0; i <= G; i++) {
      if (i) {
        p *= lh * c_md_inv_k[i];
        qd *= la * c_md_inv_k[i];
      }
#pragma unroll
      for (int r = 0; r < kMdChunk; r++) {
        if (r >= nr) break;
        const MarketRow d = mp.row[r0 + r];
        if (d.kind <= kRowSuffix) {
          if (i >= d.i0) {
            const int k = min(max(d.a + d.b * i, -1), G + 1);
            acc[r] = fmaf(p, (d.kind == kRowSuffix ? Xs : Xc)[(k + 1) * kMdThreads], acc[r]);
          }
        } else if (d.kind == kRowDiagonal) {
          acc[r] = fmaf(p, qd, acc[r]);
        }
      }
    }
    // tau on the four low-score cells, clamped at 0: the cell (i, j) adds p_i q_j (tau - 1) to the rows that cover it
    const float p1 = p0 * lh, q1 = q0 * la;
    const float d00 = (p0 * q0) * (fmaxf(1.0f - (c * lh) * la, 0.0f) - 1.0f);
    const float d01 = (p0 * q1) * (fmaxf(fmaf(c, lh, 1.0f), 0.0f) - 1.0f);
    const float d10 = (p1 * q0) * (fmaxf(fmaf(c, la, 1.0f), 0.0f) - 1.0f);
    const float d11 = (p1 * q1) * (fmaxf(1.0f - c, 0.0f) - 1.0f);
#pragma unroll
    for (int r = 0; r < kMdChunk; r++) {
      if (r >= nr) break;
      const MarketRow d = mp.row[r0 + r];
      float x = acc[r];
      if (d.corr & 1u) x += d00;
      if (d.corr & 2u) x += d01;
      if (d.corr & 4u) x += d10;
      if (d.corr & 8u) x += d11;
      if (!ok) x = __int_as_float(0x7fc00000);
      v[r] = d.kind == kRowHomeRate ? lh : d.kind == kRowAwayRate ? la : x;
    }
  };

  for (int st = 0; st < nst; st++) {
    const float* cur = buf0 + (st % kMdStages) * stage_floats;
    mbar_wait(bar0 + 8 * (st % kMdStages), (st / kMdStages) & 1);
    const int s0 = s_begin + st * NS;
    const int ns = min(NS, s_end - s0);
#pragma unroll 1
    for (int j0 = 0; j0 < ns; j0 += 4) {
      float v[4][kMdChunk];
#pragma unroll
      for (int u = 0; u < 4; u++) {
#pragma unroll
        for (int r = 0; r < kMdChunk; r++) v[u][r] = 0.0f;
        if (j0 + u < ns) {
          market(cur + (j0 + u) * gp.row_floats, v[u]);
          const bool first = st == 0 && j0 + u == 0;
#pragma unroll
          for (int r = 0; r < kMdChunk; r++) {
            if (first) shift[r] = v[u][r];
            const double d = (double)v[u][r] - (double)shift[r];
            s1[r] += d;
            s2[r] = fma(d, d, s2[r]);
          }
        }
      }
      if (out) {
#pragma unroll
        for (int r = 0; r < kMdChunk; r++) {
          if (r >= nr) break;
          float* o = out + (size_t)r * mp.ld + s0 + j0;
          if (mp.vec && j0 + 4 <= ns) {
            __stcs(reinterpret_cast<float4*>(o), make_float4(v[0][r], v[1][r], v[2][r], v[3][r]));
          } else {
#pragma unroll
            for (int u = 0; u < 4; u++)
              if (j0 + u < ns) __stcs(o + u, v[u][r]);
          }
        }
      }
    }
    __syncthreads();  // every thread is done with this buffer: refill it
    if (tid == 0 && st + kMdStages < nst) issue(st + kMdStages);
  }
  if (live) {
    const size_t FK = (size_t)gp.F * mp.K;
#pragma unroll
    for (int r = 0; r < kMdChunk; r++) {
      if (r >= nr) break;
      double* p = mp.partial + ((size_t)split * FK + (size_t)f * mp.K + r0 + r) * 3;
      p[0] = (double)shift[r];
      p[1] = s1[r];
      p[2] = s2[r];
    }
    if (bad && blockIdx.y == 0) atomicAdd(mp.invalid, bad);
  }
}

// combines the draw splits in split order (deterministic; Chan et al.'s pairwise update of count, mean and sum of
// squared deviations): stats[row] = (mean, sd with divisor S)
__global__ void market_finalize(const __grid_constant__ MarketParams mp) {
  const GridParams& gp = mp.gp;
  const size_t FK = (size_t)gp.F * mp.K;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= FK) return;
  // means relative to the first split's p0 (differences of float32 values are exact in float64): the merge keeps the
  // precision of a row that barely varies
  const double ref = mp.partial[i * 3];
  double n = 0.0, mean = 0.0, m2 = 0.0;
  for (int k = 0; k < gp.nsplit; k++) {
    const double* p = mp.partial + ((size_t)k * FK + i) * 3;
    const double nk = (double)min(gp.samples_per_split, gp.S - k * gp.samples_per_split);
    const double mk = (p[0] - ref) + p[1] / nk, m2k = fmax(p[2] - p[1] * (p[1] / nk), 0.0);
    if (k == 0) {
      n = nk, mean = mk, m2 = m2k;
    } else {
      const double d = mk - mean, nn = n + nk;
      mean += d * (nk / nn);
      m2 += m2k + d * d * (n * nk / nn);
      n = nn;
    }
  }
  mp.stats[i * 2 + 0] = ref + mean;
  mp.stats[i * 2 + 1] = sqrt(m2 / n);
}

int market_rows(const bplx_market_lines* lines, int max_goals, MarketParams* mp) {
  BPLX_REQUIRE(lines != nullptr, BPLX_E_INVALID, "markets: lines is NULL");
  const int G = max_goals;
  BPLX_REQUIRE(lines->num_total_lines >= 0 && lines->num_total_lines <= BPLX_MARKET_MAX_LINES &&
                   lines->num_margin_lines >= 0 && lines->num_margin_lines <= BPLX_MARKET_MAX_LINES,
               BPLX_E_INVALID, "markets: 0 .. %d lines of each kind (got %d total, %d margin)", BPLX_MARKET_MAX_LINES,
               lines->num_total_lines, lines->num_margin_lines);
  // the cells (i, j) of the low corner a row covers, as bits 2i + j
  auto corner = [](auto covers) {
    uint8_t m = 0;
    for (int i = 0; i < 2; i++)
      for (int j = 0; j < 2; j++)
        if (covers(i, j)) m |= (uint8_t)(1u << (2 * i + j));
    return m;
  };
  MarketRow* r = mp->row;
  int K = 0;
  r[K++] = {kRowPrefix, 1, 0, corner([](int i, int j) { return i > j; }), -1};   // home win: j <= i - 1
  r[K++] = {kRowDiagonal, 0, 0, corner([](int i, int j) { return i == j; }), 0};
  r[K++] = {kRowSuffix, 1, 0, corner([](int i, int j) { return i < j; }), 1};    // away win: j >= i + 1
  r[K++] = {kRowSuffix, 0, 1, corner([](int i, int j) { return i >= 1 && j >= 1; }), 1};  // i >= 1, j >= 1
  r[K++] = {kRowHomeRate, 0, 0, 0, 0};
  r[K++] = {kRowAwayRate, 0, 0, 0, 0};
  // a half-integer line x = m + 1/2: "over" is >= m + 1, "under" is <= m
  auto line_m = [](double x, double lo, double hi, int* m) {
    const double t = 2.0 * x;
    if (!(x >= lo && x <= hi) || t != floor(t) || fmod(fabs(t), 2.0) != 1.0) return false;
    *m = (int)floor(x);
    return true;
  };
  for (int l = 0; l < lines->num_total_lines; l++) {
    int m = 0;
    const double x = lines->total_lines[l];
    BPLX_REQUIRE(line_m(x, 0.5, 2.0 * G - 0.5, &m), BPLX_E_INVALID,
                 "markets: total line %g is not a half-integer in [0.5, %g] (max_goals %d)", x, 2.0 * G - 0.5, G);
    r[K++] = {kRowSuffix, -1, 0, corner([m](int i, int j) { return i + j >= m + 1; }), m + 1};  // j >= m + 1 - i
    r[K++] = {kRowPrefix, -1, 0, corner([m](int i, int j) { return i + j <= m; }), m};          // j <= m - i
  }
  for (int l = 0; l < lines->num_margin_lines; l++) {
    int m = 0;
    const double x = lines->margin_lines[l];
    BPLX_REQUIRE(line_m(x, -G + 0.5, G - 0.5, &m), BPLX_E_INVALID,
                 "markets: margin line %g is not a half-integer in [%g, %g] (max_goals %d)", x, -G + 0.5, G - 0.5, G);
    r[K++] = {kRowPrefix, 1, 0, corner([m](int i, int j) { return i - j >= m + 1; }), -m - 1};  // j <= i - m - 1
    r[K++] = {kRowSuffix, 1, 0, corner([m](int i, int j) { return i - j <= m; }), -m};          // j >= i - m
  }
  mp->K = K;
  return BPLX_OK;
}

size_t market_plan(MarketParams* mp, const char** err) {
  GridParams* gp = &mp->gp;
  const size_t table_bytes = table_layout(gp);
  const size_t row_bytes = (size_t)gp->row_floats * 4;
  if (row_bytes > (size_t)kMdStageBytes) {
    if (err) *err = "markets: a draw row (teams x tables) does not fit one stage buffer: too many teams";
    return 0;
  }
  int ns = (int)((size_t)kMdStageBytes / row_bytes);
  ns = ns > kGridStageMax ? kGridStageMax : ns;
  gp->ns_stage = ns >= 4 ? ns / 4 * 4 : ns;  // a multiple of 4: every stage starts on a 16-byte boundary of a matrix row
  // splits from S and the row layout only, never from F (pointwise_plan's rule): a row's statistics are the same bits
  // whichever fixtures share the call
  int best = gp->S / (4 * gp->ns_stage);
  best = best < 1 ? 1 : (best > 64 ? 64 : best);
  int sps = (gp->S + best - 1) / best;
  sps = (sps + gp->ns_stage - 1) / gp->ns_stage * gp->ns_stage;
  gp->nsplit = (gp->S + sps - 1) / sps;
  gp->samples_per_split = sps;
  return table_bytes + (size_t)gp->nsplit * gp->F * mp->K * 3 * sizeof(double);
}

int launch_market_draws(MarketParams& mp, cudaStream_t stream) {
  GridParams& gp = mp.gp;
  int rc = upload_market_constants();
  if (rc != BPLX_OK) return rc;
  mp.vec = mp.draws && mp.ld % 4 == 0 && gp.ns_stage % 4 == 0 && (reinterpret_cast<uintptr_t>(mp.draws) & 15u) == 0;
  const size_t smem = 128 + (size_t)kMdStages * gp.ns_stage * gp.row_floats * 4 + sums_bytes(gp.g);
  BPLX_REQUIRE(smem <= 227 * 1024, BPLX_E_UNSUPPORTED, "markets: %zu bytes of shared memory per CTA needed (max %d)",
               smem, 227 * 1024);
  BPLX_CUDA(cudaMemsetAsync(mp.invalid, 0, sizeof(int), stream));
  rc = launch_score_grid_tables(gp, stream);
  if (rc != BPLX_OK) return rc;
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    BPLX_CUDA(cudaFuncSetAttribute(market_draws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  dim3 grid((gp.F + kMdThreads - 1) / kMdThreads, (mp.K + kMdChunk - 1) / kMdChunk, gp.nsplit);
  market_draws_kernel<<<grid, kMdThreads, smem, stream>>>(mp);
  BPLX_CUDA(cudaGetLastError());
  const size_t FK = (size_t)gp.F * mp.K;
  market_finalize<<<(unsigned)((FK + 255) / 256), 256, 0, stream>>>(mp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(2);
  return BPLX_OK;
}

// ---- quantile kernel ------------------------------------------------------------------------------------------------
namespace {

using radix::f2key;
using radix::hist_add;
using radix::kBins;

struct MqShared {
  uint32_t target[kMqMaxRanks];   // the distinct 1-based ranks to select
  uint32_t rank[kMqMaxRanks];     // the rank inside the current bin
  uint32_t bin[kMqMaxRanks];
  uint32_t prefix[kMqMaxRanks];   // key bits selected so far
  uint32_t uprefix[kMqMaxRanks];  // the distinct prefixes of the pass
  uint32_t slot[kMqMaxRanks];     // histogram of each rank in the pass
  uint32_t wsum[kMqThreads / 32];
  long long cnt[kMqThreads / 32];
  int nr, nu;
};

// slots of the distinct values of (prefix >> shift) over the nr ranks (one thread)
__device__ void assign_slots(MqShared& sh, int shift) {
  int nu = 0;
  for (int j = 0; j < sh.nr; j++) {
    const uint32_t p = sh.prefix[j] >> shift;
    int s = 0;
    while (s < nu && sh.uprefix[s] != p) s++;
    if (s == nu) sh.uprefix[nu++] = p;
    sh.slot[j] = s;
  }
  sh.nu = nu;
}

// find_bins on each slot's histogram of nb bins, for the ranks of that slot
__device__ void find_slot_bins(const uint32_t* hist, int nb, MqShared& sh) {
  const int nu = sh.nu;  // (read once: thread 0 reassigns the slots after the last barrier)
  for (int s = 0; s < nu; s++) {
    uint32_t which = 0;
    for (int j = 0; j < sh.nr; j++)
      if (sh.slot[j] == (uint32_t)s) which |= 1u << j;
    radix::find_bins<kMqThreads, kMqMaxRanks>(hist + (size_t)s * nb, nb, which, sh.rank, sh.bin, sh.wsum);
  }
}

}  // namespace

__global__ void __launch_bounds__(kMqThreads) market_quantile_kernel(const __grid_constant__ QuantileParams qp) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  __shared__ MqShared sh;
  __shared__ int8_t lut[kBins];  // top bin -> its histogram in pass 2, -1 for bins no rank is in
  uint32_t* const hist = reinterpret_cast<uint32_t*>(smem_dyn);  // [max(1, 2 nq)][kBins]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = blockIdx.x, S = qp.S;
  const float* row = qp.rows + (size_t)r * qp.ld;
  const double odds = qp.odds ? qp.odds[r] : 0.0;

  if (tid == 0) {  // the distinct 0-based order statistics k and k + 1 of the levels, ascending
    int nr = 0;
    for (int l = 0; l < qp.nq; l++) {
      const double hv = (double)(S - 1) * qp.level[l];
      const int k = hv >= (double)(S - 1) ? S - 1 : (int)floor(hv);
      for (int kk = k; kk <= min(k + 1, S - 1); kk++) {
        int j = 0;
        while (j < nr && sh.target[j] != (uint32_t)kk + 1) j++;
        if (j == nr) sh.target[nr++] = (uint32_t)kk + 1;
      }
    }
    for (int j = 0; j < nr; j++) sh.rank[j] = sh.target[j];
    sh.nr = nr;
  }
  for (int i = tid; i < kBins; i += kMqThreads) hist[i] = 0;
  __syncthreads();

  // (1) histogram of the top 11 key bits, odds exceedances
  long long cnt = 0;
  radix::for_row<kMqThreads>(row, S, [&](float v) {
    cnt += (double)v * odds > 1.0;
    hist_add(hist, f2key(v) >> 21);
  });
#pragma unroll
  for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) sh.cnt[warp] = cnt;
  __syncthreads();
  const int nr = sh.nr;
  if (nr > 0) {
    const uint32_t all = (nr >= 32) ? 0xffffffffu : (1u << nr) - 1u;
    radix::find_bins<kMqThreads, kMqMaxRanks>(hist, kBins, all, sh.rank, sh.bin, sh.wsum);
    if (tid == 0) {
      for (int j = 0; j < nr; j++) sh.prefix[j] = sh.bin[j] << 21;
      assign_slots(sh, 21);
    }
    for (int i = tid; i < kBins; i += kMqThreads) lut[i] = -1;
    __syncthreads();
    const int nu2 = sh.nu;
    if (tid < nu2) lut[sh.uprefix[tid]] = (int8_t)tid;
    for (int i = tid; i < nu2 * kBins; i += kMqThreads) hist[i] = 0;
    __syncthreads();

    // (2) the next 11 bits of the values in a selected top bin
    radix::for_row<kMqThreads>(row, S, [&](float v) {
      const uint32_t k = f2key(v);
      const int s = lut[k >> 21];
      if (s >= 0) hist_add(hist, (uint32_t)s * kBins + ((k >> 10) & 2047u));
    });
    __syncthreads();
    find_slot_bins(hist, kBins, sh);
    if (tid == 0) {
      for (int j = 0; j < nr; j++) sh.prefix[j] |= sh.bin[j] << 10;
      assign_slots(sh, 10);
    }
    __syncthreads();
    const int nu3 = sh.nu;
    for (int i = tid; i < nu3 * 1024; i += kMqThreads) hist[i] = 0;
    __syncthreads();

    // (3) the last 10 bits of the values with a selected 22-bit prefix
    radix::for_row<kMqThreads>(row, S, [&](float v) {
      const uint32_t k = f2key(v);
      if (lut[k >> 21] >= 0) {
        for (int s = 0; s < nu3; s++)
          if ((k >> 10) == sh.uprefix[s]) {
            hist_add(hist, (uint32_t)s * 1024u + (k & 1023u));
            break;
          }
      }
    });
    __syncthreads();
    find_slot_bins(hist, 1024, sh);
  }
  if (tid == 0) {
    for (int j = 0; j < nr; j++) sh.prefix[j] |= sh.bin[j];
    if (qp.exceed) {
      long long total = 0;
      for (int w = 0; w < kMqThreads / 32; w++) total += sh.cnt[w];
      qp.exceed[r] = total;
    }
  }
  __syncthreads();
  // numpy's "linear" quantile: h = (S - 1) q, k = floor(h), t = h - k; a + (b - a) t for t < 1/2, b - (b - a)(1 - t)
  // otherwise (numpy's _lerp), in float64 without contraction
  if (tid < qp.nq) {
    const double hv = (double)(S - 1) * qp.level[tid];
    auto value = [&](int kk) {
      int j = 0;
      while (sh.target[j] != (uint32_t)kk + 1) j++;
      return (double)radix::key2f(sh.prefix[j]);
    };
    double q;
    if (hv >= (double)(S - 1)) {
      q = value(S - 1);
    } else {
      const int k = (int)floor(hv);
      const double t = __dsub_rn(hv, (double)k), lo = value(k), hi = value(k + 1);
      const double diff = __dsub_rn(hi, lo);
      q = t >= 0.5 ? __dsub_rn(hi, __dmul_rn(diff, __dsub_rn(1.0, t))) : __dadd_rn(lo, __dmul_rn(diff, t));
    }
    qp.quantiles[(size_t)r * qp.nq + tid] = q;
  }
}

int launch_market_quantiles(const QuantileParams& qp, cudaStream_t stream) {
  const size_t smem = (size_t)(qp.nq > 0 ? 2 * qp.nq : 1) * kBins * sizeof(uint32_t);
  static bool attr_done = false;  // (opt in once to the largest histogram set: the static MqShared comes on top)
  if (!attr_done) {
    BPLX_CUDA(cudaFuncSetAttribute(market_quantile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)(kMqMaxRanks * kBins * sizeof(uint32_t))));
    attr_done = true;
  }
  market_quantile_kernel<<<qp.R, kMqThreads, smem, stream>>>(qp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
