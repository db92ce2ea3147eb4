// score_grid.cu -- K3: posterior-predictive score grid + outcome probabilities.
//
// Replaces predict_score_grid_proba / predict_outcome_proba (bpl/base.py:74-148,
// bpl/neutral_dixon_coles.py:562-659, bpl/neutral_dixon_coles_WC.py:548-670) and, inside them,
// _calculate_expected_goals + predict_score_proba (bpl/dixon_coles.py:126-163,
// bpl/extended_dixon_coles.py:335-399, bpl/neutral_dixon_coles.py:399-488,
// bpl/neutral_dixon_coles_WC.py:363-474) and dixon_coles_correlation_term with weights=None
// (bpl/_util.py:35-93).  The reference materialises [S, F*g*g] temporaries and recomputes the two
// rates g*g times per fixture.  Here:
//
//   pre-pass   every rate factors as lambda = exp(home team's half) * exp(away team's half) (* the confederation
//              factors), exactly as in K1 (plan.h): the exponentials are tabulated ONCE per (sample, team) into a
//              row per sample [P1 | Q1 | P0 | EC | corr_coef], so the pair loop below has no exp of a rate and
//              two gathers instead of twelve.
//   grid       one thread owns one fixture, keeps its g x g tile of the grid in registers and walks the posterior
//              samples; sample rows are contiguous, so a stage of samples is ONE cp.async.bulk (TMA, mbarrier
//              completion) into a double-buffered ring.  Per (sample, fixture): 2-4 LDS.64, the two e^-lambda
//              (MUFU.EX2), the pmf recurrences, tau on the four low-score cells (clamped at 0, bpl/_util.py:62-68)
//              and g*g FFMA.  g <= 11: un-normalised powers lambda^k (bounded: e^-l l^k <= (k/e)^k), the 1/(i! j!)
//              applied by the finalize kernel; larger grids: 8 x 16 tiles with the normalised recurrence
//              p_k = p_{k-1} * lambda / k (never overflows, any max_goals <= 63).
//   finalize   sums the sample splits in a fixed order (deterministic), applies `scale`, and reduces the W/D/L
//              masks of bpl/base.py:140-142 in the same pass; one warp per fixture.
//
//   grid = (F / 256 fixture blocks, grid tiles, sample splits).
#include "score_grid.h"

#include <math.h>

namespace bplx {

namespace {

__constant__ float c_inv_k[64];      // 1 / k            (k >= 1)
__constant__ double c_inv_fact[16];  // 1 / k!           (k <= 10 used)

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

}  // namespace

// ---- pre-pass: the exponential tables ------------------------------------------------------------------------------
//   home venue:  lambda_h = P1[h].x * Q1[a].x,  lambda_a = P1[h].y * Q1[a].y
//   neutral:     lambda_h = P0[h].x * P0[a].y,  lambda_a = P0[h].y * P0[a].x
//   P1 = (e^(att + home_attack), e^(-def - home_defence))   Q1 = (e^(-def - away_defence), e^(att + away_attack))
//   P0 = (e^att, e^-def)            EC[c] = (e^conf, e^-conf): lambda_h *= EC[hc].x EC[ac].y, lambda_a *= EC[ac].x EC[hc].y
// (DIXON_COLES / EXTENDED: home advantage in P1.x, no other venue effect.)
__global__ void score_grid_tables(const GridParams gp) {
  const int W = gp.T + gp.Cf + 1;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)gp.S * W) return;
  const int s = (int)(i / W), col = (int)(i % W);
  const RowLayout L = row_layout(gp.T, gp.Cf, gp.ntab);
  float* row = gp.table + (size_t)s * gp.row_floats;
  if (col < gp.T) {
    const size_t k = (size_t)s * gp.T + col;
    const float att = gp.attack[k], def = gp.defence[k];
    float ha, aa = 0.0f, hd = 0.0f, ad = 0.0f;
    if (gp.model == BPLX_DIXON_COLES) ha = gp.ha[s];
    else ha = gp.ha[k];
    if (gp.ntab == 3) {
      aa = gp.aa[k];
      hd = gp.hd[k];
      ad = gp.ad[k];
      reinterpret_cast<float2*>(row + L.P0)[col] = make_float2(expf(att), expf(-def));
    }
    reinterpret_cast<float2*>(row + L.P1)[col] = make_float2(expf(att + ha), expf(-def - hd));
    reinterpret_cast<float2*>(row + L.Q1)[col] = make_float2(expf(-def - ad), expf(att + aa));
  } else if (col < gp.T + gp.Cf) {
    const int c = col - gp.T;
    const float v = gp.conf[(size_t)s * gp.Cf + c];
    reinterpret_cast<float2*>(row + L.EC)[c] = make_float2(expf(v), expf(-v));
  } else {
    row[L.C] = gp.corr[s];
    for (int k = L.C + 1; k < gp.row_floats; k++) row[k] = 0.0f;
  }
}

// ---- grid kernel ---------------------------------------------------------------------------------------------------
// R x CC tile of the grid per thread; SINGLE = the tile is the whole grid (row/col origin 0, un-normalised powers).
template <int R, int CC, bool SINGLE>
__global__ void __launch_bounds__(kGridThreads, 1) score_grid_kernel(const __grid_constant__ GridParams gp) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // [0, 16): two mbarriers; [128, ...): kGridStages stage buffers of ns_stage rows; the epilogue reuses the buffers
  float* const buf0 = reinterpret_cast<float*>(smem_raw + 128);
  const uint32_t bar0 = smem_u32(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const RowLayout L = row_layout(gp.T, gp.Cf, gp.ntab);
  const int f_raw = blockIdx.x * kGridThreads + tid;
  const int f = min(f_raw, gp.F - 1);
  const int tiles_c = (gp.g + CC - 1) / CC;
  const int r0 = SINGLE ? 0 : (blockIdx.y / tiles_c) * R;
  const int c0 = SINGLE ? 0 : (blockIdx.y % tiles_c) * CC;
  const bool corner = SINGLE || (r0 == 0 && c0 == 0);
  const int split = blockIdx.z;
  const int s_begin = split * gp.samples_per_split;
  const int s_end = min(gp.S, s_begin + gp.samples_per_split);
  const int NS = gp.ns_stage;
  const uint32_t row_bytes = (uint32_t)gp.row_floats * 4u, stage_floats = (uint32_t)NS * gp.row_floats;

  // this thread's fixture: float offsets of its two table rows (and confederation entries) inside a sample row
  const int h = gp.home[f], a = gp.away[f];
  const bool wc = gp.model == BPLX_NEUTRAL_WC;
  const bool neutral = gp.ntab == 3 && gp.nv && gp.nv[f];
  const int offH = (neutral ? L.P0 : L.P1) + 2 * h;
  const int offA = (neutral ? L.P0 : L.Q1) + 2 * a;
  const int offEh = wc ? L.EC + 2 * gp.hconf[f] : 0, offEa = wc ? L.EC + 2 * gp.aconf[f] : 0;
  const int offC = L.C;

  float acc[R][CC];
#pragma unroll
  for (int i = 0; i < R; i++)
#pragma unroll
    for (int j = 0; j < CC; j++) acc[i][j] = 0.0f;
  // normalised recurrence (tile kernels): p_k = p_{k-1} * lambda / k
  float invr[R], invc[CC];
  if (!SINGLE) {
#pragma unroll
    for (int i = 0; i < R; i++) invr[i] = c_inv_k[min(r0 + i, 63)];
#pragma unroll
    for (int i = 0; i < CC; i++) invc[i] = c_inv_k[min(c0 + i, 63)];
  }

  const int nst = (s_end - s_begin + NS - 1) / NS;
  auto issue = [&](int st) {  // one bulk copy per stage: the sample rows are contiguous
    const int s0 = s_begin + st * NS;
    const uint32_t bytes = (uint32_t)min(NS, s_end - s0) * row_bytes;
    const uint32_t slot = (uint32_t)st % kGridStages;
    mbar_arrive_expect_tx(bar0 + 8 * slot, bytes);
    tma_load_1d(smem_u32(buf0 + slot * stage_floats), gp.table + (size_t)s0 * gp.row_floats, bytes, bar0 + 8 * slot);
  };
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kGridStages; s++) mbar_init(bar0 + 8 * s, 1);
    fence_mbar_init();
    fence_proxy_async();
    for (int st = 0; st < kGridStages && st < nst; st++) issue(st);
  }
  __syncthreads();

  constexpr float kLog2e = 1.4426950408889634f;
  for (int st = 0; st < nst; st++) {
    const float* cur = buf0 + (st % kGridStages) * stage_floats;
    mbar_wait(bar0 + 8 * (st % kGridStages), (st / kGridStages) & 1);
    const int ns = min(NS, s_end - (s_begin + st * NS));
    // Software pipeline over the samples of the stage: the gathers -> rates -> e^-lambda -> pmf chain of sample j+1 sits
    // in the same basic block as the R x CC FMAs of sample j, so the scheduler hides the chain behind the FMA stream
    // (two warps per scheduler cannot hide it by themselves).
    auto vectors = [&](int j, float (&ph)[R], float (&pa)[CC], float (&tt)[4]) {
      const float* row = cur + j * gp.row_floats;
      const float2 rh = *reinterpret_cast<const float2*>(row + offH);
      const float2 ra = *reinterpret_cast<const float2*>(row + offA);
      float lh = rh.x * (neutral ? ra.y : ra.x), la = rh.y * (neutral ? ra.x : ra.y);
      if (wc) {
        const float2 eh = *reinterpret_cast<const float2*>(row + offEh);
        const float2 ea = *reinterpret_cast<const float2*>(row + offEa);
        lh *= eh.x * ea.y;
        la *= ea.x * eh.y;
      }
      lh = fminf(lh, 1e30f);  // (an overflowed rate: e^-lambda = 0 and 0 * inf would be NaN)
      la = fminf(la, 1e30f);
      const float c = row[offC];
      if (SINGLE) {
        float p = ex2_approx(-kLog2e * lh);
        ph[0] = p;
#pragma unroll
        for (int i = 1; i < R; i++) {
          p *= lh;
          ph[i] = p;
        }
        p = ex2_approx(-kLog2e * la);
        pa[0] = p;
#pragma unroll
        for (int i = 1; i < CC; i++) {
          p *= la;
          pa[i] = p;
        }
      } else {
        // normalised recurrence p_k = p_{k-1} lambda / k, first up to the tile's first row / column
        float p = ex2_approx(-kLog2e * lh);
        for (int k = 1; k <= r0; k++) p *= lh * c_inv_k[k];
        ph[0] = p;
#pragma unroll
        for (int i = 1; i < R; i++) {
          p *= lh * invr[i];
          ph[i] = p;
        }
        p = ex2_approx(-kLog2e * la);
        for (int k = 1; k <= c0; k++) p *= la * c_inv_k[k];
        pa[0] = p;
#pragma unroll
        for (int i = 1; i < CC; i++) {
          p *= la * invc[i];
          pa[i] = p;
        }
      }
      // tau on the four low-score cells, clipped at 0 (bpl/_util.py:62-68)
      tt[0] = tt[1] = tt[2] = tt[3] = 1.0f;
      if (corner) {
        tt[0] = fmaxf(1.0f - (c * lh) * la, 0.0f);
        tt[1] = fmaxf(fmaf(c, lh, 1.0f), 0.0f);  // home 0, away 1
        tt[2] = fmaxf(fmaf(c, la, 1.0f), 0.0f);  // home 1, away 0
        tt[3] = fmaxf(1.0f - c, 0.0f);
      }
    };
    float ph[R], pa[CC], tt[4];
    vectors(0, ph, pa, tt);
#pragma unroll 1
    for (int j = 0; j < ns; j++) {
      float ph_n[R], pa_n[CC], tt_n[4];
      vectors(min(j + 1, ns - 1), ph_n, pa_n, tt_n);
#pragma unroll
      for (int i = 0; i < R; i++) {
#pragma unroll
        for (int jj = 0; jj < CC; jj++) {
          float w = ph[i];
          if (i < 2 && jj < 2) w *= tt[i * 2 + jj];
          acc[i][jj] = fmaf(w, pa[jj], acc[i][jj]);
        }
      }
#pragma unroll
      for (int i = 0; i < R; i++) ph[i] = ph_n[i];
#pragma unroll
      for (int i = 0; i < CC; i++) pa[i] = pa_n[i];
#pragma unroll
      for (int i = 0; i < 4; i++) tt[i] = tt_n[i];
    }
    __syncthreads();  // every thread is done with this buffer: refill it
    if (tid == 0 && st + kGridStages < nst) issue(st + kGridStages);
  }

  // ---- epilogue: the warp's 32 tiles go through shared memory so that the partial sums leave in coalesced rows ------
  constexpr int RC = R * CC, STRIDE = RC | 1;  // odd stride: conflict-free
  float* sm = buf0 + (size_t)warp * 32 * STRIDE;
#pragma unroll
  for (int i = 0; i < R; i++)
#pragma unroll
    for (int jj = 0; jj < CC; jj++) sm[lane * STRIDE + i * CC + jj] = acc[i][jj];
  __syncwarp();
  const int f0 = blockIdx.x * kGridThreads + warp * 32;
  const int nf = min(32, gp.F - f0);
  if (nf <= 0) return;
  const int gg = gp.g * gp.g;
  float* out = gp.partial + ((size_t)split * gp.F + f0) * (size_t)gg;
  if (SINGLE && gp.g == R) {  // the warp's tiles are one contiguous range of the partial array
    for (int idx = lane; idx < nf * RC; idx += 32) out[idx] = sm[(idx / RC) * STRIDE + idx % RC];
  } else {
    for (int fl = 0; fl < nf; fl++)
      for (int e = lane; e < RC; e += 32) {
        const int i = e / CC, jj = e % CC;
        if (r0 + i < gp.g && c0 + jj < gp.g) out[(size_t)fl * gg + (r0 + i) * gp.g + c0 + jj] = sm[fl * STRIDE + e];
      }
  }
}

// sums the sample splits in a fixed order, applies scale (and 1 / (hg! ag!) for the un-normalised small grids), reduces
// home_win / draw / away_win (bpl/base.py:140-142) from the same values; one warp per fixture
__global__ void score_grid_finalize(const GridParams gp) {
  const int f = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (f >= gp.F) return;
  const int g = gp.g, gg = g * g;
  const size_t n = (size_t)gp.F * gg;
  const bool fact = g <= 11;
  float hw = 0.0f, dr = 0.0f, aw = 0.0f;
  for (int cell = lane; cell < gg; cell += 32) {
    const size_t i = (size_t)f * gg + cell;
    float s = 0.0f;
    for (int k = 0; k < gp.nsplit; k++) s += gp.partial[(size_t)k * n + i];
    const int hg = cell / g, ag = cell % g;
    const float v = fact ? (float)((double)s * (double)gp.scale * c_inv_fact[hg] * c_inv_fact[ag]) : s * gp.scale;
    gp.grid[i] = v;
    if (hg > ag) hw += v;
    else if (hg == ag) dr += v;
    else aw += v;
  }
  if (!gp.outcome) return;
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    hw += __shfl_xor_sync(0xffffffffu, hw, o);
    dr += __shfl_xor_sync(0xffffffffu, dr, o);
    aw += __shfl_xor_sync(0xffffffffu, aw, o);
  }
  if (lane == 0) {
    gp.outcome[(size_t)f * 3 + 0] = hw;
    gp.outcome[(size_t)f * 3 + 1] = dr;
    gp.outcome[(size_t)f * 3 + 2] = aw;
  }
}

// ---- host side ---------------------------------------------------------------------------------------------------
static void tile_shape(int g, int* R, int* CC, int* ntiles) {
  if (g <= 11) {
    *R = 11; *CC = 11; *ntiles = 1;
  } else {
    *R = 8; *CC = 16;
    *ntiles = ((g + 7) / 8) * ((g + 15) / 16);
  }
}

size_t table_layout(GridParams* gp) {
  const bool neu = gp->model == BPLX_NEUTRAL || gp->model == BPLX_NEUTRAL_WC;
  gp->ntab = neu ? 3 : 2;
  const RowLayout L = row_layout(gp->T, gp->Cf, gp->ntab);
  gp->row_floats = (L.C + 1 + 3) / 4 * 4;
  return ((size_t)gp->S * gp->row_floats * 4 + 255) / 256 * 256;
}

size_t score_grid_plan(GridParams* gp, const char** err) {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
      sms = 148;
  }
  const size_t table_bytes = table_layout(gp);
  const size_t row_bytes = (size_t)gp->row_floats * 4;
  if (row_bytes > (size_t)kGridStageBytes) {
    if (err) *err = "score grid: a sample row (teams x tables) does not fit one stage buffer: too many teams";
    return 0;
  }
  int ns = (int)((size_t)kGridStageBytes / row_bytes);
  gp->ns_stage = ns > kGridStageMax ? kGridStageMax : ns;
  int R, CC, ntiles;
  tile_shape(gp->g, &R, &CC, &ntiles);
  const int nfb = (gp->F + kGridThreads - 1) / kGridThreads;
  const int per_min = 4 * gp->ns_stage;  // at least four stages per split
  int max_split = gp->S / per_min;
  max_split = max_split < 1 ? 1 : (max_split > 64 ? 64 : max_split);
  int best = 1;
  double best_eff = -1.0;
  for (int k = 1; k <= max_split; k++) {
    const long long ctas = (long long)nfb * ntiles * k;
    const long long waves = (ctas + sms - 1) / sms;
    const double eff = (double)ctas / (double)(waves * sms);
    if (eff > best_eff + 1e-9) best_eff = eff, best = k;
  }
  int sps = (gp->S + best - 1) / best;
  sps = (sps + gp->ns_stage - 1) / gp->ns_stage * gp->ns_stage;
  gp->nsplit = (gp->S + sps - 1) / sps;
  gp->samples_per_split = sps;
  return table_bytes + (size_t)gp->nsplit * gp->F * gp->g * gp->g * sizeof(float);
}

int launch_score_grid_tables(const GridParams& gp, cudaStream_t stream) {
  const long long n = (long long)gp.S * (gp.T + gp.Cf + 1);
  score_grid_tables<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(gp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

template <int R, int CC, bool SINGLE>
static int launch_tile(const GridParams& gp, int ntiles, size_t smem, cudaStream_t stream) {
  auto* fn = &score_grid_kernel<R, CC, SINGLE>;
  static bool attr_done = false;  // per instantiation
  if (!attr_done) {
    BPLX_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_done = true;
  }
  dim3 grid((gp.F + kGridThreads - 1) / kGridThreads, ntiles, gp.nsplit);
  fn<<<grid, kGridThreads, smem, stream>>>(gp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

static int upload_constants() {
  static bool done = false;
  if (done) return BPLX_OK;
  float inv[64];
  double invf[16];
  double fct = 1.0;
  for (int k = 0; k < 64; k++) inv[k] = k ? (float)(1.0 / k) : 0.0f;
  for (int k = 0; k < 16; k++) {
    if (k > 1) fct *= k;
    invf[k] = 1.0 / fct;
  }
  BPLX_CUDA(cudaMemcpyToSymbol(c_inv_k, inv, sizeof inv));
  BPLX_CUDA(cudaMemcpyToSymbol(c_inv_fact, invf, sizeof invf));
  done = true;
  return BPLX_OK;
}

int launch_score_grid(const GridParams& gp, cudaStream_t stream) {
  int rc = upload_constants();
  if (rc != BPLX_OK) return rc;
  int R, CC, ntiles;
  tile_shape(gp.g, &R, &CC, &ntiles);
  const size_t stage_bytes = (size_t)kGridStages * gp.ns_stage * gp.row_floats * 4;
  const size_t epi_bytes = (size_t)(kGridThreads / 32) * 32 * ((R * CC) | 1) * 4;
  const size_t smem = 128 + (stage_bytes > epi_bytes ? stage_bytes : epi_bytes);
  BPLX_REQUIRE(smem <= 227 * 1024, BPLX_E_UNSUPPORTED, "score grid needs %zu bytes of shared memory per CTA (max %d)", smem,
               227 * 1024);
  if (!gp.reuse_tables) {
    rc = launch_score_grid_tables(gp, stream);
    if (rc != BPLX_OK) return rc;
  }
  rc = gp.g <= 11 ? launch_tile<11, 11, true>(gp, ntiles, smem, stream) : launch_tile<8, 16, false>(gp, ntiles, smem, stream);
  if (rc != BPLX_OK) return rc;
  score_grid_finalize<<<(gp.F + 7) / 8, 256, 0, stream>>>(gp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
