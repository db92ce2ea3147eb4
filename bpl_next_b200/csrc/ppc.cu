// ppc.cu -- posterior predictive checks: whole replicated datasets of the observed matches, one posterior draw per
// replicate, each reduced to its statistics on the device.
//
// Definition (the same text in include/bplx.h, oracle/ppc.py, DESIGN §3f and the docstrings):
//   replicate n = (first_draw + s) * R + r (R = sims_per_draw) uses posterior draw s; its random numbers are
//   curand_init(seed, n, 0) followed by curand() (Philox4_32_10), and words 2m and 2m + 1 become u_h and u_a of observed
//   match m through curand_uniform: the word addresses bplx_simulate_table gives fixture f.  Match m is drawn by the
//   season simulation's sampler, unchanged (sample_score, DESIGN §3c): the predict path's rates (neutral venues and
//   confederations included, Extended's clip not applied), the draw's own grid up to max_goals with tau clamped at 0,
//   normalised by its sum, inverse CDF over home goals, then over away goals given home goals.  With the same seed,
//   draws and matches the replicated scores equal simulate_table's.  Match weights are ignored.
//   Statistics per replicate (integers): score_counts [B][B] (cell min(hg, B-1), min(ag, B-1)), outcome_counts [3]
//   (home wins, draws, away wins), goals [2] (home, away), total_goals_sq (sum_m (hg + ag)^2), team_points,
//   team_goals_for, team_goals_against [T] per model team (points = (points_win, points_draw)).
//   A replicate with a non-finite rate, a normaliser that is not positive and finite, or a match naming a team or
//   confederation outside the samples is invalid: counted in `invalid`, every statistic of its row -1, the offending
//   match's scores 0xFF.
//
// Kernel: one CTA per replicate.  The draw's exponential table row (K3's pre-pass, score_grid_tables) is copied into
// shared memory, beside the replicate's accumulators (B^2 + 3T ints).  Thread p takes match pairs (2p, 2p + 1) with
// stride kPpcThreads: one Philox4x32_10 block (counter p) is the four words of the pair.  Team and score-cell counts are
// shared integer atomics; outcome and goal totals stay in registers and are reduced per warp.  Integer sums are the same
// whatever order the atomics run in, so the statistics depend neither on the launch geometry nor on the draw range.
#include "ppc.h"

#include "sample_score.cuh"

namespace bplx {

namespace {

__global__ void __launch_bounds__(kPpcThreads) ppc_kernel(const __grid_constant__ PpcParams pp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const GridParams& gp = pp.gp;
  const int T = gp.T, M = gp.F, B = pp.B, tid = threadIdx.x;
  float* const s_row = reinterpret_cast<float*>(smem_raw);
  int* const s_cells = reinterpret_cast<int*>(s_row + gp.row_floats);  // [B][B]
  int* const s_pts = s_cells + B * B;                                   // [T]
  int* const s_gf = s_pts + T;
  int* const s_ga = s_gf + T;
  __shared__ int s_outcome[3];
  __shared__ unsigned long long s_goals[3];  // home goals, away goals, sum of squared match totals
  __shared__ int s_bad;

  const int i = blockIdx.x;  // (N < 2^31 per call)
  const int s = i / pp.R, r = i - s * pp.R;
  const unsigned long long n = (unsigned long long)(pp.first_draw + s) * (unsigned long long)pp.R + (unsigned)r;
  const float4* const src = reinterpret_cast<const float4*>(gp.table + (size_t)s * gp.row_floats);
  for (int k = tid; k < gp.row_floats / 4; k += kPpcThreads) reinterpret_cast<float4*>(s_row)[k] = src[k];
  for (int k = tid; k < B * B + 3 * T; k += kPpcThreads) s_cells[k] = 0;
  if (tid < 3) {
    s_outcome[tid] = 0;
    s_goals[tid] = 0ull;
  }
  if (tid == 0) s_bad = 0;
  __syncthreads();

  const RowLayout L = row_layout(T, gp.Cf, gp.ntab);
  const float c = s_row[L.C];
  const bool wc = gp.model == BPLX_NEUTRAL_WC;
  const int pw = pp.pw, pd = pp.pd;
  int nh = 0, nd = 0, na = 0;
  unsigned gh = 0, ga = 0;
  unsigned long long sq = 0;
  bool bad = false;
  uint8_t* const sc = pp.scores ? pp.scores + (size_t)i * M * 2 : nullptr;
  // match m with the uniforms of words (wh, wa): sampled, counted, and its raw scores written
  auto play = [&](int m, unsigned wh, unsigned wa) {
    const int ht = gp.home[m], at = gp.away[m];
    const bool neutral = gp.ntab == 3 && gp.nv && gp.nv[m];
    const int hc = wc ? gp.hconf[m] : 0, ac = wc ? gp.aconf[m] : 0;
    int hg = 0xFF, ag = 0xFF;
    bool ok = ht < T && at < T && (!wc || (hc < gp.Cf && ac < gp.Cf));
    if (ok) {
      const FixtureOffsets off = fixture_offsets(L, ht, at, neutral, wc, hc, ac);
      const float2 lam = fixture_rates(s_row, off, neutral, wc);
      ok = sample_score(lam.x, lam.y, c, _curand_uniform(wh), _curand_uniform(wa), pp.G, hg, ag);
    }
    if (ok) {
      atomicAdd(&s_cells[min(hg, B - 1) * B + min(ag, B - 1)], 1);
      atomicAdd(&s_pts[ht], hg > ag ? pw : hg == ag ? pd : 0);
      atomicAdd(&s_pts[at], ag > hg ? pw : hg == ag ? pd : 0);
      atomicAdd(&s_gf[ht], hg);
      atomicAdd(&s_ga[ht], ag);
      atomicAdd(&s_gf[at], ag);
      atomicAdd(&s_ga[at], hg);
      nh += hg > ag;
      nd += hg == ag;
      na += hg < ag;
      gh += hg;
      ga += ag;
      sq += (unsigned long long)((hg + ag) * (hg + ag));
    } else {
      bad = true;
      hg = ag = 0xFF;
    }
    if (sc) *reinterpret_cast<uchar2*>(sc + 2 * m) = make_uchar2((unsigned char)hg, (unsigned char)ag);
  };
#pragma unroll 1
  for (int p = tid; 2 * p < M; p += kPpcThreads) {
    const uint4 w = philox_block(pp.seed, n, (unsigned)p);  // words 4p .. 4p + 3: matches 2p and 2p + 1
    play(2 * p, w.x, w.y);
    if (2 * p + 1 < M) play(2 * p + 1, w.z, w.w);
  }
  for (int d = 16; d > 0; d >>= 1) {
    nh += __shfl_down_sync(0xffffffffu, nh, d);
    nd += __shfl_down_sync(0xffffffffu, nd, d);
    na += __shfl_down_sync(0xffffffffu, na, d);
    gh += __shfl_down_sync(0xffffffffu, gh, d);
    ga += __shfl_down_sync(0xffffffffu, ga, d);
    sq += __shfl_down_sync(0xffffffffu, sq, d);
  }
  if ((tid & 31) == 0) {
    atomicAdd(&s_outcome[0], nh);
    atomicAdd(&s_outcome[1], nd);
    atomicAdd(&s_outcome[2], na);
    atomicAdd(&s_goals[0], (unsigned long long)gh);
    atomicAdd(&s_goals[1], (unsigned long long)ga);
    atomicAdd(&s_goals[2], sq);
  }
  if (bad) s_bad = 1;
  __syncthreads();

  // the replicate's statistics, -1 throughout when it is invalid
  const bool inv = s_bad != 0;
  for (int k = tid; k < B * B; k += kPpcThreads) pp.score_counts[(size_t)i * B * B + k] = inv ? -1 : s_cells[k];
  for (int k = tid; k < T; k += kPpcThreads) {
    pp.team_points[(size_t)i * T + k] = inv ? -1 : s_pts[k];
    pp.team_goals_for[(size_t)i * T + k] = inv ? -1 : s_gf[k];
    pp.team_goals_against[(size_t)i * T + k] = inv ? -1 : s_ga[k];
  }
  if (tid < 3) pp.outcome_counts[(size_t)i * 3 + tid] = inv ? -1 : s_outcome[tid];
  if (tid < 2) pp.goals[(size_t)i * 2 + tid] = inv ? -1ll : (long long)s_goals[tid];
  if (tid == 0) {
    pp.total_goals_sq[i] = inv ? -1ll : (long long)s_goals[2];
    if (inv) atomicAdd(pp.invalid, 1ull);
  }
}

}  // namespace

size_t ppc_smem_bytes(const PpcParams& pp) {
  return (size_t)pp.gp.row_floats * 4 + ((size_t)pp.B * pp.B + 3 * (size_t)pp.gp.T) * 4;
}

int launch_ppc(const PpcParams& pp, cudaStream_t stream) {
  int rc = upload_sim_constants();
  if (rc != BPLX_OK) return rc;
  const size_t smem = ppc_smem_bytes(pp);
  BPLX_REQUIRE(smem <= (size_t)kPpcSmemMax, BPLX_E_UNSUPPORTED,
               "posterior predictive: %zu bytes of shared memory per CTA needed for %d teams (max %d)", smem, pp.gp.T,
               kPpcSmemMax);
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    BPLX_CUDA(cudaFuncSetAttribute(ppc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  BPLX_CUDA(cudaMemsetAsync(pp.invalid, 0, 8, stream));
  rc = launch_score_grid_tables(pp.gp, stream);
  if (rc != BPLX_OK) return rc;
  ppc_kernel<<<(unsigned)pp.N, kPpcThreads, smem, stream>>>(pp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
