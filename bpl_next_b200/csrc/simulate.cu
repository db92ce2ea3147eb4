// simulate.cu -- season and group-stage simulation: every remaining fixture of a table played with the rates of ONE
// posterior draw per simulated season, then the table ranked.
//
// Definition (the same text in include/bplx.h, oracle/simulate.py and the docstrings):
//   simulation n = (first_draw + s) * R + r uses draw s; its random numbers are the outputs of curand_init(seed, n, 0)
//   followed by curand() (Philox4_32_10).  Words 2f and 2f+1 are u_h and u_a of fixture f through curand_uniform (in
//   (0, 1]); word 2F + t is the tie-break key of table slot t.  Every word has a fixed address, so a rounding difference
//   in one fixture cannot shift the random numbers of another.
//   Fixture f in draw s: lambda_h, lambda_a are the predict path's rates (neutral venues and confederations included,
//   Extended's clip not applied); G = max_goals; w(i, j) = tau+(i, j) Pois(i; lambda_h) Pois(j; lambda_a) on
//   0 <= i, j <= G with tau+ = tau clamped at 0 on the four low-score cells and 1 elsewhere; Z = sum w, m(i) = sum_j w(i, j).
//   Home goals = the smallest i with sum_{i' <= i} m(i') >= u_h Z; away goals = the smallest j with
//   sum_{j' <= j} w(i, j') >= u_a m(i); when rounding leaves a target unmet, the last index with positive mass.  A cell
//   of zero probability is never returned.
//   Table: points_win for a win, points_draw for a draw, goal difference and goals for added to the starting table.
//   Teams are ranked within their group by points, goal difference, goals for, then the tie-break key, all descending,
//   and the lower slot when even the keys are equal; position k (0-based) = the number of teams of the group ranked
//   ahead.  That is BPLX_RANK_GOAL_DIFF; under BPLX_RANK_HEAD_TO_HEAD (simulate_h2h_kernel) a set of teams level on
//   points is ordered by the points, goal difference and goals for of the matches among them (played and simulated),
//   the parts still level again by the matches among themselves, and a set that this separates nobody in by goal
//   difference, goals for, the key, then the lower slot.  Fair-play rules are not modelled.
//   A simulation with a non-finite rate, a normaliser that is not positive and finite, or a slot outside the table is
//   invalid: counted in `invalid`, left out of the histograms, its positions row 0xFF and that fixture's scores 0xFF.
//
// Kernel: one thread per simulation, simulations draw-major (the lanes of a warp share a draw when R >= 32).  The draw's
// exponential table row is K3's pre-pass (score_grid_tables), read through L1/L2.  Per fixture: the two gathered rates,
// two Philox words, one pass of the pmf recurrence p_k = p_{k-1} lambda / k over k <= G for both rates (the row sums),
// then the two cumulative walks, which stop at the sampled cell.  The pmfs are kept un-normalised (lambda^k / k!):
// e^-lambda_h e^-lambda_a cancels in the normalisation.  The team accumulators live in shared memory laid out
// [slot][thread]: every lane updates the same two slots for the same fixture, so no bank conflicts.  Ranking counts
// within the group (group member lists built once per CTA); per-CTA shared histograms are flushed with 64-bit atomics,
// so the integer counts are the same whatever order the atomics run in.
#include "simulate.h"

#include "sample_score.cuh"

#include "simulate_device.cuh"

namespace bplx {

// The kernels: simulate_body.inc with the ranking rule fixed at compile time
template <bool KO>
__global__ void __launch_bounds__(kSimThreads) simulate_kernel(const __grid_constant__ SimParams sp) {
  constexpr bool H2H = false, PAIRED = false;
#include "simulate_body.inc"
}

// the same, with the groups ranked by the head-to-head rule (bplx_ranking)
template <bool KO>
__global__ void __launch_bounds__(kSimThreads) simulate_h2h_kernel(const __grid_constant__ SimParams sp) {
  constexpr bool H2H = true, PAIRED = false;
#include "simulate_body.inc"
}

// the tournament with pairings drawn by lot (bplx_pairings), under either ranking rule
template <bool H2H_RULE>
__global__ void __launch_bounds__(kSimThreads) simulate_paired_kernel(const __grid_constant__ SimParams sp) {
  constexpr bool KO = true, H2H = H2H_RULE, PAIRED = true;
#include "simulate_body.inc"
}

// the remaining fixtures by slot pair, for the head-to-head ranking: pair_fix[pair_beg[p] .. pair_beg[p + 1]) are the
// fixtures between slots u < v, p = u NT + v, in no particular order (the ranking only sums over them).  One CTA of
// 1024 threads; a fixture with a slot outside the table or a team playing itself is left out.
__global__ void __launch_bounds__(1024) pair_index_kernel(const uint8_t* hslot, const uint8_t* aslot, int F, int NT,
                                                          int* pair_beg, int* pair_fix) {
  extern __shared__ int s_cnt[];  // [NT NT]: counts, then the cursors of the fill
  __shared__ int s_warp[32];
  const int np = NT * NT, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int p = tid; p < np; p += blockDim.x) s_cnt[p] = 0;
  __syncthreads();
  for (int f = tid; f < F; f += blockDim.x) {
    const int u = hslot[f], v = aslot[f];
    if (u != v && u < NT && v < NT) atomicAdd(&s_cnt[min(u, v) * NT + max(u, v)], 1);
  }
  __syncthreads();
  // exclusive scan: a chunk of pairs per thread, the chunk sums scanned per warp, then across the warps
  const int per = (np + blockDim.x - 1) / blockDim.x, lo = min(np, tid * per), hi = min(np, lo + per);
  int sum = 0;
  for (int p = lo; p < hi; p++) sum += s_cnt[p];
  int incl = sum;
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += o;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, w, d);
      if (lane >= d) w += o;
    }
    s_warp[lane] = w;
  }
  __syncthreads();
  int run = incl - sum + (warp ? s_warp[warp - 1] : 0);
  for (int p = lo; p < hi; p++) {
    const int c = s_cnt[p];
    s_cnt[p] = run;
    pair_beg[p] = run;
    run += c;
  }
  if (tid == (int)blockDim.x - 1) pair_beg[np] = run;
  __syncthreads();
  for (int f = tid; f < F; f += blockDim.x) {
    const int u = hslot[f], v = aslot[f];
    if (u != v && u < NT && v < NT) pair_fix[atomicAdd(&s_cnt[min(u, v) * NT + max(u, v)], 1)] = f;
  }
}

size_t simulate_smem_bytes(SimParams* sp) {
  size_t base = (size_t)sp->NT * kSimThreads * 16 + (size_t)sp->NT * sp->P * 4 + (size_t)sp->NT * 12;
  if (sp->ko.K > 0) {
    // the reach / win / decided histograms; the winner / loser bytes overlay s_gf and s_gd when they fit there (K <= 4
    // T_tab)
    base += (size_t)sp->NT * sp->ko.nr * 8 + (size_t)sp->ko.K * 8;
    sp->ko.wl_overlay = sp->ko.K <= 4 * sp->NT;
    if (!sp->ko.wl_overlay) base += (size_t)(2 * sp->ko.K + 3) / 4 * 4 * kSimThreads;
  }
  // the pool bytes of the paired kernel: in the s_key words past the qualifier map, the BEST bytes and the two 128-byte
  // per-CTA tables (row NT + bc + 2 of [row][thread]) when they fit there (4 T_tab rows), else appended
  size_t pool = 0;
  if (sp->ko.K > 0 && sp->pr.num > 0) {
    const int row = sp->NT + sp->ko.bc + 2;
    if (row + sp->pr.nbuf <= 4 * sp->NT) sp->pr.buf_off = (12 * sp->NT + row) * kSimThreads;
    else pool = (size_t)sp->pr.nbuf * kSimThreads;
  }
  // the conditional kernel's per-CTA tables (appended, 8-byte aligned) and its per-warp partial counts: in the
  // accumulators, dead once every simulation of the CTA is ranked, when they fit there (T_tab >= 4), else appended
  size_t cond = 0;
  if (sp->ko.K == 0 && sp->cd.nk > 0) {
    const size_t tab = (size_t)kCondTableWords * 8, buf = (size_t)2 * 7 * kSimThreads * 4;
    cond = 8 + tab + ((size_t)sp->NT * kSimThreads * 16 >= buf ? 0 : buf);
  }
  const size_t pts = (size_t)sp->NT * sp->B * 4;
  sp->points_in_smem = base + pool + cond + pts <= (size_t)kSimSmemMax;
  const size_t end = base + (sp->points_in_smem ? pts : 0);
  if (pool) sp->pr.buf_off = (int)end;
  if (cond) {
    sp->cd.tab_off = (int)((end + 7) / 8 * 8);
    const size_t tab_end = (size_t)sp->cd.tab_off + (size_t)kCondTableWords * 8;
    sp->cd.buf_off = (size_t)sp->NT * kSimThreads * 16 >= (size_t)2 * 7 * kSimThreads * 4 ? 0 : (int)tab_end;
    return sp->cd.buf_off ? tab_end + (size_t)2 * 7 * kSimThreads * 4 : tab_end;
  }
  return end + pool;
}

int launch_simulate(SimParams& sp, cudaStream_t stream) {
  int rc = upload_sim_constants();
  if (rc != BPLX_OK) return rc;
  const bool ko = sp.ko.K > 0;
  const size_t smem = simulate_smem_bytes(&sp);
  BPLX_REQUIRE(smem <= (size_t)kSimSmemMax, BPLX_E_UNSUPPORTED,
               "simulate: %zu bytes of shared memory per CTA needed (max %d)", smem, kSimSmemMax);
  // the dynamic shared-memory limit is an attribute of each instantiation
  static void (*const kernels[6])(const SimParams) = {
      simulate_kernel<false>,        simulate_kernel<true>,        simulate_h2h_kernel<false>,
      simulate_h2h_kernel<true>,     simulate_paired_kernel<false>, simulate_paired_kernel<true>};
  static size_t smem_set[6] = {48 * 1024, 48 * 1024, 48 * 1024, 48 * 1024, 48 * 1024, 48 * 1024};
  const bool h2h = sp.rule == BPLX_RANK_HEAD_TO_HEAD, cond = !ko && sp.cd.nk > 0;
  const int v = ko && sp.pr.num > 0 ? 4 + (int)h2h : (int)ko + (h2h ? 2 : 0);
  if (!cond && smem > smem_set[v]) {
    BPLX_CUDA(cudaFuncSetAttribute(kernels[v], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set[v] = smem;
  }
  BPLX_CUDA(cudaMemsetAsync(sp.pos_counts, 0, (size_t)sp.NT * sp.P * 8, stream));
  BPLX_CUDA(cudaMemsetAsync(sp.pts_counts, 0, (size_t)sp.NT * sp.B * 8, stream));
  BPLX_CUDA(cudaMemsetAsync(sp.invalid, 0, 8, stream));
  if (cond) {
    BPLX_CUDA(cudaMemsetAsync(sp.cd.outcome_counts, 0, (size_t)sp.cd.nk * 3 * 8, stream));
    BPLX_CUDA(cudaMemsetAsync(sp.cd.cond_counts, 0, (size_t)sp.cd.nk * 3 * sp.cd.ne * 8, stream));
  }
  if (ko) {
    BPLX_CUDA(cudaMemsetAsync(sp.ko.reach, 0, (size_t)sp.NT * sp.ko.nr * 8, stream));
    BPLX_CUDA(cudaMemsetAsync(sp.ko.win, 0, (size_t)sp.NT * sp.ko.nr * 8, stream));
    if (sp.ko.decided) BPLX_CUDA(cudaMemsetAsync(sp.ko.decided, 0, (size_t)sp.ko.K * 3 * 8, stream));
    if (sp.pr.counts)
      BPLX_CUDA(cudaMemsetAsync(sp.pr.counts, 0, (size_t)sp.pr.num * sp.NT * sp.NT * 8, stream));
  }
  rc = launch_score_grid_tables(sp.gp, stream);
  if (rc != BPLX_OK) return rc;
  if (h2h) {
    pair_index_kernel<<<1, 1024, (size_t)sp.NT * sp.NT * 4, stream>>>(sp.hslot, sp.aslot, sp.gp.F, sp.NT,
                                                                     sp.pair_beg, sp.pair_fix);
    BPLX_CUDA(cudaGetLastError());
    note_launch(1);
  }
  const unsigned grid = (unsigned)((sp.N + kSimThreads - 1) / kSimThreads);
  if (cond) return launch_simulate_cond(sp, grid, smem, stream);
  kernels[v]<<<grid, kSimThreads, smem, stream>>>(sp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
