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

namespace bplx {

namespace {

constexpr float kExtraTimeFraction = 1.0f / 3.0f;  // BPLX_EXTRA_TIME_FRACTION: 30 of 90 minutes at constant rates

// the draw's un-normalised win masses on the same clamped, truncated grid as sample_score: hw = sum_{i > j} w(i, j),
// aw = sum_{i < j} w(i, j), with running prefixes of the pmfs (O(G)); tau+ enters through the cells (1, 0) and (0, 1)
__device__ __forceinline__ void win_masses(float lh, float la, float c, int G, float& hw, float& aw) {
  float p = lh, q = la, Pc = 1.0f + lh, Qc = 1.0f + la;  // p_1, q_1, sum_{i <= 1} p_i, sum_{j <= 1} q_j
  hw = lh * fmaxf(fmaf(c, la, 1.0f), 0.0f);               // w(1, 0) = tau+(1, 0) p_1 q_0
  aw = la * fmaxf(fmaf(c, lh, 1.0f), 0.0f);               // w(0, 1)
  for (int k = 2; k <= G; k++) {
    p *= lh * c_sim_inv_k[k];
    q *= la * c_sim_inv_k[k];
    hw = fmaf(p, Qc, hw);
    aw = fmaf(q, Pc, aw);
    Qc += q;
    Pc += p;
  }
}

// word w of the Philox sequence of simulation n (philox_block): the tournament kernel reads the slot tie-break keys
// only when points, goal difference and goals for are level
__device__ __forceinline__ uint32_t philox_word(unsigned long long seed, unsigned long long n, unsigned w) {
  const uint4 o = philox_block(seed, n, w >> 2);
  const unsigned r = w & 3u;
  return r == 0 ? o.x : r == 1 ? o.y : r == 2 ? o.z : o.w;
}

}  // namespace

// Head-to-head ranking of every group of a valid simulation into k_q (k_q[gbeg + position] = slot).  Each group
// is sorted by points; bit 7 of a k_q byte marks the first position of a class of teams still level, bit 6 a class
// whose head-to-head separates nobody.  A class of two or more is sorted by the points, goal difference and goals
// for of the matches among its members (played, then this simulation's fixtures, re-sampled from their own Philox
// words: the scores that built the table); the parts still level become classes and go through that again.  A
// class that is not separated is sorted by goal difference, goals for, the key (word 2F + t), then the lower slot.
__device__ __forceinline__ void rank_head_to_head(const SimParams& sp, int tid, unsigned long long n, const RowLayout& L,
                                                  const float* row, float c, bool wc, const int* s_pts, const int* s_gf,
                                                  const int* s_gd, const int* s_members, const int* s_gcnt,
                                                  uint8_t* k_q) {
  const GridParams& gp = sp.gp;
  const int NT = sp.NT;
#define ACC(arr, t) arr[(t) * kSimThreads + tid]
#define BYTE(arr, k) arr[(k) * kSimThreads + tid]
  // fixture f's score again: words 2f, 2f + 1 are the (x, y) or (z, w) pair of Philox block f / 2
  auto rescore = [&](int f, int& hg, int& ag) {
    const uint4 w = philox_block(sp.seed, n, (unsigned)f >> 1);
    const bool neutral = gp.ntab == 3 && gp.nv && gp.nv[f];
    const FixtureOffsets off =
        fixture_offsets(L, gp.home[f], gp.away[f], neutral, wc, wc ? gp.hconf[f] : 0, wc ? gp.aconf[f] : 0);
    const float2 lam = fixture_rates(row, off, neutral, wc);
    sample_score(lam.x, lam.y, c, _curand_uniform(f & 1 ? w.z : w.x), _curand_uniform(f & 1 ? w.w : w.y), sp.G,
                 hg, ag);
  };
  // head-to-head points, goal difference and goals for of slot x against the other members of the class [a, b)
  auto h2h = [&](int x, int a, int b, int& hp, int& hd, int& hf) {
    hp = hd = hf = 0;
    for (int q = a; q < b; q++) {
      const int y = BYTE(k_q, q) & 63;
      if (y == x) continue;
      if (sp.h2h_played) {
        const int2 xy = sp.h2h_played[x * NT + y], yx = sp.h2h_played[y * NT + x];
        hp += xy.x;
        hf += xy.y;
        hd += xy.y - yx.y;
      }
      const int pr = min(x, y) * NT + max(x, y);
#pragma unroll 1
      for (int e = sp.pair_beg[pr]; e < sp.pair_beg[pr + 1]; e++) {
        const int f = sp.pair_fix[e];
        int hg = 0, ag = 0;
        rescore(f, hg, ag);
        const int gx = sp.hslot[f] == x ? hg : ag, gy = hg + ag - gx;
        hp += gx > gy ? sp.pw : gx == gy ? sp.pd : 0;
        hd += gx - gy;
        hf += gx;
      }
    }
  };
  // the end of the class that starts at position a
  auto class_end = [&](int a, int ge) {
    int b = a + 1;
    while (b < ge && !(BYTE(k_q, b) & 0x80)) b++;
    return b;
  };
  const unsigned wkey = 2u * (unsigned)gp.F;
  for (int g0 = 0; g0 < NT;) {
    const int ge = g0 + s_gcnt[s_members[g0]];
    for (int p = g0; p < ge; p++) {  // by points (insertion)
      const int x = s_members[p], px = ACC(s_pts, x);
      int q = p;
      for (; q > g0 && ACC(s_pts, BYTE(k_q, q - 1)) < px; q--) BYTE(k_q, q) = BYTE(k_q, q - 1);
      BYTE(k_q, q) = (uint8_t)x;
    }
    for (int p = g0, prev = 0; p < ge; p++) {
      const int x = BYTE(k_q, p), px = ACC(s_pts, x);
      if (p == g0 || px != prev) BYTE(k_q, p) = (uint8_t)(x | 0x80);
      prev = px;
    }
#pragma unroll 1
    for (int a = g0; a < ge;) {
      const int b = class_end(a, ge);
      if (b - a < 2 || (BYTE(k_q, a) & 0x40)) {
        a = b;
        continue;
      }
      BYTE(k_q, a) &= 63;
      // by head-to-head (insertion: the class keeps its members while a place is searched for)
#pragma unroll 1
      for (int p = a + 1; p < b; p++) {
        const int x = BYTE(k_q, p);
        int xp, xd, xf;
        h2h(x, a, b, xp, xd, xf);
        int q = p;
#pragma unroll 1
        for (; q > a; q--) {
          int yp, yd, yf;
          h2h(BYTE(k_q, q - 1), a, b, yp, yd, yf);
          if (!(xp != yp ? xp > yp : xd != yd ? xd > yd : xf > yf)) break;
        }
        for (int m = p; m > q; m--) BYTE(k_q, m) = BYTE(k_q, m - 1);
        BYTE(k_q, q) = (uint8_t)x;
      }
      // mark the parts; a class that is not split is settled, a split one is refined from its first part
      bool split = false;
#pragma unroll 1
      for (int p = a, pp = 0, pd = 0, pf = 0; p < b; p++) {
        const int x = BYTE(k_q, p) & 63;
        int xp, xd, xf;
        h2h(x, a, b, xp, xd, xf);
        const bool brk = p > a && (xp != pp || xd != pd || xf != pf);
        if (p == a || brk) BYTE(k_q, p) = (uint8_t)(x | 0x80);
        split = split || brk;
        pp = xp;
        pd = xd;
        pf = xf;
      }
      if (!split) {
        BYTE(k_q, a) |= 0x40;
        a = b;
      }
    }
    // the classes left level: goal difference, goals for, the key, then the lower slot
#pragma unroll 1
    for (int a = g0; a < ge;) {
      const int b = class_end(a, ge);
      BYTE(k_q, a) &= 63;
#pragma unroll 1
      for (int p = a + 1; p < b; p++) {
        const int x = BYTE(k_q, p), dx = ACC(s_gd, x), fx = ACC(s_gf, x);
        int q = p;
        for (; q > a; q--) {
          const int y = BYTE(k_q, q - 1), dy = ACC(s_gd, y), fy = ACC(s_gf, y);
          if (dx != dy ? dx < dy : fx != fy ? fx < fy : false) break;
          if (dx == dy && fx == fy) {
            const uint32_t kx = philox_word(sp.seed, n, wkey + x), ky = philox_word(sp.seed, n, wkey + y);
            if (kx != ky ? kx < ky : x > y) break;
          }
          BYTE(k_q, q) = (uint8_t)y;
        }
        BYTE(k_q, q) = (uint8_t)x;
      }
      a = b;
    }
    g0 = ge;
  }
#undef ACC
#undef BYTE
}

// The kernels: simulate_body.inc with the ranking rule fixed at compile time
template <bool KO>
__global__ void __launch_bounds__(kSimThreads) simulate_kernel(const __grid_constant__ SimParams sp) {
  constexpr bool H2H = false;
#include "simulate_body.inc"
}

// the same, with the groups ranked by the head-to-head rule (bplx_ranking)
template <bool KO>
__global__ void __launch_bounds__(kSimThreads) simulate_h2h_kernel(const __grid_constant__ SimParams sp) {
  constexpr bool H2H = true;
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
  const size_t pts = (size_t)sp->NT * sp->B * 4;
  sp->points_in_smem = base + pts <= (size_t)kSimSmemMax;
  return base + (sp->points_in_smem ? pts : 0);
}

int launch_simulate(SimParams& sp, cudaStream_t stream) {
  int rc = upload_sim_constants();
  if (rc != BPLX_OK) return rc;
  const bool ko = sp.ko.K > 0;
  const size_t smem = simulate_smem_bytes(&sp);
  BPLX_REQUIRE(smem <= (size_t)kSimSmemMax, BPLX_E_UNSUPPORTED,
               "simulate: %zu bytes of shared memory per CTA needed (max %d)", smem, kSimSmemMax);
  // the dynamic shared-memory limit is an attribute of each instantiation
  static void (*const kernels[4])(const SimParams) = {simulate_kernel<false>, simulate_kernel<true>,
                                                      simulate_h2h_kernel<false>, simulate_h2h_kernel<true>};
  static size_t smem_set[4] = {48 * 1024, 48 * 1024, 48 * 1024, 48 * 1024};
  const int v = (int)ko + (sp.rule == BPLX_RANK_HEAD_TO_HEAD ? 2 : 0);
  if (smem > smem_set[v]) {
    BPLX_CUDA(cudaFuncSetAttribute(kernels[v], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set[v] = smem;
  }
  BPLX_CUDA(cudaMemsetAsync(sp.pos_counts, 0, (size_t)sp.NT * sp.P * 8, stream));
  BPLX_CUDA(cudaMemsetAsync(sp.pts_counts, 0, (size_t)sp.NT * sp.B * 8, stream));
  BPLX_CUDA(cudaMemsetAsync(sp.invalid, 0, 8, stream));
  if (ko) {
    BPLX_CUDA(cudaMemsetAsync(sp.ko.reach, 0, (size_t)sp.NT * sp.ko.nr * 8, stream));
    BPLX_CUDA(cudaMemsetAsync(sp.ko.win, 0, (size_t)sp.NT * sp.ko.nr * 8, stream));
    if (sp.ko.decided) BPLX_CUDA(cudaMemsetAsync(sp.ko.decided, 0, (size_t)sp.ko.K * 3 * 8, stream));
  }
  rc = launch_score_grid_tables(sp.gp, stream);
  if (rc != BPLX_OK) return rc;
  if (v >= 2) {
    pair_index_kernel<<<1, 1024, (size_t)sp.NT * sp.NT * 4, stream>>>(sp.hslot, sp.aslot, sp.gp.F, sp.NT,
                                                                     sp.pair_beg, sp.pair_fix);
    BPLX_CUDA(cudaGetLastError());
    note_launch(1);
  }
  const unsigned grid = (unsigned)((sp.N + kSimThreads - 1) / kSimThreads);
  kernels[v]<<<grid, kSimThreads, smem, stream>>>(sp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
