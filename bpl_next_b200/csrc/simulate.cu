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
//   ahead.  Head-to-head and fair-play rules are not modelled: ties left after goals for are decided by lot.
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

#include <curand_kernel.h>
#include <float.h>

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

}  // namespace

__global__ void __launch_bounds__(kSimThreads) simulate_kernel(const __grid_constant__ SimParams sp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const GridParams& gp = sp.gp;
  const int NT = sp.NT, tid = threadIdx.x;
  // [slot][thread] accumulators, then the histograms, then the group member lists
  int* const s_pts = reinterpret_cast<int*>(smem_raw);
  int* const s_gf = s_pts + NT * kSimThreads;
  int* const s_gd = s_gf + NT * kSimThreads;  // goals against during the fixtures, goal difference for the ranking
  uint32_t* const s_key = reinterpret_cast<uint32_t*>(s_gd + NT * kSimThreads);
  unsigned* const h_pos = s_key + NT * kSimThreads;
  unsigned* const h_pts = h_pos + NT * sp.P;
  int* const s_members = reinterpret_cast<int*>(h_pts + (sp.points_in_smem ? NT * sp.B : 0));
  int* const s_gbeg = s_members + NT;
  int* const s_gcnt = s_gbeg + NT;
  __shared__ unsigned s_invalid;
  __shared__ int s_groups_fit;
#define ACC(arr, t) arr[(t) * kSimThreads + tid]

  if (tid == 0) {
    s_invalid = 0;
    s_groups_fit = 1;
  }
  for (int k = tid; k < NT * sp.P; k += kSimThreads) h_pos[k] = 0;
  if (sp.points_in_smem)
    for (int k = tid; k < NT * sp.B; k += kSimThreads) h_pts[k] = 0;
  __syncthreads();
  // group member lists: slots sorted by (group, slot); s_gbeg / s_gcnt = where a slot's group starts and its size
  for (int t = tid; t < NT; t += kSimThreads) {
    const int g = sp.group ? sp.group[t] : 0;
    int beg = 0, before = 0, cnt = 0;
    for (int u = 0; u < NT; u++) {
      const int gu = sp.group ? sp.group[u] : 0;
      beg += gu < g;
      cnt += gu == g;
      before += gu == g && u < t;
    }
    s_members[beg + before] = t;
    s_gbeg[t] = beg;
    s_gcnt[t] = cnt;
    if (cnt > sp.P) s_groups_fit = 0;
  }
  __syncthreads();

  const int i = blockIdx.x * kSimThreads + tid;  // (N < 2^31 per call)
  if (i < sp.N) {
    const int s = i / sp.R, r = i - s * sp.R;
    const unsigned long long n = (unsigned long long)(sp.first_draw + s) * (unsigned long long)sp.R + (unsigned)r;
    curandStatePhilox4_32_10_t rng;
    curand_init(sp.seed, n, 0ull, &rng);
    const RowLayout L = row_layout(gp.T, gp.Cf, gp.ntab);
    const float* const row = gp.table + (size_t)s * gp.row_floats;
    const float c = row[L.C];
    const bool wc = gp.model == BPLX_NEUTRAL_WC;
    for (int t = 0; t < NT; t++) {
      ACC(s_pts, t) = sp.start_pts[t];
      ACC(s_gf, t) = sp.start_gf[t];
      ACC(s_gd, t) = sp.start_ga[t];
    }
    bool ok = true;
    uint8_t* const sc = sp.scores ? sp.scores + (size_t)i * gp.F * 2 : nullptr;
#pragma unroll 1
    for (int f = 0; f < gp.F; f++) {
      const int hs = sp.hslot[f], as = sp.aslot[f];
      const bool neutral = gp.ntab == 3 && gp.nv && gp.nv[f];
      const FixtureOffsets off =
          fixture_offsets(L, gp.home[f], gp.away[f], neutral, wc, wc ? gp.hconf[f] : 0, wc ? gp.aconf[f] : 0);
      const float2 lam = fixture_rates(row, off, neutral, wc);
      const float uh = curand_uniform(&rng), ua = curand_uniform(&rng);
      int hg = 0, ag = 0;
      const bool fok = sample_score(lam.x, lam.y, c, uh, ua, sp.G, hg, ag) && hs < NT && as < NT;
      if (fok) {
        const int ph = hg > ag ? sp.pw : hg == ag ? sp.pd : 0;
        const int pa = ag > hg ? sp.pw : hg == ag ? sp.pd : 0;
        ACC(s_pts, hs) += ph;
        ACC(s_gf, hs) += hg;
        ACC(s_gd, hs) += ag;
        ACC(s_pts, as) += pa;
        ACC(s_gf, as) += ag;
        ACC(s_gd, as) += hg;
      } else {
        ok = false;
        hg = ag = 0xFF;
      }
      if (sc) *reinterpret_cast<uchar2*>(sc + 2 * f) = make_uchar2((unsigned char)hg, (unsigned char)ag);
    }
    for (int t = 0; t < NT; t++) {
      ACC(s_key, t) = curand(&rng);
      ACC(s_gd, t) = ACC(s_gf, t) - ACC(s_gd, t);
      const int gained = ACC(s_pts, t) - sp.start_pts[t];
      ok = ok && gained >= 0 && gained < sp.B;  // (bins sized by the caller: a short one is refused, never overrun)
    }
    ok = ok && s_groups_fit;
    uint8_t* const prow = sp.positions ? sp.positions + (size_t)i * NT : nullptr;
    if (!ok) {
      atomicAdd(&s_invalid, 1u);
      if (prow)
        for (int t = 0; t < NT; t++) prow[t] = 0xFF;
    } else {
      for (int t = 0; t < NT; t++) {
        const int pt = ACC(s_pts, t), dt = ACC(s_gd, t), ft = ACC(s_gf, t);
        const uint32_t kt = ACC(s_key, t);
        const int g0 = s_gbeg[t], gc = s_gcnt[t];
        int pos = 0;
        for (int m = 0; m < gc; m++) {
          const int u = s_members[g0 + m];
          const int pu = ACC(s_pts, u), du = ACC(s_gd, u), fu = ACC(s_gf, u);
          const uint32_t ku = ACC(s_key, u);
          pos += pu != pt ? pu > pt : du != dt ? du > dt : fu != ft ? fu > ft : ku != kt ? ku > kt : u < t;
        }
        if (prow) prow[t] = (uint8_t)pos;
        atomicAdd(&h_pos[t * sp.P + pos], 1u);
        const int gained = pt - sp.start_pts[t];
        if (sp.points_in_smem) atomicAdd(&h_pts[t * sp.B + gained], 1u);
        else atomicAdd(&sp.pts_counts[(size_t)t * sp.B + gained], 1ull);
      }
    }
  }
#undef ACC
  __syncthreads();
  for (int k = tid; k < NT * sp.P; k += kSimThreads)
    if (h_pos[k]) atomicAdd(&sp.pos_counts[k], (unsigned long long)h_pos[k]);
  if (sp.points_in_smem)
    for (int k = tid; k < NT * sp.B; k += kSimThreads)
      if (h_pts[k]) atomicAdd(&sp.pts_counts[k], (unsigned long long)h_pts[k]);
  if (tid == 0 && s_invalid) atomicAdd(sp.invalid, (unsigned long long)s_invalid);
}

size_t simulate_plan(SimParams* sp) {
  GridParams* gp = &sp->gp;
  const bool neu = gp->model == BPLX_NEUTRAL || gp->model == BPLX_NEUTRAL_WC;
  gp->ntab = neu ? 3 : 2;
  const RowLayout L = row_layout(gp->T, gp->Cf, gp->ntab);
  gp->row_floats = (L.C + 1 + 3) / 4 * 4;
  return ((size_t)gp->S * gp->row_floats * 4 + 255) / 256 * 256;
}

size_t simulate_smem_bytes(SimParams* sp) {
  const size_t base = (size_t)sp->NT * kSimThreads * 16 + (size_t)sp->NT * sp->P * 4 + (size_t)sp->NT * 12;
  const size_t pts = (size_t)sp->NT * sp->B * 4;
  sp->points_in_smem = base + pts <= (size_t)kSimSmemMax;
  return base + (sp->points_in_smem ? pts : 0);
}

static int upload_sim_constants() {
  static bool done = false;
  if (done) return BPLX_OK;
  float inv[64];
  for (int k = 0; k < 64; k++) inv[k] = k ? (float)(1.0 / k) : 0.0f;
  BPLX_CUDA(cudaMemcpyToSymbol(c_sim_inv_k, inv, sizeof inv));
  done = true;
  return BPLX_OK;
}

int launch_simulate(SimParams& sp, cudaStream_t stream) {
  int rc = upload_sim_constants();
  if (rc != BPLX_OK) return rc;
  const size_t smem = simulate_smem_bytes(&sp);
  BPLX_REQUIRE(smem <= (size_t)kSimSmemMax, BPLX_E_UNSUPPORTED,
               "simulate: %zu bytes of shared memory per CTA needed (max %d)", smem, kSimSmemMax);
  static size_t smem_set = 48 * 1024;
  if (smem > smem_set) {
    BPLX_CUDA(cudaFuncSetAttribute(simulate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set = smem;
  }
  BPLX_CUDA(cudaMemsetAsync(sp.pos_counts, 0, (size_t)sp.NT * sp.P * 8, stream));
  BPLX_CUDA(cudaMemsetAsync(sp.pts_counts, 0, (size_t)sp.NT * sp.B * 8, stream));
  BPLX_CUDA(cudaMemsetAsync(sp.invalid, 0, 8, stream));
  rc = launch_score_grid_tables(sp.gp, stream);
  if (rc != BPLX_OK) return rc;
  simulate_kernel<<<(unsigned)((sp.N + kSimThreads - 1) / kSimThreads), kSimThreads, smem, stream>>>(sp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
