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
constexpr float kExtraTimeFraction = 1.0f / 3.0f;  // BPLX_EXTRA_TIME_FRACTION: 30 of 90 minutes at constant rates

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

// words 4b .. 4b + 3 of the Philox sequence of simulation n (curand_init(seed, n, 0) followed by curand()) without a
// state: one Philox4x32_10 block
__device__ __forceinline__ uint4 philox_block(unsigned long long seed, unsigned long long n, unsigned b) {
  return curand_Philox4x32_10(make_uint4(b, 0u, (unsigned)n, (unsigned)(n >> 32)),
                              make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
}

// word w of that sequence: the tournament kernel reads the slot tie-break keys only when points, goal difference and
// goals for are level
__device__ __forceinline__ uint32_t philox_word(unsigned long long seed, unsigned long long n, unsigned w) {
  const uint4 o = philox_block(seed, n, w >> 2);
  const unsigned r = w & 3u;
  return r == 0 ? o.x : r == 1 ? o.y : r == 2 ? o.z : o.w;
}

}  // namespace

// KO = false: season / group stage (bplx_simulate_table).  KO = true: the same group stage, then the knockout bracket
// (bplx_simulate_tournament / _ex).
template <bool KO>
__global__ void __launch_bounds__(kSimThreads) simulate_kernel(const __grid_constant__ SimParams sp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const GridParams& gp = sp.gp;
  const KoParams& ko = sp.ko;
  const int NT = sp.NT, tid = threadIdx.x;
  // [slot][thread] accumulators, then the histograms, then the group member lists
  int* const s_pts = reinterpret_cast<int*>(smem_raw);
  int* const s_gf = s_pts + NT * kSimThreads;
  int* const s_gd = s_gf + NT * kSimThreads;  // goals against during the fixtures, goal difference for the ranking
  uint32_t* const s_key = reinterpret_cast<uint32_t*>(s_gd + NT * kSimThreads);
  unsigned* const h_pos = s_key + NT * kSimThreads;
  unsigned* const h_pts = h_pos + NT * sp.P;
  unsigned* const h_reach = h_pts + (sp.points_in_smem ? NT * sp.B : 0);  // tournament: [NT][nr] each
  unsigned* const h_win = h_reach + (KO ? NT * ko.nr : 0);
  // tournament: [K][2] ties settled in extra time / by u_d (the rest of the CTA's valid simulations: in normal time)
  unsigned* const h_dec = h_win + (KO ? NT * ko.nr : 0);
  int* const s_members = reinterpret_cast<int*>(h_dec + (KO ? 2 * ko.K : 0));
  int* const s_gbeg = s_members + NT;
  int* const s_gcnt = s_gbeg + NT;
  // Tournament: the keys are not stored (philox_word reads one when it is needed), so the s_key words hold bytes:
  // k_q [NT][thread] = the slot ranked p-th in its group at member index gbeg + p, k_best [bc][thread] = the slot of
  // BEST j, k_gtab = per CTA, first member index [ng] and size [ng] of each group id.  The per-tie winner / loser bytes
  // go into the thread's OWN s_gf / s_gd words once its ranking and best-placed selection are done (byte b in byte
  // b % 4 of word [b / 4][thread], so a thread that reaches its ties early never touches the words another thread is
  // still ranking), or after the member lists when 2K bytes exceed those 2 T_tab words.  A slot fits 6 bits (T_tab <=
  // 64): bits 6-7 of the winner byte hold how the tie was decided until the histograms are committed.
  uint8_t* const k_q = reinterpret_cast<uint8_t*>(s_key);
  uint8_t* const k_best = k_q + NT * kSimThreads;
  uint8_t* const k_gtab = k_best + (KO ? ko.bc : 0) * kSimThreads;
  uint8_t* const k_wl = KO && !ko.wl_overlay ? reinterpret_cast<uint8_t*>(s_gcnt + NT) : reinterpret_cast<uint8_t*>(s_gf);
  __shared__ unsigned s_invalid;
  __shared__ int s_groups_fit;
#define ACC(arr, t) arr[(t) * kSimThreads + tid]
#define BYTE(arr, k) arr[(k) * kSimThreads + tid]
#define WL(b) k_wl[(((b) >> 2) * kSimThreads + tid) * 4 + ((b) & 3)]

  if (tid == 0) {
    s_invalid = 0;
    s_groups_fit = 1;
  }
  for (int k = tid; k < NT * sp.P; k += kSimThreads) h_pos[k] = 0;
  if (sp.points_in_smem)
    for (int k = tid; k < NT * sp.B; k += kSimThreads) h_pts[k] = 0;
  if constexpr (KO) {
    for (int k = tid; k < 2 * (NT * ko.nr + ko.K); k += kSimThreads) h_reach[k] = 0;  // h_win, h_dec follow
    for (int g = tid; g < ko.ng; g += kSimThreads) {
      int beg = 0, cnt = 0;
      for (int u = 0; u < NT; u++) {
        const int gu = sp.group ? sp.group[u] : 0;
        beg += gu < g;
        cnt += gu == g;
      }
      k_gtab[g] = (uint8_t)beg;
      k_gtab[ko.ng + g] = (uint8_t)cnt;
    }
  }
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
    if constexpr (!KO) {
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
    } else {
      for (int t = 0; t < NT; t++) {
        ACC(s_gd, t) = ACC(s_gf, t) - ACC(s_gd, t);
        const int gained = ACC(s_pts, t) - sp.start_pts[t];
        ok = ok && gained >= 0 && gained < sp.B;
      }
      ok = ok && s_groups_fit;
      const unsigned wkey = 2u * (unsigned)gp.F;  // word of slot 0's tie-break key
      // a slot u ranked ahead of slot t (u != t): points, goal difference, goals for, the key, then the lower slot
      auto ahead = [&](int u, int t) -> bool {
        const int pu = ACC(s_pts, u), pt = ACC(s_pts, t);
        if (pu != pt) return pu > pt;
        const int du = ACC(s_gd, u), dt = ACC(s_gd, t);
        if (du != dt) return du > dt;
        const int fu = ACC(s_gf, u), ft = ACC(s_gf, t);
        if (fu != ft) return fu > ft;
        const uint32_t ku = philox_word(sp.seed, n, wkey + u), kt = philox_word(sp.seed, n, wkey + t);
        return ku != kt ? ku > kt : u < t;
      };
      if (ok) {
        // ranking within the groups: k_q[gbeg + position] = slot
        for (int t = 0; t < NT; t++) {
          const int g0 = s_gbeg[t], gc = s_gcnt[t];
          int pos = 0;
          for (int m = 0; m < gc; m++) {
            const int u = s_members[g0 + m];
            if (u != t) pos += ahead(u, t);
          }
          BYTE(k_q, g0 + pos) = (uint8_t)t;
        }
        // best-placed qualifiers: the slot at best_position of every group, ranked across groups
        if (ko.bc > 0) {
          unsigned mask = 0;
          int nq = 0;
          for (int g = 0; g < ko.ng; g++) {
            if (k_gtab[ko.ng + g] <= ko.bp) continue;
            const int t = BYTE(k_q, k_gtab[g] + ko.bp);
            int rk = 0;
            for (int h = 0; h < ko.ng; h++)
              if (h != g && k_gtab[ko.ng + h] > ko.bp) rk += ahead(BYTE(k_q, k_gtab[h] + ko.bp), t);
            if (rk < ko.bc) {
              nq++;
              if (ko.alloc) mask |= 1u << g;
              else BYTE(k_best, rk) = (uint8_t)t;
            }
          }
          ok = nq == ko.bc;
          if (ok && ko.alloc) {
            const uint8_t* const arow = ko.alloc + (size_t)mask * ko.bc;
            for (int j = 0; j < ko.bc; j++) {
              const int g = arow[j];
              if (g < ko.ng && ((mask >> g) & 1u)) BYTE(k_best, j) = BYTE(k_q, k_gtab[g] + ko.bp);
              else ok = false;  // an allocation row of 0xFF
            }
          }
        }
      }
      // the ties in play order; words 2F + T_tab + 3k, + 1 (the first or only match) and + 2 (the decider) of tie k,
      // and the Philox block E/4 + k (leg 2, extra time) of a tie of format 1 or 2
      skipahead((unsigned long long)NT, &rng);
      uint8_t* const ent = ko.entrants ? ko.entrants + (size_t)i * ko.K * 2 : nullptr;
      uint8_t* const ksc = ko.scores ? ko.scores + (size_t)i * ko.K * 2 : nullptr;
      uint8_t* const kwn = ko.winners ? ko.winners + (size_t)i * ko.K : nullptr;
      uint8_t* const kex = ko.extra ? ko.extra + (size_t)i * ko.K * 4 : nullptr;
#pragma unroll 1
      for (int k = 0; k < ko.K && ok; k++) {
        int e[2];
#pragma unroll
        for (int side = 0; side < 2; side++) {
          const int a0 = ko.arg0[side][k];
          switch (ko.kind[side][k]) {
            case BPLX_ENTRANT_SLOT: e[side] = a0; break;
            case BPLX_ENTRANT_GROUP_POS: {
              const int p = ko.arg1[side][k];
              ok = ok && p < k_gtab[ko.ng + a0];
              e[side] = ok ? BYTE(k_q, k_gtab[a0] + p) : 0;
              break;
            }
            case BPLX_ENTRANT_BEST: e[side] = BYTE(k_best, a0); break;
            case BPLX_ENTRANT_WINNER: e[side] = WL(2 * a0) & 63; break;
            default: e[side] = WL(2 * a0 + 1); break;
          }
        }
        const float uh = curand_uniform(&rng), ua = curand_uniform(&rng), ud = curand_uniform(&rng);
        if (!ok) break;
        const int hs = e[0], as = e[1];
        const bool neutral = gp.ntab == 3 && ko.neutral[k];
        const FixtureOffsets off = fixture_offsets(L, ko.slot_team[hs], ko.slot_team[as], neutral, wc,
                                                   wc ? ko.slot_conf[hs] : 0, wc ? ko.slot_conf[as] : 0);
        const float2 lam = fixture_rates(row, off, neutral, wc);
        int hg = 0, ag = 0;
        ok = sample_score(lam.x, lam.y, c, uh, ua, sp.G, hg, ag);
        bool home_through = hg > ag;
        int how = 0;  // decided in normal time or on aggregate (0), in extra time (1), by u_d (2)
        const int fmt = ko.format[k];
        if (fmt == BPLX_TIE_ONE_MATCH) {
          if (ok && hg == ag) {  // a drawn tie: the home entrant goes through iff u_d (hw + aw) <= hw
            float hw, aw;
            win_masses(lam.x, lam.y, c, sp.G, hw, aw);
            const float tot = hw + aw;
            ok = tot > 0.0f;
            home_through = ud * tot <= hw;
            how = 2;
          }
          if (kex) *reinterpret_cast<uchar4*>(kex + 4 * k) = make_uchar4(0xFE, 0xFE, 0xFE, 0xFE);
        } else if (ok) {
          // goals of the home entrant A and the away entrant B; extra time at the venue of the last match
          const uint4 xw = philox_block(sp.seed, n, (2u * gp.F + NT + 3u * ko.K + 3u) / 4u + k);
          int tot_a = hg, tot_b = ag, l2a = 0xFE, l2b = 0xFE, eta = 0xFE, etb = 0xFE;
          float2 last = lam;
          const bool legs = fmt == BPLX_TIE_TWO_LEGS;
          if (legs) {  // leg 2: B at home, never at a neutral venue
            const FixtureOffsets off2 = fixture_offsets(L, ko.slot_team[as], ko.slot_team[hs], false, wc,
                                                        wc ? ko.slot_conf[as] : 0, wc ? ko.slot_conf[hs] : 0);
            last = fixture_rates(row, off2, false, wc);
            ok = sample_score(last.x, last.y, c, _curand_uniform(xw.x), _curand_uniform(xw.y), sp.G, l2b, l2a);
            tot_a += l2a;
            tot_b += l2b;
          }
          if (ok && tot_a == tot_b) {
            int eh = 0, ea = 0;
            ok = sample_score(last.x * kExtraTimeFraction, last.y * kExtraTimeFraction, 0.0f, _curand_uniform(xw.z),
                              _curand_uniform(xw.w), sp.G, eh, ea);
            eta = legs ? ea : eh;
            etb = legs ? eh : ea;
            tot_a += eta;
            tot_b += etb;
            how = 1;
          }
          home_through = tot_a > tot_b;
          if (tot_a == tot_b) {  // penalties
            home_through = ud <= 0.5f;
            how = 2;
          }
          if (kex) *reinterpret_cast<uchar4*>(kex + 4 * k) = make_uchar4(l2a, l2b, eta, etb);
        }
        if (!ok) break;
        const int w = home_through ? hs : as;
        WL(2 * k) = (uint8_t)(w | how << 6);
        WL(2 * k + 1) = (uint8_t)(home_through ? as : hs);
        if (ent) *reinterpret_cast<uchar2*>(ent + 2 * k) = make_uchar2((unsigned char)hs, (unsigned char)as);
        if (ksc) *reinterpret_cast<uchar2*>(ksc + 2 * k) = make_uchar2((unsigned char)hg, (unsigned char)ag);
        if (kwn) kwn[k] = (uint8_t)w;
      }
      uint8_t* const prow = sp.positions ? sp.positions + (size_t)i * NT : nullptr;
      if (!ok) {
        atomicAdd(&s_invalid, 1u);
        if (prow)
          for (int t = 0; t < NT; t++) prow[t] = 0xFF;
        for (int k = 0; k < ko.K; k++) {
          if (ent) *reinterpret_cast<uchar2*>(ent + 2 * k) = make_uchar2(0xFF, 0xFF);
          if (ksc) *reinterpret_cast<uchar2*>(ksc + 2 * k) = make_uchar2(0xFF, 0xFF);
          if (kwn) kwn[k] = 0xFF;
          if (kex) *reinterpret_cast<uchar4*>(kex + 4 * k) = make_uchar4(0xFF, 0xFF, 0xFF, 0xFF);
        }
      } else {
        for (int m = 0; m < NT; m++) {
          const int t = BYTE(k_q, m), pos = m - s_gbeg[t];
          if (prow) prow[t] = (uint8_t)pos;
          atomicAdd(&h_pos[t * sp.P + pos], 1u);
          const int gained = ACC(s_pts, t) - sp.start_pts[t];
          if (sp.points_in_smem) atomicAdd(&h_pts[t * sp.B + gained], 1u);
          else atomicAdd(&sp.pts_counts[(size_t)t * sp.B + gained], 1ull);
        }
        for (int k = 0; k < ko.K; k++) {
          const int r = ko.round[k], wb = WL(2 * k), w = wb & 63, l = WL(2 * k + 1);
          atomicAdd(&h_reach[w * ko.nr + r], 1u);
          atomicAdd(&h_reach[l * ko.nr + r], 1u);
          atomicAdd(&h_win[w * ko.nr + r], 1u);
          if (wb >> 6) atomicAdd(&h_dec[2 * k + (wb >> 6) - 1], 1u);
        }
      }
    }
  }
#undef ACC
#undef BYTE
#undef WL
  __syncthreads();
  for (int k = tid; k < NT * sp.P; k += kSimThreads)
    if (h_pos[k]) atomicAdd(&sp.pos_counts[k], (unsigned long long)h_pos[k]);
  if (sp.points_in_smem)
    for (int k = tid; k < NT * sp.B; k += kSimThreads)
      if (h_pts[k]) atomicAdd(&sp.pts_counts[k], (unsigned long long)h_pts[k]);
  if constexpr (KO) {
    for (int k = tid; k < NT * ko.nr; k += kSimThreads) {
      if (h_reach[k]) atomicAdd(&ko.reach[k], (unsigned long long)h_reach[k]);
      if (h_win[k]) atomicAdd(&ko.win[k], (unsigned long long)h_win[k]);
    }
    if (ko.decided) {
      const unsigned valid = (unsigned)min(kSimThreads, sp.N - (int)blockIdx.x * kSimThreads) - s_invalid;
      for (int k = tid; k < ko.K; k += kSimThreads) {
        const unsigned et = h_dec[2 * k], ud = h_dec[2 * k + 1], nt = valid - et - ud;
        if (nt) atomicAdd(&ko.decided[3 * k], (unsigned long long)nt);
        if (et) atomicAdd(&ko.decided[3 * k + 1], (unsigned long long)et);
        if (ud) atomicAdd(&ko.decided[3 * k + 2], (unsigned long long)ud);
      }
    }
  }
  if (tid == 0 && s_invalid) atomicAdd(sp.invalid, (unsigned long long)s_invalid);
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
  const bool ko = sp.ko.K > 0;
  const size_t smem = simulate_smem_bytes(&sp);
  BPLX_REQUIRE(smem <= (size_t)kSimSmemMax, BPLX_E_UNSUPPORTED,
               "simulate: %zu bytes of shared memory per CTA needed (max %d)", smem, kSimSmemMax);
  // the dynamic shared-memory limit is an attribute of each instantiation
  static size_t smem_set[2] = {48 * 1024, 48 * 1024};
  if (smem > smem_set[ko]) {
    BPLX_CUDA(cudaFuncSetAttribute(ko ? simulate_kernel<true> : simulate_kernel<false>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set[ko] = smem;
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
  const unsigned grid = (unsigned)((sp.N + kSimThreads - 1) / kSimThreads);
  if (ko) simulate_kernel<true><<<grid, kSimThreads, smem, stream>>>(sp);
  else simulate_kernel<false><<<grid, kSimThreads, smem, stream>>>(sp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
