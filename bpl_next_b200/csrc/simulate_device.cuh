// simulate_device.cuh -- the device helpers of the simulation kernels (simulate.cu, simulate_cond.cu): the knockout
// win masses, single Philox words, the pairing draw and the head-to-head ranking.
// Include after simulate.h and sample_score.cuh.
#pragma once

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

__device__ __forceinline__ int nibble(unsigned long long x, int i) { return (int)(x >> (4 * i)) & 15; }
__device__ __forceinline__ unsigned long long set_nibble(unsigned long long x, int i, int v) {
  return (x & ~(0xFull << (4 * i))) | ((unsigned long long)v << (4 * i));
}
// the index of the r-th set bit of m (r < popc(m))
__device__ __forceinline__ int nth_bit(unsigned m, int r) {
  for (; r > 0; r--) m &= m - 1;
  return __ffs(m) - 1;
}

}  // namespace

// Pairing d of a simulation, its pool already resolved into the thread's pool bytes (PB(j): byte [j][thread]); the
// drawn entrants of pair i go into the winner / loser bytes of tie pr.tie[d][i], home first.  Word j of the pairing is
// component j mod 4 of Philox block P0 + 16 d + j / 4; an index uniform in [0, m) is (uint64(w) m) >> 32.
// Open: the pool in pool order, swapped in place (p[i] <-> p[i + ((w_i (n - i)) >> 32)] for i < n - 1), pair i =
// (p[2i], p[2i + 1]).  Seeded: pot A's slots at bytes [0, m), pot B's at [16, 16 + m), in pool order; adj[a] (u16
// [a][thread] at byte row 32) = the pot-B entrants a may meet.  One perfect matching of the remaining entrants is kept as
// nibbles (mate_a, mate_b, in registers); a pot-A candidate a for the drawn b is eligible iff it may meet b and either
// is b's mate or an augmenting path joins b's mate to a's mate once a and b are gone: one alternating-path search per
// candidate on bit masks, not a new matching.  Returns false when the seeded pool cannot be fully paired.
__device__ __forceinline__ bool draw_pairing(const PairParams& pr, int d, uint8_t* k_pool, const uint8_t* k_ptab,
                                             uint8_t* k_wl, int tid, unsigned long long seed, unsigned long long n) {
#define PB(j) k_pool[(j) * kSimThreads + tid]
#define WL(b) k_wl[(((b) >> 2) * kSimThreads + tid) * 4 + ((b) & 3)]
  const unsigned blk0 = pr.P0 + 16u * (unsigned)d;
  const int nd = pr.size[d];
  uint4 w4 = make_uint4(0, 0, 0, 0);
  if (pr.mode[d] == BPLX_PAIRING_OPEN) {
#pragma unroll 1
    for (int i = 0; i < nd - 1; i++) {
      if ((i & 3) == 0) w4 = philox_block(seed, n, blk0 + (unsigned)(i >> 2));
      const uint32_t w = (i & 3) == 0 ? w4.x : (i & 3) == 1 ? w4.y : (i & 3) == 2 ? w4.z : w4.w;
      const int j = i + (int)(((unsigned long long)w * (unsigned)(nd - i)) >> 32);
      const uint8_t x = PB(i);
      PB(i) = PB(j);
      PB(j) = x;
    }
#pragma unroll 1
    for (int i = 0; i < nd / 2; i++) {
      const int k = pr.tie[d][i];
      WL(2 * k) = PB(2 * i);
      WL(2 * k + 1) = PB(2 * i + 1);
    }
    return true;
  }
  const int m = nd >> 1, prot = pr.protect[d];
  uint16_t* const adj = reinterpret_cast<uint16_t*>(k_pool + 32 * kSimThreads);
#define ADJ(a) adj[(a) * kSimThreads + tid]
#pragma unroll 1
  for (int a = 0; a < m; a++) {
    const int sa = PB(a), ga = k_ptab[sa], xa = k_ptab[64 + sa];
    unsigned row = 0;
#pragma unroll 1
    for (int b = 0; b < m; b++) {
      const int sb = PB(16 + b);
      const bool clash = ((prot & BPLX_PROTECT_GROUP) && k_ptab[sb] == ga) ||
                         ((prot & BPLX_PROTECT_ASSOCIATION) && xa != 0xFF && k_ptab[64 + sb] == xa);
      row |= (unsigned)!clash << b;
    }
    ADJ(a) = (uint16_t)row;
  }
  unsigned long long mate_a = 0, mate_b = 0, parent = 0;
  // breadth-first over alternating paths from pot-A entrant src inside (ra, rb): the first pot-B entrant of `targets`
  // reached, or -1; nibble b of `parent` = the pot-A entrant b was reached from.  Every other pot-B entrant reached is
  // matched, and its mate is the next pot-A entrant of the path.
  auto search = [&](int src, unsigned ra, unsigned rb, unsigned targets) -> int {
    unsigned frontier = 1u << src, seen = 0;
    while (frontier) {
      unsigned next = 0;
      for (unsigned f = frontier; f; f &= f - 1) {
        const int a = __ffs(f) - 1;
        const unsigned nb = ADJ(a) & rb & ~seen;
        seen |= nb;
        for (unsigned g = nb; g; g &= g - 1) {
          const int b = __ffs(g) - 1;
          parent = set_nibble(parent, b, a);
          if ((targets >> b) & 1u) return b;
          next |= 1u << nibble(mate_b, b);
        }
      }
      frontier = next & ra;
    }
    return -1;
  };
  // flips the path that search(src, ...) found to b
  auto augment = [&](int src, int b) {
    for (;;) {
      const int a = nibble(parent, b), prev = nibble(mate_a, a);
      mate_a = set_nibble(mate_a, a, b);
      mate_b = set_nibble(mate_b, b, a);
      if (a == src) break;
      b = prev;
    }
  };
  const unsigned full = (1u << m) - 1u;
  unsigned free_b = full;
#pragma unroll 1
  for (int a = 0; a < m; a++) {
    const int b = search(a, full, full, free_b);
    if (b < 0) return false;
    augment(a, b);
    free_b &= ~(1u << b);
  }
  unsigned ra = full, rb = full;
#pragma unroll 1
  for (int i = 0; i < m; i++) {
    if ((i & 1) == 0) w4 = philox_block(seed, n, blk0 + (unsigned)(i >> 1));
    const uint32_t wb = i & 1 ? w4.z : w4.x, wa = i & 1 ? w4.w : w4.y;  // w_{2i}, w_{2i+1}
    const int b = nth_bit(rb, (int)(((unsigned long long)wb * (unsigned)__popc(rb)) >> 32));
    const int ab = nibble(mate_b, b);
    const unsigned rb2 = rb & ~(1u << b);
    unsigned elig = 0;
#pragma unroll 1
    for (unsigned f = ra; f; f &= f - 1) {
      const int a = __ffs(f) - 1;
      if (!((ADJ(a) >> b) & 1u)) continue;
      if (a == ab || search(ab, ra & ~(1u << a), rb2, 1u << nibble(mate_a, a)) >= 0) elig |= 1u << a;
    }
    // (never empty: b's mate is eligible)
    const int a = nth_bit(elig, (int)(((unsigned long long)wa * (unsigned)__popc(elig)) >> 32));
    if (a != ab) augment(ab, search(ab, ra & ~(1u << a), rb2, 1u << nibble(mate_a, a)));
    const int sa = PB(a), sb = PB(16 + b), k = pr.tie[d][i];
    WL(2 * k) = (uint8_t)(pr.host_b[d] ? sb : sa);
    WL(2 * k + 1) = (uint8_t)(pr.host_b[d] ? sa : sb);
    ra &= ~(1u << a);
    rb = rb2;
  }
  return true;
#undef PB
#undef WL
#undef ADJ
}

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

}  // namespace bplx
