// simulate.h -- season / group-stage simulation per posterior draw (see simulate.cu).
#pragma once
#include "score_grid.h"

namespace bplx {

constexpr int kSimThreads = 128;    // simulations per CTA (one thread per simulation)
constexpr int kSimMaxTeams = 64;    // BPLX_SIM_MAX_TEAMS
constexpr int kSimSmemMax = 227 * 1024;
constexpr int kKoMaxTies = 64;      // BPLX_KO_MAX_TIES
constexpr int kKoMaxRounds = 16;    // BPLX_KO_MAX_ROUNDS
constexpr int kKoMaxBest = 16;      // BPLX_KO_MAX_BEST

// the knockout bracket of a tournament simulation (K = 0: group stage only, the bplx_simulate_table kernel).  The per-tie
// arrays travel by value in the kernel parameters (read warp-uniformly from the constant bank).
struct KoParams {
  int K, nr, ng, bp, bc;          // ties, rounds, groups, best_position, best_count (0: no best-placed pool)
  int wl_overlay;                 // the per-tie winner / loser bytes live in the dead s_gf / s_gd accumulators
  const uint8_t* alloc;           // device [2^ng][bc] allocation table or NULL (in the workspace)
  unsigned long long *reach, *win;  // [NT][nr]
  unsigned long long* decided;    // [K][3] or NULL
  uint8_t *entrants, *scores, *winners, *extra;  // [N][K][2], [N][K][2], [N][K], [N][K][4] or NULL
  uint8_t kind[2][kKoMaxTies];    // (home, away) entrant kinds: BPLX_ENTRANT_*
  uint8_t arg0[2][kKoMaxTies];    // slot / group / j / earlier tie
  uint8_t arg1[2][kKoMaxTies];    // position of GROUP_POS
  uint8_t round[kKoMaxTies];
  uint8_t neutral[kKoMaxTies];
  uint8_t format[kKoMaxTies];     // BPLX_TIE_*
  uint16_t slot_team[kSimMaxTeams];
  uint8_t slot_conf[kSimMaxTeams];
};

constexpr int kMaxPairings = 16;      // BPLX_MAX_PAIRINGS
constexpr int kPairingMaxPool = 64;   // BPLX_PAIRING_MAX_POOL
constexpr int kPairingMaxPot = 16;    // BPLX_PAIRING_MAX_POT

// the pairings drawn by lot of a tournament (num = 0: none, the kernels without pairings).  A tie that takes a pair
// has entrant kind SLOT 0 in KoParams; the pairing writes its drawn entrants into the tie's winner / loser bytes, which
// are free until the tie is played.
struct PairParams {
  int num;
  int buf_off;                    // byte offset in dynamic shared memory of the per-thread pool bytes [nbuf][thread]
  int nbuf;                       // bytes per thread: the largest open pool, 64 for a seeded pairing
  unsigned P0;                    // Philox counter of pairing 0's first block: E/4 + K
  unsigned long long* counts;     // [num][NT][NT] or NULL
  uint8_t mode[kMaxPairings];     // BPLX_PAIRING_*
  uint8_t protect[kMaxPairings];  // BPLX_PROTECT_* bits
  uint8_t host_b[kMaxPairings];   // seeded: the pot-B entrant is at home
  uint8_t size[kMaxPairings];     // n_d
  uint8_t made_at[kKoMaxTies];    // the pairing made when tie k is reached, or 0xFF
  uint8_t of_tie[kKoMaxTies];     // the pairing tie k takes a pair of, or 0xFF
  uint8_t tie[kMaxPairings][kPairingMaxPool / 2];  // the tie that takes pair i
  uint8_t kind[kMaxPairings][kPairingMaxPool], arg0[kMaxPairings][kPairingMaxPool], arg1[kMaxPairings][kPairingMaxPool];
  uint8_t dst[kMaxPairings][kPairingMaxPool];  // pool byte of entry j: j (open); 16 pot + index in the pot (seeded)
  uint8_t assoc[kSimMaxTeams];    // slot associations, 0xFF = none
};

constexpr int kCondMaxKeys = 64;      // BPLX_SIM_MAX_KEY_FIXTURES
constexpr int kCondMaxEvents = 64;    // BPLX_SIM_MAX_EVENTS

constexpr int kCondTableWords = kSimMaxTeams + kCondMaxEvents + kCondMaxKeys / 2;

// the key fixtures and events of a conditional table simulation (nk = 0: none, the kernels without conditions)
struct CondParams {
  int nk, ne;                     // key fixtures, events
  int tab_off;                    // byte offset in dynamic shared memory of the per-CTA copy of `tables`
  int buf_off;                    // byte offset of the per-warp partial counts [2][7][kSimThreads] (uint32)
  unsigned long long *outcome_counts, *cond_counts;  // [nk][3], [nk][3][ne]
  // the events of each slot [64] (bit e: event e is about the slot), the positions of each event [64] (bit p:
  // position p is in its set), then the key fixtures as int32 [64], strictly increasing
  unsigned long long tables[kCondTableWords];
};

struct SimParams {
  GridParams gp;                  // samples (S = draws of this call), fixtures (F), table layout; gp.table = workspace
  const uint8_t *hslot, *aslot;   // [F] table slots
  const uint8_t* group;           // [NT] or NULL (one group)
  const int32_t *start_pts, *start_gf, *start_ga;  // [NT]
  int NT, P, B;                   // table slots, position bins (largest group), gained-points bins
  int G, R;                       // max_goals, simulations per draw
  int pw, pd;                     // points for a win / a draw
  unsigned long long seed;
  long long first_draw;
  int N;                          // simulations of this call = S * R (< 2^31)
  int points_in_smem;             // the gained-points histogram is kept per CTA in shared memory
  unsigned long long *pos_counts, *pts_counts, *invalid;  // [NT][P], [NT][B], [1]
  uint8_t *positions, *scores;    // [N][NT], [N][F][2] or NULL
  KoParams ko;                    // the tournament kernel only
  // the ranking rule (BPLX_RANK_*); head-to-head only: the played matches and the remaining fixtures by slot pair
  int rule;
  const int2* h2h_played;         // [NT][NT] (points, goals) of slot u against slot v in played matches, or NULL
  int *pair_beg, *pair_fix;       // [NT NT + 1], [F] in the workspace (pair_index_kernel)
  // last, so the other kernels' parameters keep their offsets.  cd shares pr's bytes: the paired tournament kernels
  // never read cd and the conditional table kernels never read pr, and a larger parameter block changed the register
  // allocation of simulate_h2h_kernel<true>.  A table call (ko.K = 0) leaves pr unused.
  union {
    PairParams pr;                // the paired tournament kernels only
    CondParams cd;                // the conditional table kernels only (cd.nk = 0 otherwise)
  };
};
static_assert(sizeof(CondParams) <= sizeof(PairParams), "cd must fit in pr's bytes");

// shared memory per CTA, and whether the points histogram fits in it (sets sp->points_in_smem); with ko.K > 0 that of
// the tournament kernel (sets sp->ko.wl_overlay), with pr.num > 0 that of the paired kernel (sets sp->pr.buf_off), with
// cd.nk > 0 that of the conditional kernel (sets sp->cd.tab_off, sp->cd.buf_off)
size_t simulate_smem_bytes(SimParams* sp);
// ko.K = 0: the group stage alone; ko.K >= 1: the tournament kernel, the same group stage, then the bracket of sp.ko.
// rule = BPLX_RANK_HEAD_TO_HEAD: the head-to-head instantiation, after the pair index is built into pair_beg / pair_fix
int launch_simulate(SimParams& sp, cudaStream_t stream);
// launch_simulate's last step for a table with conditions (cd.nk >= 1, ko.K = 0): simulate_cond_kernel, which lives in
// its own translation unit (simulate_cond.cu) so that the instantiations of simulate.cu keep their instructions
int launch_simulate_cond(const SimParams& sp, unsigned grid, size_t smem, cudaStream_t stream);

}  // namespace bplx
