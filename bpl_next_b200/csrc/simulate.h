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
};

// shared memory per CTA, and whether the points histogram fits in it (sets sp->points_in_smem); with ko.K > 0 that of
// the tournament kernel (sets sp->ko.wl_overlay)
size_t simulate_smem_bytes(SimParams* sp);
// ko.K = 0: the group stage alone; ko.K >= 1: the tournament kernel, the same group stage, then the bracket of sp.ko.
// rule = BPLX_RANK_HEAD_TO_HEAD: the head-to-head instantiation, after the pair index is built into pair_beg / pair_fix
int launch_simulate(SimParams& sp, cudaStream_t stream);

}  // namespace bplx
