// simulate.h -- season / group-stage simulation per posterior draw (see simulate.cu).
#pragma once
#include "score_grid.h"

namespace bplx {

constexpr int kSimThreads = 128;    // simulations per CTA (one thread per simulation)
constexpr int kSimMaxTeams = 64;    // BPLX_SIM_MAX_TEAMS
constexpr int kSimSmemMax = 227 * 1024;

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
};

// fills sp->gp's plan fields (model, S, T, Cf, F set) and returns the workspace bytes (the [S][row_floats] table)
size_t simulate_plan(SimParams* sp);
// shared memory per CTA, and whether the points histogram fits in it (sets sp->points_in_smem)
size_t simulate_smem_bytes(SimParams* sp);
int launch_simulate(SimParams& sp, cudaStream_t stream);

}  // namespace bplx
