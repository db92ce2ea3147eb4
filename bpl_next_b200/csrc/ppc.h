// ppc.h -- posterior predictive checks: replicated scores of the observed matches and their statistics (see ppc.cu).
#pragma once
#include "score_grid.h"

namespace bplx {

constexpr int kPpcThreads = 256;          // threads per CTA (one CTA per replicate, threads over match pairs)
constexpr int kPpcSmemMax = 227 * 1024;

struct PpcParams {
  GridParams gp;                  // samples (S = draws of this call), observed matches (F = M), table layout
  int G, B, R;                    // max_goals, score_bins, replicates per draw
  int pw, pd;                     // points for a win / a draw
  unsigned long long seed;
  long long first_draw;
  int N;                          // replicates of this call = S * R (< 2^31)
  int32_t *score_counts, *outcome_counts;           // [N][B][B], [N][3]
  long long *goals, *total_goals_sq;                // [N][2], [N]
  int32_t *team_points, *team_goals_for, *team_goals_against;  // [N][T] each
  uint8_t* scores;                // [N][M][2] or NULL
  unsigned long long* invalid;    // [1]
  // multi-gameweek call (ppc_kernel<true>): gp.table is gameweek-major ([ngw][S][row_floats], gp.S = S) and match m
  // reads the row of gameweek gw[m] of its draw
  const int32_t* gw;              // device [M], each < ngw
  int ngw;
};

// dynamic shared memory of one CTA: the draw's exponential table row(s) and the replicate's accumulators
size_t ppc_smem_bytes(const PpcParams& pp, int rows = 1);
// the exponential table pre-pass (score_grid_tables) into pp.gp.table, then one CTA per replicate
int launch_ppc(const PpcParams& pp, cudaStream_t stream);
// the same over a gameweek-major table of pp.ngw gameweeks: the pre-pass builds all ngw * S rows, each CTA copies its
// draw's row of every gameweek; BPLX_E_UNSUPPORTED when they do not fit kPpcSmemMax
int launch_ppc_gameweeks(const PpcParams& pp, cudaStream_t stream);

}  // namespace bplx
