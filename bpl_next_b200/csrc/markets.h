// markets.h -- per-draw market probabilities and their posterior quantiles (see markets.cu).
#pragma once
#include "score_grid.h"

namespace bplx {

constexpr int kMdThreads = 256;           // fixtures per CTA of the draws kernel (one thread per fixture)
constexpr int kMdStageBytes = 24 * 1024;  // budget of one stage buffer of draw rows
constexpr int kMdStages = 2;
constexpr int kMdChunk = 6;               // market rows per CTA: grid.y = ceil(K / kMdChunk)
constexpr int kMarketMaxRows = 6 + 4 * BPLX_MARKET_MAX_LINES;
constexpr int kMqThreads = 256;           // threads per row of the quantile kernel
constexpr int kMqMaxRanks = 2 * BPLX_QUANTILE_MAX_LEVELS;

// One market row of a draw.  kRowPrefix / kRowSuffix: sum over i >= i0 of p_i X(a + b i), X(k) the prefix sum
// sum_{j <= k} q_j or the suffix sum sum_{j >= k} q_j of the away pmf (0 <= j <= G); kRowDiagonal: sum over i of
// p_i q_i.  Then plus p_i q_j (tau(i, j) - 1) for each low cell (i, j) whose bit 2i + j is set in `corr`.
enum { kRowPrefix = 0, kRowSuffix = 1, kRowDiagonal = 2, kRowHomeRate = 3, kRowAwayRate = 4 };
struct MarketRow {
  int8_t kind, b, i0;
  uint8_t corr;
  int32_t a;
};

struct MarketParams {
  GridParams gp;            // samples, fixtures, table layout, stages and draw splits (gp.g = max_goals + 1)
  int K;                    // rows per fixture
  MarketRow row[kMarketMaxRows];
  float* draws;             // [F K][ld] or NULL
  size_t ld;
  int vec;                  // rows and stages are 16-byte aligned: the matrix is written with 16-byte stores
  double* partial;          // [nsplit][F K][3]  p0, sum (p - p0), sum (p - p0)^2 of each split (p0 its first value)
  double* stats;            // [F K][2]  mean, sd
  int* invalid;             // [1]
};

struct QuantileParams {
  const float* rows;        // [R][ld]
  size_t ld;
  int R, S, nq;
  double level[BPLX_QUANTILE_MAX_LEVELS];
  const double* odds;       // [R] or NULL
  double* quantiles;        // [R][nq]
  long long* exceed;        // [R] or NULL
};

// validates the lines (half-integers in range, counts) and fills mp->row / mp->K; BPLX_E_INVALID with the message set
int market_rows(const bplx_market_lines* lines, int max_goals, MarketParams* mp);
// fills mp->gp's plan fields (model, S, T, Cf, F, g set) and returns the workspace bytes (table + partial sums); 0 with
// *err set when a draw row does not fit a stage buffer or the per-thread sums do not fit shared memory
size_t market_plan(MarketParams* mp, const char** err);
int launch_market_draws(MarketParams& mp, cudaStream_t stream);
int launch_market_quantiles(const QuantileParams& qp, cudaStream_t stream);

}  // namespace bplx
