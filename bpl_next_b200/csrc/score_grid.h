// score_grid.h -- K3: posterior-predictive score grid (see score_grid.cu).
#pragma once
#include "common.cuh"

namespace bplx {

constexpr int kGridThreads = 256;   // fixtures per CTA (one thread per fixture)
constexpr int kGridStageMax = 16;   // posterior samples per TMA stage (fewer when a sample row is large)
constexpr int kGridStages = 2;      // stage buffers
constexpr int kGridStageBytes = 100 * 1024;  // budget of one stage buffer

// float offsets of the per-team tables inside a sample row of the exponential table (see score_grid_tables)
struct RowLayout {
  int P1, Q1, P0, EC, C;
};
__host__ __device__ inline RowLayout row_layout(int T, int Cf, int ntab) {
  RowLayout L;
  L.P1 = 0;
  L.Q1 = 2 * T;
  L.P0 = 4 * T;
  L.EC = 2 * T * ntab;
  L.C = L.EC + 2 * Cf;
  return L;
}

// float offsets, inside a sample row, of the table entries the rates of one fixture read (see score_grid_tables)
struct FixtureOffsets {
  int h, a, eh, ea;
};
__host__ __device__ inline FixtureOffsets fixture_offsets(const RowLayout& L, int home, int away, bool neutral, bool wc,
                                                          int home_conf, int away_conf) {
  FixtureOffsets o;
  o.h = (neutral ? L.P0 : L.P1) + 2 * home;
  o.a = (neutral ? L.P0 : L.Q1) + 2 * away;
  o.eh = wc ? L.EC + 2 * home_conf : 0;
  o.ea = wc ? L.EC + 2 * away_conf : 0;
  return o;
}

// the predict path's rates (lambda_h, lambda_a) of one fixture from one sample row: neutral venues and confederations
// included, no clip
__device__ __forceinline__ float2 fixture_rates(const float* row, const FixtureOffsets& o, bool neutral, bool wc) {
  const float2 rh = *reinterpret_cast<const float2*>(row + o.h);
  const float2 ra = *reinterpret_cast<const float2*>(row + o.a);
  float lh = rh.x * (neutral ? ra.y : ra.x), la = rh.y * (neutral ? ra.x : ra.y);
  if (wc) {
    const float2 eh = *reinterpret_cast<const float2*>(row + o.eh);
    const float2 ea = *reinterpret_cast<const float2*>(row + o.ea);
    lh *= eh.x * ea.y;
    la *= ea.x * eh.y;
  }
  return make_float2(lh, la);
}

struct GridParams {
  int model, S, T, Cf, F, g;
  int nsplit, samples_per_split;
  int ns_stage;    // samples per stage
  int ntab;        // per-team tables in a sample row: 2 (P1, Q1) or 3 (+ P0, models with neutral venues)
  int row_floats;  // floats per sample row of `table` (a multiple of 4: rows are 16-byte aligned for the bulk copies)
  int reuse_tables;  // the table in the workspace is already built for these samples
  float scale;
  // posterior samples, [S, T] row-major (home_advantage of DIXON_COLES: [S])
  const float *attack, *defence, *ha, *aa, *hd, *ad, *conf, *corr;
  const uint16_t *home, *away;
  const uint8_t *hconf, *aconf, *nv;
  float* table;    // [S][row_floats]  exponentials of the per-team log-rate halves (built by the pre-pass)
  float* partial;  // [nsplit][F][g*g]
  float* grid;     // [F][g*g]
  float* outcome;  // [F][3] or NULL
};

// fills ntab / row_floats of `gp` (model, S, T, Cf set) and returns the bytes of the [S][row_floats] exponential table,
// rounded up to 256: what follows the table in a workspace starts there
size_t table_layout(GridParams* gp);
// fills nsplit / samples_per_split / ns_stage / ntab / row_floats of `gp` (S, T, Cf, F, g, model set) and returns the
// workspace bytes (table + partial sums); 0 with *err set when a sample row does not fit a stage buffer
size_t score_grid_plan(GridParams* gp, const char** err);
int launch_score_grid(const GridParams& gp, cudaStream_t stream);
// the pre-pass alone: fills gp.table ([S][row_floats]) from the sample arrays; reads model, S, T, Cf, ntab, row_floats
int launch_score_grid_tables(const GridParams& gp, cudaStream_t stream);

}  // namespace bplx
