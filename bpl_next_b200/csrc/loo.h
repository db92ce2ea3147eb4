// loo.h -- pointwise log-likelihood and PSIS-LOO (see loo.cu).
#pragma once
#include "score_grid.h"

namespace bplx {

constexpr int kPwThreads = 256;              // matches per CTA of the pointwise kernel (one thread per match)
constexpr int kPwStageBytes = 24 * 1024;     // budget of one stage buffer
constexpr int kPwStages = 3;                 // stage buffers (72 KB: three CTAs per SM)
constexpr int kPsisThreads = 512;
constexpr int kPsisTailMax = 16384;          // longest tail (Mt draws) the PSIS kernel sorts in shared memory

struct PointwiseParams {
  GridParams gp;            // samples, fixtures (F = M), table layout, stages and sample splits
  const uint8_t *hg, *ag;   // observed goals [M]
  float* ll;                // [M][ld] or NULL
  size_t ld;
  int vec;                  // rows and stages are 16-byte aligned: the matrix is written with 16-byte stores
  double* partial;          // [nsplit][M][4]
  double* stats;            // [M][4]
  // gameweek-segmented call (pointwise_kernel<true>): CTA c takes matches [seg[c].y, seg[c].y + seg[c].z), all of
  // gameweek seg[c].x, whose draws are rows [seg[c].x * S, (seg[c].x + 1) * S) of a gameweek-major table (gp.S = S)
  const int4* seg;
  int nseg;
};

struct PsisParams {
  const float* ll;  // [M][ld]
  size_t ld;
  int M, S;
  int Mt;           // tail length ceil(min(0.2 S, 3 sqrt(S / r_eff)))
  int cap;          // power of two >= Mt: shared-memory slots of the tail sort
  double* elpd;     // [M]
  double* khat;     // [M]
};

// fills pp->gp's plan fields (pp->gp.model, S, T, Cf, F set) and returns the workspace bytes (table + partial stats);
// 0 with *err set when a sample row does not fit a stage buffer
size_t pointwise_plan(PointwiseParams* pp, const char** err);
int launch_pointwise(PointwiseParams& pp, cudaStream_t stream);
// the segmented call: the pre-pass over the ngw * S rows of the gameweek-major table, one CTA per descriptor of pp.seg
int launch_pointwise_segmented(PointwiseParams& pp, int ngw, cudaStream_t stream);

// tail length of PSIS for S draws at relative efficiency r_eff
int psis_tail_length(int S, double r_eff);
int launch_psis(const PsisParams& pp, cudaStream_t stream);

}  // namespace bplx
