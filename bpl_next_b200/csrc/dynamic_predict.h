// dynamic_predict.h -- forecast of the dynamic model's gameweeks after the fit (see dynamic_predict.cu).
#pragma once
#include "common.cuh"

namespace bplx {

constexpr int kForecastThreads = 256;  // threads per CTA: (draw, team) pairs, whole draws per CTA
constexpr int kForecastMaxTeams = kForecastThreads;  // one draw's teams fit one CTA

struct ForecastParams {
  const float *attack, *defence;  // [S][T] the walk at the last fitted gameweek G - 1
  // [h][S][T] each: attack, defence, home_attack, away_attack, home_defence, away_defence of gameweeks G .. G + h - 1
  float* out[6];
  int S, T, h;
  int draws_per_cta;
  unsigned long long key;  // seed ^ BPLX_FORECAST_KEY
  long long first_draw;
};

int launch_dynamic_forecast(ForecastParams& fp, cudaStream_t stream);

}  // namespace bplx
