/*
 * bplx.h -- C ABI of the B200-native Dixon-Coles hot path for bpl-next.
 *
 * The reference (anguswilliams91/bpl-next) has no FFI: its hot path is the numpyro model callable
 * handed to NUTS (bpl/dixon_coles.py:100, bpl/extended_dixon_coles.py:293,
 * bpl/neutral_dixon_coles.py:330, bpl/neutral_dixon_coles_WC.py:281,
 * bpl/dynamic_dixon_coles.py:279) and the eager predict_* methods (bpl/base.py:74-148).  These
 * entry points are what a jax.ffi / ctypes binding for that path binds (INTEGRATION.md shows both).
 *
 * Conventions
 *   - plain C: pointers + sizes, int return (0 = ok, <0 = bplx_status), no exceptions, no exit();
 *     bplx_last_error() gives a thread-local message for the last failing call on this thread.
 *   - device pointers are caller-owned and must stay valid until the enqueued work completes;
 *     *_fwdbwd and bplx_score_grid are asynchronous: they enqueue on `stream` (a cudaStream_t
 *     passed as void*; NULL = legacy default stream), never synchronise and never allocate.
 *   - the *_host variants take HOST buffers, do the H2D/D2H copies themselves through pinned
 *     staging owned by the handle and return after the results are in the host buffers.
 *   - a bplx_problem is immutable after create and bound to the CUDA device that was current at
 *     create time; calls may come from any host thread (one stream per concurrent caller).
 *   - all floating point is IEEE binary32 (the reference runs JAX with x64 disabled); indices are
 *     the reference's DTYPES (bpl/base.py:16-22): uint16 teams, uint8 goals / conferences / venue.
 */
#ifndef BPLX_H_
#define BPLX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BPLX_VERSION 1

typedef enum {
  BPLX_OK = 0,
  BPLX_E_INVALID = -1,     /* bad argument (null pointer, index out of range, ...) */
  BPLX_E_UNSUPPORTED = -2, /* shape outside what the kernels were built for */
  BPLX_E_CUDA = -3,        /* CUDA runtime error (message has the cudaError string) */
  BPLX_E_NOMEM = -4,
  BPLX_E_WORKSPACE = -5    /* workspace too small */
} bplx_status;

/* which bpl-next class the problem mirrors */
typedef enum {
  BPLX_DIXON_COLES = 0, /* bpl/dixon_coles.py:39-84          D = 5 + 2T            */
  BPLX_EXTENDED = 1,    /* bpl/extended_dixon_coles.py:78-248 D = 7 + 2K + 3T       */
  BPLX_NEUTRAL = 2,     /* bpl/neutral_dixon_coles.py:102-283 D = 13 + 2K + 6T      */
  BPLX_NEUTRAL_WC = 3,  /* bpl/neutral_dixon_coles_WC.py:83-232 D = 13 + 2K + 6T + Cf */
  BPLX_DYNAMIC = 4      /* bpl/dynamic_dixon_coles.py:63-247  D = 10G + 2 + 2K + 7GT */
} bplx_model;

/* memory layout of theta / grad */
typedef enum {
  BPLX_CHAIN_MAJOR = 0, /* theta[c * D + d]   -- what a vmapped jax.ffi call hands over ([C, D]) */
  BPLX_CHAIN_MINOR = 1  /* theta[d * ld + c]  -- native, fully coalesced ([D, ld], ld >= C)      */
} bplx_layout;

#define BPLX_FLAG_DYNAMIC_AS_WRITTEN 1u /* reproduce dynamic_dixon_coles.py:192-218 literally (SURVEY D1) */

/*
 * Static match data = the positional arguments of the reference `_model` after `fit`'s host prep
 * (parse_teams, bpl/_util.py:115-135).  All arrays are HOST arrays of length num_matches unless
 * stated; the library copies what it needs, the caller keeps ownership.
 */
typedef struct {
  int32_t model;            /* bplx_model */
  int32_t num_matches;      /* M */
  int32_t num_teams;        /* T */
  int32_t num_covariates;   /* K (0 = no team_covariates) */
  int32_t num_conferences;  /* Cf (NEUTRAL_WC only, else 0) */
  int32_t num_gameweeks;    /* G (DYNAMIC only, else 0) */
  uint32_t flags;
  const uint16_t* home_team;      /* [M] index into sorted team names */
  const uint16_t* away_team;      /* [M] */
  const uint8_t* home_goals;      /* [M] */
  const uint8_t* away_goals;      /* [M] */
  const uint8_t* neutral_venue;   /* [M] 1 = neutral; NULL = all 0 (required NULL-able for DC/EXT) */
  const uint8_t* home_conf;       /* [M] NEUTRAL_WC, else NULL */
  const uint8_t* away_conf;       /* [M] NEUTRAL_WC, else NULL */
  const int32_t* gameweek;        /* [M] DYNAMIC (0-based, < G), else NULL */
  const float* weights;           /* [M] match weights (time decay x game weights), NULL = unweighted
                                     (the `to_event(1)` branch, extended_dixon_coles.py:216-227) */
  const float* covariates;        /* [T*K] row-major STANDARDISED covariates
                                     (extended_dixon_coles.py:124-127), NULL iff K == 0 */
} bplx_problem_desc;

typedef struct bplx_problem bplx_problem;

/* ---- lifetime ---------------------------------------------------------------------------- */
int bplx_problem_create(const bplx_problem_desc* desc, bplx_problem** out);
void bplx_problem_destroy(bplx_problem* p);

/* number of unconstrained parameters D of the model (numpyro's flattened latent sites) */
int bplx_num_params(const bplx_problem* p);

/*
 * Layout of the flat unconstrained vector, as "name:offset:count:transform;" records
 * (transform in real|exp|sigmoid; names are numpyro's latent site names).  Pointer is owned by
 * the handle.  Replaces numpyro's ravel of the latent-site dict for this path.
 */
const char* bplx_problem_layout(const bplx_problem* p);

/*
 * Plan statistics for benchmarks / DESIGN.md: out[0..7] = matches, phase-1 entries, padded phase-1
 * entries, phase-2 (tau) entries, padded phase-2 entries, shared-memory bytes per CTA, warps per
 * CTA, (team, confederation) pairs.  Returns the number of values written.
 */
int bplx_problem_stats(const bplx_problem* p, long long* out, int n);

/*
 * What each warp of a CTA walks (static models, the plan for one CTA per group of 32 chains): out[w*12 + 0..5] =
 * phase-1 {home-form pieces, away-form pieces, home-form entries, away-form entries, teams, stages}, out[w*12 + 6..11]
 * = phase-2 {pieces, tau = 1 - c X Y entries, tau = 1 + c X entries, tau = 1 + c Y entries, teams, stages} (padded
 * counts).  Returns the number of values written (<= n); 0 for BPLX_DYNAMIC.  For tuning the plan's cost model.
 */
int bplx_problem_warp_stats(const bplx_problem* p, long long* out, int n);

/* ---- log-density + gradient: replaces value_and_grad(potential_fn) per leapfrog ---------- */
/* (numpyro potential_energy of `_model`; the returned lp is the log JOINT density, i.e. MINUS
 * the potential energy, and grad is d lp / d theta.) */
/* Workspace for num_chains chains.  For batches of num_chains x D >= 2^17 elements this includes room for one
 * transposed copy of theta and of the gradient: BPLX_CHAIN_MAJOR calls are then computed in the kernel's native
 * BPLX_CHAIN_MINOR layout (two tiled transposes around the kernel; the kernel alone is 2.2x slower on [chains, D] buffers
 * of configs[2] size).  A smaller workspace (the kernel's own need) is accepted: the call then runs on the buffers as
 * they are. */
size_t bplx_logdensity_workspace_bytes(const bplx_problem* p, int num_chains);

/*
 * Asynchronous on `stream`, capturable in a CUDA graph.  The kernel is launched with programmatic stream
 * serialization: its set-up (parameters, static plan) may overlap the end of the previous kernel of the stream, and
 * everything that reads theta or writes an output waits for that kernel to complete -- stream order is what the caller
 * sees.  Results are a pure function of the inputs (bit-reproducible).  A log-density that overflowed float32 far from
 * the typical set is reported as NaN, never as +inf.  While the call runs, grad doubles as scratch.
 */

int bplx_logdensity_fwdbwd(const bplx_problem* p, int num_chains, int layout, int ld,
                           const float* theta,   /* device, [C, D] or [D, ld] */
                           float* lp,            /* device, [C] */
                           float* grad,          /* device, same layout as theta */
                           float* corr_coef,     /* device, [C] (deterministic site "corr_coef"), may be NULL */
                           void* workspace, size_t workspace_bytes,
                           void* stream);

/*
 * Likelihood-only entry point: what a numpyro `_model` that KEEPS its prior sites hands to `numpyro.factor`
 * (bpl/dixon_coles.py:79-84; it replaces the rates -> Poisson -> tau block, e.g. bpl/neutral_dixon_coles_WC.py:188-232).
 * Input per chain: the CONSTRAINED per-team tables packed as bplx_loglik_layout() says
 *     attack[T] | defence[T] | home_advantage[1 or T]  or  home_attack, away_attack, home_defence, away_defence [T each]
 *     | confederation_strength[Cf] | corr_coef_raw (in (0,1))
 * Output: loglik[C] = sum_m w (Poisson log-pmfs) + sum_m w log tau, corr_coef[C] (the deterministic site), and
 * grad = d loglik / d (every input), same layout as the input -- the cotangent a jax.custom_vjp multiplies through.
 * No priors, no transforms, no Jacobians: those stay numpyro's.  Same launch / workspace rules as
 * bplx_logdensity_fwdbwd (bplx_logdensity_workspace_bytes gives the workspace).  DYNAMIC: BPLX_E_UNSUPPORTED.
 */
int bplx_loglik_num_inputs(const bplx_problem* p);
const char* bplx_loglik_layout(const bplx_problem* p); /* "name:offset:count:real;" records, "unit" for corr_coef_raw */
int bplx_loglik_fwdbwd(const bplx_problem* p, int num_chains, int layout, int ld,
                       const float* tables,  /* device, [C, Dl] or [Dl, ld], Dl = bplx_loglik_num_inputs */
                       float* loglik,        /* device, [C] */
                       float* grad,          /* device, same layout as tables */
                       float* corr_coef,     /* device, [C], may be NULL */
                       void* workspace, size_t workspace_bytes, void* stream);

/* host-buffer variant (chain-major [C, D]); copies in/out inside the call, returns when done.  Page-locked (pinned)
 * arrays are copied by DMA without staging, and lp / corr_coef are then written by the kernel straight into them. */
int bplx_logdensity_fwdbwd_host(bplx_problem* p, int num_chains,
                                const float* theta, float* lp, float* grad, float* corr_coef);

/* ---- posterior-predictive score grid: replaces predict_score_grid_proba/outcome_proba ---- */
/*
 * Posterior sample arrays are [S, T] row-major (the attributes `fit` stores,
 * e.g. neutral_dixon_coles_WC.py:308-334), device pointers; unused ones NULL:
 *   DIXON_COLES : attack, defence, home_advantage [S] (in `home_attack`), corr_coef
 *   EXTENDED    : attack, defence, home_advantage [S,T] (in `home_attack`), corr_coef
 *   NEUTRAL(_WC): attack, defence, home_attack, away_attack, home_defence, away_defence,
 *                 (confederation_strength [S, Cf]), corr_coef
 */
typedef struct {
  int32_t model;           /* bplx_model (DYNAMIC unsupported: reference predict is unusable, SURVEY D3) */
  int32_t num_samples;     /* S (this rank's shard) */
  int32_t num_teams;       /* T */
  int32_t num_conferences; /* Cf */
  const float* attack;
  const float* defence;
  const float* home_attack;
  const float* away_attack;
  const float* home_defence;
  const float* away_defence;
  const float* confederation_strength;
  const float* corr_coef;  /* [S] */
} bplx_samples;

typedef struct {
  int32_t num_fixtures;          /* F */
  const uint16_t* home_team;     /* device [F] */
  const uint16_t* away_team;     /* device [F] */
  const uint8_t* home_conf;      /* device [F] or NULL */
  const uint8_t* away_conf;      /* device [F] or NULL */
  const uint8_t* neutral_venue;  /* device [F] or NULL */
} bplx_fixtures;

size_t bplx_score_grid_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, int max_goals);

/*
 * grid[f, hg, ag] = scale * sum_s tau * Pois(hg; lam_h) * Pois(ag; lam_a), 0 <= hg, ag <= max_goals.
 * scale = 1/S for a single-rank call (the reference's mean over samples); a sample-sharded caller
 * passes 1/S_total and all-reduces (sum) the grids.  outcome (optional, [F, 3] = home_win, draw,
 * away_win) is summed from the SAME rank-local grid, so it is also additive across ranks.
 */
int bplx_score_grid(const bplx_samples* s, const bplx_fixtures* f, int max_goals, float scale,
                    float* grid,     /* device [F, g, g], g = max_goals + 1 */
                    float* outcome,  /* device [F, 3] or NULL */
                    void* workspace, size_t workspace_bytes, void* stream);

/*
 * Same, with flags.  BPLX_GRID_REUSE_TABLES: the workspace still holds the per-(sample, team) exponential tables a previous
 * bplx_score_grid[_ex] call built from THESE samples (same arrays, same shapes, same workspace pointer): skip the table
 * pre-pass.  For callers that cut the fixtures into ranges (e.g. to overlap a cross-GPU all-reduce with the next range).
 */
#define BPLX_GRID_REUSE_TABLES 1u
int bplx_score_grid_ex(const bplx_samples* s, const bplx_fixtures* f, int max_goals, float scale, float* grid,
                       float* outcome, void* workspace, size_t workspace_bytes, void* stream, unsigned flags);

/* host-buffer variant: every pointer in s / f / grid / outcome is a HOST pointer. */
int bplx_score_grid_host(const bplx_samples* s, const bplx_fixtures* f, int max_goals, float scale,
                         float* grid, float* outcome);

/* ---- model comparison: pointwise log-likelihood of observed scores, PSIS-LOO ------------------ */
/*
 * Observed matches: the fixtures (device index arrays, as for the score grid) and their scores.
 */
typedef struct {
  bplx_fixtures fixtures;        /* num_fixtures = M matches */
  const uint8_t* home_goals;     /* device [M] */
  const uint8_t* away_goals;     /* device [M] */
} bplx_observations;

size_t bplx_pointwise_loglik_workspace_bytes(const bplx_samples* s, const bplx_observations* obs);

/*
 * loglik[m * ld + s] = log Pois(yh; lh) + log Pois(ya; la) + log tau(yh, ya; lh, la, corr_coef[s])  (float32)
 * with the rates of the predict path (bplx_score_grid: neutral venues and confederations included, no clip of the
 * rates), tau clamped at 0 so that a match can give -inf, and no match weights: exp(loglik) averaged over s is the
 * probability bplx_score_grid gives the observed cell.  Match-major [M, ld], ld >= S; loglik may be NULL (only the
 * statistics are computed then, with no matrix traffic).
 * stats[m * 4 + 0..3] (float64) = max_s ll, sum_s exp(ll - max), sum_s ll, sum_s ll^2: lppd_m = max + log(sum exp) -
 * log S and var_s ll follow on the host.  Deterministic (sample splits are combined in a fixed order); the statistics do
 * not depend on whether loglik is NULL.  DYNAMIC: BPLX_E_UNSUPPORTED.
 */
int bplx_pointwise_loglik(const bplx_samples* s, const bplx_observations* obs, float* loglik, size_t ld, double* stats,
                          void* workspace, size_t workspace_bytes, void* stream);

/*
 * Pareto-smoothed importance-sampling leave-one-out (Vehtari et al., JMLR 2024; ArviZ's _psislw / _gpdfit) per match
 * over the rows of a match-major log-likelihood matrix loglik [M, ld] (device, float32, S draws per row):
 *   elpd_i[m]   = log sum_s exp(lw[s] + ll[s])  with lw the smoothed, normalised log-weights of the ratios -ll
 *   pareto_k[m] = the fitted shape k-hat; +inf when the tail has <= 4 draws
 * Tail length Mt = ceil(min(0.2 S, 3 sqrt(S / r_eff))); Mt <= BPLX_PSIS_MAX_TAIL (16384, the shared-memory sort of one
 * CTA), else BPLX_E_UNSUPPORTED.  S itself is not limited by shared memory.  A row with a non-finite entry gives
 * elpd_i = NaN and pareto_k = +inf.  Outputs do not depend on how tied draws are ordered.  The current kernel needs no
 * workspace: NULL, 0 is accepted.
 */
#define BPLX_PSIS_MAX_TAIL 16384
int bplx_psis_loo(const float* loglik, int num_matches, int num_samples, size_t ld, double r_eff, double* elpd_i,
                  double* pareto_k, void* workspace, size_t workspace_bytes, void* stream);

/* ---- season / group-stage simulation: finishing positions and points per posterior draw ------------------------ */
/*
 * A table of T_tab slots (T_tab <= BPLX_SIM_MAX_TEAMS), their starting points / goals for / goals against, an optional
 * group id per slot, and F remaining fixtures: `fixtures` gives the model team indices, neutral-venue flags and
 * confederations the predict path needs, home_slot / away_slot (device uint8 [F]) the table slots that play them.
 *
 * Simulation n = (first_draw + s) * R + r (R = sims_per_draw) uses draw s of `samples`.  Its random numbers are the
 * outputs of curand_init(seed, n, 0) followed by curand() (Philox4_32_10): words 2f and 2f+1 become u_h and u_a of
 * fixture f through curand_uniform (in (0, 1]), word 2F + t is the tie-break key of slot t.  Every word has a fixed
 * address, so a rounding difference in one fixture cannot shift the random numbers of any other fixture.
 *
 * Fixture f in draw s: lambda_h, lambda_a are the predict path's rates (bplx_score_grid: neutral venues and confederations
 * included, Extended's clip not applied); G = max_goals (1..63);
 *   w(i, j) = tau+(i, j) Pois(i; lambda_h) Pois(j; lambda_a),  0 <= i, j <= G,
 * tau+ = tau clamped at 0 on the four low-score cells and 1 elsewhere; Z = sum w, m(i) = sum_j w(i, j).  Home goals are
 * the smallest i with sum_{i' <= i} m(i') >= u_h Z, away goals the smallest j with sum_{j' <= j} w(i, j') >= u_a m(i);
 * when rounding leaves a target unmet, the last index with positive mass.  A cell of zero probability is never returned.
 * Per draw this is the draw's own grid normalised by its sum; averaged over draws it converges to bplx_score_grid.
 *
 * Table: points_win for a win, points_draw for a draw (0 <= points_draw <= points_win, points_win >= 1); goal
 * difference and goals for accumulate on top of the start.  Teams are ranked WITHIN THEIR GROUP by points, then goal
 * difference, then goals for, then the tie-break key, all descending; if even the keys are equal the lower slot ranks
 * first.  Position k (0-based) of slot t = the number of teams of its group ranked ahead of t.  That is ranking rule
 * BPLX_RANK_GOAL_DIFF; bplx_simulate_table_ex can rank by BPLX_RANK_HEAD_TO_HEAD instead (below).  Fair-play rules are
 * not modelled: ties left after goals for are decided by lot (the tie-break key).
 *
 * Outputs (device; integer counts, so they are the same bits whatever order the atomics run in; overwritten):
 *   position_counts [T_tab, P]  P = num_positions, the largest group size
 *   points_counts   [T_tab, B]  points GAINED in the remaining fixtures, B = num_points_bins
 *                               = points_win * max_t(remaining fixtures of t) + 1
 *   invalid [1]                 simulations in which some fixture had a non-finite rate, a normaliser that is not
 *                               positive and finite, or a slot >= T_tab (and simulations whose group is larger than P
 *                               or whose gained points do not fit B: the bins are never overrun).  They are left out of
 *                               the histograms; their positions row is 0xFF and the offending fixture's scores 0xFF.
 *   positions [N, T_tab] uint8, scores [N, F, 2] uint8 (home, away): optional, NULL to skip; N = num_samples * R, row
 *                               (s * R + r) of this call.
 * Draw ranges: calls on draws [0, k) and [k, S) (samples cut to the range, first_draw = 0 and k) give counts that sum to
 * the single call's counts and raw rows that concatenate to its rows.  The workspace holds the [S, row] exponential
 * table of bplx_score_grid's pre-pass.  DYNAMIC: BPLX_E_UNSUPPORTED; T_tab > 64 or N >= 2^31 in one call: BPLX_E_UNSUPPORTED;
 * G outside [1, 63], R < 1 or bad point values: BPLX_E_INVALID.
 */
#define BPLX_SIM_MAX_TEAMS 64
typedef struct {
  int32_t num_slots;              /* T_tab */
  int32_t num_positions;          /* P: the largest group size */
  int32_t num_points_bins;        /* B */
  int32_t points_win;
  int32_t points_draw;
  const uint8_t* group;           /* device [T_tab] group id per slot, or NULL: one group */
  const int32_t* start_points;    /* device [T_tab] */
  const int32_t* start_goals_for;
  const int32_t* start_goals_against;
} bplx_table;

size_t bplx_simulate_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, const bplx_table* t);
int bplx_simulate_table(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot, const uint8_t* away_slot,
                        const bplx_table* t, int max_goals, int sims_per_draw, unsigned long long seed,
                        long long first_draw, unsigned long long* position_counts, unsigned long long* points_counts,
                        uint8_t* positions, uint8_t* scores, unsigned long long* invalid, void* workspace,
                        size_t workspace_bytes, void* stream);

/* ---- tournament simulation: a knockout bracket after the group stage, one posterior draw per tournament --------- */
/*
 * Group stage: exactly bplx_simulate_table's definition (same simulation index n, same Philox words 2f, 2f+1 and
 * 2F + t, same ranking); with the same seed its outputs are bit-identical to a bplx_simulate_table call, except that a
 * simulation made invalid by its bracket is left out here.  F = 0 is allowed (a cup whose draw is already made).
 *
 * Bracket: K ties in play order.  Each tie has a home and an away entrant, a round id and (neutral models) a
 * neutral-venue flag; for DIXON_COLES and EXTENDED the home entrant is at home.  An entrant is
 *   BPLX_ENTRANT_SLOT t            a fixed table slot (a team already through)
 *   BPLX_ENTRANT_GROUP_POS (g, p)  the slot ranked p (0-based) in group g
 *   BPLX_ENTRANT_BEST j            the j-th best-placed qualifier (below)
 *   BPLX_ENTRANT_WINNER k'         the winner of the earlier tie k' < k
 *   BPLX_ENTRANT_LOSER k'          its loser (third-place matches)
 * Best-placed qualifiers: one pool, the slots at position best_position of every group, ranked across groups by
 * points, goal difference, goals for, then the slot tie-break key (word 2F + t), then the lower slot; the first
 * best_count qualify.  Without an allocation table BEST j is the j-th best; with one (dense [2^num_groups][best_count]
 * group ids, indexed by the bit set of the groups whose team qualified: the form of FIFA's and UEFA's third-place
 * tables) BEST j is the position-best_position slot of group alloc[mask][j].  This cross-group ranking is the same
 * under either group ranking rule (bplx_ranking: teams of different groups have no head-to-head).  Fair play and
 * rankings are not modelled: ties left after goals for are decided by lot.
 * A tie is played like a group fixture, from the draw's own clamped, truncated grid, with the rates of its entrants'
 * model teams (slot_team) and, for NEUTRAL_WC, their confederations (slot_conf).  Words 2F + T_tab + 3k and + 1 sample
 * its score, word + 2 is the decider u_d (curand_uniform); every word has a fixed address, used or not.  A drawn tie goes
 * to the home entrant iff u_d (hw_s + aw_s) <= hw_s, hw_s = sum_{i > j} w(i, j) and aw_s = sum_{i < j} w(i, j) the
 * draw's own win masses on the same grid: P(home advances | draw s) = hw_s / (hw_s + aw_s), the per-draw form of the
 * knockout renormalisation of predict_outcome_proba(knockout=True), which renormalises AFTER averaging over the draws.
 * That is tie format BPLX_TIE_ONE_MATCH; bplx_simulate_tournament_ex gives each tie a format byte:
 *   0 BPLX_TIE_ONE_MATCH     one match; a draw is decided by u_d (hw_s + aw_s) <= hw_s (above)
 *   1 BPLX_TIE_ONE_MATCH_ET  one match; drawn: extra time; still level: penalties
 *   2 BPLX_TIE_TWO_LEGS      two legs; level on aggregate: extra time in leg 2; still level: penalties
 * Legs: the home entrant A hosts leg 1, the away entrant B hosts leg 2 with the venues swapped (neutral_venue = 0 in
 * both legs; NEUTRAL_WC: A's and B's confederations swap sides).  Each leg is a 90-minute match sampled like a group
 * fixture (tau+ from the draw's own clamped, truncated grid).  Aggregate A = h1 + a2, B = a1 + h2; the higher goes
 * through (no away-goals rule).  Extra time: at the venue of the last match (format 1: the tie's neutral flag
 * included), the draw's rates times BPLX_EXTRA_TIME_FRACTION = 1/3 (30 of 90 minutes at the model's constant rates),
 * no tau correction (tau is a 90-minute low-score term): independent Poissons truncated at G.  Penalties: A goes
 * through iff u_d <= 1/2 (the model knows nothing of shoot-outs).  Neither constant is a parameter.
 * Words: tie k keeps words 2F + T_tab + 3k, + 1 ((u_h, u_a) of its first or only match) and + 2 (u_d).  With
 * E = 4 ceil((2F + T_tab + 3K) / 4), tie k owns words E + 4k .. E + 4k + 3: leg 2 (u_h, u_a), then extra time (u_h,
 * u_a), i.e. the Philox4x32_10 block of counter E/4 + k.  Every word has a fixed address, used or not, so a bracket of
 * format-0 ties reads exactly bplx_simulate_tournament's words and gives its outputs bit for bit.
 *
 * Invalid simulations (bplx_simulate_table's, and a tie with a non-finite rate or a bad normaliser in any of its
 * matches or its extra time, hw + aw not positive on a drawn format-0 tie, a GROUP_POS beyond its group, fewer than
 * best_count groups with a slot at best_position, or an allocation entry of 0xFF) are counted in `invalid` and left out
 * of every histogram; their positions, ko_entrants, ko_scores, ko_winners and ko_extra rows are 0xFF.
 *
 * Outputs (device; integer counts, additive over draw ranges; overwritten): position_counts, points_counts and invalid
 * as bplx_simulate_table; reach_counts [T_tab, num_rounds]: ties of round r the slot played; win_counts [T_tab,
 * num_rounds]: ties of round r it won (the winner of the last tie is the champion).  Optional raw rows (NULL to skip):
 * positions [N, T_tab], scores [N, F, 2], ko_entrants [N, K, 2] (slots), ko_scores [N, K, 2] (the first or only
 * match, home and away), ko_winners [N, K].  A two-legged tie counts once in its round's reach / win counts.
 * bplx_simulate_tournament_ex adds (NULL to skip): decided_counts [K, 3] (additive): how tie k was settled, in normal
 * time or on aggregate / in extra time / by u_d (penalties, or the lot of format 0); ko_extra [N, K, 4] uint8: leg-2
 * goals of (A, B), then extra-time goals of (A, B), in entrant order, 0xFE for a part not played.
 * Limits: K <= 64 ties, <= 16 rounds, best_count <= 16, num_groups <= 16 with an allocation table; T_tab <= 64 and
 * N < 2^31 per call as bplx_simulate_table; DYNAMIC: BPLX_E_UNSUPPORTED; a format byte above 2, or format 2 on a tie
 * with neutral_venue = 1: BPLX_E_INVALID.
 *
 * The bracket's arrays are HOST arrays: the call validates them (entrants reference earlier ties only, groups and
 * positions in range, BEST j < best_count, allocation entries are 0xFF or distinct groups of their mask) and passes
 * them to the kernel; the allocation table is copied into the workspace (cudaMemcpyAsync from the caller's array, so a
 * pageable array makes the call wait for the stream).
 */
#define BPLX_KO_MAX_TIES 64
#define BPLX_KO_MAX_ROUNDS 16
#define BPLX_KO_MAX_BEST 16
#define BPLX_KO_MAX_ALLOC_GROUPS 16
#define BPLX_ENTRANT_SLOT 0
#define BPLX_ENTRANT_GROUP_POS 1
#define BPLX_ENTRANT_BEST 2
#define BPLX_ENTRANT_WINNER 3
#define BPLX_ENTRANT_LOSER 4
#define BPLX_TIE_ONE_MATCH 0
#define BPLX_TIE_ONE_MATCH_ET 1
#define BPLX_TIE_TWO_LEGS 2
#define BPLX_EXTRA_TIME_FRACTION (1.0 / 3.0)
typedef struct {
  int32_t num_ties;               /* K, 1..64 */
  int32_t num_rounds;             /* 1..16 */
  int32_t num_groups;             /* group ids 0 .. num_groups-1 that GROUP_POS and the pool refer to (<= T_tab) */
  int32_t best_position;          /* position of the best-placed pool (0-based) */
  int32_t best_count;             /* 0..16 qualifiers from the pool (0: no pool) */
  const uint8_t* kind;            /* host [K, 2] (home, away) BPLX_ENTRANT_* */
  const uint8_t* arg0;            /* host [K, 2] slot / group / j / earlier tie */
  const uint8_t* arg1;            /* host [K, 2] position of GROUP_POS, else ignored */
  const uint8_t* round;           /* host [K] round id < num_rounds */
  const uint8_t* neutral_venue;   /* host [K] 1 = neutral, or NULL (all 0) */
  const uint16_t* slot_team;      /* host [T_tab] model team of each table slot */
  const uint8_t* slot_conf;       /* host [T_tab] confederation of each slot (NEUTRAL_WC), else NULL */
  const uint8_t* best_alloc;      /* host [2^num_groups, best_count] group ids or 0xFF, or NULL */
} bplx_bracket;

size_t bplx_simulate_tournament_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, const bplx_table* t,
                                                const bplx_bracket* b);
int bplx_simulate_tournament(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                             const uint8_t* away_slot, const bplx_table* t, const bplx_bracket* b, int max_goals,
                             int sims_per_draw, unsigned long long seed, long long first_draw,
                             unsigned long long* position_counts, unsigned long long* points_counts,
                             unsigned long long* reach_counts, unsigned long long* win_counts, uint8_t* positions,
                             uint8_t* scores, uint8_t* ko_entrants, uint8_t* ko_scores, uint8_t* ko_winners,
                             unsigned long long* invalid, void* workspace, size_t workspace_bytes, void* stream);
/* bplx_simulate_tournament with a format per tie: tie_format is a HOST [K] array of BPLX_TIE_* (NULL: all
 * BPLX_TIE_ONE_MATCH); decided_counts [K, 3] and ko_extra [N, K, 4] as above, or NULL.  bplx_simulate_tournament is
 * this call with the three set to NULL; bplx_simulate_tournament_workspace_bytes serves both. */
int bplx_simulate_tournament_ex(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                                const uint8_t* away_slot, const bplx_table* t, const bplx_bracket* b,
                                const uint8_t* tie_format, int max_goals, int sims_per_draw, unsigned long long seed,
                                long long first_draw, unsigned long long* position_counts,
                                unsigned long long* points_counts, unsigned long long* reach_counts,
                                unsigned long long* win_counts, unsigned long long* decided_counts, uint8_t* positions,
                                uint8_t* scores, uint8_t* ko_entrants, uint8_t* ko_scores, uint8_t* ko_winners,
                                uint8_t* ko_extra, unsigned long long* invalid, void* workspace,
                                size_t workspace_bytes, void* stream);

/* ---- ranking rules: head-to-head ------------------------------------------------------------------------------ */
/*
 * The calls above rank a group by BPLX_RANK_GOAL_DIFF: points, goal difference, goals for, then lot.  The _ex / _ranked
 * calls below take a bplx_ranking; NULL, or rule BPLX_RANK_GOAL_DIFF, gives the calls above bit for bit.  Under
 * BPLX_RANK_HEAD_TO_HEAD the teams of each group are ranked as follows:
 *   1. Points.
 *   2. Head-to-head among a level set.  For a set S of two or more teams level on points, each team's points, goal
 *      difference and goals for are computed over the matches between teams of S only: the played matches (played_h2h)
 *      and this simulation's simulated fixtures.  S is ordered by (head-to-head points, head-to-head goal difference,
 *      head-to-head goals for), all descending.
 *   3. Reapply to what is still level.  If step 2 splits S, any part of two or more teams still level on all three
 *      values goes through step 2 again, with S being that part: only the matches among that part count.
 *   4. Fall back when nobody separates.  A set in which step 2 separates nobody (its teams have not met, say) is
 *      ordered by overall goal difference, overall goals for, the tie-break key (word 2F + t), then the lower slot.
 * Position k is the team's index in this order.  This is the structure of UEFA's group-stage rule (criteria a-f); fair
 * play, coefficient rankings and a shoot-out between two level teams who meet in the last round are replaced by lot.
 * Best-placed qualifiers are still ranked across groups by points, goal difference, goals for, then lot (teams of
 * different groups have no head-to-head).  No Philox word is added or moved: a simulation reads the same words under
 * either rule, and only its group order can differ.
 *
 * played_h2h: HOST int32 [T_tab, T_tab, 2], entry (u, v) = (points of slot u, goals of slot u) in the played matches
 * between u and v (NULL: none played); the diagonal is ignored, and a negative entry is refused.  The call copies it
 * into the workspace (cudaMemcpyAsync: a pageable array makes the call wait for the stream) and indexes the remaining
 * fixtures by slot pair there from home_slot / away_slot, so a level set costs only the fixtures among its members.  An
 * unknown rule: BPLX_E_INVALID (and 0 from the workspace-size calls).
 */
#define BPLX_RANK_GOAL_DIFF 0
#define BPLX_RANK_HEAD_TO_HEAD 1
typedef struct {
  int32_t rule;                   /* BPLX_RANK_* */
  const int32_t* played_h2h;      /* host [T_tab, T_tab, 2] (points, goals) of slot u against slot v, or NULL */
} bplx_ranking;

size_t bplx_simulate_table_ex_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, const bplx_table* t,
                                              const bplx_ranking* r);
/* bplx_simulate_table with a ranking rule; bplx_simulate_table is this call with r = NULL. */
int bplx_simulate_table_ex(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                           const uint8_t* away_slot, const bplx_table* t, const bplx_ranking* r, int max_goals,
                           int sims_per_draw, unsigned long long seed, long long first_draw,
                           unsigned long long* position_counts, unsigned long long* points_counts, uint8_t* positions,
                           uint8_t* scores, unsigned long long* invalid, void* workspace, size_t workspace_bytes,
                           void* stream);
size_t bplx_simulate_tournament_ranked_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f,
                                                       const bplx_table* t, const bplx_bracket* b,
                                                       const bplx_ranking* r);
/* bplx_simulate_tournament_ex with a ranking rule for the group stage; bplx_simulate_tournament_ex is this call with
 * r = NULL. */
int bplx_simulate_tournament_ranked(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                                    const uint8_t* away_slot, const bplx_table* t, const bplx_bracket* b,
                                    const uint8_t* tie_format, const bplx_ranking* r, int max_goals, int sims_per_draw,
                                    unsigned long long seed, long long first_draw, unsigned long long* position_counts,
                                    unsigned long long* points_counts, unsigned long long* reach_counts,
                                    unsigned long long* win_counts, unsigned long long* decided_counts,
                                    uint8_t* positions, uint8_t* scores, uint8_t* ko_entrants, uint8_t* ko_scores,
                                    uint8_t* ko_winners, uint8_t* ko_extra, unsigned long long* invalid,
                                    void* workspace, size_t workspace_bytes, void* stream);

/* ---- posterior predictive checks: replicated scores of the observed matches and their statistics ------------ */
/*
 * Replicate and random numbers.  Replicate n = (first_draw + s) * R + r (R = sims_per_draw) uses posterior draw s.  Its
 * random numbers are curand_init(seed, n, 0) followed by curand() (Philox4_32_10).  Words 2m and 2m + 1 become u_h and
 * u_a of observed match m through curand_uniform.  These are exactly the word addresses bplx_simulate_table gives
 * fixture f.
 *
 * One match of one replicate.  The score is drawn by the season simulation's sampler, unchanged: the predict path's
 * rates (neutral venues and confederations included, Extended's clip not applied); the draw's own grid up to max_goals
 * (1..63), with tau clamped at 0, normalised by its sum; inverse CDF over home goals, then over away goals given home
 * goals.  As a result, with the same seed, draws and matches, the replicated scores equal bplx_simulate_table's scores.
 * A replicate that meets a non-finite rate or normaliser is counted in `invalid`, as in simulation.  Match weights are
 * ignored, as in bplx_pointwise_loglik.
 *
 * Statistics per replicate.  All are integers, so device atomics give the same bits in any order:
 *   score_counts [B, B]         matches with min(hg, B - 1) = i, min(ag, B - 1) = j (B = score_bins, 2..16)
 *   outcome_counts [3]          home wins, draws, away wins ("home" = the listed home team, neutral venue or not)
 *   goals [2]                   total home goals, total away goals
 *   total_goals_sq []           sum_m (hg + ag)^2
 *   team_points [T]             points of each model team over the matches (points_win for a win, points_draw for a draw)
 *   team_goals_for [T], team_goals_against [T]   per model team
 * Replicated goals cannot exceed max_goals.  The host computes the dispersion of total goals, the statistics of the
 * observed scores and the posterior predictive p-values (bpl_next_b200/ppc.py).
 *
 * Outputs (device; overwritten): row q = s * R + r of this call, q < N = num_samples * R.  An invalid replicate (also: a
 * match naming a team >= num_teams or a confederation >= num_conferences) has -1 in every statistic of its row and
 * 0xFF as the scores of the offending match.  scores [N, M, 2] uint8 (home, away) is optional, in the layout of
 * bplx_simulate_table's scores.  The statistics depend neither on the launch geometry nor on the draw range of the
 * call: calls on draws [0, k) and [k, S) give the rows of the single call.  The workspace holds the [S, row]
 * exponential table of bplx_score_grid's pre-pass (bplx_posterior_predictive_workspace_bytes).
 * Refusals: DYNAMIC, N >= 2^31, or more teams than one CTA's shared memory holds (about 6,000): BPLX_E_UNSUPPORTED;
 * max_goals outside 1..63, score_bins outside 2..16, R < 1, missing goals or outputs, points outside 0 <= points_draw <=
 * points_win, points_win >= 1, or max(points_win, max_goals) * M >= 2^31 (a count that could overflow): BPLX_E_INVALID.
 */
typedef struct {
  int32_t* score_counts;          /* device [N, B, B] */
  int32_t* outcome_counts;        /* device [N, 3] */
  int64_t* goals;                 /* device [N, 2] */
  int64_t* total_goals_sq;        /* device [N] */
  int32_t* team_points;           /* device [N, T] */
  int32_t* team_goals_for;        /* device [N, T] */
  int32_t* team_goals_against;    /* device [N, T] */
  uint8_t* scores;                /* device [N, M, 2] or NULL */
  unsigned long long* invalid;    /* device [1]: invalid replicates */
} bplx_ppc_output;

size_t bplx_posterior_predictive_workspace_bytes(const bplx_samples* s, const bplx_observations* obs);
int bplx_posterior_predictive(const bplx_samples* s, const bplx_observations* obs, int max_goals, int score_bins,
                              int points_win, int points_draw, int sims_per_draw, unsigned long long seed,
                              long long first_draw, const bplx_ppc_output* out, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ---- misc --------------------------------------------------------------------------------- */
/* ---- predict over sample shards: the sum of the partial grids over the ranks, over peer memory ------------- */
/*
 * One-shot all-reduce(sum) of two element ranges of SYMMETRIC buffers (one per rank, same size, each mapped into every
 * rank's address space -- e.g. torch.distributed._symmetric_memory): replaces the all_reduce that finishes the reference's
 * `.mean(axis=0)` over posterior samples (bpl/base.py:94-110) when the samples are sharded over GPUs.
 *   bufs[q]     device pointer (valid on THIS rank) to rank q's buffer, q = 0 .. nranks-1; bufs[rank] is this rank's own.
 *               Layout of every buffer: `flag_bytes` of 32-bit flags (zero before the first call; flag p of rank q's
 *               buffer = the last epoch rank p has published), then the float data.
 *   off, cnt    element ranges of the data (grid rows, outcome rows of a fixture range); cnt1 may be 0
 *   out0, out1  this rank's results (ordinary device memory): out[i] = sum over q, in rank order, of data_q[off + i] --
 *               the same bits on every rank
 *   epoch       a counter that every rank increases by one per call (all ranks make the same sequence of calls); 0 = the
 *               kernel keeps the counter itself, in word 16 of this rank's flag area (the call then has no argument that
 *               changes from one call to the next and can be replayed in a CUDA graph).  flag_bytes >= 68, multiple of 16.
 * The kernel publishes this rank's flag to all peers, waits for theirs, then reads every rank's range over NVLink.  A
 * rank may overwrite a range of its own buffer again only after a later call on that rank has returned from its wait
 * (double-buffer by call parity, as bpl_next_b200.parallel.ShardedScoreGrid does).
 */
int bplx_peer_sum(void* const* bufs, int nranks, int rank, size_t flag_bytes, size_t off0, size_t cnt0, float* out0,
                  size_t off1, size_t cnt1, float* out1, unsigned epoch, void* stream);

/* The library reads its testing / tuning switches (BPLX_NO_PDL, BPLX_SPLIT, BPLX_HOST_CHUNKS, BPLX_NUTS_GENERIC,
 * BPLX_NO_TAIL_SPLIT, BPLX_NO_TRANSPOSE) from the environment once, at first use -- never on a launch path; call this after changing them. */
void bplx_reload_env(void);
const char* bplx_last_error(void);
int bplx_version(void);
/* number of kernel launches this library has enqueued from this process (for bench accounting) */
unsigned long long bplx_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* BPLX_H_ */
