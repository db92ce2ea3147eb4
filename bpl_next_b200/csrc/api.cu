// api.cu -- the extern "C" surface declared in include/bplx.h.
#include <limits.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <new>

#include "common.cuh"
#include "plan.h"
#include "problem.h"
#include "loo.h"
#include "ppc.h"
#include "score_grid.h"
#include "simulate.h"

namespace bplx {

static thread_local char g_err[1024] = "";
static std::atomic<unsigned long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}
void note_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

static EnvSwitches g_env;
static std::once_flag g_env_once;
void reload_env_switches() {
  EnvSwitches e;
  e.no_pdl = getenv("BPLX_NO_PDL") != nullptr;
  e.nuts_generic = getenv("BPLX_NUTS_GENERIC") != nullptr;
  e.no_tail_split = getenv("BPLX_NO_TAIL_SPLIT") != nullptr;
  e.no_transpose = getenv("BPLX_NO_TRANSPOSE") != nullptr;
  if (const char* v = getenv("BPLX_TRANSPOSE_MIN_ELEMS")) e.transpose_min_elems = (size_t)atoll(v);
  if (const char* v = getenv("BPLX_SPLIT")) e.split = atoi(v);
  if (const char* v = getenv("BPLX_HOST_CHUNKS")) e.host_chunks = atoi(v);
  g_env = e;
}
const EnvSwitches& env_switches() {
  std::call_once(g_env_once, reload_env_switches);
  return g_env;
}

constexpr size_t kUploadSlack = (size_t)kMaxSplit * kMaxWarps * sizeof(EntryClip) + 64;
template <typename T>
static int upload(bplx_problem* p, const std::vector<T>& h, const T** out) {
  *out = nullptr;
  if (h.empty()) return BPLX_OK;
  void* d = nullptr;
  // kUploadSlack zero bytes follow every array: the arg-max search reads its first candidate entry of a piece before it
  // knows how many entries the piece has (logdensity.cu)
  const size_t bytes = h.size() * sizeof(T);
  BPLX_CUDA(cudaMalloc(&d, bytes + kUploadSlack));
  p->dev_allocs.push_back(d);
  BPLX_CUDA(cudaMemcpy(d, h.data(), bytes, cudaMemcpyHostToDevice));
  BPLX_CUDA(cudaMemset(static_cast<unsigned char*>(d) + bytes, 0, kUploadSlack));
  *out = static_cast<const T*>(d);
  return BPLX_OK;
}

// the device-side alias of a page-locked (cudaHostAlloc / cudaHostRegister, mapped) host array, else `fallback`
static float* mapped_or(float* host, float* fallback) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, host) != cudaSuccess) {
    cudaGetLastError();
    return fallback;
  }
  if (a.type == cudaMemoryTypeHost && a.devicePointer != nullptr) return static_cast<float*>(a.devicePointer);
  return fallback;
}

// out[c][r] = in[r][c] for an R x Cc matrix (row pitches ldi, ldo): the host entry point takes and returns [chains, D]
// arrays (what the reference's vmapped potential sees), the kernel's native layout is [D, chains].
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int R, int Cc,
                                                        size_t ldi, size_t ldo) {
  // a block moves 128 rows x 32 columns: its 16 loads per thread are all issued before the first store
  __shared__ float tile[4][32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 128;
  float v[4][4];
#pragma unroll
  for (int s = 0; s < 4; s++)
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int r = r0 + s * 32 + threadIdx.y + 8 * k, c = c0 + threadIdx.x;
      v[s][k] = (r < R && c < Cc) ? in[(size_t)r * ldi + c] : 0.0f;
    }
#pragma unroll
  for (int s = 0; s < 4; s++)
#pragma unroll
    for (int k = 0; k < 4; k++) tile[s][threadIdx.y + 8 * k][threadIdx.x] = v[s][k];
  __syncthreads();
#pragma unroll
  for (int s = 0; s < 4; s++)
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int c = c0 + threadIdx.y + 8 * k, r = r0 + s * 32 + threadIdx.x;
      if (r < R && c < Cc) out[(size_t)c * ldo + r] = tile[s][threadIdx.x][threadIdx.y + 8 * k];
    }
}
static int launch_transpose(const float* in, float* out, int R, int Cc, size_t ldi, size_t ldo, cudaStream_t s) {
  const dim3 grid((unsigned)((Cc + 31) / 32), (unsigned)((R + 127) / 128));
  BPLX_REQUIRE(grid.y <= 65535u, BPLX_E_UNSUPPORTED, "transpose of %d rows", R);
  transpose_kernel<<<grid, dim3(32, 8), 0, s>>>(in, out, R, Cc, ldi, ldo);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

// Room behind the kernel's own workspace for one transposed copy of theta and of the gradient ([D][Cpad] each): large
// [chains, D] batches are computed in the kernel's native [D, chains] layout (see enqueue).
static size_t align256(size_t n) { return (n + 255) / 256 * 256; }
static size_t transpose_room(const KernelParams& kp, int C) {
  if ((size_t)C * (size_t)kp.D < env_switches().transpose_min_elems) return 0;
  return 2 * (((size_t)C + 31) / 32 * 32) * (size_t)kp.D * sizeof(float);
}

static size_t workspace_bytes(const KernelParams& kp, int C) {
  const size_t Cpad = ((size_t)C + 31) / 32 * 32;
  if (kp.model == BPLX_DYNAMIC)  // the walk's prefix sums (+ the per-gameweek hyper-parameter table when shared memory is short)
    return ((size_t)kp.G * kp.T * 2 + (kp.dyn_hyp_ws ? (size_t)kp.G * 16 : 0)) * Cpad * sizeof(float);
  if (kp.Cf <= 0) return 0;
  return (size_t)kp.V * Cpad * sizeof(float);
}

static int enqueue(const bplx_problem* p, int C, int layout, int ld, const float* theta, float* lp, float* grad,
                   float* corr_coef, void* ws, size_t ws_bytes, cudaStream_t stream, bool pdl = false, bool lik = false) {
  BPLX_REQUIRE(p != nullptr, BPLX_E_INVALID, "problem is NULL");
  BPLX_REQUIRE(C > 0, BPLX_E_INVALID, "num_chains must be positive (got %d)", C);
  BPLX_REQUIRE(theta && lp && grad, BPLX_E_INVALID, "theta, lp and grad must not be NULL");
  if (layout == BPLX_CHAIN_MAJOR && !env_switches().no_transpose) {
    // A [chains, D] batch (what a vmapped jax.ffi call hands over): tiled transposes of theta before and of the
    // gradient after the kernel, which then runs in its native layout (configs[2], 32,768 chains: 1.6 + 0.14 ms instead
    // of 3.5 ms of strided per-chain reads) -- when the caller's workspace has the room bplx_logdensity_workspace_bytes
    // asks for.  From 2^17 elements: measured per leapfrog of a fit with chain-major sampler state, configs[1] at 4,096
    // chains x 73 parameters 45 -> 40 us, configs[2] data at 256 chains x 1,339 231 -> 153 us; configs[0] at 1,024 x 45
    // (below the threshold) 28.7 vs 29.5 us.
    const size_t base = align256(workspace_bytes(p->kp, C)), room = transpose_room(p->kp, C);
    if (room > 0 && ws != nullptr && ws_bytes >= base + room) {
      const int Dc = lik ? p->lik_D : p->kp.D;
      const size_t ldm = ld > 0 ? (size_t)ld : (size_t)Dc, Cpad = ((size_t)C + 31) / 32 * 32;
      BPLX_REQUIRE(ldm >= (size_t)Dc, BPLX_E_INVALID, "chain-major ld (%d) < D (%d)", ld, Dc);
      float* tin = reinterpret_cast<float*>(static_cast<char*>(ws) + base);
      float* tout = tin + Cpad * (size_t)p->kp.D;
      int rc = launch_transpose(theta, tin, C, Dc, ldm, Cpad, stream);
      if (rc != BPLX_OK) return rc;
      rc = enqueue(p, C, BPLX_CHAIN_MINOR, (int)Cpad, tin, lp, tout, corr_coef, ws, base, stream, pdl, lik);
      if (rc != BPLX_OK) return rc;
      return launch_transpose(tout, grad, Dc, C, Cpad, ldm, stream);
    }
  }
  KernelParams kp = p->kp;
  if (lik) {  // the same plan read through the likelihood-only site layout: constrained tables in, no priors
    BPLX_REQUIRE(kp.model != BPLX_DYNAMIC, BPLX_E_UNSUPPORTED, "bplx_loglik_fwdbwd: DYNAMIC is not supported");
    kp.lik_only = 1;
    kp.off = p->lik_off;
    for (int i = 0; i < 12; i++) kp.hyper[i] = p->lik_hyper[i];
    kp.nhyper = p->lik_nhyper;
    kp.D = p->lik_D;
    kp.K = 0;
    kp.const_term = p->lik_const;
  }
  if (layout == BPLX_CHAIN_MAJOR) {
    kp.sd = 1;
    kp.sc = ld > 0 ? ld : kp.D;
    BPLX_REQUIRE(kp.sc >= kp.D, BPLX_E_INVALID, "chain-major ld (%d) < D (%d)", ld, kp.D);
  } else if (layout == BPLX_CHAIN_MINOR) {
    kp.sc = 1;
    kp.sd = ld > 0 ? ld : C;
    BPLX_REQUIRE(kp.sd >= C, BPLX_E_INVALID, "chain-minor ld (%d) < num_chains (%d)", ld, C);
  } else {
    BPLX_REQUIRE(false, BPLX_E_INVALID, "unknown layout %d", layout);
  }
  BPLX_REQUIRE((long long)kp.D * (long long)kp.sd + (long long)C * (long long)kp.sc < (1ll << 31), BPLX_E_UNSUPPORTED,
               "theta / grad of %d x %d elements exceed the 31-bit element index of the kernel", C, kp.D);
  const size_t need = workspace_bytes(kp, C);
  BPLX_REQUIRE(ws_bytes >= need && (need == 0 || ws != nullptr), BPLX_E_WORKSPACE,
               "workspace too small: %zu bytes given, %zu needed", ws_bytes, need);
  kp.C = C;
  kp.Cpad = (C + 31) / 32 * 32;
  kp.theta = theta;
  kp.lp = lp;
  kp.grad = grad;
  kp.corr_coef = corr_coef;
  kp.scratch = static_cast<float*>(ws);
  // few chains: several CTAs (one cluster) share a group of 32 chains, as many as the device holds at once
  int si = 0;
  const int groups = (C + kChains - 1) / kChains;
  for (int i = kNumSplits - 1; i >= 1; i--)
    if (p->s1[i] && (1 << i) <= kp.split_hint && groups <= p->max_clusters[i]) {
      si = i;
      break;
    }
  if (const int want = env_switches().split) {  // testing / tuning: force 1, 2, 4 or 8 CTAs per group
    for (int i = 0; i < kNumSplits; i++)
      if ((1 << i) == want && p->s1[i] && (i == 0 || p->max_clusters[i] > 0)) si = i;
  }
  auto use_split = [&](int i) {
    kp.split = 1 << i;
    kp.stream1 = p->s1[i];
    kp.stream2 = p->s2[i];
    kp.warp_b1 = p->wb1[i];
    kp.warp_b2 = p->wb2[i];
  };
  use_split(si);
  kp.group0 = 0;
  kp.ngroups = groups;
  if (kp.model == BPLX_DYNAMIC) return launch_logdensity_dynamic(kp, stream);
  // Tail split: the kernel holds one CTA per SM, so `groups` CTAs run in waves of `sm_count`; when the last, partial
  // wave is small enough, its groups go to a second launch with 2, 4 or 8 CTAs (a cluster) per group, which fills the
  // SMs the wave would leave idle and ends sooner (configs[2] at 16,384 chains: 512 groups = 3 waves + 68 groups).
  int ti = 0;
  const int rest = p->sm_count > 0 ? groups % p->sm_count : 0;
  if (si == 0 && rest > 0 && rest < groups && !env_switches().split && !env_switches().no_tail_split) {
    for (int i = kNumSplits - 1; i >= 1; i--)
      if (p->s1[i] && (1 << i) <= kp.split_hint && rest <= p->max_clusters[i] && rest * (1 << i) <= p->sm_count) {
        ti = i;
        break;
      }
  }
  if (ti == 0) return launch_logdensity(kp, p->wb[si], stream, pdl);
  kp.ngroups = groups - rest;
  int rc = launch_logdensity(kp, p->wb[0], stream, pdl);
  if (rc != BPLX_OK) return rc;
  use_split(ti);
  kp.group0 = groups - rest;
  kp.ngroups = rest;
  return launch_logdensity(kp, p->wb[ti], stream, pdl);
}

}  // namespace bplx

using namespace bplx;

extern "C" {

int bplx_problem_create(const bplx_problem_desc* desc, bplx_problem** out) {
  BPLX_REQUIRE(desc && out, BPLX_E_INVALID, "desc / out is NULL");
  *out = nullptr;
  HostPlan hp;
  std::string err;
  int rc = build_plan(*desc, &hp, &err);
  if (rc != BPLX_OK) {
    set_error("%s", err.c_str());
    return rc;
  }
  bplx_problem* p = new (std::nothrow) bplx_problem();
  BPLX_REQUIRE(p, BPLX_E_NOMEM, "out of host memory");
  auto fail = [&](int code) {
    bplx_problem_destroy(p);
    return code;
  };
  if (cudaGetDevice(&p->device) != cudaSuccess) {
    set_error("cudaGetDevice failed: no usable CUDA device (bplx has no CPU fallback)");
    return fail(BPLX_E_CUDA);
  }
  p->kp = hp.kp;
  p->layout = hp.layout;
  p->lik_off = hp.lik_off;
  for (int i = 0; i < 12; i++) p->lik_hyper[i] = hp.lik_hyper[i];
  p->lik_nhyper = hp.lik_nhyper;
  p->lik_D = hp.lik_D;
  p->lik_const = hp.lik_const;
  p->lik_layout = hp.lik_layout;
  KernelParams& kp = p->kp;
#define UP(vec, ptr)                                 \
  if ((rc = upload(p, hp.vec, &(ptr))) != BPLX_OK) return fail(rc)
  UP(stream1, p->s1[0]);
  UP(stream2, p->s2[0]);
  UP(warp_b1, p->wb1[0]);
  UP(warp_b2, p->wb2[0]);
  for (int i = 1; i < kNumSplits; i++) {
    if (hp.more[i - 1].stream1.empty()) continue;  // (DYNAMIC has no split plans)
    UP(more[i - 1].stream1, p->s1[i]);
    UP(more[i - 1].stream2, p->s2[i]);
    UP(more[i - 1].warp_b1, p->wb1[i]);
    UP(more[i - 1].warp_b2, p->wb2[i]);
  }
  auto keep_bounds = [&](int i, const std::vector<uint32_t>& b1, const std::vector<uint32_t>& b2) {
    const size_t cap = sizeof(p->wb[i].b1) / sizeof(uint32_t);
    for (size_t k = 0; k < b1.size() && k < cap; k++) p->wb[i].b1[k] = b1[k];
    for (size_t k = 0; k < b2.size() && k < cap; k++) p->wb[i].b2[k] = b2[k];
  };
  keep_bounds(0, hp.warp_b1, hp.warp_b2);
  for (int i = 1; i < kNumSplits; i++) keep_bounds(i, hp.more[i - 1].warp_b1, hp.more[i - 1].warp_b2);
  kp.stream1 = p->s1[0];
  kp.stream2 = p->s2[0];
  kp.warp_b1 = p->wb1[0];
  kp.warp_b2 = p->wb2[0];
  kp.split = 1;
  UP(team_vptr, kp.team_vptr);
  UP(team_flags, kp.team_flags);
  UP(v_team, kp.v_team);
  UP(v_conf, kp.v_conf);
  UP(conf_vptr, kp.conf_vptr);
  UP(conf_vlist, kp.conf_vlist);
  UP(yexp, kp.yexp);
  UP(yteam, kp.yteam);
  UP(yconf, kp.yconf);
  UP(Xs, kp.Xs);
  UP(gw_tptr, kp.gw_tptr);
  UP(gw_tlist, kp.gw_tlist);
#undef UP
  rc = kp.model == BPLX_DYNAMIC ? logdensity_dynamic_set_attributes() : logdensity_set_attributes(kp);
  if (rc != BPLX_OK) return fail(rc);
  if (cudaDeviceGetAttribute(&p->sm_count, cudaDevAttrMultiProcessorCount, p->device) != cudaSuccess) p->sm_count = 0;
  p->max_clusters[0] = 1 << 30;
  if (kp.model != BPLX_DYNAMIC)
    for (int i = 1; i < kNumSplits; i++) p->max_clusters[i] = p->s1[i] ? logdensity_max_clusters(kp, 1 << i) : 0;
  p->stats[0] = desc->num_matches;
  p->stats[1] = hp.n1;
  p->stats[2] = hp.n1_padded;
  p->stats[3] = hp.n2;
  p->stats[4] = hp.n2_padded;
  p->stats[5] = kp.smem_total;
  p->stats[6] = kp.nwarps;
  p->stats[7] = kp.V;
  if (kp.model != BPLX_DYNAMIC) {  // what each warp of the split-1 plan walks (plan tuning, DESIGN.md)
    p->warp_stats.assign((size_t)kp.nwarps * 12, 0);
    for (int phase = 0; phase < 2; phase++) {
      const std::vector<unsigned char>& S = phase ? hp.stream2 : hp.stream1;
      const std::vector<uint32_t>& wb = phase ? hp.warp_b2 : hp.warp_b1;
      const size_t esz = (phase == 0 && kp.clip) ? sizeof(EntryClip) : sizeof(Entry);
      const uint32_t minp = phase ? kp.min_piece2 : kp.min_piece1;
      for (int w = 0; w < kp.nwarps && w + 1 < (int)wb.size(); w++) {
        long long* o = &p->warp_stats[(size_t)w * 12 + phase * 6];
        const uint32_t len = wb[w + 1] - wb[w];
        o[5] = (len + kp.stage_bytes - 1) / kp.stage_bytes;
        for (uint32_t st = 0; st < len; st += kp.stage_bytes) {
          uint32_t a = wb[w] + st;
          const uint32_t aend = wb[w] + std::min(len, st + kp.stage_bytes);
          while (a + minp <= aend) {
            ListHdr H;
            memcpy(&H, &S[a], sizeof H);
            if (H.n0 + H.n1 + H.n2 == 0) break;  // stage padding
            const bool home = (H.kind & 1) == 0;
            if (phase == 0) {
              o[home ? 0 : 1]++;
              o[home ? 2 : 3] += H.n0;
            } else {
              o[0]++;
              o[1] += H.n0;
              o[2] += H.n1;
              o[3] += H.n2;
            }
            if (H.flags & kTeamFirst) o[4]++;
            a += (uint32_t)sizeof(ListHdr) + (uint32_t)((H.n0 + H.n1 + H.n2) * esz);
          }
        }
      }
    }
  }
  *out = p;
  return BPLX_OK;
}

void bplx_problem_destroy(bplx_problem* p) {
  if (!p) return;
  for (void* d : p->dev_allocs) cudaFree(d);
  if (p->d_theta) cudaFree(p->d_theta);
  if (p->d_out) cudaFree(p->d_out);
  if (p->d_ws) cudaFree(p->d_ws);
  if (p->d_tin) cudaFree(p->d_tin);
  if (p->d_tout) cudaFree(p->d_tout);
  if (p->host_stream) cudaStreamDestroy(p->host_stream);
  if (p->host_in) cudaStreamDestroy(p->host_in);
  if (p->host_out) cudaStreamDestroy(p->host_out);
  for (cudaEvent_t e : p->host_ev)
    if (e) cudaEventDestroy(e);
  delete p;
}

int bplx_num_params(const bplx_problem* p) { return p ? p->kp.D : BPLX_E_INVALID; }

const char* bplx_problem_layout(const bplx_problem* p) { return p ? p->layout.c_str() : ""; }

int bplx_problem_stats(const bplx_problem* p, long long* out, int n) {
  BPLX_REQUIRE(p && out, BPLX_E_INVALID, "problem / out is NULL");
  for (int i = 0; i < n && i < 8; i++) out[i] = p->stats[i];
  return n < 8 ? n : 8;
}

int bplx_problem_warp_stats(const bplx_problem* p, long long* out, int n) {
  BPLX_REQUIRE(p && out, BPLX_E_INVALID, "problem / out is NULL");
  const int have = (int)p->warp_stats.size();
  for (int i = 0; i < n && i < have; i++) out[i] = p->warp_stats[i];
  return n < have ? n : have;
}

size_t bplx_logdensity_workspace_bytes(const bplx_problem* p, int num_chains) {
  if (!p || num_chains <= 0) return 0;
  const size_t room = transpose_room(p->kp, num_chains);
  return room ? align256(workspace_bytes(p->kp, num_chains)) + room : workspace_bytes(p->kp, num_chains);
}

int bplx_logdensity_fwdbwd(const bplx_problem* p, int num_chains, int layout, int ld, const float* theta, float* lp,
                           float* grad, float* corr_coef, void* workspace, size_t workspace_bytes, void* stream) {
  return enqueue(p, num_chains, layout, ld, theta, lp, grad, corr_coef, workspace, workspace_bytes,
                 static_cast<cudaStream_t>(stream), /*pdl=*/true);
}

int bplx_loglik_num_inputs(const bplx_problem* p) {
  if (!p) return BPLX_E_INVALID;
  return p->kp.model == BPLX_DYNAMIC ? BPLX_E_UNSUPPORTED : p->lik_D;
}

const char* bplx_loglik_layout(const bplx_problem* p) { return p ? p->lik_layout.c_str() : ""; }

int bplx_loglik_fwdbwd(const bplx_problem* p, int num_chains, int layout, int ld, const float* tables, float* loglik,
                       float* grad, float* corr_coef, void* workspace, size_t workspace_bytes, void* stream) {
  return enqueue(p, num_chains, layout, ld, tables, loglik, grad, corr_coef, workspace, workspace_bytes,
                 static_cast<cudaStream_t>(stream), /*pdl=*/true, /*lik=*/true);
}

int bplx_logdensity_fwdbwd_host(bplx_problem* p, int C, const float* theta, float* lp, float* grad, float* corr_coef) {
  BPLX_REQUIRE(p != nullptr, BPLX_E_INVALID, "problem is NULL");
  BPLX_REQUIRE(C > 0, BPLX_E_INVALID, "num_chains must be positive (got %d)", C);
  BPLX_REQUIRE(theta && lp && grad, BPLX_E_INVALID, "theta, lp and grad must not be NULL");
  std::lock_guard<std::mutex> lock(p->mu);
  BPLX_CUDA(cudaSetDevice(p->device));
  const size_t D = (size_t)p->kp.D;
  if (!p->host_stream) BPLX_CUDA(cudaStreamCreateWithFlags(&p->host_stream, cudaStreamNonBlocking));
  if (C > p->host_cap) {
    if (p->d_theta) cudaFree(p->d_theta);
    if (p->d_out) cudaFree(p->d_out);
    if (p->d_ws) cudaFree(p->d_ws);
    p->d_theta = p->d_out = nullptr;
    p->d_ws = nullptr;
    p->host_cap = 0;
    BPLX_CUDA(cudaMalloc(&p->d_theta, (size_t)C * D * sizeof(float)));
    BPLX_CUDA(cudaMalloc(&p->d_out, ((size_t)C * D + 2 * (size_t)C) * sizeof(float)));
    p->d_ws_bytes = workspace_bytes(p->kp, C);
    if (p->d_ws_bytes) BPLX_CUDA(cudaMalloc(&p->d_ws, p->d_ws_bytes));
    p->host_cap = C;
  }
  // Chains are cut into up to four chunks so that the upload of chunk k+1, the kernel of chunk k and the download
  // of chunk k-1 overlap (PCIe is full duplex); the kernels run in order on one stream and share the workspace.
  if (!p->host_in) {
    BPLX_CUDA(cudaStreamCreateWithFlags(&p->host_in, cudaStreamNonBlocking));
    BPLX_CUDA(cudaStreamCreateWithFlags(&p->host_out, cudaStreamNonBlocking));
    for (cudaEvent_t& e : p->host_ev) BPLX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  cudaStream_t s = p->host_stream;
  float* d_grad = p->d_out;
  float* d_lp = p->d_out + (size_t)C * D;
  float* d_cc = d_lp + C;
  // (only worth it when a chunk still fills the GPU: below ~16k chains K1 is latency-bound and chunking serialises it;
  //  measured on configs[1], 4,096 chains: 104 us in one piece, 138 us in four)
  // by payload (measured on configs[2] data, ms per call for 1 / 2 / 4 / 8 chunks: 22 MB each way 1.07 / 0.82 / 0.78 / 1.01,
  // 44 MB 2.10 / 1.53 / 1.32 / 1.41, 88 MB 4.08 / 2.97 / 2.48 / 2.39; 175 MB: 8 chunks)
  const size_t payload = (size_t)C * D * sizeof(float);
  int nchunk = payload >= ((size_t)80 << 20) ? 8 : (payload >= ((size_t)16 << 20) ? 4 : (payload >= ((size_t)6 << 20) ? 2 : 1));
  while (nchunk > 1 && C / nchunk < 256) nchunk /= 2;
  if (const int want = env_switches().host_chunks)  // tuning: 1, 2, 4, 8 or 16 pipelined chunks
    if (want == 1 || want == 2 || want == 4 || want == 8 || want == 16) nchunk = want;
  // Large batches go through the kernel's native chain-minor layout: a tiled transpose of theta before the kernel and of
  // the gradient after it (two passes over HBM each, ~0.1 ms for configs[2] at 32,768 chains) instead of the kernel's
  // strided per-chain reads (3.5 ms against 1.6 ms in the native layout).
  const bool native = (size_t)C * D >= std::max(env_switches().transpose_min_elems, (size_t)1 << 20) && !env_switches().no_transpose;
  if (nchunk == 1) {  // one piece: everything in order on one stream, no events (each costs microseconds at this scale)
    // lp and corr_coef are one coalesced 128-byte store per warp: when the caller's arrays are page-locked the kernel
    // writes them straight into host memory (posted PCIe writes) instead of two more copies of 6.6 us each
    float* k_lp = mapped_or(lp, d_lp);
    float* k_cc = corr_coef ? mapped_or(corr_coef, d_cc) : d_cc;
    BPLX_CUDA(cudaMemcpyAsync(p->d_theta, theta, (size_t)C * D * sizeof(float), cudaMemcpyHostToDevice, s));
    int rc;
    if (native) {
      const int ldc = (C + 31) / 32 * 32;
      if (ldc > p->tr_cap) {
        if (p->d_tin) cudaFree(p->d_tin);
        if (p->d_tout) cudaFree(p->d_tout);
        p->d_tin = p->d_tout = nullptr;
        p->tr_cap = 0;
        BPLX_CUDA(cudaMalloc(&p->d_tin, (size_t)ldc * D * sizeof(float)));
        BPLX_CUDA(cudaMalloc(&p->d_tout, (size_t)ldc * D * sizeof(float)));
        p->tr_cap = ldc;
      }
      rc = launch_transpose(p->d_theta, p->d_tin, C, (int)D, D, (size_t)ldc, s);
      if (rc != BPLX_OK) return rc;
      rc = enqueue(p, C, BPLX_CHAIN_MINOR, ldc, p->d_tin, k_lp, p->d_tout, k_cc, p->d_ws, p->d_ws_bytes, s);
      if (rc != BPLX_OK) return rc;
      rc = launch_transpose(p->d_tout, d_grad, (int)D, C, (size_t)ldc, D, s);
    } else {
      rc = enqueue(p, C, BPLX_CHAIN_MAJOR, (int)D, p->d_theta, k_lp, d_grad, k_cc, p->d_ws, p->d_ws_bytes, s);
    }
    if (rc != BPLX_OK) return rc;
    BPLX_CUDA(cudaMemcpyAsync(grad, d_grad, (size_t)C * D * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (k_lp == d_lp) BPLX_CUDA(cudaMemcpyAsync(lp, d_lp, (size_t)C * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (corr_coef && k_cc == d_cc)
      BPLX_CUDA(cudaMemcpyAsync(corr_coef, d_cc, (size_t)C * sizeof(float), cudaMemcpyDeviceToHost, s));
    BPLX_CUDA(cudaStreamSynchronize(s));
    return BPLX_OK;
  }
  const int per = ((C + nchunk - 1) / nchunk + 31) / 32 * 32;
  if (native && per > p->tr_cap) {
    if (p->d_tin) cudaFree(p->d_tin);
    if (p->d_tout) cudaFree(p->d_tout);
    p->d_tin = p->d_tout = nullptr;
    p->tr_cap = 0;
    BPLX_CUDA(cudaMalloc(&p->d_tin, (size_t)per * D * sizeof(float)));
    BPLX_CUDA(cudaMalloc(&p->d_tout, (size_t)per * D * sizeof(float)));
    p->tr_cap = per;
  }
  // chunk sizes: with four or more chunks the first and the last are cut in half -- while the first chunk uploads and the
  // last downloads, the link runs in one direction only
  int sizes[40], ns = 0, left = C;
  auto push = [&](int n) {
    n = n < left ? n : left;
    if (n > 0) sizes[ns++] = n, left -= n;
  };
  if (nchunk >= 4) {
    const int half = (per / 2 + 31) / 32 * 32;
    push(half);
    push(half);
    while (left > per) push(per);
    push((left / 2 + 31) / 32 * 32);
    push(left);
  } else {
    while (left > 0) push(per);
  }
  for (int k = 0, c0 = 0; k < ns; c0 += sizes[k], k++) {
    const int n = sizes[k];
    const size_t off = (size_t)c0 * D;
    BPLX_CUDA(cudaMemcpyAsync(p->d_theta + off, theta + off, (size_t)n * D * sizeof(float), cudaMemcpyHostToDevice, p->host_in));
    BPLX_CUDA(cudaEventRecord(p->host_ev[2 * k], p->host_in));
    BPLX_CUDA(cudaStreamWaitEvent(s, p->host_ev[2 * k], 0));
    int rc;
    if (native) {  // (the transposed buffers are shared by the chunks: everything that touches them is in order on `s`)
      rc = launch_transpose(p->d_theta + off, p->d_tin, n, (int)D, D, (size_t)per, s);
      if (rc != BPLX_OK) return rc;
      rc = enqueue(p, n, BPLX_CHAIN_MINOR, per, p->d_tin, d_lp + c0, p->d_tout, d_cc + c0, p->d_ws, p->d_ws_bytes, s);
      if (rc != BPLX_OK) return rc;
      rc = launch_transpose(p->d_tout, d_grad + off, (int)D, n, (size_t)per, D, s);
    } else {
      rc = enqueue(p, n, BPLX_CHAIN_MAJOR, (int)D, p->d_theta + off, d_lp + c0, d_grad + off, d_cc + c0, p->d_ws,
                   p->d_ws_bytes, s);
    }
    if (rc != BPLX_OK) return rc;
    BPLX_CUDA(cudaEventRecord(p->host_ev[2 * k + 1], s));
    BPLX_CUDA(cudaStreamWaitEvent(p->host_out, p->host_ev[2 * k + 1], 0));
    BPLX_CUDA(cudaMemcpyAsync(grad + off, d_grad + off, (size_t)n * D * sizeof(float), cudaMemcpyDeviceToHost, p->host_out));
    BPLX_CUDA(cudaMemcpyAsync(lp + c0, d_lp + c0, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, p->host_out));
    if (corr_coef)
      BPLX_CUDA(cudaMemcpyAsync(corr_coef + c0, d_cc + c0, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, p->host_out));
  }
  BPLX_CUDA(cudaStreamSynchronize(p->host_out));
  return BPLX_OK;
}

// ---- score grid ------------------------------------------------------------------------------------------
// samples / fixtures checks shared by the score grid and the pointwise log-likelihood (`what` prefixes the message)
// allow_no_fixtures: F = 0 is accepted (a tournament whose group stage is already played), the fixture arrays may then
// be NULL
static int check_sample_args(const bplx_samples* s, const bplx_fixtures* f, const char* what,
                             bool allow_no_fixtures = false) {
  BPLX_REQUIRE(s && f, BPLX_E_INVALID, "samples / fixtures is NULL");
  BPLX_REQUIRE(s->model >= BPLX_DIXON_COLES && s->model <= BPLX_NEUTRAL_WC, BPLX_E_UNSUPPORTED,
               "%s: model %d unsupported (DYNAMIC predict is unusable in the reference)", what, s->model);
  const bool fixtures = !(allow_no_fixtures && f->num_fixtures == 0);
  BPLX_REQUIRE(s->num_samples > 0 && s->num_teams > 0 && (f->num_fixtures > 0 || !fixtures), BPLX_E_INVALID,
               "%s: num_samples, num_teams and num_fixtures must be positive", what);
  BPLX_REQUIRE(s->attack && s->defence && s->corr_coef && (!fixtures || (f->home_team && f->away_team)), BPLX_E_INVALID,
               "%s: attack, defence, corr_coef, home_team, away_team must not be NULL", what);
  BPLX_REQUIRE(s->home_attack, BPLX_E_INVALID, "%s: home_attack (home advantage) must not be NULL", what);
  if (s->model == BPLX_NEUTRAL || s->model == BPLX_NEUTRAL_WC)
    BPLX_REQUIRE(s->away_attack && s->home_defence && s->away_defence, BPLX_E_INVALID,
                 "%s: neutral models need away_attack, home_defence, away_defence", what);
  if (s->model == BPLX_NEUTRAL_WC)
    BPLX_REQUIRE(s->confederation_strength && s->num_conferences > 0 && (!fixtures || (f->home_conf && f->away_conf)),
                 BPLX_E_INVALID, "%s: NEUTRAL_WC needs confederation_strength, home_conf, away_conf", what);
  return BPLX_OK;
}

static int check_grid_args(const bplx_samples* s, const bplx_fixtures* f, int max_goals) {
  const int rc = check_sample_args(s, f, "score grid");
  if (rc != BPLX_OK) return rc;
  BPLX_REQUIRE(max_goals >= 1 && max_goals <= 63, BPLX_E_INVALID, "max_goals must be in [1, 63] (got %d)", max_goals);
  return BPLX_OK;
}

// the shape (model, S, T, Cf, F) and the sample / fixture arrays of gp; with F = 0 the fixture arrays may be NULL
static void bind_samples(const bplx_samples* s, const bplx_fixtures* f, GridParams* gp) {
  gp->model = s->model;
  gp->S = s->num_samples;
  gp->T = s->num_teams;
  gp->Cf = s->model == BPLX_NEUTRAL_WC ? s->num_conferences : 0;
  gp->F = f->num_fixtures;
  gp->attack = s->attack;
  gp->defence = s->defence;
  gp->ha = s->home_attack;
  gp->aa = s->away_attack;
  gp->hd = s->home_defence;
  gp->ad = s->away_defence;
  gp->conf = s->confederation_strength;
  gp->corr = s->corr_coef;
  gp->home = f->home_team;
  gp->away = f->away_team;
  gp->hconf = f->home_conf;
  gp->aconf = f->away_conf;
  gp->nv = f->neutral_venue;
}

static int check_workspace(const void* workspace, size_t workspace_bytes, size_t need) {
  BPLX_REQUIRE(workspace && workspace_bytes >= need, BPLX_E_WORKSPACE,
               "workspace too small: %zu bytes given, %zu needed", workspace_bytes, need);
  BPLX_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15u) == 0, BPLX_E_INVALID, "workspace must be 16-byte aligned");
  return BPLX_OK;
}

static size_t grid_plan(const bplx_samples* s, const bplx_fixtures* f, int max_goals, GridParams* gp, const char** err) {
  bind_samples(s, f, gp);
  gp->g = max_goals + 1;
  return score_grid_plan(gp, err);
}

size_t bplx_score_grid_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, int max_goals) {
  if (!s || !f || max_goals < 1 || s->num_samples <= 0 || s->num_teams <= 0 || f->num_fixtures <= 0) return 0;
  GridParams gp{};
  return grid_plan(s, f, max_goals, &gp, nullptr);
}

int bplx_score_grid(const bplx_samples* s, const bplx_fixtures* f, int max_goals, float scale, float* grid,
                    float* outcome, void* workspace, size_t workspace_bytes, void* stream) {
  return bplx_score_grid_ex(s, f, max_goals, scale, grid, outcome, workspace, workspace_bytes, stream, 0u);
}

int bplx_score_grid_ex(const bplx_samples* s, const bplx_fixtures* f, int max_goals, float scale, float* grid,
                       float* outcome, void* workspace, size_t workspace_bytes, void* stream, unsigned flags) {
  int rc = check_grid_args(s, f, max_goals);
  if (rc != BPLX_OK) return rc;
  BPLX_REQUIRE(grid != nullptr, BPLX_E_INVALID, "grid is NULL");
  GridParams gp{};
  const char* perr = nullptr;
  const size_t need = grid_plan(s, f, max_goals, &gp, &perr);
  BPLX_REQUIRE(need > 0, BPLX_E_UNSUPPORTED, "%s", perr ? perr : "score grid: unsupported shape");
  gp.scale = scale;
  rc = check_workspace(workspace, workspace_bytes, need);
  if (rc != BPLX_OK) return rc;
  gp.table = static_cast<float*>(workspace);
  gp.partial = reinterpret_cast<float*>(static_cast<unsigned char*>(workspace) + table_layout(&gp));
  gp.grid = grid;
  gp.outcome = outcome;
  gp.reuse_tables = (flags & BPLX_GRID_REUSE_TABLES) ? 1 : 0;
  return launch_score_grid(gp, static_cast<cudaStream_t>(stream));
}

int bplx_score_grid_host(const bplx_samples* s, const bplx_fixtures* f, int max_goals, float scale, float* grid,
                         float* outcome) {
  int rc = check_grid_args(s, f, max_goals);
  if (rc != BPLX_OK) return rc;
  BPLX_REQUIRE(grid != nullptr, BPLX_E_INVALID, "grid is NULL");
  const size_t S = s->num_samples, T = s->num_teams, F = f->num_fixtures, g = max_goals + 1;
  const size_t Cf = s->model == BPLX_NEUTRAL_WC ? s->num_conferences : 0;
  for (size_t i = 0; i < F; i++) {  // host arrays: an out-of-range index would read past the staged sample rows
    BPLX_REQUIRE(f->home_team[i] < T && f->away_team[i] < T, BPLX_E_INVALID,
                 "score grid: team index out of range at fixture %zu (%u, %u; num_teams %zu)", i,
                 (unsigned)f->home_team[i], (unsigned)f->away_team[i], T);
    if (Cf)
      BPLX_REQUIRE(f->home_conf[i] < Cf && f->away_conf[i] < Cf, BPLX_E_INVALID,
                   "score grid: confederation index out of range at fixture %zu (%u, %u; num_conferences %zu)", i,
                   (unsigned)f->home_conf[i], (unsigned)f->away_conf[i], Cf);
  }
  std::vector<void*> allocs;
  auto cleanup = [&]() {
    for (void* d : allocs) cudaFree(d);
  };
  cudaStream_t st = nullptr;
  if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
    set_error("cudaStreamCreate failed: no usable CUDA device (bplx has no CPU fallback)");
    return BPLX_E_CUDA;
  }
  rc = BPLX_OK;
  auto up = [&](const void* h, size_t bytes) -> void* {
    if (!h || rc != BPLX_OK) return nullptr;
    void* d = nullptr;
    if (cudaMalloc(&d, bytes) != cudaSuccess ||
        cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) {
      set_error("score_grid_host: device allocation / copy of %zu bytes failed", bytes);
      rc = BPLX_E_CUDA;
      return nullptr;
    }
    allocs.push_back(d);
    return d;
  };
  bplx_samples ds = *s;
  bplx_fixtures df = *f;
  const size_t ha_w = s->model == BPLX_DIXON_COLES ? 1 : T;
  ds.attack = (const float*)up(s->attack, S * T * 4);
  ds.defence = (const float*)up(s->defence, S * T * 4);
  ds.home_attack = (const float*)up(s->home_attack, S * ha_w * 4);
  const bool neu = s->model == BPLX_NEUTRAL || s->model == BPLX_NEUTRAL_WC;
  ds.away_attack = neu ? (const float*)up(s->away_attack, S * T * 4) : nullptr;
  ds.home_defence = neu ? (const float*)up(s->home_defence, S * T * 4) : nullptr;
  ds.away_defence = neu ? (const float*)up(s->away_defence, S * T * 4) : nullptr;
  ds.confederation_strength = Cf ? (const float*)up(s->confederation_strength, S * Cf * 4) : nullptr;
  ds.corr_coef = (const float*)up(s->corr_coef, S * 4);
  df.home_team = (const uint16_t*)up(f->home_team, F * 2);
  df.away_team = (const uint16_t*)up(f->away_team, F * 2);
  df.home_conf = Cf ? (const uint8_t*)up(f->home_conf, F) : nullptr;
  df.away_conf = Cf ? (const uint8_t*)up(f->away_conf, F) : nullptr;
  df.neutral_venue = (neu && f->neutral_venue) ? (const uint8_t*)up(f->neutral_venue, F) : nullptr;
  const size_t ws_bytes = bplx_score_grid_workspace_bytes(s, f, max_goals);
  void *d_ws = nullptr, *d_grid = nullptr, *d_out = nullptr;
  if (rc == BPLX_OK) {
    if (cudaMalloc(&d_ws, ws_bytes) == cudaSuccess) allocs.push_back(d_ws); else rc = BPLX_E_NOMEM;
    if (cudaMalloc(&d_grid, F * g * g * 4) == cudaSuccess) allocs.push_back(d_grid); else rc = BPLX_E_NOMEM;
    if (outcome) {
      if (cudaMalloc(&d_out, F * 3 * 4) == cudaSuccess) allocs.push_back(d_out); else rc = BPLX_E_NOMEM;
    }
    if (rc != BPLX_OK) set_error("score_grid_host: out of device memory");
  }
  if (rc == BPLX_OK)
    rc = bplx_score_grid(&ds, &df, max_goals, scale, (float*)d_grid, (float*)d_out, d_ws, ws_bytes, st);
  if (rc == BPLX_OK) {
    cudaError_t e = cudaMemcpyAsync(grid, d_grid, F * g * g * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && outcome) e = cudaMemcpyAsync(outcome, d_out, F * 3 * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      set_error("score_grid_host: %s", cudaGetErrorString(e));
      rc = BPLX_E_CUDA;
    }
  } else {
    cudaStreamSynchronize(st);
  }
  cleanup();
  cudaStreamDestroy(st);
  return rc;
}

// ---- pointwise log-likelihood and PSIS-LOO -----------------------------------------------------------------------
static size_t pointwise_plan_for(const bplx_samples* s, const bplx_observations* o, PointwiseParams* pp, const char** err) {
  bind_samples(s, &o->fixtures, &pp->gp);
  return pointwise_plan(pp, err);
}

size_t bplx_pointwise_loglik_workspace_bytes(const bplx_samples* s, const bplx_observations* obs) {
  if (!s || !obs || s->num_samples <= 0 || s->num_teams <= 0 || obs->fixtures.num_fixtures <= 0) return 0;
  PointwiseParams pp{};
  return pointwise_plan_for(s, obs, &pp, nullptr);
}

int bplx_pointwise_loglik(const bplx_samples* s, const bplx_observations* obs, float* loglik, size_t ld, double* stats,
                          void* workspace, size_t workspace_bytes, void* stream) {
  BPLX_REQUIRE(obs != nullptr, BPLX_E_INVALID, "observations is NULL");
  int rc = check_sample_args(s, &obs->fixtures, "pointwise log-likelihood");
  if (rc != BPLX_OK) return rc;
  BPLX_REQUIRE(obs->home_goals && obs->away_goals, BPLX_E_INVALID,
               "pointwise log-likelihood: home_goals and away_goals must not be NULL");
  BPLX_REQUIRE(stats != nullptr, BPLX_E_INVALID, "pointwise log-likelihood: stats is NULL");
  BPLX_REQUIRE(!loglik || ld >= (size_t)s->num_samples, BPLX_E_INVALID,
               "pointwise log-likelihood: ld (%zu) < num_samples (%d)", ld, s->num_samples);
  PointwiseParams pp{};
  const char* perr = nullptr;
  const size_t need = pointwise_plan_for(s, obs, &pp, &perr);
  BPLX_REQUIRE(need > 0, BPLX_E_UNSUPPORTED, "%s", perr ? perr : "pointwise log-likelihood: unsupported shape");
  rc = check_workspace(workspace, workspace_bytes, need);
  if (rc != BPLX_OK) return rc;
  pp.gp.table = static_cast<float*>(workspace);
  pp.partial = reinterpret_cast<double*>(static_cast<unsigned char*>(workspace) + table_layout(&pp.gp));
  pp.hg = obs->home_goals;
  pp.ag = obs->away_goals;
  pp.ll = loglik;
  pp.ld = ld;
  pp.stats = stats;
  return launch_pointwise(pp, static_cast<cudaStream_t>(stream));
}

int bplx_psis_loo(const float* loglik, int num_matches, int num_samples, size_t ld, double r_eff, double* elpd_i,
                  double* pareto_k, void* workspace, size_t workspace_bytes, void* stream) {
  (void)workspace;
  (void)workspace_bytes;
  BPLX_REQUIRE(loglik && elpd_i && pareto_k, BPLX_E_INVALID, "psis loo: loglik, elpd_i and pareto_k must not be NULL");
  BPLX_REQUIRE(num_matches > 0 && num_samples > 0, BPLX_E_INVALID,
               "psis loo: num_matches and num_samples must be positive (got %d, %d)", num_matches, num_samples);
  BPLX_REQUIRE(ld >= (size_t)num_samples, BPLX_E_INVALID, "psis loo: ld (%zu) < num_samples (%d)", ld, num_samples);
  BPLX_REQUIRE(r_eff > 0.0 && r_eff <= 1e300, BPLX_E_INVALID, "psis loo: r_eff must be positive and finite (got %g)", r_eff);
  PsisParams pp{};
  pp.Mt = psis_tail_length(num_samples, r_eff);
  BPLX_REQUIRE(pp.Mt <= kPsisTailMax, BPLX_E_UNSUPPORTED,
               "psis loo: a tail of %d draws (ceil(min(0.2 S, 3 sqrt(S / r_eff)))) exceeds the kernel's limit of %d "
               "(BPLX_PSIS_MAX_TAIL)", pp.Mt, kPsisTailMax);
  pp.cap = 8;
  while (pp.cap < pp.Mt) pp.cap <<= 1;
  pp.ll = loglik;
  pp.ld = ld;
  pp.M = num_matches;
  pp.S = num_samples;
  pp.elpd = elpd_i;
  pp.khat = pareto_k;
  return launch_psis(pp, static_cast<cudaStream_t>(stream));
}

// ---- season / group-stage simulation --------------------------------------------------------------------------
// the workspace of a simulation is the [S][row_floats] exponential table
static size_t simulate_plan_for(const bplx_samples* s, const bplx_fixtures* f, SimParams* sp) {
  bind_samples(s, f, &sp->gp);
  return table_layout(&sp->gp);
}

size_t bplx_simulate_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, const bplx_table* t) {
  if (!s || !f || !t || s->num_samples <= 0 || s->num_teams <= 0 || f->num_fixtures <= 0) return 0;
  SimParams sp{};
  return simulate_plan_for(s, f, &sp);
}

// validates the arguments bplx_simulate_table and bplx_simulate_tournament share and fills *sp (its samples, fixtures
// and workspace aside: simulate_plan_for binds those)
static int simulate_setup(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                          const uint8_t* away_slot, const bplx_table* t, int max_goals, int sims_per_draw,
                          unsigned long long seed, long long first_draw, unsigned long long* position_counts,
                          unsigned long long* points_counts, uint8_t* positions, uint8_t* scores,
                          unsigned long long* invalid, const char* what, bool allow_no_fixtures, SimParams* out) {
  int rc = check_sample_args(s, f, what, allow_no_fixtures);
  if (rc != BPLX_OK) return rc;
  BPLX_REQUIRE(t != nullptr, BPLX_E_INVALID, "%s: table is NULL", what);
  BPLX_REQUIRE(t->num_slots <= BPLX_SIM_MAX_TEAMS, BPLX_E_UNSUPPORTED,
               "%s: %d table slots exceed the kernel's limit of %d (BPLX_SIM_MAX_TEAMS)", what, t->num_slots,
               BPLX_SIM_MAX_TEAMS);
  BPLX_REQUIRE(t->num_slots >= 1, BPLX_E_INVALID, "%s: the table needs at least one slot", what);
  BPLX_REQUIRE(t->num_positions >= 1 && t->num_positions <= t->num_slots && t->num_points_bins >= 1, BPLX_E_INVALID,
               "%s: num_positions must be in [1, num_slots] and num_points_bins >= 1 (got %d, %d)", what,
               t->num_positions, t->num_points_bins);
  BPLX_REQUIRE(t->points_win >= 1 && t->points_draw >= 0 && t->points_draw <= t->points_win, BPLX_E_INVALID,
               "%s: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got %d, %d)", what,
               t->points_win, t->points_draw);
  BPLX_REQUIRE(t->start_points && t->start_goals_for && t->start_goals_against, BPLX_E_INVALID,
               "%s: start_points, start_goals_for and start_goals_against must not be NULL", what);
  BPLX_REQUIRE((home_slot && away_slot) || f->num_fixtures == 0, BPLX_E_INVALID,
               "%s: home_slot and away_slot must not be NULL", what);
  BPLX_REQUIRE(max_goals >= 1 && max_goals <= 63, BPLX_E_INVALID, "%s: max_goals must be in [1, 63] (got %d)", what,
               max_goals);
  BPLX_REQUIRE(sims_per_draw >= 1, BPLX_E_INVALID, "%s: sims_per_draw must be >= 1 (got %d)", what, sims_per_draw);
  BPLX_REQUIRE(first_draw >= 0 && first_draw + s->num_samples <= LLONG_MAX / sims_per_draw, BPLX_E_INVALID,
               "%s: first_draw must be >= 0 and (first_draw + num_samples) * sims_per_draw must fit 63 bits", what);
  BPLX_REQUIRE((long long)s->num_samples * sims_per_draw <= INT_MAX, BPLX_E_UNSUPPORTED,
               "%s: num_samples * sims_per_draw must be below 2^31 per call (got %lld): cut the draws into ranges",
               what, (long long)s->num_samples * sims_per_draw);
  BPLX_REQUIRE(position_counts && points_counts && invalid, BPLX_E_INVALID,
               "%s: position_counts, points_counts and invalid must not be NULL", what);
  SimParams& sp = *out;
  sp.hslot = home_slot;
  sp.aslot = away_slot;
  sp.group = t->group;
  sp.start_pts = t->start_points;
  sp.start_gf = t->start_goals_for;
  sp.start_ga = t->start_goals_against;
  sp.NT = t->num_slots;
  sp.P = t->num_positions;
  sp.B = t->num_points_bins;
  sp.G = max_goals;
  sp.R = sims_per_draw;
  sp.pw = t->points_win;
  sp.pd = t->points_draw;
  sp.seed = seed;
  sp.first_draw = first_draw;
  sp.N = s->num_samples * sims_per_draw;
  sp.pos_counts = position_counts;
  sp.pts_counts = points_counts;
  sp.invalid = invalid;
  sp.positions = positions;
  sp.scores = scores;
  return BPLX_OK;
}

// ---- ranking rules --------------------------------------------------------------------------------------------
static bool head_to_head(const bplx_ranking* r) { return r && r->rule == BPLX_RANK_HEAD_TO_HEAD; }

// workspace bytes the ranking adds after `base` (256-aligned): head-to-head keeps the played matrix [NT][NT] int2, the
// pair offsets [NT NT + 1] and the pair fixture list [F]
static size_t ranking_bytes(const bplx_ranking* r, int NT, int F) {
  if (!head_to_head(r)) return 0;
  const size_t nn = (size_t)NT * NT;
  return (nn * 8 + 255) / 256 * 256 + ((nn + 1) * 4 + 255) / 256 * 256 + ((size_t)(F > 0 ? F : 1) * 4 + 255) / 256 * 256;
}

static int check_ranking(const bplx_ranking* r, int NT, const char* what) {
  if (!r) return BPLX_OK;
  BPLX_REQUIRE(r->rule == BPLX_RANK_GOAL_DIFF || r->rule == BPLX_RANK_HEAD_TO_HEAD, BPLX_E_INVALID,
               "%s: ranking rule %d is not a BPLX_RANK_* value", what, r->rule);
  if (head_to_head(r) && r->played_h2h)
    for (int k = 0; k < NT * NT * 2; k++)
      BPLX_REQUIRE(r->played_h2h[k] >= 0, BPLX_E_INVALID,
                   "%s: played_h2h (%d, %d) has a negative %s (%d)", what, k / 2 / NT, k / 2 % NT,
                   k % 2 ? "goal count" : "points count", r->played_h2h[k]);
  return BPLX_OK;
}

// fills the head-to-head fields of *sp from the workspace region at `base` (the played matrix is copied there)
static int bind_ranking(const bplx_ranking* r, void* workspace, size_t base, SimParams* sp, cudaStream_t stream) {
  sp->rule = r ? r->rule : BPLX_RANK_GOAL_DIFF;
  if (!head_to_head(r)) return BPLX_OK;
  const size_t nn = (size_t)sp->NT * sp->NT;
  unsigned char* p = static_cast<unsigned char*>(workspace) + base;
  if (r->played_h2h) {
    BPLX_CUDA(cudaMemcpyAsync(p, r->played_h2h, nn * 8, cudaMemcpyHostToDevice, stream));
    sp->h2h_played = reinterpret_cast<const int2*>(p);
  }
  p += (nn * 8 + 255) / 256 * 256;
  sp->pair_beg = reinterpret_cast<int*>(p);
  sp->pair_fix = reinterpret_cast<int*>(p + ((nn + 1) * 4 + 255) / 256 * 256);
  return BPLX_OK;
}

size_t bplx_simulate_table_ex_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, const bplx_table* t,
                                              const bplx_ranking* r) {
  const size_t base = bplx_simulate_workspace_bytes(s, f, t);
  if (!base || (r && r->rule != BPLX_RANK_GOAL_DIFF && r->rule != BPLX_RANK_HEAD_TO_HEAD)) return 0;
  if (t->num_slots < 1 || t->num_slots > BPLX_SIM_MAX_TEAMS) return head_to_head(r) ? 0 : base;
  return base + ranking_bytes(r, t->num_slots, f->num_fixtures);
}

int bplx_simulate_table(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot, const uint8_t* away_slot,
                        const bplx_table* t, int max_goals, int sims_per_draw, unsigned long long seed,
                        long long first_draw, unsigned long long* position_counts, unsigned long long* points_counts,
                        uint8_t* positions, uint8_t* scores, unsigned long long* invalid, void* workspace,
                        size_t workspace_bytes, void* stream) {
  return bplx_simulate_table_ex(s, f, home_slot, away_slot, t, nullptr, max_goals, sims_per_draw, seed, first_draw,
                                position_counts, points_counts, positions, scores, invalid, workspace, workspace_bytes,
                                stream);
}

int bplx_simulate_table_ex(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                           const uint8_t* away_slot, const bplx_table* t, const bplx_ranking* r, int max_goals,
                           int sims_per_draw, unsigned long long seed, long long first_draw,
                           unsigned long long* position_counts, unsigned long long* points_counts, uint8_t* positions,
                           uint8_t* scores, unsigned long long* invalid, void* workspace, size_t workspace_bytes,
                           void* stream) {
  SimParams sp{};
  int rc = simulate_setup(s, f, home_slot, away_slot, t, max_goals, sims_per_draw, seed, first_draw, position_counts,
                          points_counts, positions, scores, invalid, "simulate", false, &sp);
  if (rc != BPLX_OK) return rc;
  rc = check_ranking(r, t->num_slots, "simulate");
  if (rc != BPLX_OK) return rc;
  const size_t table = simulate_plan_for(s, f, &sp);
  rc = check_workspace(workspace, workspace_bytes, table + ranking_bytes(r, t->num_slots, f->num_fixtures));
  if (rc != BPLX_OK) return rc;
  sp.gp.table = static_cast<float*>(workspace);
  rc = bind_ranking(r, workspace, table, &sp, static_cast<cudaStream_t>(stream));
  if (rc != BPLX_OK) return rc;
  return launch_simulate(sp, static_cast<cudaStream_t>(stream));
}

// ---- tournament simulation -----------------------------------------------------------------------------------
static size_t alloc_bytes(const bplx_bracket* b) {
  return b->best_alloc ? ((size_t)b->best_count << b->num_groups) : 0;
}

size_t bplx_simulate_tournament_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f, const bplx_table* t,
                                                const bplx_bracket* b) {
  if (!s || !f || !t || !b || s->num_samples <= 0 || s->num_teams <= 0 || f->num_fixtures < 0) return 0;
  if (b->num_groups < 0 || b->num_groups > BPLX_SIM_MAX_TEAMS || b->best_count < 0) return 0;
  if (b->best_alloc && b->num_groups > BPLX_KO_MAX_ALLOC_GROUPS) return 0;
  SimParams sp{};
  return simulate_plan_for(s, f, &sp) + (alloc_bytes(b) + 255) / 256 * 256;
}

// the bracket checks the kernel relies on; fills sp->ko
static int check_bracket(const bplx_bracket* b, const uint8_t* tie_format, const bplx_samples* s, int NT, int P,
                         KoParams* ko) {
  BPLX_REQUIRE(b != nullptr, BPLX_E_INVALID, "tournament: bracket is NULL");
  const int K = b->num_ties;
  BPLX_REQUIRE(K >= 1, BPLX_E_INVALID, "tournament: the bracket needs at least one tie (got %d)", K);
  BPLX_REQUIRE(K <= BPLX_KO_MAX_TIES, BPLX_E_UNSUPPORTED,
               "tournament: %d ties exceed the kernel's limit of %d (BPLX_KO_MAX_TIES)", K, BPLX_KO_MAX_TIES);
  BPLX_REQUIRE(b->num_rounds >= 1 && b->num_rounds <= BPLX_KO_MAX_ROUNDS, BPLX_E_UNSUPPORTED,
               "tournament: num_rounds must be in [1, %d] (got %d)", BPLX_KO_MAX_ROUNDS, b->num_rounds);
  BPLX_REQUIRE(b->num_groups >= 0 && b->num_groups <= NT, BPLX_E_INVALID,
               "tournament: num_groups must be in [0, num_slots] (got %d)", b->num_groups);
  BPLX_REQUIRE(b->best_count >= 0 && b->best_count <= BPLX_KO_MAX_BEST, BPLX_E_UNSUPPORTED,
               "tournament: best_count must be in [0, %d] (got %d)", BPLX_KO_MAX_BEST, b->best_count);
  BPLX_REQUIRE(b->best_count <= b->num_groups, BPLX_E_INVALID,
               "tournament: best_count (%d) exceeds num_groups (%d)", b->best_count, b->num_groups);
  BPLX_REQUIRE(b->best_count == 0 || (b->best_position >= 0 && b->best_position < P), BPLX_E_INVALID,
               "tournament: best_position must be in [0, num_positions) (got %d)", b->best_position);
  BPLX_REQUIRE(b->kind && b->arg0 && b->arg1 && b->round && b->slot_team, BPLX_E_INVALID,
               "tournament: kind, arg0, arg1, round and slot_team must not be NULL");
  BPLX_REQUIRE(s->model != BPLX_NEUTRAL_WC || b->slot_conf, BPLX_E_INVALID, "tournament: NEUTRAL_WC needs slot_conf");
  for (int t = 0; t < NT; t++) {
    BPLX_REQUIRE(b->slot_team[t] < s->num_teams, BPLX_E_INVALID,
                 "tournament: slot_team[%d] = %d is not a model team (T = %d)", t, b->slot_team[t], s->num_teams);
    if (s->model == BPLX_NEUTRAL_WC)
      BPLX_REQUIRE(b->slot_conf[t] < s->num_conferences, BPLX_E_INVALID,
                   "tournament: slot_conf[%d] = %d is not a confederation (Cf = %d)", t, b->slot_conf[t],
                   s->num_conferences);
  }
  for (int k = 0; k < K; k++) {
    BPLX_REQUIRE(b->round[k] < b->num_rounds, BPLX_E_INVALID, "tournament: tie %d: round %d >= num_rounds (%d)", k,
                 b->round[k], b->num_rounds);
    for (int side = 0; side < 2; side++) {
      const int kind = b->kind[2 * k + side], a0 = b->arg0[2 * k + side], a1 = b->arg1[2 * k + side];
      const char* sd = side ? "away" : "home";
      switch (kind) {
        case BPLX_ENTRANT_SLOT:
          BPLX_REQUIRE(a0 < NT, BPLX_E_INVALID, "tournament: tie %d %s: slot %d outside the table (%d slots)", k, sd,
                       a0, NT);
          break;
        case BPLX_ENTRANT_GROUP_POS:
          BPLX_REQUIRE(a0 < b->num_groups && a1 < P, BPLX_E_INVALID,
                       "tournament: tie %d %s: group %d position %d out of range (%d groups, %d positions)", k, sd, a0,
                       a1, b->num_groups, P);
          break;
        case BPLX_ENTRANT_BEST:
          BPLX_REQUIRE(a0 < b->best_count, BPLX_E_INVALID, "tournament: tie %d %s: BEST %d >= best_count (%d)", k, sd,
                       a0, b->best_count);
          break;
        case BPLX_ENTRANT_WINNER:
        case BPLX_ENTRANT_LOSER:
          BPLX_REQUIRE(a0 < k, BPLX_E_INVALID, "tournament: tie %d %s: refers to tie %d, which is not earlier", k, sd,
                       a0);
          break;
        default:
          BPLX_REQUIRE(false, BPLX_E_INVALID, "tournament: tie %d %s: unknown entrant kind %d", k, sd, kind);
      }
      ko->kind[side][k] = (uint8_t)kind;
      ko->arg0[side][k] = (uint8_t)a0;
      ko->arg1[side][k] = (uint8_t)a1;
    }
    ko->round[k] = b->round[k];
    ko->neutral[k] = b->neutral_venue ? (b->neutral_venue[k] != 0) : 0;
    ko->format[k] = tie_format ? tie_format[k] : BPLX_TIE_ONE_MATCH;
    BPLX_REQUIRE(ko->format[k] <= BPLX_TIE_TWO_LEGS, BPLX_E_INVALID,
                 "tournament: tie %d: format %d is not a BPLX_TIE_* value", k, ko->format[k]);
    BPLX_REQUIRE(ko->format[k] != BPLX_TIE_TWO_LEGS || !ko->neutral[k], BPLX_E_INVALID,
                 "tournament: tie %d: a two-legged tie cannot be at a neutral venue", k);
  }
  if (b->best_alloc) {
    BPLX_REQUIRE(b->best_count >= 1, BPLX_E_INVALID, "tournament: an allocation table needs best_count >= 1");
    BPLX_REQUIRE(b->num_groups <= BPLX_KO_MAX_ALLOC_GROUPS, BPLX_E_UNSUPPORTED,
                 "tournament: an allocation table supports at most %d groups (got %d)", BPLX_KO_MAX_ALLOC_GROUPS,
                 b->num_groups);
    for (unsigned mask = 0; mask < (1u << b->num_groups); mask++) {
      unsigned seen = 0;
      for (int j = 0; j < b->best_count; j++) {
        const int g = b->best_alloc[(size_t)mask * b->best_count + j];
        if (g == 0xFF) continue;
        BPLX_REQUIRE(g < b->num_groups && ((mask >> g) & 1u) && !((seen >> g) & 1u), BPLX_E_INVALID,
                     "tournament: allocation row 0x%x entry %d: group %d is not a distinct group of the row's set", mask,
                     j, g);
        seen |= 1u << g;
      }
    }
  }
  for (int t = 0; t < NT; t++) {
    ko->slot_team[t] = b->slot_team[t];
    ko->slot_conf[t] = b->slot_conf ? b->slot_conf[t] : 0;
  }
  ko->K = K;
  ko->nr = b->num_rounds;
  ko->ng = b->num_groups;
  ko->bp = b->best_position;
  ko->bc = b->best_count;
  return BPLX_OK;
}

size_t bplx_simulate_tournament_ranked_workspace_bytes(const bplx_samples* s, const bplx_fixtures* f,
                                                       const bplx_table* t, const bplx_bracket* b,
                                                       const bplx_ranking* r) {
  const size_t base = bplx_simulate_tournament_workspace_bytes(s, f, t, b);
  if (!base || (r && r->rule != BPLX_RANK_GOAL_DIFF && r->rule != BPLX_RANK_HEAD_TO_HEAD)) return 0;
  if (t->num_slots < 1 || t->num_slots > BPLX_SIM_MAX_TEAMS) return head_to_head(r) ? 0 : base;
  return base + ranking_bytes(r, t->num_slots, f->num_fixtures);
}

int bplx_simulate_tournament_ex(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                                const uint8_t* away_slot, const bplx_table* t, const bplx_bracket* b,
                                const uint8_t* tie_format, int max_goals, int sims_per_draw, unsigned long long seed,
                                long long first_draw, unsigned long long* position_counts,
                                unsigned long long* points_counts, unsigned long long* reach_counts,
                                unsigned long long* win_counts, unsigned long long* decided_counts, uint8_t* positions,
                                uint8_t* scores, uint8_t* ko_entrants, uint8_t* ko_scores, uint8_t* ko_winners,
                                uint8_t* ko_extra, unsigned long long* invalid, void* workspace,
                                size_t workspace_bytes, void* stream) {
  return bplx_simulate_tournament_ranked(s, f, home_slot, away_slot, t, b, tie_format, nullptr, max_goals,
                                         sims_per_draw, seed, first_draw, position_counts, points_counts, reach_counts,
                                         win_counts, decided_counts, positions, scores, ko_entrants, ko_scores,
                                         ko_winners, ko_extra, invalid, workspace, workspace_bytes, stream);
}

int bplx_simulate_tournament_ranked(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                                    const uint8_t* away_slot, const bplx_table* t, const bplx_bracket* b,
                                    const uint8_t* tie_format, const bplx_ranking* r, int max_goals, int sims_per_draw,
                                    unsigned long long seed, long long first_draw, unsigned long long* position_counts,
                                    unsigned long long* points_counts, unsigned long long* reach_counts,
                                    unsigned long long* win_counts, unsigned long long* decided_counts,
                                    uint8_t* positions, uint8_t* scores, uint8_t* ko_entrants, uint8_t* ko_scores,
                                    uint8_t* ko_winners, uint8_t* ko_extra, unsigned long long* invalid,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  SimParams sp{};
  int rc = simulate_setup(s, f, home_slot, away_slot, t, max_goals, sims_per_draw, seed, first_draw, position_counts,
                          points_counts, positions, scores, invalid, "tournament", true, &sp);
  if (rc != BPLX_OK) return rc;
  rc = check_bracket(b, tie_format, s, t->num_slots, t->num_positions, &sp.ko);
  if (rc != BPLX_OK) return rc;
  BPLX_REQUIRE(reach_counts && win_counts, BPLX_E_INVALID, "tournament: reach_counts and win_counts must not be NULL");
  rc = check_ranking(r, t->num_slots, "tournament");
  if (rc != BPLX_OK) return rc;
  const size_t table = simulate_plan_for(s, f, &sp), alloc = (alloc_bytes(b) + 255) / 256 * 256;
  rc = check_workspace(workspace, workspace_bytes, table + alloc + ranking_bytes(r, t->num_slots, f->num_fixtures));
  if (rc != BPLX_OK) return rc;
  rc = bind_ranking(r, workspace, table + alloc, &sp, static_cast<cudaStream_t>(stream));
  if (rc != BPLX_OK) return rc;
  sp.gp.table = static_cast<float*>(workspace);
  sp.ko.reach = reach_counts;
  sp.ko.win = win_counts;
  sp.ko.decided = decided_counts;
  sp.ko.entrants = ko_entrants;
  sp.ko.scores = ko_scores;
  sp.ko.winners = ko_winners;
  sp.ko.extra = ko_extra;
  if (b->best_alloc) {
    uint8_t* const dst = static_cast<uint8_t*>(workspace) + table;
    BPLX_CUDA(cudaMemcpyAsync(dst, b->best_alloc, alloc_bytes(b), cudaMemcpyHostToDevice,
                              static_cast<cudaStream_t>(stream)));
    sp.ko.alloc = dst;
  }
  return launch_simulate(sp, static_cast<cudaStream_t>(stream));
}

int bplx_simulate_tournament(const bplx_samples* s, const bplx_fixtures* f, const uint8_t* home_slot,
                             const uint8_t* away_slot, const bplx_table* t, const bplx_bracket* b, int max_goals,
                             int sims_per_draw, unsigned long long seed, long long first_draw,
                             unsigned long long* position_counts, unsigned long long* points_counts,
                             unsigned long long* reach_counts, unsigned long long* win_counts, uint8_t* positions,
                             uint8_t* scores, uint8_t* ko_entrants, uint8_t* ko_scores, uint8_t* ko_winners,
                             unsigned long long* invalid, void* workspace, size_t workspace_bytes, void* stream) {
  return bplx_simulate_tournament_ex(s, f, home_slot, away_slot, t, b, nullptr, max_goals, sims_per_draw, seed,
                                     first_draw, position_counts, points_counts, reach_counts, win_counts, nullptr,
                                     positions, scores, ko_entrants, ko_scores, ko_winners, nullptr, invalid, workspace,
                                     workspace_bytes, stream);
}

// ---- posterior predictive checks ------------------------------------------------------------------------------
// the workspace is the [S][row_floats] exponential table, as for a simulation
size_t bplx_posterior_predictive_workspace_bytes(const bplx_samples* s, const bplx_observations* obs) {
  if (!s || !obs || s->num_samples <= 0 || s->num_teams <= 0 || obs->fixtures.num_fixtures <= 0) return 0;
  GridParams gp{};
  bind_samples(s, &obs->fixtures, &gp);
  return table_layout(&gp);
}

int bplx_posterior_predictive(const bplx_samples* s, const bplx_observations* obs, int max_goals, int score_bins,
                              int points_win, int points_draw, int sims_per_draw, unsigned long long seed,
                              long long first_draw, const bplx_ppc_output* out, void* workspace,
                              size_t workspace_bytes, void* stream) {
  const char* what = "posterior predictive";
  BPLX_REQUIRE(obs != nullptr && out != nullptr, BPLX_E_INVALID, "%s: observations / out is NULL", what);
  int rc = check_sample_args(s, &obs->fixtures, what);
  if (rc != BPLX_OK) return rc;
  const int M = obs->fixtures.num_fixtures;
  BPLX_REQUIRE(obs->home_goals && obs->away_goals, BPLX_E_INVALID, "%s: home_goals and away_goals must not be NULL",
               what);
  BPLX_REQUIRE(max_goals >= 1 && max_goals <= 63, BPLX_E_INVALID, "%s: max_goals must be in [1, 63] (got %d)", what,
               max_goals);
  BPLX_REQUIRE(score_bins >= 2 && score_bins <= 16, BPLX_E_INVALID, "%s: score_bins must be in [2, 16] (got %d)", what,
               score_bins);
  BPLX_REQUIRE(points_win >= 1 && points_draw >= 0 && points_draw <= points_win, BPLX_E_INVALID,
               "%s: points must satisfy 0 <= points_draw <= points_win, points_win >= 1 (got %d, %d)", what,
               points_win, points_draw);
  BPLX_REQUIRE((long long)std::max(points_win, max_goals) * M <= INT_MAX, BPLX_E_INVALID,
               "%s: max(points_win, max_goals) * num_matches must be below 2^31 (a team count could overflow)", what);
  BPLX_REQUIRE(sims_per_draw >= 1, BPLX_E_INVALID, "%s: sims_per_draw must be >= 1 (got %d)", what, sims_per_draw);
  BPLX_REQUIRE(first_draw >= 0 && first_draw + s->num_samples <= LLONG_MAX / sims_per_draw, BPLX_E_INVALID,
               "%s: first_draw must be >= 0 and (first_draw + num_samples) * sims_per_draw must fit 63 bits", what);
  BPLX_REQUIRE((long long)s->num_samples * sims_per_draw <= INT_MAX, BPLX_E_UNSUPPORTED,
               "%s: num_samples * sims_per_draw must be below 2^31 per call (got %lld): cut the draws into ranges",
               what, (long long)s->num_samples * sims_per_draw);
  BPLX_REQUIRE(out->score_counts && out->outcome_counts && out->goals && out->total_goals_sq && out->team_points &&
                   out->team_goals_for && out->team_goals_against && out->invalid,
               BPLX_E_INVALID, "%s: every output but scores must be given", what);
  PpcParams pp{};
  bind_samples(s, &obs->fixtures, &pp.gp);
  rc = check_workspace(workspace, workspace_bytes, table_layout(&pp.gp));
  if (rc != BPLX_OK) return rc;
  pp.gp.table = static_cast<float*>(workspace);
  pp.G = max_goals;
  pp.B = score_bins;
  pp.R = sims_per_draw;
  pp.pw = points_win;
  pp.pd = points_draw;
  pp.seed = seed;
  pp.first_draw = first_draw;
  pp.N = s->num_samples * sims_per_draw;
  pp.score_counts = out->score_counts;
  pp.outcome_counts = out->outcome_counts;
  pp.goals = reinterpret_cast<long long*>(out->goals);
  pp.total_goals_sq = reinterpret_cast<long long*>(out->total_goals_sq);
  pp.team_points = out->team_points;
  pp.team_goals_for = out->team_goals_for;
  pp.team_goals_against = out->team_goals_against;
  pp.scores = out->scores;
  pp.invalid = out->invalid;
  return launch_ppc(pp, static_cast<cudaStream_t>(stream));
}

void bplx_reload_env(void) {
  env_switches();
  reload_env_switches();
}
const char* bplx_last_error(void) { return g_err; }
int bplx_version(void) { return BPLX_VERSION; }
unsigned long long bplx_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

}  // extern "C"
