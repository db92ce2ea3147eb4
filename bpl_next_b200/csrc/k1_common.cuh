// k1_common.cuh -- device helpers shared by the log-density kernels (logdensity.cu, logdensity_dynamic.cu).
#pragma once
#include <float.h>

#include "common.cuh"
#include "plan.h"

namespace bplx {

namespace {


constexpr float kLn2 = 0.693147180559945309f;
constexpr unsigned kFull = 0xffffffffu;

struct Hyp {  // constrained hyper-parameters of this lane's chain
  float mu_d, sig_a, sig_d, mu[4], sig[4];
};

struct Lane {
  const float* th;  // theta + chain * sc
  float* gr;        // grad  + chain * sc
  float* sc;        // scratch + chain
  int sd;
  bool active;
  __device__ __forceinline__ float ld(int d) const { return __ldg(th + (uint32_t)(d * sd)); }
  __device__ __forceinline__ float* g(int d) const { return gr + (uint32_t)(d * sd); }
};

__device__ __forceinline__ float sigmoid_clipped(float x) {
  // numpyro SigmoidTransform: clip(expit(x), finfo.tiny, 1 - finfo.eps)
  float s = 1.0f / (1.0f + expf(-x));
  return fminf(fmaxf(s, FLT_MIN), 1.0f - FLT_EPSILON);
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void red_add(float* p, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ float ld_cg(const float* p) { return __ldcg(p); }  // L2 only: the line is red.add'ed

// (two steps, so that a kernel can issue the loads early and do the exponentials when it needs the values)
__device__ __forceinline__ Hyp load_hyp_raw(const KernelParams& kp, const Lane& ln) {
  const ThetaOffsets& o = kp.off;
  Hyp hy;
  if (kp.lik_only) {  // constrained tables come in: identity location / scale (log std = 0)
    hy.mu_d = hy.sig_a = hy.sig_d = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      hy.mu[i] = o.mean[i] >= 0 ? ln.ld(o.mean[i]) : 0.0f;
      hy.sig[i] = 0.0f;
    }
    return hy;
  }
  hy.mu_d = ln.ld(o.mean_defence);
  hy.sig_a = ln.ld(o.log_std_attack);
  hy.sig_d = ln.ld(o.log_std_defence);
#pragma unroll
  for (int i = 0; i < 4; i++) {
    hy.mu[i] = o.mean[i] >= 0 ? ln.ld(o.mean[i]) : 0.0f;
    hy.sig[i] = o.log_std[i] >= 0 ? ln.ld(o.log_std[i]) : 0.0f;
  }
  return hy;
}
__device__ __forceinline__ Hyp finish_hyp(const KernelParams& kp, Hyp hy) {
  const ThetaOffsets& o = kp.off;
  hy.sig_a = expf(hy.sig_a);
  hy.sig_d = expf(hy.sig_d);
#pragma unroll
  for (int i = 0; i < 4; i++) hy.sig[i] = (o.log_std[i] >= 0 || (kp.lik_only && i < kp.ndec)) ? expf(hy.sig[i]) : 0.0f;
  return hy;
}
__device__ __forceinline__ Hyp load_hyp(const KernelParams& kp, const Lane& ln) { return finish_hyp(kp, load_hyp_raw(kp, ln)); }

struct Hdr {
  uint32_t own_off, vteam, kind, flags, n0, n1, n2, team;
};
__device__ __forceinline__ Hdr unpack_hdr(const uint4 h) {
  Hdr H;
  H.own_off = h.x;
  H.vteam = h.y & 0xffffu;
  H.kind = (h.y >> 16) & 0xffu;
  H.flags = h.y >> 24;
  H.n0 = h.z & 0xffffu;
  H.n1 = h.z >> 16;
  H.n2 = h.w & 0xffffu;
  H.team = h.w >> 16;
  return H;
}

__device__ __forceinline__ void add_own(float (&g)[6], uint32_t kind, float gx, float gy) {
  if (kind == kH1) {
    g[eAh1] += gx; g[eBh1] += gy;
  } else if (kind == kA1) {
    g[eBa1] += gx; g[eAa1] += gy;
  } else {
    g[eB0] += gx; g[eA0] += gy;
  }
}

// exponent gradients of a team -> its raw slots (d/d att, d/d def, d/d venue effects).
// ADD = false: first touch (phase 1), plain stores.  ADD = true: red.add.
template <bool ADD>
__device__ __forceinline__ void put_raw(const KernelParams& kp, const Lane& ln, int t, const float (&g)[6], float& hacc) {
  const ThetaOffsets& o = kp.off;
  const float ra = g[eAh1] + g[eAa1] + g[eA0];
  const float rd = -(g[eBh1] + g[eBa1] + g[eB0]);
  const float rx[4] = {g[eAh1], g[eAa1], -g[eBh1], -g[eBa1]};
  if (kp.ndec == 0) hacc += rx[0];  // DIXON_COLES: scalar home advantage
  if (!ln.active) return;
  if (ADD) {
    red_add(ln.g(o.za + t), ra);
    red_add(ln.g(o.zd + t), rd);
  } else {
    *ln.g(o.za + t) = ra;
    *ln.g(o.zd + t) = rd;
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    if (i < kp.ndec) {
      if (ADD) red_add(ln.g(o.dec[i] + t), rx[i]);
      else *ln.g(o.dec[i] + t) = rx[i];
    }
  }
}

// the same sums of one side's tau lists, stored to that side's shared-memory slots (slot i of a chain at q[i * 32])
__device__ __forceinline__ void put_side(const KernelParams& kp, float* q, const float (&g)[6], float& hacc) {
  q[0] = g[eAh1] + g[eAa1] + g[eA0];
  q[32] = -(g[eBh1] + g[eBa1] + g[eB0]);
  const float rx[4] = {g[eAh1], g[eAa1], -g[eBh1], -g[eBa1]};
  if (kp.ndec == 0) hacc += rx[0];
#pragma unroll
  for (int i = 0; i < 4; i++)
    if (i < kp.ndec) q[(2 + i) * 32] = rx[i];
}

// Per-warp TMA ring over a contiguous global byte stream (the warp's list pieces of one phase).
// One elected lane issues cp.async.bulk copies of one stage into the warp's private ring and every
// lane waits on the stage's mbarrier before reading it; the same warp produces and consumes, so a
// __syncwarp() is all that is needed before a slot is refilled.  Pieces never straddle a stage.
struct Ring {
  uint32_t ring, bar;        // shared addresses: kStages stages, kStages mbarriers
  uint32_t S;                // stage bytes
  const unsigned char* src;  // current stream
  uint32_t total;            // bytes in the current stream
  uint32_t gs0, gs_next;     // ring-stage counter at the start of / after the current stream
  int lane;

  __device__ __forceinline__ void init(uint32_t ring_, uint32_t bar_, uint32_t S_, int lane_) {
    ring = ring_; bar = bar_; S = S_; lane = lane_;
    total = gs0 = gs_next = 0;
    src = nullptr;
    if (lane == 0) {
#pragma unroll
      for (int s = 0; s < kStages; s++) mbar_init(bar + 8 * s, 1);
      fence_mbar_init();
      fence_proxy_async();
    }
    __syncwarp();
  }
  __device__ __forceinline__ void issue(uint32_t k) {  // stage k of the current stream
    const uint32_t b0 = k * S;
    if (lane == 0 && b0 < total) {
      const uint32_t bytes = min(S, total - b0);
      const uint32_t slot = (gs0 + k) % kStages;
      mbar_arrive_expect_tx(bar + 8 * slot, bytes);
      tma_load_1d(ring + slot * S, src + b0, bytes, bar + 8 * slot);
    }
  }
  __device__ __forceinline__ void begin(const void* src_, uint32_t total_bytes) {
    __syncwarp();  // every lane is done with the previous stream's stages
    src = static_cast<const unsigned char*>(src_);
    total = total_bytes;
    gs0 = gs_next;
    gs_next = gs0 + (total_bytes + S - 1) / S;
#pragma unroll
    for (int s = 0; s < kStages; s++) issue(s);
  }
  __device__ __forceinline__ uint32_t num_stages() const { return (total + S - 1) / S; }
  // waits for stage k; returns its shared address, *bytes = its size
  __device__ __forceinline__ uint32_t acquire(uint32_t k, uint32_t* bytes) {
    const uint32_t idx = gs0 + k, slot = idx % kStages;
    mbar_wait(bar + 8 * slot, (idx / kStages) & 1);
    *bytes = min(S, total - k * S);
    return ring + slot * S;
  }
  __device__ __forceinline__ void release(uint32_t k) {
    __syncwarp();
    issue(k + kStages);
  }
};

// Walks the 16-byte items of a list piece: four per trip, then at most one block of two and one single -- every block
// straight-line code.  (The compiler's own remainder of an unrolled loop is a rolled loop that costs three times as
// many instructions per item, and with lists of 20-90 entries a quarter of phase 1 ran in it.)
template <typename F>
__device__ __forceinline__ void walk16(uint32_t& a, const uint32_t e_end, F&& item) {
  while (a + 64 <= e_end) {
    item(a);
    item(a + 16);
    item(a + 32);
    item(a + 48);
    a += 64;
  }
  if (a + 32 <= e_end) {
    item(a);
    item(a + 16);
    a += 32;
  }
  if (a < e_end) {
    item(a);
    a += 16;
  }
}

// The tau terms of one phase-2 piece (bpl/_util.py:54-91): entries with tau = 1 - c X Y, then 1 + c X, then 1 + c Y.
//   *lt  sum w log2 tau;  *du  d/d corr_coef;  *gx, *gy  d/d (log X, log Y) of the list's own team
// kTauPlain: model without rate clipping.  kTauClipped: rates clipped at 15 (DIXON_COLES, EXTENDED).  kTauUnclipped:
// same model, but the chain maxima say no rate of these 32 chains is at the clip -- the clipped arithmetic with
// min(x, 15) = x and every guard true, bit for bit, minus the instructions.
enum { kTauPlain = 0, kTauUnclipped = 1, kTauClipped = 2 };
template <int MODE>
__device__ __forceinline__ void tau_terms(uint32_t& a, const Hdr& L, const float2 own, const bool home, const float cc,
                                          const uint32_t tab, float& lt_out, float& du_out, float& gx_out, float& gy_out) {
  // every 16 bytes hold two entries (opponent row offset, w): their arithmetic runs as packed pairs (.x = first entry)
  const float2 one = make_float2(1.0f, 1.0f);
  float2 lt = make_float2(0.0f, 0.0f), uxy = lt, sxy_x = lt, sxy_y = lt;
  {
    const uint32_t e_end = a + L.n0 * (uint32_t)sizeof(Entry);
#pragma unroll 2
    for (; a < e_end; a += 16) {
      const uint4 q = lds128u(a);
      const float2 ea = lds64(tab + q.x), eb = lds64(tab + q.z);
      const float2 w = make_float2(__uint_as_float(q.y), __uint_as_float(q.w));
      // the two rates first, then their product, as the reference groups it: (own.x own.y) (ea.x ea.y) overflows far
      // from the typical set where the rates themselves do not
      const float2 ra = mul2(own, ea), rb = mul2(own, eb);
      float2 t;
      if (MODE == kTauClipped) t = make_float2(fminf(ra.x, 15.0f) * fminf(ra.y, 15.0f), fminf(rb.x, 15.0f) * fminf(rb.y, 15.0f));
      else t = make_float2(ra.x * ra.y, rb.x * rb.y);
      float2 tau = fma2(bc2(-cc), t, one);
      tau.x = fmaxf(tau.x, 0.0f);
      tau.y = fmaxf(tau.y, 0.0f);
      // sums of (w t) / tau as explicit fused multiply-adds, packed or scalar: the same rounding in every form (left
      // as mul + add, ptxas contracts the packed pair into an FFMA2 in one form and not in another)
      const float2 wt = mul2(w, t), rc = make_float2(rcp_approx(tau.x), rcp_approx(tau.y));
      uxy = fma2(wt, rc, uxy);
      if (MODE == kTauClipped) {
        if (ra.x < 15.0f) sxy_x.x = fmaf(wt.x, rc.x, sxy_x.x);
        if (rb.x < 15.0f) sxy_x.y = fmaf(wt.y, rc.y, sxy_x.y);
        if (ra.y < 15.0f) sxy_y.x = fmaf(wt.x, rc.x, sxy_y.x);
        if (rb.y < 15.0f) sxy_y.y = fmaf(wt.y, rc.y, sxy_y.y);
      }
      if (home) lt = fma2(w, make_float2(lg2_approx(tau.x), lg2_approx(tau.y)), lt);
    }
  }
  float u1[2] = {0.0f, 0.0f}, s1[2] = {0.0f, 0.0f};
#pragma unroll
  for (int c = 0; c < 2; c++) {
    const float oc = c == 0 ? own.x : own.y;
    const uint32_t e_end = a + (c == 0 ? L.n1 : L.n2) * (uint32_t)sizeof(Entry);
    float2 u = make_float2(0.0f, 0.0f), sm = u;
#pragma unroll 2
    for (; a < e_end; a += 16) {
      const uint4 q = lds128u(a);
      const float2 Rr = mul2(bc2(oc), make_float2(lds32(tab + q.x), lds32(tab + q.z)));  // `off` already selects .x or .y
      const float2 w = make_float2(__uint_as_float(q.y), __uint_as_float(q.w));
      const float2 R = MODE == kTauClipped ? make_float2(fminf(Rr.x, 15.0f), fminf(Rr.y, 15.0f)) : Rr;
      float2 tau = fma2(bc2(cc), R, one);
      tau.x = fmaxf(tau.x, 0.0f);
      tau.y = fmaxf(tau.y, 0.0f);
      const float2 wr = mul2(w, R), rc = make_float2(rcp_approx(tau.x), rcp_approx(tau.y));
      u = fma2(wr, rc, u);
      if (MODE == kTauClipped) {
        if (Rr.x < 15.0f) sm.x = fmaf(wr.x, rc.x, sm.x);
        if (Rr.y < 15.0f) sm.y = fmaf(wr.y, rc.y, sm.y);
      }
      if (home) lt = fma2(w, make_float2(lg2_approx(tau.x), lg2_approx(tau.y)), lt);
    }
    u1[c] = u.x + u.y;
    s1[c] = MODE == kTauClipped ? sm.x + sm.y : u1[c];
  }
  const float uxy_s = uxy.x + uxy.y;
  const float sx = MODE == kTauClipped ? sxy_x.x + sxy_x.y : uxy_s, sy = MODE == kTauClipped ? sxy_y.x + sxy_y.y : uxy_s;
  lt_out = lt.x + lt.y;
  du_out = u1[0] + u1[1] - uxy_s;
  gx_out = cc * (s1[0] - sx);
  gy_out = cc * (s1[1] - sy);
}
// Home and away lists get their own copy of the walk, with `home` a constant: an away list then issues none of the
// predicated-off MUFU.LG2 / FFMA2 that one shared walk carries through it (2 + 1 issue slots per item).  Same arithmetic,
// same bits.
template <int MODE>
__device__ __forceinline__ void tau_piece(uint32_t& a, const Hdr& L, const float2 own, const bool home, const float cc,
                                          const uint32_t tab, float& lt_out, float& du_out, float& gx_out, float& gy_out) {
  if (home) tau_terms<MODE>(a, L, own, true, cc, tab, lt_out, du_out, gx_out, gy_out);
  else tau_terms<MODE>(a, L, own, false, cc, tab, lt_out, du_out, gx_out, gy_out);
}

// the two arg-max matches of a chain (SURVEY Appendix B.3), as every warp needs them in the team pass
struct Fixup {
  uint32_t teams[2];  // per which: own team | opp team << 16 (0xffff = none)
  uint32_t confs;     // 4 x 8 bits: (which, side) -> confederation (WC)
  uint32_t vts[2];    // per which: own vteam | opp vteam << 16
  float vx[2], vy[2]; // gradient reaching the X / Y log-rate of the arg-max match
  uint32_t h1;        // bit which: the list kind is H1 (else H0)
};

// d/d (att, def, venue effects) of team t gets the fix-up of (which, side) when it is that match's team
__device__ __forceinline__ void fold_fixup(const Fixup& fx, int which, int side, float& ra, float& rd, float (&rx)[4]) {
  const bool h1 = (fx.h1 >> which) & 1u;
  const float vx = fx.vx[which], vy = fx.vy[which];
  if (side == 0) {
    if (h1) { ra += vx; rx[0] += vx; rd -= vy; rx[2] -= vy; }  // X -> A_h1, Y -> B_h1
    else { rd -= vx; ra += vy; }                                 // X -> B_0,  Y -> A_0
  } else {
    if (h1) { rd -= vx; rx[3] -= vx; ra += vy; rx[1] += vy; }  // X -> B_a1, Y -> A_a1
    else { ra += vx; rd -= vy; }                                 // X -> A_0,  Y -> B_0
  }
}
__device__ __forceinline__ float fixup_conf(const Fixup& fx, int which, int side) {  // d/d (A - B)
  const bool h1 = (fx.h1 >> which) & 1u;
  const float d = fx.vx[which] - fx.vy[which];
  return ((side == 0) == h1) ? d : -d;
}

}  // namespace

}  // namespace bplx
