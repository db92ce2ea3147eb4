// simulate_cond.cu -- season and group-stage simulation with match importance: the table kernel of simulate.cu, plus
// each simulation's key-fixture outcomes and events counted jointly (bplx_conditions, include/bplx.h).
//
// Definition (the same text in include/bplx.h, oracle/conditional.py and the docstrings):
//   key fixture j (an index into the call's F fixtures) has outcome o in {0 home win, 1 draw, 2 away win} from its
//   sampled score (hg > ag, hg = ag, hg < ag); event e = (slot t_e, position mask M_e) holds iff t_e's position within
//   its group is a bit of M_e.  outcome_counts [Kc, 3]: valid simulations in which key fixture j ended in o;
//   conditional_counts [Kc, 3, E]: valid simulations in which key fixture j ended in o and event e held.  Invalid
//   simulations are left out exactly as from position_counts.  No Philox word is added or moved: every other output is
//   bplx_simulate_table_ex's, bit for bit.
//
// Kernel: simulate_body.inc with BPLX_SIM_COND defined, under either ranking rule.  Each thread keeps two uint64 of outcome bits
// (home win, draw; set as the fixture loop passes each key fixture: the keys are sorted, so one warp-uniform cursor
// suffices) and one uint64 of event bits (set where a slot's position is known, from a per-CTA table of the events of
// each slot).  After the CTA's simulations: per warp, E ballots of the event bits (lane l keeps events l and l + 32);
// per key fixture, the outcome ballots, popc(outcome & event) per lane into per-warp partial counts in the dead
// accumulators, one barrier, then the four warps summed and flushed with 64-bit atomics, zeros skipped.  The kernel is
// in a translation unit of its own: instantiated beside the others, it changed their instructions.
#include "simulate.h"

#include "sample_score.cuh"

#include "simulate_device.cuh"

namespace bplx {

// the events that hold with slot t at position pos, from the per-CTA tables at c_tab (the
// events of each slot [64], then the positions of each event [64])
__device__ __forceinline__ unsigned long long events_at(const unsigned char* c_tab, int t, int pos) {
  const unsigned long long* const tab = reinterpret_cast<const unsigned long long*>(c_tab);
  unsigned long long ev = 0;
  for (unsigned long long m = tab[t]; m; m &= m - 1) {
    const int e = __ffsll((long long)m) - 1;
    ev |= ((tab[kSimMaxTeams + e] >> pos) & 1ull) << e;
  }
  return ev;
}


// the season / group stage with key-fixture outcomes and events counted jointly, under either ranking rule
template <bool H2H_RULE>
__global__ void __launch_bounds__(kSimThreads) simulate_cond_kernel(const __grid_constant__ SimParams sp) {
  constexpr bool KO = false, H2H = H2H_RULE, PAIRED = false;
  static_assert(kSimThreads == 128, "the conditional counts sum four warps");
#define BPLX_SIM_COND
#include "simulate_body.inc"
#undef BPLX_SIM_COND
}

int launch_simulate_cond(const SimParams& sp, unsigned grid, size_t smem, cudaStream_t stream) {
  const int rc = upload_sim_constants();  // (this translation unit's copy)
  if (rc != BPLX_OK) return rc;
  static void (*const kernels[2])(const SimParams) = {simulate_cond_kernel<false>, simulate_cond_kernel<true>};
  static size_t smem_set[2] = {48 * 1024, 48 * 1024};
  const int v = sp.rule == BPLX_RANK_HEAD_TO_HEAD;
  if (smem > smem_set[v]) {
    BPLX_CUDA(cudaFuncSetAttribute(kernels[v], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    smem_set[v] = smem;
  }
  kernels[v]<<<grid, kSimThreads, smem, stream>>>(sp);
  BPLX_CUDA(cudaGetLastError());
  note_launch(1);
  return BPLX_OK;
}

}  // namespace bplx
