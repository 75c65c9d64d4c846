// env_rules.cuh — the per-instance environment transition, shared by the API-mode step kernel
// (env.cu) and the decode loops of the rollout (rollout_env_step, rollout.cuh) so both run identical rules.
//
// Reference semantics (SURVEY App. A.1):
//   step:  visited[a]=1 (tsp.py:86); r = -||xy[cur]-xy[a]|| (tsp.py:98, vrp_graph.py:137-146);
//          IRP load -= demand[a], load=1 on the depot (irp.py:80-86); cur=a (tsp.py:90);
//          done_b = all visited BEFORE the mask rules (tsp.py:95,103-104)
//   mask:  R1 at depot -> depot bit 1 (tsp.py:141-142); R2 (VRP/IRP) away -> depot bit 0
//          (vrp.py:28-31, irp.py:141-144); R3 all visited -> depot bit 0 (tsp.py:145-146);
//          R4 (IRP) mask = visited | (demand - load > 0) in f64 (irp.py:151-155).
#pragma once
#include "common.cuh"

namespace vrpx {

struct Bits128 {
  uint32_t w[4];
};

__device__ __forceinline__ Bits128 full_bits(int N) {
  Bits128 f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int lo = i * 32;
    f.w[i] = (N >= lo + 32) ? 0xffffffffu : (N > lo ? ((1u << (N - lo)) - 1u) : 0u);
  }
  return f;
}
__device__ __forceinline__ bool bits_all(const Bits128& v, const Bits128& full) {
  return v.w[0] == full.w[0] && v.w[1] == full.w[1] && v.w[2] == full.w[2] && v.w[3] == full.w[3];
}
__device__ __forceinline__ void bit_set(Bits128& v, int n) { v.w[n >> 5] |= (1u << (n & 31)); }
__device__ __forceinline__ void bit_clr(Bits128& v, int n) { v.w[n >> 5] &= ~(1u << (n & 31)); }
__device__ __forceinline__ bool bit_get(const Bits128& v, int n) { return (v.w[n >> 5] >> (n & 31)) & 1u; }

// generate_mask rules R1-R3, in the reference's order, in place on `v`.
__device__ __forceinline__ void apply_mask_rules(Bits128& v, int kind, int N, int cur, int depot) {
  if (cur == depot) bit_set(v, depot);                  // R1
  else if (kind != VRPX_TSP) bit_clr(v, depot);         // R2
  if (bits_all(v, full_bits(N))) bit_clr(v, depot);     // R3
}

// Euclidean edge length exactly as the reference computes it: np.linalg.norm(p - q) =
// sqrt(ddot(d,d)), and the BLAS ddot evaluates dx*dx then fma(dy,dy,.) (verified bit-for-bit
// against 7k reference rewards, tests/golden/env_tapes.npz).
__device__ __forceinline__ double edge_length(const double* __restrict__ xy_b, int i, int j) {
  double dx = __dsub_rn(xy_b[2 * i], xy_b[2 * j]);
  double dy = __dsub_rn(xy_b[2 * i + 1], xy_b[2 * j + 1]);
  return __dsqrt_rn(__fma_rn(dy, dy, __dmul_rn(dx, dx)));
}

// IRP rule R4: bits of nodes whose demand exceeds the current load (f64 compare, irp.py:152).
__device__ __forceinline__ Bits128 demand_exceeds(const double* __restrict__ demand_b, int N, double load) {
  Bits128 m = {{0u, 0u, 0u, 0u}};
  for (int n = 0; n < N; ++n)
    if (__dsub_rn(demand_b[n], load) > 0.0) bit_set(m, n);
  return m;
}

struct StepResult {
  double dist;     // edge length (reward = -dist)
  bool all_before; // every node visited BEFORE the mask rules (per-instance `done`)
};

// One transition of one instance.  `v` in/out: visited bits; `cur`, `load` in/out.
__device__ __forceinline__ StepResult env_transition(int kind, int N, const double* __restrict__ xy_b,
                                                     const double* __restrict__ demand_b, int depot, int a,
                                                     Bits128& v, int& cur, double& load) {
  StepResult r;
  bit_set(v, a);
  r.dist = edge_length(xy_b, cur, a);
  if (kind == VRPX_IRP) {
    load = __dsub_rn(load, demand_b[a]);
    if (a == depot) load = 1.0;
  }
  cur = a;
  r.all_before = bits_all(v, full_bits(N));
  apply_mask_rules(v, kind, N, cur, depot);
  return r;
}

}  // namespace vrpx
