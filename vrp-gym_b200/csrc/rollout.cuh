// rollout.cuh — parameter block and the per-instance parts of a decode step outside the glimpse (graph mean, query,
// masked pointer logits, action choice, environment step), shared by the persistent rollout kernel (rollout.cu), the
// split-step kernels (rollout_steps.cu) and the recompute of the REINFORCE backward (decoder_bwd.cu).
#pragma once
#include "gemm.cuh"
#include "tile_gemm.cuh"

namespace vrpx {

struct RolloutParams {
  vrpx_env env;
  vrpx_decoder_weights w;
  const float* h;
  int mode;
  long long G;
  unsigned long long seed, offset;
  uint8_t* tape;
  int t0;
  int Tmax;
  float* logp;
  float* cost;
  int* steps;
  float* logits;
  float* qg;          // [B][1024]
  float* qg0;         // optional copy of Q~g before the `first` fold (backward)
  uint32_t* mask_hist;  // optional [Tmax][B][4] decoder-visible mask before each step (backward)
  float* load_hist;   // optional [Tmax][B] f32 vehicle load before each step (backward)
  uint32_t* gmask;    // [2][B][4] persistent kernel only: the decoder-visible masks every glimpse of step t reads are the
                      // snapshot gmask[t & 1] (the env transition of step t writes gmask[(t + 1) & 1]); reading env.mask in
                      // place would race with the transitions of tiles that are already past their pointer phase
  unsigned* bar;      // grid barrier counter
  int* notdone;       // [Tmax + 1]
  long long* prof;    // optional [8] cycle counters per phase (debug, vrpx_debug_rollout_profile)
  // split-step mode: per-episode glimpse score tables (S1 from score_table_fused.cu before the first step, S0 / SL
  // written at step 1 by rollout_steps.cu), all NULL in the persistent kernel
  const float* s1;    // [B][N][8][N]  (A_l h[b,l])_head · h[b,n]
  float* s0;          // [B][8][N]     Q~g[b]_head · h[b,n], built at step 1 (after the `first` fold)
  float* sl;          // [B][8][N]     IRP: a_load_head · h[b,n]
  const uint2* m16;   // [512][128] m_t pre-split for the fp16 tensor path (k_split_m16, tile_gemm.cuh)
  // split-step mode (rollout_steps.cu): glimpse vectors c [B][1024] and folded queries q^ [B][128] in global memory
  float* cbuf;
  float* qhat;
  // K sampled copies of a batch of Bb base instances (vrpx_rollout_samples): replica r = k·Bb + b is copy k of base
  // instance b and reads the embeddings and S1 of b; every other per-instance array is per replica (env.B = Bb·K).
  // vrpx_rollout: Bb = env.B, K = 1.
  int64_t Bb;
  int K;
  // K > 1 (NULL otherwise): replica_left[r] = replica r was unfinished after its last step (k_step_pointer), and
  // copy_left[trel][k] != 0 when some replica of copy k was unfinished after step trel (k_copy_left).  A copy whose own
  // episode is over skips the later steps: its cost, log-prob and env state stay those of the copy run alone, and its
  // tape rows get the depot.
  uint8_t* replica_left;
  int* copy_left;
};

// Warp slot s of the split-step kernels -> the replica it runs (r), that replica's base instance (b) and copy (k).  Slot
// s runs copy s mod K of base instance s / K, so the K warps that read h[b] and S1[b] are neighbours and run side by
// side.  K = 1: the identity.
struct SlotReplica {
  int64_t r, b;
  int k;
};
__device__ __forceinline__ SlotReplica slot_replica(const RolloutParams& p, int64_t s) {
  if (p.K == 1) return {s, s, 0};
  const int64_t b = s / p.K;
  const int k = (int)(s - b * p.K);
  return {k * p.Bb + b, b, k};
}

// true when copy k's own episode was over before step trel (K > 1; with K = 1 episode_over in rollout_steps.cu ends
// every launch of the step instead)
__device__ __forceinline__ bool copy_over(const RolloutParams& p, int k, int trel) {
  return p.K > 1 && trel > 0 && __ldcg(p.copy_left + (int64_t)(trel - 1) * p.K + k) == 0;
}

// rollout_steps.cu: a whole-episode table-mode rollout as launches over the whole batch — steps 0 and 1 (run_first_steps:
// they build Q~g and S0), then three launches per step (run_split_steps: glimpse, batched GEMM-B, pointer) and the final
// step count.  SplitWorkspace: transposed copies of the folded weights for the tcgen05 GEMMs ([NOUT][K] layout) and the
// split halves of m_t^T, in the rollout workspace.
struct SplitWorkspace {
  float* m_nt;     // [128][1024]  m_t^T
  float* ag_n;     // [1024][128]  ag_t^T
  float* af_n;     // [1024][128]  af_t^T (TSP / VRP)
  __half* w16b;    // 2 x [128][1024] halves: hi | lo of m_t^T * 2^8
};
int prepare_split_weights(const RolloutParams& p, const SplitWorkspace& w, GemmPlan* plan_b, cudaStream_t stream);
int run_first_steps(const RolloutParams& p, const SplitWorkspace& w, const GemmPlan& plan_b, cudaStream_t stream);
int run_split_steps(const RolloutParams& p, int t_first, const GemmPlan& plan_b, cudaStream_t stream);
// decoder_bwd.cu: G[b] = mean_n h[b, n] (warp_graph_mean) and, unless Xf is NULL, Xf[b] = h[b, tape0[b]]
int launch_episode_gather(const float* h, const uint8_t* tape0, int64_t B, int N, float* G, float* Xf, cudaStream_t stream);

// G[b] = mean_n h[b, n] (graph_decoder.py:75-77), one warp per instance: lane l returns dims 4l .. 4l+3
__device__ __forceinline__ float4 warp_graph_mean(const float* __restrict__ h, int64_t b, int N, int lane) {
  const float4* hp = reinterpret_cast<const float4*>(h + b * N * E) + lane;
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int n = 0; n < N; ++n) {
    const float4 v = __ldg(hp + n * (E / 4));
    g.x += v.x; g.y += v.y; g.z += v.z; g.w += v.w;
  }
  const float inv = 1.0f / (float)N;
  return make_float4(g.x * inv, g.y * inv, g.z * inv, g.w * inv);
}

// ---------------------------------------------------------------- the folded glimpse query q~ of one instance
// qg = the instance's Q~g row, lf = its vehicle load as f32; the load term a_load exists for IRP only.
// Step 0 (graph_decoder.py:79-81), dim c: the learned placeholder a_q0 takes the place of A_l h[last]
__device__ __forceinline__ float step0_query(const float* qg, const float* a_q0, const float* a_load, bool irp, float lf,
                                             int c) {
  const float y = qg[c] + a_q0[c];
  return irp ? fmaf(lf, a_load[c], y) : y;
}
// Steps >= 1, dims c, c+1: Q~g (+ lf · a_load), the initial accumulators of the GEMM-A tile q~ = that + A_l h[last]
__device__ __forceinline__ float2 glimpse_query_init(const float* qg, const float* a_load, bool irp, float lf, int c) {
  float2 q = *reinterpret_cast<const float2*>(qg + c);
  if (irp) {
    const float2 al = *reinterpret_cast<const float2*>(a_load + c);
    q = make_float2(fmaf(lf, al.x, q.x), fmaf(lf, al.y, q.y));
  }
  return q;
}

// Write the trace the backward replays (RolloutParams::mask_hist / load_hist) for instance b before step trel
__device__ __forceinline__ void record_trace(const RolloutParams& p, int64_t b, int trel, float lf, int lane) {
  if (p.mask_hist && lane < 4) p.mask_hist[((int64_t)trel * p.env.B + b) * 4 + lane] = __ldcg(p.env.mask + b * 4 + lane);
  if (p.load_hist && lane == 0) p.load_hist[(int64_t)trel * p.env.B + b] = lf;
}

// ---------------------------------------------------------------- the pointer phase: logits, action, environment step
// (phase P4 of the persistent kernel and the split-step pointer kernel)

// Masked logits u[i] of node 4 lane + i (graph_decoder.py:98): slot[n] where the own mask words mw leave node n open,
// -inf where masked or beyond N.  `idle` (a finished instance, see instance_idle in rollout_steps.cu): its single open
// node gets 0, which gives the same action and log-prob as any finite logit, and slot is not read.
__device__ __forceinline__ void warp_masked_logits(float (&u)[4], const float* slot, const uint32_t (&mw)[4], int N, int lane,
                                                   bool idle) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = lane * 4 + i;
    const bool ok = n < N && !((mw[n >> 5] >> (n & 31)) & 1u);
    u[i] = ok ? (idle ? 0.f : slot[n]) : -INFINITY;
  }
}

struct PointerChoice {
  int a;      // action
  float lp;   // its log-prob (0 in greedy mode)
};

// One warp picks instance b's action at step t (trel = t - p.t0) from its masked logits: u[i] = node 4 lane + i, -inf
// where masked or beyond N.  Writes them to p.logits when requested; argmax with ties to the lowest index, the Philox
// inverse-CDF sample (counter (offset + b, t, 0x5eed)) or the teacher's action; log-prob of the taken action
// (graph_decoder.py:107).  Every lane returns the same choice.
__device__ __forceinline__ PointerChoice warp_pointer_choice(const float (&u)[4], const RolloutParams& p, int64_t b, int t,
                                                             int trel, int lane) {
  if (p.logits) {
    float* lo = p.logits + ((int64_t)trel * p.env.B + b) * p.env.N;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (lane * 4 + i < p.env.N) lo[lane * 4 + i] = u[i];
  }
  // max + first-max index (argmax tie rule: lowest index)
  float mx = u[0];
  int am = lane * 4;
#pragma unroll
  for (int i = 1; i < 4; ++i)
    if (u[i] > mx) { mx = u[i]; am = lane * 4 + i; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float omx = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oam = __shfl_xor_sync(0xffffffffu, am, o);
    if (omx > mx || (omx == mx && oam < am)) { mx = omx; am = oam; }
  }
  PointerChoice c{am, 0.f};
  if (p.mode != VRPX_GREEDY) {
    float ex[4], loc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ex[i] = (u[i] == -INFINITY) ? 0.f : expf(u[i] - mx);
      loc += ex[i];
    }
    float incl = loc;  // inclusive scan of lane totals
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const float y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    const float total = __shfl_sync(0xffffffffu, incl, 31);
    if (p.mode == VRPX_SAMPLE) {
      const uint64_t gid = p.offset + (uint64_t)b;
      const uint4 r = philox4x32_10(make_uint4((uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)t, 0x5eedu),
                                    make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32)));
      const float thr = u24(r.x) * total;
      float cum = incl - loc;
      int pick = 1 << 30;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        cum += ex[i];
        if (ex[i] > 0.f && cum > thr && pick == (1 << 30)) pick = lane * 4 + i;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) pick = min(pick, __shfl_xor_sync(0xffffffffu, pick, o));
      c.a = (pick == (1 << 30)) ? am : pick;  // rounding guard: fall back to the mode
    } else {
      c.a = (int)p.tape[(int64_t)trel * p.env.B + b];
    }
    const int ai = c.a & 3;
    const float usel = ai == 0 ? u[0] : (ai == 1 ? u[1] : (ai == 2 ? u[2] : u[3]));
    const float ua = __shfl_sync(0xffffffffu, usel, c.a >> 2);
    c.lp = (ua - mx) - logf(total);
  }
  return c;
}

struct EnvStepResult {
  bool unfinished;   // some node is still unvisited after this step's visit (the instance's `done` is false)
  Bits128 mask;      // decoder-visible mask after the step
};

// One thread steps instance b at step t (trel = t - p.t0) with action a of log-prob lp: tape write (sample / greedy), env_transition
// (env_rules.cuh), state write-back, the IRP mask (rule R4), and the f32 accumulation of cost and log-prob in step order.
__device__ __forceinline__ EnvStepResult rollout_env_step(const RolloutParams& p, int64_t b, int a, float lp, int t,
                                                          int trel) {
  const int N = p.env.N, kind = p.env.kind;
  if (p.tape && p.mode != VRPX_TEACHER) p.tape[(int64_t)trel * p.env.B + b] = (uint8_t)a;
  Bits128 v;
#pragma unroll
  for (int i = 0; i < 4; ++i) v.w[i] = p.env.visited[b * 4 + i];
  int cur = p.env.cur[b];
  double load = p.env.load[b];
  const int depot = p.env.depot[b];
  const double* dem = p.env.demand ? p.env.demand + b * N : nullptr;
  const StepResult r = env_transition(kind, N, p.env.xy + b * N * 2, dem, depot, a, v, cur, load);
  p.env.cur[b] = cur;
  p.env.load[b] = load;
#pragma unroll
  for (int i = 0; i < 4; ++i) p.env.visited[b * 4 + i] = v.w[i];
  EnvStepResult res{!r.all_before, v};
  if (kind == VRPX_IRP) {
    const Bits128 x = demand_exceeds(dem, N, load);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      res.mask.w[i] = v.w[i] | x.w[i];
      p.env.mask[b * 4 + i] = res.mask.w[i];
    }
  }
  // f32 accumulation of f32(reward) in step order (graph_tsp_agent.py:85); cost = -acc_loss
  p.cost[b] = (t == 0 ? 0.f : p.cost[b]) + (float)r.dist;
  if (p.mode != VRPX_GREEDY) p.logp[b] = (t == 0 ? 0.f : p.logp[b]) + lp;
  else if (t == 0) p.logp[b] = 0.f;
  return res;
}

}  // namespace vrpx
