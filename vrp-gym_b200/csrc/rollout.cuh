// rollout.cuh — parameter block shared by the persistent rollout kernel (rollout.cu) and the split-step kernels
// (rollout_steps.cu).
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
};

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

}  // namespace vrpx
