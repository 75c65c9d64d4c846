// rollout.cu — the fused decoder + environment rollout: ONE persistent cooperative launch loops over
// every decode step of the episode (agents/graph_tsp_agent.py:78-92, graph_vrp_agent.py:69-83,
// graph_irp_agent.py:82-105 with agents/graph_decoder.py:51-115 and gym_vrp/envs/*.py step fused).
//
// Per step and per tile of 32 instances a CTA runs:
//   P0  gather X = h[b, last]                                         (graph_decoder.py:108-109)
//   P1  GEMM-A  q~ = X · A_l^T + Q~g[b]  (+ load · a_load)             context -> per-head folded query
//   P2  per instance (one warp): scores = q~_h · h_n + scrambled additive mask (graph_decoder.py:93-94),
//       softmax over nodes, c_h = sum_n p_hn h_n
//   P3  GEMM-B  q^ = C · M^T + m_c                                     (V-proj, out-proj, _att_output, _kp folded)
//   P4  per instance: u_n = 10 tanh(q^ · h_n), -inf mask, argmax / Philox sample / teacher action,
//       log-prob, then the environment transition (env_rules.cuh) in f64
// followed by a grid-wide barrier: the reference's glimpse mask of instance b reads the masks of
// instances (8b+h) mod G (SURVEY App. B-3), so all instances advance in lock-step.
// The per-instance work of P2 and P4 is done by the helpers of glimpse_mma.cuh and rollout.cuh, which the split-step
// kernels (rollout_steps.cu) call as well.
//
// Step-invariant work the reference repeats every step (K/V/kp projections, graph mean) is folded into
// host-packed weights (vrpx/packing.py) and the per-episode Q~g table built in the prologue.
#include "glimpse_mma.cuh"
#include "rollout.cuh"

namespace vrpx {


int build_score_table_fused(const float* h, const float* qk_w, int64_t B, int N, __half* w16, float* s1, cudaStream_t stream);

// Rollout tile: RMT x 16 instances.  With 16 instances per tile the working set that has to survive in L2 between the
// glimpse passes and the pointer-logit pass (all CTAs x tile x 25.6 KB) halves to 60 MB.
constexpr int RMT = 1;
constexpr int RTM = 16 * RMT;
constexpr int RQ_LD = 2 * C16_LD;   // floats per instance slot of QC: the fp16-split c rows of GEMM-B set the stride (1032)
constexpr size_t SMEM_X_MMA = smem_x_mma<RMT>(), SMEM_QC_MMA = (size_t)RTM * RQ_LD * sizeof(float);
constexpr int RNST = 2;   // depth of the per-warp weight rings of the tile GEMMs (3 measured slower: the extra 32 KiB of
                          // shared memory comes out of the L1 that buffers the embedding streams of the other phases)
constexpr size_t SMEM_W_RING = (size_t)(NT / 32) * RNST * 512 * sizeof(float);   // 64 KiB
constexpr size_t SMEM_TOTAL = SMEM_X_MMA + SMEM_QC_MMA + SMEM_W_RING;

// m_t [1024][128] f32 -> M16 [512 k-pairs][128] {hi2, lo2}: the B operand of the fp16-split GEMM-B (tile_gemm.cuh)
__global__ void k_split_m16(const float* __restrict__ m_t, uint2* __restrict__ m16) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // kp * 128 + n
  if (i >= (QW / 2) * E) return;
  const int kp = i >> 7, n = i & (E - 1);
  m16[i] = split_f16x2(m_t[(2 * kp) * E + n], m_t[(2 * kp + 1) * E + n]);
}

// ---------------------------------------------------------------- the persistent kernel
__global__ void __launch_bounds__(NT, 1) k_rollout(const RolloutParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Xs = reinterpret_cast<float*>(smem_raw);
  float* QC = reinterpret_cast<float*>(smem_raw + SMEM_X_MMA);
  float* Wb = reinterpret_cast<float*>(smem_raw + SMEM_X_MMA + SMEM_QC_MMA);
  __shared__ float s_loadf[RTM], s_lp[RTM];
  __shared__ int s_anyleft, s_act[RTM];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.env.N, kind = p.env.kind;
  const int64_t B = p.env.B;
  const int64_t ntiles = (B + RTM - 1) / RTM;
  const float* __restrict__ h = p.h;
  unsigned bar_target = 0;
  long long prof_t = clock64(), prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define VRPX_PROF(i)                                   \
  if (p.prof && tid == 0) {                            \
    long long now_ = clock64();                        \
    prof_acc[i] += now_ - prof_t;                      \
    prof_t = now_;                                     \
  }

  // ------------------------------------------------ prologue: Q~g[b] = A_g · mean_n h[b,n] + a_c
  for (int64_t tile = blockIdx.x; tile < ntiles && p.t0 == 0; tile += gridDim.x) {
    const int64_t base = tile * RTM;
    const int cnt = (int)((B - base < RTM) ? (B - base) : RTM);
    for (int m = warp; m < RTM; m += NT / 32)
      *reinterpret_cast<float4*>(Xs + m * XS_LD + lane * 4) =
          (m < cnt) ? warp_graph_mean(h, base + m, N, lane) : make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    tile_gemm_wide_mma_sw<RMT, RNST>(                                              // Q~g = A_g · g + a_c
        Xs, XS_LD, p.w.ag_t, Wb, [&](int, int c) { return *reinterpret_cast<const float2*>(p.w.a_c + c); },
        [&](int m, int c, float v0, float v1) {
          if (m >= cnt) return;
          const float2 v = make_float2(v0, v1);
          *reinterpret_cast<float2*>(p.qg + (base + m) * QW + c) = v;
          if (p.qg0) *reinterpret_cast<float2*>(p.qg0 + (base + m) * QW + c) = v;
        });
    __syncthreads();
  }

  // Snapshot of the decoder-visible masks for the glimpses of the first step (see RolloutParams::gmask), then a grid
  // barrier: no instance may step before every CTA has taken its snapshot and finished its Q~g rows.
  {
    uint32_t* gm = p.gmask + (size_t)(p.t0 & 1) * B * 4;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int64_t base = tile * RTM;
      const int cnt = (int)((B - base < RTM) ? (B - base) : RTM);
      if (tid < cnt * 4) gm[base * 4 + tid] = __ldcg(p.env.mask + base * 4 + tid);
    }
    bar_target += gridDim.x;
    grid_barrier(p.bar, bar_target);
  }

  int t = p.t0;
  for (; t < p.t0 + p.Tmax; ++t) {
    const int trel = t - p.t0;
    bool cta_unfinished = false;
    const uint32_t* __restrict__ gm_rd = p.gmask + (size_t)(t & 1) * B * 4;   // masks BEFORE step t, every instance
    uint32_t* __restrict__ gm_wr = p.gmask + (size_t)((t + 1) & 1) * B * 4;   // masks after step t
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int64_t base = tile * RTM;
      const int cnt = (int)((B - base < RTM) ? (B - base) : RTM);
      if (tid == 0) s_anyleft = 0;
      // ---------------- P0: gather last-node embeddings, vehicle load; pull this tile's Q~g rows towards L2
      for (int i = tid; i < cnt * 32; i += NT)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(p.qg + base * QW) + (size_t)i * 128));
      for (int m = warp; m < RTM; m += NT / 32) {
        float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < cnt && t > 0) {
          int last = p.env.cur[base + m];
          xv = __ldg(reinterpret_cast<const float4*>(h + ((base + m) * N + last) * E) + lane);
        }
        *reinterpret_cast<float4*>(Xs + m * XS_LD + lane * 4) = xv;
        const float lf = (m < cnt) ? (float)p.env.load[base + m] : 0.f;
        if (lane == 0) s_loadf[m] = lf;
        if (m < cnt) record_trace(p, base + m, trel, lf, lane);
      }
      __syncthreads();
      VRPX_PROF(0)
      // ---------------- P1: q~
      if (t == 0) {
        for (int o = tid; o < cnt * QW; o += NT) {
          const int m = o >> 10, c = o & (QW - 1);
          QC[m * RQ_LD + c] = step0_query(p.qg + (base + m) * QW, p.w.a_q0, p.w.a_load, kind == VRPX_IRP, s_loadf[m], c);
        }
      } else {
        if (t == 1 && kind != VRPX_IRP) {
          tile_gemm_wide_mma_sw<RMT, RNST>(                                        // fold `first` (graph_decoder.py:111-113)
              Xs, XS_LD, p.w.af_t, Wb,
              [&](int m, int c) {
                return (m < cnt) ? *reinterpret_cast<const float2*>(p.qg + (base + m) * QW + c) : make_float2(0.f, 0.f);
              },
              [&](int m, int c, float v0, float v1) {
                if (m < cnt) *reinterpret_cast<float2*>(p.qg + (base + m) * QW + c) = make_float2(v0, v1);
              });
        }
        tile_gemm_wide_mma_sw<RMT, RNST>(                                          // q~ = Q~g (+ load · a_load) + A_l · h[last]
            Xs, XS_LD, p.w.al_t, Wb,
            [&](int m, int c) {
              return (m < cnt) ? glimpse_query_init(p.qg + (base + m) * QW, p.w.a_load, kind == VRPX_IRP, s_loadf[m], c)
                               : make_float2(0.f, 0.f);
            },
            [&](int m, int c, float v0, float v1) { *reinterpret_cast<float2*>(QC + m * RQ_LD + c) = make_float2(v0, v1); });
      }
      __syncthreads();
      VRPX_PROF(1)

      // ---------------- P2: glimpse attention, one warp per instance
      for (int m = warp; m < cnt; m += NT / 32) {
        const int64_t b = base + m;
        float* slot = QC + m * RQ_LD;
        const int tq = lane & 3;
        const float4* hrow = reinterpret_cast<const float4*>(h + b * N * E);
        // ---- pass 1: scores = q~_h · h_n + scrambled additive mask
        uint32_t nb0[4], nb1[4];
        {
          const uint32_t* m0 = gm_rd + quirk_row(b, 2 * tq, p.G) * 4;
          const uint32_t* m1 = gm_rd + quirk_row(b, 2 * tq + 1, p.G) * 4;
#pragma unroll
          for (int i = 0; i < 4; ++i) { nb0[i] = __ldcg(m0 + i); nb1[i] = __ldcg(m1 + i); }
        }
        warp_glimpse_scores(slot, hrow, N, lane, [&](int n, int which, float v) {
          const uint32_t wsel = which ? nb1[n >> 5] : nb0[n >> 5];
          slot[(2 * tq + which) * E + n] = v + (float)((wsel >> (n & 31)) & 1u);
        });
        __syncwarp();
        VRPX_PROF(6)
        float pr[NH][4];
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) {
          warp_load_by_head(pr[hh], slot + hh * E, N, lane);
          warp_node_softmax(pr[hh], N);
        }
        __syncwarp();
        warp_store_by_node(slot, pr, N, lane);
        __syncwarp();
        VRPX_PROF(7)
        // ---- pass 2: c[head][dim] = sum_n P[n][head] h_n[dim], stored over P as the fp16-split A operand of GEMM-B
        float cacc[8][4];
        warp_glimpse_values_acc(cacc, slot, N, lane, glimpse_rows_global(hrow, N, lane));
        warp_glimpse_store_c16(reinterpret_cast<uint4*>(slot), cacc, lane);
      }
      // rows >= cnt of C must be finite for GEMM-B (results unused): zero them
      for (int o = cnt * QW + tid; o < RTM * QW; o += NT) QC[(o >> 10) * RQ_LD + (o & (QW - 1))] = 0.f;
      __syncthreads();
      VRPX_PROF(2)

      // ---------------- P3: q^ = C · M^T + m_c  -> Xs
      tile_gemm_tall_f16<RNST>(reinterpret_cast<const uint2*>(QC), p.m16, Wb, p.w.m_c, QC, Xs, XS_LD);
      VRPX_PROF(3)
      // ---------------- P4: logits, action, environment transition
      bool unfinished = false;
      for (int m = warp; m < cnt; m += NT / 32) {
        const int64_t b = base + m;
        float* slot = QC + m * RQ_LD;  // free scratch again
        const float4 qh = *reinterpret_cast<const float4*>(Xs + m * XS_LD + lane * 4);
        const float4* hp = reinterpret_cast<const float4*>(h + b * N * E) + lane;
        {
          float4 nxt[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) nxt[i] = (i < N) ? __ldg(hp + i * (E / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
          for (int n0 = 0; n0 < N; n0 += 8) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 hv = nxt[i];
              v[i] = fmaf(qh.x, hv.x, fmaf(qh.y, hv.y, fmaf(qh.z, hv.z, qh.w * hv.w)));
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int n = n0 + 8 + i;
              nxt[i] = (n < N) ? __ldg(hp + n * (E / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            float sc = reduce8(v, lane);
            int n = n0 + ((lane >> 2) & 7);
            if ((lane & 3) == 0 && n < N) slot[n] = 10.0f * tanhf(sc);
          }
        }
        __syncwarp();
        uint32_t mw[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) mw[i] = __ldcg(p.env.mask + b * 4 + i);
        float u[4];
        warp_masked_logits(u, slot, mw, N, lane, false);
        const PointerChoice c = warp_pointer_choice(u, p, b, t, trel, lane);
        if (lane == 0) { s_act[m] = c.a; s_lp[m] = c.lp; }
      }
      __syncthreads();
      // environment transition: one THREAD per instance, so the dependent global loads (state -> coordinates) of the
      // whole tile overlap instead of running back to back on lane 0 of each warp
      if (tid < cnt) {
        const int64_t b = base + tid;
        const EnvStepResult r = rollout_env_step(p, b, s_act[tid], s_lp[tid], t, trel);
#pragma unroll
        for (int i = 0; i < 4; ++i) gm_wr[b * 4 + i] = r.mask.w[i];
        unfinished = r.unfinished;
      }
      if (unfinished) s_anyleft = 1;  // benign race: all writers store 1
      __syncthreads();
      if (s_anyleft) cta_unfinished = true;
      __syncthreads();
      VRPX_PROF(4)
    }
    if (tid == 0 && cta_unfinished) atomicAdd(p.notdone + trel, 1);
    bar_target += gridDim.x;
    grid_barrier(p.bar, bar_target);
    VRPX_PROF(5)
    if (ld_acquire_i(p.notdone + trel) == 0) { ++t; break; }
  }
  if (p.prof && tid == 0)
    for (int i = 0; i < 8; ++i) atomicAdd(reinterpret_cast<unsigned long long*>(p.prof) + i, (unsigned long long)prof_acc[i]);
  if (blockIdx.x == 0 && tid == 0) *p.steps = t;
}

static long long* g_rollout_prof = nullptr;
static int g_split_steps = 1;                        // vrpx_debug_rollout_split (bit 0)
static int g_time_kernel = 0;                        // vrpx_debug_rollout_timing
static cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;
static bool g_ev_valid = false;
constexpr int64_t kRolloutSmall = 4096;  // barrier counter + notdone[<=513]
constexpr int64_t kRolloutM16 = (int64_t)(QW / 2) * E * sizeof(uint2);   // 512 KiB: pre-split m_t
constexpr int64_t kRolloutHdr = kRolloutSmall + kRolloutM16;             // Q~g follows

}  // namespace vrpx

using namespace vrpx;

extern "C" {

/* Debug hook: device buffer of 8 x int64 that accumulates per-phase cycles of thread 0 of every CTA (NULL disables). */
void vrpx_debug_rollout_profile(long long* dev_counters) { g_rollout_prof = dev_counters; }

void vrpx_debug_rollout_split(int32_t enable) { g_split_steps = enable & 1; }

void vrpx_debug_rollout_timing(int32_t enable) {
  g_time_kernel = enable;
  g_ev_valid = false;
}

float vrpx_debug_rollout_kernel_ms(void) {
  if (!g_ev_valid) return -1.0f;
  float ms = -1.0f;
  if (cudaEventSynchronize(g_ev1) != cudaSuccess || cudaEventElapsedTime(&ms, g_ev0, g_ev1) != cudaSuccess) return -1.0f;
  return ms;
}

// header | Q~g [B][1024] f32 | gmask [2][B][4] u32
static inline int64_t rollout_gmask_offset(int64_t B) { return kRolloutHdr + B * (int64_t)QW * (int64_t)sizeof(float); }
int64_t vrpx_rollout_workspace_bytes(int64_t B, int32_t N) {
  (void)N;
  return rollout_gmask_offset(B) + 2 * B * 4 * (int64_t)sizeof(uint32_t);
}

int64_t vrpx_rollout_workspace_qg_offset(void) { return kRolloutHdr; }

// table-mode workspace: header | Q~g | gmask | S0 | SL (IRP) | S1 | c | q^ | transposed and split weights | per-copy step
// flags | per-replica flags (the flags for K > 1 only), every segment 256-byte aligned.  S1 holds the Bb base instances, every other per-instance segment the
// Bb·K replicas.
namespace {
struct TableLayout {
  int64_t s0, sl, s1, cbuf, qhat, mnt, agn, afn, w16b, qkw16, copy_left, replica_left, total;
};
inline int64_t align256(int64_t x) { return (x + 255) & ~(int64_t)255; }
inline int64_t copy_left_bytes(int64_t K, int N) { return K > 1 ? K * 2 * N * (int64_t)sizeof(int) : 0; }   // [2N > Tmax][K]
TableLayout table_layout(int kind, int64_t Bb, int64_t K, int N) {
  TableLayout L;
  const int64_t f = (int64_t)sizeof(float), B = Bb * K;
  L.s0 = align256(vrpx_rollout_workspace_bytes(B, N));
  L.sl = align256(L.s0 + B * NH * N * f);
  L.s1 = (kind == VRPX_IRP) ? align256(L.sl + B * NH * N * f) : L.sl;
  // split-step mode (rollout_steps.cu): glimpse vectors, folded queries, transposed m_t
  L.cbuf = align256(L.s1 + Bb * N * NH * N * f);
  L.qhat = align256(L.cbuf + B * QW * f);
  L.mnt = align256(L.qhat + B * E * f);
  L.agn = align256(L.mnt + (int64_t)QW * E * f);
  L.afn = align256(L.agn + (int64_t)QW * E * f);
  L.w16b = align256(L.afn + (int64_t)QW * E * f);
  L.qkw16 = align256(L.w16b + (int64_t)2 * QW * E * 2);
  L.copy_left = align256(L.qkw16 + (int64_t)2 * 768 * E * 2);
  L.replica_left = align256(L.copy_left + copy_left_bytes(K, N));
  L.total = align256(L.replica_left + (K > 1 ? B : 0));
  return L;
}

int check_env_and_weights(const vrpx_env* env, const vrpx_decoder_weights* w) {
  VRPX_CHECK_ARG(env->kind >= 0 && env->kind <= 2 && env->N >= 2 && env->N <= VRPX_MAX_NODES && env->B >= 1,
                 "bad env header");
  VRPX_CHECK_ARG(env->xy && env->depot && env->visited && env->mask && env->cur && env->load, "env arrays");
  VRPX_CHECK_ARG(env->kind != VRPX_IRP || env->demand, "IRP env needs demand");
  VRPX_CHECK_ARG(w->ag_t && w->al_t && w->a_c && w->a_q0 && w->m_t && w->m_c, "decoder weights");
  VRPX_CHECK_ARG(env->kind == VRPX_IRP ? (w->a_load != nullptr) : (w->af_t != nullptr), "decoder weights (kind)");
  return VRPX_OK;
}

RolloutParams make_params(const vrpx_env* env, const vrpx_decoder_weights* w, const float* h, int mode, int64_t coupling,
                          uint64_t seed, uint64_t offset, uint8_t* tape, int t_begin, int Tmax, float* logp, float* cost,
                          int32_t* steps, float* logits, void* ws) {
  RolloutParams p;
  p.env = *env;
  p.w = *w;
  p.h = h;
  p.mode = mode;
  p.G = coupling;
  p.seed = seed;
  p.offset = offset;
  p.tape = tape;
  p.t0 = t_begin;
  p.Tmax = Tmax;
  p.logp = logp;
  p.cost = cost;
  p.steps = steps;
  p.logits = logits;
  p.qg0 = nullptr;
  p.mask_hist = nullptr;
  p.load_hist = nullptr;
  p.prof = g_rollout_prof;
  p.bar = reinterpret_cast<unsigned*>(ws);
  p.notdone = reinterpret_cast<int*>(ws) + 8;
  p.qg = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + kRolloutHdr);
  p.gmask = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ws) + rollout_gmask_offset(env->B));
  p.m16 = reinterpret_cast<const uint2*>(reinterpret_cast<char*>(ws) + kRolloutSmall);
  p.s1 = nullptr;
  p.s0 = p.sl = nullptr;
  p.cbuf = p.qhat = nullptr;
  p.Bb = env->B;
  p.K = 1;
  p.replica_left = nullptr;
  p.copy_left = nullptr;
  return p;
}

int decode_timing_begin(cudaStream_t stream) {
  if (g_time_kernel) {
    if (!g_ev0) {
      VRPX_CUDA(cudaEventCreate(&g_ev0));
      VRPX_CUDA(cudaEventCreate(&g_ev1));
    }
    VRPX_CUDA(cudaEventRecord(g_ev0, stream));
  }
  return VRPX_OK;
}

int decode_timing_end(cudaStream_t stream) {
  if (g_time_kernel) {
    VRPX_CUDA(cudaEventRecord(g_ev1, stream));
    g_ev_valid = true;
  }
  return VRPX_OK;
}

// Table mode: score tables over the p.Bb base instances (rollout_steps.cu reads them at each replica's base instance),
// then every decode step as launches over the p.env.B replicas.
int run_table_episode(RolloutParams& p, const TableLayout& L, void* ws, cudaStream_t stream) {
  char* base = reinterpret_cast<char*>(ws);
  float* s1 = reinterpret_cast<float*>(base + L.s1);
  int rc;
  {
    NvtxRange nvtx_tables("vrpx:score_tables");
    rc = build_score_table_fused(p.h, p.w.qk_w, p.Bb, p.env.N, reinterpret_cast<__half*>(base + L.qkw16), s1, stream);
  }
  if (rc) return rc;
  p.s1 = s1;
  p.s0 = reinterpret_cast<float*>(base + L.s0);
  p.sl = reinterpret_cast<float*>(base + L.sl);
  p.cbuf = reinterpret_cast<float*>(base + L.cbuf);
  p.qhat = reinterpret_cast<float*>(base + L.qhat);
  const SplitWorkspace sw{reinterpret_cast<float*>(base + L.mnt), reinterpret_cast<float*>(base + L.agn),
                          reinterpret_cast<float*>(base + L.afn), reinterpret_cast<__half*>(base + L.w16b)};
  GemmPlan plan_b;
  if ((rc = prepare_split_weights(p, sw, &plan_b, stream))) return rc;
  VRPX_CUDA(cudaMemsetAsync(ws, 0, kRolloutSmall, stream));
  if ((rc = decode_timing_begin(stream))) return rc;
  NvtxRange nvtx_decode("vrpx:decode_loop");
  if ((rc = run_first_steps(p, sw, plan_b, stream))) return rc;
  if ((rc = run_split_steps(p, p.t0 + 2, plan_b, stream))) return rc;   // also writes the step count
  return decode_timing_end(stream);
}
}  // namespace

int64_t vrpx_rollout_table_workspace_bytes(int32_t kind, int64_t B, int32_t N) { return table_layout(kind, B, 1, N).total; }

int64_t vrpx_rollout_samples_workspace_bytes(int32_t kind, int64_t Bb, int32_t K, int32_t N) {
  return table_layout(kind, Bb, K, N).total;
}

int vrpx_rollout(const vrpx_env* env, const vrpx_decoder_weights* w, const float* h, int32_t mode,
                 int64_t coupling, uint64_t seed, uint64_t offset, uint8_t* tape, int32_t t_begin, int32_t Tmax,
                 float* logp, float* cost, int32_t* steps, float* logits, const vrpx_rollout_trace* trace,
                 void* ws, int64_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VRPX_CHECK_ARG(env && w && h && logp && cost && steps && ws, "NULL argument");
  VRPX_DEVICE_GUARD(h);
  NvtxRange nvtx_range("vrpx:rollout");
  if (int rc = check_env_and_weights(env, w)) return rc;
  VRPX_CHECK_ARG(mode >= 0 && mode <= 2, "bad mode");
  VRPX_CHECK_ARG(mode != VRPX_TEACHER || tape, "teacher mode needs a tape");
  VRPX_CHECK_ARG(Tmax >= 1 && Tmax <= 1000 && t_begin >= 0, "t_begin / Tmax out of range");
  // attention row (b, head) reads the mask of instance quirk_row(b, head, G): it must stay inside the batch
  VRPX_CHECK_ARG(coupling >= 0 && (coupling == 0 || (coupling <= env->B && env->B % coupling == 0)),
                 "coupling group must be 0 or a divisor of the batch size");
  VRPX_CHECK_ARG(ws_bytes >= vrpx_rollout_workspace_bytes(env->B, env->N), "workspace too small");
  VRPX_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "workspace must be 16-byte aligned");
  VRPX_CHECK_ARG((int64_t)(Tmax + 1 + 8) * 4 <= kRolloutSmall, "Tmax too large for workspace header");

  RolloutParams p = make_params(env, w, h, mode, coupling, seed, offset, tape, t_begin, Tmax, logp, cost, steps, logits, ws);
  p.qg0 = trace ? trace->qg0 : nullptr;
  p.mask_hist = trace ? trace->mask_hist : nullptr;
  p.load_hist = trace ? trace->load_hist : nullptr;
  // Split-step form (default for whole-episode calls with the large workspace and the rank-48 factors): per-episode score
  // tables, then every step is a handful of launches over the whole batch (rollout_steps.cu).  The persistent kernel
  // below serves the classic mode, resumed single-step calls and vrpx_debug_rollout_split(0).
  if (g_split_steps && w->qk_w && t_begin == 0 && Tmax >= 3) {
    const TableLayout L = table_layout(env->kind, env->B, 1, env->N);
    if (ws_bytes >= L.total) return run_table_episode(p, L, ws, stream);
  }

  VRPX_CUDA(cudaMemsetAsync(ws, 0, kRolloutSmall, stream));
  k_split_m16<<<(QW / 2) * E / 256, 256, 0, stream>>>(w->m_t, reinterpret_cast<uint2*>(reinterpret_cast<char*>(ws) + kRolloutSmall));
  VRPX_LAUNCH_CHECK();
  VRPX_CUDA(cudaFuncSetAttribute(k_rollout, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_TOTAL));
  if (int rc = decode_timing_begin(stream)) return rc;
  NvtxRange nvtx_decode("vrpx:decode_loop");
  int64_t ntiles = (env->B + RTM - 1) / RTM;
  int grid = (int)((ntiles < (int64_t)num_sms()) ? ntiles : (int64_t)num_sms());
  void* args[] = {(void*)&p};
  VRPX_CUDA(cudaLaunchCooperativeKernel((void*)k_rollout, dim3(grid), dim3(NT), args, SMEM_TOTAL, stream));
  count_launch();
  return decode_timing_end(stream);
}

int vrpx_rollout_samples(const vrpx_env* env, const vrpx_decoder_weights* w, const float* h, int64_t Bb, int32_t K,
                         int64_t coupling, uint64_t seed, uint64_t offset, uint8_t* tape, int32_t Tmax, float* logp,
                         float* cost, int32_t* steps, float* logits, void* ws, int64_t ws_bytes, void* stream_) {
  return vrpx_rollout_samples_traced(env, w, h, Bb, K, coupling, seed, offset, tape, Tmax, logp, cost, steps, logits,
                                     nullptr, ws, ws_bytes, stream_);
}

int vrpx_rollout_samples_traced(const vrpx_env* env, const vrpx_decoder_weights* w, const float* h, int64_t Bb, int32_t K,
                                int64_t coupling, uint64_t seed, uint64_t offset, uint8_t* tape, int32_t Tmax, float* logp,
                                float* cost, int32_t* steps, float* logits, const vrpx_rollout_trace* trace, void* ws,
                                int64_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VRPX_CHECK_ARG(env && w && h && tape && logp && cost && steps && ws, "NULL argument");
  VRPX_DEVICE_GUARD(h);
  NvtxRange nvtx_range("vrpx:rollout_samples");
  if (int rc = check_env_and_weights(env, w)) return rc;
  VRPX_CHECK_ARG(K >= 1, "sample count K must be at least 1");
  VRPX_CHECK_ARG(Bb >= 1 && env->B % K == 0 && env->B / K == Bb, "env must hold Bb x K replicas");
  // the partner rows of quirk_row must stay inside each copy
  VRPX_CHECK_ARG(coupling >= 0 && (coupling == 0 || (coupling <= Bb && Bb % coupling == 0)),
                 "coupling group must be 0 or a divisor of the base batch size");
  VRPX_CHECK_ARG(w->qk_w, "sampling needs the score-table factors qk_w");
  VRPX_CHECK_ARG(Tmax >= 1 && Tmax <= 1000, "Tmax out of range");
  if (Tmax < 3) {
    set_error("%s: episodes of fewer than 3 steps have no table-mode decode loop (use vrpx_rollout per copy)", __func__);
    return VRPX_ERR_UNSUPPORTED;
  }
  const TableLayout L = table_layout(env->kind, Bb, K, env->N);
  VRPX_CHECK_ARG(ws_bytes >= L.total, "workspace too small");
  VRPX_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 15) == 0, "workspace must be 16-byte aligned");

  RolloutParams p = make_params(env, w, h, VRPX_SAMPLE, coupling, seed, offset, tape, 0, Tmax, logp, cost, steps, logits, ws);
  p.Bb = Bb;
  p.K = K;
  p.qg0 = trace ? trace->qg0 : nullptr;
  p.mask_hist = trace ? trace->mask_hist : nullptr;
  p.load_hist = trace ? trace->load_hist : nullptr;
  if (K > 1) {
    p.copy_left = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + L.copy_left);
    p.replica_left = reinterpret_cast<uint8_t*>(ws) + L.replica_left;
    VRPX_CUDA(cudaMemsetAsync(p.copy_left, 0, copy_left_bytes(K, env->N), stream));
  }
  return run_table_episode(p, L, ws, stream);
}

}  // extern "C"
