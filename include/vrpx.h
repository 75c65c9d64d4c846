/*
 * vrpx.h — C ABI of the B200-native VRP-Gym rollout path (libvrpx.so).
 *
 * The reference (kevin-schumann/VRP-GYM) is pure Python: it has no FFI.  Its
 * boundary is the Python class surface (SURVEY.md §8b).  This ABI sits directly
 * underneath that surface; every entry point cites the reference code it
 * replaces (paths relative to the reference root).  All pointers are DEVICE
 * pointers unless named h_*; all buffers are caller-owned; `stream` is a
 * cudaStream_t passed as void*.  Every call returns 0 or a negative
 * vrpx_status, never throws, never exits, and does not synchronise unless
 * documented.  Build: nvcc -gencode arch=compute_100a,code=sm_100a.
 */
#ifndef VRPX_H
#define VRPX_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VRPX_API __attribute__((visibility("default")))
#else
#define VRPX_API
#endif

#define VRPX_ABI_VERSION 6
#define VRPX_MAX_NODES 128 /* visited bitmask = 4 x u32 per instance */
#define VRPX_EMB 128       /* embedding width E (graph_tsp_agent.py:98) */
#define VRPX_HEADS 8       /* heads (graph_tsp_agent.py:101, :55) */
#define VRPX_FF 512        /* encoder FF width (graph_tsp_agent.py:99) */
#define VRPX_LAYERS 3      /* encoder layers (graph_tsp_agent.py:100) */

typedef enum vrpx_status {
  VRPX_OK = 0,
  VRPX_ERR_ARG = -1,     /* bad argument (NULL, N > VRPX_MAX_NODES, ...) */
  VRPX_ERR_DEVICE = -2,  /* not an sm_100 device / no device */
  VRPX_ERR_CUDA = -3,    /* CUDA runtime error, see vrpx_last_error() */
  VRPX_ERR_UNSUPPORTED = -4
} vrpx_status;

typedef enum vrpx_kind { VRPX_TSP = 0, VRPX_VRP = 1, VRPX_IRP = 2 } vrpx_kind;

/* Device-resident SoA state of a batch of routing instances.
 * Replaces: VRPNetwork/VRPGraph storage (gym_vrp/graph/vrp_network.py:9-42,
 * vrp_graph.py:27-45) and the env fields visited/current_location/load/demands
 * (gym_vrp/envs/tsp.py:162-174, irp.py:47,157-185). */
typedef struct vrpx_env {
  int32_t kind;      /* vrpx_kind */
  int32_t N;         /* nodes per instance, 2..VRPX_MAX_NODES */
  int64_t B;         /* instances */
  double* xy;        /* [B][N][2] f64 coordinates */
  int32_t* depot;    /* [B] */
  double* demand;    /* [B][N] f64 (depot 0); may be NULL for TSP/VRP */
  uint32_t* visited; /* [B][4] bit n = visited[n] AFTER the mask rules R1-R3 */
  uint32_t* mask;    /* [B][4] decoder-visible mask: IRP = visited | (demand-load>0) (irp.py:151-155);
                        TSP/VRP: must alias `visited` */
  int32_t* cur;      /* [B] current_location */
  double* load;      /* [B] f64 vehicle load (IRP; still required, unused for TSP/VRP) */
} vrpx_env;

VRPX_API int vrpx_abi_version(void);
VRPX_API const char* vrpx_last_error(void); /* thread-local message of the last failing call */
VRPX_API int vrpx_device_check(int device); /* <0 unless compute capability 10.x */

/* Philox4x32-10 instance generator (throughput mode; NOT numpy-seed compatible).
 * Fills xy (U[0,1)^2), depot (uniform), demand (U[1,10)/C, depot 0) following the
 * distributions of vrp_graph.py:29,34,41-43.  Instance b uses counter (offset + b). */
VRPX_API int vrpx_env_generate(const vrpx_env* env, uint64_t seed, uint64_t offset, void* stream);

/* Episode reset: visited=0, cur=depot, load=1, then mask rules (tsp.py:158-160,167-174; irp.py:183-185). */
VRPX_API int vrpx_env_reset(const vrpx_env* env, void* stream);

/* One environment transition for all B instances = TSPEnv.step / IRPEnv.step
 * (tsp.py:60-101, irp.py:49-99) fused with generate_mask (tsp.py:131-148, vrp.py:13-37,
 * irp.py:126-155), is_done (tsp.py:103-104) and get_distances (vrp_network.py:59-78).
 *   actions  [B] int64 (the (B,1) array of the reference, flattened)
 *   reward   [B] f64, = -euclidean distance (tsp.py:98)
 *   not_done [1] int32, must be zeroed by the caller; incremented (by >= 1) iff some instance is
 *            not fully visited BEFORE the mask rules -> done == (*not_done == 0).
 *   state    optional [B][N][4|5] f64 observation (tsp.py:106-129, irp.py:101-124), or NULL. */
VRPX_API int vrpx_env_step(const vrpx_env* env, const int64_t* actions, double* reward, int32_t* not_done,
                  double* state, void* stream);

/* Observation / mask / visited materialised in the reference layout (get_state, generate_mask).
 * state [B][N][4] = [x,y,is_depot,mask]; IRP [B][N][5] = [x,y,demand,is_depot,mask].
 * mask/visited [B][N] f64 of 0/1.  Any output may be NULL. */
VRPX_API int vrpx_env_observe(const vrpx_env* env, double* state, double* mask, double* visited, void* stream);

/* Write back a (B,N) f64 0/1 array into the bitmask (used when a caller assigns env.visited). */
VRPX_API int vrpx_env_set_visited(const vrpx_env* env, const double* visited, void* stream);

/* Recompute the decoder-visible IRP mask = visited | (demand - load > 0) (irp.py:151-155) from the CURRENT demand /
 * load arrays, e.g. after a caller edited node demands through sampler.graphs[i].nodes[n]["demand"] (the write-through
 * protocol of tests/test_env.py:31-36).  No-op for TSP / VRP (mask aliases visited). */
VRPX_API int vrpx_env_refresh_mask(const vrpx_env* env, void* stream);

/* ---------------------------------------------------------------- seed-compatible instance stream (host, C)
 * The reference draws instances from numpy's legacy global RandomState (MT19937) one graph after the other
 * (gym_vrp/graph/vrp_graph.py:29,34,42 via vrp_network.py:41-42, after tsp.py:48,55).  These entry points consume a COPY
 * of that generator state — key[624] + pos, the layout of np.random.get_state() — exactly as numpy would and leave the
 * advanced state in place, so the caller hands it back with np.random.set_state().  Host pointers (h_*), no GPU needed.
 *   vrpx_mt19937_seed              np.random.seed(seed) for 0 <= seed < 2^32
 *   vrpx_mt19937_permutation_head  np.random.choice(n, k, replace=False) = permutation(n)[:k]   (tsp.py:55 draw_idxs)
 *   vrpx_mt19937_instances         per graph: rand(N,2) -> choice(N, D, replace=False) -> uniform(1,10,(N,1))/C, depot
 *                                  demand 0; h_xy [G][N][2] f64, h_depots [G][D] int64, h_demand [G][N] f64
 *   vrpx_mt19937_random_actions    RandomAgent (agents/random_agent.py:33-35): per instance np.random.choice(feasible, 1)
 *                                  with feasible = nodes whose mask entry is 0; h_mask [B][N] f64, h_actions [B] int64 */
VRPX_API int vrpx_mt19937_seed(uint32_t seed, uint32_t* key, int32_t* pos);
VRPX_API int vrpx_mt19937_permutation_head(uint32_t* key, int32_t* pos, int64_t n, int64_t k, int64_t* h_out);
VRPX_API int vrpx_mt19937_instances(uint32_t* key, int32_t* pos, int64_t num_graphs, int32_t N, int32_t num_depots,
                                    double* h_xy, int64_t* h_depots, double* h_demand);
VRPX_API int vrpx_mt19937_random_actions(uint32_t* key, int32_t* pos, const double* h_mask, int64_t B, int32_t N,
                                         int64_t* h_actions);

/* ---------------------------------------------------------------- policy */

/* Encoder parameters, torch layouts (row-major [out][in]) — state_dict keys of SURVEY App. A.5. */
typedef struct vrpx_encoder_layer {
  const float *in_proj_w, *in_proj_b;   /* [384][128], [384]  attention_layer.in_proj_* */
  const float *out_proj_w, *out_proj_b; /* [128][128], [128] */
  const float *bn1_w, *bn1_b;           /* [128] affine */
  float *bn1_mean, *bn1_var;            /* [128] running stats (updated in train mode) */
  const float *ff0_w, *ff0_b;           /* [512][128], [512] */
  const float *ff2_w, *ff2_b;           /* [128][512], [128] */
  const float *bn2_w, *bn2_b;
  float *bn2_mean, *bn2_var;
} vrpx_encoder_layer;

typedef struct vrpx_encoder_weights {
  int32_t f;                              /* node feature count: 2 (TSP/VRP) or 3 (IRP) */
  const float *node_w, *node_b;           /* [128][f], [128]   encoder.node_embed */
  const float *depot_w, *depot_b;         /* [128][2], [128]   encoder.depot_embed, or NULL (TSP) */
  vrpx_encoder_layer layer[VRPX_LAYERS];
} vrpx_encoder_weights;

/* Bytes of scratch `ws` needed by vrpx_encoder_forward for R = B*N rows. */
VRPX_API int64_t vrpx_encoder_workspace_bytes(int64_t B, int32_t N);

/* GraphEncoder.forward / GraphDemandEncoder.forward (agents/graph_encoder.py:41-58, :95-138)
 * with MultiHeadAttentionLayer (:183-198) and BatchNorm (:141-154).
 *   x      [B][N][f] f32 node features, or NULL to read them from `env` (xy [, demand]) cast to f32
 *          exactly as graph_tsp_agent.py:72 does;
 *   depot  [B] int32 depot node per instance, or NULL (TSP: no depot embedding);
 *   train  0: running statistics; 1: batch statistics over all B*N rows + running-stat update
 *          (momentum 0.1, unbiased variance), graph_encoder.py:150-154;
 *   h      [B][N][128] f32 output embeddings;
 *   gemm_path 0: tcgen05 kind::f16 GEMMs on f16 hi/lo operand halves (~fp32 accuracy, production);
 *             1: fp32 SIMT GEMMs (debug / cross-check);
 *   saved  NULL, or (train mode) a buffer of vrpx_encoder_saved_bytes() that receives the activations the
 *          backward pass needs. */
VRPX_API int vrpx_encoder_forward(const vrpx_encoder_weights* w, const vrpx_env* env, const float* x,
                         const int32_t* depot, int64_t B, int32_t N, int32_t train, float* h, void* ws,
                         int64_t ws_bytes, int32_t gemm_path, float* saved, void* stream);

/* Bytes of the activation buffer `saved` (train mode only; pass NULL when no backward will follow). */
VRPX_API int64_t vrpx_encoder_saved_bytes(int64_t B, int32_t N);

/* Transposed copies of the dense encoder weights (dX = dY · W runs as a forward GEMM on W^T). */
typedef struct vrpx_encoder_layer_t {
  const float* in_proj_wT;  /* [128][384] */
  const float* out_proj_wT; /* [128][128] */
  const float* ff0_wT;      /* [128][512] */
  const float* ff2_wT;      /* [512][128] */
} vrpx_encoder_layer_t;
typedef struct vrpx_encoder_weights_t {
  vrpx_encoder_layer_t layer[VRPX_LAYERS];
} vrpx_encoder_weights_t;

/* Gradient buffers, same shapes as the parameters, ACCUMULATED into (+=). */
typedef struct vrpx_encoder_layer_grads {
  float *in_proj_w, *in_proj_b, *out_proj_w, *out_proj_b, *bn1_w, *bn1_b, *ff0_w, *ff0_b, *ff2_w, *ff2_b, *bn2_w, *bn2_b;
} vrpx_encoder_layer_grads;
typedef struct vrpx_encoder_grads {
  float *node_w, *node_b, *depot_w, *depot_b; /* depot_* may be NULL (TSP) */
  vrpx_encoder_layer_grads layer[VRPX_LAYERS];
} vrpx_encoder_grads;

VRPX_API int64_t vrpx_encoder_backward_workspace_bytes(int64_t B, int32_t N);

/* Backward of the train-mode encoder forward (BatchNorm with batch statistics).  `saved` is the buffer the forward
 * filled; `g` [B][N][128] holds dL/dh on entry and is overwritten (it ends as dL/d(embedding output), in the scale of
 * dL/dh on entry). */
VRPX_API int vrpx_encoder_backward(const vrpx_encoder_weights* w, const vrpx_encoder_weights_t* wt, const vrpx_env* env,
                                   const float* x, const int32_t* depot, int64_t B, int32_t N, const float* saved,
                                   float* g, const vrpx_encoder_grads* grads, void* ws, int64_t ws_bytes,
                                   int32_t gemm_path, void* stream);

/* Decoder parameters after host-side packing (agents/graph_decoder.py:29-44); vrpx/packing.py derives
 * each array from the state_dict (in float64, rounded once to f32).  With W_q/W_k/W_v/b_* the in-projections of
 * decoder.attention, W_o its out_proj, W_ao = _att_output, W_kp = _kp, W_ctx = _context_proj, and
 * Kd = blockdiag_h(W_k,h^T)/sqrt(48)  (1024 x 384; folds the per-head key projection into the query):
 *   ag_t  [128][1024]  (Kd · W_q[:, graph-embedding block])^T      IRP: W_q := W_q · W_ctx
 *   af_t  [128][1024]  same for the `first` block (TSP/VRP only, NULL for IRP)
 *   al_t  [128][1024]  same for the `last` block
 *   a_c   [1024]       Kd · b_q
 *   a_q0  [1024]       step-0 term of the learned placeholders _first_node / _last_node
 *   a_load[1024]       IRP only: Kd · W_q · W_ctx[:, 256]   (multiplied by the f32 vehicle load)
 *   m_t   [1024][128]  row h*128+d: (W_kp^T · W_ao · W_o[:, head h] · W_v,h)[:, d] / sqrt(128)
 *   m_c   [128]        W_kp^T · W_ao · (W_o · b_v + b_o) / sqrt(128)
 *   qk_w  [768][128]   optional (may be NULL): rows 0..383 = W_q[:, last block] / sqrt(48) (IRP: W_q · W_ctx), rows
 *                      384..767 = W_k — the rank-48 factors of al_t per head.  With it (and the larger workspace of
 *                      vrpx_rollout_table_workspace_bytes) a whole-episode vrpx_rollout call builds, once per episode,
 *                      the score table S1[b][l][head][n] = (A_l h[b,l])_head · h[b,n] and runs every decode step as a
 *                      few launches over the whole batch; the steps t >= 2 read their glimpse scores from the table
 *                      instead of recomputing A_l · h[last] and the score pass every step.  Without it, every step
 *                      runs in the persistent kernel (classic mode).
 * The key bias b_k shifts every score of a head equally and cancels in the softmax. */
typedef struct vrpx_decoder_weights {
  const float *ag_t, *af_t, *al_t, *a_c, *a_q0, *a_load;
  const float *m_t, *m_c;
  const float *qk_w;
} vrpx_decoder_weights;

/* Optional per-step history written by vrpx_rollout for the recompute-based backward (any field may be NULL). */
typedef struct vrpx_rollout_trace {
  uint32_t* mask_hist; /* [Tmax][B][4] decoder-visible mask bits BEFORE each step */
  float* load_hist;    /* [Tmax][B] f32 vehicle load before each step (IRP) */
  float* qg0;          /* [B][1024] per-episode query table before the `first` fold */
} vrpx_rollout_trace;

typedef enum vrpx_rollout_mode { VRPX_GREEDY = 0, VRPX_SAMPLE = 1, VRPX_TEACHER = 2 } vrpx_rollout_mode;

VRPX_API int64_t vrpx_rollout_workspace_bytes(int64_t B, int32_t N);
/* Byte offset inside the rollout workspace of the per-episode query table Q~g [B][1024] f32 (read back by the
 * recompute-based backward); the header in front of it holds the barrier/done counters and the pre-split copy of m_t. */
VRPX_API int64_t vrpx_rollout_workspace_qg_offset(void);
/* Workspace size that additionally holds the per-episode glimpse score tables (see qk_w above) and the buffers the
 * split-step launches hand between them.  A whole-episode call (t_begin == 0, Tmax >= 3) given at least this much
 * workspace and a non-NULL qk_w runs in table mode; any other call runs the classic loop in the persistent kernel. */
VRPX_API int64_t vrpx_rollout_table_workspace_bytes(int32_t kind, int64_t B, int32_t N);

/* The rollout loop TSPModel/VRPModel/IRPModel.forward (agents/graph_tsp_agent.py:78-92,
 * graph_vrp_agent.py:69-83, graph_irp_agent.py:82-105) with GraphDecoder.forward
 * (agents/graph_decoder.py:51-115) and the env transition fused, all steps in ONE persistent
 * cooperative launch.  The env must be in its reset state; on return it holds the terminal state.
 *   h        [B][N][128] encoder output
 *   mode     greedy argmax (graph_decoder.py:103), Philox sampling (:105-107), or teacher-forced
 *   coupling glimpse-mask coupling group G (graph_decoder.py:93 `mask.repeat(H,1)`): attention row (b,h)
 *            adds mask[g0 + ((b-g0)*8+h) mod G], g0 = floor(b/G)*G.  G == B is the reference at batch B;
 *            0 disables the quirk's scrambling (adds the instance's own mask) — NOT reference-equal.  Any other value
 *            must divide B (VRPX_ERR_ARG otherwise: the partner row would fall outside the batch).
 *   tape     [Tmax][B] uint8 actions: written (greedy/sample) or read (teacher); may be NULL unless teacher
 *   t_begin  first step to execute: 0 starts an episode (builds the per-episode tables in `ws`); > 0 resumes
 *            one whose `ws`, env state, logp and cost were left by the previous call (single-step decoding)
 *   Tmax     maximum number of steps to run in this call = rows of `tape`/`logits` (row 0 = step t_begin)
 *   logp     [B] f32 sum of log-probs (0 for greedy, graph_decoder.py:100)
 *   cost     [B] f32 = -(acc_loss): f32 accumulation of f32(reward) in step order (graph_tsp_agent.py:85)
 *   steps    [1] int32 number of steps executed (env.step_count)
 *   logits   optional [Tmax][B][N] f32 dump of the masked pointer logits (tests), or NULL
 *   trace    optional history for vrpx_decoder_backward, or NULL
 *   seed/offset  Philox key / global instance-id offset (shard-invariant sampling)            */
VRPX_API int vrpx_rollout(const vrpx_env* env, const vrpx_decoder_weights* w, const float* h, int32_t mode,
                 int64_t coupling, uint64_t seed, uint64_t offset, uint8_t* tape, int32_t t_begin, int32_t Tmax,
                 float* logp, float* cost, int32_t* steps, float* logits, const vrpx_rollout_trace* trace,
                 void* ws, int64_t ws_bytes, void* stream);

/* K sampled episodes per instance from one set of embeddings and one score table (best-of-K decoding).
 * The env holds Bb·K replicas in their reset state, copy-major: replica r = k·Bb + b is copy k of base instance b (same
 * xy / depot / demand).  Copy k is bit-identical to vrpx_rollout(copy k alone, h, VRPX_SAMPLE, coupling, seed,
 * offset + k·Bb, t_begin 0, Tmax) in table mode: tape rows, cost, log-prob and logits.  Each copy ends at its own step
 * count; the launches run until the slowest copy is done, so `steps` is the maximum over the copies, a copy's tape rows
 * after its own step count hold its depot and its logits rows there are not written.
 * The embeddings h [Bb][N][128] and the score table S1 exist once per base instance: the table is built over the Bb
 * base instances, and the decode kernels read both at the replica's base instance.  The always-sampling, whole-episode,
 * table-mode decode loop of vrpx_rollout runs over the Bb·K replicas, the K copies of an instance on neighbouring warps.
 *   Bb, K     base batch and sample count (K >= 1, env->B == Bb·K)
 *   coupling  0 or a divisor of Bb (the partner rows of every copy stay inside the copy)
 *   w         qk_w is required
 *   tape      [Tmax][Bb·K] uint8 actions; logp, cost [Bb·K]; logits optional [Tmax][Bb·K][N]
 *   Tmax      maximum number of steps; Tmax < 3 (TSP with N <= 3) returns VRPX_ERR_UNSUPPORTED
 *   ws        at least vrpx_rollout_samples_workspace_bytes(kind, Bb, K, N) bytes
 * VRPX_ERR_ARG for K < 1, env->B != Bb·K, a bad coupling, a NULL qk_w or a workspace that is too small.
 * vrpx_rollout_samples records no backward trace; it is vrpx_rollout_samples_traced with trace = NULL. */
VRPX_API int64_t vrpx_rollout_samples_workspace_bytes(int32_t kind, int64_t Bb, int32_t K, int32_t N);
VRPX_API int vrpx_rollout_samples(const vrpx_env* env, const vrpx_decoder_weights* w, const float* h, int64_t Bb,
                                  int32_t K, int64_t coupling, uint64_t seed, uint64_t offset, uint8_t* tape, int32_t Tmax,
                                  float* logp, float* cost, int32_t* steps, float* logits, void* ws, int64_t ws_bytes,
                                  void* stream);
/* vrpx_rollout_samples plus the history vrpx_decoder_backward_samples replays (trace may be NULL; any field may be NULL):
 *   mask_hist [Tmax][Bb·K][4], load_hist [Tmax][Bb·K], qg0 [Bb·K][1024], per replica.  Rows before a copy's own step count
 *   equal those of vrpx_rollout(copy k alone, ..., trace) bit for bit; the rows after it, up to the returned step count,
 *   hold the copy's terminal mask and load (the depot is then the only open node, so the replayed steps are inert).
 *   The per-replica Q~g after the `first` fold stays in ws at vrpx_rollout_workspace_qg_offset(). */
VRPX_API int vrpx_rollout_samples_traced(const vrpx_env* env, const vrpx_decoder_weights* w, const float* h, int64_t Bb,
                                         int32_t K, int64_t coupling, uint64_t seed, uint64_t offset, uint8_t* tape,
                                         int32_t Tmax, float* logp, float* cost, int32_t* steps, float* logits,
                                         const vrpx_rollout_trace* trace, void* ws, int64_t ws_bytes, void* stream);

/* Measurement hooks (bench.py, tools/): not part of the reference surface.
 *   vrpx_debug_rollout_profile  device buffer of 8 x int64 that accumulates per-phase cycles of thread 0 of every CTA
 *                               of the rollout kernel (NULL disables)
 *   vrpx_debug_rollout_timing   when enabled, vrpx_rollout brackets the decode launches (persistent kernel + step kernels, without the
 *                               score-table prologue kernels) with CUDA events on the launch stream
 *   vrpx_debug_rollout_kernel_ms  waits for the last bracketed launch and returns its duration (-1 if none) */
VRPX_API void vrpx_debug_rollout_profile(long long* dev_counters);
VRPX_API void vrpx_debug_rollout_timing(int32_t enable);
/* A/B switch of the whole-episode rollout (default 1):
 *   bit 0  set: table mode as described at vrpx_rollout_table_workspace_bytes (score tables, then every decode step is
 *          a handful of launches over the whole batch, rollout_steps.cu);
 *          clear: whole-episode calls skip the tables and run the classic loop in the persistent kernel (cross-check
 *          and A/B measurements)
 *   (programmatic dependent launch of the step kernels was measured and removed: 36.38 vs 36.36 ms per decode loop) */
VRPX_API void vrpx_debug_rollout_split(int32_t enable);
VRPX_API float vrpx_debug_rollout_kernel_ms(void);

/* ---------------------------------------------------------------- REINFORCE backward (decoder part)
 * loss = mean_b(advantage_b * sum_t log p(a_{b,t}))  (agents/graph_tsp_agent.py:179-186).  The backward is
 * recompute-based: it replays every decode step from (h, tape, trace) and back-propagates wts[b] = dL/dlogp_b. */
typedef struct vrpx_decoder_bwd_weights {
  const float* m_n;  /* [128][1024]  = transpose of m_t   (dc  = dq^ · M)   */
  const float* al_n; /* [1024][128]  = transpose of al_t  (dx_l = dq~ · A_l) */
} vrpx_decoder_bwd_weights;

typedef struct vrpx_decoder_grads {
  float* dH;     /* [B][N][128] accumulated (caller zero-fills): dL/dh from scores, glimpse values, logits, h[last] */
  float* D0;     /* [B][1024] dq~ of step 0            (caller zero-fills) */
  float* D1;     /* [B][1024] sum over steps >= 1 of dq~ (caller zero-fills) */
  float* Dl;     /* [B][1024] IRP: sum_t load_t dq~_t  (caller zero-fills; NULL for TSP/VRP) */
  float* d_al_t; /* [128][1024] accumulated */
  float* d_m_t;  /* [1024][128] accumulated */
  float* d_m_c;  /* [128] accumulated */
} vrpx_decoder_grads;

VRPX_API int64_t vrpx_decoder_backward_workspace_bytes(int64_t B, int32_t N);

/* Backward of vrpx_rollout for one episode.  `trace` and `qg` (the rollout workspace's Q~g table = ws + vrpx_rollout_workspace_qg_offset() bytes)
 * come from the forward call that produced `tape`; T = number of executed steps; wts [B] f32. */
VRPX_API int vrpx_decoder_backward(const vrpx_env* env, const vrpx_decoder_weights* w, const vrpx_decoder_bwd_weights* wb,
                                   const float* h, const uint8_t* tape, int32_t T, int64_t coupling,
                                   const vrpx_rollout_trace* trace, const float* qg, const float* wts,
                                   const vrpx_decoder_grads* g, void* ws, int64_t ws_bytes, void* stream);

/* Backward of vrpx_rollout_samples_traced: the K copies of Bb base instances in one launch.  env holds the Bb·K
 * copy-major replicas (only kind, N and B are read); h [Bb][N][128] are the base embeddings the rollout read, and replica
 * r = k·Bb + b reads them at row b.  tape [T][Bb·K], trace, qg [Bb·K][1024] (ws + vrpx_rollout_workspace_qg_offset() of the
 * forward call), wts [Bb·K] and every per-instance gradient buffer of g (dH [Bb·K][N][128], D0, D1, Dl) are per replica:
 * dH is NOT summed over the copies.  T = the step count of the forward call (the slowest copy's).  coupling: 0 or a divisor
 * of Bb.  Workspace: vrpx_decoder_backward_workspace_bytes(Bb·K, N).  K = 1 is vrpx_decoder_backward. */
VRPX_API int vrpx_decoder_backward_samples(const vrpx_env* env, const vrpx_decoder_weights* w,
                                           const vrpx_decoder_bwd_weights* wb, const float* h, int64_t Bb, int32_t K,
                                           const uint8_t* tape, int32_t T, int64_t coupling, const vrpx_rollout_trace* trace,
                                           const float* qg, const float* wts, const vrpx_decoder_grads* g, void* ws,
                                           int64_t ws_bytes, void* stream);

/* Small per-episode helpers used by the backward passes (decoder epilogue, encoder weight gradients):
 *   C[M][N] += A^T · Bm  with A [R][M], Bm [R][N] (reduction over rows, red.add);  out[c] += sum_r X[r][c];
 *   G[b] = mean_n h[b,n], Xf[b] = h[b, tape0[b]];  dH[b,n] += dG[b]/N, dH[b,tape0[b]] += dXf[b]. */
VRPX_API int vrpx_gemm_tn_accumulate(const float* A, const float* Bm, float* C, int64_t R, int32_t M, int32_t N, void* stream);
/* vrpx_gemm_tn_accumulate runs on tcgen05 (csrc/gemm_tn_tc.cu) when M and N are multiples of 128 and R >= 8192;
 * path 1 forces the warp-level mma.sync kernel for every shape (A/B measurements, cross-check in the tests). */
VRPX_API void vrpx_debug_gemm_tn_path(int32_t path);
VRPX_API int vrpx_colsum_accumulate(const float* X, int64_t R, int32_t Ccols, float* out, void* stream);
/* weight and bias gradient of a linear layer in one call: C += A^T · Bm and colsum_A[M] += column sums of A (may be NULL) */
VRPX_API int vrpx_gemm_tn_colsum_accumulate(const float* A, const float* Bm, float* C, float* colsum_A, int64_t R, int32_t M,
                                            int32_t N, void* stream);
VRPX_API int vrpx_episode_gather(const float* h, const uint8_t* tape0, int64_t B, int32_t N, float* G, float* Xf, void* stream);
VRPX_API int vrpx_episode_scatter(float* dH, const uint8_t* tape0, int64_t B, int32_t N, const float* dG, const float* dXf,
                                  void* stream);

/* Test hook (tests/test_gpu_gemm.py): Y[R][NOUT] = epilogue(X[R][K] · W[NOUT][K]^T) through the tcgen05 f16-split
 * path (path 0) or the fp32 SIMT path (path 1); epilogue = +bias, ReLU, +residual, *scale+shift (each optional). */
VRPX_API int vrpx_debug_gemm(const float* X, int64_t R, int32_t K, const float* W, int32_t NOUT, const float* bias,
                             int32_t relu, const float* residual, const float* scale, const float* shift, float* Y,
                             int32_t path, void* stream);

/* Test / measurement hooks of the fused encoder feed-forward kernel (csrc/ff_fused.cu):
 *   vrpx_debug_ff_fused          Y = (residual + relu(X·W1^T + b1)·W2^T + b2) * scale + shift, X/Y/residual [R][128],
 *                                W1 [512][128], W2 [128][512] (graph_encoder.py:177-181,196); scale/shift may be NULL
 *   vrpx_debug_encoder_fuse_ff   1 (default): vrpx_encoder_forward runs the FF block through that kernel whenever no
 *                                activations are saved for a backward pass; 0: two GEMMs (A/B measurements) */
VRPX_API int vrpx_debug_ff_fused(const float* X, int64_t R, const float* W1, const float* b1, const float* W2,
                                 const float* b2, const float* residual, const float* scale, const float* shift, float* Y,
                                 void* stream);
VRPX_API void vrpx_debug_encoder_fuse_ff(int32_t enable);

/* Test / measurement hooks of the fused QKV-projection + self-attention kernel (csrc/attn_fused.cu):
 *   vrpx_debug_qkv_attention            att [B·N][128] = MultiheadAttention core (8 heads, no out-projection) of
 *                                       X [B·N][128] with in_proj_w [384][128], in_proj_b [384] (graph_encoder.py:74-104)
 *   vrpx_debug_encoder_fuse_attention   1 (default): vrpx_encoder_forward runs projection + attention through that kernel
 *                                       whenever no activations are saved; 0: GEMM + attention kernel (A/B measurements) */
VRPX_API int vrpx_debug_qkv_attention(const float* X, const float* in_proj_w, const float* in_proj_b, int64_t B, int32_t N,
                                      float* att, void* stream);
VRPX_API void vrpx_debug_encoder_fuse_attention(int32_t enable);

/* Test hook of the score-table kernel of the split-step rollout (csrc/score_table_fused.cu):
 * s1 [B][N][8][N] = per-head q'·k' of every (last, node) pair with q' = h·(W_l/sqrt(48))^T, k' = h·W_k^T, from h [B·N][128]
 * and qk_w [768][128] (rows 0..383 W_l/sqrt(48), 384..767 W_k, head-major; vrpx/packing.py fold_decoder). */
VRPX_API int vrpx_debug_score_table(const float* h, const float* qk_w, int64_t B, int32_t N, float* s1, void* stream);

/* Test hook of the attention backward (csrc/attention_bwd.cu): dqkv [B·N][384] = d(loss)/d(qkv) of the per-instance
 * 8-head attention core given qkv [B·N][384], its output att [B·N][128] and datt = d(loss)/d(att)
 * (path 0: mma.sync f16-split kernel = production; path 1: fp32 SIMT kernel). */
VRPX_API int vrpx_debug_attention_backward(const float* qkv, const float* att, const float* datt, float* dqkv, int64_t B,
                                           int32_t N, int32_t path, void* stream);

/* Test hook of the encoder backward (csrc/encoder_bwd.cu): vrpx_encoder_backward with the same arguments and launches,
 * plus, for every layer whose bit is set in layer_mask (1..7), the gradients its kernels hold inside that layer, in the
 * scale of g on entry.  The selected layers' blocks follow each other in ascending layer order in `stages`; each layer's
 * part is eight stage-major blocks of R = B·N rows, 1,664 floats per row:
 *   dOUT [R][128] (g on entry to the layer), dY2 [R][128] (after the BN2 backward), dPRE [R][512] (after the ReLU-gate
 *   GEMM), dH1 [R][128] (after the residual GEMM), dY1 [R][128] (after the BN1 backward), dATT [R][128],
 *   dQKV [R][384] (after the attention backward), dX [R][128] (g after the in-projection GEMM).
 * Each block is one device-to-device cudaMemcpyAsync on `stream`. */
VRPX_API int vrpx_debug_encoder_backward_stages(const vrpx_encoder_weights* w, const vrpx_encoder_weights_t* wt,
                                                const vrpx_env* env, const float* x, const int32_t* depot, int64_t B,
                                                int32_t N, const float* saved, float* g, const vrpx_encoder_grads* grads,
                                                void* ws, int64_t ws_bytes, int32_t gemm_path, float* stages,
                                                int32_t layer_mask, void* stream);

/* Number of kernels this library has launched since load (bench.py's gpu_launches claim). */
VRPX_API int64_t vrpx_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* VRPX_H */
