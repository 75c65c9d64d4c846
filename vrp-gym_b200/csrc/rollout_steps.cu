// rollout_steps.cu — split-step form of the table-mode decode steps t >= 2 of vrpx_rollout.
//
// The persistent kernel (rollout.cu) is bound by L2 bandwidth: a 16-instance tile re-streams the 512 KiB of folded
// GEMM-B weights from L2 on every SM (32 KB per instance-step) and the embeddings cross L2 twice per step.  Larger
// tiles are not possible inside one CTA (shared memory, and the L2 working set of the embeddings).  Here the three
// phases of a table step become three launches over the WHOLE batch, with the kernel boundary as the grid barrier the
// mask coupling needs (SURVEY App. B-3):
//   k_step_glimpse   one warp per instance: scores from the per-episode tables, softmax, glimpse values
//                    c_h = sum_n p_hn h_n (mma.sync TF32 3-term split)  ->  c [B][1024] f32
//   gemm_tc          q^ = c · M^T + m_c as ONE batched tcgen05 GEMM (R = B, K = 1024, NOUT = 128): the weights are read
//                    once per 128 instances instead of once per 16
//   k_step_pointer   one warp per instance: logits 10 tanh(q^ · h_n), mask, argmax / Philox sample / teacher action,
//                    log-prob; then one thread per instance runs the environment transition (env_rules.cuh)
// Softmax, glimpse values and pointer phase are those of phases P2 and P4 of the persistent kernel: both call the helpers
// of glimpse_mma.cuh (warp_load_by_head, warp_node_softmax, warp_store_by_node, warp_glimpse_values_acc) and rollout.cuh
// (step0_query, record_trace, warp_masked_logits, warp_pointer_choice, rollout_env_step).  Against
// its classic loop the results differ only by the evaluation order of the scores (tables) and the summation order inside
// GEMM-B.  The classic mode and resumed single-step calls run in the persistent kernel.
// The launches are asynchronous on the caller's stream: no host round trip per step.  An episode that finishes early
// (VRP / IRP) turns the remaining launches into no-ops through the per-step `notdone` counters.
#include "gemm.cuh"
#include "rollout.cuh"
#include "glimpse_mma.cuh"

namespace vrpx {

constexpr int SW = 8;   // warps (= instances) per CTA of the pointer kernel
// glimpse kernel: up to 10 warps per CTA, two CTAs per SM.  Every warp streams its instance's embeddings through a
// private cp.async ring of GNS slices of 8 node rows (rows padded to 544 B: the LDS.128 fragment reads are conflict free),
// so the loads in flight cost no registers; the P[n][8] slot behind the ring is sized by N.  Measured at C4: the kernel is
// bound by dependent-instruction latency, i.e. by the number of resident warps (11 warps: 451 us, as much as the
// register-staged version at 15 warps with its exposed load latency).
constexpr int GW_MAX = 10, GNS = 2;
constexpr int G_ROW = 544;                          // bytes per staged node row (512 + 32)
constexpr int G_SLICE = 8 * G_ROW;                  // 4352 B
constexpr int G_CTA_SMEM = 113 * 1024;              // two CTAs per SM
static_assert(GNS * G_SLICE >= QW * 4, "c[1024] is staged in the ring");
__host__ __device__ inline int glimpse_warp_bytes(int N) { return GNS * G_SLICE + ((N * NH * 4 + 15) & ~15); }

// true when the episode was over before step trel: nobody was unfinished at the previous step
__device__ __forceinline__ bool episode_over(const RolloutParams& p, int trel) {
  return trel > 0 && ld_acquire_i(p.notdone + trel - 1) == 0;
}

// A finished VRP / IRP instance idles on its depot until the slowest instance of the batch is done (tsp.py:103-104): all
// nodes are visited and the vehicle stands on the depot, so rule R3 leaves the depot as the ONLY feasible node.  Its action
// (the depot), its reward (0), its log-prob (log 1 = 0 exactly) do not depend on the logits, so the step kernels skip
// the glimpse and the embedding gather for it — unless the caller asked for the logits themselves (tests).  `own` = the
// instance's decoder-visible mask words.  (At the depot rule R1 masks the depot unless everything is visited, so
// "the depot is the only candidate while cur == depot" is exactly "finished".)
__device__ __forceinline__ bool instance_idle(const uint32_t (&own)[4], int N, int cur, int depot) {
  if (cur != depot) return false;
  const Bits128 full = full_bits(N);
  int cand = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) cand += __popc(~own[i] & full.w[i]);
  return cand == 1 && !((own[depot >> 5] >> (depot & 31)) & 1u);
}

// A copy whose own episode is over skips the step, but the backward replays every replica for the launches' step count
// (the slowest copy's): its trace rows there get the copy's terminal mask and load, the tape rows get the depot
// (k_step_pointer), so the replayed step has the depot as its only open node (instance_idle) and contributes nothing.
__device__ __forceinline__ void record_terminal(const RolloutParams& p, int64_t r, int trel, int lane) {
  if (p.mask_hist || p.load_hist) record_trace(p, r, trel, (float)p.env.load[r], lane);
}

// ---------------------------------------------------------------- glimpse: tables -> softmax -> c
__global__ void __launch_bounds__(GW_MAX * 32, 2) k_step_glimpse(const RolloutParams p, int t) {
  extern __shared__ __align__(16) unsigned char gsm[];
  const int trel = t - p.t0;
  if (episode_over(p, trel)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = p.env.N, kind = p.env.kind;
  const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (s >= p.env.B) return;
  const SlotReplica sr = slot_replica(p, s);
  if (copy_over(p, sr.k, trel)) {   // see record_terminal
    record_terminal(p, sr.r, trel, lane);
    return;
  }
  const int64_t b = sr.r;
  unsigned char* ring = gsm + warp * glimpse_warp_bytes(N);
  float* slot = reinterpret_cast<float*>(ring + GNS * G_SLICE);
  const int g = lane >> 2, tq = lane & 3;
  const float4* hrow = reinterpret_cast<const float4*>(p.h + sr.b * N * E);
  // slice s = node rows 8s .. 8s+7 -> ring stage s % GNS; lane = 16-byte chunk of the row
  auto issue_slice = [&](int sidx) {
    unsigned char* dst = ring + (sidx % GNS) * G_SLICE + lane * 16;
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (8 * sidx + r < N) cp_async16(dst + r * G_ROW, hrow + (8 * sidx + r) * (E / 4) + lane);
    cp_async_commit();
  };
  const int nsl = (N + 7) / 8;
  if (kind != VRPX_TSP && !p.logits) {   // idle finished instance: its step needs no glimpse and no embeddings (see instance_idle)
    uint32_t own[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) own[i] = __ldcg(p.env.mask + b * 4 + i);
    if (instance_idle(own, N, __ldcg(p.env.cur + b), __ldg(p.env.depot + b))) {
      record_trace(p, b, trel, (float)p.env.load[b], lane);
      return;
    }
  }
#pragma unroll
  for (int sidx = 0; sidx < GNS; ++sidx) {
    if (sidx < nsl) issue_slice(sidx);
    else cp_async_commit();
  }
  const float lf = (float)p.env.load[b];
  record_trace(p, b, trel, lf, lane);

  // ---- scores = S1[b][last] + S0[b] (+ load · SL[b]) + scrambled additive mask (graph_decoder.py:93-94)
  float pr[NH][4];
  {
    const int last = __ldcg(p.env.cur + b);
    const float* r1 = p.s1 + (((size_t)sr.b * N + last) * NH) * N;
    const float* r0 = p.s0 + (size_t)b * NH * N;
    const float* rl = p.sl + (size_t)b * NH * N;
    // lane j holds mask word (j & 3) of the instance whose mask the reference adds to head j >> 2
    const uint32_t mword = __ldcg(p.env.mask + quirk_row(b, lane >> 2, p.G) * 4 + (lane & 3));
    // All table loads of a 32-node stride are issued before the first one is used (clamped addresses instead of
    // predicated loads: the source-level profile showed one exposed DRAM round trip per (head, stride) otherwise).
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (32 * i >= N) {   // uniform: no node in this stride
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) pr[hh][i] = -INFINITY;
        continue;
      }
      const int n = lane + 32 * i, nc = (n < N) ? n : N - 1;
      float v1[NH], v0[NH], vl[NH];
#pragma unroll
      for (int hh = 0; hh < NH; ++hh) {
        v1[hh] = __ldg(r1 + hh * N + nc);
        v0[hh] = __ldcg(r0 + hh * N + nc);
        vl[hh] = (kind == VRPX_IRP) ? __ldcg(rl + hh * N + nc) : 0.f;
      }
#pragma unroll
      for (int hh = 0; hh < NH; ++hh) {
        const uint32_t wsel = __shfl_sync(0xffffffffu, mword, hh * 4 + i);
        float v = v1[hh] + v0[hh];
        if (kind == VRPX_IRP) v = fmaf(lf, vl[hh], v);
        v += (float)((wsel >> lane) & 1u);
        pr[hh][i] = (n < N) ? v : -INFINITY;
      }
    }
  }
#pragma unroll
  for (int hh = 0; hh < NH; ++hh) warp_node_softmax(pr[hh], N);
  warp_store_by_node(slot, pr, N, lane);
  __syncwarp();
  // ---- c[head][dim] = sum_n P[n][head] h_n[dim], the node rows from the ring
  float cacc[8][4];
  warp_glimpse_values_acc(cacc, slot, N, lane, [&](int n0, float4 (&va)[4], float4 (&vb)[4]) {
    const int sidx = n0 >> 3;
    cp_async_wait<GNS - 1>();   // slice sidx has landed (one group per slice, possibly empty, keeps the count uniform)
    __syncwarp();
    const unsigned char* st = ring + (sidx % GNS) * G_SLICE;
#pragma unroll
    for (int cq = 0; cq < 4; ++cq) {
      va[cq] = *reinterpret_cast<const float4*>(st + tq * G_ROW + (8 * cq + g) * 16);
      vb[cq] = *reinterpret_cast<const float4*>(st + (tq + 4) * G_ROW + (8 * cq + g) * 16);
    }
    if (n0 + 8 > N) {   // uniform: only the last slice has rows beyond N (stale ring contents)
#pragma unroll
      for (int cq = 0; cq < 4; ++cq) {
        if (n0 + tq >= N) va[cq] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (n0 + tq + 4 >= N) vb[cq] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    __syncwarp();   // every lane has read the stage before it is refilled
    if (sidx + GNS < nsl) issue_slice(sidx + GNS);
    else cp_async_commit();
  });
  cp_async_wait<0>();
  // c staged in the (now idle) ring, then one coalesced copy
  float* cst = reinterpret_cast<float*>(ring);
  warp_glimpse_store_c(cst, cacc, lane);
  float4* dst = reinterpret_cast<float4*>(p.cbuf + b * QW);
  for (int i = lane; i < QW / 4; i += 32) dst[i] = *reinterpret_cast<const float4*>(cst + 4 * i);
}

// ---------------------------------------------------------------- pointer: logits -> action -> environment
__global__ void __launch_bounds__(SW * 32) k_step_pointer(const RolloutParams p, int t) {
  __shared__ float s_slot[SW][VRPX_MAX_NODES];
  __shared__ float s_lp[SW];
  __shared__ int64_t s_rep[SW];
  __shared__ int s_act[SW], s_anyleft;
  const int trel = t - p.t0;
  if (episode_over(p, trel)) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.env.N, kind = p.env.kind;
  // the CTAs walk the warp slots (slot_replica) in the opposite direction to the glimpse kernel: the embeddings that
  // kernel read last are still in L2 when this one starts, and the ones read last here are there for the next step's
  // glimpse kernel
  const int64_t B = p.env.B, base = (int64_t)(gridDim.x - 1 - blockIdx.x) * SW;
  const int cnt = (int)((B - base < SW) ? (B - base) : SW);
  if (tid == 0) s_anyleft = 0;
  const SlotReplica sr = slot_replica(p, base + (warp < cnt ? warp : 0));
  if (warp < cnt && copy_over(p, sr.k, trel)) {   // the copy's own episode is over: depot in the tape, nothing else changes
    if (lane == 0) {
      if (p.tape) p.tape[(int64_t)trel * p.env.B + sr.r] = (uint8_t)__ldg(p.env.depot + sr.r);
      s_act[warp] = -1;
    }
  } else if (warp < cnt) {
    const int64_t b = sr.r;
    float* slot = s_slot[warp];
    const float4 qh = __ldcg(reinterpret_cast<const float4*>(p.qhat + b * E) + lane);
    const float4* hp = reinterpret_cast<const float4*>(p.h + sr.b * N * E) + lane;
    // own mask (graph_decoder.py:98).  The logits of masked nodes are never used (they become -inf below), so only the
    // embedding rows of the CANDIDATE nodes are read: on average half of the instance over an episode.
    const Bits128 full = full_bits(N);
    uint32_t mw[4], cand[4];
    int cum[5];
    cum[0] = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      mw[i] = __ldcg(p.env.mask + b * 4 + i);
      cand[i] = ~mw[i] & full.w[i];
      cum[i + 1] = cum[i] + __popc(cand[i]);
    }
    // idle finished instance (see instance_idle): the depot is the only candidate and nobody reads its logit
    const bool idle = kind != VRPX_TSP && !p.logits && instance_idle(mw, N, __ldcg(p.env.cur + b), __ldg(p.env.depot + b));
    const int total = idle ? 0 : cum[4];
    // The candidate list is resolved ONCE: lane l holds the node indices of candidates l, l + 32, l + 64, l + 96 (-1 beyond
    // the list), so the gather loop below takes its row indices from registers (find-nth-set-bit inside the loop sat on
    // the critical path of every 8-row chunk).
    int cidx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int j = lane + 32 * k;
      cidx[k] = -1;
      if (j < total) {
        const int w = (j >= cum[1]) + (j >= cum[2]) + (j >= cum[3]);
        const uint32_t word = w == 0 ? cand[0] : (w == 1 ? cand[1] : (w == 2 ? cand[2] : cand[3]));
        const int base_cnt = w == 0 ? 0 : (w == 1 ? cum[1] : (w == 2 ? cum[2] : cum[3]));
        cidx[k] = 32 * w + (int)__fns(word, 0, j - base_cnt + 1);
      }
    }
    // node index of candidate j (warp-uniform j): from the lane / register that resolved it
    auto cand_node = [&](int j) {
      const int k = j >> 5;
      const int v = k == 0 ? cidx[0] : (k == 1 ? cidx[1] : (k == 2 ? cidx[2] : cidx[3]));
      return (j < total) ? __shfl_sync(0xffffffffu, v, j & 31) : -1;
    };
    {
      float4 nxt[8];
      int nn[8];   // nodes of the chunk in flight
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        nn[i] = cand_node(i);
        nxt[i] = (nn[i] >= 0) ? __ldg(hp + nn[i] * (E / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      for (int j0 = 0; j0 < total; j0 += 8) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 hv = nxt[i];
          v[i] = fmaf(qh.x, hv.x, fmaf(qh.y, hv.y, fmaf(qh.z, hv.z, qh.w * hv.w)));
        }
        int nsel = -1;   // node of the sum this lane group reduces: candidate j0 + ((lane >> 2) & 7)
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if (((lane >> 2) & 7) == i) nsel = nn[i];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          nn[i] = cand_node(j0 + 8 + i);
          nxt[i] = (nn[i] >= 0) ? __ldg(hp + nn[i] * (E / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        const float sc = reduce8(v, lane);
        if ((lane & 3) == 0 && nsel >= 0) slot[nsel] = 10.0f * tanhf(sc);
      }
    }
    __syncwarp();
    float u[4];
    warp_masked_logits(u, slot, mw, N, lane, idle);
    const PointerChoice c = warp_pointer_choice(u, p, b, t, trel, lane);
    if (lane == 0) { s_act[warp] = c.a; s_lp[warp] = c.lp; s_rep[warp] = b; }
  }
  __syncthreads();
  // environment transition: one THREAD per instance (the dependent global loads of the CTA's instances overlap)
  if (tid < cnt && s_act[tid] >= 0) {
    const bool unfinished = rollout_env_step(p, s_rep[tid], s_act[tid], s_lp[tid], t, trel).unfinished;
    if (unfinished) s_anyleft = 1;   // benign race: all writers store 1
    if (p.replica_left) p.replica_left[s_rep[tid]] = unfinished;
  }
  __syncthreads();
  if (tid == 0 && s_anyleft) atomicAdd(p.notdone + trel, 1);
}

// K > 1: copy_left[trel][k] = 1 when some replica of copy k was unfinished after step trel (replica_left, written by
// k_step_pointer), one thread per replica and one store per warp and copy
__global__ void __launch_bounds__(256) k_copy_left(const RolloutParams p, int t) {
  const int trel = t - p.t0;
  if (episode_over(p, trel)) return;
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool unfinished = r < p.env.B && __ldcg(p.replica_left + r) != 0;
  const int k = r < p.env.B ? (int)(r / p.Bb) : 0;
  const unsigned peers = __match_any_sync(0xffffffffu, k) & __ballot_sync(0xffffffffu, unfinished);
  if (unfinished && (threadIdx.x & 31) == __ffs(peers) - 1) p.copy_left[(int64_t)trel * p.K + k] = 1;
}

static int launch_pointer(const RolloutParams& p, int t, unsigned grid, cudaStream_t stream) {
  k_step_pointer<<<grid, SW * 32, 0, stream>>>(p, t);
  VRPX_LAUNCH_CHECK();
  if (p.K > 1) {
    k_copy_left<<<(unsigned)((p.env.B + 255) / 256), 256, 0, stream>>>(p, t);
    VRPX_LAUNCH_CHECK();
  }
  return VRPX_OK;
}


// ---------------------------------------------------------------- steps 0 and 1 in split form
// The first two steps have no table row yet: step 0 runs on the learned placeholders (q~ = Q~g + a_q0, graph_decoder.py:79-81),
// step 1 completes the per-episode tables (Q~g += A_f h[first]; S0 = Q~g_head · h_n; IRP: SL = a_load_head · h_n).  They
// used to run inside the persistent kernel (4.7 ms at C4, L2-bound on 16-instance tiles); here they are whole-batch
// launches like every later step: a mean / gather kernel (k_episode_gather in decoder_bwd.cu, k_gather_cur), a batched
// tcgen05 GEMM for the 128 -> 1024 query fold, and a glimpse kernel that computes the scores from q~ itself (one warp per
// instance, mma.sync TF32 3-term: the score and value contractions of glimpse_mma.cuh) instead of reading them from the
// tables.

// Xf[b] = h[b mod Bb, cur[b]]: the first chosen node after step 0 (graph_decoder.py:108-113) of every replica
__global__ void __launch_bounds__(256) k_gather_cur(const float* __restrict__ h, const int* __restrict__ cur, int64_t B,
                                                    int64_t Bb, int N, float* __restrict__ Xf) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= B) return;
  const int c = __ldcg(cur + b);
  const int64_t hb = (b < Bb) ? b : b % Bb;
  reinterpret_cast<float4*>(Xf + b * E)[lane] = __ldg(reinterpret_cast<const float4*>(h + (hb * N + c) * E) + lane);
}

// dst[c][r] = src[r][c]
__global__ void k_transpose(const float* __restrict__ src, int rows, int cols, float* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int r = i / cols, c = i - r * cols;
  dst[(size_t)c * rows + r] = src[i];
}

constexpr int FW = 8;   // warps (= instances) per CTA of the first-step glimpse kernel
__global__ void __launch_bounds__(FW * 32, 2) k_step_glimpse_first(const RolloutParams p, int t) {
  __shared__ __align__(16) float s_slot[FW][QW];
  const int trel = t - p.t0;
  if (episode_over(p, trel)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int N = p.env.N, kind = p.env.kind;
  const int64_t s = (int64_t)blockIdx.x * FW + warp;
  if (s >= p.env.B) return;
  const SlotReplica sr = slot_replica(p, s);
  if (copy_over(p, sr.k, trel)) {
    record_terminal(p, sr.r, trel, lane);
    return;
  }
  const int64_t b = sr.r;
  float* slot = s_slot[warp];
  const int tq = lane & 3;
  const float4* hrow = reinterpret_cast<const float4*>(p.h + sr.b * N * E);
  const float lf = (float)p.env.load[b];
  record_trace(p, b, trel, lf, lane);
  // ---- q~: step 0 = Q~g + a_q0 (+ load · a_load); step 1 = the finished Q~g (its scores are S0, kept for every later step)
  {
    const float* qg = p.qg + b * QW;
    for (int c = lane; c < QW; c += 32)
      slot[c] = (t == 0) ? step0_query(qg, p.w.a_q0, p.w.a_load, kind == VRPX_IRP, lf, c) : qg[c];
  }
  __syncwarp();
  float* s0 = (t == 1) ? p.s0 + (size_t)b * NH * N : nullptr;
  warp_glimpse_scores(slot, hrow, N, lane, [&](int n, int which, float v) {
    slot[(2 * tq + which) * E + n] = v;
    if (s0) s0[(2 * tq + which) * N + n] = v;
  });
  __syncwarp();
  float pr[NH][4];
#pragma unroll
  for (int hh = 0; hh < NH; ++hh) warp_load_by_head(pr[hh], slot + hh * E, N, lane);
  __syncwarp();
  if (t == 1) {
    if (kind == VRPX_IRP) {   // SL = a_load_head · h_n, and its share of this step's scores
      for (int i = lane; i < QW / 4; i += 32)
        *reinterpret_cast<float4*>(slot + 4 * i) = __ldg(reinterpret_cast<const float4*>(p.w.a_load) + i);
      __syncwarp();
      float* sl = p.sl + (size_t)b * NH * N;
      warp_glimpse_scores(slot, hrow, N, lane, [&](int n, int which, float v) {
        slot[(2 * tq + which) * E + n] = v;
        sl[(2 * tq + which) * N + n] = v;
      });
      __syncwarp();
#pragma unroll
      for (int hh = 0; hh < NH; ++hh)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int n = lane + 32 * i;
          if (n < N) pr[hh][i] = fmaf(lf, slot[hh * E + n], pr[hh][i]);
        }
      __syncwarp();
    }
    // + the table row of the node chosen at step 0: (A_l h[last])_head · h_n
    const int last = __ldcg(p.env.cur + b);
    const float* r1 = p.s1 + (((size_t)sr.b * N + last) * NH) * N;
#pragma unroll
    for (int hh = 0; hh < NH; ++hh)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int n = lane + 32 * i;
        if (n < N) pr[hh][i] += __ldg(r1 + hh * N + n);
      }
  }
  // ---- scrambled additive mask (graph_decoder.py:93-94): lane j holds word (j & 3) of the mask added to head j >> 2
  {
    const uint32_t mword = __ldcg(p.env.mask + quirk_row(b, lane >> 2, p.G) * 4 + (lane & 3));
#pragma unroll
    for (int hh = 0; hh < NH; ++hh)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t wsel = __shfl_sync(0xffffffffu, mword, hh * 4 + i);
        pr[hh][i] += (float)((wsel >> lane) & 1u);   // -inf stays -inf for the lanes beyond N
      }
  }
#pragma unroll
  for (int hh = 0; hh < NH; ++hh) warp_node_softmax(pr[hh], N);
  warp_store_by_node(slot, pr, N, lane);
  __syncwarp();
  // ---- c[head][dim] = sum_n P[n][head] h_n[dim] (the second pass over the instance's embeddings comes from L2)
  warp_glimpse_values(slot, hrow, N, lane);
  float4* dst = reinterpret_cast<float4*>(p.cbuf + b * QW);
  for (int i = lane; i < QW / 4; i += 32) dst[i] = *reinterpret_cast<const float4*>(slot + 4 * i);
}

// steps executed = first step at whose start nobody was unfinished (it still runs, like the reference's loop), else Tmax
__global__ void k_rollout_finish(const int* __restrict__ notdone, int t0, int Tmax, int* __restrict__ steps) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int t = t0 + Tmax;
  for (int i = 0; i < Tmax; ++i)
    if (notdone[i] == 0) { t = t0 + i + 1; break; }
  *steps = t;
}

int prepare_split_weights(const RolloutParams& p, const SplitWorkspace& w, GemmPlan* plan_b, cudaStream_t stream) {
  k_transpose<<<QW * E / 256, 256, 0, stream>>>(p.w.m_t, QW, E, w.m_nt);
  VRPX_LAUNCH_CHECK();
  k_transpose<<<QW * E / 256, 256, 0, stream>>>(p.w.ag_t, E, QW, w.ag_n);
  VRPX_LAUNCH_CHECK();
  if (p.w.af_t) {
    k_transpose<<<QW * E / 256, 256, 0, stream>>>(p.w.af_t, E, QW, w.af_n);
    VRPX_LAUNCH_CHECK();
  }
  // GEMM-B runs on the same buffers at every step: split m_t^T and encode its tensor maps once per rollout
  GemmArgs ga{p.cbuf, p.env.B, QW, w.m_nt, E, p.w.m_c, 0, nullptr, nullptr, nullptr, p.qhat};
  return gemm_tc_plan(ga, w.w16b, plan_b, stream);
}

static unsigned glimpse_launch_shape(int N, int64_t B, int* warps, size_t* smem) {
  int gw = G_CTA_SMEM / glimpse_warp_bytes(N);
  if (gw > GW_MAX) gw = GW_MAX;
  *warps = gw;
  *smem = (size_t)gw * glimpse_warp_bytes(N);
  return (unsigned)((B + gw - 1) / gw);
}

// steps 0 and 1 of a whole-episode table-mode rollout (p.t0 == 0)
int run_first_steps(const RolloutParams& p, const SplitWorkspace& w, const GemmPlan& plan_b, cudaStream_t stream) {
  const int64_t B = p.env.B;
  const int N = p.env.N;
  const unsigned g8 = (unsigned)((B + 7) / 8), grid_p = (unsigned)((B + SW - 1) / SW), grid_f = (unsigned)((B + FW - 1) / FW);
  int rc;
  // ---- step 0: Q~g = A_g · mean_n h + a_c (the graph part of the folded query) over the base instances, copied into
  // the rows of the other K - 1 copies (copy-major: one contiguous block each), then the placeholder step
  if ((rc = launch_episode_gather(p.h, nullptr, p.Bb, N, p.qhat, nullptr, stream))) return rc;
  GemmArgs g0{p.qhat, p.Bb, E, w.ag_n, QW, p.w.a_c, 0, nullptr, nullptr, nullptr, p.qg};
  if ((rc = gemm_tc(g0, stream))) return rc;
  const size_t qg_block = (size_t)p.Bb * QW * sizeof(float);
  for (int k = 1; k < p.K; ++k)
    VRPX_CUDA(cudaMemcpyAsync(p.qg + (size_t)k * p.Bb * QW, p.qg, qg_block, cudaMemcpyDeviceToDevice, stream));
  if (p.qg0) VRPX_CUDA(cudaMemcpyAsync(p.qg0, p.qg, (size_t)B * QW * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  k_step_glimpse_first<<<grid_f, FW * 32, 0, stream>>>(p, 0);
  VRPX_LAUNCH_CHECK();
  if ((rc = gemm_tc_launch(plan_b, stream))) return rc;
  if ((rc = launch_pointer(p, 0, grid_p, stream))) return rc;
  if (p.Tmax < 2) return VRPX_OK;
  // ---- step 1: fold the first chosen node into Q~g (graph_decoder.py:111-113; IRP has no `first` term), build S0 (, SL)
  if (p.env.kind != VRPX_IRP) {
    k_gather_cur<<<g8, 256, 0, stream>>>(p.h, p.env.cur, B, p.Bb, N, p.qhat);
    VRPX_LAUNCH_CHECK();
    GemmArgs g1{p.qhat, B, E, w.af_n, QW, nullptr, 0, p.qg, nullptr, nullptr, p.qg};
    if ((rc = gemm_tc(g1, stream))) return rc;
  }
  k_step_glimpse_first<<<grid_f, FW * 32, 0, stream>>>(p, 1);
  VRPX_LAUNCH_CHECK();
  if ((rc = gemm_tc_launch(plan_b, stream))) return rc;
  if ((rc = launch_pointer(p, 1, grid_p, stream))) return rc;
  return VRPX_OK;
}

int run_split_steps(const RolloutParams& p, int t_first, const GemmPlan& plan_b, cudaStream_t stream) {
  const int64_t B = p.env.B;
  int gw;
  size_t smem;
  const unsigned ggrid = glimpse_launch_shape(p.env.N, B, &gw, &smem), grid = (unsigned)((B + SW - 1) / SW);
  VRPX_CUDA(cudaFuncSetAttribute(k_step_glimpse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  for (int t = t_first; t < p.t0 + p.Tmax; ++t) {
    k_step_glimpse<<<ggrid, gw * 32, smem, stream>>>(p, t);
    VRPX_LAUNCH_CHECK();
    int rc = gemm_tc_launch(plan_b, stream);
    if (rc) return rc;
    if ((rc = launch_pointer(p, t, grid, stream))) return rc;
  }
  k_rollout_finish<<<1, 32, 0, stream>>>(p.notdone, p.t0, p.Tmax, p.steps);
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}

}  // namespace vrpx
