// decoder_bwd.cu — recompute-based backward of the fused decoder rollout (REINFORCE path,
// agents/graph_tsp_agent.py:178-186: loss = mean(advantage * sum_t log p(a_t)); loss.backward()).
//
// Given the action tape, every decode step depends only on (h, tape, packed weights): step t reads
// last = tape[t-1], first = tape[0], the recorded masks and loads.  So instead of storing (B,T,·) activations the
// backward RECOMPUTES each step's forward (same tile GEMMs / per-instance helpers as rollout.cu) and immediately
// back-propagates d(logp_{b,t}) * w_b, accumulating
//     dH            (B,N,128)   gradient w.r.t. the encoder output (all paths: scores, glimpse values, pointer
//                               logits, h[last]; the graph-mean / h[first] terms are added by the epilogue)
//     d_al_t, d_m_t, d_m_c      gradients of the packed per-step weights (red.global.add)
//     D0, D1 (B,1024)           dq~ at step 0 / summed over steps >= 1  -> per-episode terms (A_g, A_f, a_c, a_q0)
//     Dl (B,1024)               IRP: sum_t load_t * dq~_t -> a_load
// Tiles are the outer loop and steps the inner loop, so a CTA owns its instances' dH rows for the whole episode
// (plain read-modify-write, L2 resident) and no grid barrier is needed.
//
// Notation (DESIGN.md §3.3):  q~ = A_l x_l + Q~g (+ load a_load);  s_hn = q~_h·h_n + mask;  p = softmax_n(s);
// c_h = sum_n p_hn h_n;  q^ = M c + m_c;  z_n = q^·h_n;  u_n = 10 tanh z_n;  pi = softmax(u | unmasked).
#include "gemm.cuh"
#include "glimpse_mma.cuh"
#include "rollout.cuh"

namespace vrpx {

constexpr int SCQ = 4;   // 1024-float scratch slots per instance

struct DecBwdParams {
  int kind, N, T;
  long long B, G;
  // K sampled copies (vrpx_decoder_backward_samples): replica b = k·Bb + b' reads the embeddings h [Bb][N][128] of its
  // base instance b' = b mod Bb; every other per-instance array (tape, trace, qg, wts, dH, D0, D1, Dl) is per replica.
  // vrpx_decoder_backward: Bb = B.
  long long Bb;
  const float* h;
  const uint8_t* tape;
  const uint32_t* mask_hist;
  const float* load_hist;
  const float *qg0, *qg;
  const float* wts;
  const float *al_t, *a_q0, *a_load, *m_t, *m_c, *m_n, *al_n;
  float *dH, *D0, *D1, *Dl, *d_al_t, *d_m_t, *d_m_c;
  float* scratch;  // [grid][TM][4][1024]: q~ | p[n][8] | dz[128], q^[128] | dc
};

// Xs | QC | Wb | DQ with the padded leading dimensions of the tensor-pipe tile GEMMs (XS_LD, QC_LD): 225.5 KiB
constexpr size_t BWD_X = (size_t)TM * XS_LD * sizeof(float), BWD_QC = (size_t)TM * QC_LD * sizeof(float);
constexpr size_t BWD_SMEM = BWD_X + BWD_QC + SMEM_W + BWD_X;

__device__ __forceinline__ void red_add2(float* p, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}

// dst[r][c] += sum_m A[m][r] Bm[m][c] for the 16 x 64 block r < 16, c < 64, m over the TM instances of the tile (the
// weight gradients of B5 / B8).  Tensor pipe, TF32 3-term: A fragment (row r, col m) = A[m][r], B fragment (row m, col c)
// = Bm[m][c]; every accumulator sums the k-steps in order, then red.global.add.
__device__ __forceinline__ void warp_outer_product_tm(const float* A, int lda, const float* Bm, int ldb, float* dst, int ldd,
                                                      int lane) {
  const int g = lane >> 2, t4 = lane & 3;
  float acc[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
#pragma unroll
  for (int ks = 0; ks < TM / 8; ++ks) {
    uint32_t ah[4], al[4];
    const float* r0 = A + (ks * 8 + t4) * lda + g;
    const float* r1 = r0 + 4 * lda;
    split_tf32(r0[0], ah[0], al[0]);
    split_tf32(r0[8], ah[1], al[1]);
    split_tf32(r1[0], ah[2], al[2]);
    split_tf32(r1[8], ah[3], al[3]);
    const float* b0p = Bm + (ks * 8 + t4) * ldb + g;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      uint32_t bh0, bl0, bh1, bl1;
      split_tf32(b0p[8 * j], bh0, bl0);
      split_tf32(b0p[4 * ldb + 8 * j], bh1, bl1);
      mma_tf32_16x8x8(acc[j], al, bh0, bh1);
      mma_tf32_16x8x8(acc[j], ah, bl0, bl1);
      mma_tf32_16x8x8(acc[j], ah, bh0, bh1);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float* d = dst + (size_t)g * ldd + 8 * j + 2 * t4;
    red_add2(d, acc[j][0], acc[j][1]);
    red_add2(d + 8 * ldd, acc[j][2], acc[j][3]);
  }
}

// embedding rows of replica b: those of its base instance
__device__ __forceinline__ const float* base_rows(const DecBwdParams& p, int64_t b) {
  return p.h + ((b < p.Bb) ? b : b % p.Bb) * p.N * E;
}

__global__ void __launch_bounds__(NT, 1) k_decoder_bwd(const DecBwdParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* Xs = reinterpret_cast<float*>(smem_raw);
  float* QC = reinterpret_cast<float*>(smem_raw + BWD_X);
  float* Wb = reinterpret_cast<float*>(smem_raw + BWD_X + BWD_QC);
  float* DQ = reinterpret_cast<float*>(smem_raw + BWD_X + BWD_QC + SMEM_W);
  __shared__ float s_loadf[TM], s_w[TM];
  __shared__ int s_act[TM], s_prev[TM], s_live[TM], s_anylive;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, kind = p.kind;
  const int64_t B = p.B;
  const int64_t ntiles = (B + TM - 1) / TM;
  float* SC = p.scratch + (size_t)blockIdx.x * TM * SCQ * QW;
  float* su = Wb + warp * 128;  // per-warp scratch for u (Wb is idle outside the GEMM phases)
  float mc_acc = 0.f;           // d m_c[tid] for tid < 128, flushed once at the end

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t base = tile * TM;
    const int cnt = (int)((B - base < TM) ? (B - base) : TM);
    for (int t = 0; t < p.T; ++t) {
      // ---------------- B0: per-instance step metadata, gather x_l = h[b, tape[t-1]]
      if (tid == 0) s_anylive = 0;
      __syncthreads();
      for (int m = warp; m < TM; m += NT / 32) {
        float4 xv = make_float4(0.f, 0.f, 0.f, 0.f);
        int prev = -1, act = 0, live = 0;
        float w = 0.f, lf = 0.f;
        if (m < cnt) {
          const int64_t b = base + m;
          act = (int)p.tape[(int64_t)t * B + b];
          w = p.wts[b];
          lf = p.load_hist ? p.load_hist[(int64_t)t * B + b] : 0.f;
          if (t > 0) {
            prev = (int)p.tape[(int64_t)(t - 1) * B + b];
            xv = __ldg(reinterpret_cast<const float4*>(base_rows(p, b) + prev * E) + lane);
          }
          // an instance with a single feasible node has log p = 0 identically: no gradient
          uint32_t mw = p.mask_hist[((int64_t)t * B + b) * 4 + (lane & 3)];
          int free_cnt = 0;
#pragma unroll
          for (int i = 0; i < 4; ++i) free_cnt += __popc(~__shfl_sync(0xffffffffu, mw, i) & full_bits(N).w[i]);
          live = (w != 0.f && free_cnt > 1) ? 1 : 0;
        }
        *reinterpret_cast<float4*>(Xs + m * XS_LD + lane * 4) = xv;
        if (lane == 0) {
          s_loadf[m] = lf; s_w[m] = w; s_act[m] = act; s_prev[m] = prev; s_live[m] = live;
          if (live) s_anylive = 1;
        }
      }
      __syncthreads();
      const int anylive = s_anylive;
      __syncthreads();           // everyone has read the flag before the next iteration may reset it
      if (!anylive) continue;    // uniform: whole tile idle at this step

      // ---------------- B1: q~ (recompute)
      if (t == 0) {
        for (int o = tid; o < cnt * QW; o += NT) {
          const int m = o >> 10, c = o & (QW - 1);
          QC[m * QC_LD + c] = step0_query(p.qg0 + (base + m) * QW, p.a_q0, p.a_load, kind == VRPX_IRP, s_loadf[m], c);
        }
      } else {
        tile_gemm_wide_mma_sw<2, 2>(
            Xs, XS_LD, p.al_t, Wb,
            [&](int m, int c) {
              return (m < cnt) ? glimpse_query_init(p.qg + (base + m) * QW, p.a_load, kind == VRPX_IRP, s_loadf[m], c)
                               : make_float2(0.f, 0.f);
            },
            [&](int m, int c, float v0, float v1) {
              if (m < cnt) *reinterpret_cast<float2*>(QC + m * QC_LD + c) = make_float2(v0, v1);
            });
      }
      __syncthreads();

      // ---------------- B2: glimpse forward (scores, p, c); q~ and p are parked in the per-CTA scratch
      for (int m = warp; m < cnt; m += NT / 32) {
        const int64_t b = base + m;
        float* slot = QC + m * QC_LD;
        float* sc_q = SC + (size_t)m * SCQ * QW;
        float* sc_p = sc_q + QW;
#pragma unroll
        for (int hh = 0; hh < NH; ++hh)
          *reinterpret_cast<float4*>(sc_q + hh * E + lane * 4) = *reinterpret_cast<const float4*>(slot + hh * E + lane * 4);
        __syncwarp();
        // scores on the tensor pipe (glimpse_mma.cuh); this lane stores heads 2 tq, 2 tq + 1: their partner masks
        const int tq = lane & 3;
        uint32_t nb[2][4];
#pragma unroll
        for (int which = 0; which < 2; ++which) {
          const uint32_t* nbm = p.mask_hist + ((int64_t)t * B + quirk_row(b, 2 * tq + which, p.G)) * 4;
#pragma unroll
          for (int i = 0; i < 4; ++i) nb[which][i] = nbm[i];
        }
        const float4* hrow = reinterpret_cast<const float4*>(base_rows(p, b));
        warp_glimpse_scores(slot, hrow, N, lane, [&](int n, int which, float v) {
          const int wi = n >> 5;
          const uint32_t w0 = which ? nb[1][0] : nb[0][0], w1 = which ? nb[1][1] : nb[0][1];
          const uint32_t w2 = which ? nb[1][2] : nb[0][2], w3 = which ? nb[1][3] : nb[0][3];
          const uint32_t wsel = wi == 0 ? w0 : (wi == 1 ? w1 : (wi == 2 ? w2 : w3));
          slot[(2 * tq + which) * E + n] = v + (float)((wsel >> (n & 31)) & 1u);
        });
        __syncwarp();
        float pr[NH][4];
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) {
          warp_load_by_head(pr[hh], slot + hh * E, N, lane);
          warp_node_softmax(pr[hh], N);
        }
        __syncwarp();
        warp_store_by_node(slot, pr, N, lane);
        warp_store_by_node(sc_p, pr, N, lane);
        __syncwarp();
        warp_glimpse_values(slot, hrow, N, lane);   // c[head][dim] = sum_n p_hn h_n -> slot
      }
      for (int o = cnt * QW + tid; o < TM * QW; o += NT) QC[(o >> 10) * QC_LD + (o & (QW - 1))] = 0.f;
      __syncthreads();

      // ---------------- B3: q^ = C · M^T + m_c -> DQ   (partials go through Wb: QC must keep c for the dM update)
      tile_gemm_tall_mma_sw<2, 4, 4>(QC, QC_LD, p.m_t, Wb, p.m_c, Wb, DQ, XS_LD);   // `part` aliases the weight stage
      // ---------------- B4: pointer logits forward + backward: dz, dq^ (-> DQ), dz kept in su for B7
      for (int m = warp; m < TM; m += NT / 32) {
        float4 dqh = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < cnt && s_live[m]) {
          const int64_t b = base + m;
          const float4 qh = *reinterpret_cast<const float4*>(DQ + m * XS_LD + lane * 4);
          const float4* hp = reinterpret_cast<const float4*>(base_rows(p, b)) + lane;
          for (int n0 = 0; n0 < N; n0 += 8) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int n = n0 + i;
              const float4 hv = (n < N) ? __ldg(hp + n * (E / 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
              v[i] = fmaf(qh.x, hv.x, fmaf(qh.y, hv.y, fmaf(qh.z, hv.z, qh.w * hv.w)));
            }
            float sc = reduce8(v, lane);
            int n = n0 + ((lane >> 2) & 7);
            if ((lane & 3) == 0 && n < N) su[n] = 10.0f * tanhf(sc);
          }
          __syncwarp();
          uint32_t mw[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) mw[i] = p.mask_hist[((int64_t)t * B + b) * 4 + i];
          float u[4];
          bool ok[4];
          float mx = -INFINITY;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            int n = lane * 4 + i;
            ok[i] = n < N && !((mw[n >> 5] >> (n & 31)) & 1u);
            u[i] = (n < N) ? su[n] : 0.f;
            if (ok[i]) mx = fmaxf(mx, u[i]);
          }
          mx = warp_max(mx);
          float ex[4], loc = 0.f;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            ex[i] = ok[i] ? expf(u[i] - mx) : 0.f;
            loc += ex[i];
          }
          const float inv = 1.0f / warp_sum(loc);
          const float w = s_w[m];
          const int act = s_act[m];
          __syncwarp();
          float* sc_z = SC + (size_t)m * SCQ * QW + 2 * QW;   // dz[0..127] | q^[128..255]
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            int n = lane * 4 + i;
            // du = w (1[n==a] - pi_n);  dz = du * 10 (1 - tanh^2 z) = du * (10 - u^2 / 10)
            float du = ok[i] ? w * ((n == act ? 1.f : 0.f) - ex[i] * inv) : 0.f;
            float dz = du * (10.0f - 0.1f * u[i] * u[i]);
            if (n < N) { su[n] = dz; sc_z[n] = dz; }
          }
          __syncwarp();
          for (int n = 0; n < N; ++n) {
            const float dz = su[n];
            const float4 hv = __ldg(hp + n * (E / 4));
            dqh.x = fmaf(dz, hv.x, dqh.x); dqh.y = fmaf(dz, hv.y, dqh.y);
            dqh.z = fmaf(dz, hv.z, dqh.z); dqh.w = fmaf(dz, hv.w, dqh.w);
          }
          // dh_n += dz_n q^ is applied in B7 together with the glimpse terms (one RMW of dH per node and step)
          *reinterpret_cast<float4*>(sc_z + 128 + lane * 4) = qh;
        }
        __syncwarp();
        // every row of DQ must hold dq^ (zeros for idle instances) for the GEMMs below
        *reinterpret_cast<float4*>(DQ + m * XS_LD + lane * 4) = dqh;
      }
      __syncthreads();
      if (tid < E) {
        float s = 0.f;
        for (int m = 0; m < cnt; ++m) s += DQ[m * XS_LD + tid];
        mc_acc += s;
      }

      // ---------------- B5: d m_t[k][e] += sum_m c[m][k] dq^[m][e]     (1024 x 128 outputs, K = 32)
      // warp w owns rows [64w, 64w + 64) of d m_t
      for (int mt = 0; mt < 4; ++mt)
        for (int nh = 0; nh < 2; ++nh) {
          const int k0 = warp * 64 + mt * 16;
          warp_outer_product_tm(QC + k0, QC_LD, DQ + nh * 64, XS_LD, p.d_m_t + (size_t)k0 * E + nh * 64, E, lane);
        }
      __syncthreads();

      // ---------------- B6: dc = dq^ · M  -> QC (c is dead now)
      tile_gemm_wide_mma_sw<2, 2>(
          DQ, XS_LD, p.m_n, Wb, [](int, int) -> float2 { return make_float2(0.f, 0.f); },
          [&](int m, int c, float v0, float v1) { *reinterpret_cast<float2*>(QC + m * QC_LD + c) = make_float2(v0, v1); });
      __syncthreads();

      // ---------------- B7: glimpse backward per instance: dp, ds, dq~ (-> QC slot), dH += ...
      for (int m = warp; m < TM; m += NT / 32) {
        float* slot = QC + m * QC_LD;
        float4 dq[NH];
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) dq[hh] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < cnt && s_live[m]) {
          const int64_t b = base + m;
          const float* sc_q = SC + (size_t)m * SCQ * QW;
          const float* sc_p = sc_q + QW;
          const float* sc_z = sc_q + 2 * QW;
          float* sc_dc = SC + (size_t)m * SCQ * QW + 3 * QW;
          const float4* hrow = reinterpret_cast<const float4*>(base_rows(p, b));
          const int tq = lane & 3;
          // dc is parked in the scratch (pass Y needs it after the slot has been reused)
#pragma unroll
          for (int hh = 0; hh < NH; ++hh)
            *reinterpret_cast<float4*>(sc_dc + hh * E + lane * 4) = *reinterpret_cast<const float4*>(slot + hh * E + lane * 4);
          __syncwarp();
          // dp_hn = dc_h · h_n  -> slot[h][n]   (the score contraction with dc as the query)
          warp_glimpse_scores(slot, hrow, N, lane, [&](int n, int which, float v) { slot[(2 * tq + which) * E + n] = v; });
          __syncwarp();
          // ds_hn = p_hn (dp_hn - sum_m p_hm dp_hm), lane = node
          float ds[NH][4];
#pragma unroll
          for (int hh = 0; hh < NH; ++hh) {
            float dot = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              int n = lane + 32 * i;
              float pv = (n < N) ? sc_p[n * 8 + hh] : 0.f;
              float dp = (n < N) ? slot[hh * E + n] : 0.f;
              ds[hh][i] = pv;       // p for now
              dot = fmaf(pv, dp, dot);
              // stash dp in place of ds after the dot product is known
              if (n < N) slot[hh * E + n] = dp;
            }
            dot = warp_sum(dot);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              int n = lane + 32 * i;
              float dp = (n < N) ? slot[hh * E + n] : 0.f;
              ds[hh][i] = ds[hh][i] * (dp - dot);
            }
          }
          __syncwarp();
          warp_store_by_node(slot, ds, N, lane);
          __syncwarp();
          // pass Y: dH[b,n] += sum_h (p_hn dc_h + ds_hn q~_h) + dz_n q^     (one RMW of dH per node and step)
          {
            float4 qt[NH], dc[NH];
#pragma unroll
            for (int hh = 0; hh < NH; ++hh) {
              qt[hh] = *reinterpret_cast<const float4*>(sc_q + hh * E + lane * 4);
              dc[hh] = *reinterpret_cast<const float4*>(sc_dc + hh * E + lane * 4);
            }
            const float4 qh = *reinterpret_cast<const float4*>(sc_z + 128 + lane * 4);
            float4* dhp = reinterpret_cast<float4*>(p.dH + b * N * E) + lane;
            for (int n = 0; n < N; ++n) {
              const float4 s0 = *reinterpret_cast<const float4*>(slot + n * 8);
              const float4 s1 = *reinterpret_cast<const float4*>(slot + n * 8 + 4);
              const float4 p0 = *reinterpret_cast<const float4*>(sc_p + n * 8);
              const float4 p1 = *reinterpret_cast<const float4*>(sc_p + n * 8 + 4);
              const float dsv[NH] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
              const float pv[NH] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
              const float dz = sc_z[n];
              float4 g = make_float4(dz * qh.x, dz * qh.y, dz * qh.z, dz * qh.w);
#pragma unroll
              for (int hh = 0; hh < NH; ++hh) {
                g.x = fmaf(pv[hh], dc[hh].x, fmaf(dsv[hh], qt[hh].x, g.x));
                g.y = fmaf(pv[hh], dc[hh].y, fmaf(dsv[hh], qt[hh].y, g.y));
                g.z = fmaf(pv[hh], dc[hh].z, fmaf(dsv[hh], qt[hh].z, g.z));
                g.w = fmaf(pv[hh], dc[hh].w, fmaf(dsv[hh], qt[hh].w, g.w));
              }
              float4 o = dhp[n * (E / 4)];
              dhp[n * (E / 4)] = make_float4(o.x + g.x, o.y + g.y, o.z + g.z, o.w + g.w);
            }
          }
          // pass X: dq~_h = sum_n ds_hn h_n   (the value contraction with ds as the probabilities) -> slot[h][dim]
          __syncwarp();
          warp_glimpse_values(slot, hrow, N, lane);
#pragma unroll
          for (int hh = 0; hh < NH; ++hh) dq[hh] = *reinterpret_cast<const float4*>(slot + hh * E + lane * 4);
          // per-episode accumulators: D0 (t = 0) / D1 (t >= 1) / Dl (IRP)
          float* Dacc = (t == 0 ? p.D0 : p.D1) + b * QW;
          const float lf = s_loadf[m];
#pragma unroll
          for (int hh = 0; hh < NH; ++hh) {
            float4* dp4 = reinterpret_cast<float4*>(Dacc + hh * E + lane * 4);
            float4 o = *dp4;
            *dp4 = make_float4(o.x + dq[hh].x, o.y + dq[hh].y, o.z + dq[hh].z, o.w + dq[hh].w);
            if (kind == VRPX_IRP) {
              float4* dl4 = reinterpret_cast<float4*>(p.Dl + b * QW + hh * E + lane * 4);
              float4 ol = *dl4;
              *dl4 = make_float4(fmaf(lf, dq[hh].x, ol.x), fmaf(lf, dq[hh].y, ol.y), fmaf(lf, dq[hh].z, ol.z),
                                 fmaf(lf, dq[hh].w, ol.w));
            }
          }
        }
        __syncwarp();
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) *reinterpret_cast<float4*>(slot + hh * E + lane * 4) = dq[hh];
      }
      __syncthreads();

      if (t > 0) {
        // ---------------- B8: d al_t[j][c] += sum_m x_l[m][j] dq~[m][c]     (128 x 1024 outputs, K = 32)
        // warp w owns columns [64w, 64w + 64) of d al_t, looping over the eight 16-row j tiles
        for (int mt = 0; mt < 8; ++mt)
          warp_outer_product_tm(Xs + mt * 16, XS_LD, QC + warp * 64, QC_LD, p.d_al_t + (size_t)(mt * 16) * QW + warp * 64,
                                QW, lane);
        __syncthreads();
        // ---------------- B9: dx_l = dq~ · A_l -> DQ, then dH[b, last] += dx_l
        tile_gemm_tall_mma_sw<2, 4, 4>(QC, QC_LD, p.al_n, Wb, nullptr, Wb, DQ, XS_LD);
        for (int m = warp; m < cnt; m += NT / 32) {
          if (!s_live[m]) continue;
          const int64_t b = base + m;
          float4* dhp = reinterpret_cast<float4*>(p.dH + (b * N + s_prev[m]) * E) + lane;
          const float4 g = *reinterpret_cast<const float4*>(DQ + m * XS_LD + lane * 4);
          float4 o = *dhp;
          *dhp = make_float4(o.x + g.x, o.y + g.y, o.z + g.z, o.w + g.w);
        }
      }
      __syncthreads();
    }
  }
  if (tid < E) atomicAdd(p.d_m_c + tid, mc_acc);
}

// ---------------------------------------------------------------- small epilogue helpers (per episode, not per step)
// C[M][N] += A^T · Bm with A [R][M], Bm [R][N] row-major: reduction over rows, split across CTAs, red.add epilogue.
// Used for weight gradients (dW = dY^T X) in the decoder epilogue and the encoder backward.  64x64 output tile.
__global__ void __launch_bounds__(256) k_gemm_tn_atomic(const float* __restrict__ A, const float* __restrict__ Bm,
                                                         float* __restrict__ C, int64_t R, int M, int N,
                                                         int64_t rows_per_cta) {
  __shared__ __align__(16) float As[16][64 + 4], Bs[16][64 + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.z * 64;
  const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r_end = (r_begin + rows_per_cta < R) ? r_begin + rows_per_cta : R;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int lr = tid >> 4, lc = (tid & 15) * 4;  // loader: row lr (0..15), 4 columns at lc
  for (int64_t r0 = r_begin; r0 < r_end; r0 += 16) {
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f), bv = av;
    if (r0 + lr < r_end) {
      if (m0 + lc < M) av = *reinterpret_cast<const float4*>(A + (r0 + lr) * M + m0 + lc);
      if (n0 + lc < N) bv = *reinterpret_cast<const float4*>(Bm + (r0 + lr) * N + n0 + lc);
    }
    *reinterpret_cast<float4*>(&As[lr][lc]) = av;
    *reinterpret_cast<float4*>(&Bs[lr][lc]) = bv;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float ar[4] = {a.x, a.y, a.z, a.w}, br[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) atomicAdd(C + (size_t)m * N + n, acc[i][j]);
    }
  }
}

// Tensor-pipe version of the same reduction GEMM for M, N multiples of 64: C[M][N] += A^T · Bm on mma.sync.m16n8k8 TF32
// with the 3-term split.  CTA = 4 warps, 64 x 64 output tile; warp w owns rows [16w, 16w+16) x 64 columns; the row
// (reduction) dimension is streamed in 32-row chunks through a cp.async double buffer.
//   A fragment (m = g / g+8, k = t / t+4)  = A[r0 + t (+4)][m0 + g (+8)]   (rows of As are reduction rows)
//   B fragment (k = t / t+4, n = g)        = Bm[r0 + t (+4)][n0 + g]
constexpr int TN_LD = 64 + 8;   // (8t + g) % 32 distinct banks for both fragment patterns

__global__ void __launch_bounds__(128) k_gemm_tn_mma(const float* __restrict__ A, const float* __restrict__ Bm,
                                                      float* __restrict__ C, int64_t R, int M, int N,
                                                      int64_t rows_per_cta) {
  __shared__ __align__(16) float As[2][32][TN_LD], Bs[2][32][TN_LD];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.z * 64;
  const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r_end = (r_begin + rows_per_cta < R) ? r_begin + rows_per_cta : R;
  const int nchunks = (int)((r_end - r_begin + 31) / 32);
  float acc[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;

  auto stage = [&](int ch, int buf) {
    const int64_t r0 = r_begin + (int64_t)ch * 32;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + 128 * i;          // 32 rows x 16 float4
      const int rr = idx >> 4, c4 = (idx & 15) * 4;
      float* da = &As[buf][rr][c4];
      float* db = &Bs[buf][rr][c4];
      if (r0 + rr < r_end) {
        unsigned sa = (unsigned)__cvta_generic_to_shared(da), sb = (unsigned)__cvta_generic_to_shared(db);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(A + (r0 + rr) * M + m0 + c4) : "memory");
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sb), "l"(Bm + (r0 + rr) * N + n0 + c4) : "memory");
      } else {
        *reinterpret_cast<float4*>(da) = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(db) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  if (nchunks > 0) stage(0, 0);
  for (int ch = 0; ch < nchunks; ++ch) {
    const int buf = ch & 1;
    if (ch + 1 < nchunks) {
      stage(ch + 1, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      uint32_t ah[4], al[4];
      const float* ap = &As[buf][ks * 8 + t][warp * 16 + g];
      split_tf32(ap[0], ah[0], al[0]);               // (m = g,   k = t)
      split_tf32(ap[8], ah[1], al[1]);               // (m = g+8, k = t)
      split_tf32(ap[4 * TN_LD], ah[2], al[2]);       // (m = g,   k = t+4)
      split_tf32(ap[4 * TN_LD + 8], ah[3], al[3]);   // (m = g+8, k = t+4)
      const float* bp = &Bs[buf][ks * 8 + t][g];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        uint32_t bh0, bl0, bh1, bl1;
        split_tf32(bp[8 * j], bh0, bl0);
        split_tf32(bp[4 * TN_LD + 8 * j], bh1, bl1);
        mma_tf32_16x8x8(acc[j], al, bh0, bh1);
        mma_tf32_16x8x8(acc[j], ah, bl0, bl1);
        mma_tf32_16x8x8(acc[j], ah, bh0, bh1);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int n = n0 + 8 * j + 2 * t;
    float* c0 = C + (size_t)(m0 + warp * 16 + g) * N + n;
    float* c1 = C + (size_t)(m0 + warp * 16 + g + 8) * N + n;
    atomicAdd(c0, acc[j][0]); atomicAdd(c0 + 1, acc[j][1]);
    atomicAdd(c1, acc[j][2]); atomicAdd(c1 + 1, acc[j][3]);
  }
}

// out[c] += sum_r X[r][c]   (C <= 1024 columns, any R)
__global__ void __launch_bounds__(256) k_colsum_atomic(const float* __restrict__ X, int64_t R, int Ccols,
                                                        float* __restrict__ out, int64_t rows_per_cta) {
  const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t r_end = (r_begin + rows_per_cta < R) ? r_begin + rows_per_cta : R;
  for (int c = threadIdx.x; c < Ccols; c += 256) {
    float s = 0.f;
    for (int64_t r = r_begin; r < r_end; ++r) s += X[r * Ccols + c];
    atomicAdd(out + c, s);
  }
}

// Per-episode decoder terms: G[b] = mean_n h[b,n]; Xf[b] = h[b, tape[0][b]] unless Xf is NULL   (one warp per instance)
__global__ void __launch_bounds__(256) k_episode_gather(const float* __restrict__ h, const uint8_t* __restrict__ tape,
                                                         int64_t B, int N, float* __restrict__ G, float* __restrict__ Xf) {
  const int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  reinterpret_cast<float4*>(G + b * E)[lane] = warp_graph_mean(h, b, N, lane);
  if (Xf)
    reinterpret_cast<float4*>(Xf + b * E)[lane] = __ldg(reinterpret_cast<const float4*>(h + (b * N + (int)tape[b]) * E) + lane);
}

// dH[b,n] += dG[b] / N for every n;  dH[b, tape[0][b]] += dXf[b]
__global__ void __launch_bounds__(256) k_episode_scatter(float* __restrict__ dH, const uint8_t* __restrict__ tape,
                                                          int64_t B, int N, const float* __restrict__ dG,
                                                          const float* __restrict__ dXf) {
  const int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  float4* dp = reinterpret_cast<float4*>(dH + b * N * E) + lane;
  const float4 g = reinterpret_cast<const float4*>(dG + b * E)[lane];
  const float inv = 1.0f / (float)N;
  const int first = dXf ? (int)tape[b] : -1;
  float4 xf = make_float4(0.f, 0.f, 0.f, 0.f);
  if (dXf) xf = reinterpret_cast<const float4*>(dXf + b * E)[lane];
  for (int n = 0; n < N; ++n) {
    float4 o = dp[n * (E / 4)];
    o.x += g.x * inv; o.y += g.y * inv; o.z += g.z * inv; o.w += g.w * inv;
    if (n == first) { o.x += xf.x; o.y += xf.y; o.z += xf.z; o.w += xf.w; }
    dp[n * (E / 4)] = o;
  }
}

}  // namespace vrpx

static int g_tn_path = 0;   // vrpx_debug_gemm_tn_path

namespace vrpx {
int launch_episode_gather(const float* h, const uint8_t* tape0, int64_t B, int N, float* G, float* Xf,
                          cudaStream_t stream) {
  k_episode_gather<<<(unsigned)((B + 7) / 8), 256, 0, stream>>>(h, tape0, B, N, G, Xf);
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}

int colsum_launch(const float* X, int64_t R, int Ccols, float* out, cudaStream_t stream) {
  int64_t ctas = (R + 511) / 512;
  int64_t maxc = (int64_t)num_sms() * 8;
  if (ctas > maxc) ctas = maxc;
  int64_t rows = (R + ctas - 1) / ctas;
  ctas = (R + rows - 1) / rows;
  k_colsum_atomic<<<(unsigned)ctas, 256, 0, stream>>>(X, R, Ccols, out, rows);
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}

int gemm_tn_accumulate(const float* A, const float* Bm, float* C, float* colsum_A, int64_t R, int M, int N, cudaStream_t stream) {
  // 128-multiples with enough rows to feed every SM: tcgen05 (gemm_tn_tc.cu); the rest (embedding [128][4], tiny batches)
  // stays on the warp-level kernels
  if (g_tn_path == 0 && M % 128 == 0 && N % 128 == 0 && R >= 8192 && R <= INT32_MAX &&
      (reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(Bm) & 15) == 0)
    return gemm_tn_tc(A, Bm, C, colsum_A, R, M, N, stream);
  if (colsum_A) {
    int rc = colsum_launch(A, R, M, colsum_A, stream);
    if (rc) return rc;
  }
  int64_t ctas = (R + 2047) / 2048;
  int64_t maxc = (int64_t)num_sms() * 8;
  if (ctas > maxc) ctas = maxc;
  int64_t rows = ((R + ctas - 1) / ctas + 15) / 16 * 16;
  ctas = (R + rows - 1) / rows;
  dim3 grid((unsigned)ctas, (unsigned)((M + 63) / 64), (unsigned)((N + 63) / 64));
  if (M % 64 == 0 && N % 64 == 0) {
    rows = (rows + 31) / 32 * 32;
    grid.x = (unsigned)((R + rows - 1) / rows);
    k_gemm_tn_mma<<<grid, 128, 0, stream>>>(A, Bm, C, R, M, N, rows);
  } else {
    k_gemm_tn_atomic<<<grid, 256, 0, stream>>>(A, Bm, C, R, M, N, rows);
  }
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}
}  // namespace vrpx

using namespace vrpx;

extern "C" {

int64_t vrpx_decoder_backward_workspace_bytes(int64_t B, int32_t N) {
  (void)N;
  int64_t grid = (B + TM - 1) / TM;
  if (grid > num_sms()) grid = num_sms();
  return grid * (int64_t)TM * SCQ * QW * (int64_t)sizeof(float);
}

}  // extern "C"

namespace {
// one launch of k_decoder_bwd over env->B replicas of Bb base instances (Bb = env->B: vrpx_decoder_backward)
int decoder_backward(const vrpx_env* env, const vrpx_decoder_weights* w, const vrpx_decoder_bwd_weights* wb,
                     const float* h, int64_t Bb, const uint8_t* tape, int32_t T, int64_t coupling,
                     const vrpx_rollout_trace* trace, const float* qg, const float* wts, const vrpx_decoder_grads* g,
                     void* ws, int64_t ws_bytes, cudaStream_t stream) {
  VRPX_CHECK_ARG(env->N >= 2 && env->N <= VRPX_MAX_NODES && env->B >= 1 && T >= 1, "bad shape");
  VRPX_CHECK_ARG(trace->mask_hist && trace->qg0 && (env->kind != VRPX_IRP || trace->load_hist), "trace incomplete");
  VRPX_CHECK_ARG(g->dH && g->D0 && g->D1 && g->d_al_t && g->d_m_t && g->d_m_c && (env->kind != VRPX_IRP || g->Dl),
                 "gradient buffers");
  VRPX_CHECK_ARG(ws_bytes >= vrpx_decoder_backward_workspace_bytes(env->B, env->N), "workspace too small");
  DecBwdParams p;
  p.kind = env->kind; p.N = env->N; p.T = T; p.B = env->B; p.G = coupling; p.Bb = Bb;
  p.h = h; p.tape = tape; p.mask_hist = trace->mask_hist; p.load_hist = trace->load_hist;
  p.qg0 = trace->qg0; p.qg = qg; p.wts = wts;
  p.al_t = w->al_t; p.a_q0 = w->a_q0; p.a_load = w->a_load; p.m_t = w->m_t; p.m_c = w->m_c;
  p.m_n = wb->m_n; p.al_n = wb->al_n;
  p.dH = g->dH; p.D0 = g->D0; p.D1 = g->D1; p.Dl = g->Dl; p.d_al_t = g->d_al_t; p.d_m_t = g->d_m_t; p.d_m_c = g->d_m_c;
  p.scratch = reinterpret_cast<float*>(ws);
  int64_t ntiles = (env->B + TM - 1) / TM;
  int grid = (int)((ntiles < (int64_t)num_sms()) ? ntiles : (int64_t)num_sms());
  VRPX_CUDA(cudaFuncSetAttribute(k_decoder_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BWD_SMEM));
  k_decoder_bwd<<<grid, NT, BWD_SMEM, stream>>>(p);
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}
}  // namespace

extern "C" {

int vrpx_decoder_backward(const vrpx_env* env, const vrpx_decoder_weights* w, const vrpx_decoder_bwd_weights* wb,
                          const float* h, const uint8_t* tape, int32_t T, int64_t coupling,
                          const vrpx_rollout_trace* trace, const float* qg, const float* wts,
                          const vrpx_decoder_grads* g, void* ws, int64_t ws_bytes, void* stream_) {
  VRPX_CHECK_ARG(env && w && wb && h && tape && trace && qg && wts && g && ws, "NULL argument");
  VRPX_DEVICE_GUARD(h);
  NvtxRange nvtx_range("vrpx:decoder_backward");
  // the glimpse mask of attention row (b, head) is read at quirk_row(): it must stay inside the batch
  VRPX_CHECK_ARG(coupling >= 0 && (coupling == 0 || (coupling <= env->B && env->B % coupling == 0)),
                 "coupling group must be 0 or a divisor of the batch size");
  return decoder_backward(env, w, wb, h, env->B, tape, T, coupling, trace, qg, wts, g, ws, ws_bytes,
                          (cudaStream_t)stream_);
}

int vrpx_decoder_backward_samples(const vrpx_env* env, const vrpx_decoder_weights* w, const vrpx_decoder_bwd_weights* wb,
                                  const float* h, int64_t Bb, int32_t K, const uint8_t* tape, int32_t T, int64_t coupling,
                                  const vrpx_rollout_trace* trace, const float* qg, const float* wts,
                                  const vrpx_decoder_grads* g, void* ws, int64_t ws_bytes, void* stream_) {
  VRPX_CHECK_ARG(env && w && wb && h && tape && trace && qg && wts && g && ws, "NULL argument");
  VRPX_DEVICE_GUARD(h);
  NvtxRange nvtx_range("vrpx:decoder_backward_samples");
  VRPX_CHECK_ARG(K >= 1, "sample count K must be at least 1");
  VRPX_CHECK_ARG(Bb >= 1 && env->B % K == 0 && env->B / K == Bb, "env must hold Bb x K replicas");
  // the partner rows of quirk_row must stay inside each copy
  VRPX_CHECK_ARG(coupling >= 0 && (coupling == 0 || (coupling <= Bb && Bb % coupling == 0)),
                 "coupling group must be 0 or a divisor of the base batch size");
  return decoder_backward(env, w, wb, h, Bb, tape, T, coupling, trace, qg, wts, g, ws, ws_bytes,
                          (cudaStream_t)stream_);
}

void vrpx_debug_gemm_tn_path(int32_t path) { g_tn_path = path; }

int vrpx_gemm_tn_accumulate(const float* A, const float* Bm, float* C, int64_t R, int32_t M, int32_t N, void* stream) {
  VRPX_CHECK_ARG(A && Bm && C && R >= 1 && M >= 1 && N >= 1 && M % 4 == 0 && N % 4 == 0, "bad argument");
  VRPX_DEVICE_GUARD(A);
  return gemm_tn_accumulate(A, Bm, C, nullptr, R, M, N, (cudaStream_t)stream);
}

int vrpx_gemm_tn_colsum_accumulate(const float* A, const float* Bm, float* C, float* colsum_A, int64_t R, int32_t M, int32_t N,
                                    void* stream) {
  VRPX_CHECK_ARG(A && Bm && C && R >= 1 && M >= 1 && N >= 1 && M % 4 == 0 && N % 4 == 0, "bad argument");
  VRPX_DEVICE_GUARD(A);
  return gemm_tn_accumulate(A, Bm, C, colsum_A, R, M, N, (cudaStream_t)stream);
}

int vrpx_colsum_accumulate(const float* X, int64_t R, int32_t Ccols, float* out, void* stream) {
  VRPX_CHECK_ARG(X && out && R >= 1 && Ccols >= 1, "bad argument");
  VRPX_DEVICE_GUARD(X);
  return colsum_launch(X, R, Ccols, out, (cudaStream_t)stream);
}

int vrpx_episode_gather(const float* h, const uint8_t* tape0, int64_t B, int32_t N, float* G, float* Xf, void* stream) {
  VRPX_CHECK_ARG(h && G && B >= 1 && (Xf == nullptr || tape0 != nullptr), "bad argument");
  VRPX_DEVICE_GUARD(h);
  return launch_episode_gather(h, tape0, B, N, G, Xf, (cudaStream_t)stream);
}

int vrpx_episode_scatter(float* dH, const uint8_t* tape0, int64_t B, int32_t N, const float* dG, const float* dXf,
                         void* stream) {
  VRPX_CHECK_ARG(dH && dG && B >= 1 && (dXf == nullptr || tape0 != nullptr), "bad argument");
  VRPX_DEVICE_GUARD(dH);
  k_episode_scatter<<<(unsigned)((B + 7) / 8), 256, 0, (cudaStream_t)stream>>>(dH, tape0, B, N, dG, dXf);
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}

}  // extern "C"
