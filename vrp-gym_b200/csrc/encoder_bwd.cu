// encoder_bwd.cu — backward of the graph encoder (agents/graph_encoder.py:183-198 per layer:
//   y1 = x + MHA(x);  h1 = BN1(y1);  y2 = h1 + W2 relu(W1 h1 + b1) + b2;  out = BN2(y2)   in TRAIN mode,
// i.e. BatchNorm with batch statistics over all B*N rows, graph_encoder.py:141-154).
//
// Input: dL/d(out of the last layer) (from the decoder backward) and the activations the train-mode forward saved
// (encoder.cu, vrpx_encoder_saved_bytes).  Output: gradients of every encoder parameter, accumulated (+=).
// Dense products reuse the forward GEMM kernels (dX = dY · W through gemm_tc/gemm_simt on the transposed weight, the
// ReLU gate and the residual in its epilogue).  Weight and bias gradients go through gemm_tn_accumulate: k_gemm_tn_tc
// with its colsum_A bias sums at R >= 8192 rows, k_gemm_tn_mma + k_colsum_atomic below (decoder_bwd.cu); the embedding
// [128][4] products always take the warp-level kernels.  The per-instance attention backward runs on mma.sync
// (attention_bwd.cu; gemm_path 1: the fp32 SIMT k_enc_attention_bwd below); the BatchNorm backward (two batch-wide f64
// reductions per BN) is the pair of SIMT kernels below.
#include "gemm.cuh"

namespace vrpx {

struct BnBwdSlot {
  double s_dout[E];     // sum_r dout
  double s_dout_xh[E];  // sum_r dout * xhat
};

// Reductions for the BatchNorm backward: block = 2 row lanes x 128 features (like k_bn_stats).
__global__ void __launch_bounds__(256) k_bn_bwd_reduce(const float* __restrict__ dout, const float* __restrict__ y,
                                                        const float* __restrict__ stat, int64_t R, BnBwdSlot* slot) {
  __shared__ double s1[256], s2[256];
  const int c = threadIdx.x & 127, rl = threadIdx.x >> 7;
  const float mean = stat[c], invstd = stat[E + c];
  double a = 0.0, q = 0.0;
  for (int64_t r = (int64_t)blockIdx.x * 2 + rl; r < R; r += (int64_t)gridDim.x * 2) {
    const float d = dout[r * E + c];
    const float xh = (y[r * E + c] - mean) * invstd;
    a += (double)d;
    q += (double)d * (double)xh;
  }
  s1[threadIdx.x] = a;
  s2[threadIdx.x] = q;
  __syncthreads();
  if (rl == 0) {
    atomicAdd(&slot->s_dout[c], s1[c] + s1[c + 128]);
    atomicAdd(&slot->s_dout_xh[c], s2[c] + s2[c + 128]);
  }
}

// dy = gamma * invstd * (dout - mean(dout) - xhat * mean(dout * xhat));  in place on `g` (dout -> dy).
// Block 0 also accumulates dgamma / dbeta.  Each of the six slots serves one BN of one call (zeroed by the call's memset).
__global__ void __launch_bounds__(256) k_bn_bwd_apply(float* __restrict__ g, const float* __restrict__ y,
                                                       const float* __restrict__ stat, const float* __restrict__ gamma,
                                                       int64_t R, const BnBwdSlot* __restrict__ slot,
                                                       float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // float4 index
  if (blockIdx.x == 0 && threadIdx.x < E) {
    dgamma[threadIdx.x] += (float)slot->s_dout_xh[threadIdx.x];
    dbeta[threadIdx.x] += (float)slot->s_dout[threadIdx.x];
  }
  if (i >= R * 32) return;
  const int c = (int)(i & 31) * 4;
  float4 d = reinterpret_cast<float4*>(g)[i];
  const float4 yv = reinterpret_cast<const float4*>(y)[i];
  const float invR = 1.0f / (float)R;
  float dv[4] = {d.x, d.y, d.z, d.w};
  const float yy[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float mean = stat[c + j], invstd = stat[E + c + j];
    const float xh = (yy[j] - mean) * invstd;
    const float m1 = (float)slot->s_dout[c + j] * invR, m2 = (float)slot->s_dout_xh[c + j] * invR;
    dv[j] = gamma[c + j] * invstd * (dv[j] - m1 - xh * m2);
  }
  reinterpret_cast<float4*>(g)[i] = make_float4(dv[0], dv[1], dv[2], dv[3]);
}

// ---------------------------------------------------------------- attention backward
// One CTA per (instance, group of 4 heads), one warp per head.  For head hd with Q,K,V,dO (N x 16):
//   P = softmax(Q K^T / 4);  D_i = dO_i · O_i;  dS_ij = P_ij (dO_i · V_j - D_i)
//   dQ_i = sum_j dS_ij K_j / 4;   dK_j = sum_i dS_ij Q_i / 4;   dV_j = sum_i P_ij dO_i
// Row statistics (max, sum) are recomputed; pass A has lane = query, pass B lane = key.
__global__ void __launch_bounds__(128) k_enc_attention_bwd(const float* __restrict__ qkv, const float* __restrict__ att,
                                                            const float* __restrict__ datt, float* __restrict__ dqkv,
                                                            int N) {
  extern __shared__ __align__(16) float sm[];
  const int64_t b = blockIdx.x >> 1;
  const int hg = blockIdx.x & 1;                 // head group: heads 4*hg .. 4*hg+3
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
  const int hd = hg * 4 + w;
  // per warp: Q, K, V, dO [N][16] + m, l, D [N]
  float* base_s = sm + (size_t)w * (size_t)(((4 * 16 + 3) * N + 3) & ~3);  // 16-byte aligned per-warp region
  float* Qs = base_s; float* Ks = Qs + 16 * N; float* Vs = Ks + 16 * N; float* Os = Vs + 16 * N;
  float* ms = Os + 16 * N; float* ls = ms + N; float* Ds = ls + N;
  const float* qrow = qkv + b * N * 384;
  for (int i = lane; i < N * 4; i += 32) {       // 4 float4 per row and matrix
    const int n = i >> 2, c = (i & 3) * 4;
    *reinterpret_cast<float4*>(Qs + n * 16 + c) = *reinterpret_cast<const float4*>(qrow + (int64_t)n * 384 + hd * 16 + c);
    *reinterpret_cast<float4*>(Ks + n * 16 + c) = *reinterpret_cast<const float4*>(qrow + (int64_t)n * 384 + 128 + hd * 16 + c);
    *reinterpret_cast<float4*>(Vs + n * 16 + c) = *reinterpret_cast<const float4*>(qrow + (int64_t)n * 384 + 256 + hd * 16 + c);
    *reinterpret_cast<float4*>(Os + n * 16 + c) = *reinterpret_cast<const float4*>(datt + (b * N + n) * E + hd * 16 + c);
  }
  __syncwarp();
  // ---- pass A: lane = query i
  for (int i = lane; i < N; i += 32) {
    float q[16], dO[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) { q[d] = Qs[i * 16 + d] * 0.25f; dO[d] = Os[i * 16 + d]; }
    float D = 0.f;
    const float* orow = att + (b * N + i) * E + hd * 16;
#pragma unroll
    for (int d = 0; d < 16; ++d) D = fmaf(dO[d], orow[d], D);
    float mx = -INFINITY;
    for (int j = 0; j < N; ++j) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < 16; ++d) s = fmaf(q[d], Ks[j * 16 + d], s);
      mx = fmaxf(mx, s);
    }
    float sum = 0.f;
    for (int j = 0; j < N; ++j) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < 16; ++d) s = fmaf(q[d], Ks[j * 16 + d], s);
      sum += expf(s - mx);
    }
    const float inv = 1.0f / sum;
    float dq[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) dq[d] = 0.f;
    for (int j = 0; j < N; ++j) {
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int d = 0; d < 16; ++d) { s = fmaf(q[d], Ks[j * 16 + d], s); dp = fmaf(dO[d], Vs[j * 16 + d], dp); }
      const float pij = expf(s - mx) * inv;
      const float ds = pij * (dp - D);
#pragma unroll
      for (int d = 0; d < 16; ++d) dq[d] = fmaf(ds, Ks[j * 16 + d], dq[d]);
    }
    ms[i] = mx; ls[i] = inv; Ds[i] = D;
    float* o = dqkv + (b * N + i) * 384 + hd * 16;
#pragma unroll
    for (int d = 0; d < 16; d += 4)
      *reinterpret_cast<float4*>(o + d) = make_float4(dq[d] * 0.25f, dq[d + 1] * 0.25f, dq[d + 2] * 0.25f, dq[d + 3] * 0.25f);
  }
  __syncwarp();
  // ---- pass B: lane = key j
  for (int j = lane; j < N; j += 32) {
    float k[16], v[16], dk[16], dv[16];
#pragma unroll
    for (int d = 0; d < 16; ++d) { k[d] = Ks[j * 16 + d]; v[d] = Vs[j * 16 + d]; dk[d] = 0.f; dv[d] = 0.f; }
    for (int i = 0; i < N; ++i) {
      float s = 0.f, dp = 0.f;
#pragma unroll
      for (int d = 0; d < 16; ++d) { s = fmaf(Qs[i * 16 + d], k[d], s); dp = fmaf(Os[i * 16 + d], v[d], dp); }
      const float pij = expf(s * 0.25f - ms[i]) * ls[i];
      const float ds = pij * (dp - Ds[i]) * 0.25f;
#pragma unroll
      for (int d = 0; d < 16; ++d) { dk[d] = fmaf(ds, Qs[i * 16 + d], dk[d]); dv[d] = fmaf(pij, Os[i * 16 + d], dv[d]); }
    }
    float* ok = dqkv + (b * N + j) * 384 + 128 + hd * 16;
    float* ov = dqkv + (b * N + j) * 384 + 256 + hd * 16;
#pragma unroll
    for (int d = 0; d < 16; d += 4) {
      *reinterpret_cast<float4*>(ok + d) = make_float4(dk[d], dk[d + 1], dk[d + 2], dk[d + 3]);
      *reinterpret_cast<float4*>(ov + d) = make_float4(dv[d], dv[d + 1], dv[d + 2], dv[d + 3]);
    }
  }
}

// Feature matrices for the embedding gradients: Xn[r] = [x, y, (demand), 1] on non-depot rows (else 0),
// Xd[r] = [x, y, 0, 1] on depot rows (else 0); the bias gradient rides in column 3.
__global__ void k_embed_features(const vrpx_encoder_weights w, const double* __restrict__ xy,
                                 const double* __restrict__ demand, const float* __restrict__ x,
                                 const int32_t* __restrict__ depot, int64_t R, int N, float* __restrict__ Xn,
                                 float* __restrict__ Xd) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  float f[3] = {0.f, 0.f, 0.f};
  if (x) {
    for (int i = 0; i < w.f; ++i) f[i] = x[r * w.f + i];
  } else {
    f[0] = (float)xy[r * 2];
    f[1] = (float)xy[r * 2 + 1];
    if (w.f == 3) f[2] = (float)demand[r];
  }
  bool is_depot = false;
  if (depot && w.depot_w) {
    const int64_t b = r / N;
    is_depot = depot[b] == (int)(r - b * N);
  }
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  reinterpret_cast<float4*>(Xn)[r] = is_depot ? z : make_float4(f[0], f[1], f[2], 1.f);
  reinterpret_cast<float4*>(Xd)[r] = is_depot ? make_float4(f[0], f[1], 0.f, 1.f) : z;
}

// dW[e][f] += C[e][f] (f < nf), db[e] += C[e][3]    with C [128][4]
__global__ void k_embed_grad_unpack(const float* __restrict__ C, int nf, float* __restrict__ dW, float* __restrict__ db) {
  const int e = threadIdx.x;
  if (e >= E) return;
  for (int f = 0; f < nf; ++f) dW[e * nf + f] += C[e * 4 + f];
  db[e] += C[e * 4 + 3];
}

constexpr int64_t kBwdSmall = 16384;  // 6 BnBwdSlot (2 KiB each) + 2 x [128][4] embedding scratch
constexpr int64_t kStageWidth = 9 * E + FF;  // floats per row and layer of vrpx_debug_encoder_backward_stages

}  // namespace vrpx

using namespace vrpx;

extern "C" {

int vrpx_gemm_tn_accumulate(const float* A, const float* Bm, float* C, int64_t R, int32_t M, int32_t N, void* stream);
int vrpx_colsum_accumulate(const float* X, int64_t R, int32_t Ccols, float* out, void* stream);

int vrpx_debug_attention_backward(const float* qkv, const float* att, const float* datt, float* dqkv, int64_t B, int32_t N,
                                  int32_t path, void* stream) {
  VRPX_CHECK_ARG(qkv && att && datt && dqkv && B >= 1 && N >= 1 && N <= VRPX_MAX_NODES, "bad argument");
  VRPX_DEVICE_GUARD(qkv);
  if (path == 0) return attention_backward_mma(qkv, att, datt, dqkv, B, N, (cudaStream_t)stream);
  const int attn_smem = 4 * (((4 * 16 + 3) * N + 3) & ~3) * (int)sizeof(float);
  VRPX_CUDA(cudaFuncSetAttribute(k_enc_attention_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, attn_smem));
  k_enc_attention_bwd<<<(unsigned)(B * 2), 128, attn_smem, (cudaStream_t)stream>>>(qkv, att, datt, dqkv, N);
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}

int64_t vrpx_encoder_backward_workspace_bytes(int64_t B, int32_t N) {
  // small | T512 [R][512] | T128 [R][128] | Xn [R][4] | Xd [R][4]
  return kBwdSmall + B * (int64_t)N * (512 + 128 + 8) * (int64_t)sizeof(float);
}

}  // extern "C"

// The body of vrpx_encoder_backward.  stages == NULL: the production call.  Otherwise, for every layer l whose bit is set
// in layer_mask, the eight gradients the kernels hold inside layer l are copied into stages (see
// vrpx_debug_encoder_backward_stages) on the call's stream.
static int encoder_backward_impl(const vrpx_encoder_weights* w, const vrpx_encoder_weights_t* wt, const vrpx_env* env,
                                 const float* x, const int32_t* depot, int64_t B, int32_t N, const float* saved, float* g,
                                 const vrpx_encoder_grads* grads, void* ws, int64_t ws_bytes, int32_t gemm_path,
                                 cudaStream_t stream, float* stages, int32_t layer_mask) {
  VRPX_CHECK_ARG(w && wt && saved && g && grads && ws, "NULL argument");
  VRPX_DEVICE_GUARD(g);
  NvtxRange nvtx_range("vrpx:encoder_backward");
  VRPX_CHECK_ARG(B >= 1 && N >= 1 && N <= VRPX_MAX_NODES, "bad B or N");
  VRPX_CHECK_ARG(x || (env && env->xy && (w->f == 2 || env->demand)), "need x or an env with features");
  VRPX_CHECK_ARG(ws_bytes >= vrpx_encoder_backward_workspace_bytes(B, N), "workspace too small");
  const int64_t R = B * N;
  auto gemm = [gemm_path](const GemmArgs& ga, cudaStream_t st) { return gemm_dispatch(gemm_path, ga, st); };
  BnBwdSlot* slots = reinterpret_cast<BnBwdSlot*>(ws);
  float* embC = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + 12288);  // 2 x [128][4]
  float* T512 = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + kBwdSmall);
  float* T128 = T512 + R * 512;
  float* Xn = T128 + R * 128;
  float* Xd = Xn + R * 4;
  const float* sv_stats = saved + R * (3 * 128 + VRPX_LAYERS * 1408);
  VRPX_CUDA(cudaMemsetAsync(ws, 0, kBwdSmall, stream));
  const int attn_smem = 4 * (((4 * 16 + 3) * N + 3) & ~3) * (int)sizeof(float);
  VRPX_CUDA(cudaFuncSetAttribute(k_enc_attention_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, attn_smem));
  const unsigned ew_grid = (unsigned)((R * 32 + 255) / 256);
  int rc;
  for (int l = VRPX_LAYERS - 1; l >= 0; --l) {
    const vrpx_encoder_layer& L = w->layer[l];
    const vrpx_encoder_layer_t& LT = wt->layer[l];
    const vrpx_encoder_layer_grads& G = grads->layer[l];
    // this layer's stage blocks: behind those of the selected layers below it
    float* st = (stages && (layer_mask >> l & 1))
                    ? stages + (int64_t)__builtin_popcount(layer_mask & ((1 << l) - 1)) * R * kStageWidth
                    : nullptr;
    auto stage = [&](const float* src, int64_t col0, int width) -> int {
      if (st) VRPX_CUDA(cudaMemcpyAsync(st + R * col0, src, (size_t)(R * width) * sizeof(float), cudaMemcpyDeviceToDevice, stream));
      return VRPX_OK;
    };
    if ((rc = stage(g, 0, E))) return rc;                                                      // dOUT
    const float* Lb = saved + R * 384 + (int64_t)l * R * 1408;
    const float *QKV = Lb, *ATT = Lb + R * 384, *Y1 = Lb + R * 512, *H1 = Lb + R * 640, *F = Lb + R * 768,
                *Y2 = Lb + R * 1280;
    const float* Hin = saved + (int64_t)l * R * 128;
    // ---- BN2 backward: g = d(out) -> d(y2)
    k_bn_bwd_reduce<<<num_sms() * 4, 256, 0, stream>>>(g, Y2, sv_stats + (2 * l + 1) * 256, R, slots + 2 * l + 1);
    VRPX_LAUNCH_CHECK();
    k_bn_bwd_apply<<<ew_grid, 256, 0, stream>>>(g, Y2, sv_stats + (2 * l + 1) * 256, L.bn2_w, R, slots + 2 * l + 1,
                                                G.bn2_w, G.bn2_b);
    VRPX_LAUNCH_CHECK();
    if ((rc = stage(g, E, E))) return rc;                                                      // dY2
    // ---- FF backward:  y2 = h1 + relu(h1 W1^T + b1) W2^T + b2
    if ((rc = gemm_tn_accumulate(g, F, G.ff2_w, G.ff2_b, R, E, FF, stream))) return rc;       // dW2 [128][512] += dy2^T F, db2 += colsum(dy2)
    {
      GemmArgs a{g, R, E, LT.ff2_wT, FF, nullptr, 0, nullptr, nullptr, nullptr, T512};        // dpre = (dy2 W2) * [F > 0]
      a.gate = F;
      if ((rc = gemm(a, stream))) return rc;
    }
    if ((rc = stage(T512, 2 * E, FF))) return rc;                                              // dPRE
    if ((rc = gemm_tn_accumulate(T512, H1, G.ff0_w, G.ff0_b, R, FF, E, stream))) return rc;   // dW1 [512][128] += dpre^T h1, db1
    {
      GemmArgs a{T512, R, FF, LT.ff0_wT, E, nullptr, 0, g, nullptr, nullptr, g};              // dh1 = dy2 + dpre W1
      if ((rc = gemm(a, stream))) return rc;
    }
    if ((rc = stage(g, 2 * E + FF, E))) return rc;                                             // dH1
    // ---- BN1 backward: g = d(h1) -> d(y1)
    k_bn_bwd_reduce<<<num_sms() * 4, 256, 0, stream>>>(g, Y1, sv_stats + (2 * l) * 256, R, slots + 2 * l);
    VRPX_LAUNCH_CHECK();
    k_bn_bwd_apply<<<ew_grid, 256, 0, stream>>>(g, Y1, sv_stats + (2 * l) * 256, L.bn1_w, R, slots + 2 * l, G.bn1_w,
                                                G.bn1_b);
    VRPX_LAUNCH_CHECK();
    if ((rc = stage(g, 3 * E + FF, E))) return rc;                                             // dY1
    // ---- attention block backward:  y1 = x + att W_o^T + b_o,  att = MHA_core(x W_in^T + b_in)
    if ((rc = gemm_tn_accumulate(g, ATT, G.out_proj_w, G.out_proj_b, R, E, E, stream))) return rc;   // dW_o += dy1^T att, db_o
    {
      GemmArgs a{g, R, E, LT.out_proj_wT, E, nullptr, 0, nullptr, nullptr, nullptr, T128};    // datt = dy1 W_o
      if ((rc = gemm(a, stream))) return rc;
    }
    if ((rc = stage(T128, 4 * E + FF, E))) return rc;                                          // dATT
    float* dQKV = T512;  // [R][384]
    if (gemm_path == 0) {   // tensor pipe (attention_bwd.cu); the fp32 SIMT kernel stays as the cross-check path
      if ((rc = attention_backward_mma(QKV, ATT, T128, dQKV, B, N, stream))) return rc;
    } else {
      k_enc_attention_bwd<<<(unsigned)(B * 2), 128, attn_smem, stream>>>(QKV, ATT, T128, dQKV, N);
      VRPX_LAUNCH_CHECK();
    }
    if ((rc = stage(dQKV, 5 * E + FF, 3 * E))) return rc;                                      // dQKV
    if ((rc = gemm_tn_accumulate(dQKV, Hin, G.in_proj_w, G.in_proj_b, R, 3 * E, E, stream))) return rc;   // dW_in [384][128], db_in
    {
      GemmArgs a{dQKV, R, 3 * E, LT.in_proj_wT, E, nullptr, 0, g, nullptr, nullptr, g};       // dx = dy1 + dqkv W_in
      if ((rc = gemm(a, stream))) return rc;
    }
    if ((rc = stage(g, 8 * E + FF, E))) return rc;                                             // dX
  }
  // ---- embedding backward (graph_encoder.py:54 / :110-132)
  k_embed_features<<<(unsigned)((R + 255) / 256), 256, 0, stream>>>(
      *w, (!x && env) ? env->xy : nullptr, (!x && env) ? env->demand : nullptr, x, depot, R, N, Xn, Xd);
  VRPX_LAUNCH_CHECK();
  if ((rc = vrpx_gemm_tn_accumulate(g, Xn, embC, R, E, 4, stream))) return rc;
  k_embed_grad_unpack<<<1, E, 0, stream>>>(embC, w->f, grads->node_w, grads->node_b);
  VRPX_LAUNCH_CHECK();
  if (w->depot_w && depot) {
    VRPX_CHECK_ARG(grads->depot_w && grads->depot_b, "depot gradient buffers");
    if ((rc = vrpx_gemm_tn_accumulate(g, Xd, embC + 512, R, E, 4, stream))) return rc;
    k_embed_grad_unpack<<<1, E, 0, stream>>>(embC + 512, 2, grads->depot_w, grads->depot_b);
    VRPX_LAUNCH_CHECK();
  }
  return VRPX_OK;
}

extern "C" {

int vrpx_encoder_backward(const vrpx_encoder_weights* w, const vrpx_encoder_weights_t* wt, const vrpx_env* env,
                          const float* x, const int32_t* depot, int64_t B, int32_t N, const float* saved,
                          float* g, const vrpx_encoder_grads* grads, void* ws, int64_t ws_bytes, int32_t gemm_path,
                          void* stream) {
  return encoder_backward_impl(w, wt, env, x, depot, B, N, saved, g, grads, ws, ws_bytes, gemm_path, (cudaStream_t)stream,
                               nullptr, 0);
}

int vrpx_debug_encoder_backward_stages(const vrpx_encoder_weights* w, const vrpx_encoder_weights_t* wt,
                                       const vrpx_env* env, const float* x, const int32_t* depot, int64_t B, int32_t N,
                                       const float* saved, float* g, const vrpx_encoder_grads* grads, void* ws,
                                       int64_t ws_bytes, int32_t gemm_path, float* stages, int32_t layer_mask,
                                       void* stream) {
  VRPX_CHECK_ARG(stages && layer_mask >= 1 && layer_mask < (1 << VRPX_LAYERS), "stages buffer and a layer mask in 1..7");
  return encoder_backward_impl(w, wt, env, x, depot, B, N, saved, g, grads, ws, ws_bytes, gemm_path, (cudaStream_t)stream,
                               stages, layer_mask);
}

}  // extern "C"
