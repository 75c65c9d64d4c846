// glimpse_mma.cuh — the per-instance phases of the glimpse, one warp per instance: the score and value contractions on
// the warp-level tensor pipe with the embeddings streamed from global memory / L2 or a shared-memory ring, the softmax
// over nodes between them and the P[n][8] layout that hands the probabilities to the value contraction.  Every kernel
// that runs a glimpse calls these: phase P2 of the persistent rollout kernel (rollout.cu), the split-step glimpse kernels
// (rollout_steps.cu), and the recompute and gradients of the REINFORCE backward (decoder_bwd.cu, where the "query" is dc
// and the "probabilities" are ds).
#pragma once
#include "tile_gemm.cuh"

namespace vrpx {

// S[node][head] = h[node][:] · q[head][:] on the tensor pipe (m16n8k8 TF32 3-term; M = 16 nodes, N = 8 heads), q = 8 x 128
// floats in shared memory.  Fragment coordinates g = lane >> 2, tq = lane & 3.  The K (embedding) axis is permuted so
// that every thread streams whole float4 chunks: chunk c (0..7) of thread tq covers dims 16c + 4tq + {0,1,2,3}; k-step
// 2c + u uses mma k-index tq <-> dim 16c+4tq+2u and k-index tq+4 <-> dim 16c+4tq+2u+1, for A (node rows) and B (q)
// alike.  store(n, which, v): node n, head 2 tq + which.
template <class Store>
__device__ __forceinline__ void warp_glimpse_scores(const float* q, const float4* __restrict__ hrow, int N, int lane, Store&& store) {
  const int g = lane >> 2, tq = lane & 3;
  float4 qv[8];   // q[head g][dims of this thread]
#pragma unroll
  for (int c = 0; c < 8; ++c) qv[c] = *reinterpret_cast<const float4*>(q + g * E + 16 * c + 4 * tq);
  __syncwarp();
  for (int n0 = 0; n0 < N; n0 += 16) {
    const int na = n0 + g, nbb = n0 + g + 8;
    // six independent accumulator chains (3 split terms x even/odd k-step): a single chain would serialise the 96 mma of
    // a node tile on the tensor-pipe latency
    float acc6[2][3][4];
#pragma unroll
    for (int a_ = 0; a_ < 2; ++a_)
#pragma unroll
      for (int b_ = 0; b_ < 3; ++b_)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc6[a_][b_][i] = 0.f;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      float4 va[4], vb[4];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int c = half * 4 + cc;
        va[cc] = (na < N) ? __ldg(hrow + na * (E / 4) + 4 * c + tq) : make_float4(0.f, 0.f, 0.f, 0.f);
        vb[cc] = (nbb < N) ? __ldg(hrow + nbb * (E / 4) + 4 * c + tq) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int c = half * 4 + cc;
        const float ae[4] = {va[cc].x, va[cc].y, va[cc].z, va[cc].w};
        const float be[4] = {vb[cc].x, vb[cc].y, vb[cc].z, vb[cc].w};
        const float qe[4] = {qv[c].x, qv[c].y, qv[c].z, qv[c].w};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          uint32_t ah[4], al[4], bh0, bl0, bh1, bl1;
          split_tf32(ae[2 * u], ah[0], al[0]);       // (row g,   k = tq)
          split_tf32(be[2 * u], ah[1], al[1]);       // (row g+8, k = tq)
          split_tf32(ae[2 * u + 1], ah[2], al[2]);   // (row g,   k = tq+4)
          split_tf32(be[2 * u + 1], ah[3], al[3]);   // (row g+8, k = tq+4)
          split_tf32(qe[2 * u], bh0, bl0);           // (k = tq,   n = g)
          split_tf32(qe[2 * u + 1], bh1, bl1);       // (k = tq+4, n = g)
          mma_tf32_16x8x8(acc6[u][0], al, bh0, bh1);
          mma_tf32_16x8x8(acc6[u][1], ah, bl0, bl1);
          mma_tf32_16x8x8(acc6[u][2], ah, bh0, bh1);
        }
      }
    }
    float acc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      acc[i] = ((acc6[0][0][i] + acc6[1][0][i]) + (acc6[0][1][i] + acc6[1][1][i])) + (acc6[0][2][i] + acc6[1][2][i]);
    // C fragment: acc[0], acc[1] = node na, heads 2tq, 2tq+1;  acc[2], acc[3] = node nbb
    if (na < N) { store(na, 0, acc[0]); store(na, 1, acc[1]); }
    if (nbb < N) { store(nbb, 0, acc[2]); store(nbb, 1, acc[3]); }
  }
}

// One head's scores src[n] in the layout of warp_node_softmax: x[i] = node lane + 32 i, -inf for nodes >= N
__device__ __forceinline__ void warp_load_by_head(float (&x)[4], const float* src, int N, int lane) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = lane + 32 * i;
    x[i] = (n < N) ? src[n] : -INFINITY;
  }
}

// Softmax of one head's scores over the nodes, in place: x[i] holds node lane + 32 i (lane = node, 4 strides cover
// N <= 128), -inf for nodes >= N.  The exponential is evaluated only in the ceil(N / 32) strides that hold nodes: in them
// a lane beyond N gets exp(-inf) = 0, and a stride without nodes is 0 without it, so the result is bit for bit what
// `(n < N) ? expf(x - max) : 0` gives for every node.
__device__ __forceinline__ void warp_node_softmax(float (&x)[4], int N) {
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < 4; ++i) mx = fmaxf(mx, x[i]);
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    x[i] = (32 * i < N) ? expf(x[i] - mx) : 0.f;   // ex2.approx was measured: no time gained, mean logit error 4x larger
    sum += x[i];
  }
  sum = warp_sum(sum);
  const float inv = 1.0f / sum;
#pragma unroll
  for (int i = 0; i < 4; ++i) x[i] *= inv;
}

// v[head][i] of node n = lane + 32 i to dst[n * 8 + head] for the nodes < N: the P[n][8] layout the value contraction reads
__device__ __forceinline__ void warp_store_by_node(float* dst, const float (&v)[NH][4], int N, int lane) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = lane + 32 * i;
    if (n < N) {
      *reinterpret_cast<float4*>(dst + n * 8) = make_float4(v[0][i], v[1][i], v[2][i], v[3][i]);
      *reinterpret_cast<float4*>(dst + n * 8 + 4) = make_float4(v[4][i], v[5][i], v[6][i], v[7][i]);
    }
  }
}

// C[head][dim] = sum_n P[n][head] h_n[dim] on the tensor pipe (m16n8k8 TF32 3-term; M = 16 dims, N = 8 heads, K = 8 nodes)
// into the C fragments cacc, P read from slot[n * 8 + head].  Thread g takes the float4 chunks 8cq + g (dims 32cq + 4g + e)
// of node rows n0 + tq and n0 + tq + 4; m-tile j = 2cq + u has row g <-> dim 32cq+4g+2u and row g+8 <-> dim
// 32cq+4g+2u+1.  rows(n0, va, vb) supplies those chunks of the slice of node rows n0 .. n0+7 (va[cq]: row n0 + tq,
// vb[cq]: row n0 + tq + 4), zeros for rows >= N.
template <class Rows>
__device__ __forceinline__ void warp_glimpse_values_acc(float (&cacc)[8][4], const float* slot, int N, int lane, Rows&& rows) {
  const int g = lane >> 2, tq = lane & 3;
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int i = 0; i < 4; ++i) cacc[j][i] = 0.f;
  for (int n0 = 0; n0 < N; n0 += 8) {
    const int na = n0 + tq, nbb = n0 + tq + 4;
    float4 va[4], vb[4];
    rows(n0, va, vb);
    uint32_t bh0, bl0, bh1, bl1;
    split_tf32((na < N) ? slot[na * 8 + g] : 0.f, bh0, bl0);      // (k = tq,   n = head g)
    split_tf32((nbb < N) ? slot[nbb * 8 + g] : 0.f, bh1, bl1);    // (k = tq+4, n = head g)
#pragma unroll
    for (int cq = 0; cq < 4; ++cq) {
      const float ae[4] = {va[cq].x, va[cq].y, va[cq].z, va[cq].w};
      const float be[4] = {vb[cq].x, vb[cq].y, vb[cq].z, vb[cq].w};
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        uint32_t ah[4], al[4];
        split_tf32(ae[2 * u], ah[0], al[0]);       // (row g   = dim 32cq+4g+2u,   k = tq   = node na)
        split_tf32(ae[2 * u + 1], ah[1], al[1]);   // (row g+8 = dim 32cq+4g+2u+1, k = tq)
        split_tf32(be[2 * u], ah[2], al[2]);       // (row g,   k = tq+4 = node nbb)
        split_tf32(be[2 * u + 1], ah[3], al[3]);   // (row g+8, k = tq+4)
        mma_tf32_16x8x8(cacc[2 * cq + u], al, bh0, bh1);
        mma_tf32_16x8x8(cacc[2 * cq + u], ah, bl0, bl1);
        mma_tf32_16x8x8(cacc[2 * cq + u], ah, bh0, bh1);
      }
    }
  }
}

// rows() of warp_glimpse_values_acc for embedding rows hrow[n] in global memory / L2
__device__ __forceinline__ auto glimpse_rows_global(const float4* __restrict__ hrow, int N, int lane) {
  return [=](int n0, float4 (&va)[4], float4 (&vb)[4]) {
    const int g = lane >> 2, na = n0 + (lane & 3), nbb = na + 4;
#pragma unroll
    for (int cq = 0; cq < 4; ++cq) {
      va[cq] = (na < N) ? __ldg(hrow + na * (E / 4) + 8 * cq + g) : make_float4(0.f, 0.f, 0.f, 0.f);
      vb[cq] = (nbb < N) ? __ldg(hrow + nbb * (E / 4) + 8 * cq + g) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
}

// The C fragments of m-tile j = 2cq+u hold [0] (dim d, head 2tq), [1] (dim d, head 2tq+1), [2] (dim d+1, head 2tq),
// [3] (dim d+1, head 2tq+1) with d = 32cq + 4g + 2u.  Both stores below synchronise the warp first, so dst may be the
// slot P was read from.

// c[head][dim] as fp32 to dst[head * 128 + dim]; the warp synchronises again at the end
__device__ __forceinline__ void warp_glimpse_store_c(float* dst, const float (&cacc)[8][4], int lane) {
  const int g = lane >> 2, tq = lane & 3;
  __syncwarp();
#pragma unroll
  for (int cq = 0; cq < 4; ++cq)
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int d = 32 * cq + 4 * g + 2 * u, j = 2 * cq + u;
      *reinterpret_cast<float2*>(dst + (2 * tq) * E + d) = make_float2(cacc[j][0], cacc[j][2]);
      *reinterpret_cast<float2*>(dst + (2 * tq + 1) * E + d) = make_float2(cacc[j][1], cacc[j][3]);
    }
  __syncwarp();
}

// c as row crow of the A operand of GEMM-B, pre-split for the fp16 tensor path (tile_gemm.cuh): k = head * 128 + dim; per
// head and cq one 16-byte chunk = the two k-pairs (d0, d0+1), (d0+2, d0+3), d0 = 32cq + 4g, at the swizzled chunk
// (head*32 + 8cq + g) ^ (tq << 1)
__device__ __forceinline__ void warp_glimpse_store_c16(uint4* crow, const float (&cacc)[8][4], int lane) {
  const int g = lane >> 2, tq = lane & 3;
  __syncwarp();
#pragma unroll
  for (int cq = 0; cq < 4; ++cq)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const uint2 p01 = split_f16x2(cacc[2 * cq][e], cacc[2 * cq][e + 2]);           // dims d0, d0+1 of head 2tq+e
      const uint2 p23 = split_f16x2(cacc[2 * cq + 1][e], cacc[2 * cq + 1][e + 2]);   // dims d0+2, d0+3
      crow[(((2 * tq + e) * 32 + 8 * cq + g) ^ (tq << 1))] = make_uint4(p01.x, p01.y, p23.x, p23.y);
    }
}

// C[head][dim] = sum_n P[n][head] h_n[dim] with the rows from global memory / L2: P is read from slot[n * 8 + head], the
// result replaces it as slot[head * 128 + dim]
__device__ __forceinline__ void warp_glimpse_values(float* slot, const float4* __restrict__ hrow, int N, int lane) {
  float cacc[8][4];
  warp_glimpse_values_acc(cacc, slot, N, lane, glimpse_rows_global(hrow, N, lane));
  warp_glimpse_store_c(slot, cacc, lane);
}

}  // namespace vrpx
