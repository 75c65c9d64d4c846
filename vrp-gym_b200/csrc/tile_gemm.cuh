// tile_gemm.cuh — CTA-level building blocks shared by the persistent rollout kernel (rollout.cu) and the
// recompute-based decoder backward (decoder_bwd.cu): tiles of 16 or 32 instances, 512 threads, tile GEMMs on the
// warp-level tensor path (mma.sync TF32, 3-term split) with per-warp weight streams from L2 (cp.async rings).
#pragma once
#include "env_rules.cuh"
#include "f16split.cuh"

namespace vrpx {

constexpr int TM = 32;        // instances per tile
constexpr int NT = 512;       // threads per CTA (16 warps; <= 128 registers per thread)
constexpr int QW = NH * E;    // 1024: per-instance width of q~ / c
constexpr size_t SMEM_W = 64 * 1024;                         // weight rings of the backward kernel: 16 warps x 2 x 2 KiB

__device__ __forceinline__ unsigned ld_acquire(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ld_acquire_i(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(bar, 1u);
    while (ld_acquire(bar) < target) __nanosleep(32);
    __threadfence();
  }
  __syncthreads();
}

// Sum 8 per-lane values across the warp; lane l returns the total of v[(l >> 2) & 7].
__device__ __forceinline__ float reduce8(const float v[8], int lane) {
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
  float w4[4], w2[2], x;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float keep = b4 ? v[i + 4] : v[i], send = b4 ? v[i] : v[i + 4];
    w4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    float keep = b3 ? w4[i + 2] : w4[i], send = b3 ? w4[i] : w4[i + 2];
    w2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  {
    float keep = b2 ? w2[1] : w2[0], send = b2 ? w2[0] : w2[1];
    x = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  x += __shfl_xor_sync(0xffffffffu, x, 2);
  x += __shfl_xor_sync(0xffffffffu, x, 1);
  return x;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// glimpse-mask source row for attention row (b, hh): mask.repeat(H,1) indexing (graph_decoder.py:93)
__device__ __forceinline__ int64_t quirk_row(int64_t b, int hh, long long G) {
  if (G <= 0) return b;
  if (G < (1ll << 28) && b < (1ll << 31)) {   // 32-bit arithmetic (every per-GPU batch): two cheap divisions per call
    const uint32_t g = (uint32_t)G, bb = (uint32_t)b, g0 = (bb / g) * g;
    return (int64_t)(g0 + ((bb - g0) * NH + (uint32_t)hh) % g);
  }
  int64_t g0 = (b / G) * G;
  return g0 + (((b - g0) * NH + hh) % G);
}

// ================================================================ tensor-pipe tile GEMMs
// Two tile GEMMs (wide: [rows x 128]·[128 x 1024], tall: [rows x 1024]·[1024 x 128]) on the legacy warp-level tensor path: mma.sync.m16n8k8 TF32 with the 3-term split
// (acc += Alo·Bhi + Ahi·Blo + Ahi·Bhi, ~fp32 accuracy).  Measured on B200 (tools/mma_bench.cu): 480 MAC/clk/SM for
// mma.sync TF32 vs 123 MAC/clk/SM for FFMA, and the tensor pipe runs beside the FMA pipe.  tcgen05 needs M >= 64
// rows per instruction and operands in the UMMA smem layout; a 32-instance tile whose 1024-wide result must stay in
// shared memory for the per-instance phases does not fit that shape, so these tile GEMMs use register fragments.
// Shared-memory leading dimensions are padded so that fragment loads are bank-conflict free:
constexpr int XS_LD = E + 4;        // 132: A fragments (row g, col t): bank (4g + t) % 32
constexpr int QC_LD = QW + 4;       // 1028
template <int MT> constexpr size_t smem_x_mma() { return (size_t)(16 * MT) * XS_LD * sizeof(float); }
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32_16x8x8(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// A fragments (hi and lo) of the two 16-row tiles for one k-step, from a row-major smem matrix with leading dim ld.
template <int MT>
__device__ __forceinline__ void load_a_frags(const float* __restrict__ A, int ld, int k0, int g, int t,
                                             uint32_t (&ah)[MT][4], uint32_t (&al)[MT][4]) {
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) {
    const float* r0 = A + (mt * 16 + g) * ld + k0 + t;
    const float* r1 = r0 + 8 * ld;
    split_tf32(r0[0], ah[mt][0], al[mt][0]);
    split_tf32(r1[0], ah[mt][1], al[mt][1]);
    split_tf32(r0[4], ah[mt][2], al[mt][2]);
    split_tf32(r1[4], ah[mt][3], al[mt][3]);
  }
}

// ---------------------------------------------------------------- swizzled-stage variants, NST-deep weight pipeline
// Same tensor-pipe tile GEMMs with an UNPADDED per-warp weight stage [8 k-rows][NC = 8 NJ columns]: the 16-byte chunks of
// row r are stored at column c ^ ((r & 3) << 3), which makes the B-fragment reads (k = t, n = g) conflict free without
// the 8-float row padding, and a ring of NST stages per warp.  Both kernels run NST = 2 for the wide GEMMs: a third stage
// was measured 10 % SLOWER in the rollout kernel (59 -> 65 ms at C4) — the extra 32 KiB of shared memory comes out of the
// L1 that caches the per-instance embedding streams of the neighbouring phases.
template <int NJ>
__device__ __forceinline__ void stage_warp_kstep_sw(const float* __restrict__ src, int ld, int kstep,
                                                    float* __restrict__ dst, int lane) {
  constexpr int NC = 8 * NJ, F4 = NC / 4;
#pragma unroll
  for (int i = 0; i < (8 * F4) / 32; ++i) {
    const int idx = lane + 32 * i;
    const int r = idx / F4, c4 = idx % F4;
    cp_async16(dst + r * NC + ((c4 * 4) ^ ((r & 3) << 3)), src + (size_t)(kstep * 8 + r) * ld + c4 * 4);
  }
}

template <int MT, int NJ, int NST>
__device__ __forceinline__ void warp_gemm_mma_sw(float (&acc)[MT][NJ][4], const float* __restrict__ A, int lda, int k_base,
                                                 const float* __restrict__ wsrc, int wld, int nks,
                                                 float* __restrict__ wbuf, int lane) {
  constexpr int NC = 8 * NJ, STAGE = 8 * NC;
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int s = 0; s < NST - 1; ++s) {
    if (s < nks) stage_warp_kstep_sw<NJ>(wsrc, wld, s, wbuf + s * STAGE, lane);
    cp_async_commit();
  }
  for (int ks = 0; ks < nks; ++ks) {
    // all lanes finished reading the stage refilled below (it held k-step ks - 1) at the end of the last iteration
    if (ks + NST - 1 < nks) stage_warp_kstep_sw<NJ>(wsrc, wld, ks + NST - 1, wbuf + ((ks + NST - 1) % NST) * STAGE, lane);
    cp_async_commit();            // possibly empty: keeps the group count uniform
    cp_async_wait<NST - 1>();     // k-step ks has landed
    __syncwarp();
    uint32_t ah[MT][4], al[MT][4];
    load_a_frags<MT>(A, lda, k_base + ks * 8, g, t, ah, al);
    const float* wb = wbuf + (ks % NST) * STAGE;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int c = (8 * j + g) ^ (t << 3);
      uint32_t bh0, bl0, bh1, bl1;
      split_tf32(wb[t * NC + c], bh0, bl0);
      split_tf32(wb[(t + 4) * NC + c], bh1, bl1);
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        mma_tf32_16x8x8(acc[mt][j], al[mt], bh0, bh1);
        mma_tf32_16x8x8(acc[mt][j], ah[mt], bl0, bl1);
        mma_tf32_16x8x8(acc[mt][j], ah[mt], bh0, bh1);
      }
    }
    __syncwarp();
  }
  cp_async_wait<0>();
}

// out[16 MT][1024] = init + Xs[16 MT][128] (ld lda) · Wt[128][1024]; warp w owns columns [64w, 64w + 64).
// Wb: 16 warps x NST stages x 512 floats (NST = 2: 64 KiB, NST = 3: 96 KiB).
template <int MT, int NST, class Init, class Epi>
__device__ __forceinline__ void tile_gemm_wide_mma_sw(const float* __restrict__ Xs, int lda, const float* __restrict__ Wt,
                                                      float* __restrict__ Wb, Init init, Epi epi) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  float acc[MT][8][4];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = warp * 64 + 8 * j + 2 * t;
      const float2 i0 = init(mt * 16 + g, c), i1 = init(mt * 16 + g + 8, c);
      acc[mt][j][0] = i0.x; acc[mt][j][1] = i0.y; acc[mt][j][2] = i1.x; acc[mt][j][3] = i1.y;
    }
  warp_gemm_mma_sw<MT, 8, NST>(acc, Xs, lda, 0, Wt + warp * 64, QW, 16, Wb + warp * NST * 512, lane);
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = warp * 64 + 8 * j + 2 * t;
      epi(mt * 16 + g, c, acc[mt][j][0], acc[mt][j][1]);
      epi(mt * 16 + g + 8, c, acc[mt][j][2], acc[mt][j][3]);
    }
}

// out[16 MT][128] (ld out_ld) = Cs[16 MT][1024] (ld ldc) · Mt[1024][128] + bias, split-K over KG warp groups: warp
// (kg = w / NG, ng = w % NG), NG = 16 / KG, owns 128 / NG columns over the k range [1024 / KG · kg, +1024 / KG); the KG
// partial sums go through `part` ([KG][16 MT][128] floats; may alias Wb or Cs — it is written only after every warp has
// left the k loop).
template <int MT, int KG, int NST>
__device__ __forceinline__ void tile_gemm_tall_mma_sw(const float* __restrict__ Cs, int ldc, const float* __restrict__ Mt,
                                                      float* __restrict__ Wb, const float* __restrict__ bias,
                                                      float* __restrict__ part, float* __restrict__ out, int out_ld) {
  constexpr int TMm = 16 * MT, NG = (NT / 32) / KG, NCW = E / NG, NJ = NCW / 8, KR = QW / KG;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int kg = warp / NG, ng = warp % NG;
  float acc[MT][NJ][4];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int j = 0; j < NJ; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[mt][j][i] = 0.f;
  warp_gemm_mma_sw<MT, NJ, NST>(acc, Cs, ldc, kg * KR, Mt + (size_t)kg * KR * E + ng * NCW, E, KR / 8,
                                Wb + warp * NST * (8 * NCW), lane);
  __syncthreads();
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      // columns XOR-swizzled by the row (bits 3-4) so that the 8 rows a warp stores at once fall into distinct banks
      const int c = (ng * NCW + 8 * j + 2 * t) ^ ((g & 3) << 3);
      *reinterpret_cast<float2*>(part + (kg * TMm + mt * 16 + g) * E + c) = make_float2(acc[mt][j][0], acc[mt][j][1]);
      *reinterpret_cast<float2*>(part + (kg * TMm + mt * 16 + g + 8) * E + c) = make_float2(acc[mt][j][2], acc[mt][j][3]);
    }
  __syncthreads();
  for (int o = tid; o < TMm * E; o += NT) {
    float s = 0.f;
    const int os = o ^ (((o >> 7) & 3) << 3);
#pragma unroll
    for (int k = 0; k < KG; ++k) s += part[k * TMm * E + os];
    out[(o >> 7) * out_ld + (o & (E - 1))] = s + (bias ? bias[o & (E - 1)] : 0.f);
  }
  __syncthreads();
}

// ================================================================ fp16-split tile GEMM (rollout GEMM-B)
// f16split.cuh, scaled-lo variant.  Both operands are stored PRE-SPLIT as {hi2, lo2} = 8 bytes per pair of consecutive k,
// which is what one register of the m16n8k16 fragments holds, so the k loop has no conversion arithmetic at all.
// A operand of the fp16-split tall GEMM: C16[16][C16_LD] uint2, element (m, kp) = split pair (k = 2kp, 2kp + 1) of row m,
// stored at column kp ^ (((kp >> 7) & 3) << 2).  The XOR (by the head pair the k-pair belongs to) lets the producer
// (rollout.cu, glimpse value pass: lanes of equal g and different t write different head pairs) store 16-byte chunks
// without bank conflicts; C16_LD = 4 (mod 16) keeps the fragment reads (row g, k-pair t) conflict free.
constexpr int C16_LD = QW / 2 + 4;   // 516 uint2 = 1032 floats per row
__device__ __forceinline__ int c16_col(int kp) { return kp ^ (((kp >> 7) & 3) << 2); }

// out[16][128] (ld out_ld) = C[16][1024] · M[1024][128] + bias with pre-split operands.  M16: global [512 k-pairs][128]
// uint2.  16 warps: warp (kg = w / 4, ng = w % 4) owns columns [32 ng, +32) over k-pairs [128 kg, +128); each streams its
// slice through a private cp.async ring of NST stages of [8 k-pairs][32 columns] uint2 (2 KiB; column c of row r at
// c ^ ((r & 3) << 2): fragment reads (k-pair t, column g) conflict free).  part: [4][16][128] floats, may alias C16.
// Measured (C4): this loop is bound by the L2 -> SM stream of the weights (512 KiB per 16-instance tile on every SM at
// once), not by the tensor pipe or the issue slots: a leaner k loop (vector fragment loads, no register moves) and a
// deeper ring both left its time unchanged.
template <int NST>
__device__ __forceinline__ void tile_gemm_tall_f16(const uint2* __restrict__ C16, const uint2* __restrict__ M16,
                                                   float* __restrict__ Wb, const float* __restrict__ bias,
                                                   float* __restrict__ part, float* __restrict__ out, int out_ld) {
  constexpr int KG = 4, NG = 4, NJ = 4, KPW = (QW / 2) / KG, NKS = KPW / 8, STAGE = 8 * 32;   // STAGE in uint2
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int kg = warp / NG, ng = warp % NG;
  uint2* wbuf = reinterpret_cast<uint2*>(Wb) + warp * NST * STAGE;
  const uint2* src = M16 + (size_t)(kg * KPW) * E + ng * 32;
  auto stage = [&](int ks, uint2* dst) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = lane + 32 * i, r = idx >> 4, c2 = idx & 15;
      cp_async16(dst + r * 32 + ((2 * c2) ^ ((r & 3) << 2)), src + (size_t)(ks * 8 + r) * E + 2 * c2);
    }
  };
  float ahh[NJ][4], amx[NJ][4];
#pragma unroll
  for (int j = 0; j < NJ; ++j)
#pragma unroll
    for (int i = 0; i < 4; ++i) ahh[j][i] = amx[j][i] = 0.f;
#pragma unroll
  for (int s = 0; s < NST - 1; ++s) {
    if (s < NKS) stage(s, wbuf + s * STAGE);
    cp_async_commit();
  }
  const uint2* row0 = C16 + g * C16_LD;
  const uint2* row1 = C16 + (g + 8) * C16_LD;
  for (int ks = 0; ks < NKS; ++ks) {
    if (ks + NST - 1 < NKS) stage(ks + NST - 1, wbuf + ((ks + NST - 1) % NST) * STAGE);
    cp_async_commit();
    cp_async_wait<NST - 1>();
    __syncwarp();
    const int kp0 = kg * KPW + ks * 8;
    const int ca = c16_col(kp0 + t), cb = c16_col(kp0 + t + 4);
    const uint2 a0 = row0[ca], a1 = row1[ca], a2 = row0[cb], a3 = row1[cb];
    const uint32_t ah[4] = {a0.x, a1.x, a2.x, a3.x}, al[4] = {a0.y, a1.y, a2.y, a3.y};
    const uint2* wb = wbuf + (ks % NST) * STAGE;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int c = (8 * j + g) ^ (t << 2);
      const uint2 b0 = wb[t * 32 + c], b1 = wb[(t + 4) * 32 + c];
      mma_f16_16x8x16(ahh[j], ah, b0.x, b1.x);
      mma_f16_16x8x16(amx[j], al, b0.x, b1.x);
      mma_f16_16x8x16(amx[j], ah, b0.y, b1.y);
    }
    __syncwarp();
  }
  cp_async_wait<0>();
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int c = (ng * 32 + 8 * j + 2 * t) ^ ((g & 3) << 3);   // same row swizzle as tile_gemm_tall_mma_sw
    const float sc = 1.0f / F16_LO_SCALE;
    *reinterpret_cast<float2*>(part + (kg * 16 + g) * E + c) = make_float2(fmaf(amx[j][0], sc, ahh[j][0]), fmaf(amx[j][1], sc, ahh[j][1]));
    *reinterpret_cast<float2*>(part + (kg * 16 + g + 8) * E + c) = make_float2(fmaf(amx[j][2], sc, ahh[j][2]), fmaf(amx[j][3], sc, ahh[j][3]));
  }
  __syncthreads();
  for (int o = tid; o < 16 * E; o += NT) {
    float s = 0.f;
    const int os = o ^ (((o >> 7) & 3) << 3);
#pragma unroll
    for (int k = 0; k < KG; ++k) s += part[k * 16 * E + os];
    out[(o >> 7) * out_ld + (o & (E - 1))] = s + (bias ? bias[o & (E - 1)] : 0.f);
  }
  __syncthreads();
}

}  // namespace vrpx
