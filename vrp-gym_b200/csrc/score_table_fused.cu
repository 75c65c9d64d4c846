// score_table_fused.cu — the per-episode glimpse score table of the split-step rollout (table mode of vrpx_rollout) in
// ONE kernel: projection on tcgen05, table on mma.sync.
//
// The decoder's glimpse scores at step t >= 1 are  s[b,head,n] = q~[b,head] · h[b,n]  with
// q~ = A_l · h[b,last] + Q~g[b]  (agents/graph_decoder.py:75-94 after the folding of vrpx/packing.py).  The part that
// depends on the step, (A_l h[b,l])_head · h[b,n], takes only N different values of l per instance, and A_l has rank 48
// per head (A_l,head = W_k,head^T · W_l,head / sqrt(48), the reference's own query/key projections).  So once per
// episode
//
//     S1[b][l][head][n] = q'[b,l,head,:] · k'[b,n,head,:],   q' = h · (W_l / sqrt(48))^T,  k' = h · W_k^T
//
// and the decode steps read the 8·N scores of row (b, last) instead of running the 128 -> 1024 query GEMM and the
// 8·N·128 score pass every step.  Algorithmic cost: the table holds B·N·8·N floats (5.2 GB at TSP-50, B = 65536).
//
// Writing q' | k' ((B·N) x 768) to HBM and reading them back would move 10 GB each way at C4 for 1.7 GB of embeddings in
// and 5.2 GB of table out.  Here q' and k' never leave the SM:
//   * a tile = TI = floor(128 / N) whole instances (TI·N <= 128 rows of h), so that a tile's projection holds everything the
//     table rows of its instances need;
//   * CTAs are SPECIALISED by head pair: CTA type g = blockIdx % 4 keeps the 96 KiB of split weights of heads 2g, 2g+1
//     resident in shared memory for its whole life and walks over all tiles (streaming all 384 KiB of weights per tile
//     would need > 10 TB/s from L2).  The four types of a tile run side by side, so h comes from DRAM once;
//   * per (tile, head): D[128 x 96] = XA · W_head^T on tcgen05 (A = the tile as f16 hi/lo in tensor memory, cross terms
//     first, gemm_tc4.cu), then the epilogue warps move D to shared memory — q' rows as fp32, k' rows already split and in
//     mma.sync fragment order — and compute the table rows of the tile's instances on mma.sync.m16n8k16 with f16 hi/lo
//     halves (f16split.cuh, unscaled lo: q' and k' are O(1) projections), ~fp32 accuracy.
// Roles (16 warps): 0-3 X converters (raw fp32 smem tile -> XA in TMEM), 4 TMA producer, 5 MMA issuer (whole warp,
// elected lane), 8-15 epilogue + table (8 warps: two per TMEM lane quarter; table tasks = instance x 16-row query tile).
// TMEM: XA 128 columns | D 2 x 128 (96 used).  Shared memory: weights 96 KiB | raw X 64 KiB | q' 26 KiB | k' fragments 37.5 KiB.
#include "gemm.cuh"
#include "tc_common.cuh"
#include "tile_gemm.cuh"

namespace vrpx {
namespace stf {
using namespace tc4;

constexpr int DQK = 48;                 // decoder head dim
constexpr int HN = 2 * DQK;             // 96 projection columns per head: q' | k'
constexpr int HPC = 2;                  // heads per CTA type
constexpr int NTYPES = NH / HPC;        // 4
constexpr int NTHREADS = 512;
constexpr int W_TMA = 4, W_MMA = 5, W_EPI0 = 8;
constexpr int XBOX = 16 * 1024;         // raw X box: 128 rows x 32 floats
constexpr int WBOX = HN * 128;          // weight box: 96 rows x 128 bytes (64 halves) = 12 KiB
constexpr int W_HEAD = 4 * WBOX;        // hi k0-63 | hi k64-127 | lo k0-63 | lo k64-127 = 48 KiB
constexpr int SM_W = 0;
constexpr int SM_X = HPC * W_HEAD;      // 96 KiB
constexpr int SM_Q = SM_X + 4 * XBOX;   // q' rows: [128][QLD] f32
constexpr int QLD = 52;                 // floats per q' row (48 + 4: conflict-free fragment reads)
constexpr int SM_K = SM_Q + 128 * QLD * 4;
constexpr int KMAX = 200;               // keys of the k' fragment buffer (the host caps TI so that a tile fits, see below)
constexpr int SMEM_BYTES = SM_K + KMAX * 12 * 16 + 1024;
static_assert(SMEM_BYTES + 512 <= 227 * 1024, "shared memory budget");
constexpr uint32_t TM_XA = 0, TM_D = 128, TMEM_COLS = 512;
constexpr uint32_t IDESC = make_idesc(128, HN);

#define VRPX_TMEM_LD16(v, taddr)                                                                                    \
  asm volatile(                                                                                                     \
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                                     \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"                              \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), \
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])                    \
      : "r"(taddr)                                                                                                  \
      : "memory")

// qk_w [768][128] f32 (rows 0..383 = W_l / sqrt(48) per head, 384..767 = W_k per head) -> head-major split halves
// whi | wlo [8][96][128] f16 of W * 2^8: rows 0..47 of head h = its q' rows, 48..95 = its k' rows
__global__ void k_prepare_qkw(const float* __restrict__ qk_w, __half* __restrict__ whi, __half* __restrict__ wlo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NH * HN * E) return;
  const int k = i & (E - 1), r = (i >> 7) % HN, hh = i / (HN * E);
  const int src = (r < DQK) ? (hh * DQK + r) : (NH * DQK + hh * DQK + (r - DQK));
  const float x = qk_w[src * E + k] * W_SCALE;
  const __half hgh = __float2half_rn(x);
  whi[i] = hgh;
  wlo[i] = __float2half_rn(x - __half2float(hgh));
}

template <int NT8>
__global__ void __launch_bounds__(NTHREADS, 1)
k_score_table_fused(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapWh,
                    const __grid_constant__ CUtensorMap mapWl, float* __restrict__ s1, int64_t B, int N, int TI) {
  extern __shared__ unsigned char smem_dyn[];
  __shared__ __align__(8) uint64_t s_w_full, s_xr_full, s_xr_free, s_xa_full, s_xa_free, s_d_full[2], s_d_free[2];
  __shared__ uint32_t s_tmem;
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int type = blockIdx.x % NTYPES, stream = blockIdx.x / NTYPES, nstreams = gridDim.x / NTYPES;
  const int64_t ntiles = (B + TI - 1) / TI;
  const int head0 = type * HPC;

  if (tid == 0) {
    mbar_init(smem_u32(&s_w_full), 1);
    mbar_init(smem_u32(&s_xr_full), 1);
    mbar_init(smem_u32(&s_xr_free), 4);
    mbar_init(smem_u32(&s_xa_full), 4);
    mbar_init(smem_u32(&s_xa_free), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_d_full[i]), 1);
      mbar_init(smem_u32(&s_d_free[i]), 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // the padded keys (n >= N) of the k' fragment buffer stay zero for the whole kernel
  for (int i = tid; i < KMAX * 12; i += NTHREADS) reinterpret_cast<uint4*>(smem + SM_K)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "n"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = s_tmem;

  if (warp == W_TMA) {
    // ===================== TMA producer: the resident weights once, then the raw X tile of every visit =====================
    if (lane == 0) {
      {
        const uint32_t bar = smem_u32(&s_w_full);
        mbar_expect_tx(bar, HPC * W_HEAD);
        for (int hs = 0; hs < HPC; ++hs) {
          unsigned char* dst = smem + SM_W + hs * W_HEAD;
          const int row0 = (head0 + hs) * HN;
          tma_load_2d(smem_u32(dst), &mapWh, 0, row0, bar);
          tma_load_2d(smem_u32(dst + WBOX), &mapWh, 64, row0, bar);
          tma_load_2d(smem_u32(dst + 2 * WBOX), &mapWl, 0, row0, bar);
          tma_load_2d(smem_u32(dst + 3 * WBOX), &mapWl, 64, row0, bar);
        }
      }
      uint32_t cx = 0;
      for (int64_t tile = stream; tile < ntiles; tile += nstreams, ++cx) {
        mbar_wait(smem_u32(&s_xr_free), (cx & 1) ^ 1);
        const uint32_t bar = smem_u32(&s_xr_full);
        mbar_expect_tx(bar, 4 * XBOX);
        const int row0 = (int)(tile * TI * N);
#pragma unroll
        for (int kq = 0; kq < 4; ++kq) tma_load_2d(smem_u32(smem + SM_X + kq * XBOX), &mapX, kq * 32, row0, bar);
      }
    }
  } else if (warp < 4) {
    // ===================== X converters: raw fp32 row -> f16 hi / lo packed words -> XA (thread = tile row) =====================
    const int r = tid;
    const uint32_t xa = tmem + ((uint32_t)(warp * 32) << 16) + TM_XA;
    uint32_t xi = 0;
    for (int64_t tile = stream; tile < ntiles; tile += nstreams, ++xi) {
      mbar_wait(smem_u32(&s_xr_full), xi & 1);
#pragma unroll 1
      for (int kh = 0; kh < 2; ++kh) {
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int half = 0; half < 2; ++half)
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float4 xv = *reinterpret_cast<const float4*>(smem + SM_X + (2 * kh + half) * XBOX + r * 128 + ((c ^ (r & 7)) << 4));
            split_pair(xv.x, xv.y, hi[half * 16 + 2 * c], lo[half * 16 + 2 * c]);
            split_pair(xv.z, xv.w, hi[half * 16 + 2 * c + 1], lo[half * 16 + 2 * c + 1]);
          }
        if (kh == 0) {
          mbar_wait(smem_u32(&s_xa_free), (xi & 1) ^ 1);        // the previous visit's products are complete
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        tmem_st32(xa + kh * 32, hi);
        tmem_st32(xa + 64 + kh * 32, lo);
      }
      asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(smem_u32(&s_xr_free));                       // the raw tile may be refilled
        mbar_arrive(smem_u32(&s_xa_full));
      }
    }
  } else if (warp == W_MMA) {
    // ===================== MMA issuer (whole warp converged, elected lane issues) =====================
    mbar_wait(smem_u32(&s_w_full), 0);
    uint32_t ti = 0, dc = 0;   // tile visits, accumulator uses
    for (int64_t tile = stream; tile < ntiles; tile += nstreams, ++ti) {
      mbar_wait(smem_u32(&s_xa_full), ti & 1);
      for (int hs = 0; hs < HPC; ++hs, ++dc) {
        const uint32_t s = dc & 1, ph = (dc >> 1) & 1;
        mbar_wait(smem_u32(&s_d_free[s]), ph ^ 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d = tmem + TM_D + s * 128, xh = tmem + TM_XA, xl = tmem + TM_XA + 64;
        unsigned char* wb = smem + SM_W + hs * W_HEAD;
        const uint64_t wh[2] = {make_desc(smem_u32(wb)), make_desc(smem_u32(wb + WBOX))};
        const uint64_t wl[2] = {make_desc(smem_u32(wb + 2 * WBOX)), make_desc(smem_u32(wb + 3 * WBOX))};
#pragma unroll
        for (int kh = 0; kh < 2; ++kh)
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            const uint64_t o = (uint64_t)(2 * jj);
            const uint32_t ka = 8 * (4 * kh + jj);
            mma_f16_ts_w(d, xl + ka, wh[kh] + o, (kh | jj) ? 1u : 0u, IDESC);
            mma_f16_ts_w(d, xh + ka, wl[kh] + o, 1u, IDESC);
          }
#pragma unroll
        for (int kh = 0; kh < 2; ++kh)
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) mma_f16_ts_w(d, xh + 8 * (4 * kh + jj), wh[kh] + (uint64_t)(2 * jj), 1u, IDESC);
        mma_commit_w(smem_u32(&s_d_full[s]));
      }
      mma_commit_w(smem_u32(&s_xa_free));
    }
  } else if (warp >= W_EPI0) {
    // ===================== epilogue + table =====================
    const int ew = warp - W_EPI0, q = warp & 3, half = ew >> 2;   // TMEM lane quarter; 0: q' columns, 1: k' columns
    const int g = lane >> 2, t = lane & 3;
    float* Qs = reinterpret_cast<float*>(smem + SM_Q);
    uint4* Kf = reinterpret_cast<uint4*>(smem + SM_K);
    // query tiles per instance; keys per instance in the fragment buffer (padded to 8).  The table loop below runs over
    // the NT8 key tiles of the template bucket: tiles past KP read the next instance's keys (or the zeroed tail) into
    // accumulators that are never stored.
    const int MT = (N + 15) / 16, KP = 8 * ((N + 7) / 8);
    const bool vec_ok = (N & 1) == 0;
    uint32_t dc = 0;
    for (int64_t tile = stream; tile < ntiles; tile += nstreams) {
      const int64_t b0 = tile * TI;
      const int ninst = (int)((B - b0 < TI) ? (B - b0) : TI);
      for (int hs = 0; hs < HPC; ++hs, ++dc) {
        const uint32_t s = dc & 1, ph = (dc >> 1) & 1;
        const int head = head0 + hs;
        mbar_wait(smem_u32(&s_d_full[s]), ph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- D row (= tile row r) -> registers: this thread's 48 columns (q' or k' of the head)
        uint32_t v[48];
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + TM_D + s * 128 + half * DQK;
        VRPX_TMEM_LD16(v, taddr);
        VRPX_TMEM_LD16((v + 16), taddr + 16);
        VRPX_TMEM_LD16((v + 32), taddr + 32);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&s_d_free[s]));
        const int r = q * 32 + lane;
        if (r < ninst * N) {
          if (half == 0) {
#pragma unroll
            for (int c = 0; c < 12; ++c)
              *reinterpret_cast<float4*>(Qs + r * QLD + 4 * c) =
                  make_float4(__uint_as_float(v[4 * c]) * OUT_SCALE, __uint_as_float(v[4 * c + 1]) * OUT_SCALE,
                              __uint_as_float(v[4 * c + 2]) * OUT_SCALE, __uint_as_float(v[4 * c + 3]) * OUT_SCALE);
          } else {
            // key n of instance i -> B-fragment order of the table loop below, 16 B per [key][k16 step c][slot tt] =
            // {hi(dims 16c+2tt, +1), hi(dims 16c+2tt+8, +9), lo(..), lo(..)}: one conflict-free LDS.128 per B fragment,
            // the hi / lo pairs adjacent as the two-register HMMA operand
            const int i = r / N, n = r - i * N;
            uint4* dst = Kf + (size_t)(i * KP + n) * 12;
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
              for (int tt = 0; tt < 4; ++tt) {
                const uint2 p0 = split_f16x2_u(__uint_as_float(v[16 * c + 2 * tt]) * OUT_SCALE, __uint_as_float(v[16 * c + 2 * tt + 1]) * OUT_SCALE);
                const uint2 p1 = split_f16x2_u(__uint_as_float(v[16 * c + 2 * tt + 8]) * OUT_SCALE, __uint_as_float(v[16 * c + 2 * tt + 9]) * OUT_SCALE);
                dst[c * 4 + tt] = make_uint4(p0.x, p1.x, p0.y, p1.y);
              }
          }
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // q' and k' of the tile are in shared memory (8 epilogue warps)
        // ---- table rows: task = (instance i, 16-row query tile m), round robin over the 8 warps
        for (int task = ew; task < ninst * MT; task += 8) {
          const int i = task / MT, m = task - i * MT;
          const int la = 16 * m + g, lb = la + 8;
          const float* qa = Qs + (i * N + la) * QLD;
          const float* qb = Qs + (i * N + lb) * QLD;
          const uint4* Ks = Kf + (size_t)i * KP * 12;
          float acc[NT8][4];
#pragma unroll
          for (int j = 0; j < NT8; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[j][e] = 0.f;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            float2 a0 = make_float2(0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
            if (la < N) { a0 = *reinterpret_cast<const float2*>(qa + 16 * c + 2 * t); a2 = *reinterpret_cast<const float2*>(qa + 16 * c + 2 * t + 8); }
            if (lb < N) { a1 = *reinterpret_cast<const float2*>(qb + 16 * c + 2 * t); a3 = *reinterpret_cast<const float2*>(qb + 16 * c + 2 * t + 8); }
            const uint2 s0 = split_f16x2_u(a0.x, a0.y), s1_ = split_f16x2_u(a1.x, a1.y);
            const uint2 s2 = split_f16x2_u(a2.x, a2.y), s3 = split_f16x2_u(a3.x, a3.y);
            const uint32_t ah[4] = {s0.x, s1_.x, s2.x, s3.x}, al[4] = {s0.y, s1_.y, s2.y, s3.y};
#pragma unroll
            for (int j = 0; j < NT8; ++j) {
              const uint4 kf = Ks[((8 * j + g) * 3 + c) * 4 + t];
              mma3_f16(acc[j], ah, al, kf.x, kf.y, kf.z, kf.w);
            }
          }
          const int64_t b = b0 + i;
          float* ra = s1 + (((size_t)b * N + la) * NH + head) * N;
          float* rb = s1 + (((size_t)b * N + lb) * NH + head) * N;
#pragma unroll
          for (int j = 0; j < NT8; ++j) {
            const int n = 8 * j + 2 * t;
            if (vec_ok) {
              if (n < N) {
                if (la < N) *reinterpret_cast<float2*>(ra + n) = make_float2(acc[j][0], acc[j][1]);
                if (lb < N) *reinterpret_cast<float2*>(rb + n) = make_float2(acc[j][2], acc[j][3]);
              }
            } else {
              if (la < N) {
                if (n < N) ra[n] = acc[j][0];
                if (n + 1 < N) ra[n + 1] = acc[j][1];
              }
              if (lb < N) {
                if (n < N) rb[n] = acc[j][2];
                if (n + 1 < N) rb[n + 1] = acc[j][3];
              }
            }
          }
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // every warp is done with q' / k' before the next head overwrites them
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS) : "memory");
  }
}

template <int NT8>
static int launch(const CUtensorMap& mx, const CUtensorMap& mwh, const CUtensorMap& mwl, float* s1, int64_t B, int N, int TI,
                  cudaStream_t stream) {
  VRPX_CUDA(cudaFuncSetAttribute(k_score_table_fused<NT8>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  const int64_t ntiles = (B + TI - 1) / TI;
  int64_t streams = num_sms() / NTYPES;
  if (streams > ntiles) streams = ntiles;
  if (streams < 1) streams = 1;
  k_score_table_fused<NT8><<<(unsigned)(streams * NTYPES), NTHREADS, SMEM_BYTES, stream>>>(mx, mwh, mwl, s1, B, N, TI);
  VRPX_LAUNCH_CHECK();
  return VRPX_OK;
}

}  // namespace stf

// S1[B][N][8][N] from h [B][N][128] and qk_w [768][128]; w16 = scratch of 2 x 768 x 128 halves (head-major hi | lo)
int build_score_table_fused(const float* h, const float* qk_w, int64_t B, int N, __half* w16, float* s1, cudaStream_t stream) {
  using namespace stf;
  if (N < 2 || N > VRPX_MAX_NODES || B < 1 || (reinterpret_cast<uintptr_t>(w16) & 15)) {
    set_error("build_score_table_fused: bad argument");
    return VRPX_ERR_ARG;
  }
  constexpr int NW = NH * HN * E;
  k_prepare_qkw<<<(NW + 255) / 256, 256, 0, stream>>>(qk_w, w16, w16 + NW);
  VRPX_LAUNCH_CHECK();
  CUtensorMap mx, mwh, mwl;
  int rc;
  if ((rc = make_map(&mx, h, B * N, E, false))) return rc;
  if ((rc = make_map(&mwh, w16, NH * HN, E, true, HN))) return rc;
  if ((rc = make_map(&mwl, w16 + NW, NH * HN, E, true, HN))) return rc;
  const int nt = (N + 7) / 8, bucket = nt <= 3 ? 3 : (nt <= 7 ? 7 : (nt <= 13 ? 13 : 16));
  // instances per tile: whole instances in 128 rows, and (TI - 1) * KP + bucket * 8 keys must fit the fragment buffer
  int TI = 128 / N;
  const int cap = 1 + (KMAX - bucket * 8) / (nt * 8);
  if (TI > cap) TI = cap;
  if (TI < 1 || bucket * 8 > KMAX) {
    set_error("build_score_table_fused: key buffer too small for N=%d", N);
    return VRPX_ERR_ARG;
  }
  if (nt <= 3) return launch<3>(mx, mwh, mwl, s1, B, N, TI, stream);
  if (nt <= 7) return launch<7>(mx, mwh, mwl, s1, B, N, TI, stream);
  if (nt <= 13) return launch<13>(mx, mwh, mwl, s1, B, N, TI, stream);
  return launch<16>(mx, mwh, mwl, s1, B, N, TI, stream);
}

}  // namespace vrpx

extern "C" int vrpx_debug_score_table(const float* h, const float* qk_w, int64_t B, int32_t N, float* s1, void* stream) {
  VRPX_CHECK_ARG(h && qk_w && s1, "NULL argument");
  VRPX_DEVICE_GUARD(h);
  __half* w16 = vrpx::tc4::split_scratch((cudaStream_t)stream);
  if (!w16) return VRPX_ERR_CUDA;
  return vrpx::build_score_table_fused(h, qk_w, B, N, w16, s1, (cudaStream_t)stream);
}
