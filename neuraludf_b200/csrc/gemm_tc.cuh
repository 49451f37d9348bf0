// tcgen05 tensor-core GEMM engine for sm_100a with an fp32-grade 3xBF16 operand split.
//
//   D[128 x N] (fp32, TMEM)  =  sum over K slices of   A_hi*B_hi + A_hi*B_lo + A_lo*B_hi        (kind::f16, bf16 inputs)
//   (2 planes, 3 products, ~4e-6 vs fp64)   or, with 3 planes hi/mid/lo, the 6 products of weight >= 2^-16 (fp32-grade).
//
// x = hi + lo with hi = bf16(x), lo = bf16(x - hi): the three products keep ~16 mantissa bits of each operand, which is
// what the parity tolerance needs (plain BF16/TF32 operands do not: SURVEY.md section 0, fact 3).
//
// Structure of one CTA (320 threads, one 128-row output tile, 2-stage smem ring, K sliced by 64):
//   warps 0-7  producers: stage the fp32 A tile from global memory, split it to bf16 planes and write it into the UMMA
//              K-major SWIZZLE_128B shared-memory layout; after the last slice the same warps run the epilogue
//              (tcgen05.ld of the accumulator -> fused epilogue functor -> global): warp w reads TMEM lane quadrant
//              w%4 and every second 32-column chunk (w/4);
//   warp 8     MMA issuer: one elected lane issues tcgen05.mma (M=128, N<=256, K=16) and tcgen05.commit;
//              the warp also owns the TMEM allocation;
//   warp 9     weight loader: one lane issues cp.async.bulk (TMA engine, UBLKCP) of the pre-split, pre-swizzled weight
//              slice image (built once per optimiser step by tc_prep_weights_kernel) with mbarrier complete_tx.
// The weight-gradient variant (gemm_tn) stages BOTH operands from fp32 activations with an on-the-fly transpose
// (contraction over points); each split-K partial tile goes to its own workspace slice, added in order by sum_slices.
#pragma once
#include <cuda_bf16.h>

#include "gemm_simt.cuh"
#include "planes.cuh"

namespace nudf {
namespace tc {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int STAGES = 2;
constexpr int NPROD = 256;     // producer / epilogue threads (warps 0-7)
constexpr int THREADS = 320;   // + warp 8 (MMA issuer, TMEM owner) + warp 9 (weight loader)
constexpr int A_HALF_BYTES = BM * BK * 2;   // 16 KB: one of (hi, lo)

__host__ __device__ inline int pad16(int n) { return (n + 15) & ~15; }
__host__ __device__ inline int pad64(int k) { return (k + 63) & ~63; }
// ---- weight image --------------------------------------------------------------------------------------------------
// For operand B(n, k), n < N, k < K: n-tiles of NT rows (NT = 256 with 2 planes, 128 with 3 planes; the last tile is
// padded to a multiple of 16), k-slices of 64.  NP planes per element: p0 = bf16(x), p1 = bf16(x - p0),
// p2 = bf16(x - p0 - p1).  Image order: [n_tile][k_slice][plane][tile rows x 128 B, SWIZZLE_128B K-major].  Units: uint16.
__host__ __device__ inline int nt_of(int np) { return np == 2 ? 256 : 128; }
__host__ __device__ inline int n_tiles(int N, int np) { return (N + nt_of(np) - 1) / nt_of(np); }
__host__ __device__ inline int tile_rows(int N, int t, int np) { int r = N - nt_of(np) * t; return pad16(r < nt_of(np) ? r : nt_of(np)); }
__host__ __device__ inline int64_t tile_elems(int N, int K, int t, int np) { return (int64_t)(pad64(K) / 64) * np * tile_rows(N, t, np) * 64; }
__host__ __device__ inline int64_t tile_offset(int N, int K, int t, int np) {
  int64_t o = 0;
  for (int i = 0; i < t; ++i) o += tile_elems(N, K, i, np);
  return o;
}
__host__ __device__ inline int64_t image_elems(int N, int K, int np) { return tile_offset(N, K, n_tiles(N, np), np); }

// transposed == 0: B(n,k) = W[n*ldw + k]   (X W^T)      transposed == 1: B(n,k) = W[k*ldw + n]   (dY W)
static __device__ __forceinline__ void tc_prep_weights_body(const float* __restrict__ W, int64_t ldw, int N, int K, int transposed, int np,
                                                            uint16_t* __restrict__ img, int64_t start, int64_t stride) {
  const int Kp = pad64(K);
  const int nt = n_tiles(N, np);
  int64_t total = 0;
  for (int t = 0; t < nt; ++t) total += (int64_t)tile_rows(N, t, np) * Kp;
  for (int64_t idx = start; idx < total; idx += stride) {
    int64_t rem = idx;
    int t = 0;
    while (rem >= (int64_t)tile_rows(N, t, np) * Kp) { rem -= (int64_t)tile_rows(N, t, np) * Kp; ++t; }
    const int rows = tile_rows(N, t, np);
    const int nl = (int)(rem / Kp), k = (int)(rem - (int64_t)nl * Kp);
    const int n = t * nt_of(np) + nl;
    float x = 0.f;
    if (n < N && k < K) x = transposed ? W[(int64_t)k * ldw + n] : W[(int64_t)n * ldw + k];
    const int s = k >> 6, kl = k & 63;
    uint16_t* base = img + tile_offset(N, K, t, np) + (int64_t)s * np * rows * 64;
    const uint32_t off = sw128((uint32_t)nl, (uint32_t)kl) >> 1;
    float r = x;
    for (int p = 0; p < np; ++p) {
      __nv_bfloat16 h = __float2bfloat16_rn(r);
      base[(int64_t)p * rows * 64 + off] = __bfloat16_as_ushort(h);
      r -= __bfloat162float(h);
    }
  }
}
static __global__ void tc_prep_weights_kernel(const float* __restrict__ W, int64_t ldw, int N, int K, int transposed, int np,
                                              uint16_t* __restrict__ img) {
  tc_prep_weights_body(W, ldw, N, K, transposed, np, img, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, (int64_t)gridDim.x * blockDim.x);
}

// ---- PTX wrappers --------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(addr), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  while (!mbar_try_wait(addr, parity)) {
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// generic-proxy smem writes -> visible to the async proxy (tensor core operand fetch)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// K-major SWIZZLE_128B operand descriptor: start address, LBO = 16 B (ignored for swizzled K-major), SBO = 1024 B
// (8 rows x 128 B), version 1 (sm_100), layout type 2 (SWIZZLE_128B).  See cute/arch/mma_sm100_desc.hpp.
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D = F32, A = B = BF16, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t make_idesc(uint32_t n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float v[32]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

template <int NT>   // NT = number of producer threads (128 or 256); fetches this thread's part of a [128 x 64] fp32 slice
__device__ __forceinline__ void fetch_a(const float* __restrict__ A, int64_t lda, int64_t m0, int64_t M, int k0, int K, int tid,
                                        bool vec_ok, float4 (&v)[BM * 16 / NT]) {
  const int c = tid & 15;            // float4 chunk along k
  const int rsub = tid >> 4;         // 0 .. NT/16-1
  const int k = k0 + c * 4;
#pragma unroll
  for (int pass = 0; pass < BM * 16 / NT; ++pass) {
    const int64_t row = m0 + pass * (NT / 16) + rsub;
    v[pass] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < M) {
      const float* p = A + row * lda + k;
      if (vec_ok && k + 3 < K) {
        v[pass] = *reinterpret_cast<const float4*>(p);
      } else {
        if (k + 0 < K) v[pass].x = p[0];
        if (k + 1 < K) v[pass].y = p[1];
        if (k + 2 < K) v[pass].z = p[2];
        if (k + 3 < K) v[pass].w = p[3];
      }
    }
  }
}
// splits the fetched values into NP bf16 planes and writes them into the K-major SW128 stage (16 KB per plane)
template <int NP, int NT>
__device__ __forceinline__ void store_a(const float4 (&v)[BM * 16 / NT], uint8_t* sa, int tid) {
  const int c = tid & 15;
  const int rsub = tid >> 4;
#pragma unroll
  for (int pass = 0; pass < BM * 16 / NT; ++pass) {
    const float x[4] = {v[pass].x, v[pass].y, v[pass].z, v[pass].w};
    uint2 pl[NP];
    split4<NP>(x, pl);
    const uint32_t off = sw128((uint32_t)(pass * (NT / 16) + rsub), (uint32_t)(c * 4));
#pragma unroll
    for (int p = 0; p < NP; ++p) *reinterpret_cast<uint2*>(sa + p * A_HALF_BYTES + off) = pl[p];
  }
}
// Stage a [128 x 64] slice of row-major fp32 A (K contiguous) as NP bf16 planes.  All global loads of a thread are issued
// before the first conversion so that the whole 32 KB slice is in flight.
template <int NP, int NT>
__device__ __forceinline__ void stage_a_direct(const float* __restrict__ A, int64_t lda, int64_t m0, int64_t M, int k0, int K,
                                               uint8_t* sa, int tid, bool vec_ok) {
  float4 v[BM * 16 / NT];
  fetch_a<NT>(A, lda, m0, M, k0, K, tid, vec_ok, v);
  store_a<NP, NT>(v, sa, tid);
}

// One warp stages a [32 rows x 64 k] block of the K-major tile  T(r, k) = X[(k0 + k) * ld + m0 + r]  as 2 bf16 planes
// (on-the-fly transpose; the contraction index k runs over points).  Lane l owns the m-quad (l & 7) and, in iteration q,
// the k pair 4q + (l >> 3): every warp-level load covers 4 rows of X x 128 contiguous bytes (4 L1 wavefronts instead of
// the 32 of a lane-per-row mapping); all 16 loads of a lane are issued before the first conversion.
template <bool CSUM = false>
__device__ __forceinline__ void stage_block_t(const float* __restrict__ X, int64_t ld, int m0, int m_total, int r0, int rows,
                                              int64_t k0, int64_t k_end, uint8_t* s_hi, uint8_t* s_lo, int lane, bool vec_ok,
                                              float* csum = nullptr, bool t128 = false) {
  const int mq = lane & 7, kq = lane >> 3;
  if (r0 + 4 * mq >= rows) return;      // tile rows are padded to 16, blocks cover 32: skip quads beyond the tile
  const int m = m0 + r0 + 4 * mq;
  float4 v[8][2];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
      const int64_t k = k0 + 2 * (4 * q + kq) + kk;
      v[q][kk] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k < k_end) {
        const float* p = X + (t128 ? t128_off(k, m, ld) : k * ld + m);       // T128 (common.cuh): 4 features of a point stay contiguous
        if (vec_ok && m + 3 < m_total) {
          v[q][kk] = *reinterpret_cast<const float4*>(p);
        } else {
          if (m + 0 < m_total) v[q][kk].x = p[0];
          if (m + 1 < m_total) v[q][kk].y = p[1];
          if (m + 2 < m_total) v[q][kk].z = p[2];
          if (m + 3 < m_total) v[q][kk].w = p[3];
        }
      }
    }
  }
  if (CSUM) {                             // per-lane partial column sums of X (bias gradients), fp32
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      csum[0] += v[q][0].x + v[q][1].x; csum[1] += v[q][0].y + v[q][1].y;
      csum[2] += v[q][0].z + v[q][1].z; csum[3] += v[q][0].w + v[q][1].w;
    }
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float x0[4] = {v[q][0].x, v[q][0].y, v[q][0].z, v[q][0].w};
    const float x1[4] = {v[q][1].x, v[q][1].y, v[q][1].z, v[q][1].w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float h0 = __bfloat162float(__float2bfloat16_rn(x0[j])), h1 = __bfloat162float(__float2bfloat16_rn(x1[j]));
      const uint32_t off = sw128((uint32_t)(r0 + 4 * mq + j), (uint32_t)(2 * (4 * q + kq)));
      *reinterpret_cast<uint32_t*>(s_hi + off) = pack_bf16(h0, h1);
      *reinterpret_cast<uint32_t*>(s_lo + off) = pack_bf16(x0[j] - h0, x1[j] - h1);
    }
  }
}

struct SmemCtl {
  uint64_t full[STAGES];
  uint64_t empty[STAGES];
  uint64_t tmem_full;
  uint32_t tmem_addr;
};

__device__ __forceinline__ uint32_t tmem_cols_for(int n) { return n <= 32 ? 32u : (n <= 64 ? 64u : (n <= 128 ? 128u : 256u)); }

// Issue the MMA group of one 64-wide K slice: all plane products whose weight is >= 2^-16 (2 planes: 3 products,
// 3 planes: 6 products), smallest terms first.  a/b: shared addresses of plane 0; plane p is at +p*stride.
template <int NP>
__device__ __forceinline__ void issue_slice(uint32_t tmem_d, uint32_t a, uint32_t a_stride, uint32_t b, uint32_t b_stride, uint32_t idesc,
                                            bool first_slice) {
#pragma unroll
  for (int j = 0; j < BK / 16; ++j) {
    uint64_t da[NP], db[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) { da[p] = make_desc(a + p * a_stride + j * 32); db[p] = make_desc(b + p * b_stride + j * 32); }
    const uint32_t acc0 = (first_slice && j == 0) ? 0u : 1u;
    if (NP == 2) {
      mma_bf16(tmem_d, da[1], db[0], idesc, acc0);
      mma_bf16(tmem_d, da[0], db[1], idesc, 1u);
      mma_bf16(tmem_d, da[0], db[0], idesc, 1u);
    } else {
      mma_bf16(tmem_d, da[NP - 1], db[0], idesc, acc0);        // lo * hi
      mma_bf16(tmem_d, da[0], db[NP - 1], idesc, 1u);          // hi * lo
      mma_bf16(tmem_d, da[1], db[1], idesc, 1u);               // mid * mid
      mma_bf16(tmem_d, da[1], db[0], idesc, 1u);               // mid * hi
      mma_bf16(tmem_d, da[0], db[1], idesc, 1u);               // hi * mid
      mma_bf16(tmem_d, da[0], db[0], idesc, 1u);               // hi * hi
    }
  }
}

// Epilogue of warp w (0..7): TMEM lane quadrant w & 3 (tile rows 32 (w&3) .. +31), 32-column chunks (w >> 2), (w >> 2)+2, ...
// tcgen05.ld hands every lane one ROW (32 consecutive columns); the 32x32 block is transposed through a warp-private,
// padded shared-memory tile so that each epilogue call covers 4 rows x 32 consecutive columns per warp instruction:
// the fused epilogues' global loads / stores (activations, saved tensors, outputs) are then fully coalesced float4.
constexpr int EPI_LD = 36;                       // floats per staged row (32 + 4 pad: conflict-free STS.128 / LDS.128)
constexpr int EPI_WARP_FLOATS = 16 * EPI_LD;     // the 32x32 block goes through the staging tile in two 16-row passes
#ifndef NUDF_EPI_DEEP
#define NUDF_EPI_DEEP 1
#endif
struct NoWait {
  __device__ __forceinline__ void operator()() const {}
};
// Software pipeline: the auxiliary global loads of pass p+1 (16 rows x 32 columns per warp) are issued before pass p is
// computed and stored, and those of the very first pass before `wait()` (the accumulator-ready barrier) returns, so that
// two passes' worth of loads are in flight per warp -- the epilogues are bound by memory-level parallelism, not by math.
// G = row groups (of 4 rows x 32 columns per warp instruction) whose auxiliary loads are in flight together: 4 with 8
// epilogue warps; 2 for the 16-warp plane-fed kernel, whose threads have 112 registers (same bytes in flight per SM).
template <class Epi, class Wait = NoWait, int G = 4>
__device__ __forceinline__ void run_epilogue(uint32_t tmem_acc, int quad, int lane, int chunk0, int chunk_step, int n_acc,
                                             uint32_t acc_stride, int64_t row0, int64_t M, int col_base, int n_pad, int n_valid_end,
                                             float* stg, const Epi& epi, int rot = 0, Wait wait = Wait()) {
  const int cq = lane & 7, rsub = lane >> 3;
  if constexpr (G != 4) {
    const int n_it2 = n_pad > chunk0 ? (n_pad - chunk0 + chunk_step - 1) / chunk_step : 0;
    wait();
    for (int it = 0; it < n_it2; ++it) {
      const int c0 = chunk0 + ((it + rot) % n_it2) * chunk_step;
      const int col = col_base + c0 + 4 * cq;
      int nv = n_valid_end - col;
      nv = nv < 4 ? nv : 4;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        {
          // the accumulator block is re-read from TMEM for each 16-row pass (cheap) so that its 32 values are not live
          // across the functor's loads and stores: this path runs with 112 registers per thread
          float v[32];
          tmem_ld32(tmem_acc + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, v);
          if ((lane >> 4) == h) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              *reinterpret_cast<float4*>(stg + (lane & 15) * EPI_LD + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          }
        }
        __syncwarp();
#pragma unroll
        for (int sub = 0; sub < 4 / G; ++sub) {
          typename Epi::Aux aux[G];
#pragma unroll
          for (int i = 0; i < G; ++i) {
            const int64_t row = row0 + 16 * h + rsub + 4 * (sub * G + i);
            if (row < M && nv > 0) epi.load(row, col, nv, aux[i]);
          }
#pragma unroll
          for (int i = 0; i < G; ++i) {
            const int r = rsub + 4 * (sub * G + i);
            const float4 t = *reinterpret_cast<const float4*>(stg + r * EPI_LD + 4 * cq);
            const int64_t row = row0 + 16 * h + r;
            if (row < M && nv > 0) {
              const float x[4] = {t.x, t.y, t.z, t.w};
              epi.apply(row, col, x, nv, aux[i]);
            }
          }
        }
        __syncwarp();
      }
    }
    return;
  }
  // rot: start the column chunks at a CTA-dependent position (split-K CTAs would otherwise all reduce into the same
  // addresses at the same time)
  const int n_it = n_pad > chunk0 ? (n_pad - chunk0 + chunk_step - 1) / chunk_step : 0;
  auto chunk_col = [&](int it) { return chunk0 + ((it + rot) % n_it) * chunk_step; };
  auto load_pass = [&](int it, int h, typename Epi::Aux (&aux)[4]) {
    const int col = col_base + chunk_col(it) + 4 * cq;
    int nv = n_valid_end - col;
    nv = nv < 4 ? nv : 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int64_t row = row0 + 16 * h + rsub + 4 * i;
      if (row < M && nv > 0) epi.load(row, col, nv, aux[i]);
    }
  };
  auto do_pass = [&](int it, int h, const float (&v)[32], const typename Epi::Aux (&aux)[4]) {
    const int col = col_base + chunk_col(it) + 4 * cq;
    int nv = n_valid_end - col;
    nv = nv < 4 ? nv : 4;
    if ((lane >> 4) == h) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<float4*>(stg + (lane & 15) * EPI_LD + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = rsub + 4 * i;
      const float4 t = *reinterpret_cast<const float4*>(stg + r * EPI_LD + 4 * cq);
      const int64_t row = row0 + 16 * h + r;
      if (row < M && nv > 0) {
        const float x[4] = {t.x, t.y, t.z, t.w};
        epi.apply(row, col, x, nv, aux[i]);
      }
    }
    __syncwarp();
  };
  // Functors with 8 auxiliary floats per group (EpiTan, EpiBwd) do not fit two sets next to the 32 accumulator values in
  // the 128-register budget of the epilogue warps: they keep one set and load just in time (kDeepPipe = false).
  constexpr bool kDeep = NUDF_EPI_DEEP && sizeof(typename Epi::Aux) <= 4 * sizeof(float);
  typename Epi::Aux a0[4], a1[kDeep ? 4 : 1];
  if (n_it > 0) load_pass(0, 0, a0);
  wait();
  for (int it = 0; it < n_it; ++it) {
    const int c0 = chunk_col(it);
    if constexpr (kDeep) load_pass(it, 1, a1);
    float v[32];
    tmem_ld32(tmem_acc + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, v);
    for (int a = 1; a < n_acc; ++a) {          // per-slice partial accumulators are summed here with round-to-nearest adds
      float w[32];
      tmem_ld32(tmem_acc + a * acc_stride + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, w);
#pragma unroll
      for (int q = 0; q < 32; ++q) v[q] += w[q];
    }
    do_pass(it, 0, v, a0);
    if constexpr (kDeep) {
      if (it + 1 < n_it) load_pass(it + 1, 0, a0);
      do_pass(it, 1, v, a1);
    } else {
      load_pass(it, 1, a0);
      do_pass(it, 1, v, a0);
      if (it + 1 < n_it) load_pass(it + 1, 0, a0);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// C[M x N] = epi( A[M x K] * B^T ),  B given as a pre-split NP-plane weight image.  grid = (ceil(M/128), n_tiles(N)).
// ---------------------------------------------------------------------------------------------------------------
template <int NP, class Epi>
__global__ void __launch_bounds__(THREADS, 1)
gemm_w_kernel(const float* __restrict__ A, int64_t lda, int64_t M, int N, int K, const uint16_t* __restrict__ img, Epi epi) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int t = blockIdx.y;
  const int rows_b = tile_rows(N, t, NP);                   // padded N of this tile (multiple of 16)
  const int n_slices = pad64(K) / 64;
  const uint32_t b_half_bytes = (uint32_t)rows_b * 128u;
  const uint32_t stage_bytes = NP * (uint32_t)A_HALF_BYTES + NP * b_half_bytes;
  SmemCtl* ctl = reinterpret_cast<SmemCtl*>(smem + STAGES * stage_bytes);
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const uint16_t* img_t = img + tile_offset(N, K, t, NP);

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&ctl->full[s], NPROD + 1); mbar_init(&ctl->empty[s], 1); }
    mbar_init(&ctl->tmem_full, 1);
    fence_barrier_init();
  }
  // 3-plane (fp32-grade) variant: every K slice accumulates into its own TMEM accumulator (up to 4 x 128 columns) and the
  // epilogue adds them in fp32 with round-to-nearest: the tensor core truncates its fp32 accumulator after every MMA
  // (measured bias ~ -1e-7 per step), so short accumulation chains keep the systematic error at the FFMA level.
  const int n_acc = (NP == 3) ? (n_slices < 4 ? n_slices : 4) : 1;
  const uint32_t acc_cols = tmem_cols_for(rows_b);
  const uint32_t alloc_cols = (n_acc == 1) ? acc_cols : (n_acc == 2 ? 2 * acc_cols : 512u);
  if (warp == 8) tmem_alloc(&ctl->tmem_addr, alloc_cols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = ctl->tmem_addr;

  if (warp < 8) {
    const bool vec_ok = ((lda & 3) == 0) && aligned16(A);
    for (int ks = 0; ks < n_slices; ++ks) {
      const int s = ks & 1, u = ks >> 1;
      if (u > 0) mbar_wait(&ctl->empty[s], (uint32_t)((u - 1) & 1));
      stage_a_direct<NP, NPROD>(A, lda, m0, M, ks * BK, K, smem + s * stage_bytes, tid, vec_ok);
      fence_proxy_async();
      mbar_arrive(&ctl->full[s]);
    }
    // epilogue
    mbar_wait(&ctl->tmem_full, 0);
    tcgen05_fence_after();
    run_epilogue(tmem_base, warp & 3, lane, 32 * (warp >> 2), 64, n_acc, acc_cols, m0 + (warp & 3) * 32, M, t * nt_of(NP), rows_b, N,
                 reinterpret_cast<float*>(smem) + warp * EPI_WARP_FLOATS, epi);   // operand stages are free by now
    tcgen05_fence_before();
  } else if (warp == 8) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc((uint32_t)rows_b);
      for (int ks = 0; ks < n_slices; ++ks) {
        const int s = ks & 1, u = ks >> 1;
        mbar_wait(&ctl->full[s], (uint32_t)(u & 1));
        tcgen05_fence_after();
        const uint32_t st = smem_u32(smem + s * stage_bytes);
        issue_slice<NP>(tmem_base + (uint32_t)(ks % n_acc) * acc_cols, st, A_HALF_BYTES, st + NP * A_HALF_BYTES, b_half_bytes, idesc,
                        ks < n_acc);
        mma_commit(&ctl->empty[s]);
      }
      mma_commit(&ctl->tmem_full);
    }
    __syncwarp();
  } else {
    if (lane == 0) {
      for (int ks = 0; ks < n_slices; ++ks) {
        const int s = ks & 1, u = ks >> 1;
        if (u > 0) mbar_wait(&ctl->empty[s], (uint32_t)((u - 1) & 1));
        uint8_t* st = smem + s * stage_bytes + NP * A_HALF_BYTES;
        mbar_arrive_expect_tx(&ctl->full[s], NP * b_half_bytes);
        bulk_g2s(st, img_t + (int64_t)ks * NP * rows_b * 64, NP * b_half_bytes, &ctl->full[s]);
      }
    }
    __syncwarp();
  }
  __syncthreads();
  if (warp == 8) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, alloc_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Persistent 2-plane variant of gemm_w: one CTA per SM loops over 128-row tiles; the TMEM accumulator is double
// buffered so that the epilogue of tile i (warps 4-7) overlaps the operand staging + MMAs of tile i+1 (warps 0-3, 8, 9).
// ---------------------------------------------------------------------------------------------------------------
// profiling aid (NUDF_TC_DEBUG & 16): CTA 0 records clock64() at pipeline events
__device__ long long g_tc_trace[4][256];
#define TC_TRACE(role, idx) do { if ((dbg & 16) && blockIdx.x == 0 && blockIdx.y == 0 && (idx) < 256) g_tc_trace[role][idx] = clock64(); } while (0)

struct SmemCtlP {
  uint64_t full[STAGES];
  uint64_t empty[STAGES];
  uint64_t tfull[2];
  uint64_t tempty[2];
  uint32_t tmem_addr;
};
// Persistent kernels: 14 warps.  Measured on B200 with one CTA per SM (tools/ubench/membw.cu): the LSU path sustains
// 2.3 TB/s with 4 loading warps, 3.9 TB/s with 8, 5.9 TB/s with 16 -- it scales with the number of warps, not with the
// number of loads per thread -- so the activation operand is fetched by 8 warps.
constexpr int PPROD = 256;      // producer threads (warps 0-7)
constexpr int PTHREADS = 448;   // + warps 8-11 epilogue, warp 12 MMA issuer / TMEM owner, warp 13 weight loader

template <class Epi>
__global__ void __launch_bounds__(PTHREADS, 1)
gemm_wp_kernel(const float* __restrict__ A, int64_t lda, int64_t M, int N, int K, const uint16_t* __restrict__ img, Epi epi,
               int reverse, int dbg) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int t = blockIdx.y;
  const int rows_b = tile_rows(N, t, 2);
  const int n_slices = pad64(K) / 64;
  const uint32_t b_half_bytes = (uint32_t)rows_b * 128u;
  const uint32_t stage_bytes = 2u * A_HALF_BYTES + 2u * b_half_bytes;
  float* epi_stage = reinterpret_cast<float*>(smem + STAGES * stage_bytes);
  SmemCtlP* ctl = reinterpret_cast<SmemCtlP*>(smem + STAGES * stage_bytes + 4 * EPI_WARP_FLOATS * sizeof(float));
  const uint16_t* img_t = img + tile_offset(N, K, t, 2);
  const int64_t n_mtiles = (M + BM - 1) / BM;
  const uint32_t acc_cols = tmem_cols_for(rows_b);

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&ctl->full[s], PPROD + 1); mbar_init(&ctl->empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&ctl->tfull[a], 1); mbar_init(&ctl->tempty[a], 128); }
    fence_barrier_init();
  }
  if (warp == 12) tmem_alloc(&ctl->tmem_addr, 2 * acc_cols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = ctl->tmem_addr;
  if (tid == 0) TC_TRACE(3, 0);

  if (warp < 8) {
    // ---- A producers ----
    const bool vec_ok = ((lda & 3) == 0) && aligned16(A);
    uint32_t cnt = 0;
    for (int64_t it = blockIdx.x; it < n_mtiles; it += gridDim.x) {
      const int64_t mt = reverse ? n_mtiles - 1 - it : it;
      for (int ks = 0; ks < n_slices; ks += 2) {
        // two K slices (64 KB of fp32) are fetched before the first conversion: twice the bytes in flight per SM
        const bool two = ks + 1 < n_slices;
        float4 v0[BM * 16 / PPROD], v1[BM * 16 / PPROD];
        if (!(dbg & 1)) {
          fetch_a<PPROD>(A, lda, mt * BM, M, ks * BK, K, tid, vec_ok, v0);
          if (two) fetch_a<PPROD>(A, lda, mt * BM, M, (ks + 1) * BK, K, tid, vec_ok, v1);
        } else {
#pragma unroll
          for (int q = 0; q < BM * 16 / PPROD; ++q) { v0[q] = make_float4(1.f, 0.f, 0.f, 0.f); v1[q] = v0[q]; }
        }
        {
          const uint32_t s = cnt & 1u, u = cnt >> 1;
          if (tid == 0) TC_TRACE(0, 4 * cnt + 0);
          if (u > 0) mbar_wait(&ctl->empty[s], (u - 1) & 1u);
          if (tid == 0) TC_TRACE(0, 4 * cnt + 1);
          store_a<2, PPROD>(v0, smem + s * stage_bytes, tid);
          if (tid == 0) TC_TRACE(0, 4 * cnt + 2);
          fence_proxy_async();
          mbar_arrive(&ctl->full[s]);
          if (tid == 0) TC_TRACE(0, 4 * cnt + 3);
          ++cnt;
        }
        if (two) {
          const uint32_t s = cnt & 1u, u = cnt >> 1;
          if (u > 0) mbar_wait(&ctl->empty[s], (u - 1) & 1u);
          store_a<2, PPROD>(v1, smem + s * stage_bytes, tid);
          fence_proxy_async();
          mbar_arrive(&ctl->full[s]);
          ++cnt;
        }
      }
    }
  } else if (warp < 12) {
    // ---- epilogue ----
    uint32_t it = 0;
    for (int64_t jt = blockIdx.x; jt < n_mtiles; jt += gridDim.x, ++it) {
      const int64_t mt = reverse ? n_mtiles - 1 - jt : jt;
      const uint32_t a = it & 1u, au = it >> 1;
      if (tid == 256) TC_TRACE(2, 3 * it + 0);
      mbar_wait(&ctl->tfull[a], au & 1u);
      if (tid == 256) TC_TRACE(2, 3 * it + 1);
      tcgen05_fence_after();
      if (!(dbg & 2))
        run_epilogue(tmem_base + a * acc_cols, warp & 3, lane, 0, 32, 1, 0u, mt * BM + (warp & 3) * 32, M, t * 256, rows_b, N,
                     epi_stage + (warp & 3) * EPI_WARP_FLOATS, epi);
      tcgen05_fence_before();
      mbar_arrive(&ctl->tempty[a]);
      if (tid == 256) TC_TRACE(2, 3 * it + 2);
    }
  } else if (warp == 12) {
    // ---- MMA issuer ----
    if (lane == 0) {
      const uint32_t idesc = make_idesc((uint32_t)rows_b);
      uint32_t cnt = 0, it = 0;
      for (int64_t mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x, ++it) {
        const uint32_t a = it & 1u, au = it >> 1;
        if (au > 0) mbar_wait(&ctl->tempty[a], (au - 1) & 1u);
        tcgen05_fence_after();
        for (int ks = 0; ks < n_slices; ++ks, ++cnt) {
          const uint32_t s = cnt & 1u, u = cnt >> 1;
          TC_TRACE(1, 3 * cnt + 0);
          mbar_wait(&ctl->full[s], u & 1u);
          TC_TRACE(1, 3 * cnt + 1);
          tcgen05_fence_after();
          const uint32_t st = smem_u32(smem + s * stage_bytes);
          if (!(dbg & 8)) issue_slice<2>(tmem_base + a * acc_cols, st, A_HALF_BYTES, st + 2 * A_HALF_BYTES, b_half_bytes, idesc, ks == 0);
          mma_commit(&ctl->empty[s]);
          TC_TRACE(1, 3 * cnt + 2);
        }
        mma_commit(&ctl->tfull[a]);
      }
    }
    __syncwarp();
  } else {
    // ---- weight loader ----
    if (lane == 0) {
      uint32_t cnt = 0;
      for (int64_t mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x) {
        for (int ks = 0; ks < n_slices; ++ks, ++cnt) {
          const uint32_t s = cnt & 1u, u = cnt >> 1;
          if (u > 0) mbar_wait(&ctl->empty[s], (u - 1) & 1u);
          uint8_t* st = smem + s * stage_bytes + 2 * A_HALF_BYTES;
          if (dbg & 4) { mbar_arrive(&ctl->full[s]); continue; }
          mbar_arrive_expect_tx(&ctl->full[s], 2u * b_half_bytes);
          bulk_g2s(st, img_t + (int64_t)ks * 2 * rows_b * 64, 2u * b_half_bytes, &ctl->full[s]);
        }
      }
    }
    __syncwarp();
  }
  __syncthreads();
  if (tid == 0) TC_TRACE(3, 1);
  if (warp == 12) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 2 * acc_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Weights-resident persistent variant (K <= 256): each CTA owns one 128-column half of the output and keeps that half
// of the pre-split weight image (all K slices, <= 128 KB) in shared memory for its whole lifetime -- it is fetched once
// with a handful of 16 KB cp.async.bulk copies.  Only the activation slices stream through the 2-stage ring; the TMEM
// accumulator (128 columns) is double buffered so the epilogue of tile i overlaps the main loop of tile i+1.
// (Streaming the weight slices per tile -- gemm_wp_kernel -- turned out to be limited by the bulk-copy engine: one
// 64 KB copy per K slice per CTA took 6-10 us on B200, see profiles/.)
// ---------------------------------------------------------------------------------------------------------------
struct SmemCtlR {
  uint64_t full[STAGES];
  uint64_t empty[STAGES];
  uint64_t tfull[2];
  uint64_t tempty[2];
  uint64_t wfull;
  uint32_t tmem_addr;
};
constexpr int WR_N = 128;        // output columns per CTA
constexpr int WR_MAX_SLICES = 4; // K <= 256
// Warp-specialised layout of the weights-resident kernel: 20 warps = 5 warpgroups.  LSU streaming rate of a
// single CTA per SM scales with its number of loading warps (tools/ubench/membw.cu: 4 warps 2.3 TB/s, 8 warps 3.9 TB/s), so both the operand fetch and
// the epilogue (whose fused functors load 1-2 and store 1-2 tensors) get 8 warps each; registers are re-balanced with
// setmaxnreg (epilogue 128, MMA / loader warpgroup 32).  setmaxnreg.inc draws from the CTA pool, i.e. only from what the
// MMA / loader warpgroup released with setmaxnreg.dec: (96 - 32) x 128 threads = 8192 registers = +32 for the 256 epilogue
// threads.  Asking for more (136, 144) spins forever in USETMAXREG.TRY_ALLOC.
constexpr int RW_THREADS = 640;
constexpr int RW_PROD = 256;     // warps 0-7   (warpgroups 0-1)
constexpr int RW_EPI = 256;      // warps 8-15  (warpgroups 2-3): quadrant = warp & 3, column half = (warp >> 2) & 1
constexpr int RW_MMA_WARP = 16, RW_LOAD_WARP = 17;   // warpgroup 4 (warps 18, 19 idle)

template <class Epi>
__global__ void __launch_bounds__(RW_THREADS, 1)
gemm_wr_kernel(const float* __restrict__ A, int64_t lda, int64_t M, int N, int K, const uint16_t* __restrict__ img, Epi epi,
               int reverse) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n0 = blockIdx.y * WR_N;                          // first output column of this CTA
  const int t = n0 / 256;                                    // 256-row tile of the 2-plane image this half lives in
  const int rows_t = tile_rows(N, t, 2);                     // rows of that image tile (multiple of 16)
  const int row_in_tile = n0 - t * 256;                      // 0 or 128
  int rows_h = rows_t - row_in_tile; rows_h = rows_h < WR_N ? rows_h : WR_N;   // padded N of this CTA (multiple of 16)
  const int n_slices = pad64(K) / 64;
  const uint32_t w_plane_bytes = (uint32_t)rows_h * 128u;    // one plane of one slice of this half
  uint8_t* w_smem = smem;                                    // [slice][plane][rows_h x 128 B]
  uint8_t* a_smem = smem + (size_t)n_slices * 2 * w_plane_bytes;             // 2 stages x (2 planes x 16 KB)
  float* epi_stage = reinterpret_cast<float*>(a_smem + STAGES * 2 * A_HALF_BYTES);
  SmemCtlR* ctl = reinterpret_cast<SmemCtlR*>(reinterpret_cast<uint8_t*>(epi_stage) + 8 * EPI_WARP_FLOATS * sizeof(float));
  const uint16_t* img_t = img + tile_offset(N, K, t, 2);
  const int64_t n_mtiles = (M + BM - 1) / BM;
  const uint32_t acc_cols = tmem_cols_for(rows_h);

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&ctl->full[s], RW_PROD); mbar_init(&ctl->empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&ctl->tfull[a], 1); mbar_init(&ctl->tempty[a], RW_EPI); }
    mbar_init(&ctl->wfull, 1);
    fence_barrier_init();
  }
  if (warp == RW_MMA_WARP) tmem_alloc(&ctl->tmem_addr, 2 * acc_cols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = ctl->tmem_addr;

  if (warp < 8) {
    // ---- A producers (warpgroups 0-1): two K slices (64 KB) are fetched before the first conversion ----
    const bool vec_ok = ((lda & 3) == 0) && aligned16(A);
    uint32_t cnt = 0;
    for (int64_t it = blockIdx.x; it < n_mtiles; it += gridDim.x) {
      const int64_t mt = reverse ? n_mtiles - 1 - it : it;
      for (int ks = 0; ks < n_slices; ks += 2) {
        const bool two = ks + 1 < n_slices;
        float4 v0[BM * 16 / RW_PROD], v1[BM * 16 / RW_PROD];
        fetch_a<RW_PROD>(A, lda, mt * BM, M, ks * BK, K, tid, vec_ok, v0);
        if (two) fetch_a<RW_PROD>(A, lda, mt * BM, M, (ks + 1) * BK, K, tid, vec_ok, v1);
        {
          const uint32_t s = cnt & 1u, u = cnt >> 1;
          if (u > 0) mbar_wait(&ctl->empty[s], (u - 1) & 1u);
          store_a<2, RW_PROD>(v0, a_smem + s * 2 * A_HALF_BYTES, tid);
          fence_proxy_async();
          mbar_arrive(&ctl->full[s]);
          ++cnt;
        }
        if (two) {
          const uint32_t s = cnt & 1u, u = cnt >> 1;
          if (u > 0) mbar_wait(&ctl->empty[s], (u - 1) & 1u);
          store_a<2, RW_PROD>(v1, a_smem + s * 2 * A_HALF_BYTES, tid);
          fence_proxy_async();
          mbar_arrive(&ctl->full[s]);
          ++cnt;
        }
      }
    }
  } else if (warp < 16) {
    // ---- epilogue (warpgroups 2-3) ----
    asm volatile("setmaxnreg.inc.sync.aligned.u32 128;");
    const int ew = warp - 8;
    uint32_t it = 0;
    for (int64_t jt = blockIdx.x; jt < n_mtiles; jt += gridDim.x, ++it) {
      const int64_t mt = reverse ? n_mtiles - 1 - jt : jt;
      const uint32_t a = it & 1u, au = it >> 1;
      auto acc_ready = [&]() { mbar_wait(&ctl->tfull[a], au & 1u); tcgen05_fence_after(); };
      run_epilogue(tmem_base + a * acc_cols, ew & 3, lane, 32 * (ew >> 2), 64, 1, 0u, mt * BM + (ew & 3) * 32, M, n0, rows_h, N,
                   epi_stage + ew * EPI_WARP_FLOATS, epi, 0, acc_ready);
      tcgen05_fence_before();
      mbar_arrive(&ctl->tempty[a]);
    }
  } else {
    // ---- warpgroup 4: MMA issuer (warp 16), weight loader (warp 17) ----
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (warp == RW_MMA_WARP) {
      if (lane == 0) {
        const uint32_t idesc = make_idesc((uint32_t)rows_h);
        const uint32_t w_addr = smem_u32(w_smem);
        mbar_wait(&ctl->wfull, 0);
        uint32_t cnt = 0, it = 0;
        for (int64_t mt = blockIdx.x; mt < n_mtiles; mt += gridDim.x, ++it) {
          const uint32_t a = it & 1u, au = it >> 1;
          if (au > 0) mbar_wait(&ctl->tempty[a], (au - 1) & 1u);
          tcgen05_fence_after();
          for (int ks = 0; ks < n_slices; ++ks, ++cnt) {
            const uint32_t s = cnt & 1u, u = cnt >> 1;
            mbar_wait(&ctl->full[s], u & 1u);
            tcgen05_fence_after();
            const uint32_t st = smem_u32(a_smem + s * 2 * A_HALF_BYTES);
            issue_slice<2>(tmem_base + a * acc_cols, st, A_HALF_BYTES, w_addr + (uint32_t)ks * 2u * w_plane_bytes, w_plane_bytes, idesc,
                           ks == 0);
            mma_commit(&ctl->empty[s]);
          }
          mma_commit(&ctl->tfull[a]);
        }
      }
      __syncwarp();
    } else if (warp == RW_LOAD_WARP) {
      // weight half: fetched once per CTA; lane l < 2*n_slices copies (slice l/2, plane l%2), 16 KB each
      if (lane == 0) mbar_arrive_expect_tx(&ctl->wfull, (uint32_t)n_slices * 2u * w_plane_bytes);
      __syncwarp();
      if (lane < 2 * n_slices) {
        const int ks = lane >> 1, pl = lane & 1;
        const uint16_t* src = img_t + (int64_t)ks * 2 * rows_t * 64 + (int64_t)pl * rows_t * 64 + (int64_t)row_in_tile * 64;
        bulk_g2s(w_smem + (size_t)(ks * 2 + pl) * w_plane_bytes, src, w_plane_bytes, &ctl->wfull);
      }
      __syncwarp();
    }
  }
  __syncthreads();
  if (warp == RW_MMA_WARP) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 2 * acc_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// C[M x N] += A[K x M]^T B[K x N]  (weight gradients; contraction over points, split over gridDim.z).
// grid = (ceil(M/128), ceil(N/256), splits).  Epi is applied to the partial tile (EpiSliceStore: slice blockIdx.z).
// ---------------------------------------------------------------------------------------------------------------
constexpr int TN_PROD = 384;      // 12 loading / epilogue warps: 4 stage the [128 x 64] A^T tile, 8 the [256 x 64] B^T tile
constexpr int TN_THREADS = 416;   // + warp 12: MMA issuer and TMEM owner
template <class Epi>
__global__ void __launch_bounds__(TN_THREADS, 1)
gemm_tn_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, int M, int N, int64_t K,
               int64_t k_chunk, Epi epi, float* __restrict__ colsum_a, int t128) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * BM;
  const int n0 = blockIdx.y * 256;
  int rows_b = N - n0; rows_b = pad16(rows_b < 256 ? rows_b : 256);
  const int64_t kb = (int64_t)blockIdx.z * k_chunk;
  const int64_t ke = (kb + k_chunk < K) ? kb + k_chunk : K;
  const int n_slices = (int)((ke - kb + BK - 1) / BK);
  const uint32_t b_half_bytes = (uint32_t)rows_b * 128u;
  const uint32_t stage_bytes = 2u * A_HALF_BYTES + 2u * b_half_bytes;
  SmemCtl* ctl = reinterpret_cast<SmemCtl*>(smem + STAGES * stage_bytes);

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&ctl->full[s], TN_PROD); mbar_init(&ctl->empty[s], 1); }
    mbar_init(&ctl->tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 12) tmem_alloc(&ctl->tmem_addr, tmem_cols_for(rows_b));
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = ctl->tmem_addr;

  if (warp < 12) {
    const bool a_vec = ((lda & 3) == 0) && aligned16(A) && ((m0 & 3) == 0);
    const bool b_vec = ((ldb & 3) == 0) && aligned16(B);
    // optional fused bias gradient: column sums of A (= sum over points of dZ), taken from the values the A stagers hold
    // anyway; only the CTAs of the first N tile contribute
    const bool do_csum = colsum_a != nullptr && blockIdx.y == 0;
    float csum[4] = {0.f, 0.f, 0.f, 0.f};
    for (int ks = 0; ks < n_slices; ++ks) {
      const int s = ks & 1, u = ks >> 1;
      if (u > 0) mbar_wait(&ctl->empty[s], (uint32_t)((u - 1) & 1));
      uint8_t* st = smem + s * stage_bytes;
      const int64_t k0 = kb + (int64_t)ks * BK;
      if (warp < 4) {
        if (do_csum) stage_block_t<true>(A, lda, m0, M, 32 * warp, BM, k0, ke, st, st + A_HALF_BYTES, lane, a_vec, csum, t128 != 0);
        else stage_block_t(A, lda, m0, M, 32 * warp, BM, k0, ke, st, st + A_HALF_BYTES, lane, a_vec, nullptr, t128 != 0);
      } else if (32 * (warp - 4) < rows_b) {
        stage_block_t(B, ldb, n0, N, 32 * (warp - 4), rows_b, k0, ke, st + 2 * A_HALF_BYTES, st + 2 * A_HALF_BYTES + b_half_bytes, lane, b_vec,
                      nullptr, t128 != 0);
      }
      fence_proxy_async();
      mbar_arrive(&ctl->full[s]);
    }
    if (do_csum && warp < 4) {            // lanes (mq, kq): reduce over the 4 kq lanes, then one atomic per column
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        csum[j] += __shfl_xor_sync(0xffffffffu, csum[j], 8);
        csum[j] += __shfl_xor_sync(0xffffffffu, csum[j], 16);
      }
      if ((lane >> 3) == 0) {
        const int m = m0 + 32 * warp + 4 * (lane & 7);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (m + j < M) atomicAdd(colsum_a + (int64_t)blockIdx.z * M + m + j, csum[j]);   // this split's slice
      }
    }
    if (n_slices > 0) {
      mbar_wait(&ctl->tmem_full, 0);
      tcgen05_fence_after();
      // warp w: TMEM quadrant w & 3, 32-column chunks (w >> 2), (w >> 2) + 3, ...
      run_epilogue(tmem_base, warp & 3, lane, 32 * (warp >> 2), 96, 1, 0u, (int64_t)m0 + (warp & 3) * 32, (int64_t)M, n0, rows_b, N,
                   reinterpret_cast<float*>(smem) + warp * EPI_WARP_FLOATS, epi, (int)blockIdx.z);
      tcgen05_fence_before();
    }
  } else {
    if (lane == 0 && n_slices > 0) {
      const uint32_t idesc = make_idesc((uint32_t)rows_b);
      for (int ks = 0; ks < n_slices; ++ks) {
        const int s = ks & 1, u = ks >> 1;
        mbar_wait(&ctl->full[s], (uint32_t)(u & 1));
        tcgen05_fence_after();
        const uint32_t st = smem_u32(smem + s * stage_bytes);
        issue_slice<2>(tmem_base, st, A_HALF_BYTES, st + 2 * A_HALF_BYTES, b_half_bytes, idesc, ks == 0);
        mma_commit(&ctl->empty[s]);
      }
      mma_commit(&ctl->tmem_full);
    }
    __syncwarp();
  }
  __syncthreads();
  if (warp == 12) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, tmem_cols_for(rows_b));
  }
}

inline size_t smem_bytes_for(int rows_b, int np) {
  return (size_t)STAGES * ((size_t)np * A_HALF_BYTES + (size_t)np * rows_b * 128) + sizeof(SmemCtl) + 1024 + 64;
}

int tc_debug();   // NUDF_TC_DEBUG bit mask (profiling aid): 1 skip A fetch, 2 skip epilogue, 4 skip weight copies, 8 skip MMAs

static inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

template <class Epi>
static inline int gemm_wp(const float* A, int64_t lda, int64_t M, int N, int K, const uint16_t* img, const Epi& epi, cudaStream_t st) {
  const size_t smem = (size_t)STAGES * (2 * A_HALF_BYTES + 2 * (size_t)tile_rows(N, 0, 2) * 128) + 4 * EPI_WARP_FLOATS * sizeof(float) +
                      sizeof(SmemCtlP) + 1024 + 64;
  static bool attr_set = false;
  if (!attr_set) {
    NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_wp_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const int64_t n_mtiles = cdiv(M, BM);
  const int nt = n_tiles(N, 2);
  int64_t gx = sm_count() / nt;
  if (gx < 1) gx = 1;
  if (gx > n_mtiles) gx = n_mtiles;
  dim3 grid((unsigned)gx, (unsigned)nt);
  // consecutive layers walk the row tiles in opposite directions: the rows the previous kernel wrote last are still in
  // the 126 MB L2 when the next kernel starts with them
  static int flip = 0;
  flip ^= 1;
  LaunchTimer lt_(epi_family<Epi>::value, st);
  gemm_wp_kernel<Epi><<<grid, PTHREADS, smem, st>>>(A, lda, M, N, K, img, epi, flip, tc_debug());
  NUDF_LAUNCH_OK();
  return 0;
}

template <class Epi>
static inline int gemm_wr(const float* A, int64_t lda, int64_t M, int N, int K, const uint16_t* img, const Epi& epi, cudaStream_t st) {
  const int n_slices = pad64(K) / 64;
  const size_t smem = (size_t)n_slices * 2 * WR_N * 128 + (size_t)STAGES * 2 * A_HALF_BYTES + 8 * EPI_WARP_FLOATS * sizeof(float) +
                      sizeof(SmemCtlR) + 1024 + 64;
  static bool attr_set = false;
  if (!attr_set) {
    NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_wr_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const int64_t n_mtiles = cdiv(M, BM);
  const int nh = (int)cdiv(pad16(N), WR_N);
  int64_t gx = sm_count() / nh;
  if (gx < 1) gx = 1;
  if (gx > n_mtiles) gx = n_mtiles;
  dim3 grid((unsigned)gx, (unsigned)nh);
  static int flip = 0;
  flip ^= 1;
  LaunchTimer lt_(epi_family<Epi>::value, st);
  gemm_wr_kernel<Epi><<<grid, RW_THREADS, smem, st>>>(A, lda, M, N, K, img, epi, flip);
  NUDF_LAUNCH_OK();
  return 0;
}

template <int NP, class Epi>
static inline int gemm_w(const float* A, int64_t lda, int64_t M, int N, int K, const uint16_t* img, const Epi& epi, cudaStream_t st) {
  if (M <= 0 || N <= 0) return 0;
  if (NP == 2 && M > BM && pad64(K) <= 64 * WR_MAX_SLICES && tc_debug() != 32) return gemm_wr(A, lda, M, N, K, img, epi, st);
  if (NP == 2 && M > BM) return gemm_wp(A, lda, M, N, K, img, epi, st);
  const size_t smem = smem_bytes_for(tile_rows(N, 0, NP), NP);
  static bool attr_set = false;   // per template instantiation
  if (!attr_set) {
    NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_w_kernel<NP, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  dim3 grid((unsigned)cdiv(M, BM), (unsigned)n_tiles(N, NP));
  LaunchTimer lt_(epi_family<Epi>::value, st);
  gemm_w_kernel<NP, Epi><<<grid, THREADS, smem, st>>>(A, lda, M, N, K, img, epi);
  NUDF_LAUNCH_OK();
  return 0;
}

template <class Epi>
static inline int gemm_tn(const float* A, int64_t lda, const float* B, int64_t ldb, int M, int N, int64_t K, const Epi& epi,
                          cudaStream_t st, int split_k, float* colsum_a = nullptr, bool t128 = false) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  int64_t k_chunk = round_up(cdiv(K, split_k < 1 ? 1 : split_k), BK);
  int splits = (int)cdiv(K, k_chunk);
  if constexpr (std::is_same<Epi, EpiAtomicAdd>::value) {     // fixed-order split-K: slices + sum_slices
    const int64_t ldw = round_up(N, 4), slice = (int64_t)M * ldw, cs = colsum_a ? (int64_t)splits * M : 0;
    float* ws = nullptr;
    int rc = slices_alloc(&ws, (size_t)(slice * splits + cs), st);
    if (rc != 0) return rc;
    float* wcs = colsum_a ? ws + slice * splits : nullptr;
    if (wcs != nullptr && cudaMemsetAsync(wcs, 0, (size_t)cs * sizeof(float), st) != cudaSuccess) rc = -2;
    if (rc == 0) rc = gemm_tn(A, lda, B, ldb, M, N, K, EpiSliceStore{ws, ldw, slice}, st, split_k, wcs, t128);
    if (rc == 0) {
      SliceJobs jobs{};
      jobs.slices = splits;
      jobs.j[jobs.n++] = SliceJob{ws, slice, ldw, M, N, epi.C, epi.ldc};
      if (wcs != nullptr) jobs.j[jobs.n++] = SliceJob{wcs, M, M, 1, M, colsum_a, M};
      rc = sum_slices(jobs, st);
    }
    const int rf = slices_free(ws, st);
    return rc != 0 ? rc : rf;
  } else if constexpr (!std::is_same<Epi, EpiSliceStore>::value) {
    NUDF_REQUIRE(colsum_a == nullptr, "column sums go with a split-K reduction");
  }
  const size_t smem = smem_bytes_for(pad16(N < 256 ? N : 256), 2);
  static bool attr_set = false;
  if (!attr_set) {
    NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_tn_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  dim3 grid((unsigned)cdiv(M, BM), (unsigned)cdiv(N, 256), (unsigned)splits);
  LaunchTimer lt_(FAM_TC_WGRAD, st);
  gemm_tn_kernel<Epi><<<grid, TN_THREADS, smem, st>>>(A, lda, B, ldb, M, N, K, k_chunk, epi, colsum_a, t128 ? 1 : 0);
  NUDF_LAUNCH_OK();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Weight gradients from T128 operands (the tensors the fused UDF chains exchange, common.cuh), second generation:
//     C[M x N] += sum over pairs p of  A_p[K x M]^T B_p[K x N]          (contraction over points, split over gridDim.z)
// * up to two operand pairs per launch: the two contributions to one dW_l (D_l^T Adot_l from the tangent chain and Q_l^T A_l
//   from the backward chain) share the TMEM accumulator and ONE split-K reduction;
// * fp32 operands travel global -> shared with per-lane cp.async (LDGSTS, 16 B, zero-fill for pad rows) into a warp-private
//   raw ring: the copies of slice i+1 are in flight while slice i is split to bf16 planes, no register staging;
// * a warp copy instruction covers 32 consecutive points x 4 features = 512 contiguous bytes of the T128 layout, every 32-byte
//   sector requested once; the point-pair packing reads the raw tile back across lanes;
// * K is sliced by 32 points: the two halves (k < 32, k >= 32) of the K-major SWIZZLE_128B plane tile are the two pipeline
//   stages, MMAs of one half overlap the split of the other.
// warps 0-3 stage A (32 tile rows each), 4-11 stage B, all 12 run the split-K epilogue; warp 12 issues MMAs / owns TMEM.
// ---------------------------------------------------------------------------------------------------------------
struct TnPair {
  const float* A; int64_t lda;
  const float* B; int64_t ldb;
  float* colsum_a;                 // optional: colsum_a[m] += sum_k A[k, m]  (bias gradient)
};
constexpr int T2_BK = 32;
constexpr int T2_RING = 5;                                   // raw ring depth in half-slice granules (4 granules = 2 slices in flight)
constexpr uint32_t T2_RAW_WARP = 32u * 64u;                  // 2 KB per granule: 4 x 16 B per lane
constexpr uint32_t T2_RAW_GRAN = 12u * T2_RAW_WARP;          // 24 KB
constexpr uint32_t T2_B_HALF = 256u * 128u;                  // fixed plane stride of the B tile (32 KB)
constexpr uint32_t T2_PLANES = 2u * A_HALF_BYTES + 2u * T2_B_HALF;   // 96 KB

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N_) : "memory"); }

// One granule = half a slice of one warp: 32 points x 16 of the warp's 32 columns = 4 feature quads.  Copy: lane l moves point
// k0 + l of each quad (16 B), so every warp instruction reads 512 contiguous bytes of the T128 layout -- each 32-byte sector
// is requested exactly once (cp.async.cg bypasses L1: a mapping that splits a sector over two instructions fetches it twice
// from L2).  Raw layout of a warp's granule: [quad][slot(point)][16 B] with slot(p) = p ^ ((p >> 3) & 1): both the copy (lane = point)
// and the split (lane = point pair, two 16-byte loads) are bank-conflict free per quarter warp.  `src` = address of (point k0 + lane, first column of quad 0 of this half), or null for a
// column block beyond ld; consecutive quads are 512 floats apart in the T128 layout.
__device__ __forceinline__ void t2_issue(const float* __restrict__ src, const float* __restrict__ any, int n_quads_valid, bool row_ok,
                                         uint32_t raw_warp, int lane) {
  const uint32_t dst = raw_warp + (uint32_t)(lane ^ ((lane >> 3) & 1)) * 16u;      // slot(point) = point ^ ((point >> 3) & 1)
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const bool v = row_ok && q < n_quads_valid;                  // invalid: zero fill, source address unused
    cp_async16(dst + (uint32_t)q * 512u, v ? src + q * 512 : any, v ? 16u : 0u);
  }
}
// Split: lane (rp = lane & 15, g2 = lane >> 4) packs the point pair (2 rp, 2 rp + 1) of the quads g2 and g2 + 2.
// pre[j]: byte offset of (tile row 4 g2 + j, k = 2 rp) inside an 8-row swizzle atom, without the k half (added by the caller).
template <bool CSUM, int HALF>
__device__ __forceinline__ void t2_convert(const uint8_t* raw_warp, uint8_t* s_hi, uint8_t* s_lo, const uint32_t (&pre)[4], int lane,
                                           float* csum) {
  const int rp = lane & 15, g2 = lane >> 4;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int q = 2 * i + g2;
    const int sw = (rp >> 2) & 1;                                // points 2 rp, 2 rp + 1 -> slots (2 rp) ^ sw, (2 rp + 1) ^ sw
    const float4 a = *reinterpret_cast<const float4*>(raw_warp + q * 512 + ((2 * rp) ^ sw) * 16);
    const float4 b = *reinterpret_cast<const float4*>(raw_warp + q * 512 + ((2 * rp + 1) ^ sw) * 16);
    const float x0[4] = {a.x, a.y, a.z, a.w}, x1[4] = {b.x, b.y, b.z, b.w};
    // tile rows r0 + 16 HALF + 4 q + j = 8-row atom (r0 / 8 + 2 HALF + i), row-in-atom 4 g2 + j: s_hi / s_lo already point at
    // the warp's first atom
    uint8_t* h = s_hi + (2 * HALF + i) * 1024;
    uint8_t* l = s_lo + (2 * HALF + i) * 1024;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t hi = pack_bf16(x0[j], x1[j]);
      const uint32_t lo = pack_bf16(x0[j] - __uint_as_float(hi << 16), x1[j] - __uint_as_float(hi & 0xFFFF0000u));
      *reinterpret_cast<uint32_t*>(h + pre[j]) = hi;
      *reinterpret_cast<uint32_t*>(l + pre[j]) = lo;
      if (CSUM) csum[8 * HALF + 4 * i + j] += x0[j] + x1[j];
    }
  }
}

// ---- row-major operands (colour / NeRF++ networks): a granule = 16 points x the warp's 32 columns -------------------------
// Copy: lane l moves the 16-byte column quad (l & 7) of point 4 i + (l >> 3), i = 0..3: every warp instruction reads four
// 128-byte row segments (whole sectors).  Raw layout [point][quad ^ (point >> 1)][16 B]: conflict-free for the copy (8 lanes =
// one point, 8 distinct quads) and for the split (8 lanes = 8 point pairs of one quad).
__device__ __forceinline__ void t2_issue_rm(const float* __restrict__ X, int64_t ld, int col0, int64_t k0, int64_t k_end, uint32_t raw_warp,
                                            int lane) {
  const int c = lane & 7;
  const bool col_ok = col0 + 4 * c < ld;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int pl = 4 * i + (lane >> 3);
    const int64_t row = k0 + pl;
    const bool v = col_ok && row < k_end;
    cp_async16(raw_warp + (uint32_t)pl * 128u + (uint32_t)((c ^ (pl >> 1)) & 7) * 16u, v ? X + row * ld + col0 + 4 * c : X, v ? 16u : 0u);
  }
}
// Split: lane (p = lane & 7, g = lane >> 3) packs the point pair (2 p, 2 p + 1) of the quads g and g + 4.
// pre[j]: swizzled byte offset of (row-in-atom 4 (g & 1) + j, k = 2 p) for k half 0 / granule 0; the k position of the granule
// only flips bits of the 16-byte chunk index: offset ^= (4 khalf + 2 gran) << 4.
template <bool CSUM>
__device__ __forceinline__ void t2_convert_rm(const uint8_t* raw_warp, uint8_t* w_hi, uint8_t* w_lo, const uint32_t (&pre)[4], uint32_t kflip,
                                              int lane, float* csum) {
  const int p = lane & 7, g = lane >> 3;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int q = g + 4 * i;
    const float4 a = *reinterpret_cast<const float4*>(raw_warp + (2 * p) * 128 + ((q ^ p) & 7) * 16);
    const float4 b = *reinterpret_cast<const float4*>(raw_warp + (2 * p + 1) * 128 + ((q ^ p) & 7) * 16);
    const float x0[4] = {a.x, a.y, a.z, a.w}, x1[4] = {b.x, b.y, b.z, b.w};
    // tile rows r0 + 4 q + j = atom (r0 / 8 + 2 i + (g >> 1)), row-in-atom 4 (g & 1) + j
    uint8_t* h = w_hi + (2 * i + (g >> 1)) * 1024;
    uint8_t* l = w_lo + (2 * i + (g >> 1)) * 1024;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t hi = pack_bf16(x0[j], x1[j]);
      const uint32_t lo = pack_bf16(x0[j] - __uint_as_float(hi << 16), x1[j] - __uint_as_float(hi & 0xFFFF0000u));
      *reinterpret_cast<uint32_t*>(h + (pre[j] ^ kflip)) = hi;
      *reinterpret_cast<uint32_t*>(l + (pre[j] ^ kflip)) = lo;
      if (CSUM) csum[4 * i + j] += x0[j] + x1[j];
    }
  }
}

template <class Epi, bool RM>
__global__ void __launch_bounds__(TN_THREADS, 1)
gemm_tn2_kernel(TnPair p0, TnPair p1, int n_pairs, int M, int N, int64_t K, int64_t k_chunk, Epi epi) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * BM;
  const int n0 = blockIdx.y * 256;
  int rows_b = N - n0; rows_b = pad16(rows_b < 256 ? rows_b : 256);
  const int64_t kb = (int64_t)blockIdx.z * k_chunk;
  const int64_t ke = (kb + k_chunk < K) ? kb + k_chunk : K;
  const int n_sl = (int)((ke - kb + T2_BK - 1) / T2_BK);       // slices per pair
  const int total = n_sl * n_pairs;
  uint8_t* planes = smem;                                       // [A hi | A lo | B hi | B lo]
  uint8_t* raw = smem + T2_PLANES;                              // T2_RING granules x 12 warps x 2 KB
  SmemCtl* ctl = reinterpret_cast<SmemCtl*>(smem + T2_PLANES + T2_RING * T2_RAW_GRAN);
  if ((smem_u32(smem) & 1023u) != 0u) __trap();

  if (tid == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(&ctl->full[s], TN_PROD); mbar_init(&ctl->empty[s], 1); }
    mbar_init(&ctl->tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 12) tmem_alloc(&ctl->tmem_addr, tmem_cols_for(rows_b));
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = ctl->tmem_addr;

  if (warp < 12) {
    const bool is_a = warp < 4;
    const int r0 = is_a ? 32 * warp : 32 * (warp - 4);          // first tile row (= operand column) of this warp's block
    const bool active = is_a || r0 < rows_b;
    uint8_t* s_hi = planes + (is_a ? 0u : 2u * A_HALF_BYTES);
    uint8_t* s_lo = s_hi + (is_a ? (uint32_t)A_HALF_BYTES : T2_B_HALF);
    const uint8_t* raw_warp = raw + warp * T2_RAW_WARP;
    const uint32_t raw_warp_s = smem_u32(raw_warp);
    float csum[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) csum[j] = 0.f;
    auto pair_of = [&](int i) -> const TnPair& { return i < n_sl ? p0 : p1; };
    const int n_gran = 2 * total;
    const int col0 = (is_a ? m0 : n0) + r0;                     // first operand column of this warp
    // k_chunk is a multiple of 128 (launcher): slice i of a pair starts at point kb + 32 i, 4 slices per 128-point block of the
    // T128 layout; inside a block consecutive points are 4 floats apart, the next block is (ld / 4) * 512 floats further
    // per-pair, per-lane source bases, computed once: the copy loop only adds slice / half offsets.
    //   T128:       src(isl, half, q) = xb + (isl >> 2) * bs + (isl & 3) * 128 + half * 2048 + q * 512      (kb is a multiple of 128)
    //   row-major:  src(isl, gr, i)   = xb + (isl * 32 + 16 gr + 4 i) * ld                                  (lane = (point l >> 3, quad l & 7))
    const float* xb[2];
    int64_t bs[2];
    int nq0[2];
    int lane_row;                                               // point offset of this lane inside a granule
#pragma unroll
    for (int pi = 0; pi < 2; ++pi) {
      const TnPair& pr = pi == 0 ? p0 : p1;
      const float* X = is_a ? pr.A : pr.B;
      const int64_t ld = is_a ? pr.lda : pr.ldb;
      if (RM) {
        xb[pi] = X + (kb + (lane >> 3)) * ld + col0 + 4 * (lane & 7);
        bs[pi] = ld;
        nq0[pi] = (col0 + 4 * (lane & 7) < ld) ? 1 : 0;         // this lane's column quad exists
      } else {
        xb[pi] = X + ((kb >> 7) * (ld >> 2) + (col0 >> 2)) * 512 + lane * 4;
        bs[pi] = (ld >> 2) * 512;
        nq0[pi] = (int)(ld >> 2) - (col0 >> 2);                 // column quads of this warp's block that exist
      }
    }
    lane_row = RM ? (lane >> 3) : lane;
    const float* any = is_a ? p0.A : p0.B;
    auto issue = [&](int h) {                                   // granule h = (slice h >> 1, half h & 1); always commits a group
      if (active && h < n_gran) {
        const int i = h >> 1, half = h & 1;
        const int pi = i < n_sl ? 0 : 1;
        const int isl = i < n_sl ? i : i - n_sl;
        const uint32_t dst = raw_warp_s + (uint32_t)(h % T2_RING) * T2_RAW_GRAN;
        const int64_t row0 = kb + (int64_t)isl * T2_BK;         // first point of the slice
        if (RM) {                                               // granule = points [16 half, +16) of the slice, all 32 columns
          const float* src = xb[pi] + ((int64_t)isl * T2_BK + 16 * half) * bs[pi];
          const int c = lane & 7;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int pl = 4 * k + (lane >> 3);
            const bool v = nq0[pi] != 0 && row0 + 16 * half + pl < ke;
            cp_async16(dst + (uint32_t)pl * 128u + (uint32_t)((c ^ (pl >> 1)) & 7) * 16u, v ? src + (int64_t)(4 * k) * bs[pi] : any, v ? 16u : 0u);
          }
        } else {
          const float* src = xb[pi] + (int64_t)(isl >> 2) * bs[pi] + (isl & 3) * 128 + half * 2048;
          t2_issue(src, any, nq0[pi] - 4 * half, row0 + lane_row < ke, dst, lane);
        }
      }
      cp_async_commit();
    };
    // swizzled offsets of this lane's four tile rows (4 g2 + j) at k = 2 rp, per k half
    uint32_t pre[2][4];
#pragma unroll
    for (int kh = 0; kh < 2; ++kh)
#pragma unroll
      for (int j = 0; j < 4; ++j) pre[kh][j] = sw128((uint32_t)(4 * (lane >> 4) + j), (uint32_t)(32 * kh + 2 * (lane & 15)));
    uint32_t pre_rm[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pre_rm[j] = sw128((uint32_t)(4 * ((lane >> 3) & 1) + j), (uint32_t)(2 * (lane & 7)));
    uint8_t* w_hi = s_hi + (r0 >> 3) * 1024;
    uint8_t* w_lo = s_lo + (r0 >> 3) * 1024;
#pragma unroll
    for (int h = 0; h < T2_RING - 1; ++h) issue(h);
    for (int i = 0; i < total; ++i) {
      const int s = i & 1;
      const bool do_csum = is_a && blockIdx.y == 0 && pair_of(i).colsum_a != nullptr;
      // half 0.  __syncwarp before issue: every lane is done reading the ring slot that is refilled; after the wait: the other
      // lanes' copies of this granule are visible
      __syncwarp();
      issue(2 * i + T2_RING - 1);
      cp_async_wait<T2_RING - 1>();
      __syncwarp();
      if (i >= 2) mbar_wait(&ctl->empty[s], (uint32_t)(((i >> 1) - 1) & 1));
      if (active) {
        const uint8_t* rl = raw_warp + (uint32_t)((2 * i) % T2_RING) * T2_RAW_GRAN;
        if (RM) {
          if (do_csum) t2_convert_rm<true>(rl, w_hi, w_lo, pre_rm, (uint32_t)(4 * s) << 4, lane, csum);
          else t2_convert_rm<false>(rl, w_hi, w_lo, pre_rm, (uint32_t)(4 * s) << 4, lane, csum);
        } else if (s == 0) {
          if (do_csum) t2_convert<true, 0>(rl, w_hi, w_lo, pre[0], lane, csum); else t2_convert<false, 0>(rl, w_hi, w_lo, pre[0], lane, csum);
        } else {
          if (do_csum) t2_convert<true, 0>(rl, w_hi, w_lo, pre[1], lane, csum); else t2_convert<false, 0>(rl, w_hi, w_lo, pre[1], lane, csum);
        }
      }
      // half 1
      __syncwarp();
      issue(2 * i + T2_RING);
      cp_async_wait<T2_RING - 1>();
      __syncwarp();
      if (active) {
        const uint8_t* rl = raw_warp + (uint32_t)((2 * i + 1) % T2_RING) * T2_RAW_GRAN;
        if (RM) {
          if (do_csum) t2_convert_rm<true>(rl, w_hi, w_lo, pre_rm, (uint32_t)(4 * s + 2) << 4, lane, csum);
          else t2_convert_rm<false>(rl, w_hi, w_lo, pre_rm, (uint32_t)(4 * s + 2) << 4, lane, csum);
        } else if (s == 0) {
          if (do_csum) t2_convert<true, 1>(rl, w_hi, w_lo, pre[0], lane, csum); else t2_convert<false, 1>(rl, w_hi, w_lo, pre[0], lane, csum);
        } else {
          if (do_csum) t2_convert<true, 1>(rl, w_hi, w_lo, pre[1], lane, csum); else t2_convert<false, 1>(rl, w_hi, w_lo, pre[1], lane, csum);
        }
      }
      fence_proxy_async();
      mbar_arrive(&ctl->full[s]);
      if (is_a && blockIdx.y == 0 && (i == n_sl - 1 || i == total - 1)) {       // end of a pair: flush its column sums
        float* out = pair_of(i).colsum_a;
        if (out != nullptr) out += (int64_t)blockIdx.z * M;     // this split's slice
        if (out != nullptr && RM) {                     // lanes (p, g): columns r0 + 4 (g + 4 i) + j in csum[4 i + j]; reduce over p
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float v = csum[j];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            const int m = m0 + r0 + 4 * ((lane >> 3) + 4 * (j >> 2)) + (j & 3);
            if ((lane & 7) == 0 && m < M) atomicAdd(out + m, v);
            csum[j] = 0.f;
          }
        } else if (out != nullptr) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            float v = csum[j];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            const int m = m0 + r0 + 4 * (2 * (j >> 2) + (lane >> 4)) + (j & 3);
            if ((lane & 15) == 0 && m < M) atomicAdd(out + m, v);
            csum[j] = 0.f;
          }
        }
      }
    }
    cp_async_wait<0>();
    if (total > 0) {
      mbar_wait(&ctl->tmem_full, 0);
      tcgen05_fence_after();
      run_epilogue(tmem_base, warp & 3, lane, 32 * (warp >> 2), 96, 1, 0u, (int64_t)m0 + (warp & 3) * 32, (int64_t)M, n0, rows_b, N,
                   reinterpret_cast<float*>(smem) + warp * EPI_WARP_FLOATS, epi, (int)blockIdx.z);
      tcgen05_fence_before();
    }
  } else {
    if (lane == 0 && total > 0) {
      const uint32_t idesc = make_idesc((uint32_t)rows_b);
      const uint32_t a_hi = smem_u32(planes), a_lo = a_hi + A_HALF_BYTES, b_hi = a_hi + 2u * A_HALF_BYTES, b_lo = b_hi + T2_B_HALF;
      for (int i = 0; i < total; ++i) {
        const int s = i & 1;
        mbar_wait(&ctl->full[s], (uint32_t)((i >> 1) & 1));
        tcgen05_fence_after();
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const uint32_t o = (uint32_t)(2 * s + jj) * 32u;
          const uint64_t dah = make_desc(a_hi + o), dal = make_desc(a_lo + o), dbh = make_desc(b_hi + o), dbl = make_desc(b_lo + o);
          mma_bf16(tmem_base, dal, dbh, idesc, (i == 0 && jj == 0) ? 0u : 1u);
          mma_bf16(tmem_base, dah, dbl, idesc, 1u);
          mma_bf16(tmem_base, dah, dbh, idesc, 1u);
        }
        mma_commit(&ctl->empty[s]);
      }
      mma_commit(&ctl->tmem_full);
    }
    __syncwarp();
  }
  __syncthreads();
  if (warp == 12) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, tmem_cols_for(rows_b));
  }
}

// row_major: operands are plain [K, ld] row-major fp32 (ld % 4 == 0, 16-byte aligned bases); else T128 (common.cuh)
static inline int tn2_splits(int M, int N, int64_t K) {
  const int tiles = (int)(cdiv(M, BM) * cdiv(N, 256));
  int splits = sm_count() / tiles;
  const int max_splits = (int)cdiv(K, 256);                  // at least 8 slices of 32 points per CTA and pair
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  const int64_t k_chunk = round_up(cdiv(K, splits), 128);      // whole 128-point blocks of the T128 layout per CTA
  return (int)cdiv(K, k_chunk);
}

template <class Epi>
static inline int gemm_tn2(const TnPair* pairs, int n_pairs, int M, int N, int64_t K, const Epi& epi, cudaStream_t st, bool row_major = false) {
  if (M <= 0 || N <= 0 || K <= 0 || n_pairs <= 0) return 0;
  if constexpr (std::is_same<Epi, EpiAtomicAdd>::value) {     // fixed-order split-K: slices + sum_slices
    const int splits = tn2_splits(M, N, K);
    const int np = n_pairs > 1 ? 2 : 1;
    const int64_t ldw = round_up(N, 4), slice = (int64_t)M * ldw, cs = (int64_t)splits * M;
    float* ws = nullptr;
    int rc = slices_alloc(&ws, (size_t)(slice * splits + np * cs), st);
    if (rc != 0) return rc;
    TnPair pp[2] = {pairs[0], pairs[np - 1]};
    bool any_cs = false;
    for (int p = 0; p < np; ++p)
      if (pp[p].colsum_a != nullptr) { pp[p].colsum_a = ws + slice * splits + p * cs; any_cs = true; }
    if (any_cs && cudaMemsetAsync(ws + slice * splits, 0, (size_t)(np * cs) * sizeof(float), st) != cudaSuccess) rc = -2;
    if (rc == 0) rc = gemm_tn2(pp, np, M, N, K, EpiSliceStore{ws, ldw, slice}, st, row_major);
    if (rc == 0) {
      SliceJobs jobs{};
      jobs.slices = splits;
      jobs.j[jobs.n++] = SliceJob{ws, slice, ldw, M, N, epi.C, epi.ldc};
      for (int p = 0; p < np; ++p)
        if (pairs[p].colsum_a != nullptr) jobs.j[jobs.n++] = SliceJob{pp[p].colsum_a, M, M, 1, M, pairs[p].colsum_a, M};
      rc = sum_slices(jobs, st);
    }
    const int rf = slices_free(ws, st);
    return rc != 0 ? rc : rf;
  }
  const int splits = tn2_splits(M, N, K);
  const int64_t k_chunk = round_up(cdiv(K, splits), 128);      // whole 128-point blocks of the T128 layout per CTA
  const size_t smem = (size_t)T2_PLANES + (size_t)T2_RING * T2_RAW_GRAN + sizeof(SmemCtl) + 64;
  static bool attr_set[2] = {false, false};
  if (!attr_set[row_major ? 1 : 0]) {
    if (row_major) NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_tn2_kernel<Epi, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    else NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_tn2_kernel<Epi, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set[row_major ? 1 : 0] = true;
  }
  dim3 grid((unsigned)cdiv(M, BM), (unsigned)cdiv(N, 256), (unsigned)splits);
  LaunchTimer lt_(FAM_TC_WGRAD, st);
  const TnPair& q1 = n_pairs > 1 ? pairs[1] : pairs[0];
  if (row_major) gemm_tn2_kernel<Epi, true><<<grid, TN_THREADS, smem, st>>>(pairs[0], q1, n_pairs > 1 ? 2 : 1, M, N, K, k_chunk, epi);
  else gemm_tn2_kernel<Epi, false><<<grid, TN_THREADS, smem, st>>>(pairs[0], q1, n_pairs > 1 ? 2 : 1, M, N, K, k_chunk, epi);
  NUDF_LAUNCH_OK();
  return 0;
}

// several weight images in one launch: grid.y = job
struct PrepWJob { const float* W; uint16_t* img; int ldw, N, K, transposed, np; };
struct PrepWJobs { int n; PrepWJob j[48]; };
static __device__ __forceinline__ void tc_prep_weights_body(const float* __restrict__ W, int64_t ldw, int N, int K, int transposed, int np,
                                                            uint16_t* __restrict__ img, int64_t start, int64_t stride);
static __global__ void tc_prep_weights_jobs_kernel(const __grid_constant__ PrepWJobs jobs) {
  const PrepWJob& J = jobs.j[blockIdx.y];
  tc_prep_weights_body(J.W, J.ldw, J.N, J.K, J.transposed, J.np, J.img, (int64_t)blockIdx.x * blockDim.x + threadIdx.x,
                       (int64_t)gridDim.x * blockDim.x);
}
static inline int prep_weights_jobs(const PrepWJobs& jobs, cudaStream_t st) {
  if (jobs.n <= 0) return 0;
  int64_t mx = 0;
  for (int i = 0; i < jobs.n; ++i) {
    int64_t total = 0;
    for (int t = 0; t < n_tiles(jobs.j[i].N, jobs.j[i].np); ++t) total += (int64_t)tile_rows(jobs.j[i].N, t, jobs.j[i].np) * pad64(jobs.j[i].K);
    mx = total > mx ? total : mx;
  }
  int blocks = (int)((mx + 255) / 256);
  if (blocks > 1024) blocks = 1024;
  tc_prep_weights_jobs_kernel<<<dim3((unsigned)blocks, (unsigned)jobs.n), 256, 0, st>>>(jobs);
  NUDF_LAUNCH_OK();
  return 0;
}

static inline int prep_weights(const float* W, int64_t ldw, int N, int K, int transposed, int np, uint16_t* img, cudaStream_t st) {
  int64_t total = 0;
  for (int t = 0; t < n_tiles(N, np); ++t) total += (int64_t)tile_rows(N, t, np) * pad64(K);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 4096) blocks = 4096;
  tc_prep_weights_kernel<<<blocks, 256, 0, st>>>(W, ldw, N, K, transposed, np, img);
  NUDF_LAUNCH_OK();
  return 0;
}

}  // namespace tc
}  // namespace nudf
