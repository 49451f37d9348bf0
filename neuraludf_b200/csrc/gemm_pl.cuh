// Split-bf16 "plane" tensors and the tcgen05 kernels that consume them without a register round trip.
//
// A plane tensor stores a logical fp32 matrix X[rows x cols] (rows = points, cols = features) as two bf16 planes
// hi = bf16(x), lo = bf16(x - hi) in blocks of 64 rows x 64 cols:
//
//     [row block mb][col block cb][plane][64 rows x 128 B, SWIZZLE_128B]          (8 KB per plane block)
//
// inside a block, element (r, c) sits at sw128(r, c): 8-row atoms of 1024 B, 16-byte chunks XOR-swizzled with (r & 7).
// The SAME bytes are a valid UMMA operand in two roles:
//   * K-major   (rows = M/N index, cols = K): the A operand of the layer chains  (Y = X W^T, K = features);
//   * MN-major  (cols = M/N index, rows = K): both operands of the weight-gradient contraction dW = X^T Y (K = points).
//     Canonical MN-major SW128 layout (cute/atom/mma_traits_sm100.hpp:168-176): ((8,n),(8,k)) : ((1,LBO),(8,SBO)) in
//     16-byte units -- 64 contiguous MN elements per K row, 8 K rows per 1024-byte atom, SBO between atoms along K,
//     LBO between 64-element groups along MN.
// Producers write planes from their epilogues (pl_store4); consumers fetch 8 KB blocks with cp.async.bulk: no LSU traffic,
// no conversion, no transposition in the consumer.  Rows >= the logical row count of the last block must be ZERO
// (they are part of the contraction of the weight gradients); columns beyond the logical width may hold anything finite
// or not -- they only reach output rows / columns that are never stored.
#pragma once
#include "gemm_tc.cuh"

namespace nudf {
namespace tc {

// fp32 row-major -> planes; pad rows (up to the 64-row block) and pad columns (up to the 64-column block) are zeroed
static __global__ void pack_planes_kernel(const float* __restrict__ X, int64_t ldx, int64_t rows, int cols, Planes out) {
  const int groups = out.cb * 16;                                        // 4-column groups per row
  const int64_t rows_pad = (rows + 63) & ~(int64_t)63;
  const int64_t total = rows_pad * groups;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = idx / groups;
    const int col = (int)(idx - row * groups) * 4;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (row < rows) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (col + j < cols) v[j] = X[row * ldx + col + j];
    }
    pl_store4(out, row, col, v);
  }
}
// zero the rows [rows, round_up(rows, 64)) of a plane tensor (weight-gradient contraction pad)
static __global__ void zero_pad_rows_kernel(int64_t rows, Planes t) {
  const int groups = t.cb * 16;
  const int64_t r0 = rows, r1 = (rows + 63) & ~(int64_t)63;
  const int64_t total = (r1 - r0) * groups;
  const float z[4] = {0.f, 0.f, 0.f, 0.f};
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = r0 + idx / groups;
    pl_store4(t, row, (int)(idx % groups) * 4, z);
  }
}

// MN-major SWIZZLE_128B operand descriptor: SBO = 1024 B between 8-row K groups, LBO = bytes between 64-element MN groups
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16, D = F32, A = B = BF16, both MN-major (bits 15, 16), M = 128, N = n
__device__ __forceinline__ uint32_t make_idesc_mn(uint32_t n) { return make_idesc(n) | (1u << 15) | (1u << 16); }

// ---------------------------------------------------------------------------------------------------------------
// C[M x N] (+)= X[P x M]^T Y[P x N]   -- weight gradients, contraction over points -- both operands plane tensors.
// grid = (ceil(M/128), ceil(N/256), splits); each CTA contracts `blocks_per_split` 64-point blocks.
// warps 0-7: epilogue (after the contraction), warp 8: MMA issuer + TMEM owner, warp 9: bulk-copy issuer.
// ---------------------------------------------------------------------------------------------------------------
constexpr int TP_STAGES = 4;
constexpr int TP_THREADS = 320;
constexpr int TP_ROWS = 32;                                       // points per pipeline stage: half a block (4 atoms, contiguous)
constexpr uint32_t TP_PIECE = TP_ROWS * 128u;                     // bytes of one plane of one stage piece (4 KB)
constexpr uint32_t TP_X_BYTES = 2u * 2u * TP_PIECE;               // [plane][2 col blocks] = 16 KB
constexpr uint32_t TP_Y_BYTES = 2u * 4u * TP_PIECE;               // [plane][<= 4 col blocks] = 32 KB
constexpr uint32_t TP_STAGE_BYTES = TP_X_BYTES + TP_Y_BYTES;
struct SmemCtlT {
  uint64_t full[TP_STAGES];
  uint64_t empty[TP_STAGES];
  uint64_t tmem_full;
  uint32_t tmem_addr;
};

template <class Epi>
__global__ void __launch_bounds__(TP_THREADS, 1)
gemm_tn_pl_kernel(Planes X, int M, Planes Y, int N, int64_t P, int64_t blocks_per_split, Epi epi, int dbg) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * 128, n0 = blockIdx.y * 256;
  const int xcb0 = blockIdx.x * 2, ycb0 = blockIdx.y * 4;
  int nxb = X.cb - xcb0; nxb = nxb < 2 ? nxb : 2;
  int nyb = Y.cb - ycb0; nyb = nyb < 4 ? nyb : 4;
  const int n_mma = nyb * 64;
  const int64_t n_blocks = (P + 63) / 64;
  const int64_t kb0 = (int64_t)blockIdx.z * blocks_per_split;
  int64_t kb1 = kb0 + blocks_per_split; kb1 = kb1 < n_blocks ? kb1 : n_blocks;
  const int64_t nk = (kb1 - kb0) * (PL_BLOCK / TP_ROWS);            // pipeline stages of TP_ROWS points
  SmemCtlT* ctl = reinterpret_cast<SmemCtlT*>(smem + TP_STAGES * TP_STAGE_BYTES);
  if (nk <= 0) return;

  if (tid == 0) {
    for (int s = 0; s < TP_STAGES; ++s) { mbar_init(&ctl->full[s], 1); mbar_init(&ctl->empty[s], 1); }
    mbar_init(&ctl->tmem_full, 1);
    fence_barrier_init();
  }
  if (warp == 8) tmem_alloc(&ctl->tmem_addr, tmem_cols_for(n_mma));
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = ctl->tmem_addr;

  if (warp == 9) {
    if (lane == 0) {
      const uint32_t tx = (uint32_t)(2 * nxb + 2 * nyb) * TP_PIECE;
      for (int64_t i = 0; i < nk; ++i) {
        const int s = (int)(i % TP_STAGES);
        const int64_t u = i / TP_STAGES;
        if (u > 0) mbar_wait(&ctl->empty[s], (uint32_t)((u - 1) & 1));
        uint8_t* xs = smem + s * TP_STAGE_BYTES;
        uint8_t* ys = xs + TP_X_BYTES;
        const int64_t mb = kb0 + i / (PL_BLOCK / TP_ROWS);
        const int64_t piece = (i % (PL_BLOCK / TP_ROWS)) * (TP_PIECE / 2);        // uint16 offset inside the plane block
        if (dbg & 1) { mbar_arrive(&ctl->full[s]); continue; }
        mbar_arrive_expect_tx(&ctl->full[s], tx);
        for (int pl = 0; pl < 2; ++pl) {
          for (int c = 0; c < nxb; ++c)
            bulk_g2s(xs + (pl * 2 + c) * TP_PIECE, pl_block(X, mb, xcb0 + c, pl) + piece, TP_PIECE, &ctl->full[s]);
          for (int c = 0; c < nyb; ++c)
            bulk_g2s(ys + (pl * nyb + c) * TP_PIECE, pl_block(Y, mb, ycb0 + c, pl) + piece, TP_PIECE, &ctl->full[s]);
        }
      }
    }
    __syncwarp();
  } else if (warp == 8) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_mn((uint32_t)n_mma);
      for (int64_t i = 0; i < nk; ++i) {
        const int s = (int)(i % TP_STAGES);
        mbar_wait(&ctl->full[s], (uint32_t)((i / TP_STAGES) & 1));
        tcgen05_fence_after();
        const uint32_t xs = smem_u32(smem + s * TP_STAGE_BYTES), ys = xs + TP_X_BYTES;
        const uint32_t x_lo = 2u * TP_PIECE, y_lo = (uint32_t)nyb * TP_PIECE;
#pragma unroll
        for (int j = 0; j < TP_ROWS / 16; ++j) {          // 16 points per MMA = two 8-row atoms = 2048 B
          const uint64_t ah = make_desc_mn(xs + j * 2048u, TP_PIECE), al = make_desc_mn(xs + x_lo + j * 2048u, TP_PIECE);
          const uint64_t bh = make_desc_mn(ys + j * 2048u, TP_PIECE), bl = make_desc_mn(ys + y_lo + j * 2048u, TP_PIECE);
          if (dbg & 8) continue;
          mma_bf16(tmem_base, al, bh, idesc, (i == 0 && j == 0) ? 0u : 1u);
          mma_bf16(tmem_base, ah, bl, idesc, 1u);
          mma_bf16(tmem_base, ah, bh, idesc, 1u);
        }
        mma_commit(&ctl->empty[s]);
      }
      mma_commit(&ctl->tmem_full);
    }
    __syncwarp();
  } else {
    mbar_wait(&ctl->tmem_full, 0);
    tcgen05_fence_after();
    // the stage buffers are idle now: reuse them as the epilogue's transposition tiles
    if (!(dbg & 2))
    run_epilogue(tmem_base, warp & 3, lane, 32 * (warp >> 2), 64, 1, 0u, (int64_t)m0 + (warp & 3) * 32, (int64_t)M, n0, n_mma, N,
                 reinterpret_cast<float*>(smem) + warp * EPI_WARP_FLOATS, epi, (int)blockIdx.z);
    tcgen05_fence_before();
  }
  __syncthreads();
  if (warp == 8) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, tmem_cols_for(n_mma));
  }
}

// ---------------------------------------------------------------------------------------------------------------
// C[M x N] = epi( A[M x K] * B^T )  with A a plane tensor, B the pre-split weight image (weights-resident, K <= 256).
// Same structure as gemm_wr_kernel (gemm_tc.cuh) but the A operand is never touched by a thread: one lane issues 8 KB
// cp.async.bulk copies of plane blocks into a 3-slot ring of single-plane K slices (hi(ks), lo(ks), hi(ks+1), ...) and the
// MMAs of each slot as it lands.  The 8 producer warps of gemm_wr become 8 more epilogue warps: 16 warps drain the
// double-buffered TMEM accumulator, one 32x32 block each per tile (112 registers per epilogue thread via setmaxnreg).
// Plane tensors passed here must be allocated with their rows padded to 128 (planes_elems(round_up(M, 128), K)).
// ---------------------------------------------------------------------------------------------------------------
constexpr int PW_SLOTS = 3;
constexpr int PW_EPI_WARPS = 16;
constexpr int PW_THREADS = (PW_EPI_WARPS + 4) * 32;      // + warpgroup 4: warp 16 MMA issuer / TMEM owner, warp 17 loader, 2 idle
struct SmemCtlW {
  uint64_t full[PW_SLOTS];
  uint64_t empty[PW_SLOTS];
  uint64_t tfull[2];
  uint64_t tempty[2];
  uint64_t wfull;
  uint32_t tmem_addr;
};

template <class Epi>
__global__ void __launch_bounds__(PW_THREADS, 1)
gemm_wrp_kernel(Planes A, int64_t M, int N, int K, const uint16_t* __restrict__ img, Epi epi, int reverse, int dbg) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n0 = blockIdx.y * WR_N;
  const int t = n0 / 256;
  const int rows_t = tile_rows(N, t, 2);
  const int row_in_tile = n0 - t * 256;
  int rows_h = rows_t - row_in_tile; rows_h = rows_h < WR_N ? rows_h : WR_N;
  const int n_slices = pad64(K) / 64;
  const uint32_t w_plane_bytes = (uint32_t)rows_h * 128u;
  uint8_t* w_smem = smem;                                                    // [slice][plane][rows_h x 128 B]
  uint8_t* a_smem = smem + (size_t)n_slices * 2 * w_plane_bytes;             // PW_SLOTS x 16 KB (1024-aligned: rows_h % 16 == 0)
  float* epi_stage = reinterpret_cast<float*>(a_smem + PW_SLOTS * A_HALF_BYTES);
  SmemCtlW* ctl = reinterpret_cast<SmemCtlW*>(reinterpret_cast<uint8_t*>(epi_stage) + PW_EPI_WARPS * EPI_WARP_FLOATS * sizeof(float));
  const uint16_t* img_t = img + tile_offset(N, K, t, 2);
  const int64_t n_mtiles = (M + BM - 1) / BM;
  const uint32_t acc_cols = tmem_cols_for(rows_h);

  if (tid == 0) {
    for (int s = 0; s < PW_SLOTS; ++s) { mbar_init(&ctl->full[s], 1); mbar_init(&ctl->empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&ctl->tfull[a], 1); mbar_init(&ctl->tempty[a], PW_EPI_WARPS * 32); }
    mbar_init(&ctl->wfull, 1);
    fence_barrier_init();
  }
  if (warp == PW_EPI_WARPS) tmem_alloc(&ctl->tmem_addr, 2 * acc_cols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = ctl->tmem_addr;

  if (warp < PW_EPI_WARPS) {
    // 5 warps per scheduler cap the kernel at 96 registers per thread; the MMA / loader warpgroup hands 64 x 128 back and
    // the 512 epilogue threads take +16 each (setmaxnreg.inc only draws from the CTA's own released registers)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
    uint32_t it = 0;
    for (int64_t jt = blockIdx.x; jt < n_mtiles; jt += gridDim.x, ++it) {
      const int64_t mt = reverse ? n_mtiles - 1 - jt : jt;
      const uint32_t a = it & 1u, au = it >> 1;
      auto acc_ready = [&]() { mbar_wait(&ctl->tfull[a], au & 1u); tcgen05_fence_after(); };
      if (dbg & 2) acc_ready();
      else
      run_epilogue<Epi, decltype(acc_ready), 2>(tmem_base + a * acc_cols, warp & 3, lane, 32 * (warp >> 2), 128, 1, 0u,
                                                mt * BM + (warp & 3) * 32, M, n0, rows_h, N, epi_stage + warp * EPI_WARP_FLOATS, epi, 0,
                                                acc_ready);
      tcgen05_fence_before();
      mbar_arrive(&ctl->tempty[a]);
    }
  } else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    const int64_t my_tiles = n_mtiles > (int64_t)blockIdx.x ? (n_mtiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    const int pieces_per_tile = 2 * n_slices;
    const int64_t total = my_tiles * pieces_per_tile;
    if (warp == PW_EPI_WARPS) {
      // ---- warp 16, lane 0: MMA issuer.  It only ever waits for data (full[]) and for a free accumulator (tempty[]),
      //      never for the completion of its own MMAs: a commit -> mbarrier -> poll round trip per piece would serialise
      //      issue and completion (measured: ~0.8 us per piece, a 45 us floor per launch). ----
      if (lane == 0) {
        const uint32_t idesc = make_idesc((uint32_t)rows_h);
        const uint32_t w_addr = smem_u32(w_smem);
        mbar_wait(&ctl->wfull, 0);
        int64_t p = 0;
        for (int64_t lt = 0; lt < my_tiles; ++lt) {
          const uint32_t a = (uint32_t)(lt & 1), au = (uint32_t)(lt >> 1);
          if (au > 0) mbar_wait(&ctl->tempty[a], (au - 1) & 1u);
          tcgen05_fence_after();
          const uint32_t acc = tmem_base + a * acc_cols;
          for (int r = 0; r < pieces_per_tile; ++r, ++p) {
            const int slot = (int)(p % PW_SLOTS);
            mbar_wait(&ctl->full[slot], (uint32_t)((p / PW_SLOTS) & 1));
            tcgen05_fence_after();
            const uint32_t a_addr = smem_u32(a_smem + slot * A_HALF_BYTES);
            const uint32_t w_hi = w_addr + (uint32_t)(r >> 1) * 2u * w_plane_bytes, w_lo = w_hi + w_plane_bytes;
            if (dbg & 8) {
            } else if ((r & 1) == 0) {                // hi plane of the slice: hi * lo(W), hi * hi(W)
#pragma unroll
              for (int j = 0; j < BK / 16; ++j) {
                mma_bf16(acc, make_desc(a_addr + j * 32), make_desc(w_lo + j * 32), idesc, (r == 0 && j == 0) ? 0u : 1u);
                mma_bf16(acc, make_desc(a_addr + j * 32), make_desc(w_hi + j * 32), idesc, 1u);
              }
            } else {                                  // lo plane: lo * hi(W)
#pragma unroll
              for (int j = 0; j < BK / 16; ++j) mma_bf16(acc, make_desc(a_addr + j * 32), make_desc(w_hi + j * 32), idesc, 1u);
            }
            mma_commit(&ctl->empty[slot]);
            if (r == pieces_per_tile - 1) mma_commit(&ctl->tfull[a]);
          }
        }
      }
      __syncwarp();
    } else if (warp == PW_EPI_WARPS + 1) {
      // ---- warp 17: weight fetch (one 16 KB copy per lane), then lane 0 streams the A pieces through the ring ----
      if (lane == 0) mbar_arrive_expect_tx(&ctl->wfull, (uint32_t)n_slices * 2u * w_plane_bytes);
      __syncwarp();
      if (lane < 2 * n_slices) {
        const int ks = lane >> 1, pl = lane & 1;
        const uint16_t* src = img_t + (int64_t)ks * 2 * rows_t * 64 + (int64_t)pl * rows_t * 64 + (int64_t)row_in_tile * 64;
        bulk_g2s(w_smem + (size_t)(ks * 2 + pl) * w_plane_bytes, src, w_plane_bytes, &ctl->wfull);
      }
      __syncwarp();
      if (lane == 0) {
        // piece p -> (local tile p / ppt, slice (p % ppt) / 2, plane p % 2); two 8 KB copies (row blocks 2 mt, 2 mt + 1)
        for (int64_t p = 0; p < total; ++p) {
          const int slot = (int)(p % PW_SLOTS);
          const int64_t u = p / PW_SLOTS;
          if (u > 0) mbar_wait(&ctl->empty[slot], (uint32_t)((u - 1) & 1));
          if (dbg & 1) { mbar_arrive(&ctl->full[slot]); continue; }
          const int64_t lt = p / pieces_per_tile;
          const int r = (int)(p - lt * pieces_per_tile);
          const int64_t jt = (int64_t)blockIdx.x + lt * gridDim.x;
          const int64_t mt = reverse ? n_mtiles - 1 - jt : jt;
          uint8_t* dst = a_smem + slot * A_HALF_BYTES;
          mbar_arrive_expect_tx(&ctl->full[slot], (uint32_t)A_HALF_BYTES);
          bulk_g2s(dst, pl_block(A, 2 * mt, r >> 1, r & 1), PL_PLANE_BYTES, &ctl->full[slot]);
          bulk_g2s(dst + PL_PLANE_BYTES, pl_block(A, 2 * mt + 1, r >> 1, r & 1), PL_PLANE_BYTES, &ctl->full[slot]);
        }
      }
      __syncwarp();
    }
  }
  __syncthreads();
  if (warp == PW_EPI_WARPS) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, 2 * acc_cols);
  }
}

template <class Epi>
static inline int gemm_wrp(const Planes& A, int64_t M, int N, int K, const uint16_t* img, const Epi& epi, cudaStream_t st) {
  if (M <= 0 || N <= 0) return 0;
  const int n_slices = pad64(K) / 64;
  if (n_slices > WR_MAX_SLICES || A.cb < n_slices) {
    set_error("gemm_wrp: K = %d does not fit the weights-resident plane kernel", K);
    return -1;
  }
  const size_t smem = (size_t)n_slices * 2 * WR_N * 128 + (size_t)PW_SLOTS * A_HALF_BYTES + PW_EPI_WARPS * EPI_WARP_FLOATS * sizeof(float) +
                      sizeof(SmemCtlW) + 1024 + 64;
  static bool attr_set = false;
  if (!attr_set) {
    NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_wrp_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
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
  gemm_wrp_kernel<Epi><<<grid, PW_THREADS, smem, st>>>(A, M, N, K, img, epi, flip, tc_debug());
  NUDF_LAUNCH_OK();
  return 0;
}

static inline int pack_planes(const float* X, int64_t ldx, int64_t rows, int cols, const Planes& out, cudaStream_t st) {
  if (rows <= 0) return 0;
  const int64_t total = ((rows + 63) & ~(int64_t)63) * out.cb * 16;
  int64_t blocks = (total + 255) / 256;
  if (blocks > 8192) blocks = 8192;
  pack_planes_kernel<<<(unsigned)blocks, 256, 0, st>>>(X, ldx, rows, cols, out);
  NUDF_LAUNCH_OK();
  return 0;
}
static inline int zero_pad_rows(int64_t rows, const Planes& t, cudaStream_t st) {
  if ((rows & 63) == 0) return 0;
  const int64_t total = (64 - (rows & 63)) * t.cb * 16;
  zero_pad_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(rows, t);
  NUDF_LAUNCH_OK();
  return 0;
}

// dW[M x N] (+)= X^T Y over P points; `splits` CTAs along the contraction per output tile
template <class Epi>
static inline int gemm_tn_pl(const Planes& X, int M, const Planes& Y, int N, int64_t P, const Epi& epi, cudaStream_t st, int splits) {
  if (M <= 0 || N <= 0 || P <= 0) return 0;
  const int64_t n_blocks = (P + 63) / 64;
  if (splits < 1) splits = 1;
  const int64_t bps = cdiv(n_blocks, (int64_t)splits);
  splits = (int)cdiv(n_blocks, bps);
  if constexpr (std::is_same<Epi, EpiAtomicAdd>::value) {     // fixed-order split-K: slices + sum_slices
    const int64_t ldw = round_up(N, 4), slice = (int64_t)M * ldw;
    float* ws = nullptr;
    int rc = slices_alloc(&ws, (size_t)(slice * splits), st);
    if (rc != 0) return rc;
    rc = gemm_tn_pl(X, M, Y, N, P, EpiSliceStore{ws, ldw, slice}, st, splits);
    if (rc == 0) rc = sum_slices(ws, splits, slice, ldw, M, N, epi.C, epi.ldc, st);
    const int rf = slices_free(ws, st);
    return rc != 0 ? rc : rf;
  }
  const size_t smem = (size_t)TP_STAGES * TP_STAGE_BYTES + sizeof(SmemCtlT) + 1024 + 64;
  static bool attr_set = false;
  if (!attr_set) {
    NUDF_CUDA_OK(cudaFuncSetAttribute(gemm_tn_pl_kernel<Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  dim3 grid((unsigned)cdiv(M, 128), (unsigned)cdiv(N, 256), (unsigned)splits);
  LaunchTimer lt_(FAM_TC_WGRAD, st);
  gemm_tn_pl_kernel<Epi><<<grid, TP_THREADS, smem, st>>>(X, M, Y, N, P, bps, epi, tc_debug());
  NUDF_LAUNCH_OK();
  return 0;
}

}  // namespace tc
}  // namespace nudf
