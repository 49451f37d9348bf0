// Exact-fp32 SIMT GEMM with fused epilogues (FFMA path).
//
// Role in the design (DESIGN.md section "kernels"): this is the bit-faithful fp32 engine used for (a) every
// contraction that is too small or too oddly shaped for the tcgen05 path (K = 39/30/3, N = 1/3/13), (b) the
// parity anchor the tensor-core path is validated against on the GPU.  C = epi(A * B) with the contraction
// dimension K; operand layouts are chosen per call:
//     A(m,k) = A_KC ? A[m*lda + k] : A[k*lda + m]
//     B(k,n) = B_KC ? B[n*ldb + k] : B[k*ldb + n]
// so  X W^T (forward / tangent chains)  is <true,true>,   dY W (reverse / backward chains) is <true,false>,
// and dY^T X (weight gradients, contraction over points, split over gridDim.z into ordered slices) is <false,false>.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace nudf {

constexpr int GS_BM = 128, GS_BN = 128, GS_BK = 8, GS_PAD = 4, GS_THREADS = 256;

// Blackwell packed fp32 FMA (FFMA2): two IEEE fp32 FMAs per lane per issue slot -- the way sm_100 reaches its fp32 peak.
__device__ __forceinline__ unsigned long long pack2(float x, float y) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& x, float& y) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(v));
}
__device__ __forceinline__ void ffma2(unsigned long long& d, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}

// Tile loads are split into a register fetch (issued before the FFMA block of the current tile, so the global/L2
// latency overlaps with compute) and a shared-memory store (after the FFMA block).
template <bool KC>
__device__ __forceinline__ float4 gs_fetch(const float* __restrict__ src, int64_t ld, int64_t mn0, int64_t mn_total, int k0,
                                           int k_end, int tid, bool vec_ok) {
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
  if (KC) {
    // K contiguous in memory: each thread fetches 4 consecutive k of one row.
    int r = tid >> 1;
    int kq = (tid & 1) * 4;
    int64_t row = mn0 + r;
    if (row < mn_total) {
      const float* p = src + row * ld + (k0 + kq);
      if (vec_ok && (k0 + kq + 3) < k_end) {
        t = *reinterpret_cast<const float4*>(p);
      } else {
        if (k0 + kq + 0 < k_end) t.x = p[0];
        if (k0 + kq + 1 < k_end) t.y = p[1];
        if (k0 + kq + 2 < k_end) t.z = p[2];
        if (k0 + kq + 3 < k_end) t.w = p[3];
      }
    }
  } else {
    // M/N contiguous in memory: each thread fetches 4 consecutive m (or n) of one k.
    int k = tid >> 5;
    int q = (tid & 31) * 4;
    if (k0 + k < k_end) {
      const float* p = src + (int64_t)(k0 + k) * ld + (mn0 + q);
      if (vec_ok && (mn0 + q + 3) < mn_total) {
        t = *reinterpret_cast<const float4*>(p);
      } else {
        if (mn0 + q + 0 < mn_total) t.x = p[0];
        if (mn0 + q + 1 < mn_total) t.y = p[1];
        if (mn0 + q + 2 < mn_total) t.z = p[2];
        if (mn0 + q + 3 < mn_total) t.w = p[3];
      }
    }
  }
  return t;
}
template <bool KC>
__device__ __forceinline__ void gs_store(float4 t, float (*dst)[GS_BM + GS_PAD], int tid) {
  if (KC) {
    int r = tid >> 1;
    int kq = (tid & 1) * 4;
    dst[kq + 0][r] = t.x; dst[kq + 1][r] = t.y; dst[kq + 2][r] = t.z; dst[kq + 3][r] = t.w;   // transposed
  } else {
    int k = tid >> 5;
    int q = (tid & 31) * 4;
    *reinterpret_cast<float4*>(&dst[k][q]) = t;
  }
}

template <bool A_KC, bool B_KC, class Epi>
__global__ void __launch_bounds__(GS_THREADS, 2)   // <= 128 registers: two CTAs (16 warps) per SM hide the LDS / FFMA2 latencies
gemm_simt_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, int64_t M, int N,
                 int64_t K, int64_t k_chunk, Epi epi) {
  __shared__ __align__(16) float As[2][GS_BK][GS_BM + GS_PAD];
  __shared__ __align__(16) float Bs[2][GS_BK][GS_BN + GS_PAD];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = (int64_t)blockIdx.x * GS_BM;
  const int n0 = blockIdx.y * GS_BN;
  // contraction range of this CTA (split-K over gridDim.z; K may exceed 2^31 only through M, which it never does)
  const int64_t kb = (int64_t)blockIdx.z * k_chunk;
  const int64_t ke64 = (kb + k_chunk < K) ? kb + k_chunk : K;
  const float* Ab = A_KC ? A + kb : A + kb * lda;
  const float* Bb = B_KC ? B + kb : B + kb * ldb;
  const int k_end = (int)(ke64 - kb);
  const bool a_vec = ((lda & 3) == 0) && aligned16(Ab) && (A_KC || true);
  const bool b_vec = ((ldb & 3) == 0) && aligned16(Bb);

  unsigned long long acc2[8][4];   // acc2[i][jp] = (acc[i][2jp], acc[i][2jp+1])
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc2[i][j] = 0ull;

  const int n_tiles = (k_end + GS_BK - 1) / GS_BK;
  if (n_tiles > 0) {
    gs_store<A_KC>(gs_fetch<A_KC>(Ab, lda, m0, M, 0, k_end, tid, a_vec), As[0], tid);
    gs_store<B_KC>(gs_fetch<B_KC>(Bb, ldb, n0, N, 0, k_end, tid, b_vec), Bs[0], tid);
  }
  __syncthreads();
  for (int t = 0; t < n_tiles; ++t) {
    const int cur = t & 1;
    float4 pa = make_float4(0.f, 0.f, 0.f, 0.f), pb = pa;
    const bool more = (t + 1 < n_tiles);
    if (more) {
      pa = gs_fetch<A_KC>(Ab, lda, m0, M, (t + 1) * GS_BK, k_end, tid, a_vec);
      pb = gs_fetch<B_KC>(Bb, ldb, n0, N, (t + 1) * GS_BK, k_end, tid, b_vec);
    }
#pragma unroll
    for (int k = 0; k < GS_BK; ++k) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 4]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[cur][k][64 + ty * 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4]);
      float4 b1 = *reinterpret_cast<const float4*>(&Bs[cur][k][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const unsigned long long bp[4] = {pack2(b0.x, b0.y), pack2(b0.z, b0.w), pack2(b1.x, b1.y), pack2(b1.z, b1.w)};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const unsigned long long ap = pack2(a[i], a[i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) ffma2(acc2[i][j], ap, bp[j]);
      }
    }
    if (more) {
      gs_store<A_KC>(pa, As[cur ^ 1], tid);
      gs_store<B_KC>(pb, Bs[cur ^ 1], tid);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int64_t row = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (row >= M) continue;
#pragma unroll
    for (int jg = 0; jg < 2; ++jg) {
      int col = n0 + jg * 64 + tx * 4;
      int nv = N - col;
      if (nv <= 0) continue;
      float v[4];
      unpack2(acc2[i][jg * 2 + 0], v[0], v[1]);
      unpack2(acc2[i][jg * 2 + 1], v[2], v[3]);
      epi(row, col, v, nv < 4 ? nv : 4);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Epilogues.  Each receives 4 consecutive columns of one row (nv of them valid).
// ---------------------------------------------------------------------------------------------------------------
enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_SOFTPLUS100 = 2, ACT_SIGMOID = 3 };

__device__ __forceinline__ void ld4(const float* __restrict__ base, int64_t ld, int64_t row, int col, int nv, float out[4]) {
  const float* p = base + row * ld + col;
  if (nv == 4 && ((ld & 3) == 0) && ((col & 3) == 0) && aligned16(base)) {
    float4 t = *reinterpret_cast<const float4*>(p);
    out[0] = t.x; out[1] = t.y; out[2] = t.z; out[3] = t.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) out[j] = j < nv ? p[j] : 0.f;
  }
}
__device__ __forceinline__ void st4(float* __restrict__ base, int64_t ld, int64_t row, int col, int nv, const float v[4]) {
  float* p = base + row * ld + col;
  if (nv == 4 && ((ld & 3) == 0) && ((col & 3) == 0) && aligned16(base)) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < nv) p[j] = v[j];
  }
}

// Every epilogue has two phases so that the tensor-engine epilogue can software-pipeline them: load() fetches the
// auxiliary global data of one (row, 4-column) group into an Aux record (many groups' loads are put in flight first),
// apply() consumes the accumulator values + Aux and stores.  operator() = load + apply (used by the FFMA kernel).
#define NUDF_EPI_CALL                                                                                     \
  __device__ __forceinline__ void operator()(int64_t row, int col, const float acc[4], int nv) const {    \
    Aux aux;                                                                                              \
    load(row, col, nv, aux);                                                                              \
    apply(row, col, acc, nv, aux);                                                                        \
  }

// C[row, col] = act(acc + bias[col]) * post_scale
struct EpiAct {
  float* C; int64_t ldc; const float* bias; int act; float post_scale;
  struct Aux { float b[4]; };
  __device__ __forceinline__ void load(int64_t, int col, int nv, Aux& x) const {
#pragma unroll
    for (int j = 0; j < 4; ++j) x.b[j] = (bias != nullptr && j < nv) ? bias[col + j] : 0.f;
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float t = acc[j] + x.b[j];
      if (act == ACT_RELU) t = fmaxf(t, 0.f);
      else if (act == ACT_SOFTPLUS100) t = softplus100(t);
      else if (act == ACT_SIGMOID) t = sigmoidf_(t);
      v[j] = t * post_scale;
    }
    st4(C, ldc, row, col, nv, v);
  }
  NUDF_EPI_CALL
};

// C[row, col] += acc   (split-K partial sums of weight gradients).  The launchers run it as EpiSliceStore + sum_slices, so
// that the partials are added in a fixed order.
struct EpiAtomicAdd {
  float* C; int64_t ldc;
  struct Aux {};
  __device__ __forceinline__ void load(int64_t, int, int, Aux&) const {}
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux&) const {
    float* p = C + row * ldc + col;
    if (nv == 4 && ((ldc & 3) == 0) && ((col & 3) == 0) && aligned16(C)) {     // one 16-byte reduction instead of four
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(acc[0]), "f"(acc[1]), "f"(acc[2]), "f"(acc[3])
                   : "memory");
      return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < nv) atomicAdd(p + j, acc[j]);
  }
  NUDF_EPI_CALL
};

// (C + blockIdx.z * slice)[row, col] = acc: the partial tile of split blockIdx.z, in its own workspace slice (sum_slices)
struct EpiSliceStore {
  float* C; int64_t ldc; int64_t slice;
  struct Aux {};
  __device__ __forceinline__ void load(int64_t, int, int, Aux&) const {}
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux&) const {
    float* p = C + (int64_t)blockIdx.z * slice + row * ldc + col;
    if (nv == 4 && ((ldc & 3) == 0) && ((slice & 3) == 0) && ((col & 3) == 0) && aligned16(C)) {
      *reinterpret_cast<float4*>(p) = make_float4(acc[0], acc[1], acc[2], acc[3]);
      return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < nv) p[j] = acc[j];
  }
  NUDF_EPI_CALL
};

// Reverse sweep (grad_x udf): acc = G = d udf / d A[l].  Converts it into D_{l-1} = G * s * sigma(100 z_{l-1});
// skip-concatenated columns (>= n_main) are routed to the positional-encoding gradient buffer.
struct EpiRev {
  int n_main; float post_scale;
  const float* Anext; int64_t lda; float a_unscale;   // stored activation of layer l-1 (= A[l], first n_main cols)
  float* Dprev; int64_t ldd;
  float* Gpe; int64_t ldg;                             // [P, d_pe] or null
  struct Aux { float a[4]; };
  __device__ __forceinline__ void load(int64_t row, int col, int nv, Aux& x) const {
    int n = n_main - col;
    n = n < nv ? n : nv;
    if (n > 0) ld4(Anext, lda, row, col, n, x.a);
    else { x.a[0] = x.a[1] = x.a[2] = x.a[3] = 0.f; }
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
    if (col + nv <= n_main) {                          // whole group inside the activation block: vector path
      float d[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) d[j] = acc[j] * post_scale * sig_from_softplus(x.a[j] * a_unscale);
      st4(Dprev, ldd, row, col, nv, d);
      return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j >= nv) break;
      int c = col + j;
      float g = acc[j] * post_scale;
      if (c < n_main) Dprev[row * ldd + c] = g * sig_from_softplus(x.a[j] * a_unscale);
      else if (Gpe != nullptr) Gpe[row * ldg + (c - n_main)] = g;
    }
  }
  NUDF_EPI_CALL
};

// Last reverse GEMM (layer 0): Ge = acc + Gpe
struct EpiRevFinal {
  float* Ge; int64_t ldge; const float* Gpe; int64_t ldg;
  struct Aux { float g[4]; };
  __device__ __forceinline__ void load(int64_t row, int col, int nv, Aux& x) const {
    if (Gpe != nullptr) ld4(Gpe, ldg, row, col, nv, x.g);
    else { x.g[0] = x.g[1] = x.g[2] = x.g[3] = 0.f; }
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = acc[j] + x.g[j];
    st4(Ge, ldge, row, col, nv, v);
  }
  NUDF_EPI_CALL
};

// Tangent chain: acc = Zdot_l.  Q_l = Zdot * D_l * 100 (1 - S_l);  Adot_{l+1} = S_l * Zdot * post_scale.
struct EpiTan {
  const float* Anext; int64_t lda; float a_unscale;
  const float* D; int64_t ldd;
  float* Q; int64_t ldq;
  float* AdotNext; int64_t ldn; float post_scale;
  struct Aux { float a[4], d[4]; };
  __device__ __forceinline__ void load(int64_t row, int col, int nv, Aux& x) const {
    ld4(Anext, lda, row, col, nv, x.a);
    ld4(D, ldd, row, col, nv, x.d);
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
    float q[4], n[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float s = sig_from_softplus(x.a[j] * a_unscale);
      q[j] = acc[j] * x.d[j] * (100.0f * (1.0f - s));
      n[j] = s * acc[j] * post_scale;
    }
    st4(Q, ldq, row, col, nv, q);
    st4(AdotNext, ldn, row, col, nv, n);
  }
  NUDF_EPI_CALL
};

// Backward chain: acc = Abar wrt A[l].  Zbar_{l-1} = Abar * post_scale * S_{l-1} + Q_{l-1} (in place over Q).
struct EpiBwd {
  int n_main; float post_scale;
  const float* Anext; int64_t lda; float a_unscale;
  float* QZ; int64_t ldq;
  struct Aux { float a[4], q[4]; };
  __device__ __forceinline__ void load(int64_t row, int col, int nv, Aux& x) const {
    int n = n_main - col;
    n = n < nv ? n : nv;
    if (n > 0) { ld4(Anext, lda, row, col, n, x.a); ld4(QZ, ldq, row, col, n, x.q); }
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
    if (col >= n_main) return;
    if (col + nv > n_main) nv = n_main - col;
    float q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = acc[j] * post_scale * sig_from_softplus(x.a[j] * a_unscale) + x.q[j];
    st4(QZ, ldq, row, col, nv, q);
  }
  NUDF_EPI_CALL
};

// EpiBwd with a rank-1 term: acc += z0[row] * w0[col].  Used at the top of the backward chain, where the 257-wide last
// layer is split into its 256 feature rows (a K = 256 tensor-engine GEMM) and the udf-head row (this rank-1 update).
struct EpiBwdR1 {
  int n_main; float post_scale;
  const float* Anext; int64_t lda; float a_unscale;
  float* QZ; int64_t ldq;
  const float* z0; const float* w0;
  struct Aux { float a[4], q[4], w[4], z; };
  __device__ __forceinline__ void load(int64_t row, int col, int nv, Aux& x) const {
    int n = n_main - col;
    n = n < nv ? n : nv;
    if (n > 0) {
      ld4(Anext, lda, row, col, n, x.a); ld4(QZ, ldq, row, col, n, x.q); ld4(w0, 0, 0, col, n, x.w);
      x.z = z0[row];
    }
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
    if (col >= n_main) return;
    if (col + nv > n_main) nv = n_main - col;
    float q[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) q[j] = fmaf(x.z, x.w[j], acc[j]) * post_scale * sig_from_softplus(x.a[j] * a_unscale) + x.q[j];
    st4(QZ, ldq, row, col, nv, q);
  }
  NUDF_EPI_CALL
};

// ReLU-MLP backward: dZ_prev[row, c - col_lo] = acc * (Yprev > 0) for c in [col_lo, col_hi); optional accumulate.
struct EpiReluBwd {
  int col_lo, col_hi;
  const float* Yprev; int64_t ldy;   // post-ReLU output of the previous layer (null: no activation)
  float* dZ; int64_t ldz; int accumulate;
  struct Aux { float y[4], p[4]; };
  __device__ __forceinline__ void load(int64_t row, int col, int nv, Aux& x) const {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int c = col + j;
      bool in = (j < nv) && c >= col_lo && c < col_hi;
      int cc = c - col_lo;
      x.y[j] = (in && Yprev != nullptr) ? Yprev[row * ldy + cc] : 1.0f;
      x.p[j] = (in && accumulate) ? dZ[row * ldz + cc] : 0.0f;
    }
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j >= nv) break;
      int c = col + j;
      if (c < col_lo || c >= col_hi) continue;
      float g = x.p[j] + acc[j];
      if (!(x.y[j] > 0.f)) g = 0.f;                     // mask applies to the accumulated sum
      dZ[row * ldz + (c - col_lo)] = g;
    }
  }
  NUDF_EPI_CALL
};

// launch family of a tensor-engine layer GEMM, by its epilogue (bench.py's per-family timing table)
template <class Epi> struct epi_family { static constexpr int value = FAM_TC_OTHER; };
template <> struct epi_family<EpiRev> { static constexpr int value = FAM_TC_REV; };
template <> struct epi_family<EpiRevFinal> { static constexpr int value = FAM_TC_REV; };
template <> struct epi_family<EpiTan> { static constexpr int value = FAM_TC_TAN; };
template <> struct epi_family<EpiBwd> { static constexpr int value = FAM_TC_BWD; };
template <> struct epi_family<EpiBwdR1> { static constexpr int value = FAM_TC_BWD; };

template <bool A_KC, bool B_KC, class Epi>
static inline int gemm_simt(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int N, int64_t K,
                            const Epi& epi, cudaStream_t st, int split_k = 1) {
  if (M <= 0 || N <= 0) return 0;
  if constexpr (std::is_same<Epi, EpiAtomicAdd>::value) {     // fixed-order split-K: slices + sum_slices
    if (K <= 0) return 0;
    const int splits = split_k > 1 ? (int)cdiv(K, round_up(cdiv(K, split_k), GS_BK)) : 1;
    const int64_t ldw = round_up(N, 4), slice = M * ldw;
    float* ws = nullptr;
    int rc = slices_alloc(&ws, (size_t)(slice * splits), st);
    if (rc != 0) return rc;
    rc = gemm_simt<A_KC, B_KC, EpiSliceStore>(A, lda, B, ldb, M, N, K, EpiSliceStore{ws, ldw, slice}, st, split_k);
    if (rc == 0) rc = sum_slices(ws, splits, slice, ldw, (int)M, N, epi.C, epi.ldc, st);
    const int rf = slices_free(ws, st);
    return rc != 0 ? rc : rf;
  }
  LaunchTimer lt_(FAM_FFMA, st);
  int64_t k_chunk = K;
  if (split_k > 1) {
    k_chunk = round_up(cdiv(K, split_k), GS_BK);
    split_k = (int)cdiv(K, k_chunk);
  } else {
    split_k = 1;
  }
  dim3 grid((unsigned)cdiv(M, GS_BM), (unsigned)cdiv(N, GS_BN), (unsigned)split_k);
  gemm_simt_kernel<A_KC, B_KC, Epi><<<grid, GS_THREADS, 0, st>>>(A, lda, B, ldb, M, N, K, k_chunk, epi);
  NUDF_LAUNCH_OK();
  return 0;
}

}  // namespace nudf
