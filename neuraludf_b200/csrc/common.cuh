// Shared helpers for the nudf sm_100a kernels.
// Math helpers marked NUDF_HD are compiled for the host as well (tests/host/ builds them with g++ to check
// the per-sample formulas against the oracle on the CPU dev box, where no GPU exists).
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define NUDF_HD __host__ __device__ __forceinline__
#else
#define NUDF_HD inline
#endif

#define NUDF_MAX_LAYERS 16
#define NUDF_SQRT1_2 0.70710678118654752440f

namespace nudf {

// nn.Softplus(beta=100, threshold=20)  (reference models/fields.py:180):  z if 100 z > 20 else log1p(exp(100 z))/100.
// Device code uses the overflow-free form max(z,0) + log(1 + e^{-|100 z|})/100 with the MUFU-based __expf/__logf: the
// argument of the log is in [1,2], where __logf's absolute error is <= 2^-21.4, i.e. <= 4e-9 after the /100 -- an order
// of magnitude below fp32 resolution of the O(0.1..1) activations -- at ~1/5 of the instruction count of log1pf(expf()).
NUDF_HD float softplus100(float z) {
  float bz = 100.0f * z;
#if defined(__CUDA_ARCH__)
  float t = __expf(-fabsf(bz));
  float sp = fmaxf(z, 0.0f) + 0.01f * __logf(1.0f + t);
  return bz > 20.0f ? z : sp;
#else
  return bz > 20.0f ? z : log1pf(expf(bz)) * 0.01f;
#endif
}
// sigma(100 z) recovered from a = softplus100(z); exactly 1 in the linear regime (torch's softplus backward).
NUDF_HD float sig_from_softplus(float a) {
  float ba = 100.0f * a;
#if defined(__CUDA_ARCH__)
  return ba > 20.0f ? 1.0f : 1.0f - __expf(-ba);
#else
  return ba > 20.0f ? 1.0f : -expm1f(-ba);
#endif
}
NUDF_HD float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// "T128" layout of a [rows, ld] fp32 tensor (ld % 4 == 0, storage for round_up(rows, 128) rows): 128-row tiles, inside a tile
// the 4-column groups are outermost and the rows innermost,
//     offset(row, col) = (((row / 128) * (ld / 4) + col / 4) * 128 + row % 128) * 4 + col % 4.
// The fused chain kernels give every thread one ROW of a 128-row tile (that is how tcgen05.ld hands out the accumulator): in
// this layout the 32 lanes of a warp (32 consecutive rows, same column group) touch 512 contiguous bytes per 16-byte access
// -- fully coalesced -- where row-major would touch 32 different lines (1/8 of the L1 wavefront efficiency; measured: the
// epilogues were bound by exactly that).  The weight-gradient kernels, which contract over rows, read 4 consecutive columns of
// consecutive rows: contiguous here as well.
NUDF_HD int64_t t128_off(int64_t row, int64_t col, int64_t ld) {
  return ((((row >> 7) * (ld >> 2) + (col >> 2)) << 7) + (row & 127)) * 4 + (col & 3);
}
NUDF_HD int64_t mat_off(bool t128, int64_t row, int64_t col, int64_t ld) { return t128 ? t128_off(row, col, ld) : row * ld + col; }
NUDF_HD float clampf_(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

}  // namespace nudf

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#include <stdio.h>

namespace nudf {

void set_error(const char* fmt, ...);
void count_launch();

// Per-kernel-family device timing for bench.py (nudf_set_launch_timing): while enabled, every launch wrapped in a
// LaunchTimer is bracketed by a cudaEvent pair recorded on the launching stream; nudf_read_launch_timing() synchronises
// and sums the pairs per family.  Off by default (zero overhead besides one branch).
enum LaunchFamily {
  FAM_UDF_FWD_CHAIN = 0,   // fused UDF value chain (+ reverse sweep when the gradient is requested) (udf_chain.cuh)
  FAM_TC_REV = 1,          // one layer of the reverse sweep (grad_x udf) on tcgen05
  FAM_TC_TAN = 2,          // one layer of the tangent chain
  FAM_TC_BWD = 3,          // one layer of the backward chain
  FAM_TC_OTHER = 4,        // other tcgen05 layer GEMMs (colour / NeRF++ backward, plain forward layers)
  FAM_TC_WGRAD = 5,        // weight-gradient contractions on tcgen05
  FAM_FFMA = 6,            // exact-fp32 FFMA GEMMs
  FAM_RAY = 7,             // ray kernels: compositing forward / backward, sampling, blending
  FAM_ELEMENTWISE = 8,     // element-wise kernels of the library (PE, fold / unfold, seeds, column sums)
  FAM_UDF_BWD_CHAIN = 9,   // fused tangent + backward chains (udf_chain.cuh)
  FAM_COUNT = 10
};
bool launch_timing_on();
int launch_timer_begin(int family, cudaStream_t st);
void launch_timer_end(int slot, cudaStream_t st);
struct LaunchTimer {
  int slot; cudaStream_t st;
  LaunchTimer(int family, cudaStream_t s) : slot(-1), st(s) { if (launch_timing_on()) slot = launch_timer_begin(family, s); }
  ~LaunchTimer() { if (slot >= 0) launch_timer_end(slot, st); }
};

#define NUDF_CUDA_OK(expr)                                                              \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      nudf::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return -2;                                                                        \
    }                                                                                   \
  } while (0)

#define NUDF_LAUNCH_OK()                                                                \
  do {                                                                                  \
    nudf::count_launch();                                                               \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      nudf::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return -2;                                                                        \
    }                                                                                   \
  } while (0)

#define NUDF_REQUIRE(cond, msg)                                                         \
  do {                                                                                  \
    if (!(cond)) {                                                                      \
      nudf::set_error("%s:%d: requirement failed: %s (%s)", __FILE__, __LINE__, #cond, msg); \
      return -1;                                                                        \
    }                                                                                   \
  } while (0)

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t round_up(int64_t a, int64_t b) { return cdiv(a, b) * b; }

__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- weight-norm fold / unfold of ALL layers of a network in one launch ------------------------------------------------------
// W = g v / ||v||  (row-wise; torch._weight_norm(v, g, dim=0), reference models/fields.py:110-113) and its adjoint
// dg = <dW, v>/||v||, dv = g/||v|| (dW - dg v/||v||).  A job = one layer; grid = (max rows over the jobs, number of jobs).
constexpr int NUDF_MAX_JOBS = 32;
struct FoldJob {
  const float* g; const float* v;      // [out], [out, in]
  const float* dw; float* dg; float* dv;   // unfold only
  float* w;                            // fold only: [out, ld], columns >= in zero-filled
  int out, in, ld;
};
struct FoldJobs { int n; FoldJob j[NUDF_MAX_JOBS]; };

static __global__ void fold_jobs_kernel(const __grid_constant__ FoldJobs jobs) {
  const FoldJob& J = jobs.j[blockIdx.y];
  const int row = blockIdx.x;
  if (row >= J.out) return;
  const float* vr = J.v + (int64_t)row * J.in;
  float ss = 0.f;
  for (int k = threadIdx.x; k < J.in; k += blockDim.x) ss += vr[k] * vr[k];
  __shared__ float red[32];
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  const float s = J.g[row] / sqrtf(red[0]);
  for (int k = threadIdx.x; k < J.ld; k += blockDim.x) J.w[(int64_t)row * J.ld + k] = k < J.in ? vr[k] * s : 0.f;
}
static __global__ void unfold_jobs_kernel(const __grid_constant__ FoldJobs jobs) {
  const FoldJob& J = jobs.j[blockIdx.y];
  const int row = blockIdx.x;
  if (row >= J.out) return;
  const float* vr = J.v + (int64_t)row * J.in;
  const float* dr = J.dw + (int64_t)row * J.ld;
  float ss = 0.f, dot = 0.f;
  for (int k = threadIdx.x; k < J.in; k += blockDim.x) { ss += vr[k] * vr[k]; dot += vr[k] * dr[k]; }
  __shared__ float red[2][32];
  for (int o = 16; o > 0; o >>= 1) { ss += __shfl_xor_sync(0xffffffffu, ss, o); dot += __shfl_xor_sync(0xffffffffu, dot, o); }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = ss; red[1][threadIdx.x >> 5] = dot; }
  __syncthreads();
  if (threadIdx.x < 32) {
    float t0 = threadIdx.x < (blockDim.x >> 5) ? red[0][threadIdx.x] : 0.f;
    float t1 = threadIdx.x < (blockDim.x >> 5) ? red[1][threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) { t0 += __shfl_xor_sync(0xffffffffu, t0, o); t1 += __shfl_xor_sync(0xffffffffu, t1, o); }
    if (threadIdx.x == 0) { red[0][0] = t0; red[1][0] = t1; }
  }
  __syncthreads();
  const float n = sqrtf(red[0][0]);
  const float dgv = red[1][0] / n;
  if (threadIdx.x == 0) J.dg[row] = dgv;
  const float gn = J.g[row] / n;
  for (int k = threadIdx.x; k < J.in; k += blockDim.x) J.dv[(int64_t)row * J.in + k] = gn * (dr[k] - dgv * vr[k] / n);
}
// host: launch all jobs at once
static inline int run_fold_jobs(const FoldJobs& jobs, bool unfold, cudaStream_t st) {
  if (jobs.n <= 0) return 0;
  int max_out = 0;
  for (int i = 0; i < jobs.n; ++i) max_out = jobs.j[i].out > max_out ? jobs.j[i].out : max_out;
  const dim3 grid((unsigned)max_out, (unsigned)jobs.n);
  if (unfold) unfold_jobs_kernel<<<grid, 128, 0, st>>>(jobs);
  else fold_jobs_kernel<<<grid, 128, 0, st>>>(jobs);
  NUDF_LAUNCH_OK();
  return 0;
}

// ---- deterministic split reductions --------------------------------------------------------------------------------------------
// A contraction split over CTAs (split-K over points) writes each split's partial result into its own slice of a stream-ordered
// workspace; sum_slices then adds the slices to the destination in a fixed order.  Float atomics would add the partials in
// whatever order the CTAs finish, so the weight gradients -- and every training step after them -- would differ from run to run.
struct SliceJob {                      // C[r, c] += sum over z of ws[z * slice + r * ldw + c],  r < rows, c < cols
  const float* ws; int64_t slice, ldw;
  int rows, cols;
  float* C; int64_t ldc;
};
constexpr int NUDF_MAX_SLICE_JOBS = 3;
struct SliceJobs { int n, slices; SliceJob j[NUDF_MAX_SLICE_JOBS]; };
// grid = (elements / 32, jobs), 256 threads: lane = element, warp w sums slices w, w + 8, ... and the 8 partial sums are added
// in warp order -- a fixed tree, whatever the scheduling.
static __global__ void __launch_bounds__(256) sum_slices_kernel(const __grid_constant__ SliceJobs jobs) {
  const SliceJob& J = jobs.j[blockIdx.y];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * 32 + lane;
  const bool ok = i < (int64_t)J.rows * J.cols;
  const int64_t r = ok ? i / J.cols : 0, c = ok ? i - r * J.cols : 0;
  float s = 0.f;
  if (ok) {
    const float* p = J.ws + r * J.ldw + c;
#pragma unroll 4
    for (int z = w; z < jobs.slices; z += 8) s += __ldcs(p + (int64_t)z * J.slice);
  }
  __shared__ float part[8][32];
  part[w][lane] = s;
  __syncthreads();
  if (w == 0 && ok) {
    float t = part[0][lane];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += part[k][lane];
    J.C[r * J.ldc + c] += t;
  }
}
// status of the launch just issued (counts it like NUDF_LAUNCH_OK, but returns instead of leaving the caller's scope, so that
// a workspace can still be released)
static inline int launch_status() {
  nudf::count_launch();
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return 0;
  nudf::set_error("kernel launch -> %s", cudaGetErrorString(e));
  return -2;
}
// workspace of `floats` floats, allocated in stream order (capturable into a CUDA graph); release with slices_free
static inline int slices_alloc(float** ws, size_t floats, cudaStream_t st) {
  NUDF_CUDA_OK(cudaMallocAsync((void**)ws, floats * sizeof(float), st));
  return 0;
}
static inline int slices_free(float* ws, cudaStream_t st) {
  NUDF_CUDA_OK(cudaFreeAsync(ws, st));
  return 0;
}
static inline int sum_slices(const SliceJobs& jobs, cudaStream_t st) {
  int64_t most = 0;
  for (int k = 0; k < jobs.n; ++k) most = (int64_t)jobs.j[k].rows * jobs.j[k].cols > most ? (int64_t)jobs.j[k].rows * jobs.j[k].cols : most;
  if (most <= 0) return 0;
  sum_slices_kernel<<<dim3((unsigned)cdiv(most, 32), (unsigned)jobs.n), 256, 0, st>>>(jobs);
  return launch_status();
}
// one destination: C[r, c] += sum over z of ws[z * slice + r * ldw + c]
static inline int sum_slices(const float* ws, int slices, int64_t slice, int64_t ldw, int rows, int cols, float* C, int64_t ldc,
                             cudaStream_t st) {
  SliceJobs jobs{};
  jobs.n = 1;
  jobs.slices = slices;
  jobs.j[0] = SliceJob{ws, slice, ldw, rows, cols, C, ldc};
  return sum_slices(jobs, st);
}

}  // namespace nudf
#endif
