// ResidualRenderingNetwork ('no_normal', models/fields.py:400-495) and the NeRF++ background network
// (models/fields.py:541-628): ReLU MLPs built from the dense-layer engine (gemm_engine.cuh) with fused
// bias / activation epilogues and hand-written backward passes.
#include "../../include/nudf.h"
#include "common.cuh"
#include "ew_kernels.cuh"
#include "gemm_engine.cuh"

namespace nudf {

// =================================================================================================================
// shared pieces
// =================================================================================================================

// C[row, c] = acc routed by column range: used for d(main-stack input) = [d PE(view) | d color_base | d x_hidden]
struct EpiColorMainIn {
  int c_cb, c_hid, n_total;            // column where color_base starts, where x_hidden starts, total width
  float* dcb; int64_t ld_dcb;          // [P, d_out]  gradient wrt color_base coming through the main stack
  const float* xhid; int64_t ld_xhid;  // post-ReLU x_hidden (mask)
  float* dzb; int64_t ld_dzb;          // [P, H]      masked gradient wrt the base stack's layer n_lin-2 pre-activation
  struct Aux { float h[4]; };
  __device__ __forceinline__ void load(int64_t row, int col, int nv, Aux& x) const {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int c = col + j;
      x.h[j] = (j < nv && c >= c_hid && c < n_total) ? xhid[row * ld_xhid + (c - c_hid)] : 0.f;
    }
  }
  __device__ __forceinline__ void apply(int64_t row, int col, const float acc[4], int nv, const Aux& x) const {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (j >= nv) break;
      int c = col + j;
      if (c < c_cb) continue;
      if (c < c_hid) dcb[row * ld_dcb + (c - c_cb)] = acc[j];
      else if (c < n_total) dzb[row * ld_dzb + (c - c_hid)] = (x.h[j] > 0.f) ? acc[j] : 0.f;
    }
  }
  NUDF_EPI_CALL
};

// dY = bar * s (1 - s) for the first n_sig columns (sigmoid heads), bar elsewhere; optional extra additive term
__global__ void sigmoid_head_bwd_kernel(const float* __restrict__ bar, int ld_bar, const float* __restrict__ extra,
                                        int ld_extra, const float* __restrict__ s, int ld_s, int n_sig,
                                        const float* __restrict__ bar2, int ld_bar2, int n2, int64_t P,
                                        float* __restrict__ dy, int ld_dy) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t row = idx / ld_dy;
  int c = (int)(idx - row * ld_dy);
  if (row >= P) return;
  float v = 0.f;
  if (c < n_sig) {
    float b = bar ? bar[row * ld_bar + c] : 0.f;
    if (extra) b += extra[row * ld_extra + c];
    float sv = s[row * ld_s + c];
    v = b * sv * (1.0f - sv);
  } else if (c < n_sig + n2) {
    v = bar2 ? bar2[row * ld_bar2 + (c - n_sig)] : 0.f;
  }
  dy[row * ld_dy + c] = v;
}

// color = sigmoid(ym[:, :3]); blend = ym[:, 3:]
__global__ void color_head_kernel(const float* __restrict__ ym, int ld_ym, int d_out, int n_blend, int64_t P,
                                  float* __restrict__ color, float* __restrict__ cs, int ld_cs, float* __restrict__ blend) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int w = d_out + n_blend;
  int64_t row = idx / w;
  int c = (int)(idx - row * w);
  if (row >= P) return;
  float v = ym[row * ld_ym + c];
  if (c < d_out) {
    float s = sigmoidf_(v);
    if (color) color[row * d_out + c] = s;
    cs[row * ld_cs + c] = s;
  } else if (blend) {
    blend[row * n_blend + (c - d_out)] = v;
  }
}

__global__ void pack_pts_feat_kernel(const float* __restrict__ pts, const float* __restrict__ feat, int64_t ld_feat, int F,
                                     int64_t P, float* __restrict__ xb, int ld_xb) {
  // one thread = 4 consecutive columns of one row (ld_xb % 4 == 0: one 16-byte store; the reads of the odd-width feature
  // tensor stay scalar but consecutive across the warp)
  const int q4 = ld_xb >> 2;
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t row = idx / q4;
  int c = (int)(idx - row * q4) * 4;
  if (row >= P) return;
  float v[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int cj = c + j;
    v[j] = cj < 3 ? pts[row * 3 + cj] : (cj < 3 + F ? feat[row * ld_feat + (cj - 3)] : 0.f);
  }
  *reinterpret_cast<float4*>(xb + row * ld_xb + c) = make_float4(v[0], v[1], v[2], v[3]);
}

// Forward of a narrow head (N <= 16 outputs, K <= 128: colour_base, the colour / blending-logit head): Y[p, n] = act(<X[p, :], W[n, :]> + b[n]).
// One warp per point, lanes along K (coalesced 128-byte reads of X, which may be an unaligned column window of a wider tensor); the
// weights live in registers.  Streams X once (HBM-bound) instead of padding 3..13 output columns to a 128-wide GEMM tile.
template <int MAXN>
__global__ void __launch_bounds__(256) dense_small_forward_kernel(const float* __restrict__ X, int64_t ldx, const float* __restrict__ W, int64_t ldw,
                                                                 const float* __restrict__ bias, int N, int K, int act, float post_scale,
                                                                 float* __restrict__ C, int64_t ldc, int64_t P) {
  const int lane = threadIdx.x & 31;
  const int64_t gwarp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float w[MAXN][4];
#pragma unroll
  for (int n = 0; n < MAXN; ++n)
#pragma unroll
    for (int i = 0; i < 4; ++i) w[n][i] = (n < N && lane + 32 * i < K) ? W[(int64_t)n * ldw + lane + 32 * i] : 0.f;
  const float b = (bias != nullptr && lane < N) ? bias[lane] : 0.f;
  constexpr int R = 4;                                     // points per warp iteration: 16 independent loads in flight per lane
  for (int64_t row0 = gwarp * R; row0 < P; row0 += nwarps * R) {
    float x[R][4];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int i = 0; i < 4; ++i) x[r][i] = (row0 + r < P && lane + 32 * i < K) ? X[(row0 + r) * ldx + lane + 32 * i] : 0.f;
    float mine[R];
#pragma unroll
    for (int r = 0; r < R; ++r) mine[r] = 0.f;
#pragma unroll
    for (int n = 0; n < MAXN; ++n) {
      if (n < N) {
        float t[R];
#pragma unroll
        for (int r = 0; r < R; ++r) t[r] = x[r][0] * w[n][0] + x[r][1] * w[n][1] + x[r][2] * w[n][2] + x[r][3] * w[n][3];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int r = 0; r < R; ++r) t[r] += __shfl_xor_sync(0xffffffffu, t[r], o);
#pragma unroll
        for (int r = 0; r < R; ++r)
          if (lane == n) mine[r] = t[r];
      }
    }
    if (lane < N) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (row0 + r < P) {
          float t = mine[r] + b;
          if (act == ACT_RELU) t = fmaxf(t, 0.f);
          else if (act == ACT_SOFTPLUS100) t = softplus100(t);
          else if (act == ACT_SIGMOID) t = sigmoidf_(t);
          C[(row0 + r) * ldc + lane] = t * post_scale;
        }
      }
    }
  }
}
static inline int dense_small_forward(const float* X, int64_t ldx, const float* W, int64_t ldw, int64_t P, int N, int K, const EpiAct& e,
                                      cudaStream_t st) {
  int blocks = (int)cdiv(P, 8 * 16);                         // ~16 points per warp
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  dense_small_forward_kernel<16><<<blocks, 256, 0, st>>>(X, ldx, W, ldw, e.bias, N, K, e.act, e.post_scale, e.C, e.ldc, P);
  NUDF_LAUNCH_OK();
  return 0;
}

// Weight gradient of a narrow head (n_out <= 16: colour / density heads): dW[m, n] += sum_p dZ[p, m] X[p, n], db[m] += sum_p dZ[p, m];
// the kernel writes the partial sums of point chunk blockIdx.y to slice blockIdx.y of dW ([n_out, ldw] per slice) and db.
// Streams X once (HBM-bound) instead of padding the 3..13 output rows to a 128-wide GEMM tile.  CTA = 128 input columns x 4
// point lanes over a 256-point chunk; the lanes' partial sums meet in shared memory, then one store per (m, n) per CTA.
template <int MAXM>
__global__ void __launch_bounds__(512)
wgrad_small_kernel(const float* __restrict__ dZ, int64_t ldz, const float* __restrict__ X, int64_t ldx, int n_out, int n_in, int64_t P,
                   int64_t chunk, float* __restrict__ dW, int64_t ldw, float* __restrict__ db) {
  const int tx = threadIdx.x & 127, ty = threadIdx.x >> 7;
  const int n = blockIdx.x * 128 + tx;
  const int64_t p0 = (int64_t)blockIdx.y * chunk;
  const int64_t p1 = p0 + chunk < P ? p0 + chunk : P;
  float acc[MAXM];
#pragma unroll
  for (int m = 0; m < MAXM; ++m) acc[m] = 0.f;
  float bs = 0.f;
  __shared__ float sdz[64][MAXM];
  __shared__ float red[3][MAXM][128];
  for (int64_t pb = p0; pb < p1; pb += 64) {
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * MAXM; i += blockDim.x) {
      int r = i / MAXM, m = i - r * MAXM;
      sdz[r][m] = (pb + r < p1 && m < n_out) ? dZ[(pb + r) * ldz + m] : 0.f;
    }
    __syncthreads();
    const int cnt = (int)((p1 - pb) < 64 ? (p1 - pb) : 64);
#pragma unroll 4
    for (int r = ty; r < cnt; r += 4) {
      const float x = n < n_in ? X[(pb + r) * ldx + n] : 0.f;
#pragma unroll
      for (int m = 0; m < MAXM; ++m) acc[m] = fmaf(sdz[r][m], x, acc[m]);
    }
    if (threadIdx.x < MAXM)
      for (int r = 0; r < cnt; ++r) bs += sdz[r][threadIdx.x];
  }
  if (ty > 0) {
#pragma unroll
    for (int m = 0; m < MAXM; ++m) red[ty - 1][m][tx] = acc[m];
  }
  __syncthreads();
  if (ty == 0 && n < n_in) {
#pragma unroll
    for (int m = 0; m < MAXM; ++m)
      if (m < n_out) dW[((int64_t)blockIdx.y * n_out + m) * ldw + n] = acc[m] + red[0][m][tx] + red[1][m][tx] + red[2][m][tx];
  }
  if (db != nullptr && blockIdx.x == 0 && threadIdx.x < n_out) db[(int64_t)blockIdx.y * n_out + threadIdx.x] = bs;
}

static int wgrad(const float* dZ, int64_t ldz, const float* X, int64_t ldx, int n_out, int n_in, int64_t P, float* dW,
                 int64_t ldw, float* db, cudaStream_t st) {
  if (n_out <= 16 && P > 0) {
    const int64_t chunk = 256;
    dim3 grid((unsigned)cdiv(n_in, 128), (unsigned)cdiv(P, chunk));
    // every chunk of points writes its partial sums into its own slice; sum_slices adds them in chunk order
    const int slices = (int)grid.y;
    const int64_t slice = (int64_t)n_out * n_in;
    float* ws = nullptr;
    int rc = slices_alloc(&ws, (size_t)(slices * (slice + n_out)), st);
    if (rc != 0) return rc;
    float* wdb = db != nullptr ? ws + slices * slice : nullptr;
    wgrad_small_kernel<16><<<grid, 512, 0, st>>>(dZ, ldz, X, ldx, n_out, n_in, P, chunk, ws, n_in, wdb);
    rc = launch_status();
    if (rc == 0) {
      SliceJobs jobs{};
      jobs.slices = slices;
      jobs.j[jobs.n++] = SliceJob{ws, slice, n_in, n_out, n_in, dW, ldw};
      if (db != nullptr) jobs.j[jobs.n++] = SliceJob{wdb, n_out, n_out, 1, n_out, db, n_out};
      rc = sum_slices(jobs, st);
    }
    const int rf = slices_free(ws, st);
    return rc != 0 ? rc : rf;
  }
  int split = (int)cdiv(P, 2048);
  EpiAtomicAdd ew{dW, ldw};
  return gemm_tn(dZ, ldz, X, ldx, n_out, n_in, P, ew, st, split, TC_WGRAD, db);
}

// =================================================================================================================
// colour network
// =================================================================================================================
struct ColorPlan {
  int n_lin, F, H, d_out, n_blend, Lv, d_view;
  int dims_b[NUDF_MAX_LAYERS + 1], dims_m[NUDF_MAX_LAYERS + 1];
  int64_t wb_off[NUDF_MAX_LAYERS], wm_off[NUDF_MAX_LAYERS], wb_ld[NUDF_MAX_LAYERS], wm_ld[NUDF_MAX_LAYERS], w_total;
  int64_t bb_off[NUDF_MAX_LAYERS], bm_off[NUDF_MAX_LAYERS], b_total;
  int64_t ib_nt[NUDF_MAX_LAYERS], ib_nn[NUDF_MAX_LAYERS], im_nt[NUDF_MAX_LAYERS], im_nn[NUDF_MAX_LAYERS], img_total;
  int ld_xb, ld_xm, ld_ym, c_cb, c_hid;
};

static int color_plan(const nudf_color_desc* d, ColorPlan* p) {
  NUDF_REQUIRE(d != nullptr, "null desc");
  NUDF_REQUIRE(d->n_lin >= 3 && d->n_lin <= NUDF_MAX_LAYERS, "n_lin out of range");
  p->n_lin = d->n_lin; p->F = d->d_feature; p->H = d->d_hidden; p->d_out = d->d_out; p->n_blend = d->n_blend;
  p->Lv = d->multires_view;
  p->d_view = 3 * (1 + 2 * p->Lv);
  NUDF_REQUIRE(p->d_out >= 1 && p->d_out <= 4, "d_out must be <= 4");
  p->dims_b[0] = 3 + p->F;
  p->dims_m[0] = p->d_view + p->d_out + p->H;
  for (int l = 1; l < p->n_lin; ++l) { p->dims_b[l] = p->H; p->dims_m[l] = p->H; }
  p->dims_b[p->n_lin] = p->d_out;
  p->dims_m[p->n_lin] = p->d_out + p->n_blend;
  int64_t off = 0, boff = 0;
  for (int l = 0; l < p->n_lin; ++l) {
    p->wb_ld[l] = round_up(p->dims_b[l], 4);
    p->wb_off[l] = off; off = round_up(off + (int64_t)p->dims_b[l + 1] * p->wb_ld[l], 4);
    p->bb_off[l] = boff; boff += p->dims_b[l + 1];
  }
  for (int l = 0; l < p->n_lin; ++l) {
    p->wm_ld[l] = round_up(p->dims_m[l], 4);
    p->wm_off[l] = off; off = round_up(off + (int64_t)p->dims_m[l + 1] * p->wm_ld[l], 4);
    p->bm_off[l] = boff; boff += p->dims_m[l + 1];
  }
  p->w_total = off; p->b_total = boff;
  int64_t ioff = 0;
  for (int l = 0; l < p->n_lin; ++l) {
    p->ib_nt[l] = ioff; ioff += tc::image_elems(p->dims_b[l + 1], p->dims_b[l], 3);    // forward images: 3 planes (6 products)
    p->ib_nn[l] = ioff; ioff += tc::image_elems(p->dims_b[l], p->dims_b[l + 1], 2);
    p->im_nt[l] = ioff; ioff += tc::image_elems(p->dims_m[l + 1], p->dims_m[l], 3);
    p->im_nn[l] = ioff; ioff += tc::image_elems(p->dims_m[l], p->dims_m[l + 1], 2);
  }
  p->img_total = round_up(ioff, 8);
  p->ld_xb = (int)round_up(3 + p->F, 4);
  p->ld_xm = (int)round_up(p->dims_m[0], 4);
  p->ld_ym = (int)round_up(p->d_out + p->n_blend, 4);
  p->c_cb = p->d_view; p->c_hid = p->d_view + p->d_out;
  return 0;
}

struct ColorCtx { int64_t xb, hb[NUDF_MAX_LAYERS], xm, hm[NUDF_MAX_LAYERS], ym, cs, total; };
static void color_ctx_layout(const ColorPlan& p, int64_t P, ColorCtx* c) {
  int64_t off = 0;
  auto take = [&](int64_t n) { int64_t o = off; off += round_up(n, 4); return o; };
  c->xb = take(P * p.ld_xb);
  for (int l = 1; l <= p.n_lin - 2; ++l) c->hb[l] = take(P * p.H);   // outputs of base layers 0..n_lin-3
  c->xm = take(P * p.ld_xm);
  for (int l = 1; l <= p.n_lin - 1; ++l) c->hm[l] = take(P * p.H);   // outputs of main layers 0..n_lin-2
  c->ym = take(P * p.ld_ym);
  c->cs = take(P * 4);
  c->total = off;
}
struct ColorScratch { int64_t buf[2], dym, dyb, dcbx, total; };
static void color_scratch_layout(const ColorPlan& p, int64_t P, ColorScratch* s) {
  int64_t off = 0;
  auto take = [&](int64_t n) { int64_t o = off; off += round_up(n, 4); return o; };
  s->buf[0] = take(P * p.H); s->buf[1] = take(P * p.H);
  s->dym = take(P * p.ld_ym); s->dyb = take(P * 4); s->dcbx = take(P * 4);
  s->total = off;
}

__global__ void fold_kernel2(const float* __restrict__ g, const float* __restrict__ v, int out, int in, int64_t ld,
                             float* __restrict__ w) {
  int row = blockIdx.x;
  if (row >= out) return;
  const float* vr = v + (int64_t)row * in;
  float ss = 0.f;
  for (int k = threadIdx.x; k < in; k += blockDim.x) ss += vr[k] * vr[k];
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
  float s = g[row] / sqrtf(red[0]);
  for (int k = threadIdx.x; k < ld; k += blockDim.x) w[(int64_t)row * ld + k] = k < in ? vr[k] * s : 0.f;
}
__global__ void unfold_kernel2(const float* __restrict__ g, const float* __restrict__ v, const float* __restrict__ dw,
                               int out, int in, int64_t ld, float* __restrict__ dg, float* __restrict__ dv) {
  int row = blockIdx.x;
  if (row >= out) return;
  const float* vr = v + (int64_t)row * in;
  const float* dr = dw + (int64_t)row * ld;
  float ss = 0.f, dot = 0.f;
  for (int k = threadIdx.x; k < in; k += blockDim.x) { ss += vr[k] * vr[k]; dot += vr[k] * dr[k]; }
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
  float n = sqrtf(red[0][0]);
  float dgv = red[1][0] / n;
  if (threadIdx.x == 0) dg[row] = dgv;
  float gn = g[row] / n;
  for (int k = threadIdx.x; k < in; k += blockDim.x) dv[(int64_t)row * in + k] = gn * (dr[k] - dgv * vr[k] / n);
}

}  // namespace nudf

using namespace nudf;

extern "C" {

// One dense layer Y = act(X W^T + b): the primitive every network above is built from, exported for micro-benchmarks
// (bench.py times the dominant 256x256 layer through it) and for callers that want a single fused layer.
int nudf_dense_forward(const float* X, int64_t ldx, const float* W, int64_t ldw, const float* bias, float* Y, int64_t ldy,
                       int64_t M, int32_t N, int32_t K, int32_t act, void* stream) {
  NUDF_REQUIRE(X && W && Y, "null pointer");
  NUDF_REQUIRE(act >= 0 && act <= 3, "act must be 0 (none), 1 (relu), 2 (softplus beta=100), 3 (sigmoid)");
  NUDF_REQUIRE(ldx >= K && ldw >= K && ldy >= N, "leading dimension too small");
  EpiAct e{Y, ldy, bias, act, 1.0f};
  return gemm_nt(X, ldx, W, ldw, M, N, K, e, (cudaStream_t)stream);
}

int64_t nudf_color_folded_floats(const nudf_color_desc* d) {
  ColorPlan p;
  if (color_plan(d, &p)) return -1;
  return p.w_total + p.img_total / 2;
}

int nudf_color_fold_weights(const nudf_color_desc* d, float* wfold, void* stream) {
  ColorPlan p;
  if (int rc = color_plan(d, &p)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  {                                                     // all layers of both stacks: one launch
    FoldJobs jobs;
    jobs.n = 0;
    for (int l = 0; l < p.n_lin; ++l) {
      jobs.j[jobs.n++] = FoldJob{d->base_g[l], d->base_v[l], nullptr, nullptr, nullptr, wfold + p.wb_off[l], p.dims_b[l + 1], p.dims_b[l], (int)p.wb_ld[l]};
      jobs.j[jobs.n++] = FoldJob{d->main_g[l], d->main_v[l], nullptr, nullptr, nullptr, wfold + p.wm_off[l], p.dims_m[l + 1], p.dims_m[l], (int)p.wm_ld[l]};
    }
    if (int rc = run_fold_jobs(jobs, false, st)) return rc;
  }
  if (get_engine() == 1) {
    uint16_t* img = reinterpret_cast<uint16_t*>(wfold + p.w_total);
    tc::PrepWJobs pj;
    pj.n = 0;
    for (int l = 0; l < p.n_lin; ++l) {
      pj.j[pj.n++] = tc::PrepWJob{wfold + p.wb_off[l], img + p.ib_nt[l], (int)p.wb_ld[l], p.dims_b[l + 1], p.dims_b[l], 0, 3};
      pj.j[pj.n++] = tc::PrepWJob{wfold + p.wb_off[l], img + p.ib_nn[l], (int)p.wb_ld[l], p.dims_b[l], p.dims_b[l + 1], 1, 2};
      pj.j[pj.n++] = tc::PrepWJob{wfold + p.wm_off[l], img + p.im_nt[l], (int)p.wm_ld[l], p.dims_m[l + 1], p.dims_m[l], 0, 3};
      pj.j[pj.n++] = tc::PrepWJob{wfold + p.wm_off[l], img + p.im_nn[l], (int)p.wm_ld[l], p.dims_m[l], p.dims_m[l + 1], 1, 2};
    }
    if (int rc = tc::prep_weights_jobs(pj, st)) return rc;
  }
  return 0;
}

int64_t nudf_color_ctx_floats(const nudf_color_desc* d, int64_t P) {
  ColorPlan p;
  if (color_plan(d, &p)) return -1;
  ColorCtx c;
  color_ctx_layout(p, P, &c);
  return c.total;
}
int64_t nudf_color_scratch_floats(const nudf_color_desc* d, int64_t P) {
  ColorPlan p;
  if (color_plan(d, &p)) return -1;
  ColorScratch s;
  color_scratch_layout(p, P, &s);
  return s.total;
}

int nudf_color_forward(const nudf_color_desc* d, const float* wfold, const float* pts, const float* dirs,
                       int32_t samples_per_ray, const float* feat, int64_t ld_feat, int64_t P, float* color_base,
                       float* color, float* blend, float* ctx, void* stream) {
  ColorPlan p;
  if (int rc = color_plan(d, &p)) return rc;
  if (P <= 0) return 0;
  NUDF_REQUIRE(wfold && pts && dirs && feat && ctx, "null pointer");
  NUDF_REQUIRE(ld_feat >= p.F, "ld_feat too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int spr = samples_per_ray > 0 ? samples_per_ray : 1;
  ColorCtx c;
  color_ctx_layout(p, P, &c);
  float* xb = ctx + c.xb;
  float* xm = ctx + c.xm;
  pack_pts_feat_kernel<<<ew_blocks(P * (p.ld_xb / 4), 256), 256, 0, st>>>(pts, feat, ld_feat, p.F, P, xb, p.ld_xb);
  NUDF_LAUNCH_OK();
  ew_pe_kernel<<<ew_blocks(P, 128), 128, 0, st>>>(dirs, 3, p.Lv, spr, P, xm, p.ld_xm, 0, nullptr, 0, 0);
  NUDF_LAUNCH_OK();
  const int nl = p.n_lin;
  const uint16_t* cimg = reinterpret_cast<const uint16_t*>(wfold + p.w_total);
  // base stack
  for (int l = 0; l < nl; ++l) {
    const float* X = l == 0 ? xb : (l == nl - 1 ? xm + p.c_hid : ctx + c.hb[l]);
    int64_t ldx = l == 0 ? p.ld_xb : (l == nl - 1 ? p.ld_xm : p.H);
    EpiAct e;
    e.bias = d->base_b[l]; e.post_scale = 1.0f;
    if (l < nl - 2) { e.C = ctx + c.hb[l + 1]; e.ldc = p.H; e.act = ACT_RELU; }
    else if (l == nl - 2) { e.C = xm + p.c_hid; e.ldc = p.ld_xm; e.act = ACT_RELU; }      // x_hidden (fields.py:472-473)
    else { e.C = xm + p.c_cb; e.ldc = p.ld_xm; e.act = ACT_SIGMOID; }                      // color_base (:475-476)
    if (p.dims_b[l + 1] <= 16 && p.dims_b[l] <= 128) {
      if (int rc = dense_small_forward(X, ldx, wfold + p.wb_off[l], p.wb_ld[l], P, p.dims_b[l + 1], p.dims_b[l], e, st)) return rc;
    } else if (int rc = gemm_nt(X, ldx, wfold + p.wb_off[l], p.wb_ld[l], P, p.dims_b[l + 1], p.dims_b[l], e, st,
                                cimg + p.ib_nt[l], TC_RELU_FWD, 3)) return rc;
  }
  if (color_base) {
    ew_copy_cols_kernel<<<ew_blocks(P * p.d_out, 256), 256, 0, st>>>(xm + p.c_cb, p.ld_xm, color_base, p.d_out, 0, p.d_out, P, 1.f);
    NUDF_LAUNCH_OK();
  }
  // main stack
  for (int l = 0; l < nl; ++l) {
    const float* X = l == 0 ? xm : ctx + c.hm[l];
    int64_t ldx = l == 0 ? p.ld_xm : p.H;
    EpiAct e;
    e.bias = d->main_b[l]; e.post_scale = 1.0f;
    if (l < nl - 1) { e.C = ctx + c.hm[l + 1]; e.ldc = p.H; e.act = ACT_RELU; }
    else { e.C = ctx + c.ym; e.ldc = p.ld_ym; e.act = ACT_NONE; }
    if (p.dims_m[l + 1] <= 16 && p.dims_m[l] <= 128) {
      if (int rc = dense_small_forward(X, ldx, wfold + p.wm_off[l], p.wm_ld[l], P, p.dims_m[l + 1], p.dims_m[l], e, st)) return rc;
    } else if (int rc = gemm_nt(X, ldx, wfold + p.wm_off[l], p.wm_ld[l], P, p.dims_m[l + 1], p.dims_m[l], e, st,
                                cimg + p.im_nt[l], TC_RELU_FWD, 3)) return rc;
  }
  color_head_kernel<<<ew_blocks(P * (p.d_out + p.n_blend), 256), 256, 0, st>>>(ctx + c.ym, p.ld_ym, p.d_out, p.n_blend, P,
                                                                              color, ctx + c.cs, 4, blend);
  NUDF_LAUNCH_OK();
  return 0;
}

int nudf_color_backward(const nudf_color_desc* d, const float* wfold, int64_t P, const float* cb_bar, const float* c_bar,
                        const float* blend_bar, const float* ctx_c, float* scratch, float* dfeat, int64_t ld_df,
                        float* dwfold, float* dbias, void* stream) {
  ColorPlan p;
  if (int rc = color_plan(d, &p)) return rc;
  NUDF_REQUIRE(wfold && ctx_c && scratch && dwfold && dbias, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  NUDF_CUDA_OK(cudaMemsetAsync(dwfold, 0, sizeof(float) * p.w_total, st));
  NUDF_CUDA_OK(cudaMemsetAsync(dbias, 0, sizeof(float) * p.b_total, st));
  if (P <= 0) return 0;
  float* ctx = const_cast<float*>(ctx_c);
  ColorCtx c;
  color_ctx_layout(p, P, &c);
  ColorScratch s;
  color_scratch_layout(p, P, &s);
  const int nl = p.n_lin;
  const uint16_t* cimg = reinterpret_cast<const uint16_t*>(wfold + p.w_total);
  float* xm = ctx + c.xm;
  float* dym = scratch + s.dym;
  sigmoid_head_bwd_kernel<<<ew_blocks(P * p.ld_ym, 256), 256, 0, st>>>(c_bar, p.d_out, nullptr, 0, ctx + c.cs, 4, p.d_out,
                                                                      blend_bar, p.n_blend, p.n_blend, P, dym, p.ld_ym);
  NUDF_LAUNCH_OK();
  // ---- main stack, top down ----
  const float* dz = dym; int64_t ldz = p.ld_ym;
  int flip = 0;
  for (int l = nl - 1; l >= 0; --l) {
    const float* X = l == 0 ? xm : ctx + c.hm[l];
    int64_t ldx = l == 0 ? p.ld_xm : p.H;
    if (int rc = wgrad(dz, ldz, X, ldx, p.dims_m[l + 1], p.dims_m[l], P, dwfold + p.wm_off[l], p.wm_ld[l],
                       dbias + p.bm_off[l], st)) return rc;
    float* out = scratch + s.buf[flip];
    if (l >= 1) {
      EpiReluBwd e{0, p.H, ctx + c.hm[l], p.H, out, p.H, 0};
      if (int rc = gemm_nn(dz, ldz, wfold + p.wm_off[l], p.wm_ld[l], P, p.dims_m[l], p.dims_m[l + 1], e, st,
                           cimg + p.im_nn[l], TC_COLOR)) return rc;
    } else {
      EpiColorMainIn e{p.c_cb, p.c_hid, p.dims_m[0], scratch + s.dcbx, 4, xm + p.c_hid, p.ld_xm, out, p.H};
      if (int rc = gemm_nn(dz, ldz, wfold + p.wm_off[0], p.wm_ld[0], P, p.dims_m[0], p.dims_m[1], e, st,
                           cimg + p.im_nn[0], TC_COLOR)) return rc;
    }
    dz = out; ldz = p.H; flip ^= 1;
  }
  // dz now = masked d(pre-activation of base layer nl-2) coming through the main stack, living in buf[flip^1]
  float* dzb = const_cast<float*>(dz);
  float* dyb = scratch + s.dyb;
  sigmoid_head_bwd_kernel<<<ew_blocks(P * 4, 256), 256, 0, st>>>(cb_bar, p.d_out, scratch + s.dcbx, 4, xm + p.c_cb, p.ld_xm,
                                                                p.d_out, nullptr, 0, 0, P, dyb, 4);
  NUDF_LAUNCH_OK();
  // ---- base stack ----
  {
    const int l = nl - 1;
    if (int rc = wgrad(dyb, 4, xm + p.c_hid, p.ld_xm, p.dims_b[l + 1], p.dims_b[l], P, dwfold + p.wb_off[l], p.wb_ld[l],
                       dbias + p.bb_off[l], st)) return rc;
    EpiReluBwd e{0, p.H, xm + p.c_hid, p.ld_xm, dzb, p.H, 1};
    if (int rc = gemm_nn(dyb, 4, wfold + p.wb_off[l], p.wb_ld[l], P, p.dims_b[l], p.dims_b[l + 1], e, st)) return rc;
  }
  dz = dzb; ldz = p.H;
  for (int l = nl - 2; l >= 0; --l) {
    const float* X = l == 0 ? ctx + c.xb : ctx + c.hb[l];
    int64_t ldx = l == 0 ? p.ld_xb : p.H;
    if (int rc = wgrad(dz, ldz, X, ldx, p.dims_b[l + 1], p.dims_b[l], P, dwfold + p.wb_off[l], p.wb_ld[l],
                       dbias + p.bb_off[l], st)) return rc;
    if (l >= 1) {
      float* out = scratch + s.buf[flip];
      EpiReluBwd e{0, p.H, ctx + c.hb[l], p.H, out, p.H, 0};
      if (int rc = gemm_nn(dz, ldz, wfold + p.wb_off[l], p.wb_ld[l], P, p.dims_b[l], p.dims_b[l + 1], e, st,
                           cimg + p.ib_nn[l], TC_COLOR)) return rc;
      dz = out; flip ^= 1;
    } else if (dfeat) {
      EpiReluBwd e{3, 3 + p.F, nullptr, 0, dfeat, ld_df, 0};
      if (int rc = gemm_nn(dz, ldz, wfold + p.wb_off[0], p.wb_ld[0], P, p.dims_b[0], p.dims_b[1], e, st,
                           cimg + p.ib_nn[0], TC_COLOR)) return rc;
    }
  }
  return 0;
}

int nudf_color_unfold_grads(const nudf_color_desc* d, const float* dwfold, float* const* dg_base, float* const* dv_base,
                            float* const* dg_main, float* const* dv_main, void* stream) {
  ColorPlan p;
  if (int rc = color_plan(d, &p)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  FoldJobs jobs;
  jobs.n = 0;
  for (int l = 0; l < p.n_lin; ++l) {
    jobs.j[jobs.n++] = FoldJob{d->base_g[l], d->base_v[l], dwfold + p.wb_off[l], dg_base[l], dv_base[l], nullptr, p.dims_b[l + 1], p.dims_b[l], (int)p.wb_ld[l]};
    jobs.j[jobs.n++] = FoldJob{d->main_g[l], d->main_v[l], dwfold + p.wm_off[l], dg_main[l], dv_main[l], nullptr, p.dims_m[l + 1], p.dims_m[l], (int)p.wm_ld[l]};
  }
  return run_fold_jobs(jobs, true, st);
}

// =================================================================================================================
// NeRF++ background network
// =================================================================================================================
}  // extern "C"

namespace nudf {
struct NerfPlan {
  int D, W, d_in, L, Lv, skip, ch, chv, ld_f, ld_x5;
  int in_dim[NUDF_MAX_LAYERS];
  // tensor-engine weight images (uint16 offsets): per pts layer X W^T and dY W operands, feature layer, views layer
  int64_t ipts_nt[NUDF_MAX_LAYERS], ipts_nn[NUDF_MAX_LAYERS], ifeat_nt, ifeat_nn, iviews_nt, iviews_nn, img_total;
};
static int nerf_plan(const nudf_nerf_desc* d, NerfPlan* p) {
  NUDF_REQUIRE(d != nullptr, "null desc");
  NUDF_REQUIRE(d->D >= 2 && d->D <= NUDF_MAX_LAYERS, "D out of range");
  p->D = d->D; p->W = d->W; p->d_in = d->d_in; p->L = d->multires; p->Lv = d->multires_view; p->skip = d->skip;
  NUDF_REQUIRE(p->skip < p->D - 1, "skip on the last layer is not supported");
  NUDF_REQUIRE(p->d_in >= 1 && p->d_in <= 4, "d_in out of range");
  p->ch = p->d_in * (1 + 2 * p->L);
  p->chv = 3 * (1 + 2 * p->Lv);
  for (int i = 0; i < p->D; ++i) p->in_dim[i] = i == 0 ? p->ch : (i - 1 == p->skip ? p->W + p->ch : p->W);
  p->ld_f = (int)round_up(p->W + p->chv, 4);
  p->ld_x5 = (int)round_up(p->W + p->ch, 4);
  int64_t io = 0;
  for (int i = 0; i < p->D; ++i) {
    p->ipts_nt[i] = io; io += tc::image_elems(p->W, p->in_dim[i], 3);    // forward images: 3 planes (6 products)
    p->ipts_nn[i] = io; io += tc::image_elems(p->in_dim[i], p->W, 2);
  }
  p->ifeat_nt = io; io += tc::image_elems(p->W, p->W, 3);
  p->ifeat_nn = io; io += tc::image_elems(p->W, p->W, 2);
  p->iviews_nt = io; io += tc::image_elems(p->W / 2, p->W + p->chv, 3);
  p->iviews_nn = io; io += tc::image_elems(p->W + p->chv, p->W / 2, 2);
  p->img_total = round_up(io, 8);
  return 0;
}
struct NerfCtx { int64_t e, h[NUDF_MAX_LAYERS], f, hv, total; };
// h[i] = post-ReLU output of pts layer i; for i == skip it lives inside the concatenated buffer at column ch.
static void nerf_ctx_layout(const NerfPlan& p, int64_t P, NerfCtx* c) {
  int64_t off = 0;
  auto take = [&](int64_t n) { int64_t o = off; off += round_up(n, 4); return o; };
  c->e = take(P * round_up(p.ch, 4));
  for (int i = 0; i < p.D; ++i) c->h[i] = take(P * (i == p.skip ? p.ld_x5 : p.W));
  c->f = take(P * p.ld_f);
  c->hv = take(P * (p.W / 2));
  c->total = off;
}
struct NerfScratch { int64_t buf[2], dzv, dsig, total; };
static void nerf_scratch_layout(const NerfPlan& p, int64_t P, NerfScratch* s) {
  int64_t off = 0;
  auto take = [&](int64_t n) { int64_t o = off; off += round_up(n, 4); return o; };
  s->buf[0] = take(P * p.W); s->buf[1] = take(P * p.W);
  s->dzv = take(P * (p.W / 2));
  s->total = off;
}
// layer-i output location
static inline float* nerf_h(const NerfPlan& p, float* ctx, const NerfCtx& c, int i, int64_t* ld) {
  if (i == p.skip) { *ld = p.ld_x5; return ctx + c.h[i] + p.ch; }
  *ld = p.W; return ctx + c.h[i];
}
// layer-i input location
static inline const float* nerf_x(const NerfPlan& p, float* ctx, const NerfCtx& c, int i, int64_t* ld) {
  if (i == 0) { *ld = round_up(p.ch, 4); return ctx + c.e; }
  if (i - 1 == p.skip) { *ld = p.ld_x5; return ctx + c.h[i - 1]; }
  *ld = p.W; return ctx + c.h[i - 1];
}
}  // namespace nudf

extern "C" {

int64_t nudf_nerf_image_floats(const nudf_nerf_desc* d) {
  NerfPlan p;
  if (nerf_plan(d, &p)) return -1;
  return p.img_total / 2;
}

int nudf_nerf_prepare(const nudf_nerf_desc* d, float* wimg, void* stream) {
  NerfPlan p;
  if (int rc = nerf_plan(d, &p)) return rc;
  NUDF_REQUIRE(wimg != nullptr, "null wimg");
  cudaStream_t st = (cudaStream_t)stream;
  uint16_t* img = reinterpret_cast<uint16_t*>(wimg);
  tc::PrepWJobs pj;                                        // all images in one launch; forward (X W^T) images with 3 planes
  pj.n = 0;
  for (int i = 0; i < p.D; ++i) {
    pj.j[pj.n++] = tc::PrepWJob{d->pts_w[i], img + p.ipts_nt[i], p.in_dim[i], p.W, p.in_dim[i], 0, 3};
    pj.j[pj.n++] = tc::PrepWJob{d->pts_w[i], img + p.ipts_nn[i], p.in_dim[i], p.in_dim[i], p.W, 1, 2};
  }
  pj.j[pj.n++] = tc::PrepWJob{d->feature_w, img + p.ifeat_nt, p.W, p.W, p.W, 0, 3};
  pj.j[pj.n++] = tc::PrepWJob{d->feature_w, img + p.ifeat_nn, p.W, p.W, p.W, 1, 2};
  pj.j[pj.n++] = tc::PrepWJob{d->views_w, img + p.iviews_nt, p.W + p.chv, p.W / 2, p.W + p.chv, 0, 3};
  pj.j[pj.n++] = tc::PrepWJob{d->views_w, img + p.iviews_nn, p.W + p.chv, p.W + p.chv, p.W / 2, 1, 2};
  return tc::prep_weights_jobs(pj, st);
}

int64_t nudf_nerf_ctx_floats(const nudf_nerf_desc* d, int64_t P) {
  NerfPlan p;
  if (nerf_plan(d, &p)) return -1;
  NerfCtx c;
  nerf_ctx_layout(p, P, &c);
  return c.total;
}
int64_t nudf_nerf_scratch_floats(const nudf_nerf_desc* d, int64_t P) {
  NerfPlan p;
  if (nerf_plan(d, &p)) return -1;
  NerfScratch s;
  nerf_scratch_layout(p, P, &s);
  return s.total;
}

int nudf_nerf_forward(const nudf_nerf_desc* d, const float* wimg, const float* pts, const float* dirs, int32_t samples_per_ray,
                      int64_t P, float* sigma, float* rgb, float* ctx, void* stream) {
  NerfPlan p;
  if (int rc = nerf_plan(d, &p)) return rc;
  if (P <= 0) return 0;
  NUDF_REQUIRE(pts && dirs && sigma && rgb && ctx, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int spr = samples_per_ray > 0 ? samples_per_ray : 1;
  NerfCtx c;
  nerf_ctx_layout(p, P, &c);
  const int ld_e = (int)round_up(p.ch, 4);
  const uint16_t* img = reinterpret_cast<const uint16_t*>(wimg);   // null: exact-fp32 engine
  float* x5 = (p.skip >= 0) ? ctx + c.h[p.skip] : nullptr;
  ew_pe_kernel<<<ew_blocks(P, 128), 128, 0, st>>>(pts, p.d_in, p.L, 1, P, ctx + c.e, ld_e, 0, x5, p.ld_x5, 0);
  NUDF_LAUNCH_OK();
  ew_pe_kernel<<<ew_blocks(P, 128), 128, 0, st>>>(dirs, 3, p.Lv, spr, P, ctx + c.f, p.ld_f, p.W, nullptr, 0, 0);
  NUDF_LAUNCH_OK();
  for (int i = 0; i < p.D; ++i) {
    int64_t ldx, ldh;
    const float* X = nerf_x(p, ctx, c, i, &ldx);
    float* Hh = nerf_h(p, ctx, c, i, &ldh);
    EpiAct e{Hh, ldh, d->pts_b[i], ACT_RELU, 1.0f};
    if (int rc = gemm_nt(X, ldx, d->pts_w[i], p.in_dim[i], P, p.W, p.in_dim[i], e, st, img ? img + p.ipts_nt[i] : nullptr, TC_RELU_FWD, 3)) return rc;
  }
  int64_t ldl;
  const float* Hl = nerf_h(p, ctx, c, p.D - 1, &ldl);
  {
    EpiAct e{sigma, 1, d->alpha_b, ACT_NONE, 1.0f};
    if (int rc = gemm_nt(Hl, ldl, d->alpha_w, p.W, P, 1, p.W, e, st)) return rc;
  }
  {
    EpiAct e{ctx + c.f, p.ld_f, d->feature_b, ACT_NONE, 1.0f};
    if (int rc = gemm_nt(Hl, ldl, d->feature_w, p.W, P, p.W, p.W, e, st, img ? img + p.ifeat_nt : nullptr, TC_RELU_FWD, 3)) return rc;
  }
  {
    EpiAct e{ctx + c.hv, p.W / 2, d->views_b, ACT_RELU, 1.0f};
    if (int rc = gemm_nt(ctx + c.f, p.ld_f, d->views_w, p.W + p.chv, P, p.W / 2, p.W + p.chv, e, st, img ? img + p.iviews_nt : nullptr, TC_RELU_FWD, 3)) return rc;
  }
  {
    EpiAct e{rgb, 3, d->rgb_b, ACT_NONE, 1.0f};
    if (int rc = gemm_nt(ctx + c.hv, p.W / 2, d->rgb_w, p.W / 2, P, 3, p.W / 2, e, st)) return rc;
  }
  return 0;
}

int nudf_nerf_backward(const nudf_nerf_desc* d, const float* wimg, int64_t P, const float* sigma_bar, const float* rgb_bar,
                       const float* ctx_c, float* scratch, float* const* dparams, void* stream) {
  NerfPlan p;
  if (int rc = nerf_plan(d, &p)) return rc;
  NUDF_REQUIRE(sigma_bar && rgb_bar && ctx_c && scratch && dparams, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const uint16_t* img = reinterpret_cast<const uint16_t*>(wimg);
  const int D = p.D, W = p.W, W2 = p.W / 2;
  float* const* dpts = dparams;                 // [2*i], [2*i+1]
  float* dviews_w = dparams[2 * D + 0]; float* dviews_b = dparams[2 * D + 1];
  float* dfeat_w = dparams[2 * D + 2];  float* dfeat_b = dparams[2 * D + 3];
  float* dalpha_w = dparams[2 * D + 4]; float* dalpha_b = dparams[2 * D + 5];
  float* drgb_w = dparams[2 * D + 6];   float* drgb_b = dparams[2 * D + 7];
  for (int i = 0; i < D; ++i) {
    NUDF_CUDA_OK(cudaMemsetAsync(dpts[2 * i], 0, sizeof(float) * W * p.in_dim[i], st));
    NUDF_CUDA_OK(cudaMemsetAsync(dpts[2 * i + 1], 0, sizeof(float) * W, st));
  }
  NUDF_CUDA_OK(cudaMemsetAsync(dviews_w, 0, sizeof(float) * W2 * (W + p.chv), st));
  NUDF_CUDA_OK(cudaMemsetAsync(dviews_b, 0, sizeof(float) * W2, st));
  NUDF_CUDA_OK(cudaMemsetAsync(dfeat_w, 0, sizeof(float) * W * W, st));
  NUDF_CUDA_OK(cudaMemsetAsync(dfeat_b, 0, sizeof(float) * W, st));
  NUDF_CUDA_OK(cudaMemsetAsync(dalpha_w, 0, sizeof(float) * W, st));
  NUDF_CUDA_OK(cudaMemsetAsync(dalpha_b, 0, sizeof(float) * 1, st));
  NUDF_CUDA_OK(cudaMemsetAsync(drgb_w, 0, sizeof(float) * 3 * W2, st));
  NUDF_CUDA_OK(cudaMemsetAsync(drgb_b, 0, sizeof(float) * 3, st));
  if (P <= 0) return 0;
  float* ctx = const_cast<float*>(ctx_c);
  NerfCtx c;
  nerf_ctx_layout(p, P, &c);
  NerfScratch s;
  nerf_scratch_layout(p, P, &s);
  // rgb head
  if (int rc = wgrad(rgb_bar, 3, ctx + c.hv, W2, 3, W2, P, drgb_w, W2, drgb_b, st)) return rc;
  float* dzv = scratch + s.dzv;
  {
    EpiReluBwd e{0, W2, ctx + c.hv, W2, dzv, W2, 0};
    if (int rc = gemm_nn(rgb_bar, 3, d->rgb_w, W2, P, W2, 3, e, st)) return rc;
  }
  // views layer
  if (int rc = wgrad(dzv, W2, ctx + c.f, p.ld_f, W2, W + p.chv, P, dviews_w, W + p.chv, dviews_b, st)) return rc;
  float* dfeat = scratch + s.buf[0];
  {
    EpiReluBwd e{0, W, nullptr, 0, dfeat, W, 0};
    if (int rc = gemm_nn(dzv, W2, d->views_w, W + p.chv, P, W + p.chv, W2, e, st, img ? img + p.iviews_nn : nullptr, TC_NERF)) return rc;
  }
  // feature + alpha heads -> dZ of the last pts layer
  int64_t ldl;
  const float* Hl = nerf_h(p, ctx, c, D - 1, &ldl);
  if (int rc = wgrad(dfeat, W, Hl, ldl, W, W, P, dfeat_w, W, dfeat_b, st)) return rc;
  if (int rc = wgrad(sigma_bar, 1, Hl, ldl, 1, W, P, dalpha_w, W, dalpha_b, st)) return rc;
  float* dz = scratch + s.buf[1];
  {
    EpiReluBwd e0{0, W, nullptr, 0, dz, W, 0};
    if (int rc = gemm_nn(sigma_bar, 1, d->alpha_w, W, P, W, 1, e0, st)) return rc;
    EpiReluBwd e1{0, W, Hl, ldl, dz, W, 1};
    if (int rc = gemm_nn(dfeat, W, d->feature_w, W, P, W, W, e1, st, img ? img + p.ifeat_nn : nullptr, TC_NERF)) return rc;
  }
  int flip = 0;  // dz lives in buf[1]; next output goes to buf[0]
  for (int i = D - 1; i >= 0; --i) {
    int64_t ldx;
    const float* X = nerf_x(p, ctx, c, i, &ldx);
    if (int rc = wgrad(dz, W, X, ldx, W, p.in_dim[i], P, dpts[2 * i], p.in_dim[i], dpts[2 * i + 1], st)) return rc;
    if (i == 0) break;
    float* out = scratch + s.buf[flip];
    int64_t ldh;
    const float* Hprev = nerf_h(p, ctx, c, i - 1, &ldh);
    int col_lo = (i - 1 == p.skip) ? p.ch : 0;
    EpiReluBwd e{col_lo, col_lo + W, Hprev, ldh, out, W, 0};
    if (int rc = gemm_nn(dz, W, d->pts_w[i], p.in_dim[i], P, p.in_dim[i], W, e, st, img ? img + p.ipts_nn[i] : nullptr, TC_NERF)) return rc;
    dz = out; flip ^= 1;
  }
  return 0;
}

}  // extern "C"
