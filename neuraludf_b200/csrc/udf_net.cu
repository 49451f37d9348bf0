// UDFNetwork on B200: forward value chain, exact input-gradient (reverse sweep), and the first+second order
// parameter gradients (tangent chain + backward chain + weight-gradient contractions).
// Reference semantics: models/fields.py:115-231 (forward :192-211, gradient :219-231); maths: SURVEY.md App. A and
// tests/proto/udf_pipeline.py (the torch prototype of exactly this sequence, checked against autograd).
#include "../../include/nudf.h"
#include "common.cuh"
#include "gemm_engine.cuh"
#include "udf_chain.cuh"
#include <string.h>

namespace nudf {

struct UdfPlan {
  int n_lin, d_in, L, d_pe, d_out, skip;
  float scale;
  int in_dim[NUDF_MAX_LAYERS], out_dim[NUDF_MAX_LAYERS];
  int64_t w_off[NUDF_MAX_LAYERS], w_ld[NUDF_MAX_LAYERS], w_total;
  int64_t b_off[NUDF_MAX_LAYERS], b_total;
  int64_t img_nt[NUDF_MAX_LAYERS], img_nn[NUDF_MAX_LAYERS], img_nt3[NUDF_MAX_LAYERS], img_nn1, img_total;   // uint16 offsets of the bf16 hi/lo weight images
  int64_t img_chain[NUDF_MAX_LAYERS];   // uint16 offsets of the fused chains' fp16 slice images (udf_chain.cuh): X W_l^T operands
  int64_t img_chain_nn[NUDF_MAX_LAYERS], img_chain_nn1;   // dY W_l operands (R / B chains); nn1: feature rows 1.. of the last layer
  int64_t img_chain_t[NUDF_MAX_LAYERS];   // X W_l^T operands of the T chain (split-bf16; the F chain's exact fp16 images are img_chain)
  int chain_tb_ok;                      // the fused T + B chains support this network shape as well
  int64_t sb_off[NUDF_MAX_LAYERS], sb_total;   // float offsets (after the images) of the chain's per-layer [scale meta (4) | bias table]
  int chain_ok;                         // the fused value chain supports this network shape
  int pe_ld, y_ld;
  int stash_ld;   // the fused chains' per-CTA stash of the encoding, shifted so that the skip layer's appended columns are octet-aligned
  int a_ld[NUDF_MAX_LAYERS];    // ld of A[l] (input of layer l), l >= 1
  int o_ld[NUDF_MAX_LAYERS];    // ld of D[l] / Q[l] (out_dim rounded)
  int max_ld;
};

static int make_plan(const nudf_udf_desc* d, UdfPlan* p) {
  NUDF_REQUIRE(d != nullptr, "null desc");
  NUDF_REQUIRE(d->n_lin >= 2 && d->n_lin <= NUDF_MAX_LAYERS, "n_lin out of range");
  NUDF_REQUIRE(d->d_in == 3, "d_in must be 3");
  NUDF_REQUIRE(d->multires >= 0 && d->multires <= 16, "multires out of range");
  p->n_lin = d->n_lin; p->d_in = d->d_in; p->L = d->multires; p->d_out = d->d_out; p->skip = d->skip_layer;
  p->scale = d->scale;
  p->d_pe = d->d_in * (1 + 2 * d->multires);
  NUDF_REQUIRE(p->skip < 0 || (p->skip >= 1 && p->skip <= p->n_lin - 1), "skip_layer out of range");
  int64_t off = 0, boff = 0;
  p->max_ld = 0;
  for (int l = 0; l < p->n_lin; ++l) {
    p->in_dim[l] = d->in_dim[l]; p->out_dim[l] = d->out_dim[l];
    NUDF_REQUIRE(p->in_dim[l] > 0 && p->out_dim[l] > 0, "bad layer dims");
    p->w_ld[l] = round_up(p->in_dim[l], 4);
    p->w_off[l] = off; off += (int64_t)p->out_dim[l] * p->w_ld[l];
    off = round_up(off, 4);
    p->b_off[l] = boff; boff += p->out_dim[l];
    p->a_ld[l] = (int)round_up(p->in_dim[l], 8);        // the fused chains move 8-column octets: whole octets stay inside a tensor
    p->o_ld[l] = (int)round_up(p->out_dim[l], 8);
    if (p->a_ld[l] > p->max_ld) p->max_ld = p->a_ld[l];
    if (p->o_ld[l] > p->max_ld) p->max_ld = p->o_ld[l];
  }
  p->w_total = off; p->b_total = boff;
  int64_t ioff = 0;
  for (int l = 0; l < p->n_lin; ++l) {
    p->img_nt[l] = ioff; ioff += tc::image_elems(p->out_dim[l], p->in_dim[l], 2);   // operand of X W^T  (N = out, K = in)
    p->img_nn[l] = ioff; ioff += tc::image_elems(p->in_dim[l], p->out_dim[l], 2);   // operand of dY W   (N = in,  K = out)
    p->img_nt3[l] = ioff; ioff += tc::image_elems(p->out_dim[l], p->in_dim[l], 3);  // 3-plane image for the value chain
  }
  // feature rows 1.. of the last layer as a (N = in, K = d_out - 1) operand: the udf-head row is applied as a rank-1 update
  p->img_nn1 = ioff;
  if (p->d_out > 1) ioff += tc::image_elems(p->in_dim[p->n_lin - 1], p->d_out - 1, 2);
  ioff = round_up(ioff, 512);           // the chain image is fetched with cp.async.bulk: keep its slices 1024-byte aligned
  for (int l = 0; l < p->n_lin; ++l) { p->img_chain[l] = ioff; ioff += chain::ch_layer_elems(p->out_dim[l], p->in_dim[l]); }
  for (int l = 0; l < p->n_lin - 1; ++l) { p->img_chain_nn[l] = ioff; ioff += chain::ch_layer_elems(p->in_dim[l], p->out_dim[l]); }
  p->img_chain_nn1 = ioff;
  if (p->d_out > 1) ioff += chain::ch_layer_elems(p->in_dim[p->n_lin - 1], p->d_out - 1);
  for (int l = 0; l < p->n_lin - 1; ++l) { p->img_chain_t[l] = ioff; ioff += chain::ch_layer_elems(p->out_dim[l], p->in_dim[l]); }
  p->img_total = round_up(ioff, 8);
  int64_t soff = 0;
  for (int l = 0; l < p->n_lin; ++l) { p->sb_off[l] = soff; soff += 4 + (int64_t)chain::CH_NT * chain::ch_n_tiles(p->out_dim[l]); }
  p->sb_total = soff;
  // shapes the fused chain handles: PE fits one K slice, every contraction K <= 256, hidden layers <= 2 output tiles
  p->chain_ok = p->d_pe <= chain::CH_MAX_PE;
  for (int l = 0; l < p->n_lin; ++l) {
    if (tc::pad64(p->in_dim[l]) > 64 * chain::CH_MAX_SLICES) p->chain_ok = 0;
    if (l < p->n_lin - 1 && p->out_dim[l] + (l + 1 == p->skip ? p->d_pe : 0) > 2 * chain::CH_NT) p->chain_ok = 0;
  }
  if (2 * p->n_lin + 2 > chain::CH_MAX_STEPS) p->chain_ok = 0;
  // T + B: the last layer is split into its feature rows (a K = d_out - 1 contraction) and the udf-head row (rank-1 term)
  const int F_ = p->d_out - 1;
  p->chain_tb_ok = p->chain_ok && F_ >= 16 && F_ <= 64 * chain::CH_MAX_SLICES && (F_ % 4) == 0 && p->n_lin >= 3;
  NUDF_REQUIRE(p->in_dim[0] == p->d_pe, "in_dim[0] must equal the positional-encoding width");
  NUDF_REQUIRE(p->out_dim[p->n_lin - 1] == p->d_out, "last layer width must equal d_out");
  for (int l = 1; l < p->n_lin; ++l) {
    int expect = p->out_dim[l - 1] + (l == p->skip ? p->d_pe : 0);
    NUDF_REQUIRE(p->in_dim[l] == expect, "layer dims are not chained consistently");
  }
  p->pe_ld = (int)round_up(p->d_pe, 8);
  p->y_ld = (int)round_up(p->d_out, 8);
  p->stash_ld = (int)round_up(p->d_pe + 8, 8);
  NUDF_REQUIRE(p->stash_ld <= 64, "positional encoding too wide for the fused chains");
  return 0;
}

// Which chains run as fused kernels (udf_chain.cuh).  Like the engine and the chain mask these must not change between a
// forward call and its backward (context / scratch layouts and the folded images depend on them).
// fused_on: F + R and T + B run as fused kernels and every context / scratch tensor they exchange (and the weight-gradient
// kernels read) is stored in the T128 layout (common.cuh).
static inline bool fused_on(const UdfPlan& p) {
  return p.chain_tb_ok && tc_on(TC_FWD) && tc_on(TC_REV) && tc_on(TC_TAN) && tc_on(TC_BWD) && tc_on(TC_WGRAD) && !chain_planes_on();
}
static inline bool fused_fr_on(const UdfPlan& p) { return fused_on(p); }
static inline bool fused_tb_on(const UdfPlan& p) { return fused_on(p); }
static inline int64_t ctx_rows(const UdfPlan& p, int64_t P) { return fused_on(p) ? round_up(P, 128) : P; }

// ---- context / scratch layout (all offsets in floats; every block starts 16B-aligned) -------------------------
constexpr int64_t CHAIN_STASH_ROWS = chain::CH_MAX_GRID * 128;     // one 128-row tile per CTA of the fused chain kernels
struct UdfCtx {
  int64_t e0, a[NUDF_MAX_LAYERS], y, sgn, d[NUDF_MAX_LAYERS], gpe, ge, stash, total;
  // plane mode (chain_planes_on()): D[l] lives only as a split-bf16 plane tensor.  pl_off: float offset of the plane
  // area (aligned to 1024 B at run time), dpl[l]: uint16 offsets inside it.
  int64_t pl_off, dpl[NUDF_MAX_LAYERS];
};
static inline uint16_t* plane_area(float* base, int64_t off) {
  return reinterpret_cast<uint16_t*>((reinterpret_cast<uintptr_t>(base + off) + 1023) & ~(uintptr_t)1023);
}
static inline int cb_of(int cols) { return (cols + 63) / 64; }
static void ctx_layout(const UdfPlan& p, int64_t P_, int with_grad, UdfCtx* c) {
  const int64_t P = ctx_rows(p, P_);            // T128 tensors are stored in whole 128-row tiles
  int64_t off = 0;
  auto take = [&](int64_t n) { int64_t o = off; off += round_up(n, 4); return o; };
  c->e0 = take(P * p.pe_ld);
  c->stash = take((int64_t)CHAIN_STASH_ROWS * p.stash_ld);
  for (int l = 1; l < p.n_lin; ++l) c->a[l] = take(P * p.a_ld[l]);
  c->y = take(P * p.y_ld);
  c->sgn = take(P);
  c->pl_off = 0;
  if (with_grad) {
    if (chain_planes_on()) {
      int64_t e = 0;
      for (int l = 0; l < p.n_lin - 1; ++l) { c->d[l] = 0; c->dpl[l] = e; e += tc::planes_elems(plane_rows(P), p.out_dim[l]); }
      c->pl_off = take(e / 2 + 256);
    } else {
      for (int l = 0; l < p.n_lin - 1; ++l) c->d[l] = take(P * p.o_ld[l]);
    }
    c->gpe = take(P * p.stash_ld);                  // fused chains store it shifted (stash_ld columns)
    c->ge = take(P * p.pe_ld);
  }
  c->total = off;
}
struct UdfScratch {
  int64_t stash;
  int64_t edot, adot[2], q[NUDF_MAX_LAYERS], zlast, total;
  int64_t adot_l[NUDF_MAX_LAYERS];           // fused T chain: Adot[l], l = 1..last, all kept for the weight gradients
  int64_t pl_off, adpl[NUDF_MAX_LAYERS];     // plane mode: Adot[l] (input of layer l of the tangent chain)
};
static void scratch_layout(const UdfPlan& p, int64_t P_, UdfScratch* s) {
  const int64_t P = ctx_rows(p, P_);
  int64_t off = 0;
  auto take = [&](int64_t n) { int64_t o = off; off += round_up(n, 4); return o; };
  s->edot = take(P * p.pe_ld);
  s->stash = take((int64_t)CHAIN_STASH_ROWS * p.stash_ld);
  if (fused_tb_on(p)) {
    s->adot[0] = s->adot[1] = 0;
    for (int l = 1; l < p.n_lin; ++l) s->adot_l[l] = take(P * p.a_ld[l]);
  } else {
    s->adot[0] = take(P * p.max_ld);
    s->adot[1] = take(P * p.max_ld);
  }
  for (int l = 0; l < p.n_lin - 1; ++l) s->q[l] = take(P * p.o_ld[l]);
  s->zlast = take(P * p.y_ld);
  s->pl_off = 0;
  if (chain_planes_on()) {
    int64_t e = 0;
    for (int l = 0; l < p.n_lin; ++l) { s->adpl[l] = e; e += tc::planes_elems(plane_rows(P), p.in_dim[l]); }
    s->pl_off = take(e / 2 + 256);
  }
  s->total = off;
}

// ---- element-wise kernels ---------------------------------------------------------------------------------------

// W = g * v / ||v||  per output row (legacy weight_norm, dim=0); rows padded with zeros up to ld.
__global__ void fold_kernel(const float* __restrict__ g, const float* __restrict__ v, int out, int in, int64_t ld,
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

// dW -> dg = <dW, v>/||v|| ; dv = g/||v|| (dW - dg v/||v||)
__global__ void unfold_kernel(const float* __restrict__ g, const float* __restrict__ v, const float* __restrict__ dw,
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
  float dgv = red[1][0] / n;          // <dW, v/||v||>
  if (threadIdx.x == 0) dg[row] = dgv;
  float gn = g[row] / n;
  for (int k = threadIdx.x; k < in; k += blockDim.x) dv[(int64_t)row * in + k] = gn * (dr[k] - dgv * vr[k] / n);
}

// E0 = PE(x*scale) [P, pe_ld]; optionally also E0/sqrt2 into the skip columns of A[skip].
__global__ void pe_forward_kernel(const float* __restrict__ pts, int64_t P, int L, float scale, float* __restrict__ e0,
                                  int pe_ld, float* __restrict__ askip, int askip_ld, int askip_col) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  float x[3] = {pts[i * 3 + 0] * scale, pts[i * 3 + 1] * scale, pts[i * 3 + 2] * scale};
  float* e = e0 + i * pe_ld;
  float* a = askip ? askip + i * askip_ld + askip_col : nullptr;
  int d_pe = 3 * (1 + 2 * L);
#pragma unroll
  for (int c = 0; c < 3; ++c) { e[c] = x[c]; if (a) a[c] = x[c] * NUDF_SQRT1_2; }
  float f = 1.0f;
  for (int k = 0; k < L; ++k) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float s, co;
      sincosf(x[c] * f, &s, &co);
      e[3 + 6 * k + c] = s; e[3 + 6 * k + 3 + c] = co;
      if (a) { a[3 + 6 * k + c] = s * NUDF_SQRT1_2; a[3 + 6 * k + 3 + c] = co * NUDF_SQRT1_2; }
    }
    f *= 2.0f;
  }
  for (int c = d_pe; c < pe_ld; ++c) e[c] = 0.f;
}

// out = cat(|y0|/scale, y[1:]); sgn = sign(y0)
// y [P, y_ld] -> udf[row * ld_u] = |y0| / scale, feat[row * ld_f + j] = y[1 + j]  (the classic [P, 1 + F] tensor is udf = out,
// feat = out + 1, ld_u = ld_f = ld_out); sgn <- sign(y0)
__global__ void udf_finalize_kernel(const float* __restrict__ y, int y_ld, int d_out, int64_t P, float inv_scale,
                                    float* __restrict__ udf, int64_t ld_u, float* __restrict__ feat, int64_t ld_f, float* __restrict__ sgn, int t128) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t row = idx / d_out;
  int c = (int)(idx - row * d_out);
  if (row >= P) return;
  float v = y[mat_off(t128 != 0, row, c, y_ld)];
  if (c == 0) {
    if (sgn) sgn[row] = (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f);
    if (udf) udf[row * ld_u] = fabsf(v) * inv_scale;
  } else if (feat) {
    feat[row * ld_f + c - 1] = v;
  }
}
__global__ void udf_value_only_kernel(const float* __restrict__ y, int y_ld, int64_t P, float inv_scale, float* __restrict__ udf) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P) udf[i] = fabsf(y[i * y_ld]) * inv_scale;
}

// Reverse-sweep seed: G = (sgn/scale) W_last[0,:]  -> D[n_lin-2] (and Gpe when the last layer is the skip layer).
template <class Epi>
__global__ void rev_init_kernel(const float* __restrict__ sgn, const float* __restrict__ wlast_row0, int in_last,
                                float inv_scale, int64_t P, Epi epi) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int cols4 = (in_last + 3) / 4;
  int64_t row = idx / cols4;
  int c = (int)(idx - row * cols4) * 4;
  if (row >= P) return;
  float s = sgn[row] * inv_scale;
  float v[4];
  int nv = in_last - c < 4 ? in_last - c : 4;
#pragma unroll
  for (int j = 0; j < 4; ++j) v[j] = j < nv ? s * wlast_row0[c + j] : 0.f;
  epi(row, c, v, nv);
}

// grad_x = scale * J_e(x)^T Ge
// gpe_sh (optional, fused chains): the skip layer's part of Ge, stored shifted by `sh` columns (udf_chain.cuh), added here
__global__ void pe_vjp_kernel(const float* __restrict__ pts, const float* __restrict__ ge, int pe_ld, int64_t P, int L,
                              float scale, float* __restrict__ grad, int t128 = 0, const float* __restrict__ gpe_sh = nullptr,
                              int gpe_ld = 0, int sh = 0) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  float g[3 * (1 + 2 * 16)];
  const int d_pe_ = 3 * (1 + 2 * L);
  for (int c = 0; c < d_pe_; ++c) {
    g[c] = ge[mat_off(t128 != 0, i, c, pe_ld)];
    if (gpe_sh != nullptr) g[c] += gpe_sh[mat_off(t128 != 0, i, c + sh, gpe_ld)];
  }
  float f = 1.0f;
  float acc[3] = {g[0], g[1], g[2]};
  float x[3] = {pts[i * 3 + 0] * scale, pts[i * 3 + 1] * scale, pts[i * 3 + 2] * scale};
  for (int k = 0; k < L; ++k) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float s, co;
      sincosf(x[c] * f, &s, &co);
      acc[c] += f * (co * g[3 + 6 * k + c] - s * g[3 + 6 * k + 3 + c]);
    }
    f *= 2.0f;
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) grad[i * 3 + c] = acc[c] * scale;
}

// Edot = scale * J_e(x) gbar  [P, pe_ld]
__global__ void pe_jvp_kernel(const float* __restrict__ pts, const float* __restrict__ gbar, int64_t P, int L, float scale,
                              float* __restrict__ edot, int pe_ld) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  float* e = edot + i * pe_ld;
  float x[3] = {pts[i * 3 + 0] * scale, pts[i * 3 + 1] * scale, pts[i * 3 + 2] * scale};
  float v[3] = {gbar[i * 3 + 0] * scale, gbar[i * 3 + 1] * scale, gbar[i * 3 + 2] * scale};
  int d_pe = 3 * (1 + 2 * L);
#pragma unroll
  for (int c = 0; c < 3; ++c) e[c] = v[c];
  float f = 1.0f;
  for (int k = 0; k < L; ++k) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float s, co;
      sincosf(x[c] * f, &s, &co);
      e[3 + 6 * k + c] = f * co * v[c];
      e[3 + 6 * k + 3 + c] = -f * s * v[c];
    }
    f *= 2.0f;
  }
  for (int c = d_pe; c < pe_ld; ++c) e[c] = 0.f;
}

// dst[:, col0 + c] = src[:, c] * scale   for c < ncols
__global__ void copy_cols_kernel(const float* __restrict__ src, int64_t lds, float* __restrict__ dst, int64_t ldd, int col0,
                                 int ncols, int64_t P, float scale) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t row = idx / ncols;
  int c = (int)(idx - row * ncols);
  if (row >= P) return;
  dst[row * ldd + col0 + c] = src[row * lds + c] * scale;
}

// out[c] (+)= sum_rows w[row] * X[row, c]   (w may be null = 1).  grid: (col tiles of 32, row chunks)
__global__ void weighted_colsum_kernel(const float* __restrict__ X, int64_t ldx, const float* __restrict__ w, float wscale,
                                       int64_t P, int N, int64_t rows_per_block, float* __restrict__ out, int t128) {
  int c = blockIdx.x * 32 + (threadIdx.x & 31);
  int ry = threadIdx.x >> 5;  // 0..7
  int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  int64_t r1 = r0 + rows_per_block < P ? r0 + rows_per_block : P;
  float acc = 0.f;
  if (c < N)
    for (int64_t r = r0 + ry; r < r1; r += 8) acc += (w ? w[r] * wscale : 1.f) * X[mat_off(t128 != 0, r, c, ldx)];
  __shared__ float red[8][33];
  red[ry][threadIdx.x & 31] = acc;
  __syncthreads();
  if (ry == 0 && c < N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x & 31];
    out[(int64_t)blockIdx.y * N + c] = t;      // this row block's slice (colsum adds the slices in order)
  }
}

int colsum(const float* X, int64_t ldx, const float* w, float wscale, int64_t P, int N, float* out, cudaStream_t st, bool t128) {
  if (P <= 0 || N <= 0) return 0;
  int64_t rpb = 512;
  dim3 grid((unsigned)cdiv(N, 32), (unsigned)cdiv(P, rpb));
  float* ws = nullptr;
  int rc = slices_alloc(&ws, (size_t)grid.y * N, st);
  if (rc != 0) return rc;
  weighted_colsum_kernel<<<grid, 256, 0, st>>>(X, ldx, w, wscale, P, N, rpb, ws, t128 ? 1 : 0);
  rc = launch_status();
  if (rc == 0) rc = sum_slices(ws, (int)grid.y, N, N, 1, N, out, N, st);
  const int rf = slices_free(ws, st);
  return rc != 0 ? rc : rf;
}

// Zlast[:,0] = sgn * ob[:,0] / scale ; Zlast[:,1:] = ob[:,1:]
__global__ void zlast_kernel(const float* __restrict__ ub, int64_t ld_ub, const float* __restrict__ fb, int64_t ld_fb,
                             const float* __restrict__ sgn, float inv_scale, int d_out, int y_ld, int64_t P, float* __restrict__ z) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t row = idx / y_ld;
  int c = (int)(idx - row * y_ld);
  if (row >= P) return;
  float v = 0.f;
  if (c == 0) v = ub ? ub[row * ld_ub] * sgn[row] * inv_scale : 0.f;
  else if (c < d_out) v = fb ? fb[row * ld_fb + c - 1] : 0.f;
  z[row * y_ld + c] = v;
}

// Upstream gradient of the last layer, split: zf[:, j] = feat_bar[:, j] (features, ld = F) and z0 = sgn * udf_bar / scale (udf head);
// a null pointer stands for a zero gradient
__global__ void zlast_split_kernel(const float* __restrict__ ub, int64_t ld_ub, const float* __restrict__ fb, int64_t ld_fb,
                                   const float* __restrict__ sgn, float inv_scale, int F, int64_t P, float* __restrict__ zf,
                                   float* __restrict__ z0, int t128 = 0) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t row = idx / (F + 1);
  int c = (int)(idx - row * (F + 1));
  if (row >= P) return;
  if (c == 0) z0[row] = ub ? ub[row * ld_ub] * sgn[row] * inv_scale : 0.f;
  else zf[mat_off(t128 != 0, row, c - 1, F)] = fb ? fb[row * ld_fb + c - 1] : 0.f;
}

// Tiled versions for the T128 layout (fused chains): a CTA moves a 128-point x 32-column tile through shared memory so that
// BOTH sides are coalesced -- 16-byte accesses with the points innermost on the T128 side, 128-byte column runs on the row-major
// side (the torch-facing [P, 257] tensors: odd width, no vector access possible).  grid = (point tiles, column tiles).
// udf <- |y0| / scale, feat <- y[1:]  (separate leading dimensions);  sgn <- sign(y0)
__global__ void __launch_bounds__(256) udf_finalize_t128_kernel(const float* __restrict__ y, int y_ld, int d_out, int64_t P, float inv_scale,
                                                               float* __restrict__ udf, int64_t ld_u, float* __restrict__ feat, int64_t ld_f,
                                                               float* __restrict__ sgn) {
  __shared__ float tile[128][33];
  const int64_t r0 = (int64_t)blockIdx.x * 128;
  const int c0 = blockIdx.y * 32;
  const int t = threadIdx.x;
  {
    const int r = t & 127;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int q = (t >> 7) + 2 * k;                       // column quad of the tile
      const int c = c0 + 4 * q;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + r < P && c < y_ld) v = *reinterpret_cast<const float4*>(y + t128_off(r0 + r, c, y_ld));
      tile[r][4 * q + 0] = v.x; tile[r][4 * q + 1] = v.y; tile[r][4 * q + 2] = v.z; tile[r][4 * q + 3] = v.w;
    }
  }
  __syncthreads();
  const int cc = t & 31;
#pragma unroll 4
  for (int k = 0; k < 16; ++k) {
    const int r = (t >> 5) + 8 * k;
    const int64_t row = r0 + r;
    const int c = c0 + cc;
    if (row < P && c < d_out) {
      float v = tile[r][cc];
      if (c == 0) {
        if (sgn) sgn[row] = (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f);
        if (udf) udf[row * ld_u] = fabsf(v) * inv_scale;
      } else if (feat) {
        feat[row * ld_f + c - 1] = v;
      }
    }
  }
}
// zf[:, j] (T128, ld F) <- feat_bar[:, j];  z0 <- sgn * udf_bar / scale  (null = zero gradient)
__global__ void __launch_bounds__(256) zlast_split_t128_kernel(const float* __restrict__ ub, int64_t ld_ub, const float* __restrict__ fb,
                                                              int64_t ld_fb, const float* __restrict__ sgn, float inv_scale, int F, int64_t P,
                                                              float* __restrict__ zf, float* __restrict__ z0) {
  __shared__ float tile[128][33];
  const int64_t r0 = (int64_t)blockIdx.x * 128;
  const int c0 = blockIdx.y * 32;                           // feature columns [c0, c0 + 32) of zf = columns 1 + c0 .. of ob
  const int t = threadIdx.x;
  const int cc = t & 31;
#pragma unroll 4
  for (int k = 0; k < 16; ++k) {
    const int r = (t >> 5) + 8 * k;
    const int64_t row = r0 + r;
    float v = 0.f;
    if (fb != nullptr && row < P && c0 + cc < F) v = fb[row * ld_fb + c0 + cc];
    tile[r][cc] = v;
    if (blockIdx.y == 0 && cc == 0 && row < P) z0[row] = ub ? ub[row * ld_ub] * sgn[row] * inv_scale : 0.f;
  }
  __syncthreads();
  const int r = t & 127;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int q = (t >> 7) + 2 * k;
    const int c = c0 + 4 * q;
    if (r0 + r < P && c < F)
      *reinterpret_cast<float4*>(zf + t128_off(r0 + r, c, F)) = make_float4(tile[r][4 * q], tile[r][4 * q + 1], tile[r][4 * q + 2], tile[r][4 * q + 3]);
  }
}

static inline unsigned nblk(int64_t n, int t) { return (unsigned)cdiv(n, t); }

// ---- host orchestration -----------------------------------------------------------------------------------------

static int fold_all(const UdfPlan& p, const nudf_udf_desc* d, float* wfold, cudaStream_t st) {
  {
    FoldJobs jobs;
    jobs.n = p.n_lin;
    for (int l = 0; l < p.n_lin; ++l)
      jobs.j[l] = FoldJob{d->weight_g[l], d->weight_v[l], nullptr, nullptr, nullptr, wfold + p.w_off[l], p.out_dim[l], p.in_dim[l], (int)p.w_ld[l]};
    if (int rc = run_fold_jobs(jobs, false, st)) return rc;
  }
  if (get_engine() == 1) {
    uint16_t* img = reinterpret_cast<uint16_t*>(wfold + p.w_total);
    const int last = p.n_lin - 1;
    if (!(fused_fr_on(p) && fused_tb_on(p))) {      // split-bf16 images of the layer-by-layer tensor kernels (gemm_tc.cuh)
      for (int l = 0; l < p.n_lin; ++l) {
        if (int rc = tc::prep_weights(wfold + p.w_off[l], p.w_ld[l], p.out_dim[l], p.in_dim[l], 0, 2, img + p.img_nt[l], st)) return rc;
        if (int rc = tc::prep_weights(wfold + p.w_off[l], p.w_ld[l], p.in_dim[l], p.out_dim[l], 1, 2, img + p.img_nn[l], st)) return rc;
        if (int rc = tc::prep_weights(wfold + p.w_off[l], p.w_ld[l], p.out_dim[l], p.in_dim[l], 0, 3, img + p.img_nt3[l], st)) return rc;
      }
      if (p.d_out > 1)
        if (int rc = tc::prep_weights(wfold + p.w_off[last] + p.w_ld[last], p.w_ld[last], p.in_dim[last], p.d_out - 1, 1, 2, img + p.img_nn1, st))
          return rc;
    }
    if (p.chain_ok) {
      // fused chains (udf_chain.cuh): exact fp16 slice images of W_l as the X W^T operand of the F chain (one power-of-two
      // scale per layer, bias tables) and split-bf16 images for the R / B chains (dY W operand) and the T chain (X W^T) --
      // gradient quantities: 2^-16 relative is far inside their tolerance, 3 products.  Two launches for all layers.
      float* tab = wfold + p.w_total + p.img_total / 2;     // per layer: [4 floats of scale meta | bias table]
      chain::PrepJobs jobs;
      jobs.n = 0;
      auto add = [&](const float* W, int64_t ldw, const float* bias, int N, int K, int transposed, const float* meta, uint16_t* im,
                     float* bias_tab, int split) {
        jobs.j[jobs.n++] = chain::PrepJob{W, bias, meta, im, bias_tab, (int)ldw, N, K, transposed, split};
      };
      chain::ScaleJobs sj;
      sj.n = p.n_lin;
      for (int l = 0; l < p.n_lin; ++l) {
        float* meta = tab + p.sb_off[l];
        const float* W = wfold + p.w_off[l];
        sj.j[l] = chain::ScaleJob{W, meta, (int)p.w_ld[l], p.out_dim[l], p.in_dim[l]};
        add(W, p.w_ld[l], d->bias[l], p.out_dim[l], p.in_dim[l], 0, meta, img + p.img_chain[l], meta + 4, 0);
        if (l < last) {
          add(W, p.w_ld[l], nullptr, p.in_dim[l], p.out_dim[l], 1, meta, img + p.img_chain_nn[l], nullptr, 1);
          add(W, p.w_ld[l], nullptr, p.out_dim[l], p.in_dim[l], 0, meta, img + p.img_chain_t[l], nullptr, 1);
        } else if (p.d_out > 1) {
          add(W + p.w_ld[l], p.w_ld[l], nullptr, p.in_dim[l], p.d_out - 1, 1, meta, img + p.img_chain_nn1, nullptr, 1);
        }
      }
      if (int rc = chain::run_prep_jobs(sj, jobs, st)) return rc;
    }
  }
  return 0;
}

static inline const uint16_t* img_base(const UdfPlan& p, const float* wfold) {
  return reinterpret_cast<const uint16_t*>(wfold + p.w_total);
}

// ---- fused chains (udf_chain.cuh): step lists -------------------------------------------------------------------------
static chain::ChainStep* add_step(chain::ChainParams* cp, int kind) {
  chain::ChainStep* S = &cp->S[cp->n_steps++];
  memset(S, 0, sizeof(*S));
  S->kind = kind;
  S->post_scale = 1.0f;
  S->a_unscale = 1.0f;
  return S;
}
static void set_gemm(chain::ChainStep* S, const UdfPlan& p, const float* wfold, int layer, int K, int N, int64_t img_off) {
  const float* tab = wfold + p.w_total + p.img_total / 2;
  S->K = K; S->N = N; S->img_N = N;
  S->n_kslices = tc::pad64(K) / 64;
  S->n_tiles = chain::ch_n_tiles(N);
  S->img_off = (uint32_t)img_off;
  S->n_wpl = chain::kind_exact(S->kind) ? 3 : 2;
  S->wscale = tab + p.sb_off[layer] + 1;
}
static void chain_common(const UdfPlan& p, const float* wfold, const float* pts, int64_t P, chain::ChainParams* cp) {
  cp->n_steps = 0;
  cp->img = img_base(p, wfold);
  cp->pts = pts; cp->P = P; cp->scale = p.scale; cp->n_freq = p.L; cp->d_pe = p.d_pe;
  cp->gbar = nullptr;
  cp->pe_src = nullptr; cp->pe_ld = p.stash_ld; cp->pe_cta = 1;
  cp->pe_sh = (p.skip >= 1) ? (p.out_dim[p.skip - 1] & 7) : 0;
  cp->t128 = fused_on(p) ? 1 : 0;
  cp->udf_out = nullptr; cp->inv_scale = 1.0f / p.scale;
  cp->trace = nullptr;
}
// F chain for P points; value_only (udf != null): the last layer is restricted to its udf-head row and only udf[P] is
// written; otherwise the context tensors E0, A[1..], Y are written.  with_rev: the R chain (exact grad_x udf) follows in the
// same launch and writes D[0..last-1], Gpe, Ge.
static void build_forward(const UdfPlan& p, const float* wfold, const float* pts, int64_t P, float* ctx, const UdfCtx* c, float* udf,
                          bool with_rev, chain::ChainParams* cp) {
  const bool value_only = udf != nullptr;
  const float* tab = wfold + p.w_total + p.img_total / 2;
  const int last = p.n_lin - 1;
  chain_common(p, wfold, pts, P, cp);
  cp->udf_out = udf;
  chain::ChainStep* S = add_step(cp, chain::ST_PE);
  S->n_next = p.d_pe;
  // E0 is written for the weight gradients and re-read by the skip layer; a value-only launch keeps a 128-row stash per CTA in
  // `ctx` (= the caller's work buffer) instead, in the T128 layout
  // E0 is written for the weight gradients; the skip layer re-reads the encoding from a per-CTA stash (128 rows per CTA, T128,
  // columns shifted by pe_sh so that the appended columns are octet-aligned).  Value-only: `ctx` = the caller's work buffer.
  if (!value_only) { S->out0 = ctx + c->e0; S->ld_out0 = p.pe_ld; }
  if (p.skip >= 1) cp->pe_src = value_only ? ctx : ctx + c->stash;
  if (value_only) cp->t128 = 1;                             // no [P, ld] tensor is touched: take the fast paths
  for (int l = 0; l < last; ++l) {
    S = add_step(cp, chain::ST_FWD);
    set_gemm(S, p, wfold, l, p.in_dim[l], p.out_dim[l], p.img_chain[l]);
    S->bias = tab + p.sb_off[l] + 4;
    S->n_next = p.in_dim[l + 1];
    S->post_scale = (l + 1 == p.skip) ? NUDF_SQRT1_2 : 1.0f;
    if (!value_only) { S->out0 = ctx + c->a[l + 1]; S->ld_out0 = p.a_ld[l + 1]; }
  }
  S = add_step(cp, chain::ST_FWD_LAST);
  set_gemm(S, p, wfold, last, p.in_dim[last], value_only ? 1 : p.out_dim[last], p.img_chain[last]);
  S->bias = tab + p.sb_off[last] + 4;
  if (value_only) { S->rows_override = 16; S->img_N = p.out_dim[last]; }
  else { S->out0 = ctx + c->y; S->ld_out0 = p.y_ld; }
  if (!with_rev) return;
  auto rev_common = [&](chain::ChainStep* R, int l) {       // epilogue that turns G (w.r.t. A[l]) into D[l-1]
    R->n_main = p.out_dim[l - 1];
    R->n_next = R->n_main;
    R->post_scale = (l == p.skip) ? NUDF_SQRT1_2 : 1.0f;
    R->a_unscale = (l == p.skip) ? 1.41421356237309504880f : 1.0f;
    R->in0 = ctx + c->a[l]; R->ld_in0 = p.a_ld[l];
    R->out0 = ctx + c->d[l - 1]; R->ld_out0 = p.o_ld[l - 1];
    if (l == p.skip) { R->out1 = ctx + c->gpe; R->ld_out1 = p.stash_ld; }     // stored shifted by pe_sh columns; pe_vjp_kernel adds it
  };
  S = add_step(cp, chain::ST_REV_SEED);                     // G_last = (sgn / scale) W_last[0, :]
  S->N = p.in_dim[last];
  S->vec0 = wfold + p.w_off[last];
  S->sync_before = 1;
  rev_common(S, last);
  for (int l = last - 1; l >= 1; --l) {
    S = add_step(cp, chain::ST_REV);
    set_gemm(S, p, wfold, l, p.out_dim[l], p.in_dim[l], p.img_chain_nn[l]);
    rev_common(S, l);
  }
  S = add_step(cp, chain::ST_REV_FINAL);
  set_gemm(S, p, wfold, 0, p.out_dim[0], p.in_dim[0], p.img_chain_nn[0]);
  S->out0 = ctx + c->ge; S->ld_out0 = p.pe_ld;
}

// T chain (tangent, needs grad_bar) followed by the B chain (backward) in one launch.  Tensors: ctx (read): E0, A[l], D[l];
// scratch: Edot, Adot[l] (written by T, read later by the weight gradients), Q[l] (written by T, turned into Zbar[l] in place by
// B), zf / z0 (the split upstream gradient of the last layer, zlast_split_kernel).  with_t = false: Q was zero-filled.
static void build_backward(const UdfPlan& p, const float* wfold, const float* pts, int64_t P, const float* grad_bar, float* ctx,
                           const UdfCtx& c, float* scr, const UdfScratch& s, const float* zf, const float* z0, bool with_t,
                           chain::ChainParams* cp) {
  const int last = p.n_lin - 1;
  const int F = p.d_out - 1;
  chain_common(p, wfold, pts, P, cp);
  cp->gbar = grad_bar;
  chain::ChainStep* S;
  if (with_t) {
    S = add_step(cp, chain::ST_EDOT);
    S->n_next = p.d_pe;
    S->out0 = scr + s.edot; S->ld_out0 = p.pe_ld;
    if (p.skip >= 1) cp->pe_src = scr + s.stash;
    for (int l = 0; l < last; ++l) {
      S = add_step(cp, chain::ST_TAN);
      set_gemm(S, p, wfold, l, p.in_dim[l], p.out_dim[l], p.img_chain_t[l]);
      S->n_main = p.in_dim[l + 1];                          // width of Adot[l+1] (incl. the Edot columns at the skip layer)
      S->n_next = (l + 1 < last) ? p.in_dim[l + 1] : 0;     // Adot[last] feeds no GEMM (only a weighted column sum)
      S->post_scale = (l + 1 == p.skip) ? NUDF_SQRT1_2 : 1.0f;
      S->a_unscale = (l + 1 == p.skip) ? 1.41421356237309504880f : 1.0f;
      S->in0 = ctx + c.a[l + 1]; S->ld_in0 = p.a_ld[l + 1];
      S->in1 = ctx + c.d[l]; S->ld_in1 = p.o_ld[l];
      S->out0 = scr + s.q[l]; S->ld_out0 = p.o_ld[l];
      S->out1 = scr + s.adot_l[l + 1]; S->ld_out1 = p.a_ld[l + 1];
    }
  }
  S = add_step(cp, chain::ST_LOAD);                         // operand of the first B GEMM: the feature part of out_bar
  S->n_next = F;
  S->in0 = zf; S->ld_in0 = F;
  S->sync_before = 1;
  auto bwd_common = [&](chain::ChainStep* B, int l) {       // Abar (w.r.t. A[l]) -> Zbar[l-1] = Abar S_{l-1} + Q[l-1], in place over Q
    B->n_main = p.out_dim[l - 1];
    B->n_next = (l - 1 >= 1) ? B->n_main : 0;               // Zbar[0] feeds no further GEMM
    B->post_scale = (l == p.skip) ? NUDF_SQRT1_2 : 1.0f;
    B->a_unscale = (l == p.skip) ? 1.41421356237309504880f : 1.0f;
    B->in0 = ctx + c.a[l]; B->ld_in0 = p.a_ld[l];
    B->in1 = scr + s.q[l - 1]; B->ld_in1 = p.o_ld[l - 1];
    B->out0 = scr + s.q[l - 1]; B->ld_out0 = p.o_ld[l - 1];
  };
  S = add_step(cp, chain::ST_BWD);                          // last layer: feature rows as a K = F contraction + rank-1 udf-head term
  set_gemm(S, p, wfold, last, F, p.in_dim[last], p.img_chain_nn1);
  S->rowv = z0;
  S->vec0 = wfold + p.w_off[last];
  bwd_common(S, last);
  for (int l = last - 1; l >= 1; --l) {
    S = add_step(cp, chain::ST_BWD);
    set_gemm(S, p, wfold, l, p.out_dim[l], p.in_dim[l], p.img_chain_nn[l]);
    bwd_common(S, l);
  }
}

static int value_chain(const UdfPlan& p, const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P,
                       float* ctx, const UdfCtx& c, cudaStream_t st) {
  if (p.chain_ok && tc_on(TC_FWD)) {            // one fused tcgen05 kernel for all layers (activations stay on chip)
    chain::ChainParams cp;
    build_forward(p, wfold, pts, P, ctx, &c, nullptr, false, &cp);
    return chain::launch_chain(cp, FAM_UDF_FWD_CHAIN, st);
  }
  float* e0 = ctx + c.e0;
  float* askip = nullptr; int askip_ld = 0, askip_col = 0;
  if (p.skip >= 1) { askip = ctx + c.a[p.skip]; askip_ld = p.a_ld[p.skip]; askip_col = p.out_dim[p.skip - 1]; }
  pe_forward_kernel<<<nblk(P, 128), 128, 0, st>>>(pts, P, p.L, p.scale, e0, p.pe_ld, askip, askip_ld, askip_col);
  NUDF_LAUNCH_OK();
  for (int l = 0; l < p.n_lin; ++l) {
    const float* A = l == 0 ? e0 : ctx + c.a[l];
    int64_t lda = l == 0 ? p.pe_ld : p.a_ld[l];
    const float* W = wfold + p.w_off[l];
    int rc;
    if (l < p.n_lin - 1) {
      EpiAct epi{ctx + c.a[l + 1], p.a_ld[l + 1], d->bias[l], ACT_SOFTPLUS100, (l + 1 == p.skip) ? NUDF_SQRT1_2 : 1.0f};
      rc = gemm_nt(A, lda, W, p.w_ld[l], P, p.out_dim[l], p.in_dim[l], epi, st, img_base(p, wfold) + p.img_nt3[l], TC_FWD, 3);
    } else {
      // the last layer always runs on the exact-fp32 engine: its row 0 is the udf head
      EpiAct epi{ctx + c.y, p.y_ld, d->bias[l], ACT_NONE, 1.0f};
      rc = gemm_nt(A, lda, W, p.w_ld[l], P, p.out_dim[l], p.in_dim[l], epi, st);
    }
    if (rc) return rc;
  }
  return 0;
}

// Reverse sweep with D[l] carried as plane tensors: every GEMM fetches its A operand with cp.async.bulk (gemm_wrp_kernel).
static int reverse_chain_planes(const UdfPlan& p, const float* wfold, const float* pts, int64_t P, float* ctx, const UdfCtx& c,
                                float* grad, cudaStream_t st) {
  const int last = p.n_lin - 1;
  uint16_t* pla = plane_area(ctx, c.pl_off);
  auto dpl = [&](int l) { return tc::Planes{pla + c.dpl[l], cb_of(p.out_dim[l])}; };
  auto make_rev = [&](int l) {
    EpiRevP e;
    e.n_main = p.out_dim[l - 1];
    e.post_scale = (l == p.skip) ? NUDF_SQRT1_2 : 1.0f;
    e.Anext = ctx + c.a[l]; e.lda = p.a_ld[l]; e.a_unscale = (l == p.skip) ? 1.41421356237309504880f : 1.0f;
    e.dpl = dpl(l - 1);
    e.Gpe = (l == p.skip) ? ctx + c.gpe : nullptr; e.ldg = p.pe_ld;
    return e;
  };
  for (int l = 0; l < last; ++l)                      // rows [P, round_up(P, 64)) are part of the weight-gradient contraction
    if (int rc = tc::zero_pad_rows(P, dpl(l), st)) return rc;
  {
    EpiRevP e = make_rev(last);
    int cols4 = (p.in_dim[last] + 3) / 4;
    rev_init_kernel<EpiRevP><<<nblk(P * cols4, 256), 256, 0, st>>>(ctx + c.sgn, wfold + p.w_off[last], p.in_dim[last], 1.0f / p.scale, P, e);
    NUDF_LAUNCH_OK();
  }
  for (int l = last - 1; l >= 1; --l) {
    EpiRevP e = make_rev(l);
    if (int rc = tc::gemm_wrp(dpl(l), P, p.in_dim[l], p.out_dim[l], img_base(p, wfold) + p.img_nn[l], e, st)) return rc;
  }
  {
    EpiRevFinal e{ctx + c.ge, p.pe_ld, p.skip >= 1 ? ctx + c.gpe : nullptr, p.pe_ld};
    if (int rc = tc::gemm_wrp(dpl(0), P, p.in_dim[0], p.out_dim[0], img_base(p, wfold) + p.img_nn[0], e, st)) return rc;
  }
  pe_vjp_kernel<<<nblk(P, 128), 128, 0, st>>>(pts, ctx + c.ge, p.pe_ld, P, p.L, p.scale, grad);
  NUDF_LAUNCH_OK();
  return 0;
}

static int reverse_chain(const UdfPlan& p, const float* wfold, const float* pts, int64_t P, float* ctx, const UdfCtx& c,
                         float* grad, cudaStream_t st) {
  if (chain_planes_on()) return reverse_chain_planes(p, wfold, pts, P, ctx, c, grad, st);
  const int last = p.n_lin - 1;
  auto make_rev = [&](int l) {  // epilogue that turns G (wrt A[l]) into D[l-1]
    EpiRev e;
    e.n_main = p.out_dim[l - 1];
    e.post_scale = (l == p.skip) ? NUDF_SQRT1_2 : 1.0f;
    e.Anext = ctx + c.a[l]; e.lda = p.a_ld[l]; e.a_unscale = (l == p.skip) ? 1.41421356237309504880f : 1.0f;
    e.Dprev = ctx + c.d[l - 1]; e.ldd = p.o_ld[l - 1];
    e.Gpe = (l == p.skip) ? ctx + c.gpe : nullptr; e.ldg = p.pe_ld;
    return e;
  };
  {
    EpiRev e = make_rev(last);
    int cols4 = (p.in_dim[last] + 3) / 4;
    rev_init_kernel<EpiRev><<<nblk(P * cols4, 256), 256, 0, st>>>(ctx + c.sgn, wfold + p.w_off[last], p.in_dim[last],
                                                                  1.0f / p.scale, P, e);
    NUDF_LAUNCH_OK();
  }
  for (int l = last - 1; l >= 1; --l) {
    EpiRev e = make_rev(l);
    int rc = gemm_nn(ctx + c.d[l], p.o_ld[l], wfold + p.w_off[l], p.w_ld[l], P, p.in_dim[l], p.out_dim[l], e, st,
                     img_base(p, wfold) + p.img_nn[l], TC_REV);
    if (rc) return rc;
  }
  {
    EpiRevFinal e{ctx + c.ge, p.pe_ld, p.skip >= 1 ? ctx + c.gpe : nullptr, p.pe_ld};
    int rc = gemm_nn(ctx + c.d[0], p.o_ld[0], wfold + p.w_off[0], p.w_ld[0], P, p.in_dim[0], p.out_dim[0], e, st,
                     img_base(p, wfold) + p.img_nn[0], TC_REV);
    if (rc) return rc;
  }
  pe_vjp_kernel<<<nblk(P, 128), 128, 0, st>>>(pts, ctx + c.ge, p.pe_ld, P, p.L, p.scale, grad);
  NUDF_LAUNCH_OK();
  return 0;
}

}  // namespace nudf

using namespace nudf;

extern "C" {

int64_t nudf_udf_folded_floats(const nudf_udf_desc* d) {
  UdfPlan p;
  if (make_plan(d, &p)) return -1;
  return p.w_total + p.img_total / 2 + p.sb_total;   // fp32 folded weights, the 16-bit weight images (2 per float), the chain's (scale, bias) tables
}

int nudf_udf_fold_weights(const nudf_udf_desc* d, float* wfold, void* stream) {
  UdfPlan p;
  if (int rc = make_plan(d, &p)) return rc;
  NUDF_REQUIRE(wfold != nullptr, "null wfold");
  cudaStream_t st = (cudaStream_t)stream;
  return fold_all(p, d, wfold, st);
}

int64_t nudf_udf_ctx_floats(const nudf_udf_desc* d, int64_t P, int with_grad) {
  UdfPlan p;
  if (make_plan(d, &p)) return -1;
  UdfCtx c;
  ctx_layout(p, P, with_grad, &c);
  return c.total;
}

int64_t nudf_udf_scratch_floats(const nudf_udf_desc* d, int64_t P) {
  UdfPlan p;
  if (make_plan(d, &p)) return -1;
  UdfScratch s;
  scratch_layout(p, P, &s);
  return s.total;
}

static int udf_forward_impl(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, float* udf, int64_t ld_u, float* feat,
                            int64_t ld_f, float* grad, float* ctx, void* stream) {
  UdfPlan p;
  if (int rc = make_plan(d, &p)) return rc;
  if (P <= 0) return 0;
  NUDF_REQUIRE(wfold && pts && ctx, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  UdfCtx c;
  ctx_layout(p, P, grad != nullptr, &c);
  if (grad != nullptr && fused_fr_on(p)) {
    // value chain + reverse sweep of every 128-point tile in ONE launch (udf_chain.cuh): writes E0, A[l], Y, D[l], Gpe, Ge
    chain::ChainParams cp;
    build_forward(p, wfold, pts, P, ctx, &c, nullptr, true, &cp);
    if (int rc = chain::launch_chain(cp, FAM_UDF_FWD_CHAIN, st)) return rc;
    udf_finalize_t128_kernel<<<dim3(nblk(P, 128), nblk(p.d_out, 32)), 256, 0, st>>>(ctx + c.y, p.y_ld, p.d_out, P, 1.0f / p.scale, udf, ld_u,
                                                                                    feat, ld_f, ctx + c.sgn);
    NUDF_LAUNCH_OK();
    pe_vjp_kernel<<<nblk(P, 128), 128, 0, st>>>(pts, ctx + c.ge, p.pe_ld, P, p.L, p.scale, grad, 1, p.skip >= 1 ? ctx + c.gpe : nullptr,
                                                p.stash_ld, p.skip >= 1 ? (p.out_dim[p.skip - 1] & 7) : 0);
    NUDF_LAUNCH_OK();
    return 0;
  }
  if (int rc = value_chain(p, d, wfold, pts, P, ctx, c, st)) return rc;
  udf_finalize_kernel<<<nblk(P * p.d_out, 256), 256, 0, st>>>(ctx + c.y, p.y_ld, p.d_out, P, 1.0f / p.scale, udf, ld_u, feat, ld_f,
                                                              ctx + c.sgn, fused_on(p) ? 1 : 0);
  NUDF_LAUNCH_OK();
  if (grad) return reverse_chain(p, wfold, pts, P, ctx, c, grad, st);
  return 0;
}

int nudf_udf_forward(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, float* out, int64_t ld_out,
                     float* grad, float* ctx, void* stream) {
  NUDF_REQUIRE(d != nullptr, "null descriptor");
  NUDF_REQUIRE(out == nullptr || ld_out >= d->d_out, "ld_out too small");
  return udf_forward_impl(d, wfold, pts, P, out, ld_out, out ? out + 1 : nullptr, ld_out, grad, ctx, stream);
}

int nudf_udf_forward_split(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, float* udf, float* feat,
                           int64_t ld_feat, float* grad, float* ctx, void* stream) {
  NUDF_REQUIRE(d != nullptr, "null descriptor");
  NUDF_REQUIRE(feat == nullptr || ld_feat >= d->d_out - 1, "ld_feat too small");
  return udf_forward_impl(d, wfold, pts, P, udf, 1, feat, ld_feat, grad, ctx, stream);
}

int nudf_udf_value(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, float* udf, float* work,
                   void* stream) {
  UdfPlan p;
  if (int rc = make_plan(d, &p)) return rc;
  if (P <= 0) return 0;
  NUDF_REQUIRE(wfold && pts && udf, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  NUDF_REQUIRE(work != nullptr, "null pointer (work)");
  if (p.chain_ok && tc_on(TC_FWD)) {
    chain::ChainParams cp;
    build_forward(p, wfold, pts, P, work, nullptr, udf, false, &cp);     // work: per-CTA stash of the encoding (first ctx_rows x pe_ld floats)
    return chain::launch_chain(cp, FAM_UDF_FWD_CHAIN, st);
  }
  UdfCtx c;
  ctx_layout(p, P, 0, &c);
  // value-only: the last layer needs only its row 0 (the udf head); the 256 feature rows are skipped.
  UdfPlan pv = p;
  pv.out_dim[p.n_lin - 1] = 1;
  nudf_udf_desc dv = *d;
  if (int rc = value_chain(pv, &dv, wfold, pts, P, work, c, st)) return rc;
  udf_value_only_kernel<<<nblk(P, 256), 256, 0, st>>>(work + c.y, p.y_ld, P, 1.0f / p.scale, udf);
  NUDF_LAUNCH_OK();
  return 0;
}

static int udf_backward_impl(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, const float* ub, int64_t ld_ub,
                             const float* fb, int64_t ld_fb, const float* grad_bar, const float* ctx_c, float* scratch, float* dwfold,
                             float* dbias, void* stream);

int nudf_udf_backward(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, const float* out_bar,
                      int64_t ld_ob, const float* grad_bar, const float* ctx_c, float* scratch, float* dwfold,
                      float* dbias, void* stream) {
  return udf_backward_impl(d, wfold, pts, P, out_bar, ld_ob, out_bar ? out_bar + 1 : nullptr, ld_ob, grad_bar, ctx_c, scratch, dwfold, dbias,
                           stream);
}

int nudf_udf_backward_split(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, const float* udf_bar,
                            const float* feat_bar, int64_t ld_fb, const float* grad_bar, const float* ctx_c, float* scratch,
                            float* dwfold, float* dbias, void* stream) {
  return udf_backward_impl(d, wfold, pts, P, udf_bar, 1, feat_bar, ld_fb, grad_bar, ctx_c, scratch, dwfold, dbias, stream);
}

static int udf_backward_impl(const nudf_udf_desc* d, const float* wfold, const float* pts, int64_t P, const float* ub, int64_t ld_ub,
                             const float* fb, int64_t ld_fb, const float* grad_bar, const float* ctx_c, float* scratch, float* dwfold,
                             float* dbias, void* stream) {
  const bool out_bar = ub != nullptr || fb != nullptr;      // some upstream gradient of the value / feature outputs
  UdfPlan p;
  if (int rc = make_plan(d, &p)) return rc;
  NUDF_REQUIRE(wfold && dwfold && dbias, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  NUDF_CUDA_OK(cudaMemsetAsync(dwfold, 0, sizeof(float) * p.w_total, st));
  NUDF_CUDA_OK(cudaMemsetAsync(dbias, 0, sizeof(float) * p.b_total, st));
  if (P <= 0) return 0;
  NUDF_REQUIRE(pts && ctx_c && scratch, "null pointer");
  float* ctx = const_cast<float*>(ctx_c);  // read-only use
  UdfCtx c;
  ctx_layout(p, P, 1, &c);
  UdfScratch s;
  scratch_layout(p, P, &s);
  const int last = p.n_lin - 1;
  const int split = (int)cdiv(P, 2048);

  if (fused_tb_on(p)) {
    // ---- tangent + backward chains of every 128-point tile in ONE launch (udf_chain.cuh), then the weight gradients ----
    const int F = p.d_out - 1;
    float* zf = scratch + s.zlast;                  // [P, F] feature part of the upstream gradient of the last layer
    float* z0 = zf + ctx_rows(p, P) * F;            // [P]    udf-head part, times sgn / scale
    if (out_bar) {
      zlast_split_t128_kernel<<<dim3(nblk(P, 128), nblk(F, 32)), 256, 0, st>>>(ub, ld_ub, fb, ld_fb, ctx + c.sgn, 1.0f / p.scale, F, P, zf, z0);
      NUDF_LAUNCH_OK();
    } else {
      NUDF_CUDA_OK(cudaMemsetAsync(zf, 0, sizeof(float) * (ctx_rows(p, P) * F + P), st));
    }
    const bool with_t = grad_bar != nullptr;
    if (!with_t)
      for (int l = 0; l < last; ++l) NUDF_CUDA_OK(cudaMemsetAsync(scratch + s.q[l], 0, sizeof(float) * ctx_rows(p, P) * p.o_ld[l], st));
    {
      chain::ChainParams cp;
      build_backward(p, wfold, pts, P, grad_bar, ctx, c, scratch, s, zf, z0, with_t, &cp);
      if (int rc = chain::launch_chain(cp, FAM_UDF_BWD_CHAIN, st)) return rc;
    }
    if (with_t) {
      // g_last = W_last^T d_last with d_last = (sgn/scale) e_0  =>  dW_last[0,:] += sum_p (sgn/scale) Adot_last
      if (int rc = colsum(scratch + s.adot_l[last], p.a_ld[last], ctx + c.sgn, 1.0f / p.scale, P, p.in_dim[last], dwfold + p.w_off[last], st, true))
        return rc;
    }
    if (out_bar) {
      float* dWl = dwfold + p.w_off[last];
      EpiAtomicAdd ew{dWl + p.w_ld[last], p.w_ld[last]};
      if (int rc = gemm_tn(zf, F, ctx + c.a[last], p.a_ld[last], F, p.in_dim[last], P, ew, st, split, TC_WGRAD, dbias + p.b_off[last] + 1, true))
        return rc;
      if (int rc = colsum(ctx + c.a[last], p.a_ld[last], z0, 1.0f, P, p.in_dim[last], dWl, st, true)) return rc;
      if (int rc = colsum(z0, 1, nullptr, 1.0f, P, 1, dbias + p.b_off[last], st)) return rc;
    }
    // one launch per layer: dW_l += D_l^T Adot_l (tangent chain; Adot_0 = Edot)  +  Zbar_l^T A_l (backward chain), db_l = column
    // sums of Zbar_l -- both contractions share the accumulator and the split-K reduction
    for (int l = last - 1; l >= 0; --l) {
      tc::TnPair pr[2];
      int np = 0;
      if (with_t) pr[np++] = tc::TnPair{ctx + c.d[l], p.o_ld[l], l == 0 ? scratch + s.edot : scratch + s.adot_l[l], l == 0 ? p.pe_ld : p.a_ld[l], nullptr};
      pr[np++] = tc::TnPair{scratch + s.q[l], p.o_ld[l], l == 0 ? ctx + c.e0 : ctx + c.a[l], l == 0 ? p.pe_ld : p.a_ld[l], dbias + p.b_off[l]};
      EpiAtomicAdd ew{dwfold + p.w_off[l], p.w_ld[l]};
      if (int rc = gemm_tn_pairs(pr, np, p.out_dim[l], p.in_dim[l], P, ew, st)) return rc;
    }
    return 0;
  }

  // ---- tangent chain (second-order terms) ----
  if (grad_bar && chain_planes_on()) {
    // plane mode: D[l] (ctx) and Adot[l] (scratch) are split-bf16 plane tensors; the chain kernels and the weight gradients
    // fetch them with cp.async.bulk.  (A ctx filled without its gradient part never gets here: grad_bar is null then.)
    uint16_t* cpl = plane_area(ctx, c.pl_off);
    uint16_t* spl = plane_area(scratch, s.pl_off);
    auto dpl = [&](int l) { return tc::Planes{cpl + c.dpl[l], cb_of(p.out_dim[l])}; };
    auto adpl = [&](int l) { return tc::Planes{spl + s.adpl[l], cb_of(p.in_dim[l])}; };
    float* edot = scratch + s.edot;
    pe_jvp_kernel<<<nblk(P, 128), 128, 0, st>>>(pts, grad_bar, P, p.L, p.scale, edot, p.pe_ld);
    NUDF_LAUNCH_OK();
    if (int rc = tc::pack_planes(edot, p.pe_ld, P, p.d_pe, adpl(0), st)) return rc;
    for (int l = 1; l <= last; ++l)
      if (int rc = tc::zero_pad_rows(P, adpl(l), st)) return rc;
    float* adot_last = scratch + s.adot[0];                     // fp32 copy of Adot[last] for the weighted column sum
    for (int l = 0; l < last; ++l) {
      EpiAtomicAdd ew{dwfold + p.w_off[l], p.w_ld[l]};          // dW_l += D_l^T Adot_l
      if (int rc = gemm_tn_planes(dpl(l), p.out_dim[l], adpl(l), p.in_dim[l], P, ew, st)) return rc;
      EpiTanP et;
      et.Anext = ctx + c.a[l + 1]; et.lda = p.a_ld[l + 1];
      et.a_unscale = (l + 1 == p.skip) ? 1.41421356237309504880f : 1.0f;
      et.D = dpl(l);
      et.Q = scratch + s.q[l]; et.ldq = p.o_ld[l];
      et.npl = adpl(l + 1); et.post_scale = (l + 1 == p.skip) ? NUDF_SQRT1_2 : 1.0f;
      et.AdotNext = (l + 1 == last) ? adot_last : nullptr; et.ldn = p.a_ld[l + 1];
      if (int rc = tc::gemm_wrp(adpl(l), P, p.out_dim[l], p.in_dim[l], img_base(p, wfold) + p.img_nt[l], et, st)) return rc;
      if (l + 1 == p.skip) {
        copy_cols_planes_kernel<<<nblk(P * p.d_pe, 256), 256, 0, st>>>(edot, p.pe_ld, adpl(l + 1), p.out_dim[l], p.d_pe, P, NUDF_SQRT1_2);
        NUDF_LAUNCH_OK();
      }
    }
    if (int rc = colsum(adot_last, p.a_ld[last], ctx + c.sgn, 1.0f / p.scale, P, p.in_dim[last], dwfold + p.w_off[last], st)) return rc;
  } else if (grad_bar) {
    float* edot = scratch + s.edot;
    pe_jvp_kernel<<<nblk(P, 128), 128, 0, st>>>(pts, grad_bar, P, p.L, p.scale, edot, p.pe_ld);
    NUDF_LAUNCH_OK();
    const float* adot = edot;
    int64_t ld_adot = p.pe_ld;
    for (int l = 0; l < last; ++l) {
      // dW_l += D_l^T Adot_l
      EpiAtomicAdd ew{dwfold + p.w_off[l], p.w_ld[l]};
      if (int rc = gemm_tn(ctx + c.d[l], p.o_ld[l], adot, ld_adot, p.out_dim[l], p.in_dim[l], P, ew, st, split)) return rc;
      float* nxt = scratch + s.adot[l & 1];
      int64_t ld_nxt = p.a_ld[l + 1];
      EpiTan et;
      et.Anext = ctx + c.a[l + 1]; et.lda = p.a_ld[l + 1];
      et.a_unscale = (l + 1 == p.skip) ? 1.41421356237309504880f : 1.0f;
      et.D = ctx + c.d[l]; et.ldd = p.o_ld[l];
      et.Q = scratch + s.q[l]; et.ldq = p.o_ld[l];
      et.AdotNext = nxt; et.ldn = ld_nxt; et.post_scale = (l + 1 == p.skip) ? NUDF_SQRT1_2 : 1.0f;
      if (int rc = gemm_nt(adot, ld_adot, wfold + p.w_off[l], p.w_ld[l], P, p.out_dim[l], p.in_dim[l], et, st,
                           img_base(p, wfold) + p.img_nt[l], TC_TAN))
        return rc;
      if (l + 1 == p.skip) {
        copy_cols_kernel<<<nblk(P * p.d_pe, 256), 256, 0, st>>>(edot, p.pe_ld, nxt, ld_nxt, p.out_dim[l], p.d_pe, P,
                                                                 NUDF_SQRT1_2);
        NUDF_LAUNCH_OK();
      }
      adot = nxt; ld_adot = ld_nxt;
    }
    // g_last = W_last^T d_last with d_last = (sgn/scale) e_0  =>  dW_last[0,:] += sum_p (sgn/scale) Adot_last
    if (int rc = colsum(adot, ld_adot, ctx + c.sgn, 1.0f / p.scale, P, p.in_dim[last], dwfold + p.w_off[last], st)) return rc;
  }

  // ---- backward chain ----
  const bool has_q = grad_bar != nullptr;
  if (!has_q)
    for (int l = 0; l < last; ++l)
      NUDF_CUDA_OK(cudaMemsetAsync(scratch + s.q[l], 0, sizeof(float) * P * p.o_ld[l], st));
  float* zl = scratch + s.zlast;
  const int F = p.d_out - 1;
  const bool split_head = out_bar && tc_on(TC_BWD) && F >= 64 && (F % 4) == 0 && tc::pad64(F) <= 64 * tc::WR_MAX_SLICES;
  if (split_head) {
    // 257 = 1 udf-head row + 256 feature rows: the feature block is a K = 256 contraction for the weights-resident tensor
    // kernel, the head row a rank-1 update in its epilogue (and a weighted column sum for its weight gradient).
    float* zf = zl;
    float* z0 = zl + P * F;
    zlast_split_kernel<<<nblk(P * p.d_out, 256), 256, 0, st>>>(ub, ld_ub, fb, ld_fb, ctx + c.sgn, 1.0f / p.scale, F, P, zf, z0);
    NUDF_LAUNCH_OK();
    const float* Wl = wfold + p.w_off[last];
    float* dWl = dwfold + p.w_off[last];
    EpiAtomicAdd ew{dWl + p.w_ld[last], p.w_ld[last]};
    if (int rc = gemm_tn(zf, F, ctx + c.a[last], p.a_ld[last], F, p.in_dim[last], P, ew, st, split, TC_WGRAD, dbias + p.b_off[last] + 1))
      return rc;
    if (int rc = colsum(ctx + c.a[last], p.a_ld[last], z0, 1.0f, P, p.in_dim[last], dWl, st)) return rc;
    if (int rc = colsum(z0, 1, nullptr, 1.0f, P, 1, dbias + p.b_off[last], st)) return rc;
    EpiBwdR1 eb;
    eb.n_main = p.out_dim[last - 1]; eb.post_scale = (last == p.skip) ? NUDF_SQRT1_2 : 1.0f;
    eb.Anext = ctx + c.a[last]; eb.lda = p.a_ld[last]; eb.a_unscale = (last == p.skip) ? 1.41421356237309504880f : 1.0f;
    eb.QZ = scratch + s.q[last - 1]; eb.ldq = p.o_ld[last - 1];
    eb.z0 = z0; eb.w0 = Wl;
    if (int rc = gemm_nn(zf, F, Wl + p.w_ld[last], p.w_ld[last], P, p.in_dim[last], F, eb, st, img_base(p, wfold) + p.img_nn1, TC_BWD))
      return rc;
  } else if (out_bar) {
    zlast_kernel<<<nblk(P * p.y_ld, 256), 256, 0, st>>>(ub, ld_ub, fb, ld_fb, ctx + c.sgn, 1.0f / p.scale, p.d_out, p.y_ld, P, zl);
    NUDF_LAUNCH_OK();
    EpiAtomicAdd ew{dwfold + p.w_off[last], p.w_ld[last]};
    if (int rc = gemm_tn(zl, p.y_ld, ctx + c.a[last], p.a_ld[last], p.out_dim[last], p.in_dim[last], P, ew, st, split, TC_WGRAD,
                         dbias + p.b_off[last]))
      return rc;
    EpiBwd eb;
    eb.n_main = p.out_dim[last - 1]; eb.post_scale = (last == p.skip) ? NUDF_SQRT1_2 : 1.0f;
    eb.Anext = ctx + c.a[last]; eb.lda = p.a_ld[last]; eb.a_unscale = (last == p.skip) ? 1.41421356237309504880f : 1.0f;
    eb.QZ = scratch + s.q[last - 1]; eb.ldq = p.o_ld[last - 1];
    if (int rc = gemm_nn(zl, p.y_ld, wfold + p.w_off[last], p.w_ld[last], P, p.in_dim[last], p.out_dim[last], eb, st,
                         img_base(p, wfold) + p.img_nn[last], TC_BWD))
      return rc;
  }
  for (int l = last - 1; l >= 0; --l) {
    const float* zb = scratch + s.q[l];  // now holds Zbar_l
    const float* A = l == 0 ? ctx + c.e0 : ctx + c.a[l];
    int64_t lda = l == 0 ? p.pe_ld : p.a_ld[l];
    EpiAtomicAdd ew{dwfold + p.w_off[l], p.w_ld[l]};
    if (int rc = gemm_tn(zb, p.o_ld[l], A, lda, p.out_dim[l], p.in_dim[l], P, ew, st, split, TC_WGRAD, dbias + p.b_off[l])) return rc;
    if (l > 0) {
      EpiBwd eb;
      eb.n_main = p.out_dim[l - 1]; eb.post_scale = (l == p.skip) ? NUDF_SQRT1_2 : 1.0f;
      eb.Anext = ctx + c.a[l]; eb.lda = p.a_ld[l]; eb.a_unscale = (l == p.skip) ? 1.41421356237309504880f : 1.0f;
      eb.QZ = scratch + s.q[l - 1]; eb.ldq = p.o_ld[l - 1];
      if (int rc = gemm_nn(zb, p.o_ld[l], wfold + p.w_off[l], p.w_ld[l], P, p.in_dim[l], p.out_dim[l], eb, st,
                           img_base(p, wfold) + p.img_nn[l], TC_BWD))
        return rc;
    }
  }
  return 0;
}

int nudf_udf_unfold_grads(const nudf_udf_desc* d, const float* dwfold, float* const* dg, float* const* dv, void* stream) {
  UdfPlan p;
  if (int rc = make_plan(d, &p)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  FoldJobs jobs;
  jobs.n = p.n_lin;
  for (int l = 0; l < p.n_lin; ++l)
    jobs.j[l] = FoldJob{d->weight_g[l], d->weight_v[l], dwfold + p.w_off[l], dg[l], dv[l], nullptr, p.out_dim[l], p.in_dim[l], (int)p.w_ld[l]};
  return run_fold_jobs(jobs, true, st);
}

}  // extern "C"
