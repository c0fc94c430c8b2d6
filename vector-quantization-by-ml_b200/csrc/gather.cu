// gather.cu -- code gather + straight-through output + commitment loss in one pass over the latents,
// its backward, and the fused ResidualVQ level step.
//
// Replaces (reference file:line under vector_quantization/):
//   codebooks.py:393-397            one-hot einsum (2NKd flops) / batched_embedding gather
//   vector_quantize_pytorch.py:273  quantize = x + (quantize - x).detach()
//   vector_quantize_pytorch.py:347-364  F.mse_loss(commit_quantize, x) (masked variant included)
//   residual_vq.py:232-233          residual -= quantized ; quantized_out += quantized
// HBM-bound: per row read x (4d or 2d B) + idx (8 B), write q (4d B); codebook rows come from L2.
// One warp per row, float4 lanes, rows strided over a persistent grid; loss partials are reduced
// in a fixed order (warp shuffle -> per-block double -> single-block tree) so the loss is bitwise
// reproducible run to run.
#include "common.cuh"

namespace vqb {

constexpr int kGatherThreads = 256;

struct GatherLayout {
  size_t off_part;   // double[grid] partial sums of squared error
  size_t off_cnt;    // int64[grid]  rows used
  size_t total;
};
static int gather_grid(int64_t rows) {
  int64_t need = (rows + (kGatherThreads / 32) - 1) / (kGatherThreads / 32);
  int64_t cap = (int64_t)num_sms() * 8;
  return (int)(need < cap ? (need > 0 ? need : 1) : cap);
}
static GatherLayout gather_layout() {
  GatherLayout L;
  const size_t maxgrid = 148 * 8 * 4;   // generous upper bound on gather_grid()
  L.off_part = 0;
  L.off_cnt = align_up(maxgrid * 8);
  L.total = L.off_cnt + align_up(maxgrid * 8);
  return L;
}

// q = training ? fl(x + fl(c - x)) : c ; optional squared-error partials
template <typename T, bool kLoss>
__global__ void __launch_bounds__(kGatherThreads)
gather_st_loss_kernel(const T* __restrict__ x, const float* __restrict__ cb, const int64_t* __restrict__ idx,
                      const uint8_t* __restrict__ mask, int training, float* __restrict__ q, int64_t H, int64_t N,
                      int K, int d, double* __restrict__ part, long long* __restrict__ cntp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wpb = kGatherThreads / 32;
  const int64_t rows = H * N;
  float sq = 0.f;        // per-lane partial; one row contributes d/32 terms per lane
  double sqd = 0.0;      // folded into fp64 after every row
  long long used = 0;
  for (int64_t row = (int64_t)blockIdx.x * wpb + warp; row < rows; row += (int64_t)gridDim.x * wpb) {
    const int64_t h = row / N;
    const int64_t n = row - h * N;
    const int64_t code = idx[row];
    const bool in_loss = mask == nullptr || mask[n] != 0;
    const T* xr = x + row * (int64_t)d;
    const float* cr = cb + (h * K + code) * (int64_t)d;
    float* qr = q + row * (int64_t)d;
    sq = 0.f;
    if ((d & 7) == 0) {
      for (int j = lane * 8; j < d; j += 256) {
        const F8 xv = load8<T>(xr + j);
        const float4 c0 = __ldg(reinterpret_cast<const float4*>(cr + j)), c1 = __ldg(reinterpret_cast<const float4*>(cr + j) + 1);
        const float cv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float df = __fsub_rn(cv[e], xv.v[e]);
          o[e] = training ? __fadd_rn(xv.v[e], df) : cv[e];
          if (kLoss) sq = fmaf(df, df, sq);
        }
        __stcs(reinterpret_cast<float4*>(qr + j), make_float4(o[0], o[1], o[2], o[3]));
        __stcs(reinterpret_cast<float4*>(qr + j) + 1, make_float4(o[4], o[5], o[6], o[7]));
      }
    } else if ((d & 3) == 0) {
      for (int j = lane * 4; j < d; j += 128) {
        const float4 xv = load4<T>(xr + j);
        const float4 cv = __ldg(reinterpret_cast<const float4*>(cr + j));
        const float4 df = make_float4(__fsub_rn(cv.x, xv.x), __fsub_rn(cv.y, xv.y), __fsub_rn(cv.z, xv.z),
                                      __fsub_rn(cv.w, xv.w));
        float4 o;
        if (training) o = make_float4(__fadd_rn(xv.x, df.x), __fadd_rn(xv.y, df.y), __fadd_rn(xv.z, df.z),
                                      __fadd_rn(xv.w, df.w));
        else o = cv;
        __stcs(reinterpret_cast<float4*>(qr + j), o);
        if (kLoss) { sq = fmaf(df.x, df.x, sq); sq = fmaf(df.y, df.y, sq); sq = fmaf(df.z, df.z, sq); sq = fmaf(df.w, df.w, sq); }
      }
    } else {
      for (int j = lane; j < d; j += 32) {
        const float xv = to_f32<T>(xr[j]);
        const float cv = cr[j];
        const float df = __fsub_rn(cv, xv);
        qr[j] = training ? __fadd_rn(xv, df) : cv;
        if (kLoss) sq = fmaf(df, df, sq);
      }
    }
    if (kLoss && in_loss) { sqd += (double)sq; if (lane == 0) ++used; }
  }
  if (kLoss) {
    sqd = warp_sum(sqd);
    __shared__ double s_sq[kGatherThreads / 32];
    __shared__ long long s_n[kGatherThreads / 32];
    if (lane == 0) { s_sq[warp] = sqd; s_n[warp] = used; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      long long c = 0;
      for (int i = 0; i < wpb; ++i) { t += s_sq[i]; c += s_n[i]; }
      part[blockIdx.x] = t;
      cntp[blockIdx.x] = c;
    }
  }
}

// Narrow rows (d = 8..128, a power of two): d/8 lanes per row, so a warp works on 32/(d/8) rows at a time instead of
// leaving most lanes idle (d = 64 with one row per warp moves 256 B per warp-level load and reached 28 % of HBM).
template <typename T, bool kLoss>
__global__ void __launch_bounds__(kGatherThreads)
gather_st_loss_narrow_kernel(const T* __restrict__ x, const float* __restrict__ cb, const int64_t* __restrict__ idx,
                             const uint8_t* __restrict__ mask, int training, float* __restrict__ q, int64_t H,
                             int64_t N, int K, int d, double* __restrict__ part, long long* __restrict__ cntp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wpb = kGatherThreads / 32;
  const int lpr = d >> 3, rpi = 32 / lpr;
  const int grp = lane / lpr, j = (lane - grp * lpr) * 8;
  const int64_t rows = H * N;
  double sqd = 0.0;
  long long used = 0;
  for (int64_t row0 = ((int64_t)blockIdx.x * wpb + warp) * rpi; row0 < rows; row0 += (int64_t)gridDim.x * wpb * rpi) {
    const int64_t row = row0 + grp;
    if (row >= rows) continue;
    const int64_t h = row / N, n = row - h * N;
    const int64_t code = idx[row];
    const bool in_loss = mask == nullptr || mask[n] != 0;
    const F8 xv = load8<T>(x + row * (int64_t)d + j);
    const float* cr = cb + (h * K + code) * (int64_t)d + j;
    const float4 c0 = __ldg(reinterpret_cast<const float4*>(cr)), c1 = __ldg(reinterpret_cast<const float4*>(cr) + 1);
    const float cv[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
    float o[8], sq = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float df = __fsub_rn(cv[e], xv.v[e]);
      o[e] = training ? __fadd_rn(xv.v[e], df) : cv[e];
      if (kLoss) sq = fmaf(df, df, sq);
    }
    float* qr = q + row * (int64_t)d + j;
    __stcs(reinterpret_cast<float4*>(qr), make_float4(o[0], o[1], o[2], o[3]));
    __stcs(reinterpret_cast<float4*>(qr) + 1, make_float4(o[4], o[5], o[6], o[7]));
    if (kLoss && in_loss) { sqd += (double)sq; if (j == 0) ++used; }
  }
  if (kLoss) {
    sqd = warp_sum(sqd);
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o2);
    __shared__ double s_sq[kGatherThreads / 32];
    __shared__ long long s_n[kGatherThreads / 32];
    if (lane == 0) { s_sq[warp] = sqd; s_n[warp] = used; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      long long c = 0;
      for (int i = 0; i < wpb; ++i) { t += s_sq[i]; c += s_n[i]; }
      part[blockIdx.x] = t;
      cntp[blockIdx.x] = c;
    }
  }
}

// fixed-order reduction of the per-block partials: loss_out[0] = sum / (rows_used * d), loss_out[1] = rows_used
__global__ void loss_finalize_kernel(const double* __restrict__ part, const long long* __restrict__ cntp, int nblocks,
                                     int d, float* __restrict__ loss_out) {
  __shared__ double s[256];
  __shared__ long long c[256];
  double t = 0.0;
  long long n = 0;
  for (int i = threadIdx.x; i < nblocks; i += 256) { t += part[i]; n += cntp[i]; }
  s[threadIdx.x] = t;
  c[threadIdx.x] = n;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { s[threadIdx.x] += s[threadIdx.x + o]; c[threadIdx.x] += c[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double denom = (double)c[0] * (double)d;
    loss_out[0] = denom > 0.0 ? (float)(s[0] / denom) : __int_as_float(0x7fc00000);   // torch: mean of empty = nan
    loss_out[1] = (float)c[0];
  }
}

// Rotation-trick transport of one row (Fifty et al., arXiv:2410.06424; upstream vector-quantize-pytorch `rotate_to`):
// with sx = max(|x|, 1e-6), sc = max(|c|, 1e-6), u = x / sx, q = c / sc, w = (u + q) / max(|u + q|, 1e-12) and
// lambda = |c| / sx, the gradient g of the rotated output becomes
//   T(g) = lambda (g - 2 (g.w) w + 2 (g.q) u) = lambda g - 2 lambda (g.w) / nw (u + q) + 2 lambda (g.q) u.
// The squared norms are accumulated in fp64: at |x_i| ~ 1e-20 the fp32 squares are below the normal range and lambda
// would lose digits.  |u + q| is summed from the elementwise sums (not expanded: that cancels on antiparallel rows).
struct RotCoef {
  float sx, sc;     // max(|x|, 1e-6), max(|c|, 1e-6)
  float rx, rc;     // RN(1 / sx), RN(1 / sc)
  float lam;        // lambda
  float a;          // coefficient of (u + q): -2 lambda (g.w) / nw
  float b;          // coefficient of u: 2 lambda (g.q)
};
// nx2 = |x|^2, nc2 = |c|^2 (fp64)
__device__ __forceinline__ RotCoef rot_scales(double nx2, double nc2) {
  const double nc = sqrt(nc2), sx = fmax(sqrt(nx2), 1e-6);
  RotCoef r;
  r.sx = (float)sx;
  r.sc = (float)fmax(nc, 1e-6);
  r.rx = __frcp_rn(r.sx);
  r.rc = __frcp_rn(r.sc);
  r.lam = (float)(nc / sx);
  r.a = r.b = 0.f;
  return r;
}
// v / s from r = RN(1/s) and one fma correction: the correctly rounded quotient (Markstein) for the normal-range
// operands met here, without the slow-path call of a general division
__device__ __forceinline__ float rot_div(float v, float s, float r) {
  const float q0 = __fmul_rn(v, r);
  return fmaf(fmaf(-q0, s, v), r, q0);
}
// u and q are correctly rounded quotients and u + q is formed without contraction, so a pair that is exactly
// antiparallel after normalisation (c = -2x, or opposite signs at d = 1) sums to 0 as it does in exact arithmetic, and
// w = 0 there, as F.normalize returns; the (u + q) term then vanishes whatever g.w rounds to.
// gx = g.x, gc = g.c, nw2 = |u + q|^2
__device__ __forceinline__ void rot_finish(RotCoef& r, float gx, float gc, float nw2) {
  const float nw = fmaxf(sqrtf(nw2), 1e-12f), rnw = __frcp_rn(nw);
  const float gq = rot_div(gc, r.sc, r.rc);
  const float gw = rot_div(__fadd_rn(rot_div(gx, r.sx, r.rx), gq), nw, rnw);
  r.a = nw2 > 0.f ? -2.f * r.lam * rot_div(gw, nw, rnw) : 0.f;
  r.b = 2.f * r.lam * gq;
}
__device__ __forceinline__ float rot_u(float xv, const RotCoef& r) { return rot_div(xv, r.sx, r.rx); }
__device__ __forceinline__ float rot_sum(float xv, float cv, const RotCoef& r) {
  return __fadd_rn(rot_div(xv, r.sx, r.rx), rot_div(cv, r.sc, r.rc));
}

// grad_x = grad_q + coef * grad_loss[0] * (x - c)   (rows with mask==0: grad_q only)
// kRot: grad_x = T(grad_q) + coef * grad_loss[0] * (x - c) on the rows with mask != 0 (T above), grad_q on the others.
template <typename T, bool kRot>
__global__ void __launch_bounds__(kGatherThreads)
st_commit_backward_kernel(const float* __restrict__ gq, const float* __restrict__ gl, const T* __restrict__ x,
                          const float* __restrict__ cb, const int64_t* __restrict__ idx,
                          const uint8_t* __restrict__ mask, float coef, float* __restrict__ gx, int64_t H, int64_t N,
                          int K, int d) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wpb = kGatherThreads / 32;
  const int64_t rows = H * N;
  const float s = coef * gl[0];
  for (int64_t row = (int64_t)blockIdx.x * wpb + warp; row < rows; row += (int64_t)gridDim.x * wpb) {
    const int64_t h = row / N, n = row - h * N;
    const bool in_loss = mask == nullptr || mask[n] != 0;
    const float sc = in_loss ? s : 0.f;
    const T* xr = x + row * (int64_t)d;
    const float* cr = cb + (h * K + idx[row]) * (int64_t)d;
    const float* gr = gq + row * (int64_t)d;
    float* o = gx + row * (int64_t)d;
    if (!kRot || !in_loss) {
      for (int j = lane; j < d; j += 32) o[j] = fmaf(sc, to_f32<T>(xr[j]) - cr[j], gr[j]);
      continue;
    }
    // pass 1: |x|^2, |c|^2 (fp64), g.x, g.c -- lane-strided partials, then a fixed butterfly over the warp
    double nx2 = 0.0, nc2 = 0.0;
    float gdx = 0.f, gdc = 0.f;
    for (int j = lane; j < d; j += 32) {
      const float xv = to_f32<T>(xr[j]), cv = cr[j], g = gr[j];
      nx2 = fma((double)xv, (double)xv, nx2);
      nc2 = fma((double)cv, (double)cv, nc2);
      gdx = fmaf(g, xv, gdx);
      gdc = fmaf(g, cv, gdc);
    }
    RotCoef rc = rot_scales(warp_sum(nx2), warp_sum(nc2));
    // pass 2: |u + q|^2 from the elementwise sums (the row is in L1 now)
    float nw2 = 0.f;
    for (int j = lane; j < d; j += 32) {
      const float e = rot_sum(to_f32<T>(xr[j]), cr[j], rc);
      nw2 = fmaf(e, e, nw2);
    }
    rot_finish(rc, warp_sum(gdx), warp_sum(gdc), warp_sum(nw2));
    for (int j = lane; j < d; j += 32) {
      const float xv = to_f32<T>(xr[j]), cv = cr[j];
      o[j] = fmaf(sc, xv - cv, fmaf(rc.b, rot_u(xv, rc), fmaf(rc.a, rot_sum(xv, cv, rc), rc.lam * gr[j])));
    }
  }
}

// One ResidualVQ level: gather + ST + loss + residual/out update + next level's fp16 operand & row stats.
// Lanes own float4 column groups {lane*4 + 128*t}; the new residual row stays in registers between the
// update pass and the scaled-fp16 conversion pass (d_pad <= 512 when the next operand is requested).
__global__ void __launch_bounds__(kGatherThreads)
rvq_level_kernel(const float* res_in, float* res_out, const float* __restrict__ cb, const int64_t* __restrict__ idx,
                 const uint8_t* __restrict__ mask, int training, int first, float* __restrict__ out,
                 float* __restrict__ qout, int64_t N, int K, int d, int dp, double* __restrict__ part,
                 long long* __restrict__ cntp, __half* __restrict__ next_xb, float* __restrict__ next_xinv,
                 uint32_t* __restrict__ next_scal, __half* __restrict__ next_xaug,
                 const float* __restrict__ next_chdr, float* __restrict__ next_xn2) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wpb = kGatherThreads / 32;
  double sqd = 0.0;
  long long used = 0;
  float max_n2 = 0.f, max_r2 = 0.f;
  const bool vec = (d & 3) == 0;
  for (int64_t row = (int64_t)blockIdx.x * wpb + warp; row < N; row += (int64_t)gridDim.x * wpb) {
    const bool live = mask == nullptr || mask[row] != 0;
    const float* rr = res_in + row * (int64_t)d;
    float* ro = res_out + row * (int64_t)d;
    const float* cr = cb + idx[row] * (int64_t)d;
    float* orow = out + row * (int64_t)d;
    float sq = 0.f, m = 0.f;
    float4 keep[4];                      // new residual, columns lane*4 + 128*t (t < 4 covers d_pad <= 512)
#pragma unroll
    for (int t = 0; t < 4; ++t) keep[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec) {
      // one float4 group of columns j..j+3; returns the new residual
      auto step = [&](int j) {
        const float4 r = *reinterpret_cast<const float4*>(rr + j);
        const float4 c = __ldg(reinterpret_cast<const float4*>(cr + j));
        const float4 df = make_float4(__fsub_rn(c.x, r.x), __fsub_rn(c.y, r.y), __fsub_rn(c.z, r.z), __fsub_rn(c.w, r.w));
        float4 qv;
        // masked-out positions return the layer input itself (vector_quantize_pytorch.py:415-418)
        if (!live) qv = r;
        else if (training) qv = make_float4(__fadd_rn(r.x, df.x), __fadd_rn(r.y, df.y), __fadd_rn(r.z, df.z), __fadd_rn(r.w, df.w));
        else qv = c;
        if (out) {                         // NULL: the caller sums the levels afterwards (vqb_rvq_replay_out)
          float4 o;
          if (first) o = make_float4(__fadd_rn(0.f, qv.x), __fadd_rn(0.f, qv.y), __fadd_rn(0.f, qv.z), __fadd_rn(0.f, qv.w));
          else {
            const float4 p = *reinterpret_cast<const float4*>(orow + j);
            o = make_float4(__fadd_rn(p.x, qv.x), __fadd_rn(p.y, qv.y), __fadd_rn(p.z, qv.z), __fadd_rn(p.w, qv.w));
          }
          *reinterpret_cast<float4*>(orow + j) = o;
        }
        const float4 rn = make_float4(__fsub_rn(r.x, qv.x), __fsub_rn(r.y, qv.y), __fsub_rn(r.z, qv.z), __fsub_rn(r.w, qv.w));
        *reinterpret_cast<float4*>(ro + j) = rn;
        if (qout) *reinterpret_cast<float4*>(qout + row * (int64_t)d + j) = qv;
        sq = fmaf(df.x, df.x, sq); sq = fmaf(df.y, df.y, sq); sq = fmaf(df.z, df.z, sq); sq = fmaf(df.w, df.w, sq);
        m = fmaxf(fmaxf(fmaxf(m, fabsf(rn.x)), fmaxf(fabsf(rn.y), fabsf(rn.z))), fabsf(rn.w));
        return rn;
      };
#pragma unroll
      for (int t = 0; t < 16; ++t) {
        const int j = lane * 4 + 128 * t;
        if (j >= d) break;
        const float4 rn = step(j);
        if (t < 4) keep[t] = rn;
      }
#pragma unroll 1
      for (int j = lane * 4 + 2048; j < d; j += 128) step(j);   // rows wider than 2048 (no next operand there)
    } else {
      for (int j = lane; j < d; j += 32) {
        const float r = rr[j], c = cr[j];
        const float df = __fsub_rn(c, r);
        const float qv = live ? (training ? __fadd_rn(r, df) : c) : r;
        if (out) orow[j] = first ? __fadd_rn(0.0f, qv) : __fadd_rn(orow[j], qv);
        const float rn = __fsub_rn(r, qv);
        ro[j] = rn;
        if (qout) qout[row * (int64_t)d + j] = qv;
        sq = fmaf(df, df, sq);
        m = fmaxf(m, fabsf(rn));
      }
    }
    sq = warp_sum(sq);
    if (live) { sqd += (double)sq; ++used; }
    if (next_xb) {
#pragma unroll
      for (int o2 = 16; o2 > 0; o2 >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o2));
      float s = pow2_scale(m);
      const float a = clamp_row_scale(s, next_chdr[4], next_chdr[5]);    // bias operand of the next level's search
      const float is = 1.f / s;
      if (lane == 0) {
        next_xinv[row] = a > 0.f ? is : -is;
        const uint32_t aa = (uint32_t)__half_as_ushort(__float2half_rn(a));
        *reinterpret_cast<uint4*>(next_xaug + row * 8) = make_uint4(aa | (aa << 16), aa, 0u, 0u);
      }
      __half* xo = next_xb + row * (int64_t)dp;
      float n2 = 0.f, r2 = 0.f;
      if (vec) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const int j = lane * 4 + 128 * t;
          if (j < dp) {
            const float4 v = keep[t];     // zero beyond d
            const __half2 h0 = __floats2half2_rn(v.x * s, v.y * s), h1 = __floats2half2_rn(v.z * s, v.w * s);
            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
            uint2 pk;
            pk.x = *reinterpret_cast<const uint32_t*>(&h0);
            pk.y = *reinterpret_cast<const uint32_t*>(&h1);
            *reinterpret_cast<uint2*>(xo + j) = pk;
            const float b0 = f0.x * is, b1 = f0.y * is, b2 = f1.x * is, b3 = f1.y * is;
            n2 += b0 * b0 + b1 * b1 + b2 * b2 + b3 * b3;
            const float e0 = v.x - b0, e1 = v.y - b1, e2 = v.z - b2, e3 = v.w - b3;
            r2 += e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
          }
        }
      } else {
        __syncwarp();                     // res_out row was just written by this warp: re-read it
        for (int j = lane; j < dp; j += 32) {
          const float v = j < d ? ro[j] : 0.f;
          const __half hv = __float2half_rn(v * s);
          const float back = __half2float(hv) * is;
          xo[j] = hv;
          n2 += back * back;
          r2 += (v - back) * (v - back);
        }
      }
      n2 = warp_sum(n2);
      r2 = warp_sum(r2);
      if (lane == 0) next_xn2[row] = row_norm2_bound(n2, r2);
      max_n2 = fmaxf(max_n2, n2);
      max_r2 = fmaxf(max_r2, r2);
    }
  }
  __shared__ double s_sq[kGatherThreads / 32];
  __shared__ long long s_n[kGatherThreads / 32];
  __shared__ float s_a[kGatherThreads / 32], s_b[kGatherThreads / 32];
  if (lane == 0) { s_sq[warp] = sqd; s_n[warp] = used; s_a[warp] = max_n2; s_b[warp] = max_r2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    long long c = 0;
    float a = 0.f, b = 0.f;
    for (int i = 0; i < wpb; ++i) { t += s_sq[i]; c += s_n[i]; a = fmaxf(a, s_a[i]); b = fmaxf(b, s_b[i]); }
    part[blockIdx.x] = t;
    cntp[blockIdx.x] = c;
    if (next_scal) {
      atomicMax(next_scal + kScalXMax, batch_bound_bits(a, dp));
      atomicMax(next_scal + kScalDxMax, batch_bound_bits(b, dp));
      if (blockIdx.x == 0) next_scal[kScalTwoQ] = __float_as_uint(next_chdr[4]);   // the 2^q these operands were built with
    }
  }
}

int launch_loss_finalize(const double* part, const long long* cntp, int nblocks, int d, float* loss_out,
                         cudaStream_t st) {
  loss_finalize_kernel<<<1, 256, 0, st>>>(part, cntp, nblocks, d, loss_out);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}


// Sum of the levels' outputs of a ResidualVQ forward, replayed from the input and the chosen codes with the very IEEE
// operations of the level kernels (residual_vq.py:232-233):
//   r_0 = x;  q_l = live ? (training_l ? fl(r_l + fl(c_l - r_l)) : c_l) : r_l;  out = fl(..fl(fl(0 + q_0) + q_1)..);
//   r_{l+1} = fl(r_l - q_l)
// The level passes then do not read-modify-write `out` (2 x 4d bytes per row and level): one pass at the end reads x
// and writes out once; the Q code rows per latent come from L2 (the codebooks of a ResidualVQ are small).
constexpr int kMaxReplayLevels = 32;
struct ReplayArgs {
  const float* cb[kMaxReplayLevels];        // (K,d) codebook each level GATHERED from (before its EMA refresh)
  const int64_t* idx[kMaxReplayLevels];     // (N,)
  int training[kMaxReplayLevels];
  int Q;
};
template <int VEC>     // float4 groups per lane: d <= 128 * VEC
__global__ void __launch_bounds__(kGatherThreads)
rvq_replay_out_kernel(const float* __restrict__ x, const uint8_t* __restrict__ mask, float* __restrict__ out,
                      int64_t N, int d, const __grid_constant__ ReplayArgs A) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wpb = kGatherThreads / 32;
  for (int64_t row = (int64_t)blockIdx.x * wpb + warp; row < N; row += (int64_t)gridDim.x * wpb) {
    const bool live = mask == nullptr || mask[row] != 0;
    float4 r[VEC], acc[VEC];
#pragma unroll
    for (int t = 0; t < VEC; ++t) {
      const int j = lane * 4 + 128 * t;
      r[t] = j < d ? __ldcs(reinterpret_cast<const float4*>(x + row * (int64_t)d + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
      acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // lane l fetches level l's code id: the Q index loads are in flight together, only the code rows are chained
    const long long my_k = lane < A.Q ? (long long)A.idx[lane][row] : 0ll;
    float4 cnext[VEC];                   // code row of the next level: loaded while this level is computed
    {
      const float* cr = A.cb[0] + __shfl_sync(0xffffffffu, my_k, 0) * (int64_t)d;
#pragma unroll
      for (int t = 0; t < VEC; ++t) {
        const int j = lane * 4 + 128 * t;
        cnext[t] = j < d ? __ldg(reinterpret_cast<const float4*>(cr + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    for (int l = 0; l < A.Q; ++l) {
      float4 ccur[VEC];
#pragma unroll
      for (int t = 0; t < VEC; ++t) ccur[t] = cnext[t];
      if (l + 1 < A.Q) {
        const float* cr = A.cb[l + 1] + __shfl_sync(0xffffffffu, my_k, l + 1) * (int64_t)d;
#pragma unroll
        for (int t = 0; t < VEC; ++t) {
          const int j = lane * 4 + 128 * t;
          if (j < d) cnext[t] = __ldg(reinterpret_cast<const float4*>(cr + j));
        }
      }
      const bool tr = A.training[l] != 0;
#pragma unroll
      for (int t = 0; t < VEC; ++t) {
        const int j = lane * 4 + 128 * t;
        if (j >= d) continue;
        const float4 c = ccur[t];
        const float4 v = r[t];
        float4 qv;
        if (!live) qv = v;
        else if (tr) qv = make_float4(__fadd_rn(v.x, __fsub_rn(c.x, v.x)), __fadd_rn(v.y, __fsub_rn(c.y, v.y)),
                                      __fadd_rn(v.z, __fsub_rn(c.z, v.z)), __fadd_rn(v.w, __fsub_rn(c.w, v.w)));
        else qv = c;
        const float4 p = acc[t];             // level 0: fl(0.0f + q), as the level kernels do
        acc[t] = make_float4(__fadd_rn(p.x, qv.x), __fadd_rn(p.y, qv.y), __fadd_rn(p.z, qv.z), __fadd_rn(p.w, qv.w));
        r[t] = make_float4(__fsub_rn(v.x, qv.x), __fsub_rn(v.y, qv.y), __fsub_rn(v.z, qv.z), __fsub_rn(v.w, qv.w));
      }
    }
#pragma unroll
    for (int t = 0; t < VEC; ++t) {
      const int j = lane * 4 + 128 * t;
      if (j < d) __stcs(reinterpret_cast<float4*>(out + row * (int64_t)d + j), acc[t]);
    }
  }
}


// Input gradient of a whole ResidualVQ forward (training, EMA codebooks) in ONE pass, replayed from the level-0 input
// and the chosen codes like rvq_replay_out_kernel.  Reference autograd through residual_vq.py:212-243 and
// vector_quantize_pytorch.py:273,335-362: every level's output is r_l + (q_l - r_l).detach() (identity Jacobian), the
// next residual subtracts a DETACHED quantity (identity again), so d out / d x = Q I, and the commitment loss of level
// l, mean((c_l - r_l)^2) over the live rows, contributes coef_l (r_l - c_l) with coef_l = g_loss_l w_l 2 / (rows_l d):
//   grad_x = Q g_out + sum_l live coef_l (r_l - c_l)        (c_l from the codebook as it was BEFORE level l's EMA step)
// kRot (rotation trick): each level's output is the rotation of r_l onto c_l instead, whose Jacobian is the transport
// T_l of st_commit_backward_kernel evaluated on (r_l, c_l) -- the identity on masked rows:
//   grad_x = sum_l T_l(g_out) + sum_l live coef_l (r_l - c_l)
struct BackwardArgs {
  ReplayArgs R;
  const float* coef;       // (Q) device
};
// r_{l+1} = fl(r_l - q_l) with q_l of vqb_rvq_level
__device__ __forceinline__ float4 rvq_next_residual(float4 v, float4 c, bool live, bool tr) {
  float4 qv;
  if (!live) qv = v;
  else if (tr) qv = make_float4(__fadd_rn(v.x, __fsub_rn(c.x, v.x)), __fadd_rn(v.y, __fsub_rn(c.y, v.y)),
                                __fadd_rn(v.z, __fsub_rn(c.z, v.z)), __fadd_rn(v.w, __fsub_rn(c.w, v.w)));
  else qv = c;
  return make_float4(__fsub_rn(v.x, qv.x), __fsub_rn(v.y, qv.y), __fsub_rn(v.z, qv.z), __fsub_rn(v.w, qv.w));
}
template <int VEC, bool kRot>
__global__ void __launch_bounds__(kGatherThreads)
rvq_backward_kernel(const float* __restrict__ x, const float* __restrict__ g_out, const uint8_t* __restrict__ mask,
                    float* __restrict__ grad_x, int64_t N, int d, const __grid_constant__ BackwardArgs B) {
  const ReplayArgs& A = B.R;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wpb = kGatherThreads / 32;
  const float my_coef = lane < A.Q ? B.coef[lane] : 0.f;
  for (int64_t row = (int64_t)blockIdx.x * wpb + warp; row < N; row += (int64_t)gridDim.x * wpb) {
    const bool live = mask == nullptr || mask[row] != 0;
    float4 r[VEC], acc[VEC], g[kRot ? VEC : 1];
#pragma unroll
    for (int t = 0; t < VEC; ++t) {
      const int j = lane * 4 + 128 * t;
      r[t] = acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (kRot) g[t] = r[t];
      if (j < d) {
        r[t] = __ldcs(reinterpret_cast<const float4*>(x + row * (int64_t)d + j));
        const float4 gv = g_out ? __ldcs(reinterpret_cast<const float4*>(g_out + row * (int64_t)d + j))
                                : make_float4(0.f, 0.f, 0.f, 0.f);
        if (kRot) {
          g[t] = gv;
        } else {
          const float q = (float)A.Q;
          acc[t] = make_float4(q * gv.x, q * gv.y, q * gv.z, q * gv.w);
        }
      }
    }
    const long long my_k = lane < A.Q ? (long long)A.idx[lane][row] : 0ll;
    for (int l = 0; l < A.Q; ++l) {
      const float* cr = A.cb[l] + __shfl_sync(0xffffffffu, my_k, l) * (int64_t)d;
      const float cf = live ? __shfl_sync(0xffffffffu, my_coef, l) : 0.f;
      const bool tr = A.training[l] != 0;
      if constexpr (kRot) {
        // level l's output is rotated r_l -> c_l: acc += T_l(g_out) (identity on masked rows, whose level returns r_l);
        // five warp reductions on the row held in registers (|r|^2, |c|^2 in fp64, g.r, g.c, then |u + q|^2)
        float4 c[VEC];
#pragma unroll
        for (int t = 0; t < VEC; ++t) {
          const int j = lane * 4 + 128 * t;
          c[t] = j < d ? __ldg(reinterpret_cast<const float4*>(cr + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (live) {
          double nx2 = 0.0, nc2 = 0.0;
          float gdx = 0.f, gdc = 0.f;
#pragma unroll
          for (int t = 0; t < VEC; ++t) {
            const float4 v = r[t], cv = c[t], gv = g[t];
            nx2 = fma((double)v.x, (double)v.x, nx2); nx2 = fma((double)v.y, (double)v.y, nx2);
            nx2 = fma((double)v.z, (double)v.z, nx2); nx2 = fma((double)v.w, (double)v.w, nx2);
            nc2 = fma((double)cv.x, (double)cv.x, nc2); nc2 = fma((double)cv.y, (double)cv.y, nc2);
            nc2 = fma((double)cv.z, (double)cv.z, nc2); nc2 = fma((double)cv.w, (double)cv.w, nc2);
            gdx = fmaf(gv.x, v.x, gdx); gdx = fmaf(gv.y, v.y, gdx); gdx = fmaf(gv.z, v.z, gdx); gdx = fmaf(gv.w, v.w, gdx);
            gdc = fmaf(gv.x, cv.x, gdc); gdc = fmaf(gv.y, cv.y, gdc); gdc = fmaf(gv.z, cv.z, gdc); gdc = fmaf(gv.w, cv.w, gdc);
          }
          RotCoef rc = rot_scales(warp_sum(nx2), warp_sum(nc2));
          float nw2 = 0.f;
#pragma unroll
          for (int t = 0; t < VEC; ++t) {
            const float4 v = r[t], cv = c[t];    // zero beyond d: contributes 0
            const float e0 = rot_sum(v.x, cv.x, rc), e1 = rot_sum(v.y, cv.y, rc);
            const float e2 = rot_sum(v.z, cv.z, rc), e3 = rot_sum(v.w, cv.w, rc);
            nw2 = fmaf(e0, e0, nw2); nw2 = fmaf(e1, e1, nw2); nw2 = fmaf(e2, e2, nw2); nw2 = fmaf(e3, e3, nw2);
          }
          rot_finish(rc, warp_sum(gdx), warp_sum(gdc), warp_sum(nw2));
#pragma unroll
          for (int t = 0; t < VEC; ++t) {
            const float4 v = r[t], cv = c[t], gv = g[t];
            auto tr1 = [&](float xv, float cc, float gg) {
              return fmaf(rc.b, rot_u(xv, rc), fmaf(rc.a, rot_sum(xv, cc, rc), rc.lam * gg));
            };
            acc[t].x += tr1(v.x, cv.x, gv.x); acc[t].y += tr1(v.y, cv.y, gv.y);
            acc[t].z += tr1(v.z, cv.z, gv.z); acc[t].w += tr1(v.w, cv.w, gv.w);
          }
        } else {
#pragma unroll
          for (int t = 0; t < VEC; ++t) {
            acc[t].x += g[t].x; acc[t].y += g[t].y; acc[t].z += g[t].z; acc[t].w += g[t].w;
          }
        }
#pragma unroll
        for (int t = 0; t < VEC; ++t) {
          const float4 v = r[t];
          acc[t].x = fmaf(cf, v.x - c[t].x, acc[t].x); acc[t].y = fmaf(cf, v.y - c[t].y, acc[t].y);
          acc[t].z = fmaf(cf, v.z - c[t].z, acc[t].z); acc[t].w = fmaf(cf, v.w - c[t].w, acc[t].w);
          r[t] = rvq_next_residual(v, c[t], live, tr);
        }
      } else {
#pragma unroll
        for (int t = 0; t < VEC; ++t) {
          const int j = lane * 4 + 128 * t;
          if (j >= d) continue;
          const float4 c = __ldg(reinterpret_cast<const float4*>(cr + j));
          const float4 v = r[t];
          acc[t].x = fmaf(cf, v.x - c.x, acc[t].x); acc[t].y = fmaf(cf, v.y - c.y, acc[t].y);
          acc[t].z = fmaf(cf, v.z - c.z, acc[t].z); acc[t].w = fmaf(cf, v.w - c.w, acc[t].w);
          r[t] = rvq_next_residual(v, c, live, tr);
        }
      }
    }
#pragma unroll
    for (int t = 0; t < VEC; ++t) {
      const int j = lane * 4 + 128 * t;
      if (j < d) __stcs(reinterpret_cast<float4*>(grad_x + row * (int64_t)d + j), acc[t]);
    }
  }
}

}  // namespace vqb

using namespace vqb;

extern "C" size_t vqb_gather_workspace_bytes(int64_t H, int64_t N, int d) {
  (void)H; (void)N; (void)d;
  return gather_layout().total;
}

extern "C" int vqb_gather_st_loss(const void* x, int x_dtype, const float* codebook, const int64_t* idx,
                                  const uint8_t* mask, int training, int want_loss, float* q_out, float* loss_out,
                                  int64_t H, int64_t N, int K, int d, void* ws, size_t ws_bytes, void* stream) {
  // an empty batch has no rows to read or write (torch hands out null data pointers for it); its loss is NaN, 0
  VQB_REQUIRE(codebook && (H * N == 0 || (x && idx && q_out)), VQB_ERR_INVALID, "vqb_gather_st_loss: null pointer");
  VQB_REQUIRE(H > 0 && N >= 0 && K > 0 && d > 0, VQB_ERR_INVALID, "vqb_gather_st_loss: bad shape");
  GatherLayout L = gather_layout();
  if (want_loss) {
    VQB_REQUIRE(loss_out && ws && ws_bytes >= L.total, VQB_ERR_WORKSPACE, "gather workspace too small: %zu < %zu",
                ws_bytes, L.total);
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = gather_grid(H * N);
  double* part = want_loss ? (double*)((char*)ws + L.off_part) : nullptr;
  long long* cntp = want_loss ? (long long*)((char*)ws + L.off_cnt) : nullptr;
  const bool narrow = d >= 8 && d <= 128 && (d & (d - 1)) == 0;
  if (H * N > 0 && narrow) {
    if (want_loss) {
      VQB_DISPATCH_DTYPE(x_dtype, T,
        gather_st_loss_narrow_kernel<T, true><<<grid, kGatherThreads, 0, st>>>((const T*)x, codebook, idx, mask, training,
                                                                               q_out, H, N, K, d, part, cntp));
    } else {
      VQB_DISPATCH_DTYPE(x_dtype, T,
        gather_st_loss_narrow_kernel<T, false><<<grid, kGatherThreads, 0, st>>>((const T*)x, codebook, idx, mask, training,
                                                                                q_out, H, N, K, d, part, cntp));
    }
    VQB_LAUNCH_CHECK();
  } else if (H * N > 0) {
    // (a 4-rows-per-warp variant was measured SLOWER here: 462 vs 351 us at C2 -- the code-row gather wants occupancy)
    if (want_loss) {
      VQB_DISPATCH_DTYPE(x_dtype, T,
        gather_st_loss_kernel<T, true><<<grid, kGatherThreads, 0, st>>>((const T*)x, codebook, idx, mask, training,
                                                                        q_out, H, N, K, d, part, cntp));
    } else {
      VQB_DISPATCH_DTYPE(x_dtype, T,
        gather_st_loss_kernel<T, false><<<grid, kGatherThreads, 0, st>>>((const T*)x, codebook, idx, mask, training,
                                                                         q_out, H, N, K, d, part, cntp));
    }
    VQB_LAUNCH_CHECK();
  }
  if (want_loss) {
    loss_finalize_kernel<<<1, 256, 0, st>>>(part, cntp, H * N > 0 ? grid : 0, d, loss_out);
    VQB_LAUNCH_CHECK();
  }
  return VQB_OK;
}

extern "C" int vqb_st_commit_backward(const float* grad_q, const float* grad_loss, const void* x, int x_dtype,
                                      const float* codebook, const int64_t* idx, const uint8_t* mask, float coef,
                                      float* grad_x, int64_t H, int64_t N, int K, int d, void* stream) {
  if (H * N == 0) return VQB_OK;
  VQB_REQUIRE(grad_q && grad_loss && x && codebook && idx && grad_x, VQB_ERR_INVALID,
              "vqb_st_commit_backward: null pointer");
  const int grid = gather_grid(H * N);
  VQB_DISPATCH_DTYPE(x_dtype, T,
    st_commit_backward_kernel<T, false><<<grid, kGatherThreads, 0, (cudaStream_t)stream>>>(
        grad_q, grad_loss, (const T*)x, codebook, idx, mask, coef, grad_x, H, N, K, d));
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_rot_commit_backward(const float* grad_q, const float* grad_loss, const void* x, int x_dtype,
                                       const float* codebook, const int64_t* idx, const uint8_t* mask, float coef,
                                       float* grad_x, int64_t H, int64_t N, int K, int d, void* stream) {
  if (H * N == 0) return VQB_OK;
  VQB_REQUIRE(grad_q && grad_loss && x && codebook && idx && grad_x, VQB_ERR_INVALID,
              "vqb_rot_commit_backward: null pointer");
  const int grid = gather_grid(H * N);
  VQB_DISPATCH_DTYPE(x_dtype, T,
    st_commit_backward_kernel<T, true><<<grid, kGatherThreads, 0, (cudaStream_t)stream>>>(
        grad_q, grad_loss, (const T*)x, codebook, idx, mask, coef, grad_x, H, N, K, d));
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_rvq_level(const float* residual_in, float* residual_out, const float* codebook,
                             const int64_t* idx, const uint8_t* mask, int training, int first_level,
                             float* quantized_out, float* q_out, float* loss_out, int64_t N, int K, int d,
                             void* gather_ws, size_t gather_ws_bytes, void* next_ws, size_t next_ws_bytes,
                             const void* next_cache, void* stream) {
  VQB_REQUIRE(residual_in && residual_out && codebook && idx && loss_out && gather_ws,
              VQB_ERR_INVALID, "vqb_rvq_level: null pointer");
  GatherLayout L = gather_layout();
  VQB_REQUIRE(gather_ws_bytes >= L.total, VQB_ERR_WORKSPACE, "gather workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  LatentOperand next = {};   // all null: no next level to prepare
  const int dp = d_pad(d);
  if (next_ws && dp > 512) next_ws = nullptr;   // no tensor-core pass for this width: nothing to prepare
  if (next_ws) {
    VQB_REQUIRE(next_cache != nullptr, VQB_ERR_INVALID,
                "vqb_rvq_level: next_ws needs next_cache (the codebook cache of the level that will search it)");
    VQB_REQUIRE(next_ws_bytes >= search_layout(1, N, K, d).total, VQB_ERR_WORKSPACE,
                "next-level search workspace too small");
    next = latent_operand(next_ws, 1, N, K, d, next_cache);
    VQB_CUDA_TRY(cudaMemsetAsync(next.scal, 0, (kScalDxMax + 1) * 4, st));
  }
  const int grid = gather_grid(N);
  double* part = (double*)((char*)gather_ws + L.off_part);
  long long* cntp = (long long*)((char*)gather_ws + L.off_cnt);
  if (N > 0) {
    rvq_level_kernel<<<grid, kGatherThreads, 0, st>>>(residual_in, residual_out, codebook, idx, mask, training, first_level,
                                                      quantized_out, q_out, N, K, d, dp, part, cntp,
                                                      next.xb, next.xinv, next.scal, next.xaug, next.chdr, next.xn2);
    VQB_LAUNCH_CHECK();
  }
  loss_finalize_kernel<<<1, 256, 0, st>>>(part, cntp, N > 0 ? grid : 0, d, loss_out);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_rvq_replay_out_supported(int d, int num_levels) {
  return (d > 0 && d % 4 == 0 && d <= 512 && num_levels >= 1 && num_levels <= kMaxReplayLevels) ? 1 : 0;
}

extern "C" int vqb_rvq_replay_out(const float* x, const float* const* codebooks, const int64_t* const* idx,
                                  const int* training, int num_levels, const uint8_t* mask, float* out, int64_t N,
                                  int d, void* stream) {
  VQB_REQUIRE(x && codebooks && idx && training && out, VQB_ERR_INVALID, "vqb_rvq_replay_out: null pointer");
  VQB_REQUIRE(vqb_rvq_replay_out_supported(d, num_levels), VQB_ERR_UNSUPPORTED,
              "vqb_rvq_replay_out: d=%d (multiple of 4, <= 512), levels=%d (<= %d)", d, num_levels, kMaxReplayLevels);
  if (N <= 0) return VQB_OK;
  ReplayArgs A = {};
  A.Q = num_levels;
  for (int l = 0; l < num_levels; ++l) {
    VQB_REQUIRE(codebooks[l] && idx[l], VQB_ERR_INVALID, "vqb_rvq_replay_out: null level pointer");
    A.cb[l] = codebooks[l]; A.idx[l] = idx[l]; A.training[l] = training[l];
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = gather_grid(N);
  if (d <= 128) rvq_replay_out_kernel<1><<<grid, kGatherThreads, 0, st>>>(x, mask, out, N, d, A);
  else if (d <= 256) rvq_replay_out_kernel<2><<<grid, kGatherThreads, 0, st>>>(x, mask, out, N, d, A);
  else rvq_replay_out_kernel<4><<<grid, kGatherThreads, 0, st>>>(x, mask, out, N, d, A);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

static int rvq_backward_launch(const char* what, bool rot, const float* x, const float* const* codebooks,
                               const int64_t* const* idx, const int* training, int num_levels, const float* coef,
                               const float* g_out, const uint8_t* mask, float* grad_x, int64_t N, int d, void* stream) {
  VQB_REQUIRE(x && codebooks && idx && training && coef && grad_x, VQB_ERR_INVALID, "%s: null pointer", what);
  VQB_REQUIRE(vqb_rvq_replay_out_supported(d, num_levels), VQB_ERR_UNSUPPORTED,
              "%s: d=%d (multiple of 4, <= 512), levels=%d (<= %d)", what, d, num_levels, kMaxReplayLevels);
  if (N <= 0) return VQB_OK;
  BackwardArgs B = {};
  B.R.Q = num_levels;
  B.coef = coef;
  for (int l = 0; l < num_levels; ++l) {
    VQB_REQUIRE(codebooks[l] && idx[l], VQB_ERR_INVALID, "%s: null level pointer", what);
    B.R.cb[l] = codebooks[l]; B.R.idx[l] = idx[l]; B.R.training[l] = training[l];
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = gather_grid(N);
  if (rot) {
    if (d <= 128) rvq_backward_kernel<1, true><<<grid, kGatherThreads, 0, st>>>(x, g_out, mask, grad_x, N, d, B);
    else if (d <= 256) rvq_backward_kernel<2, true><<<grid, kGatherThreads, 0, st>>>(x, g_out, mask, grad_x, N, d, B);
    else rvq_backward_kernel<4, true><<<grid, kGatherThreads, 0, st>>>(x, g_out, mask, grad_x, N, d, B);
  } else {
    if (d <= 128) rvq_backward_kernel<1, false><<<grid, kGatherThreads, 0, st>>>(x, g_out, mask, grad_x, N, d, B);
    else if (d <= 256) rvq_backward_kernel<2, false><<<grid, kGatherThreads, 0, st>>>(x, g_out, mask, grad_x, N, d, B);
    else rvq_backward_kernel<4, false><<<grid, kGatherThreads, 0, st>>>(x, g_out, mask, grad_x, N, d, B);
  }
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_rvq_backward(const float* x, const float* const* codebooks, const int64_t* const* idx,
                                const int* training, int num_levels, const float* coef, const float* g_out,
                                const uint8_t* mask, float* grad_x, int64_t N, int d, void* stream) {
  return rvq_backward_launch("vqb_rvq_backward", false, x, codebooks, idx, training, num_levels, coef, g_out, mask,
                             grad_x, N, d, stream);
}

extern "C" int vqb_rvq_backward_rot(const float* x, const float* const* codebooks, const int64_t* const* idx,
                                    const int* training, int num_levels, const float* coef, const float* g_out,
                                    const uint8_t* mask, float* grad_x, int64_t N, int d, void* stream) {
  return rvq_backward_launch("vqb_rvq_backward_rot", true, x, codebooks, idx, training, num_levels, coef, g_out, mask,
                             grad_x, N, d, stream);
}
