// prepare.cu -- operand preparation for the tensor-core search:
//   * codebook cache: fp16(c * s_c) padded copy (s_c = power of two per codebook) + per-code norms /
//     rounding residual norms
//   * latents: fp16(x * s_row) padded copy (s_row = power of two per row) + global max row norm /
//     max rounding residual norm.  fp16 carries 3 more mantissa bits than bf16 at the same tensor-core
//     rate, which makes the rigorous rounding bound E_k (and so the re-rank rate) 8x smaller; the
//     power-of-two scales remove fp16's range problem and are undone exactly in the epilogue.
//   * per-search lower-bound bias  L_k = |c_k|^2/2 - E_k  (see search_resolve.cu for the proof sketch)
//   * l2norm of rows (reference utils/losses.py:19)
#include "common.cuh"

namespace vqb {

// max |c| per codebook -> hdr[h][2] (bits of a non-negative float order like unsigned ints)
__global__ void codebook_absmax_kernel(const float* __restrict__ cb, int64_t per_head, float* __restrict__ hdr) {
  const int h = blockIdx.y;
  const float* c = cb + (int64_t)h * per_head;
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_head; i += (int64_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(c[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<uint32_t*>(hdr + h * kHdrFloats + 2), __float_as_uint(m));
}

// one warp per code row (incl. padded rows k in [K, Kp)): fp16(c * s_c) + norms of c and of the rounding residual
__global__ void prepare_codebook_kernel(const float* __restrict__ cb, int64_t H, int K, int Kp, int d, int dp,
                                        int metric, float* __restrict__ hdr, __half* __restrict__ out,
                                        float* __restrict__ cn2h, float* __restrict__ cn, float* __restrict__ dcn) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= H * (int64_t)Kp) return;
  const int64_t h = row / Kp;
  const int k = (int)(row - h * Kp);
  const float sc = pow2_scale(hdr[h * kHdrFloats + 2]);
  const float isc = 1.f / sc;
  if (k == 0 && lane == 0) { hdr[h * kHdrFloats + 0] = sc; hdr[h * kHdrFloats + 1] = isc; }
  __half* o = out + row * dp;
  if (k >= K) {
    for (int j = lane; j < dp; j += 32) o[j] = __float2half(0.f);
    if (lane == 0) { cn2h[row] = kPadBias; cn[row] = 0.f; dcn[row] = 0.f; }
    return;
  }
  const float* c = cb + (h * K + k) * (int64_t)d;
  double n2 = 0.0, r2 = 0.0;
  for (int j = lane; j < dp; j += 32) {
    const float v = j < d ? c[j] : 0.f;
    const __half hv = __float2half_rn(v * sc);           // power-of-two scaling is exact
    const float back = __half2float(hv) * isc;
    o[j] = __hneg(hv);                                   // stored negated: accumulator = s_row s_c (|c|^2/2 - x.c)
    n2 = fma((double)v, (double)v, n2);
    const double r = (double)v - (double)back;
    r2 = fma(r, r, r2);
  }
  n2 = warp_sum(n2);
  r2 = warp_sum(r2);
  if (lane == 0) {
    const float hh = metric == VQB_EUCLID ? (float)(0.5 * n2) : 0.f;
    cn2h[row] = hh;
    if (hh > 0.f) atomicMax(reinterpret_cast<uint32_t*>(hdr + h * kHdrFloats + 3), __float_as_uint(hh));
    cn[row] = __double2float_ru(sqrt(n2)) * 1.000001f;
    dcn[row] = __double2float_ru(sqrt(r2)) * 1.000001f;
  }
}

// Scale of the bias operand: b_k = s_c 2^q (|c_k|^2/2 - E_k) must be an fp16 number; q is chosen per codebook so that
// s_c 2^q max_k |c_k|^2/2 lies in [2^12, 2^13) -- three binades of head room for E_k (make_bias_kernel checks it).
__global__ void codebook_aug_scale_kernel(int64_t H, float* __restrict__ hdr) {
  const int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  const float sc = hdr[h * kHdrFloats + 0], hmax = hdr[h * kHdrFloats + 3];
  int qe = 0;
  const float t = sc * hmax;
  if (t > 0.f && isfinite(t)) {
    int e;
    frexpf(t, &e);                 // t = m 2^e, m in [0.5, 1)
    qe = 13 - e;
    if (qe > 100) qe = 100;
    if (qe < -100) qe = -100;
  }
  hdr[h * kHdrFloats + 4] = ldexpf(1.f, qe);
  hdr[h * kHdrFloats + 5] = ldexpf(1.f, -qe);
}

// Fast variant for d % 8 == 0, d <= 256 (one 8-element group per lane): a warp converts 4 (fp32) or 8 (16-bit) rows per
// iteration with all loads issued up front -- with one 512 B row per warp in flight the kernel is latency bound (Little's law:
// ~19 KB per SM in flight ~ 3.5 TB/s).  Three blocks per SM: the register cap that measured fastest, without spills.
template <typename T>
__global__ void __launch_bounds__(256, 3)
prepare_latents4_kernel(const T* __restrict__ x, int64_t rows, int64_t rows_per_head, bool single_head, int d, int dp,
                        const float* __restrict__ chdr, __half* __restrict__ xb, float* __restrict__ xinv,
                        float* __restrict__ xn2, __half* __restrict__ xaug, uint32_t* __restrict__ scal) {
  constexpr int U = sizeof(T) == 2 ? 8 : 4;       // rows in flight per warp (32 registers of raw data)
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const int j = lane * 8;
  const bool on = j < d;
  float max_n2 = 0.f, max_r2 = 0.f;
  for (int64_t row0 = ((int64_t)blockIdx.x * wpb + (threadIdx.x >> 5)) * U; row0 < rows;
       row0 += (int64_t)gridDim.x * wpb * U) {
    Raw8<T> raw[U];
    float my_is = 0.f, my_a = 0.f, my_n2b = 0.f;
    float two_q = 1.f, two_mq = 1.f;
    if (chdr) {   // the rows of an iteration share a codebook (rows_per_head % 8 == 0 is checked by the launcher)
      const float* hd = chdr + (single_head ? 0 : (uint32_t)row0 / (uint32_t)rows_per_head) * kHdrFloats;
      two_q = hd[4]; two_mq = hd[5];
    }
#pragma unroll
    for (int u = 0; u < U; ++u)                    // all U row loads are issued before the first use
      raw[u] = load_raw8<T>(x + (on && row0 + u < rows ? (row0 + u) * (int64_t)d + j : 0));
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (row0 + u >= rows) break;                 // warp-uniform
      F8 vv = raw_to_f8(raw[u]);
      if (!on) {
#pragma unroll
        for (int e = 0; e < 8; ++e) vv.v[e] = 0.f;
      }
      float m = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) m = fmaxf(m, fabsf(vv.v[e]));
      // non-negative floats order like their bit patterns: one REDUX instead of five shuffle + max steps (same value)
      m = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(m)));
      float s = pow2_scale_bits(m);
      float a = 1.f;
      if (chdr) a = clamp_row_scale(s, two_q, two_mq);
      const float is = pow2_recip(s);
      if (lane == u) { my_is = a > 0.f ? is : -is; my_a = a; }     // lane u keeps row u's scalars for one 4-row store
      float n2 = 0.f, r2 = 0.f;
      if (sizeof(T) == 2) {
        // 16-bit latents (8 or 11 significant bits) times a power of two are fp16 numbers unless they land in
        // fp16's subnormal range, where the rounding error is at most 2^-25: |x - x~|_j <= 2^-25 / s for every j.
        // The residual norm is therefore BOUNDED analytically instead of measured, and |x~| <= |x| + |x - x~|.
        if (j < dp) {
          uint32_t pk[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float v0 = vv.v[2 * e], v1 = vv.v[2 * e + 1];
            const __half2 h = __floats2half2_rn(v0 * s, v1 * s);
            pk[e] = *reinterpret_cast<const uint32_t*>(&h);
            n2 = fmaf(v0, v0, n2);
            n2 = fmaf(v1, v1, n2);
          }
          *reinterpret_cast<uint4*>(xb + (row0 + u) * (int64_t)dp + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        n2 = warp_sum(n2);
        const float rb = 2.9802322e-8f * is;                       // 2^-25 / s
        r2 = (float)dp * rb * rb * 1.0001f;
        n2 = n2 * 1.000001f + r2 * 1.0001e6f;                      // (a + b)^2 <= a^2 (1 + e) + b^2 (1 + 1/e), e = 1e-6
      } else {
        if (j < dp) {
          uint32_t pk[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float v0 = vv.v[2 * e], v1 = vv.v[2 * e + 1];
            const __half2 h = __floats2half2_rn(v0 * s, v1 * s);
            const float2 f = __half22float2(h);
            pk[e] = *reinterpret_cast<const uint32_t*>(&h);
            const float b0 = f.x * is, b1 = f.y * is;
            n2 += b0 * b0 + b1 * b1;
            const float e0 = v0 - b0, e1 = v1 - b1;
            r2 += e0 * e0 + e1 * e1;
          }
          *reinterpret_cast<uint4*>(xb + (row0 + u) * (int64_t)dp + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        n2 = warp_sum(n2);
        r2 = warp_sum(r2);
      }
      if (lane == u) my_n2b = row_norm2_bound(n2, r2);
      max_n2 = fmaxf(max_n2, n2);
      max_r2 = fmaxf(max_r2, r2);
    }
    if (lane < U && row0 + lane < rows) {          // scales + bias operands of the U rows in one coalesced store each
      xinv[row0 + lane] = my_is;
      xn2[row0 + lane] = my_n2b;
      if (xaug) {
        const uint32_t aa = (uint32_t)__half_as_ushort(__float2half_rn(my_a));
        *reinterpret_cast<uint4*>(xaug + (row0 + lane) * 8) = make_uint4(aa | (aa << 16), aa, 0u, 0u);
      }
    }
  }
  __shared__ float s_n[32], s_r[32];
  const int w = threadIdx.x >> 5;
  if (lane == 0) { s_n[w] = max_n2; s_r[w] = max_r2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float mn = 0.f, mr = 0.f;
    for (int i = 0; i < wpb; ++i) { mn = fmaxf(mn, s_n[i]); mr = fmaxf(mr, s_r[i]); }
    atomicMax(scal + kScalXMax, batch_bound_bits(mn, dp));
    atomicMax(scal + kScalDxMax, batch_bound_bits(mr, dp));
  }
}

// Narrow rows (d_pad = 64 or 128): d_pad/8 lanes per row, so a warp converts 4 or 2 rows at a time (x U in flight)
// instead of leaving most of its lanes idle.  Same arithmetic as prepare_latents4_kernel.
template <typename T>
__global__ void __launch_bounds__(256, 3)
prepare_latents_narrow_kernel(const T* __restrict__ x, int64_t rows, int64_t rows_per_head, bool single_head, int d,
                              int dp, const float* __restrict__ chdr, __half* __restrict__ xb,
                              float* __restrict__ xinv, float* __restrict__ xn2, __half* __restrict__ xaug,
                              uint32_t* __restrict__ scal) {
  constexpr int U = sizeof(T) == 2 ? 8 : 4;
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const int lpr = dp >> 3, rpi = 32 / lpr;
  const int grp = lane / lpr, gl = lane - grp * lpr;
  const int j = gl * 8;
  const bool on = j < d;
  float max_n2 = 0.f, max_r2 = 0.f;
  for (int64_t row0 = ((int64_t)blockIdx.x * wpb + (threadIdx.x >> 5)) * (U * rpi); row0 < rows;
       row0 += (int64_t)gridDim.x * wpb * (U * rpi)) {
    Raw8<T> raw[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = row0 + u * rpi + grp;
      raw[u] = load_raw8<T>(x + (on && row < rows ? row * (int64_t)d + j : 0));
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t row = row0 + u * rpi + grp;
      const bool live = row < rows;
      F8 vv = raw_to_f8(raw[u]);
      if (!on || !live) {
#pragma unroll
        for (int e = 0; e < 8; ++e) vv.v[e] = 0.f;
      }
      float m = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) m = fmaxf(m, fabsf(vv.v[e]));
      for (int o2 = lpr >> 1; o2 > 0; o2 >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o2));
      float s = pow2_scale_bits(m);
      float a = 1.f;
      if (chdr && live) {
        const float* hd = chdr + (single_head ? 0 : (uint32_t)row / (uint32_t)rows_per_head) * kHdrFloats;
        a = clamp_row_scale(s, hd[4], hd[5]);
      }
      const float is = pow2_recip(s);
      float n2 = 0.f, r2 = 0.f;
      uint32_t pk[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float v0 = vv.v[2 * e], v1 = vv.v[2 * e + 1];
        const __half2 h = __floats2half2_rn(v0 * s, v1 * s);
        const float2 f = __half22float2(h);
        pk[e] = *reinterpret_cast<const uint32_t*>(&h);
        const float b0 = f.x * is, b1 = f.y * is;
        n2 += b0 * b0 + b1 * b1;
        const float e0 = v0 - b0, e1 = v1 - b1;
        r2 += e0 * e0 + e1 * e1;
      }
      if (live) {
        *reinterpret_cast<uint4*>(xb + row * (int64_t)dp + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        if (gl == 0) {
          xinv[row] = a > 0.f ? is : -is;
          if (xaug) {
            const uint32_t aa = (uint32_t)__half_as_ushort(__float2half_rn(a));
            *reinterpret_cast<uint4*>(xaug + row * 8) = make_uint4(aa | (aa << 16), aa, 0u, 0u);
          }
        }
      }
      for (int o2 = lpr >> 1; o2 > 0; o2 >>= 1) {
        n2 += __shfl_xor_sync(0xffffffffu, n2, o2);
        r2 += __shfl_xor_sync(0xffffffffu, r2, o2);
      }
      if (live && gl == 0) xn2[row] = row_norm2_bound(n2, r2);
      max_n2 = fmaxf(max_n2, n2);
      max_r2 = fmaxf(max_r2, r2);
    }
  }
#pragma unroll
  for (int o2 = 16; o2 > 0; o2 >>= 1) {
    max_n2 = fmaxf(max_n2, __shfl_xor_sync(0xffffffffu, max_n2, o2));
    max_r2 = fmaxf(max_r2, __shfl_xor_sync(0xffffffffu, max_r2, o2));
  }
  __shared__ float s_n[32], s_r[32];
  const int w = threadIdx.x >> 5;
  if (lane == 0) { s_n[w] = max_n2; s_r[w] = max_r2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float mn = 0.f, mr = 0.f;
    for (int i = 0; i < wpb; ++i) { mn = fmaxf(mn, s_n[i]); mr = fmaxf(mr, s_r[i]); }
    atomicMax(scal + kScalXMax, batch_bound_bits(mn, dp));
    atomicMax(scal + kScalDxMax, batch_bound_bits(mr, dp));
  }
}

// one warp per latent row: per-row power-of-two scale, fp16 copy (zero padded to dp),
// atomicMax of |x~| and |x - x~| where x~ = fp16(x s)/s is what the tensor core really sees
template <typename T>
__global__ void prepare_latents_kernel(const T* __restrict__ x, int64_t rows, int64_t rows_per_head, int d, int dp,
                                       const float* __restrict__ chdr, __half* __restrict__ xb,
                                       float* __restrict__ xinv, float* __restrict__ xn2, __half* __restrict__ xaug,
                                       uint32_t* __restrict__ scal) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  float max_n2 = 0.f, max_r2 = 0.f;          // running maxima of this warp's rows (one atomic pair per BLOCK at the end)
  for (int64_t row = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * wpb) {
    float n2 = 0.f, r2 = 0.f;
    const T* xr = x + row * (int64_t)d;
    __half* o = xb + row * (int64_t)dp;
    const bool vec = (d & 7) == 0;
    // the row stays in registers between the max pass and the conversion pass (d_pad <= 512: 2 x 8 per lane)
    F8 keep[2];
    float m = 0.f;
    if (vec) {
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int j = lane * 8 + 256 * t;
        if (j < d) keep[t] = load8<T>(xr + j);
        else {
#pragma unroll
          for (int e = 0; e < 8; ++e) keep[t].v[e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) m = fmaxf(m, fabsf(keep[t].v[e]));
      }
    } else {
      for (int j = lane; j < d; j += 32) m = fmaxf(m, fabsf(to_f32<T>(xr[j])));
    }
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o2));
    float s = pow2_scale(m);
    float a = 1.f;
    if (chdr) {
      const float* hd = chdr + (rows_per_head >= rows ? 0 : row / rows_per_head) * kHdrFloats;
      a = clamp_row_scale(s, hd[4], hd[5]);
    }
    const float is = 1.f / s;
    if (lane == 0) {
      xinv[row] = a > 0.f ? is : -is;
      if (xaug) {
        const uint32_t aa = (uint32_t)__half_as_ushort(__float2half_rn(a));
        *reinterpret_cast<uint4*>(xaug + row * 8) = make_uint4(aa | (aa << 16), aa, 0u, 0u);
      }
    }
    if (vec) {
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int j = lane * 8 + 256 * t;
        if (j >= dp) break;
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float v0 = keep[t].v[2 * e], v1 = keep[t].v[2 * e + 1];
          const __half2 h = __floats2half2_rn(v0 * s, v1 * s);
          const float2 f = __half22float2(h);
          pk[e] = *reinterpret_cast<const uint32_t*>(&h);
          const float b0 = f.x * is, b1 = f.y * is;
          n2 += b0 * b0 + b1 * b1;
          const float e0 = v0 - b0, e1 = v1 - b1;
          r2 += e0 * e0 + e1 * e1;
        }
        *reinterpret_cast<uint4*>(o + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
    } else {
      for (int j = lane; j < dp; j += 32) {
        const float v = j < d ? to_f32<T>(xr[j]) : 0.f;
        const __half hv = __float2half_rn(v * s);
        const float back = __half2float(hv) * is;
        o[j] = hv;
        n2 += back * back;
        r2 += (v - back) * (v - back);
      }
    }
    n2 = warp_sum(n2);
    r2 = warp_sum(r2);
    if (lane == 0) xn2[row] = row_norm2_bound(n2, r2);
    max_n2 = fmaxf(max_n2, n2);
    max_r2 = fmaxf(max_r2, r2);
  }
  // block-level max, then one atomic pair per block
  __shared__ float s_n[32], s_r[32];
  const int w = threadIdx.x >> 5;
  if (lane == 0) { s_n[w] = max_n2; s_r[w] = max_r2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float mn = 0.f, mr = 0.f;
    for (int i = 0; i < wpb; ++i) { mn = fmaxf(mn, s_n[i]); mr = fmaxf(mr, s_r[i]); }
    atomicMax(scal + kScalXMax, batch_bound_bits(mn, dp));
    atomicMax(scal + kScalDxMax, batch_bound_bits(mr, dp));
  }
}

int launch_prepare_latents(const void* x, int x_dtype, int64_t rows, int64_t rows_per_head, int d,
                           const LatentOperand& op, cudaStream_t st) {
  if (rows_per_head < 1) rows_per_head = 1;
  const int dp = op.dp;
  const float* chdr = op.chdr;
  __half *xb = op.xb, *xaug = op.xaug;
  float *xinv = op.xinv, *xn2 = op.xn2;
  uint32_t* scal = op.scal;
  VQB_REQUIRE(dp <= 512, VQB_ERR_UNSUPPORTED, "prepare_latents: d_pad %d > 512", dp);
  const int warps = 8;
  int64_t blocks = (rows + warps - 1) / warps;
  const int sms = num_sms();
  if (blocks > (int64_t)sms * 8) blocks = (int64_t)sms * 8;     // persistent: rows strided over the grid
  if (blocks < 1) blocks = 1;
  if ((d & 7) == 0 && dp <= 128 && rows < (1ll << 32)) {
    VQB_DISPATCH_DTYPE(x_dtype, T,
      prepare_latents_narrow_kernel<T><<<(unsigned)blocks, warps * 32, 0, st>>>((const T*)x, rows, rows_per_head,
                                                                                rows_per_head >= rows, d, dp, chdr,
                                                                                xb, xinv, xn2, xaug, scal));
  } else if ((d & 7) == 0 && d <= 256 && (rows_per_head >= rows || (rows_per_head % 8 == 0 && rows < (1ll << 32)))) {
    const int64_t want = (rows + warps - 1) / warps, cap = (int64_t)sms * 4 * 3;
    blocks = want < cap ? want : cap;      // persistent: as many blocks as fit at this register cap
    if (blocks < 1) blocks = 1;
    VQB_DISPATCH_DTYPE(x_dtype, T, (prepare_latents4_kernel<T><<<(unsigned)blocks, warps * 32, 0, st>>>(
        (const T*)x, rows, rows_per_head, rows_per_head >= rows, d, dp, chdr, xb, xinv, xn2, xaug, scal)));
  } else {
    VQB_DISPATCH_DTYPE(x_dtype, T,
      prepare_latents_kernel<T><<<(unsigned)blocks, warps * 32, 0, st>>>((const T*)x, rows, rows_per_head, d, dp, chdr,
                                                                         xb, xinv, xn2, xaug, scal));
  }
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

// Strided sample of the rows: scal[kScalXMax] = kSampleGuard * max |x_row| over the sample (in-kernel conversion, search_tc.cu).
// One warp per sampled row, d % 8 == 0, d <= 256.
template <typename T>
__global__ void __launch_bounds__(256)
sample_bound_kernel(const T* __restrict__ x, int64_t rows, int64_t stride, int64_t nsample, int d,
                    uint32_t* __restrict__ scal) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * 8 + w;
  float n2 = 0.f;
  if (i < nsample) {
    const int64_t row = i * stride < rows ? i * stride : rows - 1;
    const int j = lane * 8;
    if (j < d) {
      const F8 vv = raw_to_f8(load_raw8<T>(x + row * (int64_t)d + j));
#pragma unroll
      for (int e = 0; e < 8; ++e) n2 = fmaf(vv.v[e], vv.v[e], n2);
    }
    n2 = warp_sum(n2);
  }
  __shared__ float s_n[8];
  if (lane == 0) s_n[w] = n2;
  __syncthreads();
  if (threadIdx.x == 0) {
    float mn = 0.f;
    for (int k = 0; k < 8; ++k) mn = fmaxf(mn, s_n[k]);
    if (mn > 0.f && mn < 3.0e38f) atomicMax(scal + kScalXMax, __float_as_uint(sqrtf(mn) * kSampleGuard));
  }
}

int launch_sample_bound(const void* x, int x_dtype, int64_t rows, int d, uint32_t* scal, cudaStream_t st) {
  VQB_REQUIRE(x_dtype != VQB_F32 && d % 8 == 0 && d <= 256, VQB_ERR_UNSUPPORTED, "sample_bound: 16-bit rows of d <= 256");
  const int64_t nsample = rows < 16384 ? rows : 16384;
  const int64_t stride = rows / nsample;
  const unsigned blocks = (unsigned)((nsample + 7) / 8);
  if (x_dtype == VQB_BF16)
    sample_bound_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)x, rows, stride, nsample, d, scal);
  else
    sample_bound_kernel<__half><<<blocks, 256, 0, st>>>((const __half*)x, rows, stride, nsample, d, scal);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

// E_k = Xmax*|c_k - c~_k| + DXmax*|c_k| + accumulation slack;  bias_k = |c_k|^2/2 - E_k
__global__ void make_bias_kernel(const float* __restrict__ cn2h, const float* __restrict__ cn,
                                 const float* __restrict__ dcn, int64_t total, int Kp, int K,
                                 const float* __restrict__ hdr, uint32_t* __restrict__ scal,
                                 float* __restrict__ bias, float* __restrict__ err, int derive_dx_dp) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float e = 0.f;
  if (i < total) {
    const int k = (int)(i % Kp);
    const float hmax = hdr[(i / Kp) * kHdrFloats + 3];
    if (k >= K) {
      bias[i] = kPadBias;
      err[i] = 0.f;
    } else {
      const float xmax = __uint_as_float(scal[kScalXMax]);
      const float dxmax = derive_dx_dp > 0 ? dx_bound_16bit(xmax, derive_dx_dp, hdr[(i / Kp) * kHdrFloats + 5])
                                           : __uint_as_float(scal[kScalDxMax]);
      const float c = cn[i], h = cn2h[i];
      // products are exact in the tensor core (fp16 x fp16 = 22 bits, fits fp32); accumulation is fp32-ish:
      // allow 2^-16 of the largest possible |sum| plus the fp32 rounding of |c|^2/2.
      // (with the bias k-step |c|^2/2 goes through the same accumulator: same 2^-16 allowance, plus the
      // representation error of its three fp16 pieces, < 2^-33 relative / 2^-37 of the largest bias)
      e = xmax * dcn[i] + dxmax * c + 1.6e-5f * (xmax * c + h) + 1e-9f * hmax;
      e = e * 1.001f + 1e-30f;
      err[i] = e;
      bias[i] = h - e;
    }
  }
  // scal[kScalEmax] = max_k E_k: the search epilogue's skip test needs a bound that holds for whichever code wins
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) e = fmaxf(e, __shfl_xor_sync(0xffffffffu, e, o));
  if ((threadIdx.x & 31) == 0 && e > 0.f) atomicMax(scal + kScalEmax, __float_as_uint(e));
}

// Bias operand of the codebook for this search: three fp16 pieces (33 bits) of b_k = s_c 2^q bias_k, +inf for padded
// codes (they can never become candidates).  bias_k = |c_k|^2/2 - E_k (keys pre-lowered, window L_min + 2 E_j) whenever
// every b_k is an fp16 number; otherwise (E_k far above max |c|^2/2) bias_k = |c_k|^2/2 and scal[kScalUnlowered] = 1 tells resolve
// to use the symmetric window min + 2 Emax.
__global__ void make_bias_operand_kernel(const float* __restrict__ cn2h, const float* __restrict__ err,
                                         const float* __restrict__ hdr, int64_t total, int Kp, int K,
                                         uint32_t* __restrict__ scal, __half* __restrict__ caug) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int64_t h = i / Kp;
  const int k = (int)(i - h * Kp);
  const float* hd = hdr + h * kHdrFloats;
  const float emax = __uint_as_float(scal[kScalEmax]);
  const float scq = hd[0] * hd[4];                       // s_c 2^q (power of two)
  // per codebook; one head falling back switches resolve to the (always valid, wider) 2 Emax window for all heads
  const bool lowered = (hd[3] + emax) * scq < 60000.f;
  if (k == 0 && !lowered) scal[kScalUnlowered] = 1u;
  __half p[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) p[j] = __float2half(0.f);
  if (k >= K) {
    p[0] = __ushort_as_half((unsigned short)0x7C00);     // +inf
  } else {
    const float b = (lowered ? cn2h[i] - err[i] : cn2h[i]) * scq;
    const __half b1 = __float2half_rn(b);
    const float r1 = b - __half2float(b1);               // exact (Sterbenz)
    const __half b2 = __float2half_rn(r1);
    const __half b3 = __float2half_rn(r1 - __half2float(b2));
    p[0] = b1; p[1] = b2; p[2] = b3;
  }
  *reinterpret_cast<uint4*>(caug + i * 8) = *reinterpret_cast<const uint4*>(p);
}

int launch_make_bias(const void* cache, const CacheLayout& CL, int64_t H, int K, int metric,
                     uint32_t* scal, float* bias, float* err, __half* caug, cudaStream_t st, int derive_dx_dp) {
  (void)metric;
  const char* base = (const char*)cache;
  int64_t total = H * (int64_t)CL.Kp;
  make_bias_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
      (const float*)(base + CL.off_cn2h), (const float*)(base + CL.off_cn), (const float*)(base + CL.off_dcn),
      total, CL.Kp, K, (const float*)(base + CL.off_hdr), scal, bias, err, derive_dx_dp);
  VQB_LAUNCH_CHECK();
  if (caug) {
    make_bias_operand_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
        (const float*)(base + CL.off_cn2h), err, (const float*)(base + CL.off_hdr), total, CL.Kp, K, scal, caug);
    VQB_LAUNCH_CHECK();
  }
  return VQB_OK;
}

// reference utils/losses.py:19: x / max(|x|_2, 1e-12); one warp per row
template <typename T>
__global__ void l2norm_rows_kernel(const T* __restrict__ x, float* __restrict__ out, int64_t rows, int d) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const T* xr = x + row * (int64_t)d;
  float* o = out + row * (int64_t)d;
  float s = 0.f;
  if ((d & 3) == 0) {
    for (int j = lane * 4; j < d; j += 128) {
      float4 v = load4<T>(xr + j);
      s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s);
    }
  } else {
    for (int j = lane; j < d; j += 32) { float v = to_f32<T>(xr[j]); s = fmaf(v, v, s); }
  }
  s = warp_sum(s);
  float nrm = fmaxf(sqrtf(s), 1e-12f);
  if ((d & 3) == 0) {
    for (int j = lane * 4; j < d; j += 128) {
      float4 v = load4<T>(xr + j);
      float4 r = make_float4(__fdiv_rn(v.x, nrm), __fdiv_rn(v.y, nrm), __fdiv_rn(v.z, nrm), __fdiv_rn(v.w, nrm));
      *reinterpret_cast<float4*>(o + j) = r;
    }
  } else {
    for (int j = lane; j < d; j += 32) o[j] = __fdiv_rn(to_f32<T>(xr[j]), nrm);
  }
}


// l2norm_rows + prepare_latents in ONE pass (cosine codebooks: VectorQuantize normalises its input and the search
// then prepares the normalised rows -- two reads of N x d fp32 and one write become one read): writes x^ = x / |x|
// (same operations in the same order as l2norm_rows_kernel: bit-identical) and, from the registers, the scaled fp16
// operand, row scale, bias operand and row statistics of x^ exactly as prepare_latents_kernel does.
// d % 4 == 0, d_pad <= 512: lanes own float4 groups {lane*4 + 128 t}.
template <typename T>
__global__ void __launch_bounds__(256)
l2norm_prepare_kernel(const T* __restrict__ x, float* __restrict__ out, int64_t rows, int64_t rows_per_head,
                      bool single_head, int d, int dp, const float* __restrict__ chdr, __half* __restrict__ xb,
                      float* __restrict__ xinv, float* __restrict__ xn2, __half* __restrict__ xaug,
                      uint32_t* __restrict__ scal) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  float max_n2 = 0.f, max_r2 = 0.f;
  for (int64_t row = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * wpb) {
    const T* xr = x + row * (int64_t)d;
    float4 v[4];
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int j = lane * 4 + 128 * t;
      v[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j < d) {
        v[t] = load4<T>(xr + j);
        s = fmaf(v[t].x, v[t].x, s); s = fmaf(v[t].y, v[t].y, s); s = fmaf(v[t].z, v[t].z, s); s = fmaf(v[t].w, v[t].w, s);
      }
    }
    s = warp_sum(s);
    const float nrm = fmaxf(sqrtf(s), 1e-12f);
    float m = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int j = lane * 4 + 128 * t;
      if (j < d) {
        v[t] = make_float4(__fdiv_rn(v[t].x, nrm), __fdiv_rn(v[t].y, nrm), __fdiv_rn(v[t].z, nrm), __fdiv_rn(v[t].w, nrm));
        *reinterpret_cast<float4*>(out + row * (int64_t)d + j) = v[t];
        m = fmaxf(fmaxf(fmaxf(m, fabsf(v[t].x)), fmaxf(fabsf(v[t].y), fabsf(v[t].z))), fabsf(v[t].w));
      }
    }
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o2));
    float sc = pow2_scale_bits(m);
    float a = 1.f;
    if (chdr) {
      const float* hd = chdr + (single_head ? 0 : row / rows_per_head) * kHdrFloats;
      a = clamp_row_scale(sc, hd[4], hd[5]);
    }
    const float is = pow2_recip(sc);
    if (lane == 0) {
      xinv[row] = a > 0.f ? is : -is;
      if (xaug) {
        const uint32_t aa = (uint32_t)__half_as_ushort(__float2half_rn(a));
        *reinterpret_cast<uint4*>(xaug + row * 8) = make_uint4(aa | (aa << 16), aa, 0u, 0u);
      }
    }
    float n2 = 0.f, r2 = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int j = lane * 4 + 128 * t;
      if (j < dp) {
        const __half2 h0 = __floats2half2_rn(v[t].x * sc, v[t].y * sc), h1 = __floats2half2_rn(v[t].z * sc, v[t].w * sc);
        const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t*>(&h0);
        pk.y = *reinterpret_cast<const uint32_t*>(&h1);
        *reinterpret_cast<uint2*>(xb + row * (int64_t)dp + j) = pk;
        const float b0 = f0.x * is, b1 = f0.y * is, b2 = f1.x * is, b3 = f1.y * is;
        n2 += b0 * b0 + b1 * b1 + b2 * b2 + b3 * b3;
        const float e0 = v[t].x - b0, e1 = v[t].y - b1, e2 = v[t].z - b2, e3 = v[t].w - b3;
        r2 += e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3;
      }
    }
    n2 = warp_sum(n2);
    r2 = warp_sum(r2);
    if (lane == 0) xn2[row] = row_norm2_bound(n2, r2);
    max_n2 = fmaxf(max_n2, n2);
    max_r2 = fmaxf(max_r2, r2);
  }
  __shared__ float s_n[32], s_r[32];
  const int w = threadIdx.x >> 5;
  if (lane == 0) { s_n[w] = max_n2; s_r[w] = max_r2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float mn = 0.f, mr = 0.f;
    for (int i = 0; i < wpb; ++i) { mn = fmaxf(mn, s_n[i]); mr = fmaxf(mr, s_r[i]); }
    atomicMax(scal + kScalXMax, batch_bound_bits(mn, dp));
    atomicMax(scal + kScalDxMax, batch_bound_bits(mr, dp));
    if (blockIdx.x == 0 && chdr && single_head) scal[kScalTwoQ] = __float_as_uint(chdr[4]);   // the 2^q these operands use
  }
}

}  // namespace vqb

using namespace vqb;

extern "C" size_t vqb_codebook_cache_bytes(int64_t H, int K, int d) {
  if (H <= 0 || K <= 0 || d <= 0) return 0;
  return cache_layout(H, K, d).total;
}

extern "C" int vqb_prepare_codebook(const float* codebook, int64_t H, int K, int d, int metric,
                                    void* cache, size_t cache_bytes, void* stream) {
  VQB_REQUIRE(codebook && cache && H > 0 && K > 0 && d > 0, VQB_ERR_INVALID, "vqb_prepare_codebook: bad argument");
  VQB_REQUIRE(metric == VQB_EUCLID || metric == VQB_DOT, VQB_ERR_INVALID, "unknown metric %d", metric);
  CacheLayout CL = cache_layout(H, K, d);
  VQB_REQUIRE(cache_bytes >= CL.total, VQB_ERR_WORKSPACE, "codebook cache too small: %zu < %zu", cache_bytes, CL.total);
  char* base = (char*)cache;
  cudaStream_t st = (cudaStream_t)stream;
  float* hdr = (float*)(base + CL.off_hdr);
  VQB_CUDA_TRY(cudaMemsetAsync(hdr, 0, (size_t)H * kHdrFloats * 4, st));
  const int64_t per_head = (int64_t)K * d;
  int gx = (int)((per_head + 256 * 8 - 1) / (256 * 8));
  if (gx > 1024) gx = 1024;
  codebook_absmax_kernel<<<dim3((unsigned)gx, (unsigned)H), 256, 0, st>>>(codebook, per_head, hdr);
  VQB_LAUNCH_CHECK();
  const int warps = 8;
  int64_t rows = H * (int64_t)CL.Kp;
  prepare_codebook_kernel<<<(unsigned)((rows + warps - 1) / warps), warps * 32, 0, st>>>(
      codebook, H, K, CL.Kp, d, CL.dp, metric, hdr, (__half*)(base + CL.off_cb), (float*)(base + CL.off_cn2h),
      (float*)(base + CL.off_cn), (float*)(base + CL.off_dcn));
  VQB_LAUNCH_CHECK();
  codebook_aug_scale_kernel<<<(unsigned)((H + 63) / 64), 64, 0, st>>>(H, hdr);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_l2norm_prepare_supported(int d) { return (d % 4 == 0 && d_pad(d) <= 512) ? 1 : 0; }

extern "C" int vqb_l2norm_prepare(const void* x, int x_dtype, float* out, int64_t H, int64_t N, int K, int d,
                                  const void* cache, void* search_ws, size_t ws_bytes, void* stream) {
  VQB_REQUIRE(x && out && cache && search_ws, VQB_ERR_INVALID, "vqb_l2norm_prepare: null pointer");
  VQB_REQUIRE(H > 0 && N >= 0 && K > 0 && d > 0, VQB_ERR_INVALID, "vqb_l2norm_prepare: bad shape");
  VQB_REQUIRE(vqb_l2norm_prepare_supported(d), VQB_ERR_UNSUPPORTED, "vqb_l2norm_prepare: d=%d (d %% 4 == 0, d_pad <= 512)", d);
  SearchLayout SL = search_layout(H, N, K, d);
  VQB_REQUIRE(ws_bytes >= SL.total, VQB_ERR_WORKSPACE, "search workspace too small: %zu < %zu", ws_bytes, SL.total);
  if (N == 0) return VQB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const LatentOperand op = latent_operand(search_ws, H, N, K, d, cache);
  // the batch bounds, and scal[kScalTwoQ]: written below when H = 1, else it stays 0
  VQB_CUDA_TRY(cudaMemsetAsync(op.scal, 0, (kScalTwoQ + 1) * 4, st));
  const int64_t rows = H * N;
  int64_t blocks = (rows + 7) / 8;
  if (blocks > (int64_t)num_sms() * 8) blocks = (int64_t)num_sms() * 8;
  VQB_DISPATCH_DTYPE(x_dtype, T,
    l2norm_prepare_kernel<T><<<(unsigned)blocks, 256, 0, st>>>((const T*)x, out, rows, N, H == 1, d, op.dp, op.chdr,
                                                               op.xb, op.xinv, op.xn2, op.xaug, op.scal));
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_l2norm_rows(const void* x, int x_dtype, float* out, int64_t rows, int d, void* stream) {
  VQB_REQUIRE(x && out && rows >= 0 && d > 0, VQB_ERR_INVALID, "vqb_l2norm_rows: bad argument");
  if (rows == 0) return VQB_OK;
  const int warps = 8;
  VQB_DISPATCH_DTYPE(x_dtype, T,
    l2norm_rows_kernel<T><<<(unsigned)((rows + warps - 1) / warps), warps * 32, 0, (cudaStream_t)stream>>>(
        (const T*)x, out, rows, d));
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}
