// common.cuh -- shared helpers for libvqb200 (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/vqb.h"

namespace vqb {

// ---- error plumbing (thread-local message, C return codes) --------------------------------
void set_error(const char* fmt, ...);

#define VQB_CUDA_TRY(expr)                                                              \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      vqb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return VQB_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

#define VQB_REQUIRE(cond, code, ...)                                                    \
  do {                                                                                  \
    if (!(cond)) {                                                                      \
      vqb::set_error(__VA_ARGS__);                                                      \
      return (code);                                                                    \
    }                                                                                   \
  } while (0)

extern int64_t g_launch_count;   // every kernel launch is followed by VQB_LAUNCH_CHECK()
#define VQB_LAUNCH_CHECK()                 \
  do {                                     \
    ++vqb::g_launch_count;                 \
    VQB_CUDA_TRY(cudaGetLastError());      \
  } while (0)

// ---- geometry shared by prepare / search / resolve ----------------------------------------
constexpr int kBlockM = 128;   // latent rows per CTA tile (TMEM lanes)
constexpr int kBlockN = 256;   // codes per N tile (UMMA N)
constexpr int kBlockK = 64;    // fp16 elements per k-block = one 128B swizzle atom
constexpr int kNumCand = 24;   // candidates kept per row: 4 column quarters x 2 classes x top-3
constexpr float kPadBias = 3.0e38f;
constexpr int kHdrFloats = 8;  // per-codebook header of the cache (see CacheLayout)

__host__ __device__ inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
__host__ __device__ inline int64_t round_up64(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
inline int k_pad(int K) { return round_up(K, kBlockN); }
inline int d_pad(int d) { return round_up(d, kBlockK); }
inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Derived codebook cache layout (one caller-owned buffer).
struct CacheLayout {
  int Kp, dp;
  size_t off_hdr;    // f32  [H][8]       = {s_c (power of two), 1/s_c, max|c|, max|c|^2/2, 2^q, 2^-q, -, -}  (2^q: scale of the bias operand)
  size_t off_cb;     // fp16 [H][Kp][dp]  = -fp16(c * s_c), zero padded (negated: the accumulator is then a score)
  size_t off_cn2h;   // f32  [H][Kp]      = |c|^2 / 2   (0 for the dot metric)
  size_t off_cn;     // f32  [H][Kp]      = |c|
  size_t off_dcn;    // f32  [H][Kp]      = |c - fp16(c*s_c)/s_c|
  size_t total;
};
inline CacheLayout cache_layout(int64_t H, int K, int d) {
  CacheLayout L;
  L.Kp = k_pad(K);
  L.dp = d_pad(d);
  size_t o = 0;
  L.off_hdr = o;  o += align_up((size_t)H * kHdrFloats * 4);
  L.off_cb = o;   o += align_up((size_t)H * L.Kp * L.dp * 2);
  L.off_cn2h = o; o += align_up((size_t)H * L.Kp * 4);
  L.off_cn = o;   o += align_up((size_t)H * L.Kp * 4);
  L.off_dcn = o;  o += align_up((size_t)H * L.Kp * 4);
  L.total = o;
  return L;
}

// Slots of the u32[64] block at the head of a search workspace (SearchLayout::off_scal).  Float bounds are stored as
// their bits: non-negative floats order like unsigned ints, so atomicMax raises them.
constexpr int kScalXMax = 0;         // bound of max |x_b| over the batch (x_b = fp16(x s_row) / s_row)
constexpr int kScalDxMax = 1;        // bound of max |x - x_b| over the batch
constexpr int kScalRescanned = 2;    // rows resolved by a scan of every code
constexpr int kScalReranked = 3;     // rows queued for the warp-per-row re-rank
constexpr int kScalTcUsed = 4;       // 1: the tensor-core pass ran
constexpr int kScalMisaligned = 5;   // 1: the search kernel's dynamic shared memory was not 1024 B aligned
constexpr int kScalEmax = 6;         // max_k E_k
constexpr int kScalTwoQ = 7;         // 2^q of bias operands prepared outside the search (0: prepared by this search)
constexpr int kScalUnlowered = 8;    // 1: keys not pre-lowered by E_k (window 2 Emax)
constexpr int kScalPairs = 9;        // (row, code) pairs queued for exact scoring

// Search workspace layout (one caller-owned buffer).
struct SearchLayout {
  int dp;
  size_t off_scal;    // u32[64]: slots kScal* above
  size_t off_cnt;     // u32[3][H]: flagged rows per codebook | left to the tiled rescan | pair plan (after scal: zeroed together)
  size_t off_xb;      // fp16 [H][N][dp]  = fp16(x * s_row), zero padded
  size_t off_xinv;    // f32  [H][N]      = 1 / s_row (exact power of two); NEGATIVE marks a row whose bias operand
                      //                    s_row 2^-q is not an fp16 number: such rows are rescanned exactly
  size_t off_xn2;     // f32  [H][N]      upper bound of |x_row|^2: sizes the window of fp32 distance ties (resolve)
  size_t off_xaug;    // fp16 [H][N][8]   = {a, a, a, 0, ...}, a = s_row 2^-q: the latent side of the bias k-step
  size_t off_keys;    // u64  [H][N]      packed (score, index) min-keys of rows being rescanned
  size_t off_cand;    // {f32 key, i32 code} [H][N][kNumCand]
  size_t off_flag;    // i32 [H*N] flagged row list
  size_t off_rr;      // i32 [H*N] rows queued for the warp-per-row re-rank (length in scal[kScalReranked])
  size_t off_bias;    // f32 [H][Kp]  lower-bound bias  |c|^2/2 - E_k  (needs the row stats, so per search)
  size_t off_err;     // f32 [H][Kp]  E_k: bound on |exact score - fp16 tensor-core score| for code k
  size_t off_pairs;   // {u32 row, u32 code} [pair_cap]  (row, code) pairs scored exactly in resolve phase 2 (count in scal[kScalPairs])
  size_t pair_cap;
  size_t off_caug;    // fp16 [H][Kp][8]  three fp16 pieces of s_c 2^q bias_k (+inf for padded codes), then zeros:
                      //                  the bias term of the score as one extra MMA k-step (search_tc.cu)
  size_t total;
};
inline SearchLayout search_layout(int64_t H, int64_t N, int K, int d) {
  SearchLayout L;
  L.dp = d_pad(d);
  size_t o = 0;
  L.off_scal = o; o += 256;
  L.off_cnt = o;  o += align_up((size_t)H * 12);
  L.off_xb = o;   o += align_up((size_t)H * N * L.dp * 2);
  L.off_xinv = o; o += align_up((size_t)H * N * 4);
  L.off_xn2 = o;  o += align_up((size_t)H * N * 4);
  L.off_xaug = o; o += align_up((size_t)H * N * 16);
  L.off_keys = o; o += align_up((size_t)H * N * 8);
  L.off_cand = o; o += align_up((size_t)H * N * kNumCand * 8);
  L.off_flag = o; o += align_up((size_t)H * N * 4);
  L.off_rr = o;   o += align_up((size_t)H * N * 4);
  L.off_bias = o; o += align_up((size_t)H * k_pad(K) * 4);
  L.off_err = o;  o += align_up((size_t)H * k_pad(K) * 4);
  L.off_caug = o; o += align_up((size_t)H * k_pad(K) * 16);
  L.pair_cap = (size_t)H * N * 4 + 4096;
  L.off_pairs = o; o += align_up(L.pair_cap * 8);
  L.total = o;
  return L;
}

// The latent operand of the tensor-core search inside a search workspace (fields as in SearchLayout), and the header
// of the codebook cache whose 2^q the bias operand is built with.  make_bias and resolve rely on exactly these values
// (search_resolve.cu), the EMA kernels on scal[kScalXMax] + scal[kScalDxMax] (vqb.h).  The preparation kernels take
// its fields as separate parameters: passed as one struct, they compile to up to 8 more registers each (sm_100a).
struct LatentOperand {
  __half* xb;
  float* xinv;
  float* xn2;
  __half* xaug;
  uint32_t* scal;
  const float* chdr;
  int dp;
};
inline LatentOperand latent_operand(void* search_ws, int64_t H, int64_t N, int K, int d, const void* cache) {
  const SearchLayout SL = search_layout(H, N, K, d);
  char* w = (char*)search_ws;
  return {(__half*)(w + SL.off_xb), (float*)(w + SL.off_xinv), (float*)(w + SL.off_xn2), (__half*)(w + SL.off_xaug),
          (uint32_t*)(w + SL.off_scal), (const float*)((const char*)cache + cache_layout(H, K, d).off_hdr), SL.dp};
}

// SM count of the device that is current at the first call (persistent grids are sized from it)
inline int num_sms() {
  static const int n = [] {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    return v > 0 ? v : 148;
  }();
  return n;
}

// ---- device helpers -----------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

// load 4 consecutive elements (16B-aligned for f32, 8B for 16-bit types) as float4
template <typename T> __device__ __forceinline__ float4 load4(const T* p);
template <> __device__ __forceinline__ float4 load4<float>(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}
template <> __device__ __forceinline__ float4 load4<__nv_bfloat16>(const __nv_bfloat16* p) {
  uint2 r = __ldg(reinterpret_cast<const uint2*>(p));
  float4 o;
  o.x = __uint_as_float(r.x << 16);
  o.y = __uint_as_float(r.x & 0xffff0000u);
  o.z = __uint_as_float(r.y << 16);
  o.w = __uint_as_float(r.y & 0xffff0000u);
  return o;
}
template <> __device__ __forceinline__ float4 load4<__half>(const __half* p) {
  uint2 r = __ldg(reinterpret_cast<const uint2*>(p));
  __half2 a = *reinterpret_cast<__half2*>(&r.x), b = *reinterpret_cast<__half2*>(&r.y);
  float2 fa = __half22float2(a), fb = __half22float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}

// load 8 consecutive elements (32B-aligned for f32, 16B for 16-bit types)
struct F8 { float v[8]; };
template <typename T> __device__ __forceinline__ F8 load8(const T* p);
template <> __device__ __forceinline__ F8 load8<float>(const float* p) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  F8 o; o.v[0] = a.x; o.v[1] = a.y; o.v[2] = a.z; o.v[3] = a.w; o.v[4] = b.x; o.v[5] = b.y; o.v[6] = b.z; o.v[7] = b.w;
  return o;
}
template <> __device__ __forceinline__ F8 load8<__nv_bfloat16>(const __nv_bfloat16* p) {
  const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
  F8 o;
  o.v[0] = __uint_as_float(r.x << 16); o.v[1] = __uint_as_float(r.x & 0xffff0000u);
  o.v[2] = __uint_as_float(r.y << 16); o.v[3] = __uint_as_float(r.y & 0xffff0000u);
  o.v[4] = __uint_as_float(r.z << 16); o.v[5] = __uint_as_float(r.z & 0xffff0000u);
  o.v[6] = __uint_as_float(r.w << 16); o.v[7] = __uint_as_float(r.w & 0xffff0000u);
  return o;
}
template <> __device__ __forceinline__ F8 load8<__half>(const __half* p) {
  const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
  F8 o;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
    o.v[2 * i] = f.x; o.v[2 * i + 1] = f.y;
  }
  return o;
}

// 8 consecutive latent elements kept in their storage type while the load is in flight (half the registers of the
// fp32 form for 16-bit latents, so twice as many rows can be outstanding per thread)
template <typename T> struct Raw8 { uint4 r; };
template <> struct Raw8<float> { float4 a, b; };
template <typename T> __device__ __forceinline__ Raw8<T> load_raw8(const T* p) {
  Raw8<T> o; o.r = __ldg(reinterpret_cast<const uint4*>(p)); return o;
}
template <> __device__ __forceinline__ Raw8<float> load_raw8<float>(const float* p) {
  Raw8<float> o;
  o.a = __ldg(reinterpret_cast<const float4*>(p));
  o.b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  return o;
}
__device__ __forceinline__ F8 raw_to_f8(const Raw8<float>& w) {
  F8 o; o.v[0] = w.a.x; o.v[1] = w.a.y; o.v[2] = w.a.z; o.v[3] = w.a.w; o.v[4] = w.b.x; o.v[5] = w.b.y; o.v[6] = w.b.z; o.v[7] = w.b.w;
  return o;
}
__device__ __forceinline__ F8 raw_to_f8(const Raw8<__nv_bfloat16>& w) {
  F8 o;
  o.v[0] = __uint_as_float(w.r.x << 16); o.v[1] = __uint_as_float(w.r.x & 0xffff0000u);
  o.v[2] = __uint_as_float(w.r.y << 16); o.v[3] = __uint_as_float(w.r.y & 0xffff0000u);
  o.v[4] = __uint_as_float(w.r.z << 16); o.v[5] = __uint_as_float(w.r.z & 0xffff0000u);
  o.v[6] = __uint_as_float(w.r.w << 16); o.v[7] = __uint_as_float(w.r.w & 0xffff0000u);
  return o;
}
__device__ __forceinline__ F8 raw_to_f8(const Raw8<__half>& w) {
  const uint32_t u[4] = {w.r.x, w.r.y, w.r.z, w.r.w};
  F8 o;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u[i]));
    o.v[2 * i] = f.x; o.v[2 * i + 1] = f.y;
  }
  return o;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// dispatch a generic lambda on the latent dtype
#define VQB_DISPATCH_DTYPE(dtype, T, ...)                                                    \
  switch (dtype) {                                                                           \
    case VQB_F32:  { using T = float;          __VA_ARGS__; break; }                          \
    case VQB_BF16: { using T = __nv_bfloat16;  __VA_ARGS__; break; }                          \
    case VQB_F16:  { using T = __half;         __VA_ARGS__; break; }                          \
    default: vqb::set_error("unknown latent dtype %d", (int)(dtype)); return VQB_ERR_INVALID; \
  }

inline int dtype_size(int dt) { return dt == VQB_F32 ? 4 : 2; }

// ---- internal launchers (defined across the .cu files) --------------------------------------
// rows_per_head maps a row to its codebook's header in op.chdr
int launch_prepare_latents(const void* x, int x_dtype, int64_t rows, int64_t rows_per_head, int d,
                           const LatentOperand& op, cudaStream_t st);
// derive_dx_dp > 0: the residual bound |x - x~| is not in scal[kScalDxMax] but derived from scal[kScalXMax] by dx_bound_16bit()
// (16-bit latents converted inside the search kernel: search_tc.cu, CONV)
int launch_make_bias(const void* cache, const CacheLayout& CL, int64_t H, int K, int metric,
                     uint32_t* scal, float* bias, float* err, __half* caug, cudaStream_t st, int derive_dx_dp = 0);
// In-kernel conversion of 16-bit latents (search_tc.cu, CONV): scal[kScalXMax] = bound of the row norms from a strided sample
// (times kSampleGuard); the search kernel converts every row itself and sends rows that exceed the bound to the exact
// rescan (negative xinv), so the bound only has to be right for the rows that keep their tensor-core candidates.
// conv_outlier_bound_kernel (search_resolve.cu) then raises scal[kScalDxMax] to the norm bound of those rows, so that
// scal[kScalXMax] + scal[kScalDxMax] bounds max|x_j| over the whole batch, as a search workspace promises the EMA kernels (vqb.h).
int launch_sample_bound(const void* x, int x_dtype, int64_t rows, int d, uint32_t* scal, cudaStream_t st);
// *out = max|x_i| over n elements, exactly (atomicMax of the float bits; *out must be 0 or a smaller bound before)
int launch_absmax(const void* x, int x_dtype, int64_t n, uint32_t* out, cudaStream_t st);
struct ConvArgs {
  const void* x = nullptr;   // raw latents [H][N][d], bf16 or fp16; nullptr: operands were prepared by a separate pass
  int x_dtype = 0;
  int d = 0;
};
// xaug / caug: the bias k-step operands (not read when aug_mode is 0)
// aug_mode (search_tc_aug_mode): 0 = one row tile per codebook: search_tc_kernel adds the bias in the epilogue from
// `bias`; 1 = search_aug_kernel, bias as an extra MMA k-step; 2 = search_aug_kernel without the k-step (dot metric,
// no padded codes)
// xn2 / tie: per-row bound of |x|^2 and the tie-window coefficient (kTieSlack for the Euclidean metric, 0 for dot)
int launch_search_tc(const __half* xb, const float* xinv, const float* xn2, float tie, const __half* xaug,
                     const __half* cb, const __half* caug, const float* chdr, const float* bias, int aug_mode,
                     int64_t H, int64_t N, int K, int dp, void* cand, uint32_t* scal, bool timing, cudaStream_t st,
                     const ConvArgs& conv = ConvArgs());
int search_tc_aug_mode(int64_t N, int K, int metric);
// 1 when the search kernel converts 16-bit latents itself (no separate prepare pass) for this problem
int search_tc_conv_ok(int64_t N, int K, int d, int x_dtype, int aug_mode, int requested);

int launch_loss_finalize(const double* part, const long long* cntp, int nblocks, int d, float* loss_out,
                         cudaStream_t st);

// Row scale for the tensor-core operand and the bias operand a = s 2^-q that goes with it: s is the natural
// power-of-two scale (max|x~| in [2^13, 2^14)), lowered if needed so that a <= 2^15 stays an fp16 number
// (a smaller s only moves x~ down inside fp16's 40 binades; the rounding residual is MEASURED, not assumed).
// Returns a, or 0 when a would fall below fp16's smallest subnormal (such rows are rescanned exactly).
__device__ __forceinline__ float clamp_row_scale(float& s, float two_q, float two_mq) {
  const float cap = 32768.f * two_q;           // a = s 2^-q <= 2^15
  if (s > cap) s = cap;
  const float a = s * two_mq;
  return a >= 5.9604645e-8f ? a : 0.f;          // 2^-24
}

// The reference's distance is sqrtf(max(float(|x|^2 + |c|^2 - 2 x.c), 0)): fp32 rounding of the squared distance and of
// the root collapses codes whose exact scores differ by less than ~2^-21 of |x - c|^2 / 2 into EQUAL distances, and
// torch.argmax then takes the lowest index.  Every code that can tie with the winner must therefore be a candidate:
// the window is widened by kTieSlack * (bound of |x|^2) (+ the |score| part, covered by the packing slack).
constexpr float kTieSlack = 5.0e-7f;
// upper bound of |x|^2 from |x~|^2 and |x - x~|^2
__device__ __forceinline__ float row_norm2_bound(float n2, float r2) {
  return (n2 + 2.f * sqrtf(n2 * r2) + r2) * 1.0001f;
}

// 16-bit latents times a power of two are fp16 numbers unless they land in fp16's subnormal range, where the rounding
// error is at most 2^-25 per element: |x - x~| <= sqrt(dp) 2^-25 / s_row, and 1 / s_row <= max(|x|_max 2^-13,
// 1 / cap) with cap = 2^15 2^q the clamp of clamp_row_scale (two_mq = 2^-q).  Bound for every row with |x| <= xmax.
constexpr float kSampleGuard = 1.125f;
__device__ __forceinline__ float dx_bound_16bit(float xmax, int dp, float two_mq) {
  const float inv_s = fmaxf(xmax * 1.220703125e-4f, two_mq * 3.0517578125e-5f);     // 2^-13, 2^-15
  return sqrtf((float)dp) * 2.9802322e-8f * inv_s * 1.01f;
}

// pow2_scale(m) from the exponent field (same value for every input, a handful of integer instructions)
__device__ __forceinline__ float pow2_scale_bits(float m) {
  const uint32_t ef = (__float_as_uint(m) >> 23) & 0xffu;
  if (!(m > 0.f) || ef == 0xffu) return 1.f;
  int sh = 14 - ((int)ef - 126);            // m < 2^(ef-126); denormals: ef = 0 -> clamped below
  if (sh > 100) sh = 100;
  if (sh < -100) sh = -100;
  return __uint_as_float((uint32_t)(127 + sh) << 23);
}
// 1 / s for a normal power of two s
__device__ __forceinline__ float pow2_recip(float s) { return __uint_as_float(0x7F000000u - __float_as_uint(s)); }

// power-of-two scale that brings a magnitude bound m below 2^14 (fp16 max is 65504)
__host__ __device__ inline float pow2_scale(float m) {
  if (!(m > 0.f) || !isfinite(m)) return 1.f;
  int e = ilogbf(m) + 1;                 // m < 2^e
  int sh = 14 - e;
  if (sh > 100) sh = 100;
  if (sh < -100) sh = -100;
  return ldexpf(1.f, sh);
}

// Bits of the bound of sqrt(max2), max2 the largest of a batch's fp32 sums of squares over dp terms (|x~|^2 or
// |x - x~|^2): the sum is inflated by (1 + dp 2.4e-7) for its roundings before the square root.  Non-negative floats
// order like their bits, so atomicMax of these raises scal[kScalXMax] / scal[kScalDxMax].
__device__ __forceinline__ uint32_t batch_bound_bits(float max2, int dp) {
  const float infl = 1.f + (float)dp * 2.4e-7f;
  return __float_as_uint(sqrtf(max2 * infl) * 1.00001f);
}

}  // namespace vqb
