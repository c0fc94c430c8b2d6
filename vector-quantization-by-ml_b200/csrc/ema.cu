// ema.cu -- EMA codebook statistics and refresh.
//
// Replaces (reference file:line under vector_quantization/):
//   codebooks.py:405-408  masked one-hot column sums        -> per-code counts (exact integers)
//   codebooks.py:413      einsum("h n d, h n c -> h c d")   -> per-code sums of assigned rows (a third 2NKd SGEMM)
//   codebooks.py:411,417  ema_inplace (lerp_)               \
//   codebooks.py:419-425  laplace smoothing, divide, l2norm  > vqb_ema_apply
//   codebooks.py:241-243  dead-code replacement scatter      -> vqb_expire_scatter
//
// Reduction = sort-and-segment: a counting sort of row ids by code (histogram, scan, placement), then
// warps walk fixed 64-row chunks of the sorted order, gather each row once (coalesced 4d-byte reads)
// and accumulate per lane in registers, flushing at every code boundary.
// Determinism: the per-row contributions are converted to 64-bit fixed point (scale 2^s chosen from a
// bound on max|x| so that nothing can overflow) and added as INTEGERS -- integer addition is associative,
// so the result is bitwise independent of placement order, chunking and atomics, and its error
// (<= count * 2^-(s+1) absolute, s ~ 39 for unit-scale data) is far below one fp32 ulp of the sum.
// HBM traffic: x once (4d or 2d bytes/row) + 2 x idx + row-id permutation + K(d+1) accumulators.
#include "common.cuh"

namespace vqb {

constexpr int kChunkRows = 64;

struct EmaLayout {
  size_t off_counts;   // u32 [H][K]
  size_t off_cursor;   // u32 [H][K]
  size_t off_start;    // u32 [H][K+1]
  size_t off_scale;    // i32 [4]   s, and fp bound
  size_t off_acc;      // i64 [H][K][d]
  size_t zero_bytes;   // counts + cursor + start + scale + acc are zeroed together
  size_t off_sorted;   // i32 [H][N]
  size_t off_total;    // f32 [H]   (ema_apply scratch)
  size_t off_table;    // u32 [H][kSortBlocks][K]  per-block histograms / offsets of the counting sort (K <= kSortMaxK)
  size_t total;
};
constexpr int kSortBlocks = 148;       // one block per SM
constexpr int kSortMaxK = 12288;       // 48 KB of shared-memory counters per block
inline EmaLayout ema_layout(int64_t H, int64_t N, int K, int d) {
  EmaLayout L;
  size_t o = 0;
  L.off_counts = o; o += align_up((size_t)H * K * 4);
  L.off_cursor = o; o += align_up((size_t)H * K * 4);
  L.off_start = o;  o += align_up((size_t)H * (K + 1) * 4);
  L.off_scale = o;  o += 256;
  L.off_acc = o;    o += align_up((size_t)H * K * d * 8);
  L.zero_bytes = o;
  L.off_sorted = o; o += align_up((size_t)(H * N > 0 ? H * N : 1) * 4);
  L.off_total = o;  o += align_up((size_t)H * 4);
  L.off_table = o;  o += K <= kSortMaxK ? align_up((size_t)H * kSortBlocks * K * 4) : 0;
  L.total = o;
  return L;
}

// --- bound on max|x_j| when the caller has none: one extra read of x ---------------------------------
template <typename T>
__global__ void absmax_kernel(const T* __restrict__ x, int64_t n, uint32_t* __restrict__ out) {
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(to_f32<T>(x[i])));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));
}

int launch_absmax(const void* x, int x_dtype, int64_t n, uint32_t* out, cudaStream_t st) {
  VQB_DISPATCH_DTYPE(x_dtype, T, absmax_kernel<T><<<1184, 256, 0, st>>>((const T*)x, n, out));
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

// s = 61 - ceil(log2(bound * rows)), clamped; scale[0] = s
__global__ void ema_scale_kernel(const float* __restrict__ bound2, const uint32_t* __restrict__ own_bound,
                                 int64_t rows, int* __restrict__ scale) {
  float b = bound2 ? (bound2[0] + bound2[1]) : __uint_as_float(own_bound[0]);
  if (!(b > 0.f) || !isfinite(b)) b = 1.f;
  int e;
  frexpf(b, &e);                              // b < 2^e
  int lr = 0;
  while (((int64_t)1 << lr) < rows + 1) ++lr; // rows < 2^lr
  int s = 61 - (e + lr);
  if (s > 100) s = 100;
  if (s < -60) s = -60;
  scale[0] = s;
}

__global__ void ema_hist_kernel(const int64_t* __restrict__ idx, const uint8_t* __restrict__ mask, int64_t N, int K,
                                uint32_t* __restrict__ counts) {
  const int h = blockIdx.y;
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  if (mask && !mask[n]) return;
  const int64_t k = idx[(int64_t)h * N + n];
  if (k >= 0 && k < K) atomicAdd(counts + (int64_t)h * K + k, 1u);
}

// exclusive scan of counts -> start (one block per codebook; K <= 2^24)
__global__ void ema_scan_kernel(const uint32_t* __restrict__ counts, int K, uint32_t* __restrict__ start) {
  const int h = blockIdx.x;
  const uint32_t* c = counts + (int64_t)h * K;
  uint32_t* s = start + (int64_t)h * (K + 1);
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < K; base += 1024) {
    const int k = base + threadIdx.x;
    const uint32_t v = k < K ? c[k] : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint32_t w = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += t;
      }
      wsum[lane] = w;   // inclusive over warps
    }
    __syncthreads();
    const uint32_t before = carry + (warp ? wsum[warp - 1] : 0u) + inc - v;
    if (k < K) s[k] = before;
    __syncthreads();
    if (threadIdx.x == 1023) carry = before + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) s[K] = carry;
}

__global__ void ema_place_kernel(const int64_t* __restrict__ idx, const uint8_t* __restrict__ mask, int64_t N, int K,
                                 const uint32_t* __restrict__ start, uint32_t* __restrict__ cursor,
                                 int* __restrict__ sorted) {
  const int h = blockIdx.y;
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  if (mask && !mask[n]) return;
  const int64_t k = idx[(int64_t)h * N + n];
  if (k < 0 || k >= K) return;
  const uint32_t pos = start[(int64_t)h * (K + 1) + k] + atomicAdd(cursor + (int64_t)h * K + k, 1u);
  sorted[(int64_t)h * N + pos] = (int)n;
}


// ---------------------------------------------------------------------------------------------------------------
// Counting sort of the rows by code WITHOUT global atomics (K <= kSortMaxK): block b of kSortBlocks owns a contiguous
// range of rows; (1) histogram of its rows in shared memory -> table[b][k]; (2) per code, an exclusive prefix over the
// blocks (table[b][k] becomes the offset of block b inside the code's segment), then the usual exclusive scan over the
// codes (start[k]); (3) each block places its rows with shared-memory cursors starting at start[k] + table[b][k].
// The global-atomic form (ema_hist / ema_place: one atomic per row on K addresses) took 45 us of a C2 step and of
// every C4 level; larger codebooks keep it.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
sort_hist_kernel(const int64_t* __restrict__ idx, const uint8_t* __restrict__ mask, int64_t N, int K,
                 uint32_t* __restrict__ table) {
  extern __shared__ uint32_t s_cnt[];
  const int h = blockIdx.y, b = blockIdx.x, B = gridDim.x;
  for (int k = threadIdx.x; k < K; k += blockDim.x) s_cnt[k] = 0u;
  __syncthreads();
  const int64_t span = (N + B - 1) / B, r0 = (int64_t)b * span, r1 = r0 + span < N ? r0 + span : N;
  for (int64_t n = r0 + threadIdx.x; n < r1; n += blockDim.x) {
    if (mask && !mask[n]) continue;
    const int64_t k = idx[(int64_t)h * N + n];
    if (k >= 0 && k < K) atomicAdd(s_cnt + k, 1u);
  }
  __syncthreads();
  uint32_t* t = table + ((int64_t)h * B + b) * K;
  for (int k = threadIdx.x; k < K; k += blockDim.x) t[k] = s_cnt[k];
}

// one thread per code: table[b][k] -> exclusive prefix over the blocks b; counts[k] = total          grid (ceil(K/256), H)
__global__ void __launch_bounds__(256)
sort_prefix_kernel(uint32_t* __restrict__ table, int B, int K, uint32_t* __restrict__ counts) {
  const int h = blockIdx.y;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  uint32_t* t = table + (int64_t)h * B * K + k;
  uint32_t v = 0u;
  int b = 0;
  for (; b + 8 <= B; b += 8) {                     // 8 independent loads in flight
    uint32_t x[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) x[u] = t[(int64_t)(b + u) * K];
#pragma unroll
    for (int u = 0; u < 8; ++u) { t[(int64_t)(b + u) * K] = v; v += x[u]; }
  }
  for (; b < B; ++b) { const uint32_t x = t[(int64_t)b * K]; t[(int64_t)b * K] = v; v += x; }
  counts[(int64_t)h * K + k] = v;
}

__global__ void __launch_bounds__(1024)
sort_place_kernel(const int64_t* __restrict__ idx, const uint8_t* __restrict__ mask, int64_t N, int K,
                  const uint32_t* __restrict__ start, const uint32_t* __restrict__ table, int* __restrict__ sorted) {
  extern __shared__ uint32_t s_cur[];
  const int h = blockIdx.y, b = blockIdx.x, B = gridDim.x;
  const uint32_t* t = table + ((int64_t)h * B + b) * K;
  const uint32_t* st = start + (int64_t)h * (K + 1);
  for (int k = threadIdx.x; k < K; k += blockDim.x) s_cur[k] = st[k] + t[k];
  __syncthreads();
  const int64_t span = (N + B - 1) / B, r0 = (int64_t)b * span, r1 = r0 + span < N ? r0 + span : N;
  for (int64_t n = r0 + threadIdx.x; n < r1; n += blockDim.x) {
    if (mask && !mask[n]) continue;
    const int64_t k = idx[(int64_t)h * N + n];
    if (k < 0 || k >= K) continue;
    sorted[(int64_t)h * N + atomicAdd(s_cur + k, 1u)] = (int)n;
  }
}

// rows of every codebook sorted by code: counts, start (exclusive scan) and the permutation `sorted`
static int launch_code_sort(const int64_t* idx, const uint8_t* mask, int64_t H, int64_t N, int K, uint32_t* counts,
                            uint32_t* cursor, uint32_t* start, int* sorted, uint32_t* table, cudaStream_t st) {
  if (K <= kSortMaxK && table != nullptr && N >= 4096) {
    const dim3 g((unsigned)kSortBlocks, (unsigned)H);
    const size_t smem = (size_t)K * 4;
    sort_hist_kernel<<<g, 1024, smem, st>>>(idx, mask, N, K, table);
    VQB_LAUNCH_CHECK();
    sort_prefix_kernel<<<dim3((unsigned)((K + 255) / 256), (unsigned)H), 256, 0, st>>>(table, kSortBlocks, K, counts);
    VQB_LAUNCH_CHECK();
    ema_scan_kernel<<<(unsigned)H, 1024, 0, st>>>(counts, K, start);
    VQB_LAUNCH_CHECK();
    sort_place_kernel<<<g, 1024, smem, st>>>(idx, mask, N, K, start, table, sorted);
    VQB_LAUNCH_CHECK();
    return VQB_OK;
  }
  dim3 g1((unsigned)((N + 255) / 256), (unsigned)H);
  ema_hist_kernel<<<g1, 256, 0, st>>>(idx, mask, N, K, counts);
  VQB_LAUNCH_CHECK();
  ema_scan_kernel<<<(unsigned)H, 1024, 0, st>>>(counts, K, start);
  VQB_LAUNCH_CHECK();
  ema_place_kernel<<<g1, 256, 0, st>>>(idx, mask, N, K, start, cursor, sorted);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

// one warp per 64 consecutive positions of the sorted order; lanes own columns {cb*128 + lane*4 .. +3}
template <typename T>
__global__ void __launch_bounds__(256, 3)
ema_segsum_kernel(const T* __restrict__ x, const int64_t* __restrict__ idx, const int* __restrict__ sorted,
                  const uint32_t* __restrict__ start, int64_t N, int K, int d, const int* __restrict__ scale_p,
                  unsigned long long* __restrict__ acc) {
  const int h = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int64_t chunk = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t total = start[(int64_t)h * (K + 1) + K];     // rows that take part (mask applied)
  const int64_t p0 = chunk * kChunkRows;
  if (p0 >= total) return;
  const int64_t p1 = p0 + kChunkRows < total ? p0 + kChunkRows : total;
  const float scale = ldexpf(1.f, scale_p[0]);
  const T* xh = x + (int64_t)h * N * d;
  const int64_t* idxh = idx + (int64_t)h * N;
  const int* srt = sorted + (int64_t)h * N;
  unsigned long long* acch = acc + (int64_t)h * K * d;
  const bool vec = (d & 3) == 0;

  // row ids and codes of the chunk live in registers (2 per lane) and are broadcast with shuffles,
  // so the only dependent memory access in the row loop is the row itself
  const int n = (int)(p1 - p0);
  const int r_lo = lane < n ? srt[p0 + lane] : 0;
  const int r_hi = lane + 32 < n ? srt[p0 + 32 + lane] : 0;
  const int k_lo = lane < n ? (int)idxh[r_lo] : -1;
  const int k_hi = lane + 32 < n ? (int)idxh[r_hi] : -1;

  if ((d & 7) == 0) {
    // column blocks of 256 (8 per lane: one 16-byte load per row for 16-bit latents)
    for (int c0 = 0; c0 < d; c0 += 256) {
      const int j = c0 + lane * 8;
      const bool on = j < d;
      long long a[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) a[e] = 0;
      int cur = -1;
      for (int i0 = 0; i0 < n; i0 += 4) {
        F8 v[4];
        int kk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {            // 4 independent row loads in flight
          const int i = i0 + u;
          const int r = __shfl_sync(0xffffffffu, i < 32 ? r_lo : r_hi, i & 31);
          kk[u] = __shfl_sync(0xffffffffu, i < 32 ? k_lo : k_hi, i & 31);
          if (i < n && on) v[u] = load8<T>(xh + (int64_t)r * d + j);
          else {
#pragma unroll
            for (int e = 0; e < 8; ++e) v[u].v[e] = 0.f;
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (i0 + u < n) {
            if (kk[u] != cur) {                   // warp-uniform: code boundary -> flush
              if (cur >= 0 && on) {
                unsigned long long* o = acch + (int64_t)cur * d + j;
#pragma unroll
                for (int e = 0; e < 8; ++e) if (a[e]) atomicAdd(o + e, (unsigned long long)a[e]);
              }
#pragma unroll
              for (int e = 0; e < 8; ++e) a[e] = 0;
              cur = kk[u];
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) a[e] += __float2ll_rn(v[u].v[e] * scale);
          }
        }
      }
      if (cur >= 0 && on) {
        unsigned long long* o = acch + (int64_t)cur * d + j;
#pragma unroll
        for (int e = 0; e < 8; ++e) if (a[e]) atomicAdd(o + e, (unsigned long long)a[e]);
      }
    }
    return;
  }

  for (int c0 = 0; c0 < d; c0 += 128) {        // column block of 128 (4 per lane)
    const int j = c0 + lane * 4;
    const bool on = j < d;
    long long a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    int cur = -1;
    for (int i0 = 0; i0 < n; i0 += 4) {
      float4 v[4];
      int kk[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {            // 4 independent row loads in flight
        const int i = i0 + u;
        const int r = __shfl_sync(0xffffffffu, i < 32 ? r_lo : r_hi, i & 31);
        kk[u] = __shfl_sync(0xffffffffu, i < 32 ? k_lo : k_hi, i & 31);
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n && on) {
          const T* xr = xh + (int64_t)r * d + j;
          if (vec) v[u] = load4<T>(xr);
          else {
            v[u].x = to_f32<T>(xr[0]);
            v[u].y = j + 1 < d ? to_f32<T>(xr[1]) : 0.f;
            v[u].z = j + 2 < d ? to_f32<T>(xr[2]) : 0.f;
            v[u].w = j + 3 < d ? to_f32<T>(xr[3]) : 0.f;
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (i0 + u < n) {
          if (kk[u] != cur) {                   // warp-uniform: code boundary -> flush
            if (cur >= 0 && on) {
              unsigned long long* o = acch + (int64_t)cur * d + j;
              if (a0) atomicAdd(o + 0, (unsigned long long)a0);
              if (j + 1 < d && a1) atomicAdd(o + 1, (unsigned long long)a1);
              if (j + 2 < d && a2) atomicAdd(o + 2, (unsigned long long)a2);
              if (j + 3 < d && a3) atomicAdd(o + 3, (unsigned long long)a3);
            }
            a0 = a1 = a2 = a3 = 0;
            cur = kk[u];
          }
          a0 += __float2ll_rn(v[u].x * scale);
          a1 += __float2ll_rn(v[u].y * scale);
          a2 += __float2ll_rn(v[u].z * scale);
          a3 += __float2ll_rn(v[u].w * scale);
        }
      }
    }
    if (cur >= 0 && on) {
      unsigned long long* o = acch + (int64_t)cur * d + j;
      if (a0) atomicAdd(o + 0, (unsigned long long)a0);
      if (j + 1 < d && a1) atomicAdd(o + 1, (unsigned long long)a1);
      if (j + 2 < d && a2) atomicAdd(o + 2, (unsigned long long)a2);
      if (j + 3 < d && a3) atomicAdd(o + 3, (unsigned long long)a3);
    }
  }
}

// stats[h][k][:d] = fixed -> float, stats[h][k][d] = count
__global__ void ema_finalize_kernel(const long long* __restrict__ acc, const uint32_t* __restrict__ counts,
                                    const int* __restrict__ scale_p, int64_t HK, int d, float* __restrict__ stats) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = HK * (d + 1);
  if (i >= n) return;
  const int64_t k = i / (d + 1);
  const int j = (int)(i - k * (d + 1));
  if (j == d) stats[i] = (float)counts[k];
  else stats[i] = (float)ldexp((double)acc[k * d + j], -scale_p[0]);
}


// ---------------------------------------------------------------------------------------------------
// Fused tail of the training step: gather + straight-through + commitment loss + EMA sums in ONE pass
// over the latents, walking them in code-sorted order (vqb_quantize_ema).  A row is read once; the code
// row stays in registers for the whole run of rows assigned to it.
//   lanes: LPR = d/8 lanes (d <= 256) or 32 lanes x NB column blocks (d = 512) own 8 columns each of a row;
//          a warp therefore works on RPI = 32/LPR rows at a time, each lane group with its own running segment.
//   sums : fixed point by the "magic constant" trick -- t = v + M1 rounds v to a multiple of q1 = ulp(M1) and the
//          integer v/q1 is bits(t) - bits(M1): one FADD + one IADD per element instead of a 64-bit F2I (16/clk/SM).
//          fp32 latents add a second term for the rounding error v - (t - M1) (exact, Fast2Sum) with quantum
//          q2 = 2^-(P-22) q1, so the result carries P <= 44 bits below the bound; 16-bit latents (8 / 11 significant
//          bits) are already exact down to 2^-14 / 2^-11 of the bound with one term.  Integer sums are associative:
//          the result does not depend on the (atomic) placement order -- bitwise reproducible.
//   loss : (c - x)^2 summed per row in a fixed lane order, one float per row, reduced afterwards in a fixed tree.
struct FusedScale { int s; int pad; int e; int P; };   // ws scale block: quantum 2^-s, |v| < 2^e, P total bits

__global__ void fused_scale_kernel(const float* __restrict__ bound2, const uint32_t* __restrict__ own_bound,
                                   int64_t rows, int two_terms, int* __restrict__ scale) {
  float b = bound2 ? (bound2[0] + bound2[1]) : __uint_as_float(own_bound[0]);
  if (!(b > 0.f) || !isfinite(b)) b = 1.f;
  int e;
  frexpf(b, &e);                  // b < 2^e
  e += 1;                         // one binade of head room: t = v + M1 never reaches the next binade
  if (e > 100) e = 100;
  if (e < -100) e = -100;
  int lr = 0;
  while (((int64_t)1 << lr) < rows + 1) ++lr;
  int P = 22;
  if (two_terms) { P = 62 - lr; if (P > 44) P = 44; }
  scale[0] = P - e;               // value = integer * 2^(e-P)
  scale[2] = e;
  scale[3] = P;
}


constexpr int kFusedChunkRows = 128;   // sorted positions per warp in the fused pass

// ResidualVQ level extras (RVQ = true, H = 1, fp32 residual): the same pass also does residual_vq.py:232-233 and prepares
// the next level's search operand (what vqb_rvq_level does in row order):
//   out = first ? 0 + q : out + q ;  r_next = r - q ;  next operand = scaled fp16 of r_next + row scale + bias operand
struct RvqExtra {
  float* out;             // (N,d) running sum of the levels' outputs, updated in place
  float* res_out;         // (N,d) next residual
  float* q_level;         // (N,d) this level's output, nullable
  __half* next_xb;        // nullable: no next level
  float* next_xinv;
  float* next_xn2;
  __half* next_xaug;
  uint32_t* next_scal;
  const float* next_chdr;
  int first;
  int dp;
};

template <typename T, int NB, int TERMS, bool RVQ>
__global__ void __launch_bounds__(256, 2)
quantize_ema_kernel(const T* __restrict__ x, const float* __restrict__ cb, const int64_t* __restrict__ idx,
                    const int* __restrict__ sorted, const uint32_t* __restrict__ start, int64_t N, int K, int d,
                    int training, const int* __restrict__ scale_p, float* __restrict__ q,
                    float* __restrict__ loss_rows, unsigned long long* __restrict__ acc, const RvqExtra R) {
  // rows in flight per lane group: 32 registers of raw data (half of that in the register-hungry RVQ form)
  constexpr int U0 = (sizeof(T) == 2 ? 8 : 4) / NB;
  constexpr int U = RVQ ? (U0 > 1 ? U0 / 2 : 1) : U0;
  const int h = blockIdx.y;
  const int lane = threadIdx.x & 31;
  const int64_t chunk = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t total = start[(int64_t)h * (K + 1) + K];
  const int64_t p0 = chunk * kFusedChunkRows;
  if (p0 >= total) return;
  const int n = (int)((p0 + kFusedChunkRows < total ? p0 + kFusedChunkRows : total) - p0);
  const int lpr = NB == 1 ? d >> 3 : 32;        // lanes per row
  const int rpi = 32 / lpr;                     // rows per warp iteration
  const int grp = lane / lpr, gl = lane - grp * lpr;
  const int j = gl * 8;                         // first owned column (of column block 0)
  const int e = scale_p[2], P = scale_p[3];
  const float M1 = ldexpf(1.5f, e + 1);         // ulp(M1) = 2^(e-22)
  const float M2 = ldexpf(1.5f, e + 23 - P);    // ulp(M2) = 2^(e-P)
  const uint32_t M1b = __float_as_uint(M1), M2b = __float_as_uint(M2);
  const int shift = P - 22;
  const T* xh = x + (int64_t)h * N * d;
  const float* cbh = cb + (int64_t)h * K * d;
  const int64_t* idxh = idx + (int64_t)h * N;
  const int* srt = sorted + (int64_t)h * N;
  float* qh = q + (int64_t)h * N * d;
  unsigned long long* acch = acc + (int64_t)h * K * d;

  // row ids and codes of the chunk: 4 registers each per lane, broadcast with shuffles in the row loop
  int rid[4], kid[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    rid[t] = lane + 32 * t < n ? srt[p0 + 32 * t + lane] : 0;
    kid[t] = lane + 32 * t < n ? (int)idxh[rid[t]] : -1;
  }

  uint32_t sh[NB][8], sl[NB][8];                // wrapped sums of bits(t) (and bits(t2))
  float c[NB][8];
#pragma unroll
  for (int b = 0; b < NB; ++b)
#pragma unroll
    for (int t = 0; t < 8; ++t) { sh[b][t] = 0u; sl[b][t] = 0u; c[b][t] = 0.f; }
  int cur = -1;
  uint32_t cnt = 0;                             // rows in the open segment of this lane group
  float max_n2 = 0.f, max_r2 = 0.f;             // RVQ: statistics of the next level's operand

  auto flush = [&]() {
    if (cur >= 0) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        unsigned long long* o = acch + (int64_t)cur * d + b * 256 + j;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          long long v = (long long)(int)(sh[b][t] - cnt * M1b);
          if (TERMS == 2) v = (v << shift) + (long long)(int)(sl[b][t] - cnt * M2b);
          if (v) atomicAdd(o + t, (unsigned long long)v);
          sh[b][t] = 0u; sl[b][t] = 0u;
        }
      }
    }
    cnt = 0;
  };

  for (int i0 = 0; i0 < n; i0 += U * rpi) {
    Raw8<T> raw[U][NB];
    int kk[U], rr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {               // U independent row loads in flight per group
      const int i = i0 + u * rpi + grp;
      const int w = (i >> 5) & 3;
      const int rsel = w == 0 ? rid[0] : (w == 1 ? rid[1] : (w == 2 ? rid[2] : rid[3]));
      const int ksel = w == 0 ? kid[0] : (w == 1 ? kid[1] : (w == 2 ? kid[2] : kid[3]));
      rr[u] = __shfl_sync(0xffffffffu, rsel, i & 31);
      kk[u] = __shfl_sync(0xffffffffu, ksel, i & 31);
      if (i >= n) kk[u] = -1;
#pragma unroll
      for (int b = 0; b < NB; ++b)
        raw[u][b] = load_raw8<T>(xh + (int64_t)(kk[u] >= 0 ? rr[u] : 0) * d + b * 256 + j);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float sq = 0.f;
      F8 rn[NB];                                // RVQ: the new residual stays in registers for the fp16 conversion
      float mabs = 0.f;
      if (RVQ) {
#pragma unroll
        for (int b = 0; b < NB; ++b)
#pragma unroll
          for (int t = 0; t < 8; ++t) rn[b].v[t] = 0.f;
      }
      if (kk[u] >= 0) {
        if (kk[u] != cur) {                     // group-uniform: segment boundary
          flush();
          cur = kk[u];
#pragma unroll
          for (int b = 0; b < NB; ++b) {
            const float4 a0 = __ldg(reinterpret_cast<const float4*>(cbh + (int64_t)cur * d + b * 256 + j));
            const float4 a1 = __ldg(reinterpret_cast<const float4*>(cbh + (int64_t)cur * d + b * 256 + j) + 1);
            c[b][0] = a0.x; c[b][1] = a0.y; c[b][2] = a0.z; c[b][3] = a0.w;
            c[b][4] = a1.x; c[b][5] = a1.y; c[b][6] = a1.z; c[b][7] = a1.w;
          }
        }
        ++cnt;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          float o[8];
          const F8 v = raw_to_f8(raw[u][b]);
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const float xv = v.v[t];
            const float df = __fsub_rn(c[b][t], xv);
            o[t] = training ? __fadd_rn(xv, df) : c[b][t];
            sq = fmaf(df, df, sq);
            const float t1 = __fadd_rn(xv, M1);
            sh[b][t] += __float_as_uint(t1);
            if (TERMS == 2) {
              const float lo = __fsub_rn(xv, __fsub_rn(t1, M1));
              sl[b][t] += __float_as_uint(__fadd_rn(lo, M2));
            }
          }
          const int64_t off = (int64_t)rr[u] * d + b * 256 + j;
          if (!RVQ) {
            __stcs(reinterpret_cast<float4*>(qh + off), make_float4(o[0], o[1], o[2], o[3]));
            __stcs(reinterpret_cast<float4*>(qh + off) + 1, make_float4(o[4], o[5], o[6], o[7]));
          } else {
            if (R.out) {                          // NULL: the caller sums the levels afterwards (vqb_rvq_replay_out)
            float acc8[8];
            if (R.first) {
#pragma unroll
              for (int t = 0; t < 8; ++t) acc8[t] = __fadd_rn(0.f, o[t]);
            } else {
              const float4 p0 = *reinterpret_cast<const float4*>(R.out + off), p1 = *(reinterpret_cast<const float4*>(R.out + off) + 1);
              const float pv[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
#pragma unroll
              for (int t = 0; t < 8; ++t) acc8[t] = __fadd_rn(pv[t], o[t]);
            }
            *reinterpret_cast<float4*>(R.out + off) = make_float4(acc8[0], acc8[1], acc8[2], acc8[3]);
            *(reinterpret_cast<float4*>(R.out + off) + 1) = make_float4(acc8[4], acc8[5], acc8[6], acc8[7]);
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              rn[b].v[t] = __fsub_rn(v.v[t], o[t]);
              mabs = fmaxf(mabs, fabsf(rn[b].v[t]));
            }
            *reinterpret_cast<float4*>(R.res_out + off) = make_float4(rn[b].v[0], rn[b].v[1], rn[b].v[2], rn[b].v[3]);
            *(reinterpret_cast<float4*>(R.res_out + off) + 1) = make_float4(rn[b].v[4], rn[b].v[5], rn[b].v[6], rn[b].v[7]);
            if (R.q_level) {
              *reinterpret_cast<float4*>(R.q_level + off) = make_float4(o[0], o[1], o[2], o[3]);
              *(reinterpret_cast<float4*>(R.q_level + off) + 1) = make_float4(o[4], o[5], o[6], o[7]);
            }
          }
        }
      }
      if (RVQ && R.next_xb) {                   // next level's operand (shuffles: every lane takes part)
        const bool live = kk[u] >= 0;
        for (int o2 = lpr >> 1; o2 > 0; o2 >>= 1) mabs = fmaxf(mabs, __shfl_xor_sync(0xffffffffu, mabs, o2));
        float s = pow2_scale_bits(mabs);
        const float a = clamp_row_scale(s, R.next_chdr[4], R.next_chdr[5]);
        const float is = pow2_recip(s);
        if (gl == 0 && live) {
          R.next_xinv[rr[u]] = a > 0.f ? is : -is;
          const uint32_t aa = (uint32_t)__half_as_ushort(__float2half_rn(a));
          *reinterpret_cast<uint4*>(R.next_xaug + (int64_t)rr[u] * 8) = make_uint4(aa | (aa << 16), aa, 0u, 0u);
        }
        float n2 = 0.f, r2 = 0.f;
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          uint32_t pk[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float v0 = rn[b].v[2 * t], v1 = rn[b].v[2 * t + 1];
            const __half2 hh = __floats2half2_rn(v0 * s, v1 * s);
            const float2 f = __half22float2(hh);
            pk[t] = *reinterpret_cast<const uint32_t*>(&hh);
            const float b0 = f.x * is, b1 = f.y * is;
            n2 += b0 * b0 + b1 * b1;
            const float e0 = v0 - b0, e1 = v1 - b1;
            r2 += e0 * e0 + e1 * e1;
          }
          if (live)
            *reinterpret_cast<uint4*>(R.next_xb + (int64_t)rr[u] * R.dp + b * 256 + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        for (int o2 = lpr >> 1; o2 > 0; o2 >>= 1) {
          n2 += __shfl_xor_sync(0xffffffffu, n2, o2);
          r2 += __shfl_xor_sync(0xffffffffu, r2, o2);
        }
        if (gl == 0 && live) R.next_xn2[rr[u]] = row_norm2_bound(n2, r2);
        max_n2 = fmaxf(max_n2, n2);
        max_r2 = fmaxf(max_r2, r2);
      }
      if (loss_rows) {                          // fixed-order sum over the lanes of the row
        for (int o2 = lpr >> 1; o2 > 0; o2 >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o2);
        if (kk[u] >= 0 && gl == 0) loss_rows[(int64_t)h * N + rr[u]] = sq;
      }
    }
  }
  flush();
  if (RVQ && R.next_xb) {
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) {
      max_n2 = fmaxf(max_n2, __shfl_xor_sync(0xffffffffu, max_n2, o2));
      max_r2 = fmaxf(max_r2, __shfl_xor_sync(0xffffffffu, max_r2, o2));
    }
    if (lane == 0) {
      const float infl = 1.f + (float)R.dp * 2.4e-7f;
      atomicMax(R.next_scal + 0, __float_as_uint(sqrtf(max_n2 * infl) * 1.00001f));
      atomicMax(R.next_scal + 1, __float_as_uint(sqrtf(max_r2 * infl) * 1.00001f));
      if (blockIdx.x == 0 && threadIdx.x == 0) R.next_scal[7] = __float_as_uint(R.next_chdr[4]);
    }
  }
}

// fixed-order partial sums of the per-row squared errors: block b owns rows [b*span, (b+1)*span)
__global__ void __launch_bounds__(256)
loss_rows_partial_kernel(const float* __restrict__ loss_rows, int64_t rows, int64_t span, double* __restrict__ part,
                         long long* __restrict__ cntp) {
  const int64_t r0 = (int64_t)blockIdx.x * span;
  const int64_t r1 = r0 + span < rows ? r0 + span : rows;
  double t = 0.0;
  for (int64_t r = r0 + threadIdx.x; r < r1; r += 256) t += (double)loss_rows[r];
  __shared__ double s[256];
  s[threadIdx.x] = t;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) { part[blockIdx.x] = s[0]; cntp[blockIdx.x] = r1 > r0 ? r1 - r0 : 0; }
}

constexpr int kLossBlocks = 1024;
struct FusedLayout {
  EmaLayout E;
  size_t off_loss_rows;   // f32 [H*N]
  size_t off_part;        // f64 [kLossBlocks]
  size_t off_cnt;         // i64 [kLossBlocks]
  size_t total;
};
inline FusedLayout fused_layout(int64_t H, int64_t N, int K, int d) {
  FusedLayout L;
  L.E = ema_layout(H, N, K, d);
  size_t o = L.E.total;
  L.off_loss_rows = o; o += align_up((size_t)(H * N > 0 ? H * N : 1) * 4);
  L.off_part = o;      o += align_up((size_t)kLossBlocks * 8);
  L.off_cnt = o;       o += align_up((size_t)kLossBlocks * 8);
  L.total = o;
  return L;
}
inline bool fused_width_ok(int d) { return d == 512 || (d >= 8 && d <= 256 && (d & (d - 1)) == 0); }


// ---------------------------------------------------------------------------------------------------------------
// Column moments of the latents (affine re-parametrisation, reference codebooks.py:300-347: batch mean and biased
// variance over the rows of each codebook's batch): per (h, column) sum and sum of squares over the rows with
// mask != 0, accumulated in fp64 in ONE pass over the latents.  out (H, d, 2) fp64 must be zero; rows_used (H) int64.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kMomentRows = 256;          // rows per block
template <typename T>
__global__ void __launch_bounds__(256)
column_moments_kernel(const T* __restrict__ x, const uint8_t* __restrict__ mask, int64_t N, int d,
                      double* __restrict__ out, long long* __restrict__ rows_used) {
  const int h = blockIdx.y;
  const int64_t r0 = (int64_t)blockIdx.x * kMomentRows;
  const int64_t r1 = r0 + kMomentRows < N ? r0 + kMomentRows : N;
  const T* xh = x + (int64_t)h * N * d;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    double s = 0.0, ss = 0.0;
    for (int64_t r = r0; r < r1; ++r) {
      if (mask && !mask[r]) continue;
      const double v = (double)to_f32<T>(xh[r * d + c]);
      s += v;
      ss = fma(v, v, ss);
    }
    atomicAdd(out + ((int64_t)h * d + c) * 2, s);
    atomicAdd(out + ((int64_t)h * d + c) * 2 + 1, ss);
  }
  if (threadIdx.x == 0) {
    long long n = 0;
    for (int64_t r = r0; r < r1; ++r) n += (!mask || mask[r]) ? 1 : 0;
    atomicAdd(reinterpret_cast<unsigned long long*>(rows_used + h), (unsigned long long)n);
  }
}

// --- apply ------------------------------------------------------------------------------------------
__device__ __forceinline__ float torch_lerp(float a, float b, float w) {
  // ATen lerp: |w| < 0.5 ? a + w*(b-a) : b - (b-a)*(1-w), evaluated with one fma (both the CPU vector
  // kernel and nvcc's contraction do that)
  const float diff = b - a;
  return fabsf(w) < 0.5f ? fmaf(w, diff, a) : fmaf(w - 1.f, diff, b);
}

// one block per codebook: cluster_size <- lerp(cluster_size, counts, w); total[h] = sum(cluster_size)
__global__ void ema_apply_counts_kernel(const float* __restrict__ stats, float* __restrict__ cluster_size, float w,
                                        int K, int d, float* __restrict__ total) {
  const int h = blockIdx.x;
  __shared__ double s[1024];
  double t = 0.0;
  for (int k = threadIdx.x; k < K; k += 1024) {
    const int64_t i = (int64_t)h * K + k;
    const float v = torch_lerp(cluster_size[i], stats[i * (d + 1) + d], w);
    cluster_size[i] = v;
    t += (double)v;
  }
  s[threadIdx.x] = t;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) total[h] = (float)s[0];
}

// one warp per code: embed_avg <- lerp; embeddings <- reg(embed_avg / smoothed)
__global__ void __launch_bounds__(256)
ema_apply_rows_kernel(const float* __restrict__ stats, const float* __restrict__ cluster_size,
                      float* __restrict__ embed_avg, float* __restrict__ embeddings, float w, float eps, float keps,
                      int l2, int64_t H, int K, int d, const float* __restrict__ total) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= H * K) return;
  const int64_t h = row / K;
  const float tot = total[h];
  // laplace_smoothing(cs, K, eps) * cs.sum()   (utils/general.py:154-156, codebooks.py:419-421)
  const float smoothed = __fmul_rn(__fdiv_rn(__fadd_rn(cluster_size[row], eps), __fadd_rn(tot, keps)), tot);
  const float* st = stats + row * (int64_t)(d + 1);
  float* ea = embed_avg + row * (int64_t)d;
  float* em = embeddings + row * (int64_t)d;
  float n2 = 0.f;
  for (int j = lane; j < d; j += 32) {
    const float a = torch_lerp(ea[j], st[j], w);
    ea[j] = a;
    const float e = __fdiv_rn(a, smoothed);
    if (l2) n2 = fmaf(e, e, n2);
    else em[j] = e;
  }
  if (l2) {
    n2 = warp_sum(n2);
    const float nrm = fmaxf(sqrtf(n2), 1e-12f);
    for (int j = lane; j < d; j += 32) em[j] = __fdiv_rn(__fdiv_rn(ea[j], smoothed), nrm);
  }
}

// --- expiry: the j-th dead code (ascending) takes sample row j -------------------------------------------
template <typename T>
__global__ void __launch_bounds__(1024)
expire_scatter_kernel(const T* __restrict__ x, const int64_t* __restrict__ rows, int64_t m, float thr, float reset,
                      int l2, float* __restrict__ cluster_size, float* __restrict__ embed_avg,
                      float* __restrict__ embeddings, int64_t N, int K, int d) {
  __shared__ int dead_k[1024];
  __shared__ uint32_t wsum[32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < K; base += 1024) {
    const int k = base + threadIdx.x;
    const uint32_t dead = (k < K && cluster_size[k] < thr) ? 1u : 0u;
    uint32_t inc = dead;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      uint32_t v = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
      }
      wsum[lane] = v;
    }
    __syncthreads();
    const uint32_t local = (warp ? wsum[warp - 1] : 0u) + inc - dead;   // dead codes before k in this chunk
    const uint32_t ndead = wsum[31];
    const uint32_t c0 = carry;
    if (dead) dead_k[local] = k;
    __syncthreads();
    // warps copy the chunk's dead codes, one code per warp at a time
    for (uint32_t i = warp; i < ndead; i += 32) {
      const int kk = dead_k[i];
      const int64_t j = (int64_t)c0 + i;
      if (j < m) {
        int64_t r = rows[j];
        if (r < 0) r = 0;
        if (r >= N) r = N - 1;
        const T* xr = x + r * (int64_t)d;
        float nrm = 1.f;
        if (l2) {
          float n2 = 0.f;
          for (int c = lane; c < d; c += 32) { const float v = to_f32<T>(xr[c]); n2 = fmaf(v, v, n2); }
          n2 = warp_sum(n2);
          nrm = fmaxf(sqrtf(n2), 1e-12f);
        }
        for (int c = lane; c < d; c += 32) {
          float v = to_f32<T>(xr[c]);
          if (l2) v = __fdiv_rn(v, nrm);
          embeddings[(int64_t)kk * d + c] = v;
          embed_avg[(int64_t)kk * d + c] = __fmul_rn(v, reset);
        }
        if (lane == 0) cluster_size[kk] = reset;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) carry = c0 + ndead;
    __syncthreads();
  }
}

// --- sharded-codebook keys --------------------------------------------------------------------------
__global__ void minkey_pack_kernel(const float* __restrict__ score, const int64_t* __restrict__ idx, int64_t n,
                                   long long* __restrict__ keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t u = __float_as_uint(score[i]);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);       // monotone: float order -> unsigned order
  u ^= 0x80000000u;                                     // unsigned order -> signed int64 order of the packed key
  keys[i] = (long long)(((unsigned long long)u << 32) | (unsigned long long)(uint32_t)idx[i]);
}
__global__ void minkey_unpack_kernel(const long long* __restrict__ keys, int64_t n, int64_t* __restrict__ idx,
                                     float* __restrict__ score) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long kq = (unsigned long long)keys[i];
  idx[i] = (int64_t)(uint32_t)(kq & 0xffffffffull);
  if (score) {
    uint32_t u = (uint32_t)(kq >> 32) ^ 0x80000000u;
    u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
    score[i] = __uint_as_float(u);
  }
}

}  // namespace vqb

using namespace vqb;

extern "C" size_t vqb_ema_workspace_bytes(int64_t H, int64_t N, int K, int d) {
  if (H <= 0 || N < 0 || K <= 0 || d <= 0) return 0;
  return ema_layout(H, N, K, d).total;
}

extern "C" int vqb_ema_reduce(const void* x, int x_dtype, const int64_t* idx, const uint8_t* mask,
                              const float* absmax_bound2, int64_t H, int64_t N, int K, int d, float* stats,
                              void* ws, size_t ws_bytes, void* stream) {
  VQB_REQUIRE(x && idx && stats && ws, VQB_ERR_INVALID, "vqb_ema_reduce: null pointer");
  VQB_REQUIRE(H > 0 && N >= 0 && K > 0 && d > 0 && H < 65536, VQB_ERR_INVALID, "vqb_ema_reduce: bad shape");
  VQB_REQUIRE(N < (1ll << 31), VQB_ERR_UNSUPPORTED, "N must be < 2^31");
  EmaLayout L = ema_layout(H, N, K, d);
  VQB_REQUIRE(ws_bytes >= L.total, VQB_ERR_WORKSPACE, "ema workspace too small: %zu < %zu", ws_bytes, L.total);
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)ws;
  uint32_t* counts = (uint32_t*)(w + L.off_counts);
  uint32_t* cursor = (uint32_t*)(w + L.off_cursor);
  uint32_t* start = (uint32_t*)(w + L.off_start);
  int* scale = (int*)(w + L.off_scale);
  long long* acc = (long long*)(w + L.off_acc);
  int* sorted = (int*)(w + L.off_sorted);
  VQB_CUDA_TRY(cudaMemsetAsync(w, 0, L.zero_bytes, st));
  if (N > 0) {
    if (!absmax_bound2)
      if (int rc = launch_absmax(x, x_dtype, H * N * (int64_t)d, (uint32_t*)(scale + 1), st)) return rc;
    ema_scale_kernel<<<1, 1, 0, st>>>(absmax_bound2, (const uint32_t*)(scale + 1), N, scale);
    VQB_LAUNCH_CHECK();
    if (int rc = launch_code_sort(idx, mask, H, N, K, counts, cursor, start, sorted,
                                  K <= kSortMaxK ? (uint32_t*)(w + L.off_table) : nullptr, st)) return rc;
    const int64_t chunks = (N + kChunkRows - 1) / kChunkRows;
    dim3 g2((unsigned)((chunks + 7) / 8), (unsigned)H);
    VQB_DISPATCH_DTYPE(x_dtype, T,
      ema_segsum_kernel<T><<<g2, 256, 0, st>>>((const T*)x, idx, sorted, start, N, K, d, scale,
                                               (unsigned long long*)acc));
    VQB_LAUNCH_CHECK();
  }
  const int64_t n = H * (int64_t)K * (d + 1);
  ema_finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(acc, counts, scale, H * (int64_t)K, d, stats);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_quantize_ema_supported(int d) { return fused_width_ok(d) ? 1 : 0; }

extern "C" size_t vqb_quantize_ema_workspace_bytes(int64_t H, int64_t N, int K, int d) {
  if (H <= 0 || N < 0 || K <= 0 || d <= 0) return 0;
  return fused_layout(H, N, K, d).total;
}

// shared by vqb_quantize_ema (rvq == nullptr) and vqb_rvq_level_ema
static int quantize_ema_impl(const void* x, int x_dtype, const float* codebook, const int64_t* idx,
                             const float* absmax_bound2, int training, int want_loss, float* q_out,
                             float* loss_out, float* stats, int64_t H, int64_t N, int K, int d, void* ws,
                             size_t ws_bytes, const RvqExtra* rvq, void* stream) {
  VQB_REQUIRE(x && codebook && idx && (q_out || rvq) && stats && ws, VQB_ERR_INVALID, "vqb_quantize_ema: null pointer");
  VQB_REQUIRE(H > 0 && N >= 0 && K > 0 && d > 0 && H < 65536, VQB_ERR_INVALID, "vqb_quantize_ema: bad shape");
  VQB_REQUIRE(N < (1ll << 31), VQB_ERR_UNSUPPORTED, "N must be < 2^31");
  VQB_REQUIRE(fused_width_ok(d), VQB_ERR_UNSUPPORTED, "vqb_quantize_ema: d=%d (need a power of two <= 256, or 512)", d);
  VQB_REQUIRE(!want_loss || loss_out, VQB_ERR_INVALID, "vqb_quantize_ema: loss_out is null");
  FusedLayout L = fused_layout(H, N, K, d);
  VQB_REQUIRE(ws_bytes >= L.total, VQB_ERR_WORKSPACE, "quantize_ema workspace too small: %zu < %zu", ws_bytes, L.total);
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)ws;
  uint32_t* counts = (uint32_t*)(w + L.E.off_counts);
  uint32_t* cursor = (uint32_t*)(w + L.E.off_cursor);
  uint32_t* start = (uint32_t*)(w + L.E.off_start);
  int* scale = (int*)(w + L.E.off_scale);
  long long* acc = (long long*)(w + L.E.off_acc);
  int* sorted = (int*)(w + L.E.off_sorted);
  float* loss_rows = want_loss ? (float*)(w + L.off_loss_rows) : nullptr;
  double* part = (double*)(w + L.off_part);
  long long* cntp = (long long*)(w + L.off_cnt);
  const int two_terms = x_dtype == VQB_F32 ? 1 : 0;
  VQB_CUDA_TRY(cudaMemsetAsync(w, 0, L.E.zero_bytes, st));
  if (N > 0) {
    if (!absmax_bound2)
      if (int rc = launch_absmax(x, x_dtype, H * N * (int64_t)d, (uint32_t*)(scale + 1), st)) return rc;
    fused_scale_kernel<<<1, 1, 0, st>>>(absmax_bound2, (const uint32_t*)(scale + 1), N, two_terms, scale);
    VQB_LAUNCH_CHECK();
    // the next level's statistics usually live in the workspace absmax_bound2 points into: zero them only now
    if (rvq && rvq->next_scal) VQB_CUDA_TRY(cudaMemsetAsync(rvq->next_scal, 0, 8, st));
    if (int rc = launch_code_sort(idx, nullptr, H, N, K, counts, cursor, start, sorted,
                                  K <= kSortMaxK ? (uint32_t*)(w + L.E.off_table) : nullptr, st)) return rc;
    const int64_t chunks = (N + kFusedChunkRows - 1) / kFusedChunkRows;
    dim3 g2((unsigned)((chunks + 7) / 8), (unsigned)H);
#define VQB_QE_LAUNCH(T, NB, TERMS)                                                                          \
    quantize_ema_kernel<T, NB, TERMS, false><<<g2, 256, 0, st>>>((const T*)x, codebook, idx, sorted, start, N, K, d, \
                                                                 training, scale, q_out, loss_rows,              \
                                                                 (unsigned long long*)acc, RvqExtra{})
    if (rvq) {
      if (d == 512)
        quantize_ema_kernel<float, 2, 2, true><<<g2, 256, 0, st>>>((const float*)x, codebook, idx, sorted, start, N, K, d,
                                                                   training, scale, nullptr, loss_rows,
                                                                   (unsigned long long*)acc, *rvq);
      else
        quantize_ema_kernel<float, 1, 2, true><<<g2, 256, 0, st>>>((const float*)x, codebook, idx, sorted, start, N, K, d,
                                                                   training, scale, nullptr, loss_rows,
                                                                   (unsigned long long*)acc, *rvq);
    } else if (d == 512) {
      if (x_dtype == VQB_F32) VQB_QE_LAUNCH(float, 2, 2);
      else if (x_dtype == VQB_BF16) VQB_QE_LAUNCH(__nv_bfloat16, 2, 1);
      else if (x_dtype == VQB_F16) VQB_QE_LAUNCH(__half, 2, 1);
      else { set_error("unknown latent dtype %d", x_dtype); return VQB_ERR_INVALID; }
    } else {
      if (x_dtype == VQB_F32) VQB_QE_LAUNCH(float, 1, 2);
      else if (x_dtype == VQB_BF16) VQB_QE_LAUNCH(__nv_bfloat16, 1, 1);
      else if (x_dtype == VQB_F16) VQB_QE_LAUNCH(__half, 1, 1);
      else { set_error("unknown latent dtype %d", x_dtype); return VQB_ERR_INVALID; }
    }
#undef VQB_QE_LAUNCH
    VQB_LAUNCH_CHECK();
  }
  const int64_t n = H * (int64_t)K * (d + 1);
  ema_finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(acc, counts, scale, H * (int64_t)K, d, stats);
  VQB_LAUNCH_CHECK();
  if (want_loss) {
    const int64_t rows = H * N;
    int nblocks = 0;
    if (rows > 0) {
      const int64_t span = (rows + kLossBlocks - 1) / kLossBlocks;
      nblocks = (int)((rows + span - 1) / span);
      loss_rows_partial_kernel<<<nblocks, 256, 0, st>>>(loss_rows, rows, span, part, cntp);
      VQB_LAUNCH_CHECK();
    }
    int rc = launch_loss_finalize(part, cntp, nblocks, d, loss_out, st);
    if (rc) return rc;
  }
  return VQB_OK;
}

extern "C" int vqb_quantize_ema(const void* x, int x_dtype, const float* codebook, const int64_t* idx,
                                const float* absmax_bound2, int training, int want_loss, float* q_out,
                                float* loss_out, float* stats, int64_t H, int64_t N, int K, int d, void* ws,
                                size_t ws_bytes, void* stream) {
  return quantize_ema_impl(x, x_dtype, codebook, idx, absmax_bound2, training, want_loss, q_out, loss_out, stats, H, N,
                           K, d, ws, ws_bytes, nullptr, stream);
}

extern "C" int vqb_rvq_level_ema_supported(int d) { return (d == 64 || d == 128 || d == 256 || d == 512) ? 1 : 0; }

extern "C" int vqb_rvq_level_ema(const float* residual_in, float* residual_out, const float* codebook,
                                 const int64_t* idx, const float* absmax_bound2, int training, int first_level,
                                 float* quantized_out, float* q_out, float* loss_out, float* stats, int64_t N, int K,
                                 int d, void* ws, size_t ws_bytes, void* next_ws, size_t next_ws_bytes,
                                 const void* next_cache, void* stream) {
  VQB_REQUIRE(residual_in && residual_out && loss_out, VQB_ERR_INVALID, "vqb_rvq_level_ema: null pointer");
  VQB_REQUIRE(vqb_rvq_level_ema_supported(d), VQB_ERR_UNSUPPORTED, "vqb_rvq_level_ema: d=%d (64, 128, 256 or 512)", d);
  VQB_REQUIRE(residual_in != residual_out, VQB_ERR_INVALID, "vqb_rvq_level_ema: rows are visited in code order, the "
              "residual cannot be updated in place");
  RvqExtra R = {};
  R.out = quantized_out; R.res_out = residual_out; R.q_level = q_out; R.first = first_level; R.dp = d_pad(d);
  if (next_ws) {
    VQB_REQUIRE(next_cache != nullptr, VQB_ERR_INVALID, "vqb_rvq_level_ema: next_ws needs next_cache");
    SearchLayout SL = search_layout(1, N, K, d);
    VQB_REQUIRE(next_ws_bytes >= SL.total, VQB_ERR_WORKSPACE, "next-level search workspace too small");
    R.next_xb = (__half*)((char*)next_ws + SL.off_xb);
    R.next_xaug = (__half*)((char*)next_ws + SL.off_xaug);
    R.next_xinv = (float*)((char*)next_ws + SL.off_xinv);
    R.next_xn2 = (float*)((char*)next_ws + SL.off_xn2);
    R.next_scal = (uint32_t*)((char*)next_ws + SL.off_scal);
    R.next_chdr = (const float*)((const char*)next_cache + cache_layout(1, K, d).off_hdr);
  }
  return quantize_ema_impl(residual_in, VQB_F32, codebook, idx, absmax_bound2, training, 1, nullptr, loss_out, stats, 1,
                           N, K, d, ws, ws_bytes, &R, stream);
}

extern "C" int vqb_ema_apply_counts(const float* stats, float* cluster_size, float weight, int64_t H, int K, int d,
                                    float* totals_out, void* stream) {
  VQB_REQUIRE(stats && cluster_size && totals_out, VQB_ERR_INVALID, "vqb_ema_apply_counts: null pointer");
  VQB_REQUIRE(H > 0 && K > 0 && d > 0, VQB_ERR_INVALID, "vqb_ema_apply_counts: bad shape");
  ema_apply_counts_kernel<<<(unsigned)H, 1024, 0, (cudaStream_t)stream>>>(stats, cluster_size, weight, K, d, totals_out);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_ema_apply_rows(const float* stats, const float* cluster_size, float* embed_avg, float* embeddings,
                                  float weight, double eps, int64_t k_total, int l2norm, int64_t H, int K, int d,
                                  const float* totals, void* stream) {
  VQB_REQUIRE(stats && cluster_size && embed_avg && embeddings && totals, VQB_ERR_INVALID,
              "vqb_ema_apply_rows: null pointer");
  VQB_REQUIRE(H > 0 && K > 0 && d > 0 && k_total >= K, VQB_ERR_INVALID, "vqb_ema_apply_rows: bad shape");
  const int64_t rows = H * (int64_t)K;
  ema_apply_rows_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      stats, cluster_size, embed_avg, embeddings, weight, (float)eps, (float)((double)k_total * eps), l2norm, H, K, d,
      totals);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_ema_apply(const float* stats, float* cluster_size, float* embed_avg, float* embeddings,
                             float weight, double eps, int l2norm, int64_t H, int K, int d, void* ws,
                             size_t ws_bytes, void* stream) {
  VQB_REQUIRE(ws != nullptr && ws_bytes >= (size_t)H * 4, VQB_ERR_WORKSPACE, "ema_apply workspace too small");
  int rc = vqb_ema_apply_counts(stats, cluster_size, weight, H, K, d, (float*)ws, stream);
  if (rc) return rc;
  return vqb_ema_apply_rows(stats, cluster_size, embed_avg, embeddings, weight, eps, K, l2norm, H, K, d,
                            (const float*)ws, stream);
}

extern "C" int vqb_expire_scatter(const void* x, int x_dtype, const int64_t* sample_rows, int64_t m, float threshold,
                                  float reset, int l2norm, float* cluster_size, float* embed_avg, float* embeddings,
                                  int64_t N, int K, int d, void* stream) {
  VQB_REQUIRE(x && cluster_size && embed_avg && embeddings, VQB_ERR_INVALID, "vqb_expire_scatter: null pointer");
  VQB_REQUIRE(m >= 0 && N > 0 && K > 0 && d > 0, VQB_ERR_INVALID, "vqb_expire_scatter: bad shape");
  if (m == 0) return VQB_OK;
  VQB_REQUIRE(sample_rows != nullptr, VQB_ERR_INVALID, "vqb_expire_scatter: sample_rows is null");
  VQB_DISPATCH_DTYPE(x_dtype, T,
    expire_scatter_kernel<T><<<1, 1024, 0, (cudaStream_t)stream>>>((const T*)x, sample_rows, m, threshold, reset,
                                                                  l2norm, cluster_size, embed_avg, embeddings, N, K, d));
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_minkey_pack(const float* score, const int64_t* idx, int64_t n, int64_t* keys, void* stream) {
  VQB_REQUIRE(score && idx && keys && n >= 0, VQB_ERR_INVALID, "vqb_minkey_pack: bad argument");
  if (n == 0) return VQB_OK;
  minkey_pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(score, idx, n, (long long*)keys);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_minkey_unpack(const int64_t* keys, int64_t n, int64_t* idx, float* score, void* stream) {
  VQB_REQUIRE(keys && idx && n >= 0, VQB_ERR_INVALID, "vqb_minkey_unpack: bad argument");
  if (n == 0) return VQB_OK;
  minkey_unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const long long*)keys, n, idx,
                                                                                       score);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_column_moments(const void* x, int x_dtype, const uint8_t* mask, int64_t H, int64_t N, int d,
                                  double* sums_out, int64_t* rows_used_out, void* stream) {
  VQB_REQUIRE(H >= 1 && H <= 65535 && N >= 0 && d >= 1, VQB_ERR_INVALID, "vqb_column_moments: bad shape");
  VQB_REQUIRE(sums_out && rows_used_out && (x || N == 0), VQB_ERR_INVALID, "vqb_column_moments: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  VQB_CUDA_TRY(cudaMemsetAsync(sums_out, 0, (size_t)H * d * 2 * sizeof(double), st));
  VQB_CUDA_TRY(cudaMemsetAsync(rows_used_out, 0, (size_t)H * sizeof(int64_t), st));
  if (N == 0) return VQB_OK;
  const dim3 grid((unsigned)((N + kMomentRows - 1) / kMomentRows), (unsigned)H);
  VQB_DISPATCH_DTYPE(x_dtype, T, (column_moments_kernel<T><<<grid, 256, 0, st>>>(
      (const T*)x, mask, N, d, sums_out, (long long*)rows_used_out)));
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}
