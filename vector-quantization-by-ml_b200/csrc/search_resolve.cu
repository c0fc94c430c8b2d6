// search_resolve.cu -- turns tensor-core candidates into the reference's fp32 argmin, exactly.
//
// Why the candidate set is complete (per row x, metric score e_k = |c_k|^2/2 - x.c_k, or -x.c_k):
//   the tensor-core pass computes a_k = bias_k - x_b.c_bk with bf16 roundings x_b, c_bk, and
//   |e_k - (a_k + E_k)| <= E_k  where  E_k >= |x_b|.|c_k - c_bk| + |x - x_b|.|c_k| + fp32 accumulation slack
//   (Cauchy-Schwarz; |x_b|, |x - x_b| replaced by their maxima over the batch, prepare.cu).
//   The kernel stores L_k = a_k (already lowered by E_k): L_k <= e_k <= L_k + 2 E_k.
//   With j = argmin_k L_k the true argmin k* satisfies L_k* <= e_k* <= e_j <= L_j + 2 E_j, so
//   every possible winner has L <= thr := L_j + 2 E_j (+ slack for the 5 id bits packed into L).
//   The epilogue keeps, per 64-column group (one class of one column quarter of a pair of N tiles), the two
//   smallest L, and per class (8 per row: 4 quarters x 2 classes) the three smallest of those.  Therefore a possible winner is missing only if
//     (i)  the third entry of some class is <= thr (a fourth could exist)  -> full exact rescan, or
//     (ii) two entries <= thr come from the same 64-column group (a third could hide there)
//                                                                          -> rescan those 64 columns.
//   Both are detected here; neither is assumed away.
//   (x_b, c_bk above stand for the scaled-fp16 values x~ = fp16(x s_row)/s_row, c~ = fp16(c s_c)/s_c.)
//
// Two phases: a streaming one-thread-per-row classification (accept / queue / flag), then one warp per queued
// row where lane i evaluates candidate i exactly.
//
// "Exact" score = the reference's recipe (SURVEY A.1) evaluated with fp64 accumulation:
//   euclid: sqrtf(max(float(|x|^2 + |c|^2 - 2 x.c), 0))   dot: float(-x.c); lowest index wins ties.
#include "common.cuh"

namespace vqb {

template <typename T>
__device__ __forceinline__ double row_norm2(const T* __restrict__ xr, int d) {
  double s = 0.0;
  if ((d & 3) == 0) {
#pragma unroll 8
    for (int j = 0; j < d; j += 4) {
      float4 v = load4<T>(xr + j);
      s = fma((double)v.x, (double)v.x, s); s = fma((double)v.y, (double)v.y, s);
      s = fma((double)v.z, (double)v.z, s); s = fma((double)v.w, (double)v.w, s);
    }
  } else {
    for (int j = 0; j < d; ++j) { double v = (double)to_f32<T>(xr[j]); s = fma(v, v, s); }
  }
  return s;
}

// exact score of (row, code); xn2 = |x|^2 in fp64 (ignored for the dot metric)
template <typename T>
__device__ __forceinline__ float exact_score(const T* __restrict__ xr, const float* __restrict__ cr, int d, int metric,
                                             double xn2) {
  double dot = 0.0, cn2 = 0.0;
  if ((d & 3) == 0) {
#pragma unroll 8          // 16 independent loads in flight; the fma chains keep their order (same result)
    for (int j = 0; j < d; j += 4) {
      float4 a = load4<T>(xr + j);
      float4 c = __ldg(reinterpret_cast<const float4*>(cr + j));
      dot = fma((double)a.x, (double)c.x, dot); dot = fma((double)a.y, (double)c.y, dot);
      dot = fma((double)a.z, (double)c.z, dot); dot = fma((double)a.w, (double)c.w, dot);
      cn2 = fma((double)c.x, (double)c.x, cn2); cn2 = fma((double)c.y, (double)c.y, cn2);
      cn2 = fma((double)c.z, (double)c.z, cn2); cn2 = fma((double)c.w, (double)c.w, cn2);
    }
  } else {
    for (int j = 0; j < d; ++j) {
      double a = (double)to_f32<T>(xr[j]), c = (double)cr[j];
      dot = fma(a, c, dot);
      cn2 = fma(c, c, cn2);
    }
  }
  if (metric == VQB_DOT) return (float)(-dot);
  float d2 = (float)(xn2 + cn2 - 2.0 * dot);
  return sqrtf(fmaxf(d2, 0.f));
}

// exact_score(xr, cr, d, metric, row_norm2(xr, d)) in ONE walk over the latent row: three independent fma chains, each in
// the order of the two functions above, so the value is bit-identical (the pair scorer walked every row twice)
template <typename T>
__device__ __forceinline__ float exact_score_norm(const T* __restrict__ xr, const float* __restrict__ cr, int d,
                                                  int metric) {
  double dot = 0.0, cn2 = 0.0, n2 = 0.0;
  if ((d & 3) == 0) {
#pragma unroll 8
    for (int j = 0; j < d; j += 4) {
      float4 a = load4<T>(xr + j);
      float4 c = __ldg(reinterpret_cast<const float4*>(cr + j));
      n2 = fma((double)a.x, (double)a.x, n2); n2 = fma((double)a.y, (double)a.y, n2);
      n2 = fma((double)a.z, (double)a.z, n2); n2 = fma((double)a.w, (double)a.w, n2);
      dot = fma((double)a.x, (double)c.x, dot); dot = fma((double)a.y, (double)c.y, dot);
      dot = fma((double)a.z, (double)c.z, dot); dot = fma((double)a.w, (double)c.w, dot);
      cn2 = fma((double)c.x, (double)c.x, cn2); cn2 = fma((double)c.y, (double)c.y, cn2);
      cn2 = fma((double)c.z, (double)c.z, cn2); cn2 = fma((double)c.w, (double)c.w, cn2);
    }
  } else {
    for (int j = 0; j < d; ++j) {
      double a = (double)to_f32<T>(xr[j]), c = (double)cr[j];
      n2 = fma(a, a, n2);
      dot = fma(a, c, dot);
      cn2 = fma(c, c, cn2);
    }
  }
  if (metric == VQB_DOT) return (float)(-dot);
  float d2 = (float)(n2 + cn2 - 2.0 * dot);
  return sqrtf(fmaxf(d2, 0.f));
}

constexpr float kPackSlack = 6.2e-5f;   // 2 keys x 2^-17 (6 id bits) + fma rounding, with margin

// candidate bookkeeping shared by both resolve phases ------------------------------------------------
struct RowCands {
  float key[kNumCand];
  int code[kNumCand];
  float thr;
  int c1;
  int ncand;
  bool full_rescan;   // hazard (i)
  bool local_rescan;  // hazard (ii) somewhere
};

// emax > 0: the keys are NOT pre-lowered by E_k (no bias k-step, or E_k too large for the fp16 bias operand) and the
// window is the symmetric min + 2 Emax for every code
__device__ __forceinline__ void load_cands(const uint2* __restrict__ cand, int64_t gid, int K, int Kp, int64_t h,
                                           const float* __restrict__ err, float emax, float tie_win, RowCands& R) {
  const uint4* c4 = reinterpret_cast<const uint4*>(cand + gid * kNumCand);
#pragma unroll
  for (int i = 0; i < kNumCand / 2; ++i) {
    const uint4 v = __ldg(c4 + i);
    R.key[2 * i] = __uint_as_float(v.x); R.code[2 * i] = (int)v.y;
    R.key[2 * i + 1] = __uint_as_float(v.z); R.code[2 * i + 1] = (int)v.w;
  }
  float m1 = __int_as_float(0x7f800000);
  int c1 = -1;
#pragma unroll
  for (int i = 0; i < kNumCand; ++i) {
    const bool valid = R.code[i] >= 0 && R.code[i] < K;
    if (!valid) R.key[i] = __int_as_float(0x7f800000);
    if (valid && R.key[i] < m1) { m1 = R.key[i]; c1 = R.code[i]; }
  }
  const float E1 = emax > 0.f ? emax : (c1 >= 0 ? err[h * Kp + c1] : 0.f);
  // 2 E_j, plus the 6 packed id bits (<= 2^-17 relative per key) and the bias fma rounding
  // + the codes that the reference's fp32 rounding of the distance can make EQUAL to the winner (kTieSlack, common.cuh)
  R.thr = m1 + 2.f * E1 + (fabsf(m1) + E1) * kPackSlack + tie_win;
  R.c1 = c1;
  R.ncand = 0;
  R.full_rescan = c1 < 0;
  R.local_rescan = false;
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    const float k0 = R.key[3 * g], k1 = R.key[3 * g + 1], k2 = R.key[3 * g + 2];
    if (k0 <= R.thr) ++R.ncand;
    if (k1 <= R.thr) {
      ++R.ncand;
      if ((R.code[3 * g] >> 9) == (R.code[3 * g + 1] >> 9)) R.local_rescan = true;   // (ii)
    }
    if (k2 <= R.thr) { ++R.ncand; R.full_rescan = true; }                            // (i)
  }
}

// phase 1, one thread per row, pure streaming: accept the unique candidate, or queue the row for the
// warp-per-row re-rank (phase 2), or flag it for the exact rescan
// SCORE (the caller wants the exact score of every row: sharded codebooks merge (score, index) keys across GPUs): a row
// with a single candidate evaluates that one exact score right here -- same functions, same fma order as the pair
// scorer -- instead of going through the queue: with every row queued the one-atomic-per-row append of
// rerank_emit_kernel alone cost 5 ms for the 4M rows of config 5.
template <typename T, bool SCORE>
__global__ void __launch_bounds__(256)
resolve_classify_kernel(const uint2* __restrict__ cand, const float* __restrict__ err, int64_t H, int64_t N, int K,
                        int Kp, int64_t idx_offset, int64_t* __restrict__ idx_out,
                        int* __restrict__ rr_list, int* __restrict__ flag_list, uint32_t* __restrict__ flag_cnt,
                        unsigned long long* __restrict__ keys, uint32_t* __restrict__ scal,
                        const float* __restrict__ xinv, const float* __restrict__ chdr, int aug,
                        const float* __restrict__ xn2, float tie, const T* __restrict__ x,
                        const float* __restrict__ cb, int d, int metric, float* __restrict__ score_out) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool queue = false;
  int64_t direct_code = -1;                   // SCORE: flat index (h K + code) of the accepted single candidate
  if (gid < H * N) {
    const int64_t h = gid / N;
    RowCands R;
    load_cands(cand, gid, K, Kp, h, err, (aug == 2 || scal[8]) ? __uint_as_float(scal[6]) : 0.f, tie * xn2[gid], R);
    // no fp16 bias operand for this row (prepare.cu), or operands prepared by vqb_rvq_level against a cache that
    // has been rebuilt with another 2^q since (scal[7] records the one used): rescan exactly
    if (aug && (xinv[gid] < 0.f || (scal[7] != 0u && scal[7] != __float_as_uint(chdr[h * kHdrFloats + 4]))))
      R.full_rescan = true;
    if (R.full_rescan) {
      const uint32_t pos = atomicAdd(flag_cnt + h, 1u);
      flag_list[h * N + pos] = (int)(gid - h * N);
      keys[gid] = ~0ull;                      // min-key accumulator of the K-split rescan
    } else if (R.ncand == 1 && !R.local_rescan) {
      idx_out[gid] = (int64_t)R.c1 + idx_offset;
      if (SCORE) direct_code = (h * K + (int64_t)R.c1);
    } else {
      queue = true;
      keys[gid] = ~0ull;                      // min-key accumulator of the pair scoring
    }
  }
  if (SCORE) {
    // Exact score of the accepted candidate, same fma chains in the same order as exact_score() / row_norm2() (the
    // sharded merge compares scores across GPUs and across resolve paths).  A thread walking its own 4d-byte row
    // touches 32 different lines per warp-load; the block's rows are staged through shared memory instead, 32
    // dimensions at a time with fully coalesced loads (stride 33: conflict-free reads), and only the code row --
    // a gather in any case, served by L2 -- is read directly.
    __shared__ float xs[256][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row0 = (int64_t)blockIdx.x * blockDim.x;
    const int64_t total = H * N;
    const float* cr = direct_code >= 0 ? cb + direct_code * (int64_t)d : cb;
    double dot = 0.0, cn2 = 0.0, n2 = 0.0;
    for (int d0 = 0; d0 < d; d0 += 32) {
      __syncthreads();
#pragma unroll 8
      for (int r = 0; r < 32; ++r) {
        const int64_t row = row0 + warp * 32 + r;
        xs[warp * 32 + r][lane] = (row < total && d0 + lane < d) ? to_f32<T>(x[row * (int64_t)d + d0 + lane]) : 0.f;
      }
      __syncthreads();
      if (direct_code >= 0) {
        const int lim = d - d0 < 32 ? d - d0 : 32;
        if ((d & 3) == 0) {              // code row as float4: a warp-load of 32 different rows costs 32 L1 wavefronts
#pragma unroll 2
          for (int c = 0; c < lim; c += 4) {
            const float4 c4 = __ldg(reinterpret_cast<const float4*>(cr + d0 + c));
            const float cvs[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const double a = (double)xs[threadIdx.x][c + t], cv = (double)cvs[t];
              n2 = fma(a, a, n2);
              dot = fma(a, cv, dot);
              cn2 = fma(cv, cv, cn2);
            }
          }
        } else {
          for (int c = 0; c < lim; ++c) {
            const double a = (double)xs[threadIdx.x][c], cv = (double)__ldg(cr + d0 + c);
            n2 = fma(a, a, n2);
            dot = fma(a, cv, dot);
            cn2 = fma(cv, cv, cn2);
          }
        }
      }
    }
    if (direct_code >= 0)
      score_out[gid] = metric == VQB_DOT ? (float)(-dot) : sqrtf(fmaxf((float)(n2 + cn2 - 2.0 * dot), 0.f));
  }
  // warp-aggregated append to the re-rank list (scal[3] is its length)
  const uint32_t m = __ballot_sync(0xffffffffu, queue);
  if (m) {
    const int lane = threadIdx.x & 31;
    uint32_t base = 0;
    if (lane == __ffs(m) - 1) base = atomicAdd(scal + 3, (uint32_t)__popc(m));
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (queue) rr_list[base + __popc(m & ((1u << lane) - 1u))] = (int)gid;
  }
}

// phase 2 works on (row, code) PAIRS so that every lane of the scoring kernel is busy: a queued row has 24 candidate
// slots but typically only 2-3 of them inside the window, and a warp-per-row kernel spends its issue slots (the
// fp32 -> fp64 conversions run at 16 lanes/clk/SM) on 2-3 active lanes.
//   2a  one warp per queued row: window from the 24 candidates, emit one pair per candidate inside it and, for
//       hazard (ii), the 64 columns of the group; a row that does not fit the pair list goes to the exact rescan
//   2b  one THREAD per pair: exact score (same fma order as everywhere else), 64-bit atomicMin of (orderable score,
//       index) into the row's key -- the lowest index wins ties, like torch.argmax
//   2c  one thread per queued row: unpack the key
__device__ __forceinline__ unsigned long long pack_key(float score, int idx);
__device__ __forceinline__ float unpack_score(unsigned long long key);

__global__ void __launch_bounds__(256)
rerank_emit_kernel(const uint2* __restrict__ cand, const float* __restrict__ err, int64_t N, int K, int Kp,
                   const int* __restrict__ rr_list, uint32_t* __restrict__ scal, int aug, uint2* __restrict__ pairs,
                   uint32_t pair_cap, int* __restrict__ flag_list, uint32_t* __restrict__ flag_cnt,
                   const float* __restrict__ xn2, float tie) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t count = scal[3];
  // the pair slots of the 8 rows a block handles per iteration are reserved with ONE atomic (a row at a time, 250 k
  // queued rows of a d = 64 search serialised on that one counter for 0.24 ms)
  __shared__ uint32_t s_n[8], s_base;
  for (int64_t it0 = (int64_t)blockIdx.x * (blockDim.x >> 5); it0 < count; it0 += nwarps) {   // block-uniform trip count
    const int64_t it = it0 + warp;
    const bool have = it < count;
    const int64_t gid = rr_list[have ? it : it0];
    const int64_t h = gid / N;
    float key = __int_as_float(0x7f800000);
    int code = -1;
    if (lane < kNumCand) {
      const uint2 v = __ldg(cand + gid * kNumCand + lane);
      code = (int)v.y;
      if (code >= 0 && code < K) key = __uint_as_float(v.x); else code = -1;
    }
    float m1 = key;
    int c1 = code;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float om = __shfl_xor_sync(0xffffffffu, m1, o);
      const int oc = __shfl_xor_sync(0xffffffffu, c1, o);
      if (om < m1 || (om == m1 && oc > c1)) { m1 = om; c1 = oc; }   // any consistent tie rule: only E(c1) is used
    }
    const float E1 = (aug == 2 || scal[8]) ? __uint_as_float(scal[6]) : (c1 >= 0 ? err[h * Kp + c1] : 0.f);
    const float thr = m1 + 2.f * E1 + (fabsf(m1) + E1) * kPackSlack + tie * xn2[gid];
    const bool act = code >= 0 && key <= thr;
    // hazard (ii): entries 3g and 3g+1 both within thr and from the same pair of N tiles -> that 64-column group
    const float key_next = __shfl_down_sync(0xffffffffu, key, 1);
    const int code_next = __shfl_down_sync(0xffffffffu, code, 1);
    const bool req = lane < kNumCand && (lane % 3) == 0 && key <= thr && key_next <= thr && code >= 0 &&
                     code_next >= 0 && (code >> 9) == (code_next >> 9);
    const uint32_t acts = __ballot_sync(0xffffffffu, act);
    uint32_t reqs = __ballot_sync(0xffffffffu, req);
    const uint32_t n = have ? (uint32_t)__popc(acts) + 64u * (uint32_t)__popc(reqs) : 0u;
    if (lane == 0) s_n[warp] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t t = 0;
      for (int w2 = 0; w2 < (int)(blockDim.x >> 5); ++w2) t += s_n[w2];
      s_base = t ? atomicAdd(scal + 9, t) : 0u;
    }
    __syncthreads();
    uint32_t base = s_base;
    for (int w2 = 0; w2 < warp; ++w2) base += s_n[w2];
    __syncthreads();                    // s_n / s_base are rewritten in the next iteration
    if (!have) continue;
    if (base + n > pair_cap) {          // no room: the exact rescan takes the row (its key is already ~0)
      if (lane == 0) flag_list[h * N + atomicAdd(flag_cnt + h, 1u)] = (int)(gid - h * N);
      for (uint32_t i = base + lane; i < base + n && i < pair_cap; i += 32)   // void the reserved slots
        pairs[i] = make_uint2((uint32_t)gid, 0xffffffffu);
      continue;
    }
    if (act) pairs[base + __popc(acts & ((1u << lane) - 1u))] = make_uint2((uint32_t)gid, (uint32_t)code);
    uint32_t off = base + (uint32_t)__popc(acts);
    while (reqs) {
      const int src = __ffs(reqs) - 1;
      reqs &= reqs - 1;
      const int c0 = __shfl_sync(0xffffffffu, code, src);
      const int g = src / 3;                                     // group = quarter*2 + class
#pragma unroll
      for (int t = 0; t < 2; ++t) {                              // the group spans a pair of N tiles: 64 columns
        const int k = ((c0 >> 9) * 2 + t) * kBlockN + (g >> 1) * 64 + (g & 1) + 2 * lane;
        // columns beyond K cannot win: repeat the requesting candidate instead (harmless duplicate)
        pairs[off + t * 32 + lane] = make_uint2((uint32_t)gid, (uint32_t)(k < K ? k : c0));
      }
      off += 64;
    }
  }
}

// A handful of flagged rows are cheaper as (row, code) pairs over ALL codes than as a tiled rescan (whose latency
// is ~60 us however few rows there are).  Per codebook: if its flagged rows x K fit the budget and the pair list,
// reserve the pairs (plan[h] = first slot) and leave nothing for the tiled rescan (scan_cnt[h] = 0).
constexpr uint32_t kFlagPairBudget = 1u << 17;
__global__ void flag_plan_kernel(const uint32_t* __restrict__ flag_cnt, int H, int K, uint32_t pair_cap,
                                 uint32_t* __restrict__ scal, uint32_t* __restrict__ scan_cnt,
                                 uint32_t* __restrict__ plan) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  const uint32_t n = flag_cnt[h];
  scan_cnt[h] = n;
  plan[h] = 0xffffffffu;
  if (n == 0 || (uint64_t)n * (uint64_t)K > kFlagPairBudget) return;
  const uint32_t need = n * (uint32_t)K;
  const uint32_t base = atomicAdd(scal + 9, need);
  if ((uint64_t)base + need > pair_cap) return;     // (the over-reservation is clamped away by pair_score_kernel)
  plan[h] = base;
  scan_cnt[h] = 0;
  atomicAdd(scal + 2, n);                           // statistics: rows resolved by a scan of every code
}
__global__ void __launch_bounds__(256)
flag_emit_kernel(const int* __restrict__ flag_list, const uint32_t* __restrict__ flag_cnt,
                 const uint32_t* __restrict__ plan, int64_t N, int K, uint2* __restrict__ pairs) {
  const int h = blockIdx.y;
  const uint32_t base = plan[h];
  if (base == 0xffffffffu) return;
  const uint64_t total = (uint64_t)flag_cnt[h] * (uint64_t)K;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t p = (uint32_t)(i / (uint32_t)K), k = (uint32_t)(i - (uint64_t)p * (uint32_t)K);
    pairs[base + i] = make_uint2((uint32_t)((int64_t)h * N + flag_list[(int64_t)h * N + p]), k);
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
pair_score_kernel(const T* __restrict__ x, const float* __restrict__ cb, const uint2* __restrict__ pairs,
                  const uint32_t* __restrict__ scal, uint32_t pair_cap, int64_t total_rows, int64_t N, int K, int d,
                  int metric, unsigned long long* __restrict__ keys) {
  uint32_t count = scal[9];
  if (count > pair_cap) count = pair_cap;      // over-reserved by rows that were diverted to the rescan
  for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < count; p += gridDim.x * blockDim.x) {
    const uint2 pr = pairs[p];
    const int64_t gid = pr.x;
    // voided slot (row diverted to the rescan), or a slot of a reservation that did not fit and was never written:
    // whatever in-range (row, code) such a slot holds is a true score of a real code -- harmless for the minimum
    if (pr.y >= (uint32_t)K || gid >= total_rows) continue;
    const int64_t h = gid / N;
    const T* xr = x + gid * (int64_t)d;
    const float s = exact_score_norm<T>(xr, cb + (h * K + (int64_t)pr.y) * d, d, metric);
    atomicMin(keys + gid, pack_key(s, (int)pr.y));
  }
}

__global__ void rerank_finalize_kernel(const int* __restrict__ rr_list, const uint32_t* __restrict__ scal,
                                       const unsigned long long* __restrict__ keys, int64_t idx_offset,
                                       int64_t* __restrict__ idx_out, float* __restrict__ score_out) {
  const int64_t count = scal[3];
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < count; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t gid = rr_list[p];
    const unsigned long long key = keys[gid];
    if (key == ~0ull) continue;                // diverted to the rescan: rescan_finalize writes it
    idx_out[gid] = (int64_t)(uint32_t)(key & 0xffffffffull) + idx_offset;
    if (score_out) score_out[gid] = unpack_score(key);
  }
}

// ------------------------------------------------------------------------------------------
// exact scan of every code for a list of rows (flagged rows, or all rows with FORCE_EXACT / d_pad > 512).
// Tile: 32 rows x 64 codes per 256-thread block, fp64 accumulators, same fma order as exact_score.
// ------------------------------------------------------------------------------------------
constexpr int kER = 32, kEC = 64, kEK = 32;

__device__ __forceinline__ unsigned long long pack_key(float score, int idx) {
  uint32_t u = __float_as_uint(score);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);      // float order -> unsigned order
  return ((unsigned long long)u << 32) | (unsigned long long)(uint32_t)idx;
}
__device__ __forceinline__ float unpack_score(unsigned long long key) {
  uint32_t u = (uint32_t)(key >> 32);
  u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  return __uint_as_float(u);
}

// kSplit: blockIdx.z owns the code range [z*ksplit_codes, (z+1)*ksplit_codes) and the per-row result is merged
// with a 64-bit atomicMin on (orderable score, index) keys -- the lowest index wins ties, like torch.argmax.
template <typename T, bool kSplit>
__global__ void __launch_bounds__(256)
exact_scan_kernel(const T* __restrict__ x, const float* __restrict__ cb, const int* __restrict__ flag_list,
                  const uint32_t* __restrict__ flag_cnt, int64_t N, int K, int d, int metric, int64_t idx_offset,
                  int64_t* __restrict__ idx_out, float* __restrict__ score_out, uint32_t* __restrict__ scal,
                  int ksplit_codes, unsigned long long* __restrict__ keys) {
  __shared__ float xs[kER][kEK + 1];
  __shared__ float cs[kEC][kEK + 1];
  __shared__ int rows_s[kER];
  const int h = blockIdx.y;
  const int64_t count = flag_list ? (int64_t)flag_cnt[h] : N;
  const int* list = flag_list ? flag_list + (int64_t)h * N : nullptr;
  const T* xh = x + (int64_t)h * N * d;
  const float* cbh = cb + (int64_t)h * K * d;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;   // codes tx+16j (j<4), rows ty+16i (i<2)
  if (flag_list && blockIdx.x == 0 && blockIdx.z == 0 && threadIdx.x == 0 && count) atomicAdd(scal + 2, (uint32_t)count);
  const int kbeg = kSplit ? (int)blockIdx.z * ksplit_codes : 0;
  const int kend = kSplit ? (kbeg + ksplit_codes < K ? kbeg + ksplit_codes : K) : K;
  if (kbeg >= kend) return;

  for (int64_t t0 = (int64_t)blockIdx.x * kER; t0 < count; t0 += (int64_t)gridDim.x * kER) {
    __syncthreads();
    if (threadIdx.x < kER) {
      const int64_t r = t0 + threadIdx.x;
      rows_s[threadIdx.x] = r < count ? (list ? list[r] : (int)r) : -1;
    }
    __syncthreads();
    float best[2] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000)};
    int bidx[2] = {0x7fffffff, 0x7fffffff};
    // |x|^2 of this thread's two rows, fp64, same order as row_norm2 (recomputed per code tile: cheap)
    for (int k0 = kbeg; k0 < kend; k0 += kEC) {
      double acc[2][4], xn[2] = {0.0, 0.0}, cn[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
      for (int d0 = 0; d0 < d; d0 += kEK) {
        __syncthreads();
        for (int e = threadIdx.x; e < kER * kEK; e += 256) {
          const int r = e / kEK, c = e % kEK;
          const int rr = rows_s[r];
          xs[r][c] = (rr >= 0 && d0 + c < d) ? to_f32<T>(xh[(int64_t)rr * d + d0 + c]) : 0.f;
        }
        for (int e = threadIdx.x; e < kEC * kEK; e += 256) {
          const int r = e / kEK, c = e % kEK;
          cs[r][c] = (k0 + r < kend && d0 + c < d) ? cbh[(int64_t)(k0 + r) * d + d0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int c = 0; c < kEK; ++c) {
          double xv[2], cv[4];
#pragma unroll
          for (int i = 0; i < 2; ++i) { xv[i] = (double)xs[ty + 16 * i][c]; xn[i] = fma(xv[i], xv[i], xn[i]); }
#pragma unroll
          for (int j = 0; j < 4; ++j) { cv[j] = (double)cs[tx + 16 * j][c]; cn[j] = fma(cv[j], cv[j], cn[j]); }
#pragma unroll
          for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = fma(xv[i], cv[j], acc[i][j]);
        }
      }
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = k0 + tx + 16 * j;
          if (k < kend) {
            float s;
            if (metric == VQB_DOT) s = (float)(-acc[i][j]);
            else s = sqrtf(fmaxf((float)(xn[i] + cn[j] - 2.0 * acc[i][j]), 0.f));
            if (s < best[i] || (s == best[i] && k < bidx[i])) { best[i] = s; bidx[i] = k; }
          }
        }
    }
    // reduce over the 16 threads (tx) that share a row: lanes of one half-warp
#pragma unroll
    for (int i = 0; i < 2; ++i) {
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best[i], o);
        const int oi = __shfl_xor_sync(0xffffffffu, bidx[i], o);
        if (ob < best[i] || (ob == best[i] && oi < bidx[i])) { best[i] = ob; bidx[i] = oi; }
      }
      const int rr = rows_s[ty + 16 * i];
      if (tx == 0 && rr >= 0) {
        if (kSplit) {
          atomicMin(keys + (int64_t)h * N + rr, pack_key(best[i], bidx[i]));
        } else {
          idx_out[(int64_t)h * N + rr] = (int64_t)bidx[i] + idx_offset;
          if (score_out) score_out[(int64_t)h * N + rr] = best[i];
        }
      }
    }
  }
}

// unpack the merged keys of the rescanned rows
__global__ void rescan_finalize_kernel(const int* __restrict__ flag_list, const uint32_t* __restrict__ flag_cnt,
                                       const unsigned long long* __restrict__ keys, int64_t N, int64_t idx_offset,
                                       int64_t* __restrict__ idx_out, float* __restrict__ score_out) {
  const int h = blockIdx.y;
  const int64_t count = flag_cnt[h];
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < count; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = (int64_t)h * N + flag_list[(int64_t)h * N + p];
    const unsigned long long key = keys[g];
    idx_out[g] = (int64_t)(uint32_t)(key & 0xffffffffull) + idx_offset;
    if (score_out) score_out[g] = unpack_score(key);
  }
}

// In-kernel conversion: scal[0] bounds only the rows within the sampled bound; the search kernel gave the others a
// negative xinv (they are rescanned exactly).  Their norm bound xn2 (>= |x|^2) goes into scal[1], which nothing reads on
// this route once make_bias has run, so that scal[0] + scal[1] >= max|x_j| over the batch, as the EMA kernels read it
// (vqb.h, vqb_ema_reduce).
__global__ void __launch_bounds__(256)
conv_outlier_bound_kernel(const float* __restrict__ xinv, const float* __restrict__ xn2, int64_t rows,
                          uint32_t* __restrict__ scal) {
  float m = 0.f;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x)
    if (xinv[r] < 0.f) m = fmaxf(m, sqrtf(xn2[r]));
  m = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(m)));   // non-negative: bit order = float order
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(scal + 1, __float_as_uint(m));
}

static int g_num_sms = 0;
static int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

}  // namespace vqb

using namespace vqb;

extern "C" size_t vqb_search_workspace_bytes(int64_t H, int64_t N, int K, int d) {
  if (H <= 0 || N < 0 || K <= 0 || d <= 0) return 0;
  return search_layout(H, N, K, d).total;
}

extern "C" int vqb_search(const void* x, int x_dtype, const float* codebook, const void* cache, int metric,
                          int64_t H, int64_t N, int K, int d, int64_t idx_offset, int64_t* idx_out,
                          float* score_out, int flags, void* ws, size_t ws_bytes, void* stream) {
  VQB_REQUIRE(x && codebook && idx_out && ws, VQB_ERR_INVALID, "vqb_search: null pointer");
  VQB_REQUIRE(H > 0 && N >= 0 && K > 0 && d > 0, VQB_ERR_INVALID, "vqb_search: bad shape H=%lld N=%lld K=%d d=%d",
              (long long)H, (long long)N, K, d);
  VQB_REQUIRE(metric == VQB_EUCLID || metric == VQB_DOT, VQB_ERR_INVALID, "unknown metric %d", metric);
  VQB_REQUIRE(H * N < (1ll << 31), VQB_ERR_UNSUPPORTED, "H*N must be < 2^31");
  VQB_REQUIRE(H < 65536, VQB_ERR_UNSUPPORTED, "too many codebooks");
  SearchLayout SL = search_layout(H, N, K, d);
  VQB_REQUIRE(ws_bytes >= SL.total, VQB_ERR_WORKSPACE, "search workspace too small: %zu < %zu", ws_bytes, SL.total);
  if (N == 0) return VQB_OK;
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)ws;
  uint32_t* scal = (uint32_t*)(w + SL.off_scal);
  uint32_t* cnt = (uint32_t*)(w + SL.off_cnt);          // [H] flagged rows | [H] of them left to the tiled rescan | [H] plan
  uint32_t* scan_cnt = cnt + H;
  uint32_t* plan = cnt + 2 * H;
  int* flag_list = (int*)(w + SL.off_flag);
  const bool prepared = (flags & VQB_SEARCH_LATENTS_PREPARED) != 0;
  const bool tc = !(flags & VQB_SEARCH_FORCE_EXACT) && SL.dp <= 512 && cache != nullptr;
  // scal[0..1] hold the row statistics: keep them when the caller prepared the latents
  if (prepared) {   // keep [0..1] (row statistics) and [7] (2^q of the prepared bias operands)
    VQB_CUDA_TRY(cudaMemsetAsync((char*)scal + 8, 0, 20, st));
    VQB_CUDA_TRY(cudaMemsetAsync((char*)scal + 32, 0, (SL.off_cnt - SL.off_scal) + (size_t)H * 12 - 32, st));
  } else {
    VQB_CUDA_TRY(cudaMemsetAsync((char*)scal, 0, (SL.off_cnt - SL.off_scal) + (size_t)H * 12, st));
  }

  const int grid_scan = (int)((N + kER - 1) / kER < 4 * (int64_t)num_sms() ? (N + kER - 1) / kER : 4 * num_sms());
  if (!tc) {
    // nothing on this route writes the row statistics: scal[0] = max|x_j| for the EMA kernels (vqb.h, vqb_ema_reduce)
    if (int rc = launch_absmax(x, x_dtype, H * N * (int64_t)d, scal, st)) return rc;
    VQB_DISPATCH_DTYPE(x_dtype, T,
      exact_scan_kernel<T, false><<<dim3((unsigned)grid_scan, (unsigned)H), 256, 0, st>>>(
          (const T*)x, codebook, nullptr, nullptr, N, K, d, metric, idx_offset, idx_out, score_out, scal, 0, nullptr));
    VQB_LAUNCH_CHECK();
    return VQB_OK;
  }

  CacheLayout CL = cache_layout(H, K, d);
  const char* cbase = (const char*)cache;
  __half* xb = (__half*)(w + SL.off_xb);
  float* xinv = (float*)(w + SL.off_xinv);
  float* xn2 = (float*)(w + SL.off_xn2);
  const float tie = metric == VQB_EUCLID ? kTieSlack : 0.f;
  unsigned long long* keys = (unsigned long long*)(w + SL.off_keys);
  float* bias = (float*)(w + SL.off_bias);
  float* err = (float*)(w + SL.off_err);
  int rc;
  __half* xaug = (__half*)(w + SL.off_xaug);
  const float* chdr = (const float*)(cbase + CL.off_hdr);
  const int aug = search_tc_aug_mode(N, K, metric);
  // 16-bit latents and enough tensor work per row tile: the search kernel converts the rows itself, overlapped with
  // its MMAs (search_tc.cu, CONV); all that runs ahead of it is a strided sample that bounds the row norms
  ConvArgs conv;
  const int conv_mode = prepared ? 0 : search_tc_conv_ok(N, K, d, x_dtype, aug, (flags & VQB_SEARCH_FUSED_PREP) != 0);
  if (conv_mode == 2) {
    rc = launch_prepare_latents(x, x_dtype, H * N, N, d, SL.dp, chdr, xb, xinv, xn2, xaug, scal, st);
    if (rc) return rc;
    conv.x = x; conv.x_dtype = -1; conv.d = d;
  } else if (conv_mode == 1) {
    conv.x = x; conv.x_dtype = x_dtype; conv.d = d;
    rc = launch_sample_bound(x, x_dtype, H * N, d, scal, st);
    if (rc) return rc;
  } else if (!prepared) {
    rc = launch_prepare_latents(x, x_dtype, H * N, N, d, SL.dp, chdr, xb, xinv, xn2, xaug, scal, st);
    if (rc) return rc;
  }
  __half* caug = (__half*)(w + SL.off_caug);
  rc = launch_make_bias(cache, CL, H, K, metric, scal, bias, err, aug == 1 ? caug : nullptr, st, conv_mode == 1 ? SL.dp : 0);
  if (rc) return rc;
  rc = launch_search_tc(xb, xinv, xn2, tie, xaug, (const __half*)(cbase + CL.off_cb), caug, chdr,
                        bias, aug, H, N, K, SL.dp, w + SL.off_cand, scal, (flags & VQB_SEARCH_TIMING) != 0, st, conv);
  if (rc) return rc;
  const int64_t total = H * N;
  if (conv_mode == 1) {
    const int64_t want = (total + 255) / 256, cap = 4 * (int64_t)num_sms();
    conv_outlier_bound_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(xinv, xn2, total, scal);
    VQB_LAUNCH_CHECK();
  }
  int* rr_list = (int*)(w + SL.off_rr);
  if (score_out) {
    VQB_DISPATCH_DTYPE(x_dtype, T,
      (resolve_classify_kernel<T, true><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
          (const uint2*)(w + SL.off_cand), err, H, N, K, CL.Kp, idx_offset, idx_out, rr_list, flag_list, cnt, keys, scal,
          xinv, chdr, aug, xn2, tie, (const T*)x, codebook, d, metric, score_out)));
  } else {
    resolve_classify_kernel<float, false><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
        (const uint2*)(w + SL.off_cand), err, H, N, K, CL.Kp, idx_offset, idx_out, rr_list, flag_list, cnt, keys, scal,
        xinv, chdr, aug, xn2, tie, nullptr, codebook, d, metric, nullptr);
  }
  VQB_LAUNCH_CHECK();
  {
    uint2* pairs = (uint2*)(w + SL.off_pairs);
    const uint32_t pair_cap = (uint32_t)(SL.pair_cap < 0xffffff00ull ? SL.pair_cap : 0xffffff00ull);
    int64_t want = (total / 16 + 7) / 8 + 1;   // blocks of 8 warps
    const int64_t cap = (int64_t)num_sms() * 8;
    const int grid_rr = (int)(want < cap ? want : cap);
    rerank_emit_kernel<<<grid_rr, 256, 0, st>>>((const uint2*)(w + SL.off_cand), err, N, K, CL.Kp, rr_list, scal, aug,
                                                pairs, pair_cap, flag_list, cnt, xn2, tie);
    VQB_LAUNCH_CHECK();
    flag_plan_kernel<<<(unsigned)((H + 63) / 64), 64, 0, st>>>(cnt, (int)H, K, pair_cap, scal, scan_cnt, plan);
    VQB_LAUNCH_CHECK();
    flag_emit_kernel<<<dim3(64, (unsigned)H), 256, 0, st>>>(flag_list, cnt, plan, N, K, pairs);
    VQB_LAUNCH_CHECK();
    int64_t wantp = (total / 8 + 255) / 256 + 1;
    const int grid_ps = (int)(wantp < cap ? wantp : cap);
    VQB_DISPATCH_DTYPE(x_dtype, T,
      pair_score_kernel<T><<<grid_ps, 256, 0, st>>>((const T*)x, codebook, pairs, scal, pair_cap, total, N, K, d, metric,
                                                    keys));
    VQB_LAUNCH_CHECK();
    rerank_finalize_kernel<<<grid_rr, 256, 0, st>>>(rr_list, scal, keys, idx_offset, idx_out, score_out);
    VQB_LAUNCH_CHECK();
  }
  // flagged rows (count is device-side): fixed grid, code range split over blockIdx.z so that even a handful of
  // rows spreads over the whole chip; blocks exit at once when there is nothing to do
  const int ksplit_codes = K <= 16384 ? 64 : (K <= 65536 ? 128 : 64 * ((K + 64 * 4096 - 1) / (64 * 4096)));
  const int nsplit = (K + ksplit_codes - 1) / ksplit_codes;
  int grid_rows = (2 * num_sms() + nsplit - 1) / nsplit;
  if (grid_rows > grid_scan) grid_rows = grid_scan;
  if (grid_rows < 1) grid_rows = 1;
  VQB_REQUIRE(nsplit <= 65535, VQB_ERR_UNSUPPORTED, "codebook too large for the rescan grid");
  VQB_DISPATCH_DTYPE(x_dtype, T,
    exact_scan_kernel<T, true><<<dim3((unsigned)grid_rows, (unsigned)H, (unsigned)nsplit), 256, 0, st>>>(
        (const T*)x, codebook, flag_list, scan_cnt, N, K, d, metric, idx_offset, idx_out, score_out, scal, ksplit_codes,
        keys));
  VQB_LAUNCH_CHECK();
  rescan_finalize_kernel<<<dim3(8, (unsigned)H), 256, 0, st>>>(flag_list, cnt, keys, N, idx_offset, idx_out, score_out);
  VQB_LAUNCH_CHECK();
  return VQB_OK;
}

extern "C" int vqb_search_stats(const void* ws, int64_t* host_out3, void* stream) {
  VQB_REQUIRE(ws && host_out3, VQB_ERR_INVALID, "vqb_search_stats: null pointer");
  uint32_t hbuf[8];
  VQB_CUDA_TRY(cudaMemcpyAsync(hbuf, ws, sizeof(hbuf), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  VQB_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  host_out3[0] = hbuf[3];
  host_out3[1] = hbuf[2];
  host_out3[2] = hbuf[4];
  if (hbuf[5]) { set_error("search_tc: dynamic shared memory base was not 1024B aligned"); return VQB_ERR_CUDA; }
  return VQB_OK;
}
