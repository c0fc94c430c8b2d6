// search_tc.cu -- fused nearest-code search on the 5th-gen tensor cores (sm_100a).
//
// Replaces reference codebooks.py:386 (-cdist / einsum: an N x K fp32 matrix in HBM) and
// utils/general.py:128-129 (argmax + one_hot) with ONE persistent kernel:
//
//   TMA (cp.async.bulk.tensor, 128B swizzle)  ->  smem ring      (one lane of the TMA warp)
//   tcgen05.mma kind::f16, fp16 x fp16 -> fp32 in TMEM            (one lane of the MMA warp)
//   tcgen05.ld + bias + packed running top-2 per row              (16 epilogue warps)
//
// Per CTA: a 128-row tile of latents stays resident in smem (A operand, d/64 slabs of 16 KB);
// the whole codebook streams through a ring of 32 KB stages (B operand, 256 codes x 64 dims).
// Accumulators are double buffered in TMEM (2 x 256 columns) so the epilogue of N-tile i
// overlaps the MMAs of N-tile i+1.  The N x K score matrix never leaves the SM.
// search_tc_kernel (bias added in the epilogue) serves problems with one row tile per codebook; every other search
// runs search_aug_kernel (CTA pairs, bias as an extra MMA k-step), below.
//
// Operands are fp16 with exact power-of-two scales (per latent row, per codebook) that the epilogue
// undoes with the same FFMA that adds the bias.
// The scores are lower bounds  L_k = |c_k|^2/2 - E_k - x~.c~_k  (bias precomputed per search,
// prepare.cu); each row keeps, for 8 disjoint column groups (4 column quarters x 2 classes), the three smallest L
// (low 6 mantissa bits carry the column id inside a 64-column group = one class of one quarter of a PAIR of N tiles).  search_resolve.cu turns these 16 candidates into
// the exact fp32 argmin or proves that it cannot and flags the row for an exact rescan.
// (tile-local top-2 per 32-column group feeds a running top-3 per class: see search_resolve.cu)
#include <cuda.h>

#include "common.cuh"

namespace vqb {

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a protocol bug must trap (kernel error), never hang the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  for (uint32_t it = 0; it < (1u << 26); ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return;
  }
  printf("vqb search_tc: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", (int)blockIdx.x,
         (int)threadIdx.x, bar, parity);
  __trap();
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// true in exactly one lane of a fully active warp; unlike `lane == 0` the compiler knows the enclosing code stays
// warp-uniform, so the tensor-core / TMA issue instructions (uniform datapath) are not wrapped in election loops
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
      "elect.sync rx|px, %1;\n\t"
      "@px mov.s32 %0, 1;\n\t}"
      : "+r"(pred) : "r"(0xFFFFFFFFu));
  return pred != 0;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

constexpr uint64_t kEvictFirst = 0x12F0000000000000ull;
constexpr uint64_t kEvictLast = 0x14F0000000000000ull;

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2,
                                            uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(hint) : "memory");
}

// ---- 2-CTA ("pair") forms: one tcgen05.mma.cta_group::2 covers 256 rows (128 per CTA) x 256 codes (each CTA holds
// 128 of them in ITS shared memory), issued by the leader CTA only.  Shared-window addresses of the odd CTA carry
// bit 24; clearing it addresses the same offset in the even (leader) CTA.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0,
                                                 int c1, int c2, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "l"(hint) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {   // arrives on `bar` in BOTH CTAs of the pair
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {  // arrive on the leader CTA's copy of `bar`
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar & kPeerBitMask) : "memory");
}

// D[tmem] (+)= A[smem] . B[smem]^T, fp16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once all previously issued MMAs have completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// K-major, 128B-swizzled smem operand descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 (unused for swizzled K-major) | [32,46) SBO>>4 = 1024B between 8-row groups
//   [46,48) version=1 | [61,64) layout=2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// cute::UMMA::InstrDescriptor: c=f32 [4,6)=1, a=f16 [7,10)=0, b=f16 [10,13)=0, K-major both,
// N>>3 at [17,23), M>>4 at [24,29)
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(kBlockN >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);
constexpr uint32_t kIdescPair = (1u << 4) | ((uint32_t)(kBlockN >> 3) << 17) | ((uint32_t)((2 * kBlockM) >> 4) << 24);

#define TMEM_LD32(taddr, r)                                                                                      \
  asm volatile(                                                                                                  \
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                  \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                                  \
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                  \
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),          \
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),    \
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),  \
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])   \
      : "r"(taddr))
#define TMEM_LD16(taddr, r)                                                                                      \
  asm volatile(                                                                                                  \
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                                  \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"                           \
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),          \
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])     \
      : "r"(taddr))
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float min3f(float a, float b, float c) {
  float r;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
// running two smallest of a stream, fed two values at a time: 5 ALU ops per pair
__device__ __forceinline__ void top2_pair(float& m1, float& m2, float a, float b) {
  float lo = fminf(a, b), hi = fmaxf(a, b);
  float t = fmaxf(m1, lo);
  m2 = min3f(m2, hi, t);
  m1 = fminf(m1, lo);
}

#ifdef VQB_TRACE
// bring-up only (-DVQB_TRACE): cluster 0 stamps clock64 per tile.  g_trace_mma[role][tile]: 0 tmem_empty seen,
// 1 MMAs + commits issued, 2 (with -DVQB_TRACE_MMA_LAT) tmem_full seen by the issuing warp itself.
// g_trace_epi[role][cta rank * 16 + warp][tile]: 0 tmem_full seen, 1 loads done + arrive sent, 2 ranked.
// The two CTAs of the pair run on different SMs: their clocks are not comparable, intervals are.
constexpr int kTraceTiles = 256;
__device__ long long g_trace_mma[3][kTraceTiles];
__device__ long long g_trace_epi[3][32][kTraceTiles];
#define VQB_STAMP_MMA(role, t) do { if ((t) < kTraceTiles) g_trace_mma[role][t] = clock64(); } while (0)
#define VQB_STAMP_EPI(role, w, t) do { if ((t) < kTraceTiles) g_trace_epi[role][w][t] = clock64(); } while (0)
#endif
constexpr float kPackSlackTC = 6.2e-5f;   // must equal kPackSlack in search_resolve.cu

// order-preserving float <-> int (involution): lets shared-memory atomicMin work on scores of either sign
__device__ __forceinline__ int f2ord(float f) { const int i = __float_as_int(f); return i ^ ((i >> 31) & 0x7fffffff); }
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }

// key = (bits & mask) | id in ONE LOP3 (mask lives in a register, id is an immediate); lut 0xEA = (a & b) | c
template <uint32_t ID>
__device__ __forceinline__ float pack_id(float v, uint32_t mask) {
  uint32_t r;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(r) : "r"(__float_as_uint(v)), "r"(mask), "n"(ID));
  return __uint_as_float(r);
}

// The epilogue is a software pipeline over 16-column chunks of one thread's row: a thread owns one row (TMEM lane)
// and a 64-column quarter of the tile = 4 chunks.  Measured with in-kernel cycle counters: a tcgen05.ld -> wait round
// trip costs ~400 cycles of latency plus ~8 cycles per column of transfer while the tensor pipe is accumulating into
// TMEM; with four epilogue warps per sub-partition those waits overlap.
//   scores : wait for the chunk's accumulators (tcgen05.wait::ld), score = acc*ninv + bias (FFMA, undoes the operand
//            scales and adds |c|^2/2 - E_k), chunk minimum with an FMNMX3 tree.  The accumulator registers are dead
//            afterwards, so the NEXT chunk's tcgen05.ld is issued right here and is in flight during
//   rank   : FAST PATH -- a score can be a candidate of the final answer only if it is <= thr_final = m + |m| slack
//            + 2E (m = final row minimum); thr is monotone in m and the running minimum only decreases, so if every
//            score of the chunk exceeds t_run = thr(running minimum, Emax) for every row of the warp, the chunk holds
//            no candidate and nothing else is done.  SLOW PATH -- 6-bit id PARITY*32 + CH*8 + i packed into the low
//            mantissa bits (column j = 2*i + c is class c), running top-2 per class, exactly as if no chunk had been
//            skipped.
__device__ __forceinline__ float chunk_scores(const uint32_t (&r)[16], const float4* bias4, float ninv,
                                              float (&key)[16]) {
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 b = bias4[i];          // shared memory, same address in every lane: broadcast
    key[4 * i + 0] = fmaf(__uint_as_float(r[4 * i + 0]), ninv, b.x);
    key[4 * i + 1] = fmaf(__uint_as_float(r[4 * i + 1]), ninv, b.y);
    key[4 * i + 2] = fmaf(__uint_as_float(r[4 * i + 2]), ninv, b.z);
    key[4 * i + 3] = fmaf(__uint_as_float(r[4 * i + 3]), ninv, b.w);
  }
  float cm[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) cm[c] = fminf(min3f(key[c], key[4 + c], key[8 + c]), key[12 + c]);
  return fminf(min3f(cm[0], cm[1], cm[2]), cm[3]);
}

template <uint32_t ID>
__device__ __forceinline__ void pack_pair(float (&key)[16], int i, uint32_t mask) {
  key[2 * i + 0] = pack_id<ID>(key[2 * i + 0], mask);
  key[2 * i + 1] = pack_id<ID>(key[2 * i + 1], mask);
}

template <int PARITY, int CH>
__device__ __forceinline__ void chunk_rank(float (&key)[16], float cmin, uint32_t idmask, float tconst, float& m_run,
                                           float& t_run, int* row_slot, float (&a1)[2], float (&a2)[2],
                                           bool& any_slow) {
  if (__any_sync(0xffffffffu, cmin <= t_run)) {
    any_slow = true;
    constexpr uint32_t kBase = (uint32_t)(PARITY * 32 + CH * 8);
    pack_pair<kBase + 0>(key, 0, idmask); pack_pair<kBase + 1>(key, 1, idmask);
    pack_pair<kBase + 2>(key, 2, idmask); pack_pair<kBase + 3>(key, 3, idmask);
    pack_pair<kBase + 4>(key, 4, idmask); pack_pair<kBase + 5>(key, 5, idmask);
    pack_pair<kBase + 6>(key, 6, idmask); pack_pair<kBase + 7>(key, 7, idmask);
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
      top2_pair(a1[0], a2[0], key[2 * i + 0], key[2 * i + 2]);
      top2_pair(a1[1], a2[1], key[2 * i + 1], key[2 * i + 3]);
    }
    if (cmin < m_run) {
      m_run = cmin;
      t_run = fminf(t_run, fmaf(fabsf(cmin), kPackSlackTC, cmin) + tconst);
      if (row_slot) atomicMin(row_slot, f2ord(cmin));     // publish to the other quarter-warps of this row
    }
  }
}

// insert (v, c) into the ascending triple (M1,M2,M3) with payloads (C1,C2,C3)
__device__ __forceinline__ void top3_insert(float& M1, float& M2, float& M3, int& C1, int& C2, int& C3, float v,
                                            int c) {
  const bool p1 = v < M1, p2 = v < M2, p3 = v < M3;
  M3 = p2 ? M2 : (p3 ? v : M3);
  C3 = p2 ? C2 : (p3 ? c : C3);
  M2 = p1 ? M1 : (p2 ? v : M2);
  C2 = p1 ? C1 : (p2 ? c : C2);
  M1 = p1 ? v : M1;
  C1 = p1 ? c : C1;
}

// ------------------------------------------------------------------------------------------
// kernel
// ------------------------------------------------------------------------------------------
// 20 warps: 0..15 epilogue (4 per SM sub-partition: TMEM-load latencies of one warp hide behind the other three),
// 16 bias stager, 17 TMEM allocator, 18 TMA producer, 19 MMA issuer.  Epilogue warp w reads TMEM lane quadrant
// w & 3 (hardware rule: a warp may only touch lanes 32*(warp%4)..+31) and the 64-column quarter w >> 2 of a tile.
constexpr int kThreads = 640;
constexpr int kNumEpiWarps = 16;
constexpr int kWarpStager = 16, kWarpAlloc = 17, kWarpTma = 18, kWarpMma = 19;
constexpr int kSlabBytes = kBlockM * kBlockK * 2;     // 16 KB: 128 rows x 64 fp16
constexpr int kStageBytes = kBlockN * kBlockK * 2;    // 32 KB: 256 codes x 64 fp16
constexpr int kMaxKB = 8;                              // d_pad <= 512
constexpr int kMaxStages = 12;
constexpr int kTmemCols = 512;

struct SearchParams {
  const float* bias;   // [H][Kp]
  const float* xn2;    // [H][N]   bound of |x_row|^2
  float tie;           // kTieSlack (Euclidean) or 0: window of fp32 distance ties = tie * xn2 (common.cuh)
  const float* xinv;   // [H][N]   1 / s_row
  const float* chdr;   // [H][4]   {s_c, 1/s_c, ..}
  void* cand;          // [H][N][24] {f32 key, i32 code}
  uint32_t* scal;
  int64_t N;           // rows per codebook
  int Kp;              // padded codes
  int H;
  int KB;              // k-blocks = d_pad / 64
  int NT;              // N tiles = Kp / 256
  int S;               // B stages
  int MT;              // row tiles per head = ceil(N/128)
};

struct Barriers {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t a_full[kMaxKB];
  uint64_t a_empty[kMaxKB];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint64_t bias_full[2];
  uint32_t tmem_base;
  uint32_t pad;
  alignas(16) float bias[2][kBlockN];   // per-accumulator-buffer copy of the N tile's biases (staged by warp 3)
  // Running row minima shared by the four quarter-warps of a row (order-preserving int encoding of the float), three
  // slots rotating with the row tile: slot (i+1)%3 is reset when a warp starts its i-th row tile.  Epilogue warps are
  // never more than ~2 N tiles apart (tmem_empty needs all of them), so with NT >= 4 no value of an older row tile
  // can land in a slot after its last reset.  Any value in the slot is a score of the CURRENT row, hence an upper
  // bound of its final minimum -- all the skip test needs.
  int rowmin[3][kBlockM];
};

// Persistent, one CTA per SM and no clusters: each CTA walks the (codebook, 128-row tile) items with a stride of the
// grid.  Launched for problems with a single row tile per codebook (search_tc_aug_mode() == 0).
__global__ void __launch_bounds__(kThreads, 1)
search_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_c,
                 const SearchParams P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t a_base = smem_base;
  const uint32_t b_base = smem_base + (uint32_t)P.KB * kSlabBytes;
  Barriers* bars = reinterpret_cast<Barriers*>(smem + (size_t)P.KB * kSlabBytes + (size_t)P.S * kStageBytes);

  const int cta = blockIdx.x;
  const int num_ctas = gridDim.x;
  const int G = P.H * P.MT;                    // (codebook, row tile) work items

  if (threadIdx.x == 0 && (smem_base & 1023u)) {   // the swizzle pattern assumes 1024B-aligned tiles
    atomicExch(P.scal + 5, 1u);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) P.scal[4] = 1u;   // "tensor-core pass ran" marker for vqb_search_stats
  if (warp == kWarpTma && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_c) : "memory");
  }
  if (warp == kWarpMma && lane == 0) {
    for (int i = 0; i < P.S; ++i) {
      mbar_init(smem_u32(&bars->full[i]), 1);
      mbar_init(smem_u32(&bars->empty[i]), 1);
    }
    for (int i = 0; i < P.KB; ++i) {
      mbar_init(smem_u32(&bars->a_full[i]), 1);
      mbar_init(smem_u32(&bars->a_empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&bars->tmem_full[i]), 1);
      mbar_init(smem_u32(&bars->tmem_empty[i]), kNumEpiWarps);
      mbar_init(smem_u32(&bars->bias_full[i]), 1);
    }
    fence_barrier_init();
  }
  if (threadIdx.x < 3 * kBlockM) (&bars->rowmin[0][0])[threadIdx.x] = 0x7fffffff;
  if (warp == kWarpAlloc) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(&bars->tmem_base)), "n"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == kWarpTma) {
    // =============================== TMA producer ===============================
    // The whole warp runs the loop (barrier waits are warp-uniform); one elected lane issues expect_tx + TMA.
    uint32_t stage = 0, ph = 0, a_ph = 0;
    for (int g = cta; g < G; g += num_ctas) {
      const int h = g / P.MT;
      const int row0 = (g - h * P.MT) * kBlockM;
      for (int nt = 0; nt < P.NT; ++nt) {
        for (int kb = 0; kb < P.KB; ++kb) {
          if (nt == 0) {   // (re)load slab kb of this row tile as soon as the previous tile's MMAs released it
            mbar_wait(smem_u32(&bars->a_empty[kb]), a_ph ^ 1u);
            if (elect_one()) {
              mbar_expect_tx(smem_u32(&bars->a_full[kb]), kSlabBytes);
              tma_load_3d(a_base + kb * kSlabBytes, &map_x, smem_u32(&bars->a_full[kb]), kb * kBlockK, row0, h,
                          kEvictFirst);
            }
            __syncwarp();
          }
          mbar_wait(smem_u32(&bars->empty[stage]), ph ^ 1u);
          if (elect_one()) {
            mbar_expect_tx(smem_u32(&bars->full[stage]), kStageBytes);
            tma_load_3d(b_base + stage * kStageBytes, &map_c, smem_u32(&bars->full[stage]), kb * kBlockK,
                        nt * kBlockN, h, kEvictLast);
          }
          __syncwarp();
          if (++stage == (uint32_t)P.S) { stage = 0; ph ^= 1u; }
        }
      }
      a_ph ^= 1u;
    }
  } else if (warp == kWarpMma) {
    // =============================== MMA issuer ===============================
    // The whole warp runs the loop; one elected lane issues the tcgen05.mma / tcgen05.commit instructions.
    uint32_t stage = 0, ph = 0, a_ph = 0, acc = 0, acc_ph = 0;
    for (int g = cta; g < G; g += num_ctas) {
      for (int nt = 0; nt < P.NT; ++nt) {
        mbar_wait(smem_u32(&bars->tmem_empty[acc]), acc_ph ^ 1u);   // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * (uint32_t)kBlockN;
        for (int kb = 0; kb < P.KB; ++kb) {
          if (nt == 0) mbar_wait(smem_u32(&bars->a_full[kb]), a_ph);
          mbar_wait(smem_u32(&bars->full[stage]), ph);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t adesc = make_sw128_desc(a_base + kb * kSlabBytes);
            const uint64_t bdesc = make_sw128_desc(b_base + stage * kStageBytes);
#pragma unroll
            for (int kk = 0; kk < kBlockK / 16; ++kk) {
              // +32 B per 16-element k step inside the 128B swizzle atom = +2 in the (addr>>4) field
              umma_f16(d_tmem, adesc + (uint64_t)(kk * 2), bdesc + (uint64_t)(kk * 2), kIdesc,
                       (kb | kk) != 0 ? 1u : 0u);
            }
            umma_commit(smem_u32(&bars->empty[stage]));
            if (nt == P.NT - 1) umma_commit(smem_u32(&bars->a_empty[kb]));     // slab kb may be overwritten
            if (kb == P.KB - 1) umma_commit(smem_u32(&bars->tmem_full[acc]));  // accumulator complete
          }
          __syncwarp();
          if (++stage == (uint32_t)P.S) { stage = 0; ph ^= 1u; }
        }
        if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
      }
      a_ph ^= 1u;
    }
  } else if (warp == kWarpStager) {
    // =============================== bias stager ===============================
    // Only ~34 KB of L1 is left next to 193 KB of dynamic smem, and the bias vector (4 B per code) is re-read for
    // every row tile, so global loads in the epilogue would miss L1 and sit in its dependency chain.  This warp
    // copies each N tile's 256 biases into smem, one slot per accumulator buffer, as soon as the epilogue has
    // released that buffer (same cadence as the MMA warp).
    // The loads of tile i+1 are issued before the wait for tile i's slot, so their L2 latency is off the critical path.
    uint32_t acc = 0, acc_ph = 0;
    int g = cta, nt = 0;
    float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
    if (g < G) {
      const float* b = P.bias + (size_t)(g / P.MT) * P.Kp;
      v0 = __ldg(reinterpret_cast<const float4*>(b) + lane);
      v1 = __ldg(reinterpret_cast<const float4*>(b) + 32 + lane);
    }
    while (g < G) {
      int g2 = g, nt2 = nt + 1;
      if (nt2 == P.NT) { nt2 = 0; g2 += num_ctas; }
      float4 n0 = v0, n1 = v1;
      if (g2 < G) {
        const float* b = P.bias + (size_t)(g2 / P.MT) * P.Kp + nt2 * kBlockN;
        n0 = __ldg(reinterpret_cast<const float4*>(b) + lane);
        n1 = __ldg(reinterpret_cast<const float4*>(b) + 32 + lane);
      }
      mbar_wait(smem_u32(&bars->tmem_empty[acc]), acc_ph ^ 1u);
      reinterpret_cast<float4*>(bars->bias[acc])[lane] = v0;
      reinterpret_cast<float4*>(bars->bias[acc])[32 + lane] = v1;
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars->bias_full[acc]));   // release semantics order the stores
      if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
      v0 = n0; v1 = n1; g = g2; nt = nt2;
    }
  } else if (warp < kNumEpiWarps) {
    // =============================== epilogue: bias + packed running top-2 ===============================
    const int q = warp & 3;                       // TMEM lane quadrant this warp may touch
    const int quarter = warp >> 2;                // which 64 of the tile's 256 columns
    uint32_t acc = 0, acc_ph = 0;
    const float INF = __int_as_float(0x7f800000);
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + quarter * 64;
    // Emax * (2 + slack): the part of the candidate threshold that does not depend on the row minimum
    const float tconst = __uint_as_float(P.scal[6]) * (2.f + kPackSlackTC);
    uint32_t r[16];
    uint32_t tile_it = 0;                           // row tiles processed by this CTA so far
    if (cta < G) {   // pipeline prologue: first chunk of the very first tile (later ones are prefetched in the loop)
      mbar_wait(smem_u32(&bars->tmem_full[0]), 0);
      tc_fence_after();
      TMEM_LD16(lane_addr, r);
    }
    for (int g = cta; g < G; g += num_ctas) {
      const int h = g / P.MT;
      const int64_t row = (int64_t)(g - h * P.MT) * kBlockM + q * 32 + lane;
      float M1[2], M2[2], M3[2];
      int C1[2], C2[2], C3[2];
#pragma unroll
      for (int c = 0; c < 2; ++c) { M1[c] = INF; M2[c] = INF; M3[c] = INF; C1[c] = -1; C2[c] = -1; C3[c] = -1; }
      // acc = (x s_row).(-c s_c)  ->  score = bias + acc / (s_row s_c): one FFMA per element
      const float ninv = row < P.N ? fabsf(P.xinv[(size_t)h * P.N + row]) * P.chdr[h * kHdrFloats + 1] : 0.f;
      // candidate window of THIS row: Emax part + the fp32 distance-tie part
      const float trow = tconst + (row < P.N ? P.tie * P.xn2[(size_t)h * P.N + row] : 0.f);
      // the id mask lives in a register so that "(bits & mask) | id" is a single LOP3 (opaque to constant folding)
      uint32_t idmask;
      asm volatile("mov.u32 %0, 0xFFFFFFC0;" : "=r"(idmask));
      float m_run = INF, t_run = INF;              // running row minimum (this thread's columns) and its threshold
      // shared running minimum of the row (all four quarters); disabled for tiny codebooks (see Barriers::rowmin)
      int* row_slot = nullptr;
      if (P.NT >= 4) {
        bars->rowmin[(tile_it + 1) % 3][q * 32 + lane] = 0x7fffffff;        // reset the NEXT row tile's slot
        row_slot = &bars->rowmin[tile_it % 3][q * 32 + lane];
      }
      ++tile_it;
      for (int nt = 0; nt < P.NT; nt += 2) {       // N tiles in pairs: one top-3 merge per 512 codes
        if (row_slot) {                            // tighten the threshold with what the other quarters have seen
          const float gmin = ord2f(*reinterpret_cast<volatile int*>(row_slot));
          t_run = fminf(t_run, fmaf(fabsf(gmin), kPackSlackTC, gmin) + trow);
        }
        float a1[2], a2[2];
#pragma unroll
        for (int c = 0; c < 2; ++c) { a1[c] = INF; a2[c] = INF; }
        bool any_slow = false;
#pragma unroll
        for (int par = 0; par < 2; ++par) {
          if (nt + par < P.NT) {
            // r[] already holds (or is receiving) chunk 0 of this tile
            const uint32_t taddr = lane_addr + acc * (uint32_t)kBlockN;
            mbar_wait(smem_u32(&bars->bias_full[acc]), acc_ph);
            const float4* bias4 = reinterpret_cast<const float4*>(bars->bias[acc] + quarter * 64);
            float key[16];
            float cmin;
#define VQB_CHUNK(CH)                                                                                      \
            cmin = chunk_scores(r, bias4 + (CH) * 4, ninv, key);                                           \
            TMEM_LD16(taddr + ((CH) + 1) * 16, r);                                                         \
            if (par == 0) chunk_rank<0, (CH)>(key, cmin, idmask, trow, m_run, t_run, row_slot, a1, a2, any_slow); \
            else chunk_rank<1, (CH)>(key, cmin, idmask, trow, m_run, t_run, row_slot, a1, a2, any_slow);
            VQB_CHUNK(0) VQB_CHUNK(1) VQB_CHUNK(2)
#undef VQB_CHUNK
            // last chunk: once its scores are formed every TMEM read of this tile is complete -> hand the buffer
            // back to the MMA warp, then start loading the next tile's first chunk (before this chunk's ranking
            // work if that accumulator is already complete)
            cmin = chunk_scores(r, bias4 + 12, ninv, key);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&bars->tmem_empty[acc]));
            if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
            const bool more = (nt + par + 1 < P.NT) || (g + num_ctas < G);
            bool issued = false;
            if (more && mbar_try(smem_u32(&bars->tmem_full[acc]), acc_ph)) {
              tc_fence_after();
              TMEM_LD16(lane_addr + acc * (uint32_t)kBlockN, r);
              issued = true;
            }
            if (par == 0) chunk_rank<0, 3>(key, cmin, idmask, trow, m_run, t_run, row_slot, a1, a2, any_slow);
            else chunk_rank<1, 3>(key, cmin, idmask, trow, m_run, t_run, row_slot, a1, a2, any_slow);
            if (more && !issued) {
              mbar_wait(smem_u32(&bars->tmem_full[acc]), acc_ph);
              tc_fence_after();
              TMEM_LD16(lane_addr + acc * (uint32_t)kBlockN, r);
            }
          }
        }
        if (!any_slow) continue;                   // warp-uniform: nothing was ranked in this tile pair
        // merge this tile pair's top-2 into the running top-3 of the class (with global code ids):
        // id bit 5 = which tile of the pair, bits 0..4 = position inside the class (column = 2*pos + class)
        const int col0 = nt * kBlockN + quarter * 64;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const uint32_t i1 = __float_as_uint(a1[c]) & 63u, i2 = __float_as_uint(a2[c]) & 63u;
          top3_insert(M1[c], M2[c], M3[c], C1[c], C2[c], C3[c], a1[c],
                      col0 + (int)(i1 >> 5) * kBlockN + (int)((i1 & 31u) << 1) + c);
          top3_insert(M1[c], M2[c], M3[c], C1[c], C2[c], C3[c], a2[c],
                      col0 + (int)(i2 >> 5) * kBlockN + (int)((i2 & 31u) << 1) + c);
        }
      }
      if (row < P.N) {
        // 6 entries {key, code} = 48 B per (row, quarter): class-major, ascending inside a class
        uint4* out4 = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(P.cand) +
                                               (((size_t)h * P.N + row) * kNumCand + quarter * (kNumCand / 4)) * 8);
        out4[0] = make_uint4(__float_as_uint(M1[0]), (uint32_t)C1[0], __float_as_uint(M2[0]), (uint32_t)C2[0]);
        out4[1] = make_uint4(__float_as_uint(M3[0]), (uint32_t)C3[0], __float_as_uint(M1[1]), (uint32_t)C1[1]);
        out4[2] = make_uint4(__float_as_uint(M2[1]), (uint32_t)C2[1], __float_as_uint(M3[1]), (uint32_t)C3[1]);
      }
    }
  }

  // teardown: everything issued has been consumed (epilogue waited on the last tmem_full)
  tc_fence_before();
  __syncthreads();
  if (warp == kWarpAlloc)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
}

// ------------------------------------------------------------------------------------------
// Bias in the MMA ("aug") variant, cta_group::2 only.
// The codebook operand is stored negated and every N tile gets ONE extra k-step whose operands are
//   A: {a, a, a, 0...} per row, a = s_row 2^-q          (fp16, written by prepare_latents)
//   B: {b1, b2, b3, 0...} per code, b1+b2+b3 = s_c 2^q |c_k|^2/2 to 33 bits (codebook cache; +inf for padded codes)
// so the fp32 accumulator IS the score times the positive row constant s_row s_c:
//   acc = s_row s_c (|c_k|^2/2 - x~.c~_k).
// The epilogue is then a pure packed min over raw accumulators: no FFMA, no bias in shared memory, no stager warp.
// Thresholds are applied in the row's scaled units; keys are unscaled once, when the 24 candidates are written.
// The bound |exact - key| <= E_k is symmetric here (the key is not pre-lowered by E_k), so the candidate window
// is min + 2 Emax: resolve uses Emax for every code (search_resolve.cu).
// Operand plumbing: the two 16-byte-per-row aug chunks use the no-swizzle K-major canonical layout (8-row core
// matrices of 128 B, SBO = 128 B); the second k-chunk (k = 8..15) of both operands is one shared block of zeros
// addressed through LBO.  The aug chunk of B rides in a 2 KB tail of every B stage and completes on the stage's
// barrier with the last k-block; the aug chunk of A completes on the last slab's barrier: no extra barriers.
// ------------------------------------------------------------------------------------------
constexpr int kAugChunkBytes = kBlockM * 16;                 // 128 rows x 8 fp16
constexpr int kStageStrideAug = kStageBytes / 2 + kAugChunkBytes;

__device__ __forceinline__ uint64_t make_nosw_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}

struct AugParams {
  const float* xn2;    // [H][N]   bound of |x_row|^2
  float tie;           // see SearchParams
  const float* xinv;   // [H][N]   +-1 / s_row
  const float* chdr;   // [H][kHdrFloats]
  void* cand;
  uint32_t* scal;
  int64_t N;
  int Kp, H, KB, NT, S, GPH;
  int aug;             // 0: dot metric with K % 256 == 0 -- no bias k-step at all
  // CONV: the kernel converts the caller's 16-bit latents itself (two extra warps, a row tile or two ahead of the
  // TMA producer) into the fp16 operand arrays that the pointers above name
  const void* xraw;    // [H][N][d] bf16 / fp16
  const __half* xb_w;  // [H][N][dp] the A operand array behind map_x
  const __half* xaug_w;
  int xdtype, d, dp;
};

struct AugBarriers {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t a_full[kMaxKB];
  uint64_t a_empty[kMaxKB];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint64_t conv_full[2];      // CONV: both converter warps wrote the operands of a row tile (count 2)
  uint64_t conv_empty[2];     // CONV: the producer took that row tile: the converters may run two tiles ahead
  uint32_t tmem_base;
  uint32_t pad;
  int rowmin[3][kBlockM];     // see Barriers::rowmin
};

// One warp converts rows [r0, r1) of codebook `h` exactly as prepare_latents4_kernel does for 16-bit latents (same
// scale, same fp16 values, same bounds), 8 rows in flight.  A row whose statistics exceed the bounds the bias
// operand was built with (scal[0] from the strided sample, the residual bound derived from it) gets a NEGATIVE xinv:
// resolve rescans it exactly.
template <typename T>
__device__ __forceinline__ void convert_rows16(const T* __restrict__ x, int64_t base, int64_t r0, int64_t r1, int d,
                                               int dp, float two_q, float two_mq, float x0sq, float x1sq,
                                               __half* __restrict__ xb, float* __restrict__ xinv,
                                               float* __restrict__ xn2, __half* __restrict__ xaug, int lane) {
  // Few registers on purpose: this code shares the kernel's 96-register budget with the epilogue; when it spilled,
  // its local-memory traffic went through the 13 KB of L1 that the kernel leaves and slowed the epilogue warps too.
  constexpr int U = 4;
  const int j = lane * 8;
  const bool on = j < d;
  const float infl = (1.f + (float)dp * 2.4e-7f) * 1.00003f;
  for (int64_t row0 = r0; row0 < r1; row0 += U) {
    Raw8<T> raw[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
      raw[u] = load_raw8<T>(x + (on && row0 + u < r1 ? (base + row0 + u) * (int64_t)d + j : 0));
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (row0 + u >= r1) break;                 // warp-uniform
      F8 vv = raw_to_f8(raw[u]);
      if (!on) {
#pragma unroll
        for (int e = 0; e < 8; ++e) vv.v[e] = 0.f;
      }
      float m = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) m = fmaxf(m, fabsf(vv.v[e]));
      // non-negative floats order like their bit patterns: one REDUX instead of five shuffle + max steps
      m = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(m)));
      float s = pow2_scale_bits(m);
      const float a = clamp_row_scale(s, two_q, two_mq);
      const float is = pow2_recip(s);
      float n2 = 0.f;
      uint32_t pk[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float v0 = vv.v[2 * e], v1 = vv.v[2 * e + 1];
        const __half2 hh = __floats2half2_rn(v0 * s, v1 * s);
        pk[e] = *reinterpret_cast<const uint32_t*>(&hh);
        n2 = fmaf(v0, v0, n2);
        n2 = fmaf(v1, v1, n2);
      }
      if (j < dp)
        *reinterpret_cast<uint4*>(xb + (base + row0 + u) * (int64_t)dp + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      // |x|^2 as an integer sum (one REDUX): the lane's part in units of m^2 2^-20, rounded UP; 8 m^2 per lane at most
      // -> < 2^24 per lane, < 2^29 per row.  An upper bound of the fp32 sum prepare_latents4 forms, within 2^-15.
      const float unit = m * m * 9.5367431640625e-7f;     // m^2 2^-20
      const uint32_t q = unit > 0.f ? (uint32_t)__float2uint_ru(__fdividef(n2, unit) * 1.000001f) + 1u : 0u;
      n2 = (float)__reduce_add_sync(0xffffffffu, q) * unit * 1.000001f;
      const float rb = 2.9802322e-8f * is;                       // 2^-25 / s
      const float r2 = m > 0.f ? (float)dp * rb * rb * 1.0001f : 0.f;   // an all-zero row converts exactly
      n2 = n2 * 1.000001f + r2 * 1.0001e6f;
      const bool ok = n2 * infl <= x0sq && r2 * infl <= x1sq;      // squares of the bounds: no square roots here
      if (lane == 0) {
        xinv[base + row0 + u] = (a > 0.f && ok) ? is : -is;
        xn2[base + row0 + u] = n2 * 1.0001f + r2 * 10002.f;        // (|x~| + |x - x~|)^2 <= n2 (1 + e) + r2 (1 + 1/e)
        const uint32_t aa = (uint32_t)__half_as_ushort(__float2half_rn(a));
        *reinterpret_cast<uint4*>(xaug + (base + row0 + u) * 8) = make_uint4(aa | (aa << 16), aa, 0u, 0u);
      }
    }
  }
}

__device__ __forceinline__ float chunk_min16(const uint32_t (&r)[16]) {
  float cm[4];
#pragma unroll
  for (int c = 0; c < 4; ++c)
    cm[c] = fminf(min3f(__uint_as_float(r[c]), __uint_as_float(r[4 + c]), __uint_as_float(r[8 + c])),
                  __uint_as_float(r[12 + c]));
  return fminf(min3f(cm[0], cm[1], cm[2]), cm[3]);
}

// The epilogue DRAINS: an epilogue warp first copies its whole 64-column quarter of the accumulator into registers and
// hands the TMEM buffer back, THEN ranks from the registers.  The buffer is then held for ~150 cycles instead of the
// whole epilogue of the tile, so the next-but-one tile's MMAs (and the barrier round trips around them) overlap the
// ranking: with a chunk-by-chunk form the epilogue warps of a d = 64 search waited for `tmem_full` a third of the time
// and the MMA warp for `tmem_empty` 63 % of it (ncu source page / cycle counters), each side waiting for the other's
// latency.  Costs 64 live accumulator registers: 18 warps (the TMA warp also allocates TMEM and writes the zero
// chunk) x 32 x 112 registers.
constexpr int kThreadsAug = 576;
constexpr int kThreadsConv = 640;      // + two converter warps (18, 19)
template <bool CONV>
__global__ void __launch_bounds__(CONV ? kThreadsConv : kThreadsAug, 1)
search_aug_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_c,
                  const __grid_constant__ CUtensorMap map_xa, const __grid_constant__ CUtensorMap map_ca,
                  const AugParams P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr int kWarpTma = 16, kWarpMma = 17, kWarpAlloc = 16, kWarpStager = 16;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t a_base = smem_base;
  const uint32_t b_base = smem_base + (uint32_t)P.KB * kSlabBytes;
  const uint32_t xa_base = b_base + (uint32_t)P.S * kStageStrideAug;       // A aug chunk (2 KB)
  const uint32_t zero_base = xa_base + kAugChunkBytes;                     // shared zero k-chunk (2 KB)
  AugBarriers* bars = reinterpret_cast<AugBarriers*>(smem + (size_t)P.KB * kSlabBytes + (size_t)P.S * kStageStrideAug +
                                                     2 * kAugChunkBytes);
  const uint32_t rank = cluster_ctarank();
  const int cid = blockIdx.x / 2;
  const int num_clusters = gridDim.x / 2;
  const int G = P.H * P.GPH;
  const bool aug = P.aug != 0;

  if (threadIdx.x == 0 && (smem_base & 1023u)) atomicExch(P.scal + 5, 1u);
  if (blockIdx.x == 0 && threadIdx.x == 0) P.scal[4] = 1u;
  if (warp == kWarpTma && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_c) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_xa) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ca) : "memory");
  }
  if (warp == kWarpMma && lane == 0) {
    for (int i = 0; i < P.S; ++i) {
      mbar_init(smem_u32(&bars->full[i]), 1);
      mbar_init(smem_u32(&bars->empty[i]), 1);
    }
    for (int i = 0; i < P.KB; ++i) {
      mbar_init(smem_u32(&bars->a_full[i]), 1);
      mbar_init(smem_u32(&bars->a_empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&bars->tmem_full[i]), 1);
      mbar_init(smem_u32(&bars->tmem_empty[i]), 2 * kNumEpiWarps);
      mbar_init(smem_u32(&bars->conv_full[i]), 2);
      mbar_init(smem_u32(&bars->conv_empty[i]), 1);
    }
    fence_barrier_init();
  }
  if (threadIdx.x < 3 * kBlockM) (&bars->rowmin[0][0])[threadIdx.x] = 0x7fffffff;
  if (warp == kWarpStager) {   // the zero k-chunk, read by the tensor core (async proxy)
    for (int i = lane; i < kAugChunkBytes / 16; i += 32)
      reinterpret_cast<uint4*>(smem + (zero_base - smem_base))[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
  }
  if (warp == kWarpAlloc) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(smem_u32(&bars->tmem_base)), "n"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == kWarpTma) {
    // =============================== TMA producer ===============================
    uint32_t stage = 0, ph = 0, a_ph = 0, c_it = 0;
    for (int g = cid; g < G; g += num_clusters) {
      const int h = g / P.GPH;
      const int mt = (g - h * P.GPH) * 2 + (int)rank;
      const int row0 = mt * kBlockM;
      if (CONV) {   // the operands of this row tile are in global memory (written by this CTA's converter warps)
#ifdef VQB_TRACE
        if (cid == 0 && rank == 0 && lane == 0) VQB_STAMP_EPI(0, 20, (int)c_it);
#endif
        mbar_wait(smem_u32(&bars->conv_full[c_it & 1u]), (c_it >> 1) & 1u);
#ifdef VQB_TRACE
        if (cid == 0 && rank == 0 && lane == 0) VQB_STAMP_EPI(1, 20, (int)c_it);
#endif
        if (elect_one()) mbar_arrive(smem_u32(&bars->conv_empty[c_it & 1u]));
        __syncwarp();
        ++c_it;
      }
      for (int nt = 0; nt < P.NT; ++nt) {
        for (int kb = 0; kb < P.KB; ++kb) {
          const bool last = kb == P.KB - 1;
          if (nt == 0) {
            mbar_wait(smem_u32(&bars->a_empty[kb]), a_ph ^ 1u);
            if (elect_one()) {
              const uint32_t bar = smem_u32(&bars->a_full[kb]);
              if (rank == 0) mbar_expect_tx(bar, 2 * kSlabBytes + (last && aug ? 2 * kAugChunkBytes : 0));
              tma_load_3d_pair(a_base + kb * kSlabBytes, &map_x, bar & kPeerBitMask, kb * kBlockK, row0, h, kEvictFirst);
              if (last && aug) tma_load_3d_pair(xa_base, &map_xa, bar & kPeerBitMask, 0, row0, h, kEvictFirst);
            }
            __syncwarp();
          }
          mbar_wait(smem_u32(&bars->empty[stage]), ph ^ 1u);
          if (elect_one()) {
            const uint32_t bar = smem_u32(&bars->full[stage]);
            if (rank == 0) mbar_expect_tx(bar, kStageBytes + (last && aug ? 2 * kAugChunkBytes : 0));
            const uint32_t dst = b_base + stage * kStageStrideAug;
            const int code0 = nt * kBlockN + (int)rank * (kBlockN / 2);
            tma_load_3d_pair(dst, &map_c, bar & kPeerBitMask, kb * kBlockK, code0, h, kEvictLast);
            if (last && aug) tma_load_3d_pair(dst + kStageBytes / 2, &map_ca, bar & kPeerBitMask, 0, code0, h, kEvictLast);
          }
          __syncwarp();
          if (++stage == (uint32_t)P.S) { stage = 0; ph ^= 1u; }
        }
      }
      a_ph ^= 1u;
    }
  } else if (warp == kWarpMma) {
    // =============================== MMA issuer (leader CTA) ===============================
    if (rank == 0) {
      uint32_t stage = 0, ph = 0, a_ph = 0, acc = 0, acc_ph = 0;
#ifdef VQB_TRACE
      int tr_t = 0;
#endif
      for (int g = cid; g < G; g += num_clusters) {
        for (int nt = 0; nt < P.NT; ++nt) {
          const uint32_t d_tmem = tmem_base + acc * (uint32_t)kBlockN;
          if (P.KB == 1) {
            // d_pad = 64: one stage per N tile, and the accumulator hand-off is the critical path (clock stamps,
            // tools/trace_d64.py: buffer free -> MMAs issued took 760 cycles with the stage wait and the descriptor
            // arithmetic after the `tmem_empty` wait, 350 with them before it).  The stage has been full for a long
            // time (the ring runs ahead), so everything that does not need the accumulator goes first.
            if (nt == 0) mbar_wait(smem_u32(&bars->a_full[0]), a_ph);
            mbar_wait(smem_u32(&bars->full[stage]), ph);
            const uint32_t b_addr = b_base + stage * kStageStrideAug;
            const uint32_t ca = b_addr + kStageBytes / 2;
            const uint64_t adesc = make_sw128_desc(a_base);
            const uint64_t bdesc = make_sw128_desc(b_addr);
            const uint64_t xdesc = make_nosw_desc(xa_base, zero_base - xa_base, 128);
            const uint64_t cdesc = make_nosw_desc(ca, zero_base - ca, 128);
            asm volatile("" ::"l"(adesc), "l"(bdesc), "l"(xdesc), "l"(cdesc));   // materialised here, not after the wait
            mbar_wait(smem_u32(&bars->tmem_empty[acc]), acc_ph ^ 1u);   // epilogues of both CTAs drained this buffer
#ifdef VQB_TRACE
            if (cid == 0 && lane == 0) VQB_STAMP_MMA(0, tr_t);
#endif
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
              for (int kk = 0; kk < kBlockK / 16; ++kk)
                umma_f16_pair(d_tmem, adesc + (uint64_t)(kk * 2), bdesc + (uint64_t)(kk * 2), kIdescPair, kk != 0 ? 1u : 0u);
              if (aug) umma_f16_pair(d_tmem, xdesc, cdesc, kIdescPair, 1u);   // + a (b1 + b2 + b3) = s_row s_c |c|^2/2
              umma_commit_pair(smem_u32(&bars->tmem_full[acc]));              // the hand-off first
              umma_commit_pair(smem_u32(&bars->empty[stage]));
              if (nt == P.NT - 1) umma_commit_pair(smem_u32(&bars->a_empty[0]));
            }
            __syncwarp();
            if (++stage == (uint32_t)P.S) { stage = 0; ph ^= 1u; }
          } else {
            mbar_wait(smem_u32(&bars->tmem_empty[acc]), acc_ph ^ 1u);
            tc_fence_after();
            for (int kb = 0; kb < P.KB; ++kb) {
              if (nt == 0) mbar_wait(smem_u32(&bars->a_full[kb]), a_ph);
              mbar_wait(smem_u32(&bars->full[stage]), ph);
              tc_fence_after();
              if (elect_one()) {
                const uint32_t b_addr = b_base + stage * kStageStrideAug;
                const uint64_t adesc = make_sw128_desc(a_base + kb * kSlabBytes);
                const uint64_t bdesc = make_sw128_desc(b_addr);
#pragma unroll
                for (int kk = 0; kk < kBlockK / 16; ++kk)
                  umma_f16_pair(d_tmem, adesc + (uint64_t)(kk * 2), bdesc + (uint64_t)(kk * 2), kIdescPair,
                                (kb | kk) != 0 ? 1u : 0u);
                if (kb == P.KB - 1 && aug) {        // + a (b1 + b2 + b3) = s_row s_c |c|^2/2
                  const uint32_t ca = b_addr + kStageBytes / 2;
                  umma_f16_pair(d_tmem, make_nosw_desc(xa_base, zero_base - xa_base, 128),
                                make_nosw_desc(ca, zero_base - ca, 128), kIdescPair, 1u);
                }
                umma_commit_pair(smem_u32(&bars->empty[stage]));
                if (nt == P.NT - 1) umma_commit_pair(smem_u32(&bars->a_empty[kb]));
                if (kb == P.KB - 1) umma_commit_pair(smem_u32(&bars->tmem_full[acc]));
              }
              __syncwarp();
              if (++stage == (uint32_t)P.S) { stage = 0; ph ^= 1u; }
            }
          }
#ifdef VQB_TRACE
          if (cid == 0 && lane == 0) VQB_STAMP_MMA(1, tr_t);
#ifdef VQB_TRACE_MMA_LAT
          mbar_wait(smem_u32(&bars->tmem_full[acc]), acc_ph);   // the issuing warp itself watches the accumulator complete
#endif
#endif
#ifdef VQB_TRACE
          if (cid == 0 && lane == 0) VQB_STAMP_MMA(2, tr_t);
          ++tr_t;
#endif
          if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
        }
        a_ph ^= 1u;
      }
    }
  } else if (CONV && warp >= 18) {
    // =============================== converter warps (CONV) ===============================
    // Each converts 64 of the CTA's 128 rows of every row tile, in the CTA's own tile order, at most two row tiles
    // ahead of the producer: the fp16 rows are still in L2 when the TMA load comes for them.  The tensor pipe is the
    // bound of this kernel and HBM nearly idle, so the conversion pass costs nothing on the step's critical path.
    const int cw = warp - 18;
    const float x0 = __uint_as_float(P.scal[0]);
    const float x0sq = x0 * x0 * 0.99999f;
    uint32_t c_it = 0;
    for (int g = cid; g < G; g += num_clusters, ++c_it) {
      const int h = g / P.GPH;
      const int mt = (g - h * P.GPH) * 2 + (int)rank;
#ifdef VQB_TRACE
      if (cid == 0 && rank == 0 && lane == 0) VQB_STAMP_EPI(0, 18 + cw, (int)c_it);
#endif
      mbar_wait(smem_u32(&bars->conv_empty[c_it & 1u]), ((c_it >> 1) & 1u) ^ 1u);
#ifdef VQB_TRACE
      if (cid == 0 && rank == 0 && lane == 0) VQB_STAMP_EPI(1, 18 + cw, (int)c_it);
#endif
      const int64_t r0 = (int64_t)mt * kBlockM + cw * (kBlockM / 2);
      const int64_t r1 = r0 + kBlockM / 2 < P.N ? r0 + kBlockM / 2 : P.N;
      const float two_q = P.chdr[h * kHdrFloats + 4], two_mq = P.chdr[h * kHdrFloats + 5];
      const float x1 = dx_bound_16bit(x0, P.dp, two_mq);
      const float x1sq = x1 * x1 * 0.99999f;
      const int64_t base = (int64_t)h * P.N;
      if (r0 < r1 && P.xdtype >= 0) {
        if (P.xdtype == VQB_BF16)
          convert_rows16<__nv_bfloat16>((const __nv_bfloat16*)P.xraw, base, r0, r1, P.d, P.dp, two_q, two_mq, x0sq, x1sq,
                                        const_cast<__half*>(P.xb_w), const_cast<float*>(P.xinv),
                                        const_cast<float*>(P.xn2), const_cast<__half*>(P.xaug_w), lane);
        else
          convert_rows16<__half>((const __half*)P.xraw, base, r0, r1, P.d, P.dp, two_q, two_mq, x0sq, x1sq,
                                 const_cast<__half*>(P.xb_w), const_cast<float*>(P.xinv), const_cast<float*>(P.xn2),
                                 const_cast<__half*>(P.xaug_w), lane);
      }
      // generic-proxy global writes -> read by the TMA unit (async proxy) of this CTA
      asm volatile("fence.proxy.async;" ::: "memory");
      __threadfence_block();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars->conv_full[c_it & 1u]));
#ifdef VQB_TRACE
      if (cid == 0 && rank == 0 && lane == 0) VQB_STAMP_EPI(2, 18 + cw, (int)c_it);
#endif
    }
  } else if (warp < kNumEpiWarps) {
    // =============================== epilogue: packed running top-2 on raw accumulators ===============================
    const int q = warp & 3;
    const int quarter = warp >> 2;
    uint32_t acc = 0, acc_ph = 0;
    const float INF = __int_as_float(0x7f800000);
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + quarter * 64;
    const float tconst = __uint_as_float(P.scal[6]) * (2.f + kPackSlackTC);
    uint32_t rD[4][16];                      // the whole 64-column quarter
    uint32_t tile_it = 0;
    for (int g = cid; g < G; g += num_clusters) {
      const int h = g / P.GPH;
      const int mt = (g - h * P.GPH) * 2 + (int)rank;
      const int64_t row = (int64_t)mt * kBlockM + q * 32 + lane;
      float M1[2], M2[2], M3[2];
      int C1[2], C2[2], C3[2];
#pragma unroll
      for (int c = 0; c < 2; ++c) { M1[c] = INF; M2[c] = INF; M3[c] = INF; C1[c] = -1; C2[c] = -1; C3[c] = -1; }
      // key = s_row s_c score: inv undoes it (exact, powers of two); thresholds live in the scaled units
      // CONV: the row scalars are written by this CTA's converter warps, possibly only moments ago (first row tile of
      // the kernel): they are read after the row tile's first `tmem_full` wait, which orders them (converter ->
      // producer -> TMA -> MMA -> here); read at this point they could still be what an earlier search left behind
      float inv = 0.f, trow = 0.f;
      if (!CONV) {
        inv = row < P.N ? fabsf(P.xinv[(size_t)h * P.N + row]) * P.chdr[h * kHdrFloats + 1] : 0.f;
        // candidate window of this row in its scaled units: Emax part + the fp32 distance-tie part
        trow = inv > 0.f ? (tconst + P.tie * P.xn2[(size_t)h * P.N + row]) / inv : 0.f;
      }
      uint32_t idmask;
      asm volatile("mov.u32 %0, 0xFFFFFFC0;" : "=r"(idmask));
      float m_run = INF, t_run = INF;
      int* row_slot = nullptr;
      if (P.NT >= 4) {
        bars->rowmin[(tile_it + 1) % 3][q * 32 + lane] = 0x7fffffff;
        row_slot = &bars->rowmin[tile_it % 3][q * 32 + lane];
      }
      ++tile_it;
      for (int nt = 0; nt < P.NT; nt += 2) {
        if (row_slot) {
          const float gmin = ord2f(*reinterpret_cast<volatile int*>(row_slot));
          t_run = fminf(t_run, fmaf(fabsf(gmin), kPackSlackTC, gmin) + trow);
        }
        float a1[2], a2[2];
#pragma unroll
        for (int c = 0; c < 2; ++c) { a1[c] = INF; a2[c] = INF; }
        bool any_slow = false;
#pragma unroll
        for (int par = 0; par < 2; ++par) {
          if (nt + par < P.NT) {
            const uint32_t taddr = lane_addr + acc * (uint32_t)kBlockN;
            mbar_wait(smem_u32(&bars->tmem_full[acc]), acc_ph);
            if (CONV && nt == 0 && par == 0) {
              const volatile float* vx = P.xinv;
              const volatile float* vn = P.xn2;
              inv = row < P.N ? fabsf(vx[(size_t)h * P.N + row]) * P.chdr[h * kHdrFloats + 1] : 0.f;
              trow = inv > 0.f ? (tconst + P.tie * vn[(size_t)h * P.N + row]) / inv : 0.f;
            }
#ifdef VQB_TRACE
            const int tr_t = (int)(tile_it - 1) * P.NT + nt + par;
            const bool tr_on = cid == 0 && lane == 0;
            const int tr_w = (int)rank * 16 + warp;
            if (tr_on) VQB_STAMP_EPI(0, tr_w, tr_t);
#endif
            tc_fence_after();
            TMEM_LD16(taddr, rD[0]);
            TMEM_LD16(taddr + 16, rD[1]);
            TMEM_LD16(taddr + 32, rD[2]);
            TMEM_LD16(taddr + 48, rD[3]);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(smem_u32(&bars->tmem_empty[acc]));   // buffer handed back: rank from registers
#ifdef VQB_TRACE
            if (tr_on) VQB_STAMP_EPI(1, tr_w, tr_t);
#endif
            if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
            float cmin;
            // the accumulator registers ARE the keys
#define VQB_RANK_CHUNK(CH)                                                                                  \
            cmin = chunk_min16(rD[CH]);                                                                     \
            if (par == 0) chunk_rank<0, (CH)>(reinterpret_cast<float(&)[16]>(rD[CH]), cmin, idmask, trow, m_run, \
                                              t_run, row_slot, a1, a2, any_slow);                           \
            else chunk_rank<1, (CH)>(reinterpret_cast<float(&)[16]>(rD[CH]), cmin, idmask, trow, m_run, t_run,   \
                                     row_slot, a1, a2, any_slow);
            VQB_RANK_CHUNK(0) VQB_RANK_CHUNK(1) VQB_RANK_CHUNK(2) VQB_RANK_CHUNK(3)
#undef VQB_RANK_CHUNK
#ifdef VQB_TRACE
            if (tr_on) VQB_STAMP_EPI(2, tr_w, tr_t);
#endif
          }
        }
        if (!any_slow) continue;
        const int col0 = nt * kBlockN + quarter * 64;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const uint32_t i1 = __float_as_uint(a1[c]) & 63u, i2 = __float_as_uint(a2[c]) & 63u;
          top3_insert(M1[c], M2[c], M3[c], C1[c], C2[c], C3[c], a1[c],
                      col0 + (int)(i1 >> 5) * kBlockN + (int)((i1 & 31u) << 1) + c);
          top3_insert(M1[c], M2[c], M3[c], C1[c], C2[c], C3[c], a2[c],
                      col0 + (int)(i2 >> 5) * kBlockN + (int)((i2 & 31u) << 1) + c);
        }
      }
      if (row < P.N) {
        uint4* out4 = reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(P.cand) +
                                               (((size_t)h * P.N + row) * kNumCand + quarter * (kNumCand / 4)) * 8);
#pragma unroll
        for (int c = 0; c < 2; ++c) { M1[c] *= inv; M2[c] *= inv; M3[c] *= inv; }   // inf stays inf
        out4[0] = make_uint4(__float_as_uint(M1[0]), (uint32_t)C1[0], __float_as_uint(M2[0]), (uint32_t)C2[0]);
        out4[1] = make_uint4(__float_as_uint(M3[0]), (uint32_t)C3[0], __float_as_uint(M1[1]), (uint32_t)C1[1]);
        out4[2] = make_uint4(__float_as_uint(M2[1]), (uint32_t)C2[1], __float_as_uint(M3[1]), (uint32_t)C3[1]);
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == kWarpAlloc)
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = (EncodeTiledFn)p;
  return fn;
}

// 3-D fp16 tensor (inner, rows, heads), box (box_inner, box_rows, 1), OOB rows read as zero;
// 128B swizzle for the 64-wide operand tiles, none for the 8-wide bias chunks
static int make_map(CUtensorMap* m, const void* base, int inner, int64_t rows, int64_t heads, int box_rows,
                    int box_inner = kBlockK) {
  EncodeTiledFn enc = get_encode_fn();
  VQB_REQUIRE(enc != nullptr, VQB_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)rows, (cuuint64_t)heads};
  cuuint64_t strides[2] = {(cuuint64_t)inner * 2, (cuuint64_t)inner * 2 * (cuuint64_t)rows};
  cuuint32_t box[3] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE,
                   box_inner == kBlockK ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VQB_REQUIRE(r == CUDA_SUCCESS, VQB_ERR_CUDA, "cuTensorMapEncodeTiled failed: %d (inner=%d rows=%lld heads=%lld)",
              (int)r, inner, (long long)rows, (long long)heads);
  return VQB_OK;
}

// timing ring for VQB_SEARCH_TIMING: event pairs recorded on the search stream around the kernel launch
constexpr int kTimingSlots = 64;
static cudaEvent_t g_ev0[kTimingSlots], g_ev1[kTimingSlots];
static bool g_ev_made = false;
static int g_ev_dev = -1;              // the events belong to the device of the first timed search
static int g_ev_count = 0;
static int g_num_sms = 0;              // SMs of the device of the first search: one CTA per SM

// Launches a persistent search kernel: clusters of `cluster` CTAs, one CTA per SM but no more clusters than the G
// work items, 227 KB of dynamic shared memory allowed; `timing` brackets the launch with an event pair of the ring.
template <auto Kernel, typename... Args>
static int launch_search_kernel(int cluster, int G, int threads, size_t smem_bytes, bool timing, cudaStream_t st,
                                const Args&... args) {
  static bool configured[64] = {};      // function attributes are per device
  int dev = 0;
  VQB_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    VQB_CUDA_TRY(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  if (!g_num_sms) VQB_CUDA_TRY(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  int nclusters = g_num_sms / cluster;
  if (nclusters > G) nclusters = G;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(nclusters * cluster));
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int slot = -1;
  if (timing && (g_ev_dev < 0 || g_ev_dev == dev)) {
    if (!g_ev_made) {
      g_ev_dev = dev;
      for (int i = 0; i < kTimingSlots; ++i) {
        VQB_CUDA_TRY(cudaEventCreate(&g_ev0[i]));
        VQB_CUDA_TRY(cudaEventCreate(&g_ev1[i]));
      }
      g_ev_made = true;
    }
    if (g_ev_count < kTimingSlots) slot = g_ev_count++;
  }
  if (slot >= 0) VQB_CUDA_TRY(cudaEventRecord(g_ev0[slot], st));
  VQB_CUDA_TRY(cudaLaunchKernelEx(&cfg, Kernel, args...));
  ++g_launch_count;
  if (slot >= 0) VQB_CUDA_TRY(cudaEventRecord(g_ev1[slot], st));
  return VQB_OK;
}

// 0: one row tile per codebook, bias added in the epilogue (search_tc_kernel); 1: search_aug_kernel with the bias
// k-step; 2: search_aug_kernel without any bias (dot metric, no padded codes).  The pair kernel needs >= 2 row tiles.
int search_tc_aug_mode(int64_t N, int K, int metric) {
  if ((N + kBlockM - 1) / kBlockM < 2) return 0;
  return (metric == VQB_DOT && K % kBlockN == 0) ? 2 : 1;
}

// In-kernel conversion of 16-bit latents (CONV, opt-in: VQB_SEARCH_FUSED_PREP): the two converter warps keep up when
// a row tile carries enough tensor work; below that the separate prepare pass stays.
// env VQB_FUSED_PREP: 1 = on for every qualifying search, 0 = never, 2 = bring-up (converter warps present but idle,
// operands from the separate pass); unset: the caller's flag decides.
int search_tc_conv_ok(int64_t N, int K, int d, int x_dtype, int aug_mode, int requested) {
  static int env = -2;
  if (env == -2) { const char* e = getenv("VQB_FUSED_PREP"); env = e ? atoi(e) : -1; }
  const int on = env >= 0 ? env : (requested ? 1 : 0);
  if (on == 2) return 2;
  if (!on || !aug_mode || x_dtype == VQB_F32 || (d & 7) || d > 256) return 0;
  const int dp = d_pad(d);
  const int64_t work = (int64_t)(k_pad(K) / kBlockN) * (dp / kBlockK);       // MMA k-blocks per row tile
  return (work >= 96 && N >= 64 * kBlockM) ? 1 : 0;
}

static int launch_aug(const __half* xb, const float* xinv, const float* xn2, float tie, const __half* xaug,
                      const __half* cb, const __half* caug,
                      const float* chdr, int64_t H, int64_t N, int K, int dp, int aug_on, void* cand, uint32_t* scal,
                      bool timing, cudaStream_t st, const ConvArgs& conv) {
  const int Kp = k_pad(K);
  AugParams P;
  P.xraw = conv.x; P.xdtype = conv.x_dtype; P.d = conv.d; P.dp = dp; P.xb_w = xb; P.xaug_w = xaug;
  P.xinv = xinv; P.xn2 = xn2; P.tie = tie; P.chdr = chdr; P.cand = cand; P.scal = scal; P.N = N; P.Kp = Kp;
  P.H = (int)H;
  P.KB = dp / kBlockK;
  P.NT = Kp / kBlockN;
  P.aug = aug_on;
  const size_t fixed = (size_t)P.KB * kSlabBytes + 2 * kAugChunkBytes + sizeof(AugBarriers);
  int S = (int)((227 * 1024 - fixed) / kStageStrideAug);
  if (S > kMaxStages) S = kMaxStages;
  VQB_REQUIRE(S >= 2, VQB_ERR_UNSUPPORTED, "not enough shared memory for d_pad=%d", dp);
  P.S = S;
  const int MT = (int)((N + kBlockM - 1) / kBlockM);
  P.GPH = (MT + 1) / 2;
  const size_t smem_bytes = fixed + (size_t)S * kStageStrideAug;
  const int G = (int)H * P.GPH;
  CUtensorMap mx, mc, mxa, mca;
  int rc = make_map(&mx, xb, dp, N, H, kBlockM);
  if (rc) return rc;
  rc = make_map(&mc, cb, dp, Kp, H, kBlockN / 2);
  if (rc) return rc;
  rc = make_map(&mxa, xaug, 8, N, H, kBlockM, 8);
  if (rc) return rc;
  rc = make_map(&mca, caug, 8, Kp, H, kBlockN / 2, 8);
  if (rc) return rc;
  if (conv.x != nullptr)
    return launch_search_kernel<search_aug_kernel<true>>(2, G, kThreadsConv, smem_bytes, timing, st, mx, mc, mxa, mca, P);
  return launch_search_kernel<search_aug_kernel<false>>(2, G, kThreadsAug, smem_bytes, timing, st, mx, mc, mxa, mca, P);
}

int launch_search_tc(const __half* xb, const float* xinv, const float* xn2, float tie, const __half* xaug,
                     const __half* cb, const __half* caug, const float* chdr, const float* bias, int aug_mode,
                     int64_t H, int64_t N, int K, int dp, void* cand, uint32_t* scal, bool timing, cudaStream_t st,
                     const ConvArgs& conv) {
  const int Kp = k_pad(K);
  VQB_REQUIRE(conv.x == nullptr || aug_mode, VQB_ERR_INVALID, "in-kernel latent conversion needs the bias k-step kernel");
  if (aug_mode) {
    VQB_REQUIRE(xaug && caug, VQB_ERR_INVALID, "search: bias operands missing");
    VQB_REQUIRE(dp % kBlockK == 0 && dp / kBlockK <= kMaxKB, VQB_ERR_UNSUPPORTED, "d_pad %d unsupported by the TC path", dp);
    VQB_REQUIRE(N < (1ll << 31) - kBlockM, VQB_ERR_UNSUPPORTED, "N too large for TMA coordinates");
    return launch_aug(xb, xinv, xn2, tie, xaug, cb, caug, chdr, H, N, K, dp, aug_mode == 1 ? 1 : 0, cand, scal, timing,
                      st, conv);
  }
  VQB_REQUIRE(dp % kBlockK == 0 && dp / kBlockK <= kMaxKB, VQB_ERR_UNSUPPORTED, "d_pad %d unsupported by the TC path", dp);
  VQB_REQUIRE(N < (1ll << 31) - kBlockM, VQB_ERR_UNSUPPORTED, "N too large for TMA coordinates");
  SearchParams P;
  P.bias = bias; P.xinv = xinv; P.xn2 = xn2; P.tie = tie; P.chdr = chdr; P.cand = cand; P.scal = scal; P.N = N;
  P.Kp = Kp; P.H = (int)H;
  P.KB = dp / kBlockK;
  P.NT = Kp / kBlockN;
  const size_t fixed = (size_t)P.KB * kSlabBytes + sizeof(Barriers);
  int S = (int)((227 * 1024 - fixed) / kStageBytes);
  if (S > kMaxStages) S = kMaxStages;
  VQB_REQUIRE(S >= 2, VQB_ERR_UNSUPPORTED, "not enough shared memory for d_pad=%d", dp);
  P.S = S;
  P.MT = (int)((N + kBlockM - 1) / kBlockM);
  const size_t smem_bytes = fixed + (size_t)S * kStageBytes;

  CUtensorMap mx, mc;
  int rc = make_map(&mx, xb, dp, N, H, kBlockM);
  if (rc) return rc;
  rc = make_map(&mc, cb, dp, Kp, H, kBlockN);
  if (rc) return rc;
  return launch_search_kernel<search_tc_kernel>(1, (int)H * P.MT, kThreads, smem_bytes, timing, st, mx, mc, P);
}

int search_timing(float* host_ms, int cap) {
  const int n = g_ev_count;
  for (int i = 0; i < n; ++i) {
    VQB_CUDA_TRY(cudaEventSynchronize(g_ev1[i]));
    float ms = 0.f;
    VQB_CUDA_TRY(cudaEventElapsedTime(&ms, g_ev0[i], g_ev1[i]));
    if (i < cap && host_ms) host_ms[i] = ms;
  }
  g_ev_count = 0;
  return n;
}

}  // namespace vqb

#ifdef VQB_TRACE
extern "C" int vqb_debug_trace(long long* mma, long long* epi) {   // [3][kTraceTiles], [3][32][kTraceTiles]
  if (cudaMemcpyFromSymbol(mma, vqb::g_trace_mma, sizeof(long long) * 3 * vqb::kTraceTiles) != cudaSuccess) return -1;
  return cudaMemcpyFromSymbol(epi, vqb::g_trace_epi, sizeof(long long) * 96 * vqb::kTraceTiles) == cudaSuccess ? 0 : -1;
}
#endif
extern "C" int vqb_search_timing(float* host_ms, int cap) { return vqb::search_timing(host_ms, cap); }
