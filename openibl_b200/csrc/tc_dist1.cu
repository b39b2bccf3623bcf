// Query x database distance + top-k, screening in ONE tensor-core pass (SURVEY 8 rows a8/a9; replaces
// pairwise_distance + np.argsort, reference ibl/evaluators.py:127-129,143, for the ranks evaluate_all reads).
//
// Round 1 screened with the bf16x3 split (3 MMAs per product) although every survivor is re-scored in exact
// fp32 anyway.  Here:
//   1. rows_f16_kernel        one pass per matrix: fp16 plane of each row scaled by a power of two (row max in
//                             [0.5,1): no overflow, 11 significant bits), exact fp32 |x|^2 (same summation order as
//                             planes_sqnorm_kernel, so the exact distances below are unchanged) and the row's
//                             representation error |x - plane * 2^e| (exact per element, fp16 subnormals included);
//   2. gemm2_f16_top16_kernel tcgen05.mma.cta_group::2 kind::f16 (fp16 x fp16 -> fp32 in TMEM), ONE MMA per
//                             K step, 256 queries x 256 database rows per SM pair, 6-stage TMA ring, running
//                             top-16 per query in registers across the pair's database range;
//   3. dist_finish_kernel     per query: merge of the per-range candidate lists, exact fp32 re-scoring of the 16
//                             survivors (|q|^2 + |d|^2 - 2 q.d, bit-identical to round 1's rescore_sort_kernel),
//                             final (dist, idx) sort, and the GUARD: a database row that was NOT kept has a
//                             screened distance >= s16 (the 16th screened distance); its exact distance is
//                             >= s16 - B with B = screen_guard_bound (common.cuh), a bound for any input: the
//                             representation errors of the query and of the worst database row (Cauchy-Schwarz),
//                             the TMEM accumulator's truncation (d/16 MMAs, per-MMA loss from the kind::bf16
//                             measurement x 18) and fp32 rounding of both distance expressions.  Unless
//                             s16 - B > (k-th exact distance) the query is appended to a device-side list;
//   4. dist_exact_chunk_kernel / dist_exact_merge_kernel   listed queries (none on descriptor-like data: B is
//                             ~8e-4 for unit 4096-d rows, the k-th to 16th gap is larger) are ranked again by exact
//                             fp32 brute force, without any host round trip: the kernels size their work from the
//                             device counter.  The bf16x3 paths of ibl_l2dist_topk use the same fallback.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace ibl {

using namespace tc;

// ---- 1. fp16 planes -----------------------------------------------------------------------------
// aux[r] = {|x|^2 (exact fp32), 2^e (x = plane * 2^e), |x - plane * 2^e|, 0}
__global__ void __launch_bounds__(256)
rows_f16_kernel(const float* __restrict__ x, int D, __half* __restrict__ plane, float4* __restrict__ aux) {
  __shared__ float red[8], redm[8];
  __shared__ float scale_s, tot_s;
  const long long r = blockIdx.x;
  const float4* p = reinterpret_cast<const float4*>(x + r * D);
  float ss = 0.f, mx = 0.f;
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) {
    const float4 v = __ldg(p + i);
    ss = fmaf(v.x, v.x, ss); ss = fmaf(v.y, v.y, ss); ss = fmaf(v.z, v.z, ss); ss = fmaf(v.w, v.w, ss);
    mx = fmaxf(fmaxf(mx, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = ss; redm[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f, m = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { tot += red[i]; m = fmaxf(m, redm[i]); }
    int e = 0;
    if (m > 0.f && m < INFINITY) frexpf(m, &e);       // m = f * 2^e, f in [0.5, 1)
    scale_s = ldexpf(1.f, -e);
    tot_s = tot;
  }
  __syncthreads();
  const float inv = scale_s, sc = 1.f / inv;
  uint2* ph = reinterpret_cast<uint2*>(plane + r * D);
  float se = 0.f;
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) {   // second read of the row: L1/L2 hits
    const float4 v = __ldg(p + i);
    const __half2 a = __floats2half2_rn(v.x * inv, v.y * inv), b = __floats2half2_rn(v.z * inv, v.w * inv);
    ph[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
    // x - plane * 2^e: the product is exact and the difference is exact (Sterbenz; or plane = 0)
    const float e0 = v.x - __low2float(a) * sc, e1 = v.y - __high2float(a) * sc;
    const float e2 = v.z - __low2float(b) * sc, e3 = v.w - __high2float(b) * sc;
    se = fmaf(e0, e0, se); se = fmaf(e1, e1, se); se = fmaf(e2, e2, se); se = fmaf(e3, e3, se);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
  __syncthreads();                                     // red[] of the first reduction has been read
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = se;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tote = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tote += red[i];
    aux[r] = make_float4(tot_s, sc, sqrtf(tote), 0.f);
  }
}

// max over the database rows of (|x - x'|, |x|^2): the guard's bound for rows that were not kept.  sq / err are
// read with a stride (4: the float4 aux of this file; 1: plain arrays of the bf16x3 path).
__global__ void dist_colmax_kernel(const float* __restrict__ sq, const float* __restrict__ err, int stride, int n,
                                   float* __restrict__ out2) {
  float a = 0.f, c = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    a = fmaxf(a, __ldg(err + (long long)i * stride));
    c = fmaxf(c, __ldg(sq + (long long)i * stride));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, o));
    c = fmaxf(c, __shfl_xor_sync(0xffffffffu, c, o));
  }
  if ((threadIdx.x & 31) == 0) {     // non-negative floats order like their bit patterns
    atomicMax(reinterpret_cast<int*>(out2), __float_as_int(a));
    atomicMax(reinterpret_cast<int*>(out2) + 1, __float_as_int(c));
  }
}

int launch_dist_colmax(const float* sq, const float* err, int stride, int n, float* out2, cudaStream_t s) {
  if (n <= 0) return IBL_OK;
  dist_colmax_kernel<<<cdiv(n, 256) < 64 ? cdiv(n, 256) : 64, 256, 0, s>>>(sq, err, stride, n, out2);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}

// ---- 2. screening GEMM on SM pairs ----------------------------------------------------------------
struct Dist1Args {
  int M, N, K;
  int n_tiles, nt_per_item, items_per_mpair, total_items, n_valid;
  const float4* a_aux;  // per query  {|q|^2, 2^eq, ...}
  const float4* b_aux;  // per db row {|d|^2, 2^ed, ...}
  float* cand_d;        // [items_per_mpair][M][16] screened distances
  int* cand_i;          // [items_per_mpair][M][16] local database rows (-1: none)
  unsigned* gate;       // [M] orderable bits of the smallest 16th-best distance any work item of this query has reached
};

__host__ __device__ constexpr uint32_t umma_idesc_f16_f32(int M, int N) {   // kind::f16, fp16 A/B, fp32 accumulator
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ uint32_t d1_ord(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float d1_unord(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__device__ __forceinline__ void d1_sts64(uint32_t addr, float x, float y) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(x), "f"(y) : "memory");
}
__device__ __forceinline__ float2 d1_lds64(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr) : "memory");
  return v;
}

constexpr int D1_BN = 256, D1_BK = 64;
constexpr int D1_PEND = 32;                            // pending candidates per row between two merges (see the epilogue)
constexpr int D1_A_BYTES = 128 * D1_BK * 2;            // 16 KiB: this CTA's 128 query rows
constexpr int D1_BH_BYTES = (D1_BN / 2) * D1_BK * 2;   // 16 KiB: this CTA's half of one 256-row database sub-tile

// SUB = 256-row database sub-tiles per work tile.  SUB = 1 (default): 256 x 256 tiles, two 256-column accumulators, the
// epilogue of tile i runs under the main loop of tile i+1.  SUB = 2 (IBL_DIST_BN=512): a 256 x 512 tile reuses every
// staged query block for two MMAs (48 KiB per stage instead of 2 x 32: 25 % less L2->SM traffic) but has ONE 512-column
// accumulator, so epilogue and main loop alternate.  Measured (profiles/r02_dist_variants_s8.jsonl, whole call,
// 6.8k x {10k, 31k, 250k} x 4096): SUB = 1 0.70 / 1.62 / 11.9 ms, SUB = 2 0.79 / 1.80 / 12.4 ms.
template <int SUB> struct D1Cfg {
  static constexpr int STAGES = SUB == 1 ? 6 : 4;
  static constexpr int STAGE = D1_A_BYTES + SUB * D1_BH_BYTES;
  static constexpr int TILE_N = D1_BN * SUB;
  static constexpr int ACC_BUFS = SUB == 1 ? 2 : 1;
  static constexpr int BARS = 256;                      // mbarriers + the TMEM slot
  static constexpr int BSTAGE = 4 * 32 * 8;             // per epilogue warp: {|d|^2, 2^e} of the 32 columns of a chunk
  static constexpr int PEND = 128 * D1_PEND * 8;        // per query row: D1_PEND pending (distance, column) pairs
  static constexpr int SMEM = STAGES * STAGE + BARS + BSTAGE + PEND + 1024;
};

// SM pairs: the peer CTA's producer does NOT arrive on the leader's full barrier.  The leader's single
// arrive.expect_tx names the bytes of BOTH CTAs; the peer's TMA completions decrement the same transaction count
// (complete_tx may land before the expect_tx: the phase still cannot complete before the leader's arrival).  Round 1
// had the peer do an `mbarrier.arrive.release.cluster` per stage; removing it was worth ~2 %.  The peer cannot lap the
// ring: it waits on its local empty barrier, which the leader's multicast commit signals.
//
// What actually bounded this kernel (ncu source view, profiles/r02_dist_f16_v{2,3,4}*.md): the EPILOGUE.  At 10 k
// database rows per query the sorted insertion ran for half of all columns (any of a warp's 32 rows inserting) at
// ~110 instructions a time, one warp per scheduler: 968 us with the tensor pipe 27 % active.  The pending-list epilogue
// below brought the kernel to the MMA/L2 bound (whole call 1.24 -> 0.70 ms).
template <int SUB>
__global__ void __launch_bounds__(192, 1)
gemm2_f16_top16_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                       const Dist1Args g) {
  using C = D1Cfg<SUB>;
  constexpr int STAGES = C::STAGES, STAGE = C::STAGE, TILE_N = C::TILE_N;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int unit0 = blockIdx.x >> 1, unit_stride = gridDim.x >> 1;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE);
  uint64_t* full_bar = bars;                    // leader's are used: count 1 (the leader's arrive.expect_tx for both CTAs)
  uint64_t* empty_bar = bars + STAGES;          // local, count 1 (multicast commit)
  uint64_t* tfull_bar = bars + 2 * STAGES;      // local, count 1 (multicast commit)
  uint64_t* tempty_bar = bars + 2 * STAGES + 2; // leader's are used: count 8 (4 epilogue warps x 2 CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b);
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&tfull_bar[0], 1); mbar_init(&tfull_bar[1], 1);
    mbar_init(&tempty_bar[0], 8); mbar_init(&tempty_bar[1], 8);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc_2sm(tmem_slot, 512);   // both CTAs, same warp id: one allocation spanning the pair
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto decode = [&](int item, int& mp, int& nt0, int& ntn) {
    mp = item / g.items_per_mpair;
    const int sub = item - mp * g.items_per_mpair;
    nt0 = sub * g.nt_per_item;
    ntn = (nt0 + g.nt_per_item <= g.n_tiles) ? g.nt_per_item : (g.n_tiles - nt0);
  };
  const int kiters = g.K / D1_BK;

  if (warp == 0) {
    // TMA producer (both CTAs): convergent warp, one elected lane issues, warp-uniform operands (tc_conv.cu)
    {
      const uint32_t smem_a = warp_uniform(smem_u32(smem));
      const uint32_t bars_a = smem_a + STAGES * STAGE;
      const uint32_t full_a = bars_a, empty_a = bars_a + 8 * STAGES;
      const uint32_t full_c = warp_uniform(mapa_u32(full_a, 0));   // the leader's barriers, shared::cluster addresses
      const int rank_u = (int)warp_uniform(rank);
      int stage = 0; uint32_t phase = 0;
      for (int item = unit0; item < g.total_items; item += unit_stride) {
        int mp, nt0, ntn;
        decode(item, mp, nt0, ntn);
        const int row0 = (int)warp_uniform((uint32_t)((mp * 2 + rank_u) * 128));
        for (int nt = nt0; nt < nt0 + ntn; ++nt) {
          const int col0 = (int)warp_uniform((uint32_t)(nt * TILE_N + rank_u * (D1_BN / 2)));
          for (int kit = 0; kit < kiters; ++kit) {
            const uint32_t sg = warp_uniform((uint32_t)stage);
            mbar_wait_warp_a(empty_a + 8 * sg, phase ^ 1);
            const uint32_t st = smem_a + sg * STAGE;
            const int k0 = (int)warp_uniform((uint32_t)(kit * D1_BK));
            if (elect_one()) {
              if (leader) mbar_arrive_expect_tx_a(full_a + 8 * sg, 2 * STAGE);   // bytes of BOTH CTAs; the peer only loads
              tma_load_2d_2sm_a(st, &tm_a, full_c + 8 * sg, k0, row0);
#pragma unroll
              for (int j = 0; j < SUB; ++j)     // rows beyond the matrix are zero-filled by the TMA unit
                tma_load_2d_2sm_a(st + D1_A_BYTES + j * D1_BH_BYTES, &tm_b, full_c + 8 * sg, k0, col0 + j * D1_BN);
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // whole warp in convergent code, one elected lane issues, ring position / bases warp-uniform: every tcgen05 operand lives in a
    // uniform register (tc_conv.cu, MMA issuer)
    if (warp_uniform(leader ? 1u : 0u)) {
      constexpr uint32_t idesc = umma_idesc_f16_f32(256, D1_BN);
      const uint32_t tmem_u = warp_uniform(tmem_base);
      const uint32_t smem_a = warp_uniform(smem_u32(smem));
      const uint32_t bars_a = smem_a + STAGES * STAGE;
      const uint32_t full_a = bars_a, empty_a = bars_a + 8 * STAGES;
      const uint32_t tfull_a = bars_a + 16 * STAGES, tempty_a = tfull_a + 16;
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      for (int item = unit0; item < g.total_items; item += unit_stride) {
        int mp, nt0, ntn;
        decode(item, mp, nt0, ntn);
        for (int nt = nt0; nt < nt0 + ntn; ++nt, ++it) {
          const uint32_t as = warp_uniform((uint32_t)(C::ACC_BUFS == 2 ? (it & 1) : 0));
          const uint32_t aphase = C::ACC_BUFS == 2 ? ((it >> 1) & 1) : (it & 1);
          mbar_wait_warp_a(tempty_a + 8 * as, aphase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_u + as * D1_BN;
          for (int kit = 0; kit < kiters; ++kit) {
            const uint32_t st = warp_uniform((uint32_t)stage);
            mbar_wait_warp_a(full_a + 8 * st, phase);
            tc_fence_after();
            const uint32_t sa = smem_a + st * STAGE;
            if (elect_one()) {
              const uint64_t a = umma_desc_kmajor_sw128(sa);
#pragma unroll
              for (int k = 0; k < D1_BK / 16; ++k) {
#pragma unroll
                for (int j = 0; j < SUB; ++j) {
                  const uint64_t b = umma_desc_kmajor_sw128(sa + D1_A_BYTES + j * D1_BH_BYTES);
                  umma_bf16_2sm(d_tmem + j * D1_BN, a + (uint64_t)(k * 2), b + (uint64_t)(k * 2), idesc,
                                (kit > 0 || k > 0) ? 1u : 0u);
                }
              }
              umma_commit_2sm_mc_a(empty_a + 8 * st, 0x3);
              if (kit == kiters - 1) umma_commit_2sm_mc_a(tfull_a + 8 * as, 0x3);   // same elected thread as the MMAs
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else {
    // Epilogue: one warp per scheduler, one thread per query row, 256+ accumulator columns per tile.  With a single
    // warp per scheduler every instruction counts (no other warp hides a dependent issue), and ncu's source view of the
    // first version -- a sorted 16-entry insertion behind `if (d < td[15])` for every column -- showed ~85 executed
    // warp instructions per column: whenever ANY of the 32 rows of the warp inserts (half of all columns at 10 k
    // database rows per query) the whole warp walks the ~110-instruction insertion.  Here the per-column work is
    // scale + compare + a predicated 8-byte shared-memory append to a per-row pending list; the lists are merged into
    // the sorted top-16 in a compact loop (trip count = the longest list of the warp) when one could overflow within
    // the next 16 columns, and at the end of every tile.  All 32 rows insert side by side in that loop, so the walk runs
    // once per ~16 appended candidates of the fullest row instead of once per column with a candidate anywhere.
    const int q = warp & 3;
    const int rloc = q * 32 + lane;
    // shared-state-space addresses (the generic pointer arithmetic above makes the compiler emit generic LD/ST)
    const uint32_t bst = smem_u32(smem + STAGES * STAGE + C::BARS) + q * 256;
    const uint32_t pend = smem_u32(smem + STAGES * STAGE + C::BARS + C::BSTAGE) + rloc * 8;   // [slot][128 rows] x 8 B
    int it = 0;
    for (int item = unit0; item < g.total_items; item += unit_stride) {
      int mp, nt0, ntn;
      decode(item, mp, nt0, ntn);
      const int row = (mp * 2 + (int)rank) * 128 + rloc;
      const bool row_ok = row < g.M;
      float an = 0.f, m2sa = 0.f;
      if (row_ok) { const float4 t = __ldg(g.a_aux + row); an = t.x; m2sa = -2.f * t.y; }
      float td[16];
      int ti[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) { td[j] = INFINITY; ti[j] = -1; }
      uint32_t paddr = pend;                               // next free slot of this row's pending list
      float thr = row_ok ? INFINITY : -INFINITY;           // rows beyond the matrix never append
      // merge this row's pending list into the sorted top-16; the 32 rows of the warp run the loop together
      auto merge_pending = [&]() {
        const int cnt = (int)((paddr - pend) >> 10);
        const int longest = __reduce_max_sync(0xffffffffu, cnt);
#pragma unroll 1
        for (int e = 0; e < longest; ++e) {
          if (e < cnt) {
            const float2 v = d1_lds64(pend + e * 1024);
            const float d = v.x;
            if (d < td[15]) {
              const int col = __float_as_int(v.y);
              // Sorted insert without a dependency chain: the slot is counted with 16 independent compares and every
              // entry is rewritten from the OLD values of itself and its left neighbour (descending s).
              int pos = 0;
#pragma unroll
              for (int s = 0; s < 16; ++s) pos += (td[s] <= d) ? 1 : 0;
#pragma unroll
              for (int s = 15; s > 0; --s) {
                const bool shift = s > pos, here = s == pos;
                td[s] = shift ? td[s - 1] : (here ? d : td[s]);
                ti[s] = shift ? ti[s - 1] : (here ? col : ti[s]);
              }
              if (pos == 0) { td[0] = d; ti[0] = col; }
            }
          }
        }
        paddr = pend;
      };
      for (int nt = nt0; nt < nt0 + ntn; ++nt, ++it) {
        const int as = C::ACC_BUFS == 2 ? (it & 1) : 0;
        const uint32_t aphase = C::ACC_BUFS == 2 ? ((it >> 1) & 1) : (it & 1);
        // Shared gate: the work items of one query block scan different database ranges concurrently, each keeping its
        // own top-16.  An element that is not below the 16th-best distance ANY of them has already reached cannot be in
        // the merged top-16, so every item publishes its 16th-best (atomicMin) after each tile and reads the common
        // value before the next: the gate tightens with the UNION of the columns scanned so far.  A stale read only
        // costs efficiency.  Ties at the gate are dropped: the guard's error bound covers them.
        if (row_ok) {
          const unsigned gv = *reinterpret_cast<volatile unsigned*>(g.gate + row);
          if (gv != 0xFFFFFFFFu) thr = fminf(thr, d1_unord(gv));       // 0xFFFFFFFF = "no gate yet" (the memset pattern)
        }
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + as * D1_BN;
#pragma unroll 1
        for (int ch = 0; ch < TILE_N / 32; ++ch) {
          const int col0 = nt * TILE_N + ch * 32;
          if (col0 >= g.n_valid) break;                    // warp-uniform: the rest of the tile is padding
          // The per-column terms {|d|^2, 2^e} of this chunk: ONE coalesced load (lane j fetches column col0 + j) staged
          // in shared memory and read back as warp-wide broadcasts.  A `__ldg(b_aux + col)` per column, as round 1's
          // kernels did, is a chain of 256 dependent L2-latency loads per tile.
          float2 mine = make_float2(INFINITY, 0.f);        // padding columns: +inf, never below the threshold
          if (col0 + lane < g.n_valid) { const float4 t = __ldg(g.b_aux + col0 + lane); mine = make_float2(t.x, t.y); }
          uint32_t raw[32];
          tmem_ld_32x32(t_row + ch * 32, raw);
          __syncwarp();                                    // the previous chunk's broadcast reads are done
          d1_sts64(bst + lane * 8, mine.x, mine.y);
          __syncwarp();
          tmem_ld_wait();
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (__any_sync(0xffffffffu, paddr > pend + (D1_PEND - 16) * 1024)) {   // could overflow within 16 columns: merge first
              merge_pending();
              thr = fminf(thr, td[15]);
            }
            float2 c[16];
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) c[jj] = d1_lds64(bst + (h * 16 + jj) * 8);   // issued back to back
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const int j = h * 16 + jj;
              const float d = fmaf(m2sa * c[jj].y, __uint_as_float(raw[j]), an + c[jj].x);
              if (d < thr) { d1_sts64(paddr, d, __int_as_float(col0 + j)); paddr += 1024; }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (leader) mbar_arrive(&tempty_bar[as]);
          else mbar_arrive_remote(mapa_u32(smem_u32(&tempty_bar[as]), 0));
        }
        merge_pending();                                   // after the accumulator is released: overlaps the next main loop
        if (row_ok && td[15] < thr) {
          thr = td[15];
          atomicMin(g.gate + row, d1_ord(thr));
        }
      }
      if (row_ok) {
        const int sub = item % g.items_per_mpair;
        float4* od = reinterpret_cast<float4*>(g.cand_d + ((long long)sub * g.M + row) * 16);
        int4* oi = reinterpret_cast<int4*>(g.cand_i + ((long long)sub * g.M + row) * 16);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          od[j] = make_float4(td[4 * j], td[4 * j + 1], td[4 * j + 2], td[4 * j + 3]);
          oi[j] = make_int4(ti[4 * j], ti[4 * j + 1], ti[4 * j + 2], ti[4 * j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// ---- 3. merge + exact re-scoring + sort + guard ---------------------------------------------------------

// exact distance of query row (staged at qrow) and database row ci, one warp; same arithmetic as round 1's
// rescore_sort_kernel: lane-strided float4 FMAs, xor-shuffle tree, fmaf(-2, dot, |q|^2 + |d|^2)
__device__ __forceinline__ float d1_exact(const float* qrow, const float* __restrict__ dp, int d, int lane, float an,
                                          float bn) {
  float acc = 0.f;
#pragma unroll 2
  for (int i = lane * 4; i < d; i += 128) {   // unrolled: several row loads in flight (the FMA order is unchanged)
    const float4 a = *reinterpret_cast<const float4*>(qrow + i);
    const float4 b = __ldg(reinterpret_cast<const float4*>(dp + i));
    acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc);
    acc = fmaf(a.z, b.z, acc); acc = fmaf(a.w, b.w, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return fmaf(-2.f, acc, an + bn);
}

struct FinishArgs {
  const float* q; const float* db;
  const float4* q_aux; const float4* db_aux;
  const float* db_max2;          // {max |x - x'|, max |x|^2} over the database rows
  const float* cand_d; const int* cand_i;
  int m, d, runs, k_out, n_valid;
  long long idx_base;
  float* out_dist; long long* out_idx;
  int* flag_count; int* flag_list;
};

__global__ void __launch_bounds__(128)
dist_finish_kernel(const FinishArgs g) {
  extern __shared__ __align__(16) float qs[];   // [d] when it fits
  __shared__ unsigned long long keys[128];
  __shared__ unsigned long long skeys[128];
  const long long row = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int d = g.d;
  const bool staged = d <= 16384;
  if (staged) {
    for (int i = threadIdx.x * 4; i < d; i += 128 * 4)
      *reinterpret_cast<float4*>(qs + i) = __ldg(reinterpret_cast<const float4*>(g.q + row * d + i));
  }
  const float* qrow = staged ? qs : (g.q + row * d);
  // ---- merge: the 16 best screened candidates of runs x 16 (runs <= 8) ----
  const int total = g.runs * 16;
  {
    unsigned long long key = ~0ull;
    if ((int)threadIdx.x < total) {
      const int r = threadIdx.x >> 4, j = threadIdx.x & 15;
      const long long src = ((long long)r * g.m + row) * 16 + j;
      const int ci = g.cand_i[src];
      if (ci >= 0) key = ((unsigned long long)d1_ord(g.cand_d[src]) << 32) | (unsigned)ci;
    }
    skeys[threadIdx.x] = key;
  }
  for (int size = 2; size <= 128; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      if (threadIdx.x < 64) {
        const int i = threadIdx.x;
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool up = ((lo & size) == 0);
        const unsigned long long a = skeys[lo], b = skeys[hi];
        if ((a > b) == up) { skeys[lo] = b; skeys[hi] = a; }
      }
    }
  }
  __syncthreads();
  const float4 qa = __ldg(g.q_aux + row);
  // ---- exact fp32 re-scoring of the 16 survivors ----
  for (int c = wid; c < 128; c += 4) {
    unsigned long long key = ~0ull;
    if (c < 16) {
      const unsigned long long sk = skeys[c];
      if (sk != ~0ull) {
        const long long ci = (long long)(uint32_t)(sk & 0xffffffffu);
        const float dist = d1_exact(qrow, g.db + ci * d, d, lane, qa.x, __ldg(&g.db_aux[ci].x));
        key = ((unsigned long long)d1_ord(dist) << 32) | (unsigned)ci;
      }
    }
    if (lane == 0) keys[c] = key;
  }
  for (int size = 2; size <= 16; size <<= 1) {          // only keys[0..15] can be valid
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      if (threadIdx.x < 8) {
        const int i = threadIdx.x;
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool up = ((lo & size) == 0);
        const unsigned long long a = keys[lo], b = keys[hi];
        if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
      }
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < g.k_out) {
    const unsigned long long key = keys[threadIdx.x];
    if (key == ~0ull) {
      g.out_dist[row * g.k_out + threadIdx.x] = INFINITY;
      g.out_idx[row * g.k_out + threadIdx.x] = -1;
    } else {
      g.out_dist[row * g.k_out + threadIdx.x] = d1_unord((uint32_t)(key >> 32));
      g.out_idx[row * g.k_out + threadIdx.x] = g.idx_base + (long long)(uint32_t)(key & 0xffffffffu);
    }
  }
  // ---- guard ----
  if (threadIdx.x == 0 && g.n_valid > 16) {              // with <= 16 rows everything was re-scored
    const unsigned long long s16k = skeys[15];
    const int kk = g.k_out < 16 ? g.k_out : 16;
    const unsigned long long ek = keys[kk - 1];
    bool flag = (s16k == ~0ull) || (ek == ~0ull);        // cannot happen with n_valid > 16; be safe
    if (!flag) {
      const float s16 = d1_unord((uint32_t)(s16k >> 32)), e_k = d1_unord((uint32_t)(ek >> 32));
      const float bound = screen_guard_bound(qa.x, qa.z, __ldg(g.db_max2 + 1), __ldg(g.db_max2), d, d / 16, 0.f);
      flag = !(s16 - bound > e_k);                       // also catches NaN
    }
    if (flag) g.flag_list[atomicAdd(g.flag_count, 1)] = (int)row;
  }
}

// ---- 4. exact brute force for the listed queries ----------------------------------------------------
constexpr int DX_KMAX = 128;
constexpr int DX_G = 8;                 // listed queries per work item of the exact brute force
constexpr int DX_QSTAGE = 32768;        // floats of staged queries per work item (128 KiB)
// database rows per work item: at most 64 items per listed query (bounds the scratch), at least 128 rows, so that a
// few listed queries still spread over all SMs (each warp's rows are a chain of L2 latencies)
static int dx_chunk_rows(int n_valid) {
  const int c = cdiv(cdiv(n_valid > 0 ? n_valid : 1, 64), 64) * 64;
  return c > 128 ? c : 128;
}

struct ExactArgs {
  const float* q; const float* db;
  const float* qn; const float* dbn;   // |x|^2, read with a stride (4 for the float4 aux of this file)
  int qn_stride, dbn_stride;
  int m, d, n_valid, k, chunk, nchunks, group;
  long long idx_base;
  const int* flag_count; const int* flag_list;
  unsigned long long* scratch;   // [m][nchunks][k] keys
  float* out_dist; long long* out_idx;
};

// number of keys below `key` in nl sorted lists of length k (stride k); keys are distinct (they hold the row)
__device__ __forceinline__ int dx_rank(const unsigned long long* lists, int nl, int k, unsigned long long key) {
  int rank = 0;
  for (int l = 0; l < nl && rank < k; ++l) {
    const unsigned long long* L = lists + (long long)l * k;
    int lo = 0, hi = k;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (L[mid] < key) lo = mid + 1; else hi = mid; }
    rank += lo;
  }
  return rank;
}

// work item = (chunk c of the database, group of up to g.group listed queries): every database row of the chunk is read
// once for the whole group (one warp per row, the group's queries staged in shared memory), so a handful of listed
// queries costs about one pass over the database.  Per query and warp a sorted list of the k best keys; at the end of
// the item the 8 lists of each query are merged by rank into scratch.  The dot products use d1_exact's arithmetic
// (lane-strided FMAs in the same order, the same xor tree), so the distances are bit-identical to the re-scoring.
__global__ void __launch_bounds__(256)
dist_exact_chunk_kernel(const ExactArgs g) {
  extern __shared__ __align__(16) float dsm[];   // [group][d] queries when staged | [group][8 warps][k] keys
  const int G = g.group, k = g.k, d = g.d;
  const bool staged = (long long)G * d <= DX_QSTAGE;
  unsigned long long* lists = reinterpret_cast<unsigned long long*>(dsm + (staged ? G * d : 0));
  const int count = *g.flag_count;
  const int ngroups = (count + G - 1) / G;
  const int items = ngroups * g.nchunks;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    const int c = item / ngroups, grp = item - c * ngroups;   // the groups of one chunk run side by side: L2 hits
    const int f0 = grp * G, gn = min(G, count - f0);
    __syncthreads();
    if (staged)
      for (int t = 0; t < gn; ++t) {
        const long long row = g.flag_list[f0 + t];
        for (int i = threadIdx.x * 4; i < d; i += 256 * 4)
          *reinterpret_cast<float4*>(dsm + t * d + i) = __ldg(reinterpret_cast<const float4*>(g.q + row * d + i));
      }
    for (int s = threadIdx.x; s < G * 8 * k; s += 256) lists[s] = ~0ull;
    __syncthreads();
    const float* qp[DX_G];
    float an[DX_G];
#pragma unroll
    for (int t = 0; t < DX_G; ++t) {
      const long long row = t < gn ? g.flag_list[f0 + t] : 0;
      qp[t] = staged ? dsm + t * d : g.q + row * d;
      an[t] = t < gn ? __ldg(g.qn + row * g.qn_stride) : 0.f;
    }
    const int j0 = c * g.chunk, j1 = min(g.n_valid, j0 + g.chunk);
    for (int j = j0 + wid; j < j1; j += 8) {
      const float* dp = g.db + (long long)j * d;
      float acc[DX_G];
#pragma unroll
      for (int t = 0; t < DX_G; ++t) acc[t] = 0.f;
#pragma unroll 2
      for (int i = lane * 4; i < d; i += 128) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(dp + i));
#pragma unroll
        for (int t = 0; t < DX_G; ++t) {
          if (t < gn) {
            const float4 a = *reinterpret_cast<const float4*>(qp[t] + i);
            acc[t] = fmaf(a.x, b.x, acc[t]); acc[t] = fmaf(a.y, b.y, acc[t]);
            acc[t] = fmaf(a.z, b.z, acc[t]); acc[t] = fmaf(a.w, b.w, acc[t]);
          }
        }
      }
      const float bn = __ldg(g.dbn + (long long)j * g.dbn_stride);
#pragma unroll
      for (int t = 0; t < DX_G; ++t) {
        if (t >= gn) break;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[t] += __shfl_xor_sync(0xffffffffu, acc[t], o);
        const float dist = fmaf(-2.f, acc[t], an[t] + bn);
        const unsigned long long key = ((unsigned long long)d1_ord(dist) << 32) | (unsigned)j;
        unsigned long long* L = lists + (t * 8 + wid) * k;
        if (key < L[k - 1]) {                  // warp-uniform: sorted insert, each lane moves the slots it owns
          unsigned long long left[DX_KMAX / 32], cur[DX_KMAX / 32];
#pragma unroll
          for (int u = 0; u < DX_KMAX / 32; ++u) {
            const int s = lane + 32 * u;
            left[u] = (s > 0 && s < k) ? L[s - 1] : 0ull;
            cur[u] = s < k ? L[s] : 0ull;
          }
          __syncwarp();
#pragma unroll
          for (int u = 0; u < DX_KMAX / 32; ++u) {
            const int s = lane + 32 * u;
            if (s < k) {
              if (s > 0 && left[u] > key) L[s] = left[u];
              else if (cur[u] > key) L[s] = key;
            }
          }
          __syncwarp();
        }
      }
    }
    __syncthreads();
    // per query: the k smallest of its 8 sorted lists, placed by rank
    for (int t = 0; t < gn; ++t) {
      const long long row = g.flag_list[f0 + t];
      unsigned long long* out = g.scratch + ((long long)row * g.nchunks + c) * k;
      for (int s = threadIdx.x; s < k; s += 256) out[s] = ~0ull;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < gn * 8 * k; i += 256) {
      const unsigned long long key = lists[i];
      if (key == ~0ull) continue;
      const int t = i / (8 * k);
      const int rank = dx_rank(lists + t * 8 * k, 8, k, key);
      if (rank < k) g.scratch[((long long)g.flag_list[f0 + t] * g.nchunks + c) * k + rank] = key;
    }
  }
}

// one block per listed query: the k smallest of its nchunks sorted lists (staged in shared memory), placed by rank
__global__ void __launch_bounds__(128)
dist_exact_merge_kernel(const ExactArgs g) {
  extern __shared__ unsigned long long src[];   // [nchunks][k]
  const int count = *g.flag_count;
  for (int f = blockIdx.x; f < count; f += gridDim.x) {
    const long long row = g.flag_list[f];
    __syncthreads();
    for (int i = threadIdx.x; i < g.nchunks * g.k; i += blockDim.x) src[i] = g.scratch[row * g.nchunks * g.k + i];
    for (int t = threadIdx.x; t < g.k; t += blockDim.x) {
      g.out_dist[row * g.k + t] = INFINITY;
      g.out_idx[row * g.k + t] = -1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < g.nchunks * g.k; i += blockDim.x) {
      const unsigned long long key = src[i];
      if (key == ~0ull) continue;
      const int rank = dx_rank(src, g.nchunks, g.k, key);
      if (rank < g.k) {
        g.out_dist[row * g.k + rank] = d1_unord((uint32_t)(key >> 32));
        g.out_idx[row * g.k + rank] = g.idx_base + (long long)(uint32_t)(key & 0xffffffffu);
      }
    }
    __syncthreads();
  }
}

size_t dist_exact_scratch_bytes(int m, int n_valid, int k) {
  const int nchunks = cdiv(n_valid > 0 ? n_valid : 1, 128);    // >= the chunks of any n_valid' <= n_valid
  return (size_t)m * (nchunks < 64 ? nchunks : 64) * k * sizeof(unsigned long long);
}

// exact fp32 brute force of the queries in flag_list[0 .. *flag_count): no host round trip, the kernels size their
// work from the device counter and exit at once when nothing is listed.  scratch: dist_exact_scratch_bytes(m, n_valid, k)
int launch_dist_exact_fallback(const float* q, const float* qn, int qn_stride, int m, const float* db, const float* dbn,
                               int dbn_stride, int n_valid, int d, int k, long long idx_base, const int* flag_count,
                               const int* flag_list, unsigned long long* scratch, float* out_dist, long long* out_idx,
                               cudaStream_t s) {
  IBL_REQUIRE(k >= 1 && k <= DX_KMAX && d % 4 == 0, "exact fallback: 1 <= k <= 128, d % 4 == 0");
  static DeviceOnce attr_done;   // the attribute is per device
  if (!attr_done.done()) {
    IBL_CUDA_OK(cudaFuncSetAttribute(dist_exact_chunk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     DX_QSTAGE * 4 + DX_G * 8 * DX_KMAX * 8));
    IBL_CUDA_OK(cudaFuncSetAttribute(dist_exact_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    attr_done.mark();
  }
  ExactArgs x{};
  x.q = q; x.db = db; x.qn = qn; x.dbn = dbn; x.qn_stride = qn_stride; x.dbn_stride = dbn_stride;
  x.m = m; x.d = d; x.n_valid = n_valid; x.k = k;
  x.group = d <= DX_QSTAGE / DX_G ? DX_G : (d <= DX_QSTAGE ? DX_QSTAGE / d : 1);
  x.chunk = dx_chunk_rows(n_valid);
  x.nchunks = cdiv(n_valid > 0 ? n_valid : 1, x.chunk); x.idx_base = idx_base; x.flag_count = flag_count;
  x.flag_list = flag_list; x.scratch = scratch; x.out_dist = out_dist; x.out_idx = out_idx;
  const size_t csm = ((long long)x.group * d <= DX_QSTAGE ? (size_t)x.group * d * 4 : 0) + (size_t)x.group * 8 * k * 8;
  dist_exact_chunk_kernel<<<device_sm_count() * 2, 256, csm, s>>>(x);
  dist_exact_merge_kernel<<<128, 128, (size_t)x.nchunks * k * sizeof(unsigned long long), s>>>(x);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}

// ---- host -----------------------------------------------------------------------------------------
static int pick_runs1(int m_pairs, int n_tiles) {
  const int G = device_sm_count() / 2;
  int best = 1;
  double best_eff = -1.0;
  for (int r = 1; r <= n_tiles && r <= 8; ++r) {          // dist_finish_kernel merges up to 8 x 16 candidates
    const int per = cdiv(n_tiles, r), runs = cdiv(n_tiles, per);
    const long long total = (long long)m_pairs * runs, waves = (total + G - 1) / G;
    const double eff = (double)m_pairs * n_tiles / ((double)waves * G * per);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = runs; }
  }
  return best;
}

size_t dist1_workspace_bytes(int m, int n, int d, size_t* off /*[8]*/) {
  // layout: q plane | db plane | q aux | db aux | db max2 + flag count (256 B) | flag list | cand_d | cand_i | scratch
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at = o; o += (bytes + 255) & ~(size_t)255; return at; };
  off[0] = take((size_t)m * d * 2);
  off[1] = take((size_t)n * d * 2);
  off[2] = take((size_t)m * 16);
  off[3] = take((size_t)n * 16);
  off[4] = take(256);
  off[5] = take((size_t)m * 4 + (size_t)m * 4);     // guard list | shared gates
  off[6] = take((size_t)8 * m * 16 * 4);
  off[7] = take((size_t)8 * m * 16 * 4);
  off[8] = take(dist_exact_scratch_bytes(m, n, 16));
  return o;
}

// q [m,d], db [n,d] fp32 (device); n_valid <= n; k <= 12.  ws: dist1_workspace_bytes(m, n, d).
int launch_dist_topk_1pass(const float* q, int m, const float* db, int n, int n_valid, int d, int k, long long idx_base,
                           void* ws, float* out_dist, long long* out_idx, uint64_t* launches, cudaStream_t s) {
  IBL_REQUIRE(d % 64 == 0 && k >= 1 && k <= 12 && n_valid >= 1, "1-pass distance: d % 64 == 0, 1 <= k <= 12");
  size_t off[9];
  dist1_workspace_bytes(m, n, d, off);
  uint8_t* w = reinterpret_cast<uint8_t*>(ws);
  __half* qp = reinterpret_cast<__half*>(w + off[0]);
  __half* dp = reinterpret_cast<__half*>(w + off[1]);
  float4* qa = reinterpret_cast<float4*>(w + off[2]);
  float4* da = reinterpret_cast<float4*>(w + off[3]);
  float* dmax2 = reinterpret_cast<float*>(w + off[4]);
  int* fcount = reinterpret_cast<int*>(w + off[4] + 16);
  int* flist = reinterpret_cast<int*>(w + off[5]);
  unsigned* gate = reinterpret_cast<unsigned*>(w + off[5] + (size_t)m * 4);
  float* cd = reinterpret_cast<float*>(w + off[6]);
  int* ci = reinterpret_cast<int*>(w + off[7]);
  unsigned long long* scratch = reinterpret_cast<unsigned long long*>(w + off[8]);

  IBL_CUDA_OK(cudaMemsetAsync(w + off[4], 0, 32, s));      // db max2 (2 floats) | flag count at +16
  IBL_CUDA_OK(cudaMemsetAsync(gate, 0xFF, (size_t)m * 4, s));      // orderable +max: no gate yet
  rows_f16_kernel<<<m, 256, 0, s>>>(q, d, qp, qa);
  rows_f16_kernel<<<n, 256, 0, s>>>(db, d, dp, da);
  IBL_CUDA_OK(cudaGetLastError());
  IBL_RET(launch_dist_colmax(&da->x, &da->z, 4, n_valid, dmax2, s));

  CUtensorMap ma, mb;
  {
    uint64_t dims_a[2] = {(uint64_t)d, (uint64_t)m}, dims_b[2] = {(uint64_t)d, (uint64_t)n};
    uint64_t str[1] = {(uint64_t)d * 2};
    uint32_t box[2] = {64, 128};
    IBL_RET(make_tmap(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, qp, dims_a, str, box));
    IBL_RET(make_tmap(&mb, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, dp, dims_b, str, box));
  }
  // default: 256 x 256 tiles with two overlapped accumulators; IBL_DIST_BN=512 selects the 256 x 512 tile (variant tests)
  static const int tile_env = [] { const char* v = getenv("IBL_DIST_BN"); return v ? atoi(v) : 256; }();
  const int SUBn = tile_env == 256 ? 1 : 2;
  Dist1Args g{};
  g.M = m; g.N = n; g.K = d;
  g.n_tiles = cdiv(n_valid, D1_BN * SUBn);
  const int m_pairs = cdiv(cdiv(m, 128), 2);
  const int runs = pick_runs1(m_pairs, g.n_tiles);
  g.nt_per_item = cdiv(g.n_tiles, runs);
  g.items_per_mpair = cdiv(g.n_tiles, g.nt_per_item);
  g.total_items = m_pairs * g.items_per_mpair;
  g.n_valid = n_valid;
  g.a_aux = qa; g.b_aux = da; g.cand_d = cd; g.cand_i = ci; g.gate = gate;
  static DeviceOnce attr_done;   // the attributes are per device
  if (!attr_done.done()) {
    IBL_CUDA_OK(cudaFuncSetAttribute(gemm2_f16_top16_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, D1Cfg<1>::SMEM));
    IBL_CUDA_OK(cudaFuncSetAttribute(gemm2_f16_top16_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, D1Cfg<2>::SMEM));
    IBL_CUDA_OK(cudaFuncSetAttribute(dist_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    attr_done.mark();
  }
  const int pairs = device_sm_count() / 2;
  const int units = g.total_items < pairs ? g.total_items : pairs;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * units);
  cfg.blockDim = dim3(192);
  cfg.dynamicSmemBytes = SUBn == 1 ? D1Cfg<1>::SMEM : D1Cfg<2>::SMEM;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (SUBn == 1) IBL_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm2_f16_top16_kernel<1>, ma, mb, g));
  else IBL_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm2_f16_top16_kernel<2>, ma, mb, g));

  FinishArgs f{};
  f.q = q; f.db = db; f.q_aux = qa; f.db_aux = da; f.db_max2 = dmax2; f.cand_d = cd; f.cand_i = ci;
  f.m = m; f.d = d; f.runs = g.items_per_mpair; f.k_out = k; f.n_valid = n_valid; f.idx_base = idx_base;
  f.out_dist = out_dist; f.out_idx = out_idx; f.flag_count = fcount; f.flag_list = flist;
  const size_t qsm = d <= 16384 ? (size_t)d * sizeof(float) : 16;
  dist_finish_kernel<<<m, 128, qsm, s>>>(f);
  IBL_CUDA_OK(cudaGetLastError());

  IBL_RET(launch_dist_exact_fallback(q, &qa->x, 4, m, db, &da->x, 4, n_valid, d, k, idx_base, fcount, flist, scratch,
                                     out_dist, out_idx, s));
  if (launches) *launches += 7;
  return IBL_OK;
}

// device address of the guard's counter of listed queries in a workspace of dist1_workspace_bytes(m, n, d)
int* dist1_flag_count(void* ws, int m, int n, int d) {
  size_t off[9];
  dist1_workspace_bytes(m, n, d, off);
  return reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(ws) + off[4] + 16);
}

}  // namespace ibl
