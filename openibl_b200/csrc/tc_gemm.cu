// tcgen05 "NT" GEMM with fp32-grade operands:  acc[i,j] = sum_k A[i,k] * B[j,k]
// A [M,K] and B [N,K] are row-major fp32 matrices carried as bf16 hi/lo planes; every K-chunk
// issues A_lo.B_hi + A_hi.B_lo + A_hi.B_hi into an fp32 TMEM accumulator (see tc_conv.cu).
//
// Used for
//   * stage (iii-b) query x database L2 distance (reference ibl/evaluators.py:127-129), with
//       EPI_TOP16  a per-query running top-16 kept in registers across the CTA's sweep over its
//                  database range -- the [m,n] matrix is never written (replaces np.argsort, :143)
//       EPI_DENSE  the dense matrix, for callers that need it (netvlad_img.py:78) and for k > 12
//   * stage (iii-a) PCA-whitening GEMM (netvlad.py:105-108 / pca.py:117-121), split along K:
//       EPI_PARTIAL partial[z][j][i]
//
// Work item = (row tile of 128, a run of column tiles, a run of K chunks); items are dealt
// round-robin to a persistent grid.  Warp roles as in tc_conv.cu.
#include <stdlib.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace ibl {

using namespace tc;

enum { EPI_TOP16 = 0, EPI_DENSE = 1, EPI_PARTIAL = 2 };

struct GemmTcArgs {
  int M, N, K;
  int n_tiles;          // ceil(N / BN)
  int nt_per_item;      // column tiles per item
  int items_per_mtile;  // column-runs per row tile (EPI_TOP16/DENSE) or K-splits (EPI_PARTIAL)
  int kit_per_item;     // K chunks (of 64) per item
  int total_items;
  int n_valid;          // columns >= n_valid are ignored
  const float* an;      // |A_i|^2   (distance epilogues)
  const float* bn;      // |B_j|^2
  float* out;           // DENSE: [M, ld_out];  PARTIAL: [splits][N][M]
  long long ld_out;
  float* cand_d;        // TOP16: [items_per_mtile][M][16]
  long long* cand_i;
};

constexpr int GT_BM = 128;

// MC = true: the grid is launched as clusters of two CTAs that walk the same column tiles with adjacent
// row tiles.  Each CTA fetches only half of every B tile and TMA-multicasts it into both CTAs' shared
// memory, so the per-SM L2->SM operand traffic drops from A+B to A+B/2 per K chunk (the kernel is bound by
// the L2 latency x bandwidth product against the ~190 KiB of stages that fit, profiles/r01_dist_tc.md).
// A stage may be refilled only when BOTH CTAs' MMAs have released it: the MMA warp's tcgen05.commit is
// multicast to the empty barrier of both CTAs (arrival count 2).
template <int BN, int STAGES, int EPI, bool MC, int BK = 64>
__global__ void __launch_bounds__(192, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tm_ahi, const __grid_constant__ CUtensorMap tm_alo,
               const __grid_constant__ CUtensorMap tm_bhi, const __grid_constant__ CUtensorMap tm_blo,
               const GemmTcArgs g) {
  constexpr int CL = MC ? 2 : 1;
  uint32_t cta_rank = 0;
  if (MC) asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta_rank));
  const int unit0 = blockIdx.x / CL, unit_stride = gridDim.x / CL;   // a unit = one CTA or one CTA pair
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // BK = 64: 128-byte rows, 128B swizzle.  BK = 32: 64-byte rows, 64B swizzle -- half-size stages, so a
  // 256-column tile still gets a 4-deep pipeline.
  constexpr int A_BYTES = GT_BM * BK * 2;
  constexpr int B_BYTES = BN * BK * 2;
  constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tfull_bar = bars + 2 * STAGES;
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  constexpr uint32_t TMEM_COLS = (2 * BN < 32) ? 32 : 2 * BN;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_ahi);
    tma_prefetch_desc(&tm_alo);
    tma_prefetch_desc(&tm_bhi);
    tma_prefetch_desc(&tm_blo);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], CL);
    }
    mbar_init(&tfull_bar[0], 1);
    mbar_init(&tfull_bar[1], 1);
    mbar_init(&tempty_bar[0], 4);
    mbar_init(&tempty_bar[1], 4);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  if (MC) cluster_sync_all();     // the peer's barriers exist before anything is multicast into this CTA
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // item -> (row tile, first column tile, #column tiles, first K chunk, #K chunks); with MC an item is a
  // pair of adjacent row tiles and this CTA takes the one matching its rank in the cluster
  auto decode = [&](int item, int& mt, int& nt0, int& ntn, int& k0, int& kn) {
    mt = item / g.items_per_mtile;
    const int sub = item - mt * g.items_per_mtile;
    mt = mt * CL + (int)cta_rank;
    if (EPI == EPI_PARTIAL) {
      nt0 = 0; ntn = g.n_tiles;
      k0 = sub * g.kit_per_item;
      const int ktot = g.K / BK;
      kn = (k0 + g.kit_per_item <= ktot) ? g.kit_per_item : (ktot - k0);
    } else {
      nt0 = sub * g.nt_per_item;
      ntn = (nt0 + g.nt_per_item <= g.n_tiles) ? g.nt_per_item : (g.n_tiles - nt0);
      k0 = 0; kn = g.K / BK;
    }
  };

  if (warp == 0) {
    // TMA producer: convergent warp, one elected lane issues, warp-uniform operands (tc_conv.cu explains why)
    {
      const uint32_t smem_a = warp_uniform(smem_u32(smem));
      const uint32_t bars_a = smem_a + STAGES * STAGE_BYTES;
      const uint32_t full_a = bars_a, empty_a = bars_a + 8 * STAGES;
      const int rank_u = (int)warp_uniform(cta_rank);
      int stage = 0;
      uint32_t phase = 0;
      for (int item = unit0; item < g.total_items; item += unit_stride) {
        int mt, nt0, ntn, k0, kn;
        decode(item, mt, nt0, ntn, k0, kn);
        const int row0 = (int)warp_uniform((uint32_t)(mt * GT_BM));
        for (int nt = nt0; nt < nt0 + ntn; ++nt) {
          const int col0 = (int)warp_uniform((uint32_t)(nt * BN));
          for (int kit = k0; kit < k0 + kn; ++kit) {
            const uint32_t sg = warp_uniform((uint32_t)stage);
            mbar_wait_warp_a(empty_a + 8 * sg, phase ^ 1);
            const uint32_t st = smem_a + sg * STAGE_BYTES, fb = full_a + 8 * sg;
            const int kc = (int)warp_uniform((uint32_t)(kit * BK));
            if (elect_one()) {
              mbar_arrive_expect_tx_a(fb, STAGE_BYTES);
              tma_load_2d_a(st, &tm_ahi, fb, kc, row0);
              tma_load_2d_a(st + A_BYTES, &tm_alo, fb, kc, row0);
              if (MC) {   // this CTA's half of the B tile, delivered to both CTAs of the pair
                constexpr int HB = B_BYTES / 2;
                tma_load_2d_mc_a(st + 2 * A_BYTES + rank_u * HB, &tm_bhi, fb, kc, col0 + rank_u * (BN / 2), 0x3);
                tma_load_2d_mc_a(st + 2 * A_BYTES + B_BYTES + rank_u * HB, &tm_blo, fb, kc, col0 + rank_u * (BN / 2), 0x3);
              } else {
                tma_load_2d_a(st + 2 * A_BYTES, &tm_bhi, fb, kc, col0);
                tma_load_2d_a(st + 2 * A_BYTES + B_BYTES, &tm_blo, fb, kc, col0);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // MMA issuer: convergent warp, one elected lane issues, ring position and bases warp-uniform (tc_conv.cu explains why)
    {
      constexpr uint32_t idesc = umma_idesc_bf16_f32(GT_BM, BN);
      const uint32_t tmem_u = warp_uniform(tmem_base);
      const uint32_t smem_a = warp_uniform(smem_u32(smem));
      const uint32_t bars_a = smem_a + STAGES * STAGE_BYTES;
      const uint32_t full_a = bars_a, empty_a = bars_a + 8 * STAGES;
      const uint32_t tfull_a = bars_a + 16 * STAGES, tempty_a = tfull_a + 16;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int item = unit0; item < g.total_items; item += unit_stride) {
        int mt, nt0, ntn, k0, kn;
        decode(item, mt, nt0, ntn, k0, kn);
        for (int nt = nt0; nt < nt0 + ntn; ++nt, ++it) {
          const uint32_t as = warp_uniform((uint32_t)(it & 1));
          const uint32_t aphase = (it >> 1) & 1;
          mbar_wait_warp_a(tempty_a + 8 * as, aphase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_u + as * BN;
          for (int kit = 0; kit < kn; ++kit) {
            const uint32_t sg = warp_uniform((uint32_t)stage);
            mbar_wait_warp_a(full_a + 8 * sg, phase);
            tc_fence_after();
            const uint32_t sa = smem_a + sg * STAGE_BYTES;
            if (elect_one()) {
              const uint64_t a_hi = umma_desc_kmajor<BK>(sa);
              const uint64_t a_lo = umma_desc_kmajor<BK>(sa + A_BYTES);
              const uint64_t b_hi = umma_desc_kmajor<BK>(sa + 2 * A_BYTES);
              const uint64_t b_lo = umma_desc_kmajor<BK>(sa + 2 * A_BYTES + B_BYTES);
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                const uint64_t ko = (uint64_t)(k * 2);
                umma_bf16(d_tmem, a_lo + ko, b_hi + ko, idesc, (kit > 0 || k > 0) ? 1u : 0u);
                umma_bf16(d_tmem, a_hi + ko, b_lo + ko, idesc, 1u);
                umma_bf16(d_tmem, a_hi + ko, b_hi + ko, idesc, 1u);
              }
              if (MC) umma_commit_mc_a(empty_a + 8 * sg, 0x3);   // frees the slot in both CTAs of the pair
              else umma_commit_a(empty_a + 8 * sg);
              if (kit == kn - 1) umma_commit_a(tfull_a + 8 * as);   // same elected thread as the MMAs it covers
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else {
    const int q = warp & 3;
    const int rloc = q * 32 + lane;
    int it = 0;
    for (int item = unit0; item < g.total_items; item += unit_stride) {
      int mt, nt0, ntn, k0, kn;
      decode(item, mt, nt0, ntn, k0, kn);
      const int row = mt * GT_BM + rloc;
      const bool row_ok = row < g.M;
      float an = 0.f;
      if (EPI != EPI_PARTIAL && row_ok) an = __ldg(g.an + row);
      float td[16];
      int ti[16];
      if (EPI == EPI_TOP16) {
#pragma unroll
        for (int j = 0; j < 16; ++j) { td[j] = INFINITY; ti[j] = -1; }
      }
      for (int nt = nt0; nt < nt0 + ntn; ++nt, ++it) {
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&tfull_bar[as], aphase);
        tc_fence_after();
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + as * BN;
#pragma unroll 1
        for (int ch = 0; ch < BN / 32; ++ch) {
          uint32_t raw[32];
          tmem_ld_32x32(t_row + ch * 32, raw);
          tmem_ld_wait();
          const int col0 = nt * BN + ch * 32;
          if (EPI == EPI_PARTIAL) {
            const int split = item % g.items_per_mtile;
            float* o = g.out + ((long long)split * g.N) * g.M;
            if (row_ok) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < g.N) o[(long long)(col0 + j) * g.M + row] = __uint_as_float(raw[j]);
            }
          } else if (EPI == EPI_DENSE) {
            if (row_ok) {
              float* o = g.out + (long long)row * g.ld_out + col0;
              if (col0 + 32 <= g.n_valid && (g.ld_out & 3) == 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 b = __ldg(reinterpret_cast<const float4*>(g.bn + col0) + j);
                  float4 v;
                  v.x = fmaf(-2.f, __uint_as_float(raw[4 * j + 0]), an + b.x);
                  v.y = fmaf(-2.f, __uint_as_float(raw[4 * j + 1]), an + b.y);
                  v.z = fmaf(-2.f, __uint_as_float(raw[4 * j + 2]), an + b.z);
                  v.w = fmaf(-2.f, __uint_as_float(raw[4 * j + 3]), an + b.w);
                  reinterpret_cast<float4*>(o)[j] = v;
                }
              } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                  if (col0 + j < g.n_valid)
                    o[j] = fmaf(-2.f, __uint_as_float(raw[j]), an + __ldg(g.bn + col0 + j));
              }
            }
          } else {  // EPI_TOP16
            // one coalesced load of the chunk's |d|^2 terms + shuffles, chain-free sorted insert (see tc_dist1.cu)
            const float bmine = (col0 + (int)(threadIdx.x & 31) < g.n_valid) ? __ldg(g.bn + col0 + (threadIdx.x & 31)) : INFINITY;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int col = col0 + j;
              const float d = fmaf(-2.f, __uint_as_float(raw[j]), an + __shfl_sync(0xffffffffu, bmine, j));
              if (d < td[15]) {
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
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty_bar[as]);
      }
      if (EPI == EPI_TOP16 && row_ok) {
        const int sub = item % g.items_per_mtile;
        float* od = g.cand_d + ((long long)sub * g.M + row) * 16;
        long long* oi = g.cand_i + ((long long)sub * g.M + row) * 16;
#pragma unroll
        for (int j = 0; j < 16; ++j) { od[j] = td[j]; oi[j] = ti[j]; }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (MC) cluster_sync_all();     // no CTA leaves while its peer may still multicast into it or arrive on its barriers
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---- host ------------------------------------------------------------------------------------
static int sm_count() { return device_sm_count(); }   // per device: one process may drive several GPUs

template <int BN, int STAGES, int EPI, bool MC = false, int BK = 64>
static int launch_gemm_variant(const CUtensorMap* maps, const GemmTcArgs& g, cudaStream_t s) {
  constexpr int smem = STAGES * (2 * GT_BM * BK * 2 + 2 * BN * BK * 2) + 1024 + 256;
  static DeviceOnce attr_done;   // the attribute is per device
  if (!attr_done.done()) {
    IBL_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<BN, STAGES, EPI, MC, BK>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_done.mark();
  }
  if (!MC) {
    const int grid = g.total_items < sm_count() ? g.total_items : sm_count();
    gemm_tc_kernel<BN, STAGES, EPI, false, BK><<<grid, 192, smem, s>>>(maps[0], maps[1], maps[2], maps[3], g);
    IBL_CUDA_OK(cudaGetLastError());
    return IBL_OK;
  }
  // clusters of two CTAs; g.total_items counts PAIRS of row tiles
  const int pairs = sm_count() / 2;
  const int units = g.total_items < pairs ? g.total_items : pairs;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * units);
  cfg.blockDim = dim3(192);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  IBL_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, STAGES, EPI, true, BK>, maps[0], maps[1], maps[2], maps[3], g));
  return IBL_OK;
}

static int make_plane_maps(CUtensorMap* maps, const __nv_bfloat16* a_hi, const __nv_bfloat16* a_lo, int M,
                           const __nv_bfloat16* b_hi, const __nv_bfloat16* b_lo, int N, int K, int bn, int bk = 64) {
  uint64_t dims_a[2] = {(uint64_t)K, (uint64_t)M}, dims_b[2] = {(uint64_t)K, (uint64_t)N};
  uint64_t str[1] = {(uint64_t)K * 2};
  uint32_t box_a[2] = {(uint32_t)bk, 128}, box_b[2] = {(uint32_t)bk, (uint32_t)bn};
  const int sw = bk == 64 ? 128 : 64;
  IBL_RET(make_tmap(&maps[0], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a_hi, dims_a, str, box_a, sw));
  IBL_RET(make_tmap(&maps[1], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a_lo, dims_a, str, box_a, sw));
  IBL_RET(make_tmap(&maps[2], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, b_hi, dims_b, str, box_b, sw));
  IBL_RET(make_tmap(&maps[3], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, b_lo, dims_b, str, box_b, sw));
  return IBL_OK;
}

// choose the number of column runs per row tile so the round-robin deal fills whole waves
static int pick_runs(int m_tiles, int n_tiles, int min_tiles_per_run, int units = 0) {
  const int G = units > 0 ? units : sm_count();
  int best = 1;
  double best_eff = -1.0;
  const int rmax = n_tiles / (min_tiles_per_run > 0 ? min_tiles_per_run : 1);
  for (int r = 1; r <= (rmax < 1 ? 1 : rmax) && r <= 64; ++r) {
    const int per = cdiv(n_tiles, r);
    const int runs = cdiv(n_tiles, per);
    const long long total = (long long)m_tiles * runs;
    const long long waves = (total + G - 1) / G;
    // time ~ waves * per (column tiles per item)
    const double eff = (double)m_tiles * n_tiles / ((double)waves * G * per);
    if (eff > best_eff + 1e-9) { best_eff = eff; best = runs; }
  }
  return best;
}

// Distance + running top-16 per (query, column run): cand_* [runs][M][16]; returns runs.
// Tile shape of the distance kernel (measured on 6.8k x 10k x 4096, whole retrieval call, same process):
//   BN=128, BK=64 (128B swizzle), 3 stages                      1.945 ms
//   BN=128, BK=64, 3 stages, CTA pairs + TMA multicast of B     1.890 ms   (IBL_DIST_BN=128 IBL_GEMM_MC=1)
//   BN=256, BK=32 (64B swizzle), 4 stages                       1.846 ms   (default)
// A 256-column tile needs 96 instead of 128 B/clk of shared-memory operand reads per MMA, and the half-size
// K chunk keeps a 4-deep pipeline inside 192 KiB.  All three land near 1.3 ms for the GEMM itself
// (~1285 TF/s of issued bf16 MMA, ~0.89 of the power-capped cuBLAS rate).
// clusters of two CTAs with TMA multicast of the database tile (only with BN=128; IBL_GEMM_MC=0 disables)
static bool gemm_mc() {
  static int mc = -1;
  if (mc < 0) { const char* v = getenv("IBL_GEMM_MC"); mc = (v && atoi(v) == 0) ? 0 : 1; }
  return mc != 0;
}

static int dist_bn() {
  static int bn = 0;
  if (!bn) { const char* v = getenv("IBL_DIST_BN"); bn = (v && atoi(v) == 128) ? 128 : 256; }
  return bn;
}

int launch_dist_top16_tc(const __nv_bfloat16* q_hi, const __nv_bfloat16* q_lo, const float* qn, int m,
                         const __nv_bfloat16* d_hi, const __nv_bfloat16* d_lo, const float* dn, int n,
                         int n_valid, int K, float* cand_d, long long* cand_i, int max_runs, int* runs_out,
                         cudaStream_t s) {
  IBL_REQUIRE(K % 64 == 0, "tcgen05 distance needs dim % 64 == 0");
  const int BN = dist_bn();
  const int m_tiles = cdiv(m, GT_BM);
  const bool mc = gemm_mc() && BN == 128 && m_tiles >= 2;
  const int bk = BN == 256 ? 32 : 64;
  CUtensorMap maps[4];
  IBL_RET(make_plane_maps(maps, q_hi, q_lo, m, d_hi, d_lo, n, K, mc ? BN / 2 : BN, bk));
  GemmTcArgs g{};
  g.M = m; g.N = n; g.K = K;
  g.n_tiles = cdiv(n_valid > 0 ? n_valid : 1, BN);
  const int m_units = mc ? cdiv(m_tiles, 2) : m_tiles;
  int runs = pick_runs(m_units, g.n_tiles, BN == 256 ? 1 : 2, mc ? sm_count() / 2 : 0);
  if (runs > max_runs) runs = max_runs;
  g.nt_per_item = cdiv(g.n_tiles, runs);
  g.items_per_mtile = cdiv(g.n_tiles, g.nt_per_item);
  g.kit_per_item = K / bk;
  g.total_items = m_units * g.items_per_mtile;
  g.n_valid = n_valid;
  g.an = qn; g.bn = dn;
  g.cand_d = cand_d; g.cand_i = cand_i;
  *runs_out = g.items_per_mtile;
  if (mc) return launch_gemm_variant<128, 3, EPI_TOP16, true>(maps, g, s);
  if (BN == 256) return launch_gemm_variant<256, 4, EPI_TOP16, false, 32>(maps, g, s);
  return launch_gemm_variant<128, 3, EPI_TOP16>(maps, g, s);
}

int dist_top16_max_runs(int m, int n_valid) {
  const int BN = dist_bn();
  const int m_tiles = cdiv(m, GT_BM);
  const bool mc = gemm_mc() && BN == 128 && m_tiles >= 2;
  return pick_runs(mc ? cdiv(m_tiles, 2) : m_tiles, cdiv(n_valid > 0 ? n_valid : 1, BN), BN == 256 ? 1 : 2,
                   mc ? sm_count() / 2 : 0);
}

int launch_dist_dense_tc(const __nv_bfloat16* q_hi, const __nv_bfloat16* q_lo, const float* qn, int m,
                         const __nv_bfloat16* d_hi, const __nv_bfloat16* d_lo, const float* dn, int n, int K,
                         float* out, long long ld_out, cudaStream_t s) {
  IBL_REQUIRE(K % 64 == 0, "tcgen05 distance needs dim % 64 == 0");
  constexpr int BN = 128;
  const int m_tiles = cdiv(m, GT_BM);
  const bool mc = gemm_mc() && m_tiles >= 2;
  CUtensorMap maps[4];
  IBL_RET(make_plane_maps(maps, q_hi, q_lo, m, d_hi, d_lo, n, K, mc ? BN / 2 : BN));
  GemmTcArgs g{};
  g.M = m; g.N = n; g.K = K;
  g.n_tiles = cdiv(n, BN);
  const int m_units = mc ? cdiv(m_tiles, 2) : m_tiles;
  const int runs = pick_runs(m_units, g.n_tiles, 1, mc ? sm_count() / 2 : 0);
  g.nt_per_item = cdiv(g.n_tiles, runs);
  g.items_per_mtile = cdiv(g.n_tiles, g.nt_per_item);
  g.kit_per_item = K / 64;
  g.total_items = m_units * g.items_per_mtile;
  g.n_valid = n;
  g.an = qn; g.bn = dn;
  g.out = out; g.ld_out = ld_out;
  if (mc) return launch_gemm_variant<BN, 3, EPI_DENSE, true>(maps, g, s);
  return launch_gemm_variant<BN, 3, EPI_DENSE>(maps, g, s);
}

// PCA GEMM: A = W planes [P,D], B = descriptor planes [N,D]; partial [splits][N][P]
int launch_pca_partial_tc(const __nv_bfloat16* w_hi, const __nv_bfloat16* w_lo, int P,
                          const __nv_bfloat16* v_hi, const __nv_bfloat16* v_lo, int N, int D,
                          float* partial, int* splits_out, cudaStream_t s) {
  IBL_REQUIRE(D % 64 == 0, "tcgen05 PCA needs D % 64 == 0");
  IBL_REQUIRE(N >= 1 && N <= 32, "tcgen05 PCA handles up to 32 rows per call");
  constexpr int BN = 32;
  CUtensorMap maps[4];
  IBL_RET(make_plane_maps(maps, w_hi, w_lo, P, v_hi, v_lo, N, D, BN));
  GemmTcArgs g{};
  g.M = P; g.N = N; g.K = D;
  g.n_tiles = 1;
  const int m_tiles = cdiv(P, GT_BM);
  const int ktot = D / 64;
  int splits = sm_count() / (m_tiles > 0 ? m_tiles : 1);
  if (splits < 1) splits = 1;
  if (splits > ktot) splits = ktot;
  g.kit_per_item = cdiv(ktot, splits);
  g.items_per_mtile = cdiv(ktot, g.kit_per_item);
  g.nt_per_item = 1;
  g.total_items = m_tiles * g.items_per_mtile;
  g.n_valid = N;
  g.out = partial;
  *splits_out = g.items_per_mtile;
  return launch_gemm_variant<BN, 5, EPI_PARTIAL>(maps, g, s);
}

int pca_tc_splits(int P, int D) {
  const int m_tiles = cdiv(P, GT_BM), ktot = D / 64;
  int splits = sm_count() / (m_tiles > 0 ? m_tiles : 1);
  if (splits < 1) splits = 1;
  if (splits > ktot) splits = ktot;
  const int per = cdiv(ktot, splits);
  return cdiv(ktot, per);
}

// ---- exact fp32 re-scoring of a candidate list + final ordering ---------------------------------
// one block (128 threads) per query: dist = |q|^2 + |d|^2 - 2 q.d with an fp32 dot product, then
// (dist, idx)-ascending sort of the kc <= 128 candidates; writes the first k_out.  Guard: a database row that was not
// kept has a screened distance >= s_kc (the largest screened distance kept), so its exact distance is >= s_kc - B
// (screen_guard_bound, 3 MMAs per 16-wide K step).  Unless s_kc - B > (k-th exact distance) the query is listed for
// the exact brute force of tc_dist1.cu.
__device__ __forceinline__ uint32_t f32_ord(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(128)
rescore_sort_kernel(const float* __restrict__ q, const float* __restrict__ qn,
                    const float* __restrict__ db, const float* __restrict__ dbn, int d,
                    const long long* __restrict__ cand_i, int kc, int k_out, long long idx_base,
                    float* __restrict__ out_dist, long long* __restrict__ out_idx, const RescoreGuard gd) {
  extern __shared__ __align__(16) float qs[];   // [d]
  __shared__ unsigned long long keys[128];
  const long long row = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  // the query row is staged in shared memory when it fits (d <= 16384, e.g. the 4096-d PCA
  // descriptors); the 32768-d raw VLAD is read through L1 instead
  const bool staged = d <= 16384;
  if (staged) {
    for (int i = threadIdx.x * 4; i < d; i += 128 * 4)
      *reinterpret_cast<float4*>(qs + i) = __ldg(reinterpret_cast<const float4*>(q + row * d + i));
  }
  const float* qrow = staged ? qs : (q + row * d);
  __syncthreads();
  const float an = __ldg(qn + row);
  for (int c = wid; c < 128; c += 4) {
    unsigned long long key = ~0ull;
    if (c < kc) {
      const long long ci = cand_i[row * kc + c];
      if (ci >= 0) {
        const float* dp = db + ci * d;
        float acc = 0.f;
        for (int i = lane * 4; i < d; i += 128) {
          const float4 a = *reinterpret_cast<const float4*>(qrow + i);
          const float4 b = __ldg(reinterpret_cast<const float4*>(dp + i));
          acc = fmaf(a.x, b.x, acc); acc = fmaf(a.y, b.y, acc);
          acc = fmaf(a.z, b.z, acc); acc = fmaf(a.w, b.w, acc);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        const float dist = fmaf(-2.f, acc, an + __ldg(dbn + ci));
        key = ((unsigned long long)f32_ord(dist) << 32) | (unsigned)ci;
      }
    }
    if (lane == 0) keys[c] = key;
  }
  // bitonic sort of 128 keys, one per thread pair
  for (int size = 2; size <= 128; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      if (threadIdx.x < 64) {
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
  if (threadIdx.x < k_out) {
    const unsigned long long key = keys[threadIdx.x];
    if (key == ~0ull) {
      out_dist[row * k_out + threadIdx.x] = INFINITY;
      out_idx[row * k_out + threadIdx.x] = -1;
    } else {
      const uint32_t u = (uint32_t)(key >> 32);
      out_dist[row * k_out + threadIdx.x] = __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
      out_idx[row * k_out + threadIdx.x] = idx_base + (long long)(uint32_t)(key & 0xffffffffu);
    }
  }
  if (threadIdx.x == 0 && gd.n_valid > kc) {            // with <= kc rows everything was re-scored
    const unsigned long long ek = keys[k_out - 1];
    bool flag = ek == ~0ull;
    float s_kc = -INFINITY;
    for (int c = 0; c < kc; ++c) {
      if (cand_i[row * kc + c] < 0) flag = true;         // fewer than kc candidates: cannot happen; be safe
      s_kc = fmaxf(s_kc, gd.cand_sd[row * kc + c]);
    }
    if (!flag) {
      const uint32_t u = (uint32_t)(ek >> 32);
      const float e_k = __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
      const float bound = screen_guard_bound(an, __ldg(gd.q_err + row), __ldg(gd.db_max2 + 1), __ldg(gd.db_max2), d,
                                             3 * (d / 16), 1.5411377e-5f);   // |ql||dl| <= (2^-8 (1 + 2^-8))^2 |q||d|
      flag = !(s_kc - bound > e_k);                     // also catches NaN
    }
    if (flag) gd.flag_list[atomicAdd(gd.flag_count, 1)] = (int)row;
  }
}

int launch_rescore_sort(const float* q, const float* qn, int m, const float* db, const float* dbn, int d,
                        const long long* cand_i, int kc, int k_out, long long idx_base, float* out_dist,
                        long long* out_idx, const RescoreGuard& guard, cudaStream_t s) {
  IBL_REQUIRE(kc >= 1 && kc <= 128 && k_out >= 1 && k_out <= 128, "rescore: 1 <= k <= 128");
  IBL_REQUIRE(d % 4 == 0, "rescore: dim must be a multiple of 4");
  static DeviceOnce attr_done;   // the attribute is per device
  if (!attr_done.done()) {
    IBL_CUDA_OK(cudaFuncSetAttribute(rescore_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    attr_done.mark();
  }
  if (m == 0) return IBL_OK;
  rescore_sort_kernel<<<m, 128, d <= 16384 ? d * sizeof(float) : 16, s>>>(q, qn, db, dbn, d, cand_i, kc, k_out, idx_base,
                                                       out_dist, out_idx, guard);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}

}  // namespace ibl
