// Shared declarations for libiblb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <string>

#include "../../include/iblb200.h"

namespace ibl {

void set_last_error(const std::string& s);

#define IBL_CUDA_OK(expr)                                                          \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      ::ibl::set_last_error(std::string(#expr) + ": " + cudaGetErrorString(_e) +   \
                            " (" __FILE__ ":" + std::to_string(__LINE__) + ")");   \
      return IBL_ERR_CUDA;                                                         \
    }                                                                              \
  } while (0)

#define IBL_RET(expr)                 \
  do {                                \
    int _s = (expr);                  \
    if (_s != IBL_OK) return _s;      \
  } while (0)

#define IBL_REQUIRE(cond, msg)                                  \
  do {                                                          \
    if (!(cond)) {                                              \
      ::ibl::set_last_error(std::string("bad argument: ") + msg); \
      return IBL_ERR_BAD_ARG;                                   \
    }                                                           \
  } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// "Done once" flag per CUDA device: function attributes (cudaFuncSetAttribute) and device properties belong
// to a device, and one process may drive several GPUs (one engine each).  done()/mark() look at the calling
// thread's current device; setting an attribute twice from two threads is harmless, launching before it
// is set is not, so mark() comes after the setter.
struct DeviceOnce {
  std::atomic<unsigned long long> mask[4];
  DeviceOnce() { for (auto& m : mask) m.store(0); }
  static int cur() { int d = 0; cudaGetDevice(&d); return d & 255; }
  bool done() const { const int d = cur(); return (mask[d >> 6].load(std::memory_order_acquire) >> (d & 63)) & 1ull; }
  void mark() { const int d = cur(); mask[d >> 6].fetch_or(1ull << (d & 63), std::memory_order_release); }
};

// Screening guard of the distance/top-k paths: an upper bound on |e(q,d) - s(q,d)| for ANY database row d, where
// e = fmaf(-2, q.d, |q|^2 + |d|^2) with an fp32 dot product (lane-strided FMAs, d/32 per lane, then a 5-level tree)
// and s = |q|^2 + |d|^2 - 2 q'.d' with q', d' the tensor-core representations, accumulated in TMEM.
//   representation:  q.d - q'.d' = dq.d' + q'.dd + dq.dd (+ the product the bf16x3 split drops, ql.dl)
//                    |.| <= |dq||d| + |q||dd| + |dq||dd| (+ |ql||dl|), all |x - x'| computed exactly per row;
//   accumulation:    the fp32 TMEM accumulator truncates once per MMA; every partial sum is <= |q'||d'|;
//   fp32 rounding:   of both the dot product and the two distance expressions.
// an = |q|^2, qe = |q - q'|, dmax_sq / dmax_err = max over the database rows of |d|^2 and |d - d'|,
// n_mma = MMAs accumulated per dot product, lolo = bound of |ql||dl| / (|q||d|) (0 for the fp16 plane).
// SCREEN_MMA_REL: the per-MMA truncation measured for kind::bf16 is 1.32e-8 of the accumulator
// (profiles/r01_diag_tc_accumulator_bias.txt, mean over 108..864 MMAs); 2^-22 = 2 fp32 ulps is 18x that.
#define SCREEN_MMA_REL 2.3841858e-7f
__host__ __device__ __forceinline__ float screen_guard_bound(float an, float qe, float dmax_sq, float dmax_err, int d,
                                                             int n_mma, float lolo) {
  const float nq = sqrtf(an) * 1.001f, nd = sqrtf(dmax_sq) * 1.001f;   // 1.001: fp32 sums and sqrt of the norms
  const float rep = qe * nd + nq * dmax_err + qe * dmax_err;
  const float rel = lolo + (float)n_mma * SCREEN_MMA_REL * 1.01f + (float)(d / 32 + 8) * 5.9604645e-8f;
  return 1.001f * (2.f * (rep + rel * nq * nd) + 4.7683716e-7f * (an + dmax_sq));   // 2^-21 (|q|^2 + |d|^2)
}

// SM count of the calling thread's current device
static inline int device_sm_count() {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  return sms;
}

// One conv layer of the VGG16 trunk.
struct ConvLayer {
  int cin, cout;
  bool relu;       // ReLU after the conv (all but conv5_3, vgg.py:41-42)
  bool pool;       // MaxPool2x2 after the ReLU (blocks 1-4)
};

// Device-side parameter store of one conv layer.
struct ConvParams {
  float* w_tck = nullptr;            // SIMT layout  [9][Cin][Cout] fp32
  float* bias = nullptr;             // [Cout]
  __nv_bfloat16* w_hi = nullptr;     // TC layout    [9][Cout][Cin_pad] bf16 (hi part)
  __nv_bfloat16* w_lo = nullptr;     //                                      (lo part)
  int cin_pad = 0;
};

// ---- launchers implemented in the .cu files ------------------------------------------------
// simt_conv.cu
int launch_repack_weights(const float* w_oihw, int cout, int cin, ConvParams& p, cudaStream_t s);
int launch_conv3x3_simt(const float* x_nhwc, const ConvParams& p, int N, int H, int W, int cin,
                        int cout, bool relu, float* y_nhwc, cudaStream_t s);
int launch_conv1_1(const float* x_nchw, const ConvParams& p, int N, int H, int W, bool to_planes,
                   float* y_nhwc, __nv_bfloat16* y_hi, __nv_bfloat16* y_lo, cudaStream_t s);
int launch_maxpool2x2(const float* x, int N, int H, int W, int C, float* y, cudaStream_t s);
int launch_nhwc_to_nchw(const float* x, int N, int S, int C, float* y, cudaStream_t s);
int launch_u8_hwc_to_nchw_norm(const uint8_t* x, int N, int H, int W, const float* mean, const float* stdv, float* y,
                               cudaStream_t s);
int launch_global_maxpool_nhwc(const float* x, int N, int S, int C, float* y, cudaStream_t s);
int launch_planes_to_f32(const __nv_bfloat16* hi, const __nv_bfloat16* lo, size_t n, float* y,
                         cudaStream_t s);
int launch_f32_to_planes(const float* x, size_t n, __nv_bfloat16* hi, __nv_bfloat16* lo,
                         cudaStream_t s);

// tc_conv.cu  (tcgen05 + TMA implicit GEMM, bf16 hi/lo split operands)
struct TcConvPlan;   // opaque per-engine cache of TMA descriptors
int tc_driver_init();   // resolves cuTensorMapEncodeTiled; IBL_ERR_NO_DEVICE if unavailable
int launch_conv3x3_tc(const __nv_bfloat16* x_hi, const __nv_bfloat16* x_lo, const ConvParams& p,
                      int N, int H, int W, int cin, int cout, bool relu, bool pool,
                      __nv_bfloat16* y_hi, __nv_bfloat16* y_lo, float* y_f32, cudaStream_t s,
                      float* ssq = nullptr, int* ssq_parts = nullptr);
int launch_conv1_fused_tc(const float* x_nchw, const float* w1_oihw, const float* bias1, const ConvParams& p2, int N, int H,
                          int W, __nv_bfloat16* y_hi, __nv_bfloat16* y_lo, cudaStream_t s);
int launch_maxpool2x2_planes(const __nv_bfloat16* hi, const __nv_bfloat16* lo, int N, int H, int W,
                             int C, __nv_bfloat16* yhi, __nv_bfloat16* ylo, cudaStream_t s);
int tc_selftest(float* max_rel_err, cudaStream_t s);
// sort_rows.cu  (full argsort of distance-matrix rows: the training samplers' mining)
int launch_argsort_rows(const float* dist, long long ld, int m, int n, long long* idx, unsigned long long* scratch,
                        cudaStream_t s, uint64_t* launches);
// resize.cu  (Pillow-exact 8-bit bilinear resample)
int launch_resize_bilinear_u8(const uint8_t* x, int N, int Hin, int Win, int Hout, int Wout, const int* bounds_h,
                              const int* kk_h, int ksize_h, const int* bounds_v, const int* kk_v, int ksize_v,
                              uint8_t* tmp, uint8_t* out, cudaStream_t s, uint64_t* launches);
// tc_conv_bwd.cu  (dgrad filter re-layout, tcgen05 wgrad, ReLU mask, pool backward, conv1_1 wgrad)
int launch_repack_weights_dgrad(const float* w_tck, int cout, int cin, __nv_bfloat16* w_hi, __nv_bfloat16* w_lo,
                                cudaStream_t s);
int launch_relu_mask_planes(const float* g, const float* y, size_t n, bool relu, __nv_bfloat16* hi, __nv_bfloat16* lo,
                            cudaStream_t s);
int launch_maxpool2x2_bwd(const float* x, const float* gy, int N, int H, int W, int C, float* gx, cudaStream_t s);
int wgrad_tc_splits(int N, int H, int W, int cin, int cout);
int launch_conv_wgrad_tc(const __nv_bfloat16* g_hi, const __nv_bfloat16* g_lo, const __nv_bfloat16* x_hi,
                         const __nv_bfloat16* x_lo, int N, int H, int W, int cin, int cout, float* part, int splits,
                         float* bpart, float* dw_oihw, float* db, cudaStream_t s);
int launch_conv1_1_wgrad(const float* x_nchw, const __nv_bfloat16* g_hi, const __nv_bfloat16* g_lo, int N, int H, int W,
                         float* part, float* dw_oihw, float* db, cudaStream_t s);
// tc_conv1.cu
int launch_conv1_1_tc(const float* x_nchw, const float* w_oihw, const float* bias, int N, int H, int W,
                      __nv_bfloat16* y_hi, __nv_bfloat16* y_lo, cudaStream_t s);
// tc_netvlad.cu
int debug_gemm_tn(const float* A, const float* B, float* C, cudaStream_t s);
int netvlad_tc_units(int B, int S);
// tc_probe.cu
int debug_umma_strided(const void* A, int rows, const void* B, int s0, int group_rows, int base_mode, float* D,
                       cudaStream_t s);
int launch_netvlad_tc(const __nv_bfloat16* x_hi, const __nv_bfloat16* x_lo, int B, int S,
                      const __nv_bfloat16* w_hi, const __nv_bfloat16* w_lo, const float* ssq, int ssq_parts,
                      const float* cent, bool normalize_input, float* part, float* asum_part, int* ticket,
                      float* vlad_raw, float* vlad_norm, cudaStream_t s);
int launch_global_maxpool_planes(const __nv_bfloat16* hi, const __nv_bfloat16* lo, int N, int S, int C, float* y,
                                 cudaStream_t s);

// tc_gemm.cu  (tcgen05 NT GEMM on bf16 hi/lo planes: distance/top-16, dense distance, PCA partials)
int dist_top16_max_runs(int m, int n_valid);
int launch_dist_top16_tc(const __nv_bfloat16* q_hi, const __nv_bfloat16* q_lo, const float* qn, int m,
                         const __nv_bfloat16* d_hi, const __nv_bfloat16* d_lo, const float* dn, int n,
                         int n_valid, int K, float* cand_d, long long* cand_i, int max_runs, int* runs_out,
                         cudaStream_t s);
int launch_dist_dense_tc(const __nv_bfloat16* q_hi, const __nv_bfloat16* q_lo, const float* qn, int m,
                         const __nv_bfloat16* d_hi, const __nv_bfloat16* d_lo, const float* dn, int n, int K,
                         float* out, long long ld_out, cudaStream_t s);
// tc_gemm2.cu  (same contract on SM pairs: tcgen05.mma.cta_group::2, 256-row tiles)
int dist_top16_2sm_max_runs(int m, int n_valid);
int launch_dist_top16_2sm(const __nv_bfloat16* q_hi, const __nv_bfloat16* q_lo, const float* qn, int m,
                          const __nv_bfloat16* d_hi, const __nv_bfloat16* d_lo, const float* dn, int n,
                          int n_valid, int K, float* cand_d, long long* cand_i, int* runs_out, cudaStream_t s);
// tc_dist1.cu  (single-pass fp16 screening on SM pairs + exact re-scoring + guard + exact fallback)
size_t dist1_workspace_bytes(int m, int n, int d, size_t* off /*[9]*/);
int launch_dist_topk_1pass(const float* q, int m, const float* db, int n, int n_valid, int d, int k, long long idx_base,
                           void* ws, float* out_dist, long long* out_idx, uint64_t* launches, cudaStream_t s);
int* dist1_flag_count(void* ws, int m, int n, int d);
int launch_dist_colmax(const float* sq, const float* err, int stride, int n, float* out2, cudaStream_t s);
size_t dist_exact_scratch_bytes(int m, int n_valid, int k);
int launch_dist_exact_fallback(const float* q, const float* qn, int qn_stride, int m, const float* db, const float* dbn,
                               int dbn_stride, int n_valid, int d, int k, long long idx_base, const int* flag_count,
                               const int* flag_list, unsigned long long* scratch, float* out_dist, long long* out_idx,
                               cudaStream_t s);
int pca_tc_splits(int P, int D);
int launch_pca_partial_tc(const __nv_bfloat16* w_hi, const __nv_bfloat16* w_lo, int P,
                          const __nv_bfloat16* v_hi, const __nv_bfloat16* v_lo, int N, int D,
                          float* partial, int* splits_out, cudaStream_t s);
// guard inputs of launch_rescore_sort: the bf16x3 representation errors and the screened candidate distances
struct RescoreGuard {
  const float* cand_sd;   // [m][kc] screened distances of the candidates
  const float* q_err;     // [m] |q - (hi + lo)|
  const float* db_max2;   // {max |d - (hi + lo)|, max |d|^2} over the valid database rows
  int n_valid;
  int* flag_count; int* flag_list;
};
int launch_rescore_sort(const float* q, const float* qn, int m, const float* db, const float* dbn, int d,
                        const long long* cand_i, int kc, int k_out, long long idx_base, float* out_dist,
                        long long* out_idx, const RescoreGuard& guard, cudaStream_t s);
int launch_pca_finalize(const float* partial, int splits, int N, int P, const float* bias, float* out,
                        cudaStream_t s);

// netvlad.cu
struct NetvladWorkspace {
  float* assign = nullptr;   // [N,S,K]  soft-assignment * inv-norm handled in kernel
  float* invnorm = nullptr;  // [N,S]
  float* asum = nullptr;     // [N,K]
  float* raw = nullptr;      // [N,K,C]  (used when the caller does not want vlad_raw)
  size_t cap_N = 0;
  int cap_S = 0, cap_K = 0, cap_C = 0;
};
int launch_netvlad(const float* feat, bool nhwc, int N, int C, int S, const float* conv_w,
                   const float* centroids, int K, bool normalize_input, float* assign,
                   float* invnorm, float* asum, float* vlad_raw, float* vlad_norm,
                   cudaStream_t s, uint64_t* launches);
int launch_vlad_normalize(const float* raw, int N, int K, int C, float* out, cudaStream_t s);
int launch_netvlad_assign(const float* feat, bool nhwc, int N, int C, int S, const float* conv_w,
                          bool normalize_input, float* assign, float* invnorm, cudaStream_t s);
// netvlad_bwd.cu
int launch_netvlad_backward(const float* x, bool nhwc, int N, int C, int S, const float* conv_w,
                            const float* centroids, const float* g, bool normalize_input, float* assign,
                            float* invnorm, float* dz, float* part, int splits, float* dx, float* dW,
                            float* dcent, cudaStream_t s, uint64_t* launches);

// gemm_simt.cu  (C = A[m,K] . B[n,K]^T family)
int launch_pca_l2(const float* v, int N, int D, const float* W, const float* b, int P,
                  float* partial, int splits, float* out, cudaStream_t s, uint64_t* launches);
int launch_l2_normalize_rows(const float* x, int N, int D, float* out, cudaStream_t s);
int launch_row_sqnorm(const float* x, int N, int D, float* out, cudaStream_t s);
int launch_scale(const float* x, float s, int n, float* y, cudaStream_t st);
// err (may be null): |x - (hi + lo)| per row, exact up to the fp32 sum of squares
int launch_planes_sqnorm(const float* x, int N, int D, __nv_bfloat16* hi, __nv_bfloat16* lo, float* sq,
                         cudaStream_t st, float* err = nullptr);
int launch_l2dist_dense(const float* q, const float* qn, int m, const float* db, const float* dbn,
                        int n, int d, float* out, long long ld_out, cudaStream_t s);

// topk.cu
int launch_topk_rows(const float* dist, long long ld, int m, int n_valid, int k, int64_t idx_base,
                     float* out_dist, int64_t* out_idx, bool accumulate, cudaStream_t s);
int launch_topk_merge(const float* cand_dist, const int64_t* cand_idx, int parts, int m, int k_in,
                      int k_out, float* out_dist, int64_t* out_idx, cudaStream_t s);

}  // namespace ibl
