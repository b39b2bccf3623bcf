/*
 * iblb200.h -- C ABI of the B200-native OpenIBL hot path (libiblb200.so).
 *
 * Drop-in boundary for the one data-parallel path of yxgeee/OpenIBL:
 *   VGG16 conv1_1..conv5_3 -> NetVLAD (+intra-norm, L2) -> PCA-whiten + L2
 *   -> query x database L2 distance -> top-k.
 * The reference is pure Python on torch ops and has no FFI of its own; each
 * entry point below names the reference call site (file:line under the
 * reference root) whose arithmetic it replaces.  The host-side mirror of the
 * reference API (ibl.models / ibl.evaluators / ibl.pca) binds these symbols with
 * ctypes -- see INTEGRATION.md for the stub a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - Every function returns an ibl_status (0 = OK) and never throws.
 *   - Unless a name ends in _host, pointers are DEVICE pointers on the engine's
 *     device; fp32, contiguous.  `stream` is a cudaStream_t passed as void*
 *     (NULL = legacy default stream).  No hidden synchronisation except in the
 *     *_host entry points, which return after their result is in host memory.
 *   - The caller owns every input and output buffer.  The engine owns only its
 *     workspace and re-laid-out weight copies.
 *   - One engine per (process, GPU); not thread-safe (the reference drives one
 *     GPU from one Python thread, scripts/test_dist.sh:27).
 */
#ifndef IBLB200_H_
#define IBLB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IBLB200_ABI_VERSION 1

typedef enum ibl_status {
  IBL_OK = 0,
  IBL_ERR_BAD_ARG = 1,       /* null pointer, non-positive size, unsupported shape */
  IBL_ERR_NOT_READY = 2,     /* weights for the requested stage were never set */
  IBL_ERR_CUDA = 3,          /* a CUDA runtime/driver call failed (see ibl_last_error) */
  IBL_ERR_NO_DEVICE = 4,     /* no usable sm_100 device: there is NO CPU fallback */
  IBL_ERR_OOM = 5,           /* workspace allocation failed */
  IBL_ERR_UNSUPPORTED = 6    /* valid request this build cannot serve */
} ibl_status;

typedef struct ibl_engine ibl_engine;

/* extraction flags for ibl_extract / ibl_extract_host */
#define IBL_OUT_VLAD 0x1u  /* out = L2(flatten(intra-norm(vlad)))  [N, K*C]   (EmbedNet, netvlad.py:73-82) */
#define IBL_OUT_PCA  0x2u  /* out = L2(W out_vlad + b)              [N, P]     (EmbedNetPCA, netvlad.py:95-110) */
#define IBL_OUT_POOL 0x4u  /* also write pool [N,512]               (vgg.py:67-70) */

/* conv math mode (ibl_engine_set_conv_mode) */
#define IBL_CONV_SIMT_FP32 0  /* fp32 CUDA-core implicit GEMM (verification path)              */
#define IBL_CONV_TC_BF16X3 1  /* tcgen05 implicit GEMM, bf16 hi/lo split, 3 MMAs, fp32 accum   */

int ibl_abi_version(void);
const char* ibl_status_string(int status);
/* Text of the most recent failure on this thread ("" if none). */
const char* ibl_last_error(void);

/* ---- engine lifetime ------------------------------------------------------- */
int ibl_engine_create(int device, ibl_engine** out);
int ibl_engine_destroy(ibl_engine* e);
int ibl_engine_set_conv_mode(ibl_engine* e, int mode);
int ibl_engine_get_conv_mode(ibl_engine* e, int* mode);
/* Math mode of the distance and PCA GEMMs (same two values; default tcgen05 bf16x3 with exact fp32
 * re-scoring of the top-k candidates). */
int ibl_engine_set_gemm_mode(ibl_engine* e, int mode);
/* Number of kernels this library has launched through `e` since creation. */
int ibl_engine_launch_count(ibl_engine* e, uint64_t* count);

/* ---- parameters ------------------------------------------------------------ */
/* VGG16 trunk parameters, reference layout: weights[i] is OIHW [Cout,Cin,3,3],
 * biases[i] is [Cout], i = conv1_1..conv5_3 (state-dict slots
 * base.{0,2,5,7,10,12,14,17,19,21,24,26,28}, vgg.py:40-42).  The engine keeps
 * re-laid-out copies; call again after the parameters change. */
int ibl_engine_set_vgg16(ibl_engine* e, const float* const* weights13,
                         const float* const* biases13, void* stream);
/* NetVLAD parameters: conv_w [K,C] (net_vlad.conv.weight squeezed), centroids [K,C]
 * (netvlad.py:28-29). */
int ibl_engine_set_netvlad(ibl_engine* e, const float* conv_w, const float* centroids,
                           int K, int C, void* stream);
/* PCA-whitening layer: W [P,D] (pca_layer.weight squeezed == PCA.load weight,
 * pca.py:105), b [P]. */
int ibl_engine_set_pca(ibl_engine* e, const float* W, const float* b, int P, int D, void* stream);

/* ---- stage (i): backbone --------------------------------------------------- */
/* VGG.forward -> self.base (vgg.py:61-62) and gap (vgg.py:67-70).
 * x NCHW [N,3,H,W]  ->  feat_nhwc [N,H/16,W/16,512] (engine-native layout, may be NULL),
 * feat_nchw [N,512,H/16,W/16] (reference layout, may be NULL), pool [N,512] (may be NULL). */
int ibl_vgg16_forward(ibl_engine* e, const float* x_nchw, int N, int H, int W,
                      float* feat_nhwc, float* feat_nchw, float* pool, void* stream);

/* ---- stage (i), training surface (config 5: SFRS trains conv5_x, vgg.py:50-53) --------------- */
/* Layers are numbered 0..12 (conv1_1..conv5_3); activations cross the boundary as fp32 NHWC.
 * Frozen prefix: layers [0, n_layers) with their ReLUs and pools -> out_nhwc (the activation entering layer
 * n_layers); what autograd skips for requires_grad=False layers (vgg.py:50-53). */
int ibl_vgg16_prefix_forward(ibl_engine* e, const float* x_nchw, int N, int H, int W, int n_layers,
                             float* out_nhwc, void* stream);
/* One trainable layer: y = [ReLU](conv3x3(x) + b), no pooling (vgg.py:61-62 one nn.Conv2d + nn.ReLU).
 * layer 0 reads the NCHW image, layers >= 1 fp32 NHWC [N,H,W,Cin]; y [N,H,W,Cout]. */
int ibl_vgg16_layer_forward(ibl_engine* e, int layer, const float* x, int N, int H, int W, float* y_nhwc,
                            void* stream);
/* nn.MaxPool2d(2, 2) forward / backward on fp32 NHWC (gradient to the first maximum of each window). */
int ibl_maxpool2x2_forward(ibl_engine* e, const float* x_nhwc, int N, int H, int W, int C, float* y_nhwc,
                           void* stream);
int ibl_maxpool2x2_backward(ibl_engine* e, const float* x_nhwc, const float* gy_nhwc, int N, int H, int W, int C,
                            float* gx_nhwc, void* stream);
/* Backward of one trainable layer (what autograd + cuDNN dgrad/wgrad compute for vgg.py:61-62): x = the layer's
 * input, y = its post-ReLU output (read only if the layer has a ReLU), gy = dL/dy.  gx = dL/dx (NULL for the first
 * trainable layer), gw [Cout,Cin,3,3], gb [Cout].  dgrad and wgrad run on tcgen05 (bf16x3). */
int ibl_vgg16_layer_backward(ibl_engine* e, int layer, const float* x, const float* y, const float* gy, int N,
                             int H, int W, float* gx, float* gw, float* gb, void* stream);

/* ---- stage (ii): NetVLAD --------------------------------------------------- */
/* NetVLAD.forward (netvlad.py:44-61) + EmbedNet normalisation (netvlad.py:78-80), fused.
 * feat is [N,S,C] if nhwc != 0 else [N,C,S].  conv_w/centroids [K,C] are read directly.
 * vlad_raw [N,K,C] (un-normalised, what NetVLAD.forward returns; may be NULL)
 * vlad_norm [N,K*C] (intra-norm + flatten + L2; may be NULL). */
int ibl_netvlad_forward(ibl_engine* e, const float* feat, int nhwc, int N, int C, int S,
                        const float* conv_w, const float* centroids, int K,
                        int normalize_input, float* vlad_raw, float* vlad_norm, void* stream);
/* Backward of NetVLAD.forward (what autograd derives for netvlad.py:44-61; SURVEY 8 row a11, used by the SFRS
 * training step, netvlad.py:139-146).  grad_vlad [N,K,C] -> grad_feat (same layout as feat), grad_conv_w [K,C],
 * grad_centroids [K,C] (both summed over the batch).  fp32 CUDA cores; the soft-assignment is recomputed. */
int ibl_netvlad_backward(ibl_engine* e, const float* feat, int nhwc, int N, int C, int S,
                         const float* conv_w, const float* centroids, int K, int normalize_input,
                         const float* grad_vlad, float* grad_feat, float* grad_conv_w,
                         float* grad_centroids, void* stream);
/* Only the two normalisations (netvlad.py:78-80): vlad_raw [N,K,C] -> out [N,K*C]. */
int ibl_vlad_normalize(ibl_engine* e, const float* vlad_raw, int N, int K, int C,
                       float* out, void* stream);

/* ---- stage (iii-a): PCA-whiten + L2 ---------------------------------------- */
/* EmbedNetPCA.pca_layer + F.normalize (netvlad.py:105-108) == PCA.infer (pca.py:108-123).
 * v [N,D], W [P,D], b [P] -> out [N,P]. */
int ibl_pca_l2(ibl_engine* e, const float* v, int N, int D, const float* W, const float* b,
               int P, float* out, void* stream);
/* F.normalize(x, p=2, dim=-1) (evaluators.py:29-33): rows [N,D] in place or to out. */
int ibl_l2_normalize_rows(ibl_engine* e, const float* x, int N, int D, float* out, void* stream);

/* ---- whole extraction ------------------------------------------------------ */
/* extract_cnn_feature + pca (evaluators.py:22-34,56-57) with parameters set on the engine.
 * out is [N,K*C] for IBL_OUT_VLAD, [N,P] for IBL_OUT_VLAD|IBL_OUT_PCA; pool [N,512] if
 * IBL_OUT_POOL. */
int ibl_extract(ibl_engine* e, const float* x_nchw, int N, int H, int W, unsigned flags,
                float* out, float* pool, void* stream);
/* Same through HOST buffers (pinned or pageable): H2D of x, the pipeline, D2H of out (+pool),
 * then a stream synchronise -- the reference's per-batch `.cuda()` ... `.cpu()`
 * (evaluators.py:24,58). */
int ibl_extract_host(ibl_engine* e, const float* x_nchw_host, int N, int H, int W,
                     unsigned flags, float* out_host, float* pool_host, void* stream);

/* Two-deep pipelined form of ibl_extract_host (the overlap a loader loop gets in the reference from pin_memory +
 * non_blocking .cuda(), evaluators.py:24, here inside the library): submit(slot) enqueues H2D on the engine's copy
 * stream, the extraction and the D2H of the descriptors, and returns without synchronising; wait(slot) blocks until
 * that batch's descriptors are in out_host.  slot is 0 or 1; the host buffers must stay valid until wait returns. */
int ibl_extract_host_submit(ibl_engine* e, int slot, const float* x_nchw_host, int N, int H, int W, unsigned flags,
                            float* out_host, float* pool_host, void* stream);
int ibl_extract_host_wait(ibl_engine* e, int slot);

/* ---- input side: ToTensor + Normalize on the GPU ----------------------------- */
/* The reference's test transform after the resize (ibl/utils/data/__init__.py:37-42: T.ToTensor(),
 * T.Normalize(mean, std)) applied to decoded uint8 HWC pixels: out[n,c,h,w] = ((x[n,h,w,c]/255) - mean[c]) / std[c],
 * IEEE fp32 operations in that order (bit-identical to torchvision on the CPU).  x_nhwc device uint8 [N,H,W,3],
 * mean3/std3 HOST float[3], out device fp32 [N,3,H,W]. */
int ibl_preprocess_u8(ibl_engine* e, const uint8_t* x_nhwc, int N, int H, int W, const float* mean3,
                      const float* std3, float* out_nchw, void* stream);
/* T.Resize((H, W)) on a PIL image (the first stage of the reference's test transform, utils/data/__init__.py:37-42):
 * Pillow's 8-bit bilinear resample (antialiased, fixed point, horizontal pass then vertical pass), bit-exact.
 * x [N,Hin,Win,3] -> out [N,Hout,Wout,3], device uint8.  bounds_* [out,2] (first sample, count) and kk_* [out,ksize]
 * (coefficients with 22 fractional bits) are DEVICE int32 tables built by the host as Pillow's precompute_coeffs /
 * normalize_coeffs_8bpc do (openibl_b200/utils/data/gpu_resize.py); a pass whose sizes are equal is skipped. */
int ibl_resize_bilinear_u8(ibl_engine* e, const uint8_t* x_nhwc, int N, int Hin, int Win, int Hout, int Wout,
                           const int* bounds_h, const int* kk_h, int ksize_h, const int* bounds_v, const int* kk_v,
                           int ksize_v, uint8_t* out_nhwc, void* stream);
/* ibl_extract_host for a loader that hands over decoded uint8 HWC images (Preprocessor.__getitem__,
 * ibl/utils/data/preprocessor.py:31-42, minus the CPU transform): H2D of N*H*W*3 bytes (a quarter of the fp32
 * tensor), the transform above on the device, the extraction path, D2H of the descriptors, stream sync. */
int ibl_extract_host_u8(ibl_engine* e, const uint8_t* x_nhwc_host, int N, int H, int W, const float* mean3,
                        const float* std3, unsigned flags, float* out_host, float* pool_host, void* stream);

/* ---- stage (iii-b): distance + ranking ------------------------------------- */
/* pairwise_distance(features) with query = gallery = None (evaluators.py:106-114):
 * out[i,j] = 2|x_i|^2 - 2 x_i.x_j, x [n,d], out [n,n]. */
int ibl_l2dist_self(ibl_engine* e, const float* x, int n, int d, float* out, void* stream);
/* pairwise_distance (evaluators.py:127-129): out[i,j] = |q_i|^2 + |db_j|^2 - 2 q_i.db_j,
 * q [m,d], db [n,d], out [m,n].  Kept for the callers that need the dense matrix
 * (netvlad_img.py:78). */
int ibl_l2dist_dense(ibl_engine* e, const float* q, int m, const float* db, int n, int d,
                     float* out, void* stream);
/* Fused distance + per-query top-k over one database shard; replaces pairwise_distance +
 * np.argsort (evaluators.py:127-129,143) for the ranks evaluate_all reads (:151-159).
 * out_dist [m,k] ascending, out_idx [m,k] = idx_base + row in db; ties: lowest index first.
 * n_valid <= n rows of db are real (the rest is DistributedSliceSampler padding,
 * sampler.py:208-219, and is ignored).  k <= 128.  Tensor cores screen, exact fp32 decides: only the
 * candidates a screening pass keeps are re-scored exactly, and a guard with a bound that holds for any input
 * (representation errors, accumulator truncation, fp32 rounding) sends every query whose ranking the screening could
 * have changed to an exact brute force on the device, without host synchronisation.  With k >= 121 the bf16x3 path
 * keeps fewer than 8 spare candidates, and most queries take that brute force. */
int ibl_l2dist_topk(ibl_engine* e, const float* q, int m, const float* db, int n, int n_valid,
                    int d, int k, int64_t idx_base, float* out_dist, int64_t* out_idx,
                    void* stream);
/* Per-row top-k of an existing dense matrix dist [m,n] (row stride n): the ranks evaluate_all reads
 * from np.argsort (evaluators.py:143,151-159).  Same ordering rule as ibl_l2dist_topk.  1 <= k <= 1024. */
int ibl_topk_rows(ibl_engine* e, const float* dist, int m, int n, int k, float* out_dist,
                  int64_t* out_idx, void* stream);
/* torch.argsort(distmat, dim=1) of the training samplers' refresh (ibl/utils/data/sampler.py:46-54,126-135) on the
 * device: dist [m,n] -> out_idx [m,n], every row ascending by (distance, index). */
int ibl_argsort_rows(ibl_engine* e, const float* dist, int m, int n, int64_t* out_idx, void* stream);
/* k-way merge of per-shard candidates (after the NCCL all-gather): cand_* [parts,m,k_in]
 * -> out_* [m,k_out] ascending by (dist, idx). Entries with idx < 0 are ignored. */
int ibl_topk_merge(ibl_engine* e, const float* cand_dist, const int64_t* cand_idx, int parts,
                   int m, int k_in, int k_out, float* out_dist, int64_t* out_idx, void* stream);
/* Host-buffer variant of ibl_l2dist_topk for the e2e measurement: H2D of q and db, kernel,
 * D2H of results, synchronise. */
int ibl_l2dist_topk_host(ibl_engine* e, const float* q_host, int m, const float* db_host, int n,
                         int d, int k, float* out_dist_host, int64_t* out_idx_host, void* stream);

/* C[m,n] = alpha * A[m,k] . B[n,k]^T on the engine's GEMM kernels: the products of PCA.train (pca.py:38-67,
 * torch.matmul there).  mode IBL_CONV_SIMT_FP32 (fp32 CUDA cores) or IBL_CONV_TC_BF16X3 (tcgen05, k % 64 == 0). */
int ibl_gemm_nt(ibl_engine* e, const float* A, int m, const float* B, int n, int k, float alpha, float* C, int mode,
                void* stream);

/* ---- self-tests (GPU) ------------------------------------------------------ */
/* Queries that the screening guard re-ranked by exact brute force in the last ibl_l2dist_topk call, whichever
 * tensor-core path it took (-1: the call took the CUDA-core path).  Synchronises. */
int ibl_debug_dist_flagged(ibl_engine* e, int* count, void* stream);
/* Runs the tcgen05/TMA building blocks against CUDA-core results on the device;
 * returns IBL_OK when all agree. max_rel_err (may be NULL) receives the worst error. */
int ibl_selftest_tc(ibl_engine* e, float* max_rel_err);

/* One 3x3/s1/p1 conv layer in isolation (test hook): x NHWC [N,H,W,Cin] fp32, w OIHW, optional
 * ReLU and fused 2x2 max-pool, y NHWC fp32.  mode: IBL_CONV_SIMT_FP32, IBL_CONV_TC_BF16X3 (fp32
 * epilogue) or 2 (tcgen05 with the bf16 hi/lo plane epilogue, converted back to fp32).
 * bn_override forces the N tile (64/128/256) when it divides Cout, 0 = default. Synchronises. */
int ibl_debug_conv3x3(ibl_engine* e, const float* x_nhwc, int N, int H, int W, int cin,
                      const float* w_oihw, const float* bias, int cout, int relu, int pool, int mode,
                      int bn_override, float* y_nhwc, void* stream);

/* MN-major tcgen05 operand self-test: C[128,64] = A^T B for A [128 k,128 m], B [128 k,64 n] (fp32, device),
 * bf16x3 on the tensor core.  Synchronises. */
int ibl_debug_gemm_tn(ibl_engine* e, const float* A, const float* B, float* C, void* stream);
/* Hardware probe (tools/probe_umma_stride.py): D[128,64] = view(A) . B^T on tcgen05 where view row m is row
 * s0 + (m/8)*group_rows + (m%8) of the TMA-staged, 128B-swizzled [rows][64] bf16 tile A; base_mode 1 sets the
 * descriptor's base_offset field to the start row's swizzle phase.  Decides whether a conv can read its nine
 * taps out of one halo tile. */
int ibl_debug_umma_strided(ibl_engine* e, const void* A, int rows, const void* B, int s0, int group_rows,
                           int base_mode, float* D, void* stream);
/* Average device time (ms) of one backbone layer over `reps` launches, weights from the engine
 * (tools/bench_layers.py).  layer 0 = conv1_1 (x NCHW [N,3,H,W]); 1..12 = conv1_2..conv5_3
 * (x NHWC [N,H,W,Cin] fp32).  Synchronises. */
int ibl_debug_time_layer(ibl_engine* e, int layer, const float* x, int N, int H, int W, int bn_override,
                         int reps, float* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* IBLB200_H_ */
