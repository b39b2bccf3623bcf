// C-ABI entry points of libiblb200 (see include/iblb200.h).  The engine owns the workspace
// arena and the re-laid-out weights; every entry point validates its arguments, enqueues
// kernels on the caller's stream and returns a status code -- it never throws and never
// synchronises, except for the *_host variants.
#include <stdlib.h>

#include <mutex>
#include <new>
#include <vector>

#include "common.cuh"

namespace ibl {

static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
void tc_set_bn_override(int bn);

static const ConvLayer kVgg16[13] = {
    {3, 64, true, false},    {64, 64, true, true},     // block 1
    {64, 128, true, false},  {128, 128, true, true},   // block 2
    {128, 256, true, false}, {256, 256, true, false}, {256, 256, true, true},   // block 3
    {256, 512, true, false}, {512, 512, true, false}, {512, 512, true, true},   // block 4
    {512, 512, true, false}, {512, 512, true, false}, {512, 512, false, false}  // block 5 (no ReLU last)
};

// A growable device buffer.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return IBL_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_last_error("workspace cudaMalloc(" + std::to_string(bytes) + " B) failed: " + cudaGetErrorString(e));
      return IBL_ERR_OOM;
    }
    cap = bytes;
    return IBL_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

}  // namespace ibl

using namespace ibl;

struct ibl_engine {
  int device = 0;
  int conv_mode = IBL_CONV_TC_BF16X3;
  int gemm_mode = IBL_CONV_TC_BF16X3;   // distance / PCA GEMMs: same two math modes
  uint64_t launches = 0;
  bool vgg_ready = false;
  ConvParams conv[13];
  float* w0_oihw = nullptr;   // conv1_1 filters in the reference OIHW layout (tcgen05 conv1_1 builds its own operand)
  // borrowed NetVLAD / PCA parameters (owned by the caller's torch Parameters)
  const float* nv_w = nullptr;
  const float* nv_c = nullptr;
  int nv_K = 0, nv_C = 0;
  const float* pca_W = nullptr;
  const float* pca_b = nullptr;
  int pca_P = 0, pca_D = 0;
  // workspace
  DevBuf act[2];       // activation ping-pong (fp32 NHWC, or bf16 hi|lo planes back to back)
  DevBuf feat;         // conv5_3 output, fp32 NHWC
  DevBuf nv_assign, nv_inv, nv_raw, vlad;
  DevBuf pca_partial;
  DevBuf qn, dbn, dist_chunk, cand_d, cand_i;
  DevBuf stage_in, stage_out, stage_out2, stage_u8;
  DevBuf q_pl, db_pl, v_pl, pca_pl;     // bf16 hi|lo planes of queries, database shard, descriptors, PCA W
  const float* pca_pl_src = nullptr;    // W pointer the cached planes were made from
  DevBuf mrg_d, mrg_i;
  DevBuf bw_g, bw_x, bw_part, bw_w;      // conv backward: dY planes, X planes, wgrad/bias partials, dgrad filter planes
  DevBuf d1_ws;                          // workspace of the single-pass distance/top-k path (tc_dist1.cu)
  DevBuf dguard;                         // guard + exact fallback of the bf16x3 distance/top-k paths
  const int* dist_flags = nullptr;       // flag counter of the last ibl_l2dist_topk call (null: CUDA-core path)
  DevBuf ssq, nv_part, nv_asum, nvw_pl;  // fused NetVLAD: |x|^2 partials, unit partials, W planes [64,512]
  DevBuf nv_ticket;                      // [images] arrival counters of the fused NetVLAD kernel (zero between launches)
  const float* nvw_pl_src = nullptr;
  cudaStream_t copy_stream = nullptr;   // H2D staging of ibl_extract_host overlaps compute
  cudaEvent_t copy_ev[2] = {nullptr, nullptr};
  // two-deep pipelined host entry point (ibl_extract_host_submit / _wait): per slot an input staging buffer, an
  // output staging buffer, "H2D done" and "slot done" events
  DevBuf pipe_in[2], pipe_out[2], pipe_pool[2];
  cudaEvent_t pipe_h2d[2] = {nullptr, nullptr}, pipe_done[2] = {nullptr, nullptr};
  bool pipe_busy[2] = {false, false};
};

// conv5_3 output as bf16 hi/lo planes (fused-NetVLAD path)
struct FeatPlanes {
  __nv_bfloat16* hi = nullptr;
  __nv_bfloat16* lo = nullptr;
  int ssq_parts = 0;
};

namespace {

inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// arrival counters of the fused NetVLAD kernel: zeroed when (re)allocated, left at zero by every launch
int ensure_tickets(ibl_engine* e, int n_images, cudaStream_t s) {
  const size_t need = (size_t)(n_images > 1024 ? n_images : 1024) * sizeof(int);
  if (e->nv_ticket.cap >= need) return IBL_OK;
  IBL_RET(e->nv_ticket.ensure(need));
  IBL_CUDA_OK(cudaMemsetAsync(e->nv_ticket.p, 0, e->nv_ticket.cap, s));
  return IBL_OK;
}

int vgg_forward_impl(ibl_engine* e, const float* x, int N, int H, int W, float* feat_nhwc,
                     cudaStream_t s, FeatPlanes* planes_out = nullptr, int last_layer = 12) {
  // largest activation: conv1_x output, N*H*W*64 values of 4 bytes (fp32, or bf16 hi + bf16 lo)
  const size_t act_bytes = (size_t)N * H * W * 64 * 4;
  IBL_RET(e->act[0].ensure(act_bytes));
  IBL_RET(e->act[1].ensure(act_bytes));
  int h = H, w = W;
  int cur = 0;
  if (e->conv_mode == IBL_CONV_SIMT_FP32) {
    IBL_RET(launch_conv1_1(x, e->conv[0], N, h, w, false, e->act[0].as<float>(), nullptr, nullptr, s));
    e->launches++;
    for (int l = 1; l <= last_layer; ++l) {
      const ConvLayer& L = kVgg16[l];
      const bool last = (l == last_layer);
      float* dst = (last && !L.pool) ? feat_nhwc : e->act[cur ^ 1].as<float>();
      IBL_RET(launch_conv3x3_simt(e->act[cur].as<float>(), e->conv[l], N, h, w, L.cin, L.cout, L.relu, dst, s));
      e->launches++;
      cur ^= 1;
      if (L.pool) {
        IBL_RET(launch_maxpool2x2(e->act[cur].as<float>(), N, h, w, L.cout, last ? feat_nhwc : e->act[cur ^ 1].as<float>(), s));
        e->launches++;
        cur ^= 1;
        h /= 2;
        w /= 2;
      }
    }
    return IBL_OK;
  }
  // tcgen05 path: activations are two bf16 planes, hi then lo, each `plane` elements apart
  auto hi_of = [&](int b, size_t elems) { (void)elems; return e->act[b].as<__nv_bfloat16>(); };
  auto lo_of = [&](int b, size_t elems) { return e->act[b].as<__nv_bfloat16>() + elems; };
  size_t elems = (size_t)N * h * w * 64;
  int first_l = 1;
  // conv1_1 + conv1_2 + pool in one kernel (tc_conv.cu: conv1_fused_tc_kernel): the 2.5 GB conv1_1 activation never
  // goes to HBM.  IBL_CONV1_FUSED=0 keeps the two separate kernels (A/B measurements, variant tests).
  static const bool fused1_env = [] { const char* v = getenv("IBL_CONV1_FUSED"); return !v || atoi(v) != 0; }();
  const bool fused1 = fused1_env && last_layer >= 2 && h >= 2 && w >= 2;
  if (fused1) {
    const size_t out_elems = (size_t)N * (h / 2) * (w / 2) * 64;
    IBL_RET(launch_conv1_fused_tc(x, e->w0_oihw, e->conv[0].bias, e->conv[1], N, h, w, hi_of(1, out_elems),
                                  lo_of(1, out_elems), s));
    e->launches++;
    cur = 1;
    h /= 2;
    w /= 2;
    first_l = 2;
  } else {
    static int simt1 = -1;   // IBL_CONV1_SIMT=1: keep conv1_1 on the CUDA cores (A/B experiments)
    if (simt1 < 0) { const char* v = getenv("IBL_CONV1_SIMT"); simt1 = (v && atoi(v)) ? 1 : 0; }
    if (simt1)
      IBL_RET(launch_conv1_1(x, e->conv[0], N, h, w, true, nullptr, hi_of(0, elems), lo_of(0, elems), s));
    else
      IBL_RET(launch_conv1_1_tc(x, e->w0_oihw, e->conv[0].bias, N, h, w, hi_of(0, elems), lo_of(0, elems), s));
    e->launches++;
  }
  for (int l = first_l; l <= last_layer; ++l) {
    const ConvLayer& L = kVgg16[l];
    const bool last = (l == last_layer);
    const size_t in_elems = (size_t)N * h * w * L.cin;
    const int oh = L.pool ? h / 2 : h, ow = L.pool ? w / 2 : w;
    const size_t out_elems = (size_t)N * oh * ow * L.cout;
    if (last && planes_out) {
      // fused-NetVLAD path: conv5_3 leaves hi/lo planes + per-pixel |x|^2 partials instead of fp32
      IBL_RET(e->ssq.ensure((size_t)8 * N * oh * ow * sizeof(float)));
      IBL_RET(launch_conv3x3_tc(hi_of(cur, in_elems), lo_of(cur, in_elems), e->conv[l], N, h, w, L.cin,
                                L.cout, L.relu, L.pool, hi_of(cur ^ 1, out_elems), lo_of(cur ^ 1, out_elems),
                                nullptr, s, e->ssq.as<float>(), &planes_out->ssq_parts));
      planes_out->hi = hi_of(cur ^ 1, out_elems);
      planes_out->lo = lo_of(cur ^ 1, out_elems);
      e->launches++;
      return IBL_OK;
    }
    IBL_RET(launch_conv3x3_tc(hi_of(cur, in_elems), lo_of(cur, in_elems), e->conv[l], N, h, w, L.cin,
                              L.cout, L.relu, L.pool, last ? nullptr : hi_of(cur ^ 1, out_elems),
                              last ? nullptr : lo_of(cur ^ 1, out_elems), last ? feat_nhwc : nullptr, s));
    e->launches++;
    cur ^= 1;
    h = oh;
    w = ow;
  }
  return IBL_OK;
}

}  // namespace

extern "C" {

int ibl_abi_version(void) { return IBLB200_ABI_VERSION; }

const char* ibl_status_string(int status) {
  switch (status) {
    case IBL_OK: return "ok";
    case IBL_ERR_BAD_ARG: return "bad argument";
    case IBL_ERR_NOT_READY: return "parameters for this stage were not set";
    case IBL_ERR_CUDA: return "CUDA error";
    case IBL_ERR_NO_DEVICE: return "no usable sm_100 CUDA device (this library has no CPU fallback)";
    case IBL_ERR_OOM: return "out of device memory";
    case IBL_ERR_UNSUPPORTED: return "unsupported request";
    default: return "unknown status";
  }
}

const char* ibl_last_error(void) { return g_last_error.c_str(); }

int ibl_engine_create(int device, ibl_engine** out) {
  if (!out) return IBL_ERR_BAD_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
    cudaGetLastError();
    set_last_error("no CUDA device visible; libiblb200 has no CPU fallback");
    return IBL_ERR_NO_DEVICE;
  }
  IBL_REQUIRE(device >= 0 && device < count, "device index out of range");
  cudaDeviceProp prop;
  IBL_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_last_error(std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                   std::to_string(prop.minor) + "; this library is built for sm_100a only");
    return IBL_ERR_NO_DEVICE;
  }
  ibl_engine* e = new (std::nothrow) ibl_engine();
  if (!e) return IBL_ERR_OOM;
  e->device = device;
  *out = e;
  return IBL_OK;
}

int ibl_engine_destroy(ibl_engine* e) {
  if (!e) return IBL_OK;
  DeviceGuard g(e->device);
  for (auto& c : e->conv) {
    if (c.w_tck) cudaFree(c.w_tck);
    if (c.bias) cudaFree(c.bias);
    if (c.w_hi) cudaFree(c.w_hi);
    if (c.w_lo) cudaFree(c.w_lo);
  }
  if (e->w0_oihw) cudaFree(e->w0_oihw);
  if (e->copy_stream) { cudaStreamDestroy(e->copy_stream); cudaEventDestroy(e->copy_ev[0]); cudaEventDestroy(e->copy_ev[1]); }
  for (int i = 0; i < 2; ++i) {
    if (e->pipe_h2d[i]) cudaEventDestroy(e->pipe_h2d[i]);
    if (e->pipe_done[i]) cudaEventDestroy(e->pipe_done[i]);
    e->pipe_in[i].release(); e->pipe_out[i].release(); e->pipe_pool[i].release();
  }
  DevBuf* bufs[] = {&e->act[0], &e->act[1], &e->feat, &e->nv_assign, &e->nv_inv, &e->nv_raw, &e->vlad,
                    &e->pca_partial, &e->qn, &e->dbn, &e->dist_chunk, &e->cand_d, &e->cand_i,
                    &e->stage_in, &e->stage_out, &e->stage_out2, &e->stage_u8, &e->q_pl, &e->db_pl, &e->v_pl, &e->pca_pl,
                    &e->mrg_d, &e->mrg_i, &e->d1_ws, &e->dguard, &e->bw_g, &e->bw_x, &e->bw_part, &e->bw_w, &e->ssq, &e->nv_part, &e->nv_asum, &e->nvw_pl, &e->nv_ticket};
  for (DevBuf* b : bufs) b->release();
  delete e;
  return IBL_OK;
}

int ibl_engine_set_conv_mode(ibl_engine* e, int mode) {
  IBL_REQUIRE(e, "null engine");
  IBL_REQUIRE(mode == IBL_CONV_SIMT_FP32 || mode == IBL_CONV_TC_BF16X3, "unknown conv mode");
  e->conv_mode = mode;
  return IBL_OK;
}
int ibl_engine_get_conv_mode(ibl_engine* e, int* mode) {
  IBL_REQUIRE(e && mode, "null argument");
  *mode = e->conv_mode;
  return IBL_OK;
}
int ibl_engine_set_gemm_mode(ibl_engine* e, int mode) {
  IBL_REQUIRE(e, "null engine");
  IBL_REQUIRE(mode == IBL_CONV_SIMT_FP32 || mode == IBL_CONV_TC_BF16X3, "unknown gemm mode");
  e->gemm_mode = mode;
  return IBL_OK;
}
int ibl_engine_launch_count(ibl_engine* e, uint64_t* count) {
  IBL_REQUIRE(e && count, "null argument");
  *count = e->launches;
  return IBL_OK;
}

int ibl_engine_set_vgg16(ibl_engine* e, const float* const* w13, const float* const* b13, void* stream) {
  IBL_REQUIRE(e && w13 && b13, "null argument");
  DeviceGuard g(e->device);
  for (int l = 0; l < 13; ++l) {
    IBL_REQUIRE(w13[l] && b13[l], "null weight/bias pointer");
    const ConvLayer& L = kVgg16[l];
    ConvParams& p = e->conv[l];
    const size_t nw = (size_t)L.cout * L.cin * 9;
    if (!p.w_tck) IBL_CUDA_OK(cudaMalloc(&p.w_tck, nw * sizeof(float)));
    if (!p.bias) IBL_CUDA_OK(cudaMalloc(&p.bias, L.cout * sizeof(float)));
    if (L.cin % 64 == 0) {
      if (!p.w_hi) IBL_CUDA_OK(cudaMalloc(&p.w_hi, nw * sizeof(__nv_bfloat16)));
      if (!p.w_lo) IBL_CUDA_OK(cudaMalloc(&p.w_lo, nw * sizeof(__nv_bfloat16)));
      p.cin_pad = L.cin;
    }
    IBL_RET(launch_repack_weights(w13[l], L.cout, L.cin, p, S(stream)));
    IBL_CUDA_OK(cudaMemcpyAsync(p.bias, b13[l], L.cout * sizeof(float), cudaMemcpyDeviceToDevice, S(stream)));
    if (l == 0) {
      if (!e->w0_oihw) IBL_CUDA_OK(cudaMalloc(&e->w0_oihw, nw * sizeof(float)));
      IBL_CUDA_OK(cudaMemcpyAsync(e->w0_oihw, w13[0], nw * sizeof(float), cudaMemcpyDeviceToDevice, S(stream)));
    }
    e->launches++;
  }
  e->vgg_ready = true;
  return IBL_OK;
}

int ibl_engine_set_netvlad(ibl_engine* e, const float* conv_w, const float* centroids, int K, int C,
                           void* stream) {
  IBL_REQUIRE(e && conv_w && centroids, "null argument");
  IBL_REQUIRE(K == 64, "NetVLAD kernels are built for K=64 clusters");
  IBL_REQUIRE(C >= 4 && C % 4 == 0, "NetVLAD dim must be a positive multiple of 4");
  e->nv_w = conv_w;
  e->nv_c = centroids;
  e->nv_K = K;
  e->nv_C = C;
  e->nvw_pl_src = nullptr;
  if (K == 64 && C == 512) {
    DeviceGuard g(e->device);
    const size_t n = (size_t)K * C;
    IBL_RET(e->nvw_pl.ensure(n * 4));
    IBL_RET(launch_f32_to_planes(conv_w, n, e->nvw_pl.as<__nv_bfloat16>(), e->nvw_pl.as<__nv_bfloat16>() + n, S(stream)));
    e->launches++;
    e->nvw_pl_src = conv_w;
  }
  return IBL_OK;
}

int ibl_engine_set_pca(ibl_engine* e, const float* W, const float* b, int P, int D, void* stream) {
  (void)stream;
  IBL_REQUIRE(e && W && b, "null argument");
  IBL_REQUIRE(P >= 1 && D >= 4 && D % 4 == 0, "bad PCA shape");
  e->pca_W = W;
  e->pca_b = b;
  e->pca_P = P;
  e->pca_D = D;
  e->pca_pl_src = nullptr;
  if (D % 64 == 0) {
    DeviceGuard g(e->device);
    const size_t n = (size_t)P * D;
    IBL_RET(e->pca_pl.ensure(n * 4));
    IBL_RET(launch_f32_to_planes(W, n, e->pca_pl.as<__nv_bfloat16>(), e->pca_pl.as<__nv_bfloat16>() + n, S(stream)));
    e->launches++;
    e->pca_pl_src = W;
  }
  return IBL_OK;
}

int ibl_vgg16_forward(ibl_engine* e, const float* x, int N, int H, int W, float* feat_nhwc,
                      float* feat_nchw, float* pool, void* stream) {
  IBL_REQUIRE(e && x, "null argument");
  IBL_REQUIRE(N >= 1 && H >= 16 && W >= 16, "VGG16 trunk needs N>=1 and H,W>=16");
  if (!e->vgg_ready) { set_last_error("ibl_engine_set_vgg16 was not called"); return IBL_ERR_NOT_READY; }
  DeviceGuard g(e->device);
  const int fh = H / 16, fw = W / 16;
  const size_t fbytes = (size_t)N * fh * fw * 512 * sizeof(float);
  float* f = feat_nhwc;
  if (!f) {
    IBL_RET(e->feat.ensure(fbytes));
    f = e->feat.as<float>();
  }
  IBL_RET(vgg_forward_impl(e, x, N, H, W, f, S(stream)));
  if (feat_nchw) { IBL_RET(launch_nhwc_to_nchw(f, N, fh * fw, 512, feat_nchw, S(stream))); e->launches++; }
  if (pool) { IBL_RET(launch_global_maxpool_nhwc(f, N, fh * fw, 512, pool, S(stream))); e->launches++; }
  return IBL_OK;
}

// ---- training surface of the trunk (SURVEY 8 f1, config 5): frozen prefix, per-layer forward and backward --------
// Layers are numbered 0..12 (conv1_1 .. conv5_3).  Activations cross this boundary as fp32 NHWC.

// Frozen prefix: conv layers [0, n_layers) with their ReLUs and pools (inference kernels, nothing saved).
// out_nhwc: [N, h, w, C] of the activation that enters layer n_layers.
int ibl_vgg16_prefix_forward(ibl_engine* e, const float* x, int N, int H, int W, int n_layers, float* out_nhwc,
                             void* stream) {
  IBL_REQUIRE(e && x && out_nhwc, "null argument");
  IBL_REQUIRE(n_layers >= 1 && n_layers <= 13, "prefix length must be 1..13");
  IBL_REQUIRE(N >= 1 && H >= 16 && W >= 16, "VGG16 trunk needs N>=1 and H,W>=16");
  if (!e->vgg_ready) { set_last_error("ibl_engine_set_vgg16 was not called"); return IBL_ERR_NOT_READY; }
  DeviceGuard g(e->device);
  if (n_layers == 1) {
    e->launches++;
    return launch_conv1_1(x, e->conv[0], N, H, W, false, out_nhwc, nullptr, nullptr, S(stream));
  }
  return vgg_forward_impl(e, x, N, H, W, out_nhwc, S(stream), nullptr, n_layers - 1);
}

// One trainable layer forward: y = [ReLU](conv(x) + b), NO pooling (the caller pools, so that the pre-pool
// activation is available to the backward).  layer 0 takes the NCHW image, layers >= 1 fp32 NHWC.
int ibl_vgg16_layer_forward(ibl_engine* e, int layer, const float* x, int N, int H, int W, float* y_nhwc, void* stream) {
  IBL_REQUIRE(e && x && y_nhwc, "null argument");
  IBL_REQUIRE(layer >= 0 && layer < 13 && N >= 1 && H >= 1 && W >= 1, "bad layer / shape");
  if (!e->vgg_ready) { set_last_error("ibl_engine_set_vgg16 was not called"); return IBL_ERR_NOT_READY; }
  DeviceGuard g(e->device);
  cudaStream_t s = S(stream);
  const ConvLayer& L = kVgg16[layer];
  if (layer == 0) {
    e->launches++;
    return launch_conv1_1(x, e->conv[0], N, H, W, false, y_nhwc, nullptr, nullptr, s);
  }
  if (e->conv_mode == IBL_CONV_SIMT_FP32) {
    e->launches++;
    return launch_conv3x3_simt(x, e->conv[layer], N, H, W, L.cin, L.cout, L.relu, y_nhwc, s);
  }
  const size_t in_e = (size_t)N * H * W * L.cin;
  IBL_RET(e->act[0].ensure(in_e * 4));
  __nv_bfloat16* xh = e->act[0].as<__nv_bfloat16>();
  IBL_RET(launch_f32_to_planes(x, in_e, xh, xh + in_e, s));
  IBL_RET(launch_conv3x3_tc(xh, xh + in_e, e->conv[layer], N, H, W, L.cin, L.cout, L.relu, false, nullptr, nullptr,
                            y_nhwc, s));
  e->launches += 2;
  return IBL_OK;
}

int ibl_maxpool2x2_forward(ibl_engine* e, const float* x_nhwc, int N, int H, int W, int C, float* y_nhwc, void* stream) {
  IBL_REQUIRE(e && x_nhwc && y_nhwc && N >= 1 && H >= 2 && W >= 2 && C >= 4 && C % 4 == 0, "bad argument");
  DeviceGuard g(e->device);
  e->launches++;
  return launch_maxpool2x2(x_nhwc, N, H, W, C, y_nhwc, S(stream));
}

int ibl_maxpool2x2_backward(ibl_engine* e, const float* x_nhwc, const float* gy_nhwc, int N, int H, int W, int C,
                            float* gx_nhwc, void* stream) {
  IBL_REQUIRE(e && x_nhwc && gy_nhwc && gx_nhwc && N >= 1 && H >= 2 && W >= 2 && C >= 1, "bad argument");
  DeviceGuard g(e->device);
  e->launches++;
  return launch_maxpool2x2_bwd(x_nhwc, gy_nhwc, N, H, W, C, gx_nhwc, S(stream));
}

// Backward of one trainable layer.  x: the layer's input (fp32 NHWC; NCHW image for layer 0), y: its post-ReLU,
// pre-pool output (only read when the layer has a ReLU), gy: dL/dy.  Outputs: gx (dL/dx, nullable -- not needed for
// the first trainable layer), gw [Cout,Cin,3,3] (OIHW, the parameter's layout), gb [Cout].
int ibl_vgg16_layer_backward(ibl_engine* e, int layer, const float* x, const float* y, const float* gy, int N, int H,
                             int W, float* gx, float* gw, float* gb, void* stream) {
  IBL_REQUIRE(e && x && gy && gw && gb, "null argument");
  IBL_REQUIRE(layer >= 0 && layer < 13 && N >= 1 && H >= 1 && W >= 1, "bad layer / shape");
  if (!e->vgg_ready) { set_last_error("ibl_engine_set_vgg16 was not called"); return IBL_ERR_NOT_READY; }
  const ConvLayer& L = kVgg16[layer];
  IBL_REQUIRE(!L.relu || y, "the layer has a ReLU: its output is needed for the mask");
  DeviceGuard g(e->device);
  cudaStream_t s = S(stream);
  const size_t out_e = (size_t)N * H * W * L.cout, in_e = (size_t)N * H * W * L.cin;
  // dY (after the ReLU mask) as bf16 hi/lo planes: the operand of dgrad, wgrad and the bias gradient
  IBL_RET(e->bw_g.ensure(out_e * 4));
  __nv_bfloat16* gh = e->bw_g.as<__nv_bfloat16>();
  IBL_RET(launch_relu_mask_planes(gy, y, out_e, L.relu, gh, gh + out_e, s));
  e->launches++;
  if (layer == 0) {
    IBL_REQUIRE(!gx, "conv1_1 has no input gradient (its input is the image)");
    IBL_RET(e->bw_part.ensure((size_t)1024 * 64 * 28 * sizeof(float)));
    IBL_RET(launch_conv1_1_wgrad(x, gh, gh + out_e, N, H, W, e->bw_part.as<float>(), gw, gb, s));
    e->launches += 2;
    return IBL_OK;
  }
  IBL_RET(e->bw_x.ensure(in_e * 4));
  __nv_bfloat16* xh = e->bw_x.as<__nv_bfloat16>();
  IBL_RET(launch_f32_to_planes(x, in_e, xh, xh + in_e, s));
  const int splits = wgrad_tc_splits(N, H, W, L.cin, L.cout);
  IBL_RET(e->bw_part.ensure(((size_t)splits * 9 * L.cout * L.cin + (size_t)256 * L.cout) * sizeof(float)));
  float* part = e->bw_part.as<float>();
  IBL_RET(launch_conv_wgrad_tc(gh, gh + out_e, xh, xh + in_e, N, H, W, L.cin, L.cout, part, splits,
                               part + (size_t)splits * 9 * L.cout * L.cin, gw, gb, s));
  e->launches += 5;
  if (gx) {
    // dgrad = the forward implicit-GEMM kernel on dY with the 180-degree-rotated, role-swapped filter bank
    const size_t nw = (size_t)L.cout * L.cin * 9;
    IBL_RET(e->bw_w.ensure(nw * 4 + (size_t)L.cin * sizeof(float)));
    ConvParams p;
    p.w_hi = e->bw_w.as<__nv_bfloat16>();
    p.w_lo = p.w_hi + nw;
    p.bias = reinterpret_cast<float*>(p.w_lo + nw);
    p.cin_pad = L.cout;
    IBL_CUDA_OK(cudaMemsetAsync(p.bias, 0, (size_t)L.cin * sizeof(float), s));
    IBL_RET(launch_repack_weights_dgrad(e->conv[layer].w_tck, L.cout, L.cin, p.w_hi, p.w_lo, s));
    IBL_RET(launch_conv3x3_tc(gh, gh + out_e, p, N, H, W, L.cout, L.cin, false, false, nullptr, nullptr, gx, s));
    e->launches += 2;
  }
  return IBL_OK;
}

int ibl_netvlad_forward(ibl_engine* e, const float* feat, int nhwc, int N, int C, int S_, const float* conv_w,
                        const float* centroids, int K, int normalize_input, float* vlad_raw,
                        float* vlad_norm, void* stream) {
  IBL_REQUIRE(e && feat && conv_w && centroids, "null argument");
  IBL_REQUIRE(N >= 1 && C >= 1 && S_ >= 1, "empty NetVLAD input");
  IBL_REQUIRE(K == 64, "NetVLAD kernels are built for K=64 clusters");
  IBL_REQUIRE(vlad_raw || vlad_norm, "no output requested");
  DeviceGuard g(e->device);
  if (nhwc && C == 512 && K == 64 && e->gemm_mode == IBL_CONV_TC_BF16X3) {
    cudaStream_t s = S(stream);
    const size_t ne = (size_t)N * S_ * C, nw = (size_t)K * C;
    IBL_RET(e->v_pl.ensure(ne * 4));
    IBL_RET(e->q_pl.ensure(nw * 4));
    IBL_RET(e->ssq.ensure((size_t)N * S_ * sizeof(float)));
    __nv_bfloat16 *xh = e->v_pl.as<__nv_bfloat16>(), *wh = e->q_pl.as<__nv_bfloat16>();
    IBL_RET(launch_f32_to_planes(feat, ne, xh, xh + ne, s));
    IBL_RET(launch_f32_to_planes(conv_w, nw, wh, wh + nw, s));
    IBL_RET(launch_row_sqnorm(feat, N * S_, C, e->ssq.as<float>(), s));
    const int G = netvlad_tc_units(N, S_);
    IBL_RET(e->nv_part.ensure((size_t)N * G * 64 * 512 * sizeof(float)));
    IBL_RET(e->nv_asum.ensure((size_t)N * G * 64 * sizeof(float)));
    IBL_RET(ensure_tickets(e, N, s));
    IBL_RET(launch_netvlad_tc(xh, xh + ne, N, S_, wh, wh + nw, e->ssq.as<float>(), 1, centroids,
                              normalize_input != 0, e->nv_part.as<float>(), e->nv_asum.as<float>(),
                              e->nv_ticket.as<int>(), vlad_raw, vlad_norm, s));
    e->launches += 4;
    return IBL_OK;
  }
  IBL_RET(e->nv_assign.ensure((size_t)N * S_ * K * sizeof(float)));
  IBL_RET(e->nv_inv.ensure((size_t)N * S_ * sizeof(float)));
  float* raw = vlad_raw;
  if (!raw) {
    IBL_RET(e->nv_raw.ensure((size_t)N * K * C * sizeof(float)));
    raw = e->nv_raw.as<float>();
  }
  return launch_netvlad(feat, nhwc != 0, N, C, S_, conv_w, centroids, K, normalize_input != 0,
                        e->nv_assign.as<float>(), e->nv_inv.as<float>(), nullptr, raw, vlad_norm,
                        S(stream), &e->launches);
}

int ibl_netvlad_backward(ibl_engine* e, const float* feat, int nhwc, int N, int C, int S_, const float* conv_w,
                         const float* centroids, int K, int normalize_input, const float* grad_vlad,
                         float* grad_feat, float* grad_conv_w, float* grad_centroids, void* stream) {
  IBL_REQUIRE(e && feat && conv_w && centroids && grad_vlad && grad_feat && grad_conv_w && grad_centroids,
              "null argument");
  IBL_REQUIRE(N >= 1 && C >= 64 && S_ >= 1, "empty NetVLAD input");
  IBL_REQUIRE(K == 64, "NetVLAD kernels are built for K=64 clusters");
  DeviceGuard g(e->device);
  const int splits = 64;
  IBL_RET(e->nv_assign.ensure((size_t)N * S_ * K * sizeof(float)));
  IBL_RET(e->nv_inv.ensure((size_t)N * S_ * sizeof(float)));
  IBL_RET(e->nv_raw.ensure((size_t)N * S_ * K * sizeof(float)));                 // dz
  IBL_RET(e->nv_part.ensure((size_t)splits * K * C * sizeof(float)));            // dW partials
  return launch_netvlad_backward(feat, nhwc != 0, N, C, S_, conv_w, centroids, grad_vlad, normalize_input != 0,
                                 e->nv_assign.as<float>(), e->nv_inv.as<float>(), e->nv_raw.as<float>(),
                                 e->nv_part.as<float>(), splits, grad_feat, grad_conv_w, grad_centroids, S(stream),
                                 &e->launches);
}

int ibl_vlad_normalize(ibl_engine* e, const float* vlad_raw, int N, int K, int C, float* out, void* stream) {
  IBL_REQUIRE(e && vlad_raw && out, "null argument");
  IBL_REQUIRE(N >= 1 && K >= 1 && C >= 1 && K <= 4096, "bad shape");
  DeviceGuard g(e->device);
  e->launches++;
  return launch_vlad_normalize(vlad_raw, N, K, C, out, S(stream));
}

int ibl_pca_l2(ibl_engine* e, const float* v, int N, int D, const float* W, const float* b, int P,
               float* out, void* stream) {
  IBL_REQUIRE(e && v && W && b && out, "null argument");
  IBL_REQUIRE(N >= 1 && P >= 1 && D >= 4, "bad shape");
  IBL_REQUIRE((size_t)P * sizeof(float) <= 48 * 1024, "PCA output dim above 12288 is not supported");
  DeviceGuard g(e->device);
  if (e->gemm_mode == IBL_CONV_TC_BF16X3 && W == e->pca_pl_src && P == e->pca_P && D == e->pca_D) {
    const size_t nw = (size_t)P * D;
    const int splits = pca_tc_splits(P, D);
    for (int n0 = 0; n0 < N; n0 += 32) {
      const int nb = N - n0 < 32 ? N - n0 : 32;
      const size_t nv = (size_t)nb * D;
      IBL_RET(e->v_pl.ensure(nv * 4));
      IBL_RET(e->pca_partial.ensure((size_t)splits * nb * P * sizeof(float)));
      __nv_bfloat16* vh = e->v_pl.as<__nv_bfloat16>();
      IBL_RET(launch_f32_to_planes(v + (size_t)n0 * D, nv, vh, vh + nv, S(stream)));
      int sp = 0;
      IBL_RET(launch_pca_partial_tc(e->pca_pl.as<__nv_bfloat16>(), e->pca_pl.as<__nv_bfloat16>() + nw, P, vh,
                                    vh + nv, nb, D, e->pca_partial.as<float>(), &sp, S(stream)));
      IBL_RET(launch_pca_finalize(e->pca_partial.as<float>(), sp, nb, P, b, out + (size_t)n0 * P, S(stream)));
      e->launches += 3;
    }
    return IBL_OK;
  }
  // enough K-splits to fill the machine: tiles = ceil(P/128)*ceil(N/64)*splits >= ~2 waves of 148 SMs
  int tiles = cdiv(P, 128) * cdiv(N, 64);
  int splits = cdiv(2 * 148, tiles);
  if (splits < 1) splits = 1;
  if (splits > 32) splits = 32;
  while (splits > 1 && D / splits < 256) --splits;
  IBL_RET(e->pca_partial.ensure((size_t)splits * N * P * sizeof(float)));
  return launch_pca_l2(v, N, D, W, b, P, e->pca_partial.as<float>(), splits, out, S(stream), &e->launches);
}

int ibl_l2_normalize_rows(ibl_engine* e, const float* x, int N, int D, float* out, void* stream) {
  IBL_REQUIRE(e && x && out, "null argument");
  IBL_REQUIRE(N >= 0 && D >= 1, "bad shape");
  DeviceGuard g(e->device);
  e->launches++;
  return launch_l2_normalize_rows(x, N, D, out, S(stream));
}

int ibl_extract(ibl_engine* e, const float* x, int N, int H, int W, unsigned flags, float* out,
                float* pool, void* stream) {
  IBL_REQUIRE(e && x && out, "null argument");
  IBL_REQUIRE(flags & IBL_OUT_VLAD, "ibl_extract: IBL_OUT_VLAD is required");
  IBL_REQUIRE(!(flags & IBL_OUT_POOL) || pool, "IBL_OUT_POOL needs a pool buffer");
  IBL_REQUIRE(N >= 1 && H >= 16 && W >= 16, "VGG16 trunk needs N>=1 and H,W>=16");
  if (!e->vgg_ready || !e->nv_w) { set_last_error("VGG16 / NetVLAD parameters were not set"); return IBL_ERR_NOT_READY; }
  const bool pca = (flags & IBL_OUT_PCA) != 0;
  if (pca && !e->pca_W) { set_last_error("PCA parameters were not set"); return IBL_ERR_NOT_READY; }
  IBL_REQUIRE(e->nv_C == 512, "NetVLAD dim must match the VGG16 feature dim (512)");
  DeviceGuard g(e->device);
  const int fh = H / 16, fw = W / 16, Sp = fh * fw;
  const int K = e->nv_K, C = e->nv_C, D = K * C;
  if (pca) IBL_REQUIRE(e->pca_D == D, "PCA input dim must equal K*C");
  const int out_dim = pca ? e->pca_P : D;
  // micro-batches bound the workspace (157 MB / image at 480x640)
  const int MB = 32;
  for (int n0 = 0; n0 < N; n0 += MB) {
    const int nb = (N - n0 < MB) ? (N - n0) : MB;
    const float* xb = x + (size_t)n0 * 3 * H * W;
    float* vdst = out + (size_t)n0 * out_dim;
    if (pca) {
      IBL_RET(e->vlad.ensure((size_t)nb * D * sizeof(float)));
      vdst = e->vlad.as<float>();
    }
    const bool fused = e->conv_mode == IBL_CONV_TC_BF16X3 && e->gemm_mode == IBL_CONV_TC_BF16X3 &&
                       e->nvw_pl_src == e->nv_w && K == 64 && C == 512;
    if (fused) {
      // conv5_3 -> hi/lo planes + |x|^2 partials -> one tcgen05 NetVLAD kernel (+ finalize)
      FeatPlanes fp;
      IBL_RET(vgg_forward_impl(e, xb, nb, H, W, nullptr, S(stream), &fp));
      if (flags & IBL_OUT_POOL) {
        IBL_RET(launch_global_maxpool_planes(fp.hi, fp.lo, nb, Sp, 512, pool + (size_t)n0 * 512, S(stream)));
        e->launches++;
      }
      const int G = netvlad_tc_units(nb, Sp);
      IBL_RET(e->nv_part.ensure((size_t)nb * G * 64 * 512 * sizeof(float)));
      IBL_RET(e->nv_asum.ensure((size_t)nb * G * 64 * sizeof(float)));
      IBL_RET(ensure_tickets(e, nb, S(stream)));
      const size_t nw = (size_t)64 * 512;
      IBL_RET(launch_netvlad_tc(fp.hi, fp.lo, nb, Sp, e->nvw_pl.as<__nv_bfloat16>(), e->nvw_pl.as<__nv_bfloat16>() + nw,
                                e->ssq.as<float>(), fp.ssq_parts, e->nv_c, true, e->nv_part.as<float>(),
                                e->nv_asum.as<float>(), e->nv_ticket.as<int>(), nullptr, vdst, S(stream)));
      e->launches += 1;                     // ONE launch: partials, centroid term, intra-norm and L2 inside the kernel
    } else {
      IBL_RET(e->feat.ensure((size_t)nb * Sp * 512 * sizeof(float)));
      IBL_RET(vgg_forward_impl(e, xb, nb, H, W, e->feat.as<float>(), S(stream)));
      if (flags & IBL_OUT_POOL) {
        IBL_RET(launch_global_maxpool_nhwc(e->feat.as<float>(), nb, Sp, 512, pool + (size_t)n0 * 512, S(stream)));
        e->launches++;
      }
      IBL_RET(ibl_netvlad_forward(e, e->feat.as<float>(), 1, nb, C, Sp, e->nv_w, e->nv_c, K, 1, nullptr, vdst, stream));
    }
    if (pca)
      IBL_RET(ibl_pca_l2(e, vdst, nb, D, e->pca_W, e->pca_b, e->pca_P, out + (size_t)n0 * out_dim, stream));
  }
  return IBL_OK;
}

int ibl_extract_host(ibl_engine* e, const float* x_host, int N, int H, int W, unsigned flags,
                     float* out_host, float* pool_host, void* stream) {
  IBL_REQUIRE(e && x_host && out_host, "null argument");
  IBL_REQUIRE(N >= 1 && H >= 16 && W >= 16, "VGG16 trunk needs N>=1 and H,W>=16");
  DeviceGuard g(e->device);
  const bool pca = (flags & IBL_OUT_PCA) != 0;
  const int out_dim = pca ? e->pca_P : e->nv_K * e->nv_C;
  const size_t in_bytes = (size_t)N * 3 * H * W * sizeof(float);
  IBL_RET(e->stage_in.ensure(in_bytes));
  IBL_RET(e->stage_out.ensure((size_t)N * out_dim * sizeof(float)));
  if (flags & IBL_OUT_POOL) IBL_RET(e->stage_out2.ensure((size_t)N * 512 * sizeof(float)));
  // Two half-batches: the H2D copy of the second half runs on the engine's copy stream while the
  // first half is being computed (the reference serialises .cuda() and the forward, evaluators.py:24).
  const int halves = N >= 16 ? 2 : 1;
  if (!e->copy_stream) {
    IBL_CUDA_OK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->copy_ev[0], cudaEventDisableTiming));
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->copy_ev[1], cudaEventDisableTiming));
  }
  const size_t img_elems = (size_t)3 * H * W;
  // uneven split: only the first (small) part's copy is exposed; the rest streams in behind its compute
  static const int split_div = [] { const char* v = getenv("IBL_HOST_SPLIT"); const int d = v ? atoi(v) : 0; return d >= 2 ? d : 4; }();
  const int n_first = halves == 2 ? (N / split_div > 0 ? N / split_div : 1) : N;
  for (int i = 0; i < halves; ++i) {
    const int n0 = i == 0 ? 0 : n_first, nb = i == 0 ? n_first : N - n_first;
    IBL_CUDA_OK(cudaMemcpyAsync(e->stage_in.as<float>() + n0 * img_elems, x_host + n0 * img_elems,
                                nb * img_elems * sizeof(float), cudaMemcpyHostToDevice, e->copy_stream));
    IBL_CUDA_OK(cudaEventRecord(e->copy_ev[i], e->copy_stream));
  }
  for (int i = 0; i < halves; ++i) {
    const int n0 = i == 0 ? 0 : n_first, nb = i == 0 ? n_first : N - n_first;
    IBL_CUDA_OK(cudaStreamWaitEvent(S(stream), e->copy_ev[i], 0));
    IBL_RET(ibl_extract(e, e->stage_in.as<float>() + n0 * img_elems, nb, H, W, flags,
                        e->stage_out.as<float>() + (size_t)n0 * out_dim,
                        (flags & IBL_OUT_POOL) ? e->stage_out2.as<float>() + (size_t)n0 * 512 : nullptr, stream));
  }
  IBL_CUDA_OK(cudaMemcpyAsync(out_host, e->stage_out.p, (size_t)N * out_dim * sizeof(float),
                              cudaMemcpyDeviceToHost, S(stream)));
  if ((flags & IBL_OUT_POOL) && pool_host)
    IBL_CUDA_OK(cudaMemcpyAsync(pool_host, e->stage_out2.p, (size_t)N * 512 * sizeof(float),
                                cudaMemcpyDeviceToHost, S(stream)));
  IBL_CUDA_OK(cudaStreamSynchronize(S(stream)));
  return IBL_OK;
}

// Pipelined host entry point: what a loader loop overlaps by hand in the reference (pin_memory + non_blocking .cuda(),
// evaluators.py:24) -- submit(slot) enqueues H2D of this batch on the engine's copy stream, the extraction behind it
// on the caller's stream and the D2H of the descriptors, and returns WITHOUT synchronising; wait(slot) blocks until
// that batch's descriptors are in out_host.  With two slots the copy of batch i+1 runs under the compute of batch i.
// x_host / out_host (/ pool_host) must stay valid (and should be pinned) until wait(slot) returns.
int ibl_extract_host_submit(ibl_engine* e, int slot, const float* x_host, int N, int H, int W, unsigned flags,
                            float* out_host, float* pool_host, void* stream) {
  IBL_REQUIRE(e && x_host && out_host, "null argument");
  IBL_REQUIRE(slot == 0 || slot == 1, "slot must be 0 or 1");
  IBL_REQUIRE(N >= 1 && H >= 16 && W >= 16, "VGG16 trunk needs N>=1 and H,W>=16");
  IBL_REQUIRE(!e->pipe_busy[slot], "slot is in flight: call ibl_extract_host_wait first");
  DeviceGuard g(e->device);
  const bool pca = (flags & IBL_OUT_PCA) != 0;
  const int out_dim = pca ? e->pca_P : e->nv_K * e->nv_C;
  const size_t in_bytes = (size_t)N * 3 * H * W * sizeof(float), out_bytes = (size_t)N * out_dim * sizeof(float);
  if (!e->copy_stream) {
    IBL_CUDA_OK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->copy_ev[0], cudaEventDisableTiming));
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->copy_ev[1], cudaEventDisableTiming));
  }
  if (!e->pipe_h2d[slot]) {
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->pipe_h2d[slot], cudaEventDisableTiming));
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->pipe_done[slot], cudaEventDisableTiming));
  }
  // growing a buffer frees the old one: make sure nothing of an earlier use of this slot is still running
  if (e->pipe_in[slot].cap < in_bytes || e->pipe_out[slot].cap < out_bytes) IBL_CUDA_OK(cudaEventSynchronize(e->pipe_done[slot]));
  IBL_RET(e->pipe_in[slot].ensure(in_bytes));
  IBL_RET(e->pipe_out[slot].ensure(out_bytes));
  if (flags & IBL_OUT_POOL) IBL_RET(e->pipe_pool[slot].ensure((size_t)N * 512 * sizeof(float)));
  // the copy stream may overwrite this slot's input buffer only after the slot's previous extraction has read it
  IBL_CUDA_OK(cudaStreamWaitEvent(e->copy_stream, e->pipe_done[slot], 0));
  IBL_CUDA_OK(cudaMemcpyAsync(e->pipe_in[slot].p, x_host, in_bytes, cudaMemcpyHostToDevice, e->copy_stream));
  IBL_CUDA_OK(cudaEventRecord(e->pipe_h2d[slot], e->copy_stream));
  IBL_CUDA_OK(cudaStreamWaitEvent(S(stream), e->pipe_h2d[slot], 0));
  IBL_RET(ibl_extract(e, e->pipe_in[slot].as<float>(), N, H, W, flags, e->pipe_out[slot].as<float>(),
                      (flags & IBL_OUT_POOL) ? e->pipe_pool[slot].as<float>() : nullptr, stream));
  IBL_CUDA_OK(cudaMemcpyAsync(out_host, e->pipe_out[slot].p, out_bytes, cudaMemcpyDeviceToHost, S(stream)));
  if ((flags & IBL_OUT_POOL) && pool_host)
    IBL_CUDA_OK(cudaMemcpyAsync(pool_host, e->pipe_pool[slot].p, (size_t)N * 512 * sizeof(float), cudaMemcpyDeviceToHost,
                                S(stream)));
  IBL_CUDA_OK(cudaEventRecord(e->pipe_done[slot], S(stream)));
  e->pipe_busy[slot] = true;
  return IBL_OK;
}

int ibl_extract_host_wait(ibl_engine* e, int slot) {
  IBL_REQUIRE(e, "null engine");
  IBL_REQUIRE(slot == 0 || slot == 1, "slot must be 0 or 1");
  if (!e->pipe_busy[slot]) return IBL_OK;
  DeviceGuard g(e->device);
  IBL_CUDA_OK(cudaEventSynchronize(e->pipe_done[slot]));
  e->pipe_busy[slot] = false;
  return IBL_OK;
}

int ibl_preprocess_u8(ibl_engine* e, const uint8_t* x_nhwc, int N, int H, int W, const float* mean3,
                      const float* std3, float* out_nchw, void* stream) {
  IBL_REQUIRE(e && x_nhwc && mean3 && std3 && out_nchw, "null argument");
  IBL_REQUIRE(N >= 1 && H >= 1 && W >= 1, "empty image batch");
  IBL_REQUIRE(std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f, "zero std");
  DeviceGuard g(e->device);
  e->launches++;
  return launch_u8_hwc_to_nchw_norm(x_nhwc, N, H, W, mean3, std3, out_nchw, S(stream));
}

// T.Resize((H, W)) of the reference's test transform (ibl/utils/data/__init__.py:37-42) on decoded uint8 HWC batches,
// bit-exact with Pillow's bilinear resample.  bounds_* [out,2] and kk_* [out,ksize] are DEVICE int32 tables built by
// the host exactly as Pillow builds them (openibl_b200/utils/data/gpu_resize.py); a pass with equal sizes is skipped.
int ibl_resize_bilinear_u8(ibl_engine* e, const uint8_t* x_nhwc, int N, int Hin, int Win, int Hout, int Wout,
                           const int* bounds_h, const int* kk_h, int ksize_h, const int* bounds_v, const int* kk_v,
                           int ksize_v, uint8_t* out_nhwc, void* stream) {
  IBL_REQUIRE(e && x_nhwc && out_nhwc, "null argument");
  IBL_REQUIRE(N >= 1 && Hin >= 1 && Win >= 1 && Hout >= 1 && Wout >= 1, "empty image batch");
  IBL_REQUIRE(Wout == Win || (bounds_h && kk_h && ksize_h >= 1), "horizontal pass needs its coefficient table");
  IBL_REQUIRE(Hout == Hin || (bounds_v && kk_v && ksize_v >= 1), "vertical pass needs its coefficient table");
  DeviceGuard g(e->device);
  uint8_t* tmp = nullptr;
  if (Wout != Win && Hout != Hin) {
    IBL_RET(e->stage_u8.ensure((size_t)N * Hin * Wout * 3));
    tmp = e->stage_u8.as<uint8_t>();
  }
  return launch_resize_bilinear_u8(x_nhwc, N, Hin, Win, Hout, Wout, bounds_h, kk_h, ksize_h, bounds_v, kk_v, ksize_v, tmp,
                                   out_nhwc, S(stream), &e->launches);
}

int ibl_extract_host_u8(ibl_engine* e, const uint8_t* x_nhwc_host, int N, int H, int W, const float* mean3,
                        const float* std3, unsigned flags, float* out_host, float* pool_host, void* stream) {
  IBL_REQUIRE(e && x_nhwc_host && mean3 && std3 && out_host, "null argument");
  IBL_REQUIRE(N >= 1 && H >= 16 && W >= 16, "VGG16 trunk needs N>=1 and H,W>=16");
  IBL_REQUIRE(std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f, "zero std");
  DeviceGuard g(e->device);
  const bool pca = (flags & IBL_OUT_PCA) != 0;
  const int out_dim = pca ? e->pca_P : e->nv_K * e->nv_C;
  const size_t img_px = (size_t)H * W;
  IBL_RET(e->stage_u8.ensure((size_t)N * img_px * 3));
  IBL_RET(e->stage_in.ensure((size_t)N * img_px * 3 * sizeof(float)));
  IBL_RET(e->stage_out.ensure((size_t)N * out_dim * sizeof(float)));
  if (flags & IBL_OUT_POOL) IBL_RET(e->stage_out2.ensure((size_t)N * 512 * sizeof(float)));
  if (!e->copy_stream) {
    IBL_CUDA_OK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->copy_ev[0], cudaEventDisableTiming));
    IBL_CUDA_OK(cudaEventCreateWithFlags(&e->copy_ev[1], cudaEventDisableTiming));
  }
  // same two-part overlap as ibl_extract_host, with a quarter of the bytes on the wire
  const int parts = N >= 16 ? 2 : 1;
  const int n_first = parts == 2 ? N / 4 : N;
  uint8_t* du8 = e->stage_u8.as<uint8_t>();
  for (int i = 0; i < parts; ++i) {
    const int n0 = i == 0 ? 0 : n_first, nb = i == 0 ? n_first : N - n_first;
    IBL_CUDA_OK(cudaMemcpyAsync(du8 + n0 * img_px * 3, x_nhwc_host + n0 * img_px * 3, nb * img_px * 3,
                                cudaMemcpyHostToDevice, e->copy_stream));
    IBL_CUDA_OK(cudaEventRecord(e->copy_ev[i], e->copy_stream));
  }
  for (int i = 0; i < parts; ++i) {
    const int n0 = i == 0 ? 0 : n_first, nb = i == 0 ? n_first : N - n_first;
    IBL_CUDA_OK(cudaStreamWaitEvent(S(stream), e->copy_ev[i], 0));
    float* xin = e->stage_in.as<float>() + n0 * img_px * 3;
    IBL_RET(launch_u8_hwc_to_nchw_norm(du8 + n0 * img_px * 3, nb, H, W, mean3, std3, xin, S(stream)));
    e->launches++;
    IBL_RET(ibl_extract(e, xin, nb, H, W, flags, e->stage_out.as<float>() + (size_t)n0 * out_dim,
                        (flags & IBL_OUT_POOL) ? e->stage_out2.as<float>() + (size_t)n0 * 512 : nullptr, stream));
  }
  IBL_CUDA_OK(cudaMemcpyAsync(out_host, e->stage_out.p, (size_t)N * out_dim * sizeof(float), cudaMemcpyDeviceToHost,
                              S(stream)));
  if ((flags & IBL_OUT_POOL) && pool_host)
    IBL_CUDA_OK(cudaMemcpyAsync(pool_host, e->stage_out2.p, (size_t)N * 512 * sizeof(float), cudaMemcpyDeviceToHost,
                                S(stream)));
  IBL_CUDA_OK(cudaStreamSynchronize(S(stream)));
  return IBL_OK;
}

int ibl_l2dist_dense(ibl_engine* e, const float* q, int m, const float* db, int n, int d, float* out,
                     void* stream) {
  IBL_REQUIRE(e && q && db && out, "null argument");
  IBL_REQUIRE(m >= 1 && n >= 1 && d >= 4 && d % 4 == 0, "bad shape");
  DeviceGuard g(e->device);
  IBL_RET(e->qn.ensure((size_t)m * sizeof(float)));
  IBL_RET(e->dbn.ensure((size_t)n * sizeof(float)));
  IBL_RET(launch_row_sqnorm(q, m, d, e->qn.as<float>(), S(stream)));
  IBL_RET(launch_row_sqnorm(db, n, d, e->dbn.as<float>(), S(stream)));
  if (e->gemm_mode == IBL_CONV_TC_BF16X3 && d % 64 == 0) {
    const size_t qe = (size_t)m * d, de = (size_t)n * d;
    IBL_RET(e->q_pl.ensure(qe * 4));
    IBL_RET(e->db_pl.ensure(de * 4));
    __nv_bfloat16 *qh = e->q_pl.as<__nv_bfloat16>(), *dh = e->db_pl.as<__nv_bfloat16>();
    IBL_RET(launch_f32_to_planes(q, qe, qh, qh + qe, S(stream)));
    IBL_RET(launch_f32_to_planes(db, de, dh, dh + de, S(stream)));
    IBL_RET(launch_dist_dense_tc(qh, qh + qe, e->qn.as<float>(), m, dh, dh + de, e->dbn.as<float>(), n, d, out, n,
                                 S(stream)));
    e->launches += 5;
    return IBL_OK;
  }
  IBL_RET(launch_l2dist_dense(q, e->qn.as<float>(), m, db, e->dbn.as<float>(), n, d, out, n, S(stream)));
  e->launches += 3;
  return IBL_OK;
}

// C[m,n] = alpha * A[m,k] . B[n,k]^T on the engine's own GEMM kernels (PCA.train's covariance / dual products and
// projection, reference ibl/pca.py:38-67, torch.matmul there).  mode: IBL_CONV_SIMT_FP32 = fp32 CUDA cores,
// IBL_CONV_TC_BF16X3 = tcgen05 bf16x3 (k % 64 == 0).  Built on the distance tile with zero norm terms:
// (0 + 0 - 2 a.b) * (-alpha / 2).
int ibl_gemm_nt(ibl_engine* e, const float* A, int m, const float* B, int n, int k, float alpha, float* C, int mode,
                void* stream) {
  IBL_REQUIRE(e && A && B && C, "null argument");
  IBL_REQUIRE(m >= 1 && n >= 1 && k >= 4 && k % 4 == 0, "bad shape (k must be a positive multiple of 4)");
  IBL_REQUIRE((long long)m * n < (1ll << 31), "output too large for one call");
  IBL_REQUIRE(mode == IBL_CONV_SIMT_FP32 || mode == IBL_CONV_TC_BF16X3, "unknown gemm mode");
  DeviceGuard g(e->device);
  cudaStream_t s = S(stream);
  IBL_RET(e->qn.ensure((size_t)m * sizeof(float)));
  IBL_RET(e->dbn.ensure((size_t)n * sizeof(float)));
  IBL_CUDA_OK(cudaMemsetAsync(e->qn.p, 0, (size_t)m * sizeof(float), s));
  IBL_CUDA_OK(cudaMemsetAsync(e->dbn.p, 0, (size_t)n * sizeof(float), s));
  if (mode == IBL_CONV_TC_BF16X3 && k % 64 == 0) {
    const size_t ae = (size_t)m * k, be = (size_t)n * k;
    IBL_RET(e->q_pl.ensure(ae * 4));
    IBL_RET(e->db_pl.ensure(be * 4));
    __nv_bfloat16 *ah = e->q_pl.as<__nv_bfloat16>(), *bh = e->db_pl.as<__nv_bfloat16>();
    IBL_RET(launch_f32_to_planes(A, ae, ah, ah + ae, s));
    IBL_RET(launch_f32_to_planes(B, be, bh, bh + be, s));
    IBL_RET(launch_dist_dense_tc(ah, ah + ae, e->qn.as<float>(), m, bh, bh + be, e->dbn.as<float>(), n, k, C, n, s));
    e->launches += 3;
  } else {
    IBL_RET(launch_l2dist_dense(A, e->qn.as<float>(), m, B, e->dbn.as<float>(), n, k, C, n, s));
    e->launches += 1;
  }
  IBL_RET(launch_scale(C, -0.5f * alpha, m * n, C, s));
  e->launches += 1;
  return IBL_OK;
}

// pairwise_distance(features) with query=gallery=None (evaluators.py:106-114):
// out[i,j] = 2|x_i|^2 - 2 x_i.x_j  (the reference broadcasts 2|x_i|^2 over the whole row)
int ibl_l2dist_self(ibl_engine* e, const float* x, int n, int d, float* out, void* stream) {
  IBL_REQUIRE(e && x && out, "null argument");
  IBL_REQUIRE(n >= 1 && d >= 4 && d % 4 == 0, "bad shape");
  DeviceGuard g(e->device);
  cudaStream_t s = S(stream);
  IBL_RET(e->qn.ensure((size_t)n * sizeof(float)));
  IBL_RET(e->dbn.ensure((size_t)n * sizeof(float)));
  IBL_RET(launch_row_sqnorm(x, n, d, e->qn.as<float>(), s));
  IBL_RET(launch_scale(e->qn.as<float>(), 2.f, n, e->qn.as<float>(), s));   // row term 2|x_i|^2
  IBL_CUDA_OK(cudaMemsetAsync(e->dbn.p, 0, (size_t)n * sizeof(float), s));   // no column term
  if (e->gemm_mode == IBL_CONV_TC_BF16X3 && d % 64 == 0) {
    const size_t ne = (size_t)n * d;
    IBL_RET(e->q_pl.ensure(ne * 4));
    __nv_bfloat16* xh = e->q_pl.as<__nv_bfloat16>();
    IBL_RET(launch_f32_to_planes(x, ne, xh, xh + ne, s));
    IBL_RET(launch_dist_dense_tc(xh, xh + ne, e->qn.as<float>(), n, xh, xh + ne, e->dbn.as<float>(), n, d, out, n, s));
    e->launches += 4;
    return IBL_OK;
  }
  IBL_RET(launch_l2dist_dense(x, e->qn.as<float>(), n, x, e->dbn.as<float>(), n, d, out, n, s));
  e->launches += 3;
  return IBL_OK;
}

int ibl_l2dist_topk(ibl_engine* e, const float* q, int m, const float* db, int n, int n_valid, int d,
                    int k, int64_t idx_base, float* out_dist, int64_t* out_idx, void* stream) {
  IBL_REQUIRE(e && q && db && out_dist && out_idx, "null argument");
  IBL_REQUIRE(m >= 1 && n >= 1 && d >= 4 && d % 4 == 0, "bad shape");
  IBL_REQUIRE(n_valid >= 0 && n_valid <= n, "n_valid out of range");
  IBL_REQUIRE(k >= 1 && k <= 128, "top-k supports 1 <= k <= 128");
  DeviceGuard g(e->device);
  // IBL_DIST_SCREEN=3 selects round 1's bf16x3 screening kernels (A/B measurements, variant tests)
  static const int screen_env = [] { const char* v = getenv("IBL_DIST_SCREEN"); return v ? atoi(v) : 1; }();
  if (e->gemm_mode == IBL_CONV_TC_BF16X3 && d % 64 == 0 && n_valid > 0 && k <= 12 && m > 128 && screen_env != 3) {
    // single fp16 tensor-core pass to screen, exact fp32 to decide, guard + exact fallback on the device
    size_t off[9];
    IBL_RET(e->d1_ws.ensure(dist1_workspace_bytes(m, n, d, off)));
    e->dist_flags = dist1_flag_count(e->d1_ws.p, m, n, d);
    return launch_dist_topk_1pass(q, m, db, n, n_valid, d, k, (long long)idx_base, e->d1_ws.p, out_dist,
                                  reinterpret_cast<long long*>(out_idx), &e->launches, S(stream));
  }
  if (e->gemm_mode == IBL_CONV_TC_BF16X3 && d % 64 == 0 && n_valid > 0) {
    cudaStream_t s = S(stream);
    IBL_RET(e->qn.ensure((size_t)m * sizeof(float)));
    IBL_RET(e->dbn.ensure((size_t)n * sizeof(float)));
    const size_t qe = (size_t)m * d, de = (size_t)n * d;
    IBL_RET(e->q_pl.ensure(qe * 4));
    IBL_RET(e->db_pl.ensure(de * 4));
    __nv_bfloat16 *qh = e->q_pl.as<__nv_bfloat16>(), *dh = e->db_pl.as<__nv_bfloat16>();
    // guard workspace: q err [m] | db err [n] | db max2 + flag count (256 B) | flag list [m] | fallback scratch
    const int kk = k <= 12 ? 16 : (k + 8 > 128 ? 128 : k + 8);   // candidates kept per query before exact re-scoring
    const size_t g_qe = 0, g_de = g_qe + (((size_t)m * 4 + 255) & ~(size_t)255), g_mx = g_de + (((size_t)n * 4 + 255) & ~(size_t)255);
    const size_t g_fl = g_mx + 256, g_sc = g_fl + (((size_t)m * 4 + 255) & ~(size_t)255);
    IBL_RET(e->dguard.ensure(g_sc + dist_exact_scratch_bytes(m, n_valid, k)));
    uint8_t* gw = reinterpret_cast<uint8_t*>(e->dguard.p);
    float* q_err = reinterpret_cast<float*>(gw + g_qe);
    float* db_err = reinterpret_cast<float*>(gw + g_de);
    RescoreGuard gd{};
    gd.q_err = q_err; gd.db_max2 = reinterpret_cast<float*>(gw + g_mx); gd.n_valid = n_valid;
    gd.flag_count = reinterpret_cast<int*>(gw + g_mx + 16); gd.flag_list = reinterpret_cast<int*>(gw + g_fl);
    e->dist_flags = gd.flag_count;
    IBL_CUDA_OK(cudaMemsetAsync(gw + g_mx, 0, 32, s));      // db max2 (2 floats) | flag count at +16
    // one pass per matrix: bf16 hi/lo planes for the tensor-core GEMM + exact fp32 squared norms + the guard's
    // representation errors
    IBL_RET(launch_planes_sqnorm(q, m, d, qh, qh + qe, e->qn.as<float>(), s, q_err));
    IBL_RET(launch_planes_sqnorm(db, n, d, dh, dh + de, e->dbn.as<float>(), s, db_err));
    IBL_RET(launch_dist_colmax(e->dbn.as<float>(), db_err, 1, n_valid, reinterpret_cast<float*>(gw + g_mx), s));
    e->launches += 3;
    // exact brute force of the queries the guard of launch_rescore_sort listed (none, usually)
    auto fallback = [&]() {
      e->launches += 2;
      return launch_dist_exact_fallback(q, e->qn.as<float>(), 1, m, db, e->dbn.as<float>(), 1, n_valid, d, k, idx_base,
                                        gd.flag_count, gd.flag_list, reinterpret_cast<unsigned long long*>(gw + g_sc),
                                        out_dist, reinterpret_cast<long long*>(out_idx), s);
    };
    const int kc = 16;
    if (k <= 12) {
      // SM pairs (tcgen05.mma.cta_group::2, tc_gemm2.cu) unless there is a single 128-query tile; IBL_DIST_2SM=0
      // selects the one-SM kernel of tc_gemm.cu
      static const bool two_sm_env = [] { const char* v = getenv("IBL_DIST_2SM"); return !v || atoi(v) != 0; }();
      const bool two_sm = two_sm_env && m > 128;
      const int max_runs = two_sm ? dist_top16_2sm_max_runs(m, n_valid) : dist_top16_max_runs(m, n_valid);
      IBL_RET(e->cand_d.ensure((size_t)max_runs * m * kc * sizeof(float)));
      IBL_RET(e->cand_i.ensure((size_t)max_runs * m * kc * sizeof(int64_t)));
      int runs = 0;
      if (two_sm) {
        IBL_RET(launch_dist_top16_2sm(qh, qh + qe, e->qn.as<float>(), m, dh, dh + de, e->dbn.as<float>(), n,
                                      n_valid, d, e->cand_d.as<float>(), e->cand_i.as<long long>(), &runs, s));
      } else {
        IBL_RET(launch_dist_top16_tc(qh, qh + qe, e->qn.as<float>(), m, dh, dh + de, e->dbn.as<float>(), n,
                                     n_valid, d, e->cand_d.as<float>(), e->cand_i.as<long long>(), max_runs,
                                     &runs, s));
      }
      e->launches++;
      const long long* ci = e->cand_i.as<long long>();
      gd.cand_sd = e->cand_d.as<float>();
      if (runs > 1) {
        IBL_RET(e->mrg_d.ensure((size_t)m * kc * sizeof(float)));
        IBL_RET(e->mrg_i.ensure((size_t)m * kc * sizeof(int64_t)));
        IBL_RET(launch_topk_merge(e->cand_d.as<float>(), e->cand_i.as<int64_t>(), runs, m, kc, kc,
                                  e->mrg_d.as<float>(), e->mrg_i.as<int64_t>(), s));
        e->launches++;
        ci = e->mrg_i.as<long long>();
        gd.cand_sd = e->mrg_d.as<float>();
      }
      IBL_RET(launch_rescore_sort(q, e->qn.as<float>(), m, db, e->dbn.as<float>(), d, ci, kc, k, idx_base,
                                  out_dist, reinterpret_cast<long long*>(out_idx), gd, s));
      e->launches++;
      return fallback();
    }
    // k > 12: dense tiles on the tensor cores, row select, then the same exact re-scoring.  k >= 121 keeps fewer than
    // 8 candidates beyond the k-th: expect the guard to send most such queries to the exact brute force.
    const int CHT = 32768;
    const int ncht = cdiv(n_valid, CHT);
    IBL_REQUIRE((long long)ncht * kk <= 8192, "database shard too large for one call; shard it");
    const int chw = n_valid < CHT ? cdiv(n_valid, 4) * 4 : CHT;
    IBL_RET(e->dist_chunk.ensure((size_t)m * chw * sizeof(float)));
    IBL_RET(e->cand_d.ensure((size_t)ncht * m * kk * sizeof(float)));
    IBL_RET(e->cand_i.ensure((size_t)ncht * m * kk * sizeof(int64_t)));
    for (int c = 0; c < ncht; ++c) {
      const int j0 = c * CHT;
      const int nc = (n_valid - j0 < CHT) ? (n_valid - j0) : CHT;
      IBL_RET(launch_dist_dense_tc(qh, qh + qe, e->qn.as<float>(), m, dh + (size_t)j0 * d, dh + de + (size_t)j0 * d,
                                   e->dbn.as<float>() + j0, nc, d, e->dist_chunk.as<float>(), chw, s));
      IBL_RET(launch_topk_rows(e->dist_chunk.as<float>(), chw, m, nc, kk, j0, e->cand_d.as<float>() + (size_t)c * m * kk,
                               e->cand_i.as<int64_t>() + (size_t)c * m * kk, false, s));
      e->launches += 2;
    }
    const long long* ci = e->cand_i.as<long long>();
    gd.cand_sd = e->cand_d.as<float>();
    if (ncht > 1) {
      IBL_RET(e->mrg_d.ensure((size_t)m * kk * sizeof(float)));
      IBL_RET(e->mrg_i.ensure((size_t)m * kk * sizeof(int64_t)));
      IBL_RET(launch_topk_merge(e->cand_d.as<float>(), e->cand_i.as<int64_t>(), ncht, m, kk, kk,
                                e->mrg_d.as<float>(), e->mrg_i.as<int64_t>(), s));
      e->launches++;
      ci = e->mrg_i.as<long long>();
      gd.cand_sd = e->mrg_d.as<float>();
    }
    IBL_RET(launch_rescore_sort(q, e->qn.as<float>(), m, db, e->dbn.as<float>(), d, ci, kk, k, idx_base, out_dist,
                                reinterpret_cast<long long*>(out_idx), gd, s));
    e->launches++;
    return fallback();
  }
  e->dist_flags = nullptr;
  const int CH = 32768;                         // database rows per dense chunk
  const int nch = n_valid > 0 ? cdiv(n_valid, CH) : 1;
  IBL_REQUIRE((long long)nch * k <= 8192, "database shard too large for one call; shard it");
  IBL_RET(e->qn.ensure((size_t)m * sizeof(float)));
  IBL_RET(e->dbn.ensure((size_t)n * sizeof(float)));
  const int chw = n_valid < CH ? (n_valid > 0 ? n_valid : 1) : CH;
  IBL_RET(e->dist_chunk.ensure((size_t)m * chw * sizeof(float)));
  IBL_RET(launch_row_sqnorm(q, m, d, e->qn.as<float>(), S(stream)));
  IBL_RET(launch_row_sqnorm(db, n, d, e->dbn.as<float>(), S(stream)));
  e->launches += 2;
  float* cd = out_dist;
  int64_t* ci = out_idx;
  if (nch > 1) {
    IBL_RET(e->cand_d.ensure((size_t)nch * m * k * sizeof(float)));
    IBL_RET(e->cand_i.ensure((size_t)nch * m * k * sizeof(int64_t)));
    cd = e->cand_d.as<float>();
    ci = e->cand_i.as<int64_t>();
  }
  for (int c = 0; c < nch; ++c) {
    const int j0 = c * CH;
    const int nc = (n_valid - j0 < CH) ? (n_valid - j0) : CH;
    if (nc > 0)
      IBL_RET(launch_l2dist_dense(q, e->qn.as<float>(), m, db + (size_t)j0 * d, e->dbn.as<float>() + j0, nc,
                                  d, e->dist_chunk.as<float>(), chw, S(stream)));
    IBL_RET(launch_topk_rows(e->dist_chunk.as<float>(), chw, m, nc > 0 ? nc : 0, k, idx_base + j0,
                             cd + (size_t)c * m * k, ci + (size_t)c * m * k, false, S(stream)));
    e->launches += 2;
  }
  if (nch > 1) {
    IBL_RET(launch_topk_merge(cd, ci, nch, m, k, k, out_dist, out_idx, S(stream)));
    e->launches++;
  }
  return IBL_OK;
}

int ibl_topk_rows(ibl_engine* e, const float* dist, int m, int n, int k, float* out_dist, int64_t* out_idx,
                  void* stream) {
  IBL_REQUIRE(e && dist && out_dist && out_idx, "null argument");
  IBL_REQUIRE(m >= 0 && n >= 1 && k >= 1 && k <= 1024, "bad shape (ibl_topk_rows: 1 <= k <= 1024)");
  DeviceGuard g(e->device);
  e->launches++;
  return launch_topk_rows(dist, n, m, n, k, 0, out_dist, out_idx, false, S(stream));
}

// torch.argsort(distmat, dim=1) of the training samplers (ibl/utils/data/sampler.py:46-54,126-135) on the device:
// dist [m,n] -> out_idx [m,n], ascending by (distance, index).
int ibl_argsort_rows(ibl_engine* e, const float* dist, int m, int n, int64_t* out_idx, void* stream) {
  IBL_REQUIRE(e && dist && out_idx, "null argument");
  IBL_REQUIRE(m >= 0 && n >= 1, "bad shape");
  DeviceGuard g(e->device);
  unsigned long long* scratch = nullptr;
  if (n > 16384) {
    IBL_RET(e->dist_chunk.ensure((size_t)2 * m * n * sizeof(unsigned long long)));
    scratch = e->dist_chunk.as<unsigned long long>();
  }
  return launch_argsort_rows(dist, n, m, n, reinterpret_cast<long long*>(out_idx), scratch, S(stream), &e->launches);
}

int ibl_topk_merge(ibl_engine* e, const float* cand_dist, const int64_t* cand_idx, int parts, int m,
                   int k_in, int k_out, float* out_dist, int64_t* out_idx, void* stream) {
  IBL_REQUIRE(e && cand_dist && cand_idx && out_dist && out_idx, "null argument");
  IBL_REQUIRE(parts >= 1 && m >= 0 && k_in >= 1, "bad shape");
  DeviceGuard g(e->device);
  e->launches++;
  return launch_topk_merge(cand_dist, cand_idx, parts, m, k_in, k_out, out_dist, out_idx, S(stream));
}

int ibl_l2dist_topk_host(ibl_engine* e, const float* q_host, int m, const float* db_host, int n, int d,
                         int k, float* out_dist_host, int64_t* out_idx_host, void* stream) {
  IBL_REQUIRE(e && q_host && db_host && out_dist_host && out_idx_host, "null argument");
  IBL_REQUIRE(m >= 1 && n >= 1 && d >= 4 && k >= 1 && k <= 128, "bad shape");
  DeviceGuard g(e->device);
  const size_t qb = (size_t)m * d * sizeof(float), dbb = (size_t)n * d * sizeof(float);
  IBL_RET(e->stage_in.ensure(qb + dbb));
  IBL_RET(e->stage_out.ensure((size_t)m * k * sizeof(float)));
  IBL_RET(e->stage_out2.ensure((size_t)m * k * sizeof(int64_t)));
  float* dq = e->stage_in.as<float>();
  float* ddb = dq + (size_t)m * d;
  IBL_CUDA_OK(cudaMemcpyAsync(dq, q_host, qb, cudaMemcpyHostToDevice, S(stream)));
  IBL_CUDA_OK(cudaMemcpyAsync(ddb, db_host, dbb, cudaMemcpyHostToDevice, S(stream)));
  IBL_RET(ibl_l2dist_topk(e, dq, m, ddb, n, n, d, k, 0, e->stage_out.as<float>(), e->stage_out2.as<int64_t>(), stream));
  IBL_CUDA_OK(cudaMemcpyAsync(out_dist_host, e->stage_out.p, (size_t)m * k * sizeof(float), cudaMemcpyDeviceToHost, S(stream)));
  IBL_CUDA_OK(cudaMemcpyAsync(out_idx_host, e->stage_out2.p, (size_t)m * k * sizeof(int64_t), cudaMemcpyDeviceToHost, S(stream)));
  IBL_CUDA_OK(cudaStreamSynchronize(S(stream)));
  return IBL_OK;
}

// test hook: how many queries the screening guard listed in the last ibl_l2dist_topk call (they were re-ranked by
// exact brute force on the device), whichever tensor-core path it took; -1 after the CUDA-core path.  Synchronises.
int ibl_debug_dist_flagged(ibl_engine* e, int* count, void* stream) {
  IBL_REQUIRE(e && count, "null argument");
  *count = -1;
  if (!e->dist_flags) return IBL_OK;
  DeviceGuard g(e->device);
  IBL_CUDA_OK(cudaMemcpyAsync(count, e->dist_flags, sizeof(int), cudaMemcpyDeviceToHost, S(stream)));
  IBL_CUDA_OK(cudaStreamSynchronize(S(stream)));
  return IBL_OK;
}

int ibl_selftest_tc(ibl_engine* e, float* max_rel_err) {
  IBL_REQUIRE(e, "null engine");
  DeviceGuard g(e->device);
  return tc_selftest(max_rel_err, nullptr);
}

// One conv layer in isolation, fp32 NHWC in / out, either math mode (test hook).
int ibl_debug_conv3x3(ibl_engine* e, const float* x_nhwc, int N, int H, int W, int cin, const float* w_oihw,
                      const float* bias, int cout, int relu, int pool, int mode, int bn_override,
                      float* y_nhwc, void* stream) {
  IBL_REQUIRE(e && x_nhwc && w_oihw && bias && y_nhwc, "null argument");
  IBL_REQUIRE(cin % 64 == 0 && cout % 64 == 0, "debug conv needs Cin%64==0, Cout%64==0");
  DeviceGuard g(e->device);
  cudaStream_t s = S(stream);
  ConvParams p;
  const size_t nw = (size_t)cout * cin * 9;
  IBL_CUDA_OK(cudaMalloc(&p.w_tck, nw * 4));
  IBL_CUDA_OK(cudaMalloc(&p.bias, cout * 4));
  IBL_CUDA_OK(cudaMalloc(&p.w_hi, nw * 2));
  IBL_CUDA_OK(cudaMalloc(&p.w_lo, nw * 2));
  int rc = launch_repack_weights(w_oihw, cout, cin, p, s);
  cudaMemcpyAsync(p.bias, bias, cout * 4, cudaMemcpyDeviceToDevice, s);
  const size_t in_e = (size_t)N * H * W * cin;
  const int oh = pool ? H / 2 : H, ow = pool ? W / 2 : W;
  const size_t out_e = (size_t)N * oh * ow * cout;
  if (rc == IBL_OK && mode == IBL_CONV_SIMT_FP32) {
    if (!pool) {
      rc = launch_conv3x3_simt(x_nhwc, p, N, H, W, cin, cout, relu != 0, y_nhwc, s);
    } else {
      float* tmp = nullptr;
      if (cudaMalloc(&tmp, (size_t)N * H * W * cout * 4) != cudaSuccess) rc = IBL_ERR_OOM;
      if (rc == IBL_OK) rc = launch_conv3x3_simt(x_nhwc, p, N, H, W, cin, cout, relu != 0, tmp, s);
      if (rc == IBL_OK) rc = launch_maxpool2x2(tmp, N, H, W, cout, y_nhwc, s);
      cudaStreamSynchronize(s);
      if (tmp) cudaFree(tmp);
    }
  } else if (rc == IBL_OK) {
    __nv_bfloat16 *xh = nullptr, *xl = nullptr;
    if (cudaMalloc(&xh, in_e * 2) != cudaSuccess || cudaMalloc(&xl, in_e * 2) != cudaSuccess) rc = IBL_ERR_OOM;
    if (rc == IBL_OK) rc = launch_f32_to_planes(x_nhwc, in_e, xh, xl, s);
    tc_set_bn_override(bn_override);
    if (mode == 2) {
      __nv_bfloat16 *yh = nullptr, *yl = nullptr;
      if (cudaMalloc(&yh, out_e * 2) != cudaSuccess || cudaMalloc(&yl, out_e * 2) != cudaSuccess) rc = IBL_ERR_OOM;
      if (rc == IBL_OK) rc = launch_conv3x3_tc(xh, xl, p, N, H, W, cin, cout, relu != 0, pool != 0, yh, yl, nullptr, s);
      if (rc == IBL_OK) rc = launch_planes_to_f32(yh, yl, out_e, y_nhwc, s);
      cudaStreamSynchronize(s);
      if (yh) cudaFree(yh);
      if (yl) cudaFree(yl);
    } else if (rc == IBL_OK) {
      rc = launch_conv3x3_tc(xh, xl, p, N, H, W, cin, cout, relu != 0, pool != 0, nullptr, nullptr, y_nhwc, s);
    }
    tc_set_bn_override(0);
    cudaStreamSynchronize(s);
    if (xh) cudaFree(xh);
    if (xl) cudaFree(xl);
  }
  cudaError_t ce = cudaStreamSynchronize(s);
  cudaFree(p.w_tck); cudaFree(p.bias); cudaFree(p.w_hi); cudaFree(p.w_lo);
  if (rc == IBL_OK && ce != cudaSuccess) {
    set_last_error(std::string("debug conv: ") + cudaGetErrorString(ce));
    return IBL_ERR_CUDA;
  }
  e->launches += 3;
  return rc;
}

int ibl_debug_gemm_tn(ibl_engine* e, const float* A, const float* B, float* C, void* stream) {
  IBL_REQUIRE(e && A && B && C, "null argument");
  DeviceGuard g(e->device);
  e->launches += 3;
  return debug_gemm_tn(A, B, C, S(stream));
}

int ibl_debug_umma_strided(ibl_engine* e, const void* A, int rows, const void* B, int s0, int group_rows,
                            int base_mode, float* D, void* stream) {
  IBL_REQUIRE(e && A && B && D, "null argument");
  DeviceGuard g(e->device);
  e->launches += 1;
  return debug_umma_strided(A, rows, B, s0, group_rows, base_mode, D, S(stream));
}

// Timing hooks (tools/bench_layers.py): average device time of one backbone layer over `reps`
// back-to-back launches, weights taken from the engine (ibl_engine_set_vgg16).  layer 0 = conv1_1
// (x is NCHW [N,3,H,W]); layers 1..12 take x NHWC [N,H,W,Cin] fp32 (converted to planes once).
int ibl_debug_time_layer(ibl_engine* e, int layer, const float* x, int N, int H, int W, int bn_override,
                         int reps, float* ms_out) {
  IBL_REQUIRE(e && x && ms_out && layer >= 0 && layer <= 13 && reps >= 1, "bad argument");
  if (!e->vgg_ready) { set_last_error("ibl_engine_set_vgg16 was not called"); return IBL_ERR_NOT_READY; }
  DeviceGuard g(e->device);
  if (layer == 13) {   // the fused conv1_1 + conv1_2 + pool kernel: x is the NCHW image batch
    const size_t out_e = (size_t)N * (H / 2) * (W / 2) * 64;
    IBL_RET(e->act[1].ensure(out_e * 4));
    cudaEvent_t e0, e1;
    IBL_CUDA_OK(cudaEventCreate(&e0));
    IBL_CUDA_OK(cudaEventCreate(&e1));
    __nv_bfloat16* oh_ = e->act[1].as<__nv_bfloat16>();
    int rc = IBL_OK;
    for (int r = -1; r < reps && rc == IBL_OK; ++r) {
      if (r == 0) cudaEventRecord(e0, nullptr);
      rc = launch_conv1_fused_tc(x, e->w0_oihw, e->conv[0].bias, e->conv[1], N, H, W, oh_, oh_ + out_e, nullptr);
    }
    cudaEventRecord(e1, nullptr);
    cudaError_t ce = cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc == IBL_OK && ce != cudaSuccess) { set_last_error(cudaGetErrorString(ce)); return IBL_ERR_CUDA; }
    *ms_out = ms / reps;
    e->launches += reps + 1;
    return rc;
  }
  const ConvLayer& L = kVgg16[layer];
  const size_t in_e = (size_t)N * H * W * L.cin;
  const int oh = L.pool ? H / 2 : H, ow = L.pool ? W / 2 : W;
  const size_t out_e = (size_t)N * oh * ow * L.cout;
  IBL_RET(e->act[0].ensure((in_e > out_e ? in_e : out_e) * 4));
  IBL_RET(e->act[1].ensure((in_e > out_e ? in_e : out_e) * 4));
  cudaEvent_t e0, e1;
  IBL_CUDA_OK(cudaEventCreate(&e0));
  IBL_CUDA_OK(cudaEventCreate(&e1));
  __nv_bfloat16* ih = e->act[0].as<__nv_bfloat16>();
  __nv_bfloat16* oh_ = e->act[1].as<__nv_bfloat16>();
  int rc = IBL_OK;
  if (layer > 0) rc = launch_f32_to_planes(x, in_e, ih, ih + in_e, nullptr);
  tc_set_bn_override(bn_override);
  for (int r = -1; r < reps && rc == IBL_OK; ++r) {       // r = -1 is a warm-up launch
    if (r == 0) cudaEventRecord(e0, nullptr);
    if (layer == 0)
      rc = bn_override == 1 ? launch_conv1_1(x, e->conv[0], N, H, W, true, nullptr, oh_, oh_ + out_e, nullptr)
                            : launch_conv1_1_tc(x, e->w0_oihw, e->conv[0].bias, N, H, W, oh_, oh_ + out_e, nullptr);
    else
      rc = launch_conv3x3_tc(ih, ih + in_e, e->conv[layer], N, H, W, L.cin, L.cout, L.relu, L.pool,
                             layer == 12 ? nullptr : oh_, layer == 12 ? nullptr : oh_ + out_e,
                             layer == 12 ? e->act[1].as<float>() : nullptr, nullptr);
  }
  tc_set_bn_override(0);
  cudaEventRecord(e1, nullptr);
  cudaError_t ce = cudaEventSynchronize(e1);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (rc == IBL_OK && ce != cudaSuccess) { set_last_error(cudaGetErrorString(ce)); return IBL_ERR_CUDA; }
  *ms_out = ms / reps;
  e->launches += reps + 1;
  return rc;
}

}  // extern "C"
