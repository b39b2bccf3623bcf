// CUDA-core fp32 "NT" GEMM family  C[i,j] = sum_k A[i,k] * B[j,k]  (both operands K-major)
// used by
//   * PCA-whitening  y = W v + b, L2          (netvlad.py:105-108 / pca.py:117-121)
//   * dense L2 distance |q|^2 + |d|^2 - 2 q.d (evaluators.py:127-129)
// plus the row-norm helpers (evaluators.py:29-33).
#include "common.cuh"

namespace ibl {

constexpr int G_BM = 128, G_BN = 64, G_BK = 16;

enum { EPI_PCA_PARTIAL = 0, EPI_L2DIST = 1 };

struct GemmArgs {
  const float* A;   // [M, K] row-major (ld = lda)
  const float* B;   // [Ncol, K] row-major (ld = ldb)
  long long lda, ldb;
  int M, Ncol;
  int k_begin_stride;  // K range of split z is [z*k_per_split, min(K,(z+1)*k_per_split))
  int K;
  // epilogue
  float* out;          // PCA: partial [splits][Ncol][M];  L2DIST: out [M][ld_out]
  long long ld_out;
  const float* an;     // L2DIST: |A_i|^2
  const float* bn;     // L2DIST: |B_j|^2
};

template <int EPI>
__global__ void __launch_bounds__(256) gemm_nt_kernel(GemmArgs g) {
  __shared__ __align__(16) float As[G_BK][G_BM];
  __shared__ __align__(16) float Bs[G_BK][G_BN];
  const int t = threadIdx.x;
  const int tn = t & 15, tm = t >> 4;
  const int m0 = blockIdx.x * G_BM, n0 = blockIdx.y * G_BN;
  const int kb = blockIdx.z * g.k_begin_stride;
  const int ke = min(g.K, kb + g.k_begin_stride);

  const int lm = t & 127, kq0 = t >> 7;       // A loader: row lm, k-quads kq0, kq0+2
  const int bnr = t >> 2, bkq = t & 3;        // B loader: row bnr, k-quad bkq
  const bool a_ok = (m0 + lm) < g.M;
  const bool b_ok = (n0 + bnr) < g.Ncol;
  const float* ap = g.A + (long long)(m0 + lm) * g.lda;
  const float* bp = g.B + (long long)(n0 + bnr) * g.ldb;

  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = kb; k0 < ke; k0 += G_BK) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int kq = kq0 + 2 * j;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a_ok && k0 + kq * 4 + 3 < ke) v = __ldg(reinterpret_cast<const float4*>(ap + k0 + kq * 4));
      As[kq * 4 + 0][lm] = v.x;
      As[kq * 4 + 1][lm] = v.y;
      As[kq * 4 + 2][lm] = v.z;
      As[kq * 4 + 3][lm] = v.w;
    }
    {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b_ok && k0 + bkq * 4 + 3 < ke) v = __ldg(reinterpret_cast<const float4*>(bp + k0 + bkq * 4));
      Bs[bkq * 4 + 0][bnr] = v.x;
      Bs[bkq * 4 + 1][bnr] = v.y;
      Bs[bkq * 4 + 2][bnr] = v.z;
      Bs[bkq * 4 + 3][bnr] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < G_BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[k][tm * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[k][tm * 8 + 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tn * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }

  if (EPI == EPI_PCA_PARTIAL) {
    // partial[z][j][i]: i (= output feature) contiguous
    float* o = g.out + (long long)blockIdx.z * g.Ncol * (long long)g.M;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = n0 + tn * 4 + j;
      if (col >= g.Ncol) continue;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = m0 + tm * 8 + i;
        if (row < g.M) o[(long long)col * g.M + row] = acc[i][j];
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = m0 + tm * 8 + i;
      if (row >= g.M) continue;
      const float an = __ldg(g.an + row);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int col = n0 + tn * 4 + j;
        if (col < g.Ncol) {
          // evaluators.py:127-129: (|x|^2 + |y|^2) + (-2) * x.y
          g.out[(long long)row * g.ld_out + col] = fmaf(-2.f, acc[i][j], an + __ldg(g.bn + col));
        }
      }
    }
  }
}

// out[n][p] = normalize( bias[p] + sum_z partial[z][n][p] )
__global__ void __launch_bounds__(256)
pca_finalize_kernel(const float* __restrict__ partial, int splits, int N, int P,
                    const float* __restrict__ bias, float* __restrict__ out) {
  extern __shared__ float row[];  // [P]
  __shared__ float red[8];
  __shared__ float inv_s;
  const long long n = blockIdx.x;
  float ss = 0.f;
  for (int p = threadIdx.x; p < P; p += blockDim.x) {
    float v = 0.f;
    for (int z = 0; z < splits; ++z) v += partial[((long long)z * N + n) * P + p];
    v += __ldg(bias + p);
    row[p] = v;
    ss = fmaf(v, v, ss);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
    inv_s = 1.f / fmaxf(sqrtf(tot), 1e-12f);
  }
  __syncthreads();
  const float inv = inv_s;
  for (int p = threadIdx.x; p < P; p += blockDim.x) out[n * P + p] = row[p] * inv;
}

int launch_pca_finalize(const float* partial, int splits, int N, int P, const float* bias, float* out,
                        cudaStream_t s) {
  pca_finalize_kernel<<<N, 256, P * sizeof(float), s>>>(partial, splits, N, P, bias, out);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}

int launch_pca_l2(const float* v, int N, int D, const float* W, const float* b, int P,
                  float* partial, int splits, float* out, cudaStream_t s, uint64_t* launches) {
  IBL_REQUIRE(D % 4 == 0, "PCA input dim must be a multiple of 4");
  GemmArgs g{};
  g.A = W; g.lda = D; g.M = P;
  g.B = v; g.ldb = D; g.Ncol = N;
  g.K = D;
  int kps = cdiv(D, splits);
  kps = cdiv(kps, G_BK) * G_BK;
  g.k_begin_stride = kps;
  g.out = partial;
  dim3 grid((unsigned)cdiv(P, G_BM), (unsigned)cdiv(N, G_BN), (unsigned)cdiv(D, kps));
  gemm_nt_kernel<EPI_PCA_PARTIAL><<<grid, 256, 0, s>>>(g);
  IBL_CUDA_OK(cudaGetLastError());
  pca_finalize_kernel<<<N, 256, P * sizeof(float), s>>>(partial, (int)grid.z, N, P, b, out);
  IBL_CUDA_OK(cudaGetLastError());
  *launches += 2;
  return IBL_OK;
}

int launch_l2dist_dense(const float* q, const float* qn, int m, const float* db, const float* dbn,
                        int n, int d, float* out, long long ld_out, cudaStream_t s) {
  IBL_REQUIRE(d % 4 == 0, "descriptor dim must be a multiple of 4");
  GemmArgs g{};
  g.A = q; g.lda = d; g.M = m;
  g.B = db; g.ldb = d; g.Ncol = n;
  g.K = d;
  g.k_begin_stride = cdiv(d, G_BK) * G_BK;
  g.out = out; g.ld_out = ld_out; g.an = qn; g.bn = dbn;
  dim3 grid((unsigned)cdiv(m, G_BM), (unsigned)cdiv(n, G_BN), 1);
  gemm_nt_kernel<EPI_L2DIST><<<grid, 256, 0, s>>>(g);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}

// ---- row helpers ----------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
row_sqnorm_kernel(const float* __restrict__ x, int D, float* __restrict__ out) {
  __shared__ float red[8];
  const long long r = blockIdx.x;
  const float* p = x + r * D;
  float ss = 0.f;
  for (int i = threadIdx.x; i < D; i += blockDim.x) { const float v = __ldg(p + i); ss = fmaf(v, v, ss); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
    out[r] = tot;
  }
}

int launch_row_sqnorm(const float* x, int N, int D, float* out, cudaStream_t s) {
  if (N == 0) return IBL_OK;
  row_sqnorm_kernel<<<N, 256, 0, s>>>(x, D, out);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}

__global__ void __launch_bounds__(256)
l2_normalize_rows_kernel(const float* __restrict__ x, int D, float* __restrict__ out) {
  __shared__ float red[8];
  __shared__ float inv_s;
  const long long r = blockIdx.x;
  const float* p = x + r * D;
  float ss = 0.f;
  for (int i = threadIdx.x; i < D; i += blockDim.x) { const float v = p[i]; ss = fmaf(v, v, ss); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
    inv_s = 1.f / fmaxf(sqrtf(tot), 1e-12f);
  }
  __syncthreads();
  const float inv = inv_s;
  for (int i = threadIdx.x; i < D; i += blockDim.x) out[r * D + i] = p[i] * inv;
}

int launch_l2_normalize_rows(const float* x, int N, int D, float* out, cudaStream_t s) {
  if (N == 0) return IBL_OK;
  l2_normalize_rows_kernel<<<N, 256, 0, s>>>(x, D, out);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}

}  // namespace ibl

namespace ibl {
__global__ void scale_kernel(const float* __restrict__ x, float s, int n, float* __restrict__ y) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = x[i] * s;
}
int launch_scale(const float* x, float s, int n, float* y, cudaStream_t st) {
  if (n <= 0) return IBL_OK;
  scale_kernel<<<cdiv(n, 256), 256, 0, st>>>(x, s, n, y);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}
}  // namespace ibl

namespace ibl {
// One pass over a row-major fp32 matrix: bf16 hi/lo planes + squared row norms (what the distance GEMM and
// its epilogue need), instead of separate f32_to_planes and row_sqnorm passes.  One block per row.  err (may be
// null): |x - (hi + lo)| of the row, for the screening guard; x - hi and (x - hi) - lo are exact in fp32.
__global__ void __launch_bounds__(256)
planes_sqnorm_kernel(const float* __restrict__ x, int D, __nv_bfloat16* __restrict__ hi,
                     __nv_bfloat16* __restrict__ lo, float* __restrict__ sq, float* __restrict__ err) {
  __shared__ float red[8], rede[8];
  const long long r = blockIdx.x;
  const float4* p = reinterpret_cast<const float4*>(x + r * D);
  uint2* ph = reinterpret_cast<uint2*>(hi + r * D);
  uint2* pl = reinterpret_cast<uint2*>(lo + r * D);
  float ss = 0.f, se = 0.f;
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) {
    const float4 v = __ldg(p + i);
    ss = fmaf(v.x, v.x, ss); ss = fmaf(v.y, v.y, ss); ss = fmaf(v.z, v.z, ss); ss = fmaf(v.w, v.w, ss);
    const __nv_bfloat16 h0 = __float2bfloat16_rn(v.x), h1 = __float2bfloat16_rn(v.y);
    const __nv_bfloat16 h2 = __float2bfloat16_rn(v.z), h3 = __float2bfloat16_rn(v.w);
    __nv_bfloat162 a(h0, h1), b(h2, h3);
    const float r0 = v.x - __bfloat162float(h0), r1 = v.y - __bfloat162float(h1);
    const float r2 = v.z - __bfloat162float(h2), r3 = v.w - __bfloat162float(h3);
    __nv_bfloat162 c = __floats2bfloat162_rn(r0, r1);
    __nv_bfloat162 d = __floats2bfloat162_rn(r2, r3);
    if (err) {
      const float e0 = r0 - __low2float(c), e1 = r1 - __high2float(c), e2 = r2 - __low2float(d), e3 = r3 - __high2float(d);
      se = fmaf(e0, e0, se); se = fmaf(e1, e1, se); se = fmaf(e2, e2, se); se = fmaf(e3, e3, se);
    }
    ph[i] = make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b));
    pl[i] = make_uint2(*reinterpret_cast<uint32_t*>(&c), *reinterpret_cast<uint32_t*>(&d));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    se += __shfl_xor_sync(0xffffffffu, se, o);
  }
  if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5] = ss; rede[threadIdx.x >> 5] = se; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f, tote = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { tot += red[i]; tote += rede[i]; }
    sq[r] = tot;
    if (err) err[r] = sqrtf(tote);
  }
}
int launch_planes_sqnorm(const float* x, int N, int D, __nv_bfloat16* hi, __nv_bfloat16* lo, float* sq,
                         cudaStream_t st, float* err) {
  IBL_REQUIRE(D % 4 == 0, "planes_sqnorm: D must be a multiple of 4");
  if (N <= 0) return IBL_OK;
  planes_sqnorm_kernel<<<N, 256, 0, st>>>(x, D, hi, lo, sq, err);
  IBL_CUDA_OK(cudaGetLastError());
  return IBL_OK;
}
}  // namespace ibl
