// fp32 SIMT tile GEMM with loader / store functors (shared by conv_simt.cu and seg_head.cu).
#pragma once
#include "common.cuh"

namespace iic {

constexpr int ST_BM = 64, ST_BN = 64, ST_BK = 16, ST_THREADS = 256;

// ---- loaders -----------------------------------------------------------------------------
template <typename T>
struct DenseLoad {  // element (i, k) at ptr[i*si + k*sk]; i is the M (or N) index
  const T* ptr;
  long long si, sk;
  int rows, K;
  __device__ __forceinline__ float operator()(int i, int k) const {
    return (i < rows && k < K) ? to_f(ptr[i * si + k * sk]) : 0.f;
  }
};

// rows = output pixels (n,oy,ox); k = (a, b, ci) over an NHWC input.  transposed==0: fprop
// gather iy = oy*s - p + a*d.  transposed==1: dgrad gather over dy: ty = oy + p - a*d must be a
// multiple of s, iy = ty / s (rows are then pixels of dx, "input" is dy with C = cout).
template <typename T>
struct Im2colLoad {
  const T* x;
  int H, W, C;        // tensor being gathered from
  int OH, OW;         // pixel grid that the row index enumerates
  int KH, KW, s, p, d, transposed;
  int rows, K;        // rows = n*OH*OW ; K = KH*KW*C
  __device__ __forceinline__ float operator()(int i, int k) const {
    if (i >= rows || k >= K) return 0.f;
    const int ox = i % OW;
    const int t = i / OW;
    const int oy = t % OH;
    const int n = t / OH;
    const int ci = k % C;
    const int t2 = k / C;
    const int b = t2 % KW;
    const int a = t2 / KW;
    int iy, ix;
    if (!transposed) {
      iy = oy * s - p + a * d;
      ix = ox * s - p + b * d;
    } else {
      const int ty = oy + p - a * d, tx = ox + p - b * d;
      if (ty < 0 || tx < 0 || (ty % s) != 0 || (tx % s) != 0) return 0.f;
      iy = ty / s;
      ix = tx / s;
    }
    if (iy < 0 || iy >= H || ix < 0 || ix >= W) return 0.f;
    return to_f(x[(((long long)n * H + iy) * W + ix) * C + ci]);
  }
};

// ---- stores ------------------------------------------------------------------------------
template <typename T>
struct StoreOut {
  T* out;
  const T* addend;
  long long ldc;
  __device__ __forceinline__ void operator()(int z, int m, int n, int M, int N, float v) const {
    long long o = (long long)m * ldc + n;
    if (addend != nullptr) v += to_f(addend[o]);
    out[o] = from_f<T>(v);
  }
};
struct StorePartial {
  float* ws;
  __device__ __forceinline__ void operator()(int z, int m, int n, int M, int N, float v) const {
    ws[((long long)z * M + m) * N + n] = v;
  }
};

// AK / BK: true if consecutive k are contiguous in memory for that operand (picks the
// thread->element mapping of the tile fill so global reads coalesce).
template <class AL, class BL, class ST, bool AK, bool BKC>
__global__ void __launch_bounds__(ST_THREADS) simt_gemm_kernel(AL A, BL B, ST S, int M, int N, int K, int klen) {
  __shared__ float As[ST_BK][ST_BM + 4];
  __shared__ float Bs[ST_BK][ST_BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  const int m0 = blockIdx.y * ST_BM, n0 = blockIdx.x * ST_BN;
  const int kbeg = blockIdx.z * klen;
  const int kend = min(K, kbeg + klen);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = kbeg; k0 < kend; k0 += ST_BK) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int idx = tid + j * ST_THREADS;
      int mi, ki;
      if (AK) { ki = idx % ST_BK; mi = idx / ST_BK; } else { mi = idx % ST_BM; ki = idx / ST_BM; }
      const int k = k0 + ki;
      As[ki][mi] = (k < kend) ? A(m0 + mi, k) : 0.f;
      int ni, kj;
      if (BKC) { kj = idx % ST_BK; ni = idx / ST_BK; } else { ni = idx % ST_BN; kj = idx / ST_BN; }
      const int k2 = k0 + kj;
      Bs[kj][ni] = (k2 < kend) ? B(n0 + ni, k2) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < ST_BK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) S(blockIdx.z, m, n, M, N, acc[i][j]);
    }
  }
}

// out[i] (=|+=) sum_z ws[z][i]   (fixed order => deterministic)
static __global__ void splitk_reduce_kernel(const float* __restrict__ ws, float* __restrict__ out, long long count, int splits,
                                     int accumulate) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    float t = 0.f;
    for (int z = 0; z < splits; ++z) t += ws[(long long)z * count + i];
    out[i] = accumulate ? out[i] + t : t;
  }
}

template <class AL, class BL, class ST, bool AK, bool BKC>
static inline int launch_simt(AL A, BL B, ST S, int M, int N, int K, int splits, cudaStream_t st) {
  const int klen = ((K + splits - 1) / splits + ST_BK - 1) / ST_BK * ST_BK;
  dim3 grid(cdiv(N, ST_BN), cdiv(M, ST_BM), splits);
  simt_gemm_kernel<AL, BL, ST, AK, BKC><<<grid, ST_THREADS, 0, st>>>(A, B, S, M, N, K, klen);
  IIC_LAUNCH_CHECK();
  count_launch();
  return IIC_OK;
}

// ---- skinny dense GEMMs of the heads (conv_simt.cu: sub-heads; semisup.cu: Linear layers) ----------------------------
// Split-K for the skinny head GEMMs (N = S*k = 10..350 columns, K = 512..4608): with one 64x64 tile per 64 rows the
// ClusterNet6c logits (1400 x 4608 x 50) ran on 22 CTAs.  Partials in a per-device scratch (conv_simt.cu), folded in split
// order.  accumulate != 0: out += A B^T instead of out = A B^T.
float* heads_scratch(size_t bytes);

static inline int heads_splits(int M, int N, int K) {
  const long long tiles = (long long)cdiv(M, ST_BM) * cdiv(N, ST_BN);
  const int sms = device_sm_count();
  if (tiles >= sms || K < 512) return 1;
  long long s = (2ll * sms) / tiles;
  if (s > K / 128) s = K / 128;
  if (s > 32) s = 32;
  return (int)(s < 1 ? 1 : s);
}
template <class AL, class BL, bool AK, bool BKC>
static int heads_gemm(AL A, BL B, float* out, long long ldc, int M, int N, int K, cudaStream_t st, int accumulate = 0) {
  const int splits = heads_splits(M, N, K);
  if (splits == 1 || ldc != N) {
    StoreOut<float> St{out, accumulate ? out : nullptr, ldc};
    return launch_simt<AL, BL, StoreOut<float>, AK, BKC>(A, B, St, M, N, K, 1, st);
  }
  float* ws = heads_scratch((size_t)splits * M * N * sizeof(float));
  IIC_REQUIRE(ws != nullptr, IIC_ERR_CUDA, "heads: scratch allocation failed");
  StorePartial Sp{ws};
  int rc = launch_simt<AL, BL, StorePartial, AK, BKC>(A, B, Sp, M, N, K, splits, st);
  if (rc != IIC_OK) return rc;
  const long long count = (long long)M * N;
  long long blocks = cdiv(count, 256);
  if (blocks > 1024) blocks = 1024;
  splitk_reduce_kernel<<<(int)blocks, 256, 0, st>>>(ws, out, count, splits, accumulate);
  IIC_LAUNCH_CHECK();
  count_launch();
  return IIC_OK;
}

}  // namespace iic
