// Reference-precision (fp32 SIMT) implicit-GEMM convolution + the small dense GEMMs of the heads.
//
// This is the IIC_F32 mode of the conv entry points: every multiply-add is an fp32 FFMA, so the
// trunk matches the reference (fp32 cuDNN/MKL) to rounding.  It doubles as the on-device
// cross-check for the tcgen05 path (conv_tc2.cu, conv_tf32.cu) and runs the tiny head GEMMs in both modes.
//
//   C[M][N] = sum_k A(m,k) * B(k,n), 64x64 tiles, BK=16, 256 threads x (4x4) register tiles,
//   operands fetched through loader functors (dense strided / im2col gather / transposed-conv
//   gather), optional split-K over blockIdx.z with deterministic second-pass reduction.
//
// Reference ops replaced: nn.Conv2d fprop/dgrad/wgrad (residual.py:4-7,:53-55; vgg.py:25-27),
// nn.Linear in the sub-heads (net5g_two_head.py:22-24).
#include "simt_gemm.cuh"

namespace iic {

static int wgrad_splits_simt(const iic_conv_geom* g) {
  const long long P = (long long)g->n * g->oh * g->ow;
  const long long tiles = (long long)cdiv(g->cout, ST_BM) * cdiv((long long)g->kh * g->kw * g->cin, ST_BN);
  long long want = ((long long)device_sm_count() * 4 + tiles - 1) / tiles;
  long long maxs = (P + 255) / 256;
  if (want > maxs) want = maxs;
  if (want < 1) want = 1;
  if (want > 512) want = 512;
  return (int)want;
}

int simt_conv_fprop(const float* x, const float* w, float* y, const iic_conv_geom* g, cudaStream_t st) {
  const int M = g->n * g->oh * g->ow, N = g->cout, K = g->kh * g->kw * g->cin;
  Im2colLoad<float> A{x, g->h, g->w, g->cin, g->oh, g->ow, g->kh, g->kw, g->stride, g->pad, g->dil, 0, M, K};
  DenseLoad<float> B{w, (long long)K, 1, N, K};
  StoreOut<float> S{y, nullptr, (long long)N};
  return launch_simt<Im2colLoad<float>, DenseLoad<float>, StoreOut<float>, true, true>(A, B, S, M, N, K, 1, st);
}

int simt_conv_dgrad(const float* dy, const float* wt, const float* addend, float* dx, const iic_conv_geom* g,
                    cudaStream_t st) {
  const int M = g->n * g->h * g->w, N = g->cin, K = g->kh * g->kw * g->cout;
  Im2colLoad<float> A{dy, g->oh, g->ow, g->cout, g->h, g->w, g->kh, g->kw, g->stride, g->pad, g->dil, 1, M, K};
  DenseLoad<float> B{wt, (long long)K, 1, N, K};
  StoreOut<float> S{dx, addend, (long long)N};
  return launch_simt<Im2colLoad<float>, DenseLoad<float>, StoreOut<float>, true, true>(A, B, S, M, N, K, 1, st);
}

long long simt_conv_wgrad_workspace(const iic_conv_geom* g) {
  return (long long)wgrad_splits_simt(g) * g->cout * g->kh * g->kw * g->cin * (long long)sizeof(float);
}

// B operand of wgrad: element (nidx=(a,b,ci), k=pixel)
struct WgradXLoad {
  Im2colLoad<float> im;
  __device__ __forceinline__ float operator()(int nidx, int k) const { return im(k, nidx); }
};

int simt_conv_wgrad(const float* x, const float* dy, float* dw, float* ws, const iic_conv_geom* g, cudaStream_t st) {
  const int M = g->cout, N = g->kh * g->kw * g->cin;
  const long long P = (long long)g->n * g->oh * g->ow;
  IIC_REQUIRE(P < (1ll << 31), IIC_ERR_UNSUPPORTED, "simt wgrad: too many pixels");
  const int K = (int)P;
  const int splits = wgrad_splits_simt(g);
  DenseLoad<float> A{dy, 1, (long long)g->cout, M, K};  // A(co, pix) = dy[pix*cout + co]
  WgradXLoad B{Im2colLoad<float>{x, g->h, g->w, g->cin, g->oh, g->ow, g->kh, g->kw, g->stride, g->pad, g->dil, 0, K, N}};
  StorePartial S{ws};
  int rc = launch_simt<DenseLoad<float>, WgradXLoad, StorePartial, false, false>(A, B, S, M, N, K, splits, st);
  if (rc != IIC_OK) return rc;
  const long long count = (long long)M * N;
  int blocks = cdiv(count, 256);
  splitk_reduce_kernel<<<blocks, 256, 0, st>>>(ws, dw, count, splits, 0);
  IIC_LAUNCH_CHECK();
  count_launch();
  return IIC_OK;
}

// ---- heads: S x (Linear + Softmax(dim=1)) -- net5g_two_head.py:22-36 ---------------------------
// logits [n][S*k] -> z [S][n][k]; one warp per (row, sub-head)
__global__ void heads_softmax_kernel(const float* __restrict__ logits, float* __restrict__ z, int n, int S, int k) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n * S) return;
  const int r = warp / S, s = warp % S;
  const float* l = logits + (long long)r * S * k + (long long)s * k;
  float m = -INFINITY;
  for (int j = lane; j < k; j += 32) m = fmaxf(m, l[j]);
  m = warp_max(m);
  float sum = 0.f;
  for (int j = lane; j < k; j += 32) sum += expf(l[j] - m);
  sum = warp_sum(sum);
  float* o = z + ((long long)s * n + r) * k;
  for (int j = lane; j < k; j += 32) o[j] = expf(l[j] - m) / sum;
}
// dlogits[r][s*k+j] = z * (dz - sum_j dz*z)
__global__ void heads_softmax_bwd_kernel(const float* __restrict__ z, const float* __restrict__ dz,
                                         float* __restrict__ dlogits, int n, int S, int k) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n * S) return;
  const int r = warp / S, s = warp % S;
  const float* zz = z + ((long long)s * n + r) * k;
  const float* dd = dz + ((long long)s * n + r) * k;
  float dot = 0.f;
  for (int j = lane; j < k; j += 32) dot = fmaf(zz[j], dd[j], dot);
  dot = warp_sum(dot);
  float* o = dlogits + (long long)r * S * k + (long long)s * k;
  for (int j = lane; j < k; j += 32) o[j] = zz[j] * (dd[j] - dot);
}
__global__ void add_bias_kernel(float* __restrict__ logits, const float* __restrict__ b, long long n, int cols) {
  const long long total = n * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    logits[i] += b[i % cols];
}
__global__ void colsum_kernel(const float* __restrict__ a, float* __restrict__ out, int n, int cols) {
  // one block per 32 columns; deterministic
  __shared__ float sh[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), rg = threadIdx.x >> 5;
  float t = 0.f;
  if (c < cols)
    for (int r = rg; r < n; r += 8) t += a[(long long)r * cols + c];
  sh[rg][threadIdx.x & 31] = t;
  __syncthreads();
  if (rg == 0 && c < cols) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += sh[i][threadIdx.x & 31];
    out[c] = s;
  }
}

}  // namespace iic

using namespace iic;

// Per-device split-K scratch of heads_gemm (simt_gemm.cuh): grown, never freed -- a captured CUDA graph
// (iic_b200/graph.py) may hold the old pointer, and a later eager call with a larger batch (an evaluation pass between
// graphed training steps) must not pull it from under the replays.
float* iic::heads_scratch(size_t bytes) {
  static float* buf[64] = {nullptr};
  static size_t cap[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (cap[dev] < bytes) {
    float* nb = nullptr;
    if (cudaMalloc(&nb, bytes) != cudaSuccess) return nullptr;
    buf[dev] = nb;
    cap[dev] = bytes;
  }
  return buf[dev];
}

extern "C" int iic_heads_fwd(const float* feat, const float* w, const float* b, float* logits_ws, float* z, int n,
                             int F, int S, int k, void* stream) {
  IIC_REQUIRE(feat && w && b && logits_ws && z && n > 0 && F > 0 && S > 0 && k > 0, IIC_ERR_BAD_ARG,
              "iic_heads_fwd: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = S * k;
  DenseLoad<float> A{feat, (long long)F, 1, n, F};
  DenseLoad<float> B{w, (long long)F, 1, N, F};
  int rc = heads_gemm<DenseLoad<float>, DenseLoad<float>, true, true>(A, B, logits_ws, (long long)N, n, N, F, st);
  if (rc != IIC_OK) return rc;
  add_bias_kernel<<<cdiv((long long)n * N, 256), 256, 0, st>>>(logits_ws, b, n, N);
  IIC_LAUNCH_CHECK();
  count_launch();
  heads_softmax_kernel<<<cdiv((long long)n * S * 32, 256), 256, 0, st>>>(logits_ws, z, n, S, k);
  IIC_LAUNCH_CHECK();
  count_launch();
  return IIC_OK;
}

extern "C" int iic_heads_bwd(const float* feat, const float* w, const float* z, const float* dz, float* dlogits_ws,
                             float* dw, float* db, float* dfeat, int n, int F, int S, int k, void* stream) {
  IIC_REQUIRE(feat && w && z && dz && dlogits_ws && dw && db && n > 0 && F > 0 && S > 0 && k > 0, IIC_ERR_BAD_ARG,
              "iic_heads_bwd: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = S * k;
  heads_softmax_bwd_kernel<<<cdiv((long long)n * S * 32, 256), 256, 0, st>>>(z, dz, dlogits_ws, n, S, k);
  IIC_LAUNCH_CHECK();
  count_launch();
  colsum_kernel<<<cdiv(N, 32), 256, 0, st>>>(dlogits_ws, db, n, N);
  IIC_LAUNCH_CHECK();
  count_launch();
  {  // dw[N][F] = dlogits^T [N][n] x feat [n][F]
    DenseLoad<float> A{dlogits_ws, 1, (long long)N, N, n};  // A(i=col, k=row)
    DenseLoad<float> B{feat, 1, (long long)F, F, n};        // B(i=f, k=row)
    int rc = heads_gemm<DenseLoad<float>, DenseLoad<float>, false, false>(A, B, dw, (long long)F, N, F, n, st);
    if (rc != IIC_OK) return rc;
  }
  if (dfeat != nullptr) {  // dfeat[n][F] = dlogits [n][N] x w [N][F]
    DenseLoad<float> A{dlogits_ws, (long long)N, 1, n, N};
    DenseLoad<float> B{w, 1, (long long)F, F, N};  // B(i=f, k=col) = w[col*F + f]
    StoreOut<float> St{dfeat, nullptr, (long long)F};
    int rc = launch_simt<DenseLoad<float>, DenseLoad<float>, StoreOut<float>, true, false>(A, B, St, n, F, N, 1, st);
    if (rc != IIC_OK) return rc;
  }
  return IIC_OK;
}
