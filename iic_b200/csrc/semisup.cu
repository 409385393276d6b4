// Semi-supervised finetuning (code/scripts/semisup/IID_semisup_STL10.py): the supervised loss and the small dense
// layers of SupHead5 (code/archs/semisup/sup_head5.py) and of the `semisup` TwoHead heads (net5g_two_head.py:22-24,
// net6c_two_head.py:31-33).
//
//   iic_cross_entropy   nn.CrossEntropyLoss() (mean) over fp32 logits + its gradient, one launch: a thread-block
//                       cluster whose CTAs take fixed slices of rows; per-CTA fp64 sums are folded in rank order through
//                       distributed shared memory (no float atomics, bitwise reproducible, nothing to zero beforehand)
//   iic_linear_fwd/bwd  fp32 nn.Linear on the split-K SIMT GEMM of the sub-heads (heads_gemm, simt_gemm.cuh)
//   iic_col_sum         column sums of an fp32 / bf16 matrix (the bias gradient of a Linear whose output feeds a
//                       BatchNorm computed on the convolution engine)
//
// The wide first Linear of SupHead5 (dlen -> 2048) does not live here: it runs as a 1x1 convolution over n images of
// 1x1 pixels on the convolution entry points (conv_api.cu), see DESIGN.md S3.
#include <cooperative_groups.h>
#include <math.h>

#include "simt_gemm.cuh"

namespace cg = cooperative_groups;

namespace iic {

constexpr int CE_THREADS = 256;
constexpr int CE_MAX_CLUSTER = 8;

// One warp per row (rows strided over the whole cluster).  Per row: m = max, s = sum exp(l - m),
// nll = (m - l[t]) + log s, dlogits = (exp(l - m) / s - [j == t]) / n.  A target outside [0, k) makes that row's nll
// and its gradient NaN (so the mean is NaN); nothing traps and the host is not involved.
__global__ void __launch_bounds__(CE_THREADS) cross_entropy_kernel(const float* __restrict__ logits,
                                                                   const long long* __restrict__ targets, int n, int k,
                                                                   float* __restrict__ loss, float* __restrict__ dlogits) {
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ double red[33];
  __shared__ double part;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = CE_THREADS / 32;
  const int rank = (int)cluster.block_rank();
  const int gwarps = nwarps * (int)cluster.num_blocks();
  const float inv_n = 1.0f / (float)n;
  double acc = 0.0;  // lane 0: sum of this warp's row losses, in row order
  for (int r = rank * nwarps + warp; r < n; r += gwarps) {
    const float* l = logits + (long long)r * k;
    const long long t = targets[r];
    const bool valid = t >= 0 && t < k;
    float m = -INFINITY;
    for (int j = lane; j < k; j += 32) m = fmaxf(m, l[j]);
    m = warp_max(m);
    float s = 0.f;
    for (int j = lane; j < k; j += 32) s += expf(l[j] - m);
    s = warp_sum(s);
    const float inv_s = 1.0f / s;
    float* d = dlogits + (long long)r * k;
    for (int j = lane; j < k; j += 32) {
      const float p = expf(l[j] - m) * inv_s;
      d[j] = valid ? (p - (j == (int)t ? 1.0f : 0.0f)) * inv_n : __int_as_float(0x7fc00000);
    }
    if (lane == 0) acc += valid ? ((double)(m - l[t]) + (double)logf(s)) : (double)__int_as_float(0x7fc00000);
  }
  const double blk = block_sum(lane == 0 ? acc : 0.0, red);
  if (threadIdx.x == 0) part = blk;
  cluster.sync();
  if (rank == 0 && threadIdx.x == 0) {
    double tot = 0.0;
    for (int b = 0; b < (int)cluster.num_blocks(); ++b) tot += *cluster.map_shared_rank(&part, b);
    loss[0] = (float)(tot / (double)n);
  }
  cluster.sync();  // no CTA leaves while rank 0 still reads its shared memory
}

__global__ void bias_add_kernel(float* __restrict__ y, const float* __restrict__ b, long long rows, int cols) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    y[i] += b[i % cols];
}

// out[c] (=|+=) sum_r x[r][c]: one block per 32 columns, 8 row groups, folded in a fixed order (deterministic)
template <typename T>
__global__ void col_sum_kernel(const T* __restrict__ x, long long rows, int cols, float* __restrict__ out, int accumulate) {
  __shared__ float sh[8][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31), rg = threadIdx.x >> 5;
  float t = 0.f;
  if (c < cols)
    for (long long r = rg; r < rows; r += 8) t += to_f(x[r * cols + c]);
  sh[rg][threadIdx.x & 31] = t;
  __syncthreads();
  if (rg == 0 && c < cols) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += sh[i][threadIdx.x & 31];
    out[c] = accumulate ? out[c] + s : s;
  }
}

}  // namespace iic

using namespace iic;

extern "C" int iic_cross_entropy(const float* logits, const long long* targets, int n, int k, float* loss, float* dlogits,
                                 void* stream) {
  IIC_REQUIRE(logits && targets && loss && dlogits && n > 0 && k > 0, IIC_ERR_BAD_ARG, "iic_cross_entropy: bad arguments");
  int C = CE_MAX_CLUSTER;
  while (C > 1 && (n + C - 1) / C < CE_THREADS / 32) C >>= 1;  // small batches: fewer CTAs
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(C, 1, 1);
  cfg.blockDim = dim3(CE_THREADS, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  IIC_CUDA(cudaLaunchKernelEx(&cfg, cross_entropy_kernel, logits, targets, n, k, loss, dlogits));
  count_launch();
  return IIC_OK;
}

extern "C" int iic_linear_fwd(const float* x, const float* w, const float* b, float* y, int n, int K, int N, void* stream) {
  IIC_REQUIRE(x && w && y && n > 0 && K > 0 && N > 0, IIC_ERR_BAD_ARG, "iic_linear_fwd: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  DenseLoad<float> A{x, (long long)K, 1, n, K};
  DenseLoad<float> B{w, (long long)K, 1, N, K};
  int rc = heads_gemm<DenseLoad<float>, DenseLoad<float>, true, true>(A, B, y, (long long)N, n, N, K, st);
  if (rc != IIC_OK) return rc;
  if (b != nullptr) {
    long long blocks = cdiv((long long)n * N, 256);
    if (blocks > 1024) blocks = 1024;
    bias_add_kernel<<<(int)blocks, 256, 0, st>>>(y, b, n, N);
    IIC_LAUNCH_CHECK();
    count_launch();
  }
  return IIC_OK;
}

extern "C" int iic_linear_bwd(const float* x, const float* w, const float* dy, float* dw, float* db, float* dx, int accumulate,
                              int n, int K, int N, void* stream) {
  IIC_REQUIRE(x && w && dy && dw && n > 0 && K > 0 && N > 0, IIC_ERR_BAD_ARG, "iic_linear_bwd: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (db != nullptr) {
    col_sum_kernel<float><<<cdiv(N, 32), 256, 0, st>>>(dy, n, N, db, accumulate);
    IIC_LAUNCH_CHECK();
    count_launch();
  }
  {  // dw[N][K] (+)= dy^T [N][n] x x [n][K]
    DenseLoad<float> A{dy, 1, (long long)N, N, n};  // A(i = column of dy, k = row)
    DenseLoad<float> B{x, 1, (long long)K, K, n};   // B(i = feature, k = row)
    int rc = heads_gemm<DenseLoad<float>, DenseLoad<float>, false, false>(A, B, dw, (long long)K, N, K, n, st, accumulate);
    if (rc != IIC_OK) return rc;
  }
  if (dx != nullptr) {  // dx[n][K] = dy [n][N] x w [N][K]
    DenseLoad<float> A{dy, (long long)N, 1, n, N};
    DenseLoad<float> B{w, 1, (long long)K, K, N};  // B(i = feature, k = output) = w[k*K + i]
    StoreOut<float> St{dx, nullptr, (long long)K};
    int rc = launch_simt<DenseLoad<float>, DenseLoad<float>, StoreOut<float>, true, false>(A, B, St, n, K, N, 1, st);
    if (rc != IIC_OK) return rc;
  }
  return IIC_OK;
}

extern "C" int iic_col_sum(const void* x, int dtype, long long rows, int cols, float* out, int accumulate, void* stream) {
  IIC_REQUIRE(x && out && rows > 0 && cols > 0, IIC_ERR_BAD_ARG, "iic_col_sum: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == IIC_F32)
    col_sum_kernel<float><<<cdiv(cols, 32), 256, 0, st>>>((const float*)x, rows, cols, out, accumulate);
  else if (dtype == IIC_BF16)
    col_sum_kernel<__nv_bfloat16><<<cdiv(cols, 32), 256, 0, st>>>((const __nv_bfloat16*)x, rows, cols, out, accumulate);
  else
    IIC_REQUIRE(false, IIC_ERR_BAD_ARG, "iic_col_sum: bad dtype %d", dtype);
  IIC_LAUNCH_CHECK();
  count_launch();
  return IIC_OK;
}
