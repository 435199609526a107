// bsg_impute.cu -- snp_fastImputeSimple (R/impute.R:189-203 -> _bigsnpr_impute, src/impute-simple.cpp:10-73) over host
// bytes: the n x m FBM.code256 codes (CODE_012: 0 / 1 / 2, anything else missing) are imputed IN PLACE, column blocks
// uploaded, counted and filled on the device and downloaded again, on two streams so one block's copies run under the
// other's kernel and an FBM larger than HBM works.  Values written, as the reference writes them:
//   1 mode        4 + argmax(c0, c1, c2) with the reference's tie order (:51-57)
//   2 mean0       4 + fround(mean, 0),        mean = (c1 + 2.0 c2) / c
//   3 mean2       7 + fround(100 mean, 0)     (a CODE_DOSAGE code)
//   4 random      4 + two Bernoulli(af) draws, af = (0.5 c1 + c2) / c
// fround(x, 0) is R's round-half-to-even (nearbyint; R documents round(0.5) == 0).  The reference draws method 4 with
// R's Rf_rbinom, which cannot be reproduced outside R: here the draws come from a counter-based generator keyed by
// (seed, column, row), success iff u < rint(af 2^32) for a 32-bit u -- mirrored bit for bit by tests/impute_ref.py.  A
// column without any non-missing value (c = 0) is undefined behaviour in the reference for methods 2-4 (NaN cast to
// unsigned char): its bytes are left as they are and the column is counted in *n_all_missing; mode writes 4 like the
// reference.
#include <math.h>

#include <algorithm>

#include "bsg_internal.cuh"

namespace bsg {
namespace imp {

__device__ __forceinline__ uint64_t mix64(uint64_t x) {  // splitmix64 finaliser, as the synthetic generator
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

constexpr uint64_t DOMAIN = 0x696D707574650000ull;  // keeps these draws apart from the synthetic generator's

// one block per column of the block; col0 = global index of the first column
__global__ void __launch_bounds__(256) k_impute(uint8_t *__restrict__ X, int n, int ncols, int64_t col0, int method,
                                                uint64_t seed, int *__restrict__ n_all_missing) {
  __shared__ int cnt[3];
  __shared__ int fill;  // value to write (-1: leave the column as it is); method 4: 1
  __shared__ unsigned long long thr;
  for (int jj = blockIdx.x; jj < ncols; jj += gridDim.x) {
    uint8_t *col = X + (int64_t)jj * n;
    if (threadIdx.x < 3) cnt[threadIdx.x] = 0;
    __syncthreads();
    int c1 = 0, c2 = 0, cna = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const uint8_t g = col[i];
      c1 += g == 1;
      c2 += g == 2;
      cna += g > 2;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      c1 += __shfl_xor_sync(0xffffffffu, c1, o);
      c2 += __shfl_xor_sync(0xffffffffu, c2, o);
      cna += __shfl_xor_sync(0xffffffffu, cna, o);
    }
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(&cnt[0], c1);
      atomicAdd(&cnt[1], c2);
      atomicAdd(&cnt[2], cna);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      const int k1 = cnt[0], k2 = cnt[1], c = n - cnt[2];
      int v = -1;
      if (cnt[2] > 0) {
        if (c == 0) atomicAdd(n_all_missing, 1);
        if (method == 1) {
          const int c0 = c - (k1 + k2);
          int imputed = 0;
          if (k1 > c0) imputed = 1;
          if (imputed == 0 && k2 > c0) imputed = 2;
          if (imputed == 1 && k2 > k1) imputed = 2;
          v = imputed + 4;
        } else if (c > 0) {
          if (method == 4) {
            const double af = (0.5 * k1 + k2) / c;
            thr = (unsigned long long)rint(af * 4294967296.0);
            v = 1;
          } else {
            const double mean = (k1 + 2.0 * k2) / c;
            v = method == 2 ? (int)rint(mean) + 4 : (int)rint(100 * mean) + 7;
          }
        }
      }
      fill = v;
    }
    __syncthreads();
    const int v = fill;
    if (v >= 0) {
      const uint64_t kj = mix64((seed ^ DOMAIN) ^ mix64((uint64_t)(col0 + jj)));
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        if (col[i] <= 2) continue;
        if (method == 4) {
          const uint64_t h = mix64(kj + (uint64_t)i * 0xD1342543DE82EF95ull);
          const int d = ((h & 0xFFFFFFFFull) < thr) + ((h >> 32) < thr);
          col[i] = (uint8_t)(4 + d);
        } else {
          col[i] = (uint8_t)v;
        }
      }
    }
    __syncthreads();  // fill / cnt are rewritten for the next column
  }
}

}  // namespace imp
}  // namespace bsg

using namespace bsg;

extern "C" int bsg_impute(uint8_t *bytes, int n, int m, int method, uint64_t seed, int device, int *n_all_missing) {
  if (!bytes && (int64_t)n * m > 0) return fail(BSG_ERR_ARG, "null argument");
  if (n <= 0 || m < 0) return fail(BSG_ERR_ARG, "n must be positive and m non-negative.");
  if (method < 1 || method > 4) return fail(BSG_ERR_ARG, "Parameter 'method' should be 1, 2, 3, or 4.");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(BSG_ERR_CUDA, "No CUDA device available: libbsgpu has no CPU fallback.");
  if (device < 0 || device >= ndev) return fail(BSG_ERR_ARG, "device %d out of range (0..%d).", device, ndev - 1);
  BSG_CUDA(cudaSetDevice(device));
  if (n_all_missing) *n_all_missing = 0;
  if (m == 0) return BSG_OK;
  // blocks of columns of <= 256 MB, two in flight
  const int bc = (int)std::max<int64_t>(1, std::min<int64_t>(m, (int64_t)(256 << 20) / n));
  cudaStream_t st[2] = {nullptr, nullptr};
  uint8_t *buf[2] = {nullptr, nullptr};
  int *d_cnt = nullptr;
  int rc = BSG_OK;
  for (int k = 0; k < 2 && !rc; k++) {
    e = cudaStreamCreateWithFlags(&st[k], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&buf[k], (size_t)bc * n);
    if (e != cudaSuccess) rc = cuda_fail(e, "impute buffers");
  }
  if (!rc) {
    e = cudaMalloc(&d_cnt, sizeof(int));
    if (e == cudaSuccess) e = cudaMemsetAsync(d_cnt, 0, sizeof(int), st[0]);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st[0]);
    if (e != cudaSuccess) rc = cuda_fail(e, "impute counter");
  }
  for (int64_t j0 = 0, b = 0; j0 < m && !rc; j0 += bc, b++) {
    const int k = (int)(b & 1), nb = (int)std::min<int64_t>(bc, m - j0);
    const size_t len = (size_t)nb * n;
    e = cudaMemcpyAsync(buf[k], bytes + j0 * n, len, cudaMemcpyHostToDevice, st[k]);
    if (e == cudaSuccess) {
      imp::k_impute<<<std::min(nb, 148 * 8), 256, 0, st[k]>>>(buf[k], n, nb, j0, method, seed, d_cnt);
      count_launch();
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(bytes + j0 * n, buf[k], len, cudaMemcpyDeviceToHost, st[k]);
    if (e != cudaSuccess) rc = cuda_fail(e, "impute block");
  }
  for (int k = 0; k < 2; k++)
    if (st[k]) {
      e = cudaStreamSynchronize(st[k]);
      if (e != cudaSuccess && !rc) rc = cuda_fail(e, "impute");
    }
  if (!rc && n_all_missing) {
    e = cudaMemcpy(n_all_missing, d_cnt, sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = cuda_fail(e, "impute counter");
  }
  for (int k = 0; k < 2; k++) {
    if (buf[k]) cudaFree(buf[k]);
    if (st[k]) cudaStreamDestroy(st[k]);
  }
  if (d_cnt) cudaFree(d_cnt);
  return rc;
}
