// bsg_core.cu -- handles, staging of the packed genotypes to HBM, layout transforms, counts.
//
// Replaces class bed / bedXPtr of the reference (src/bed-acc.h:18-48, src/bed-acc-xptr.cpp:14-55):
// instead of an mmap that every accessor call walks byte by byte, the file is validated with the
// same three checks, recoded once to the "staged code" (bsg_internal.cuh) and kept in HBM.
#include <errno.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <vector>

#include "bsg_internal.cuh"

namespace bsg {

thread_local std::string g_err;
static std::atomic<long long> g_launches{0};

void count_launch(int n) { g_launches += n; }

int fail(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

int cuda_fail(cudaError_t e, const char *what) {
  return fail(BSG_ERR_CUDA, "CUDA error: %s (%s)", cudaGetErrorString(e), what);
}

int DevBuf::ensure(size_t bytes) {
  if (bytes <= cap && p) return BSG_OK;
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
  size_t want = bytes < 256 ? 256 : bytes;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(scratch)");
  cap = want;
  return BSG_OK;
}

void DevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}

// Large per-call work buffers (expanded Gram operands, pair statistics) come from the device's stream-ordered pool with a
// high release threshold: the second call of a session (LD scores, then correlations, then clumping on the same data) reuses
// the pages instead of paying cudaMalloc / cudaFree of tens of GB each time.  cudaFree on such a pointer returns it to
// the pool.
cudaError_t pool_alloc(void **p, size_t bytes, int device, cudaStream_t s) {
  static unsigned configured = 0;  // one bit per device
  if (!(configured >> (device & 31) & 1u)) {
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long thr = (unsigned long long)48 << 30;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    cudaGetLastError();
    configured |= 1u << (device & 31);
  }
  cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 16, s);
  if (e != cudaSuccess) {  // pool exhausted or fragmented: trim and take the plain path
    cudaGetLastError();
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
    cudaGetLastError();
    e = cudaMalloc(p, bytes ? bytes : 16);
  }
  return e;
}

// First touch of a large, possibly untouched host OUTPUT buffer from several threads (one write per 4 KB page): a fresh
// allocation faults in at ~1.5 GB/s when one thread (or the copy engine's staging loop) touches it, which dominated the
// calls that return GBs (CSC of bsg_cor, K of bsg_tcrossprod).  Only for buffers the call overwrites completely.
void prefault_pages(void *p, size_t bytes) {
  if (bytes < ((size_t)64 << 20)) return;
  unsigned hw = std::thread::hardware_concurrency();
  const int nt = (int)std::max(1u, std::min(hw ? hw : 1u, 16u));
  std::vector<std::thread> th;
  const size_t per = (bytes / nt + 4095) & ~(size_t)4095;
  for (int t = 0; t < nt; t++) {
    const size_t b0 = (size_t)t * per, b1 = std::min(bytes, b0 + per);
    if (b0 >= b1) break;
    th.emplace_back([=]() {
      volatile char *q = static_cast<volatile char *>(p);
      for (size_t o = b0; o < b1; o += 4096) q[o] = 0;
      q[b1 - 1] = 0;
    });
  }
  for (auto &x : th) x.join();
}

int bind_device(const bsg_bed *h) {
  BSG_CUDA(cudaSetDevice(h->device));
  return BSG_OK;
}

// ---------------------------------------------------------------------------------------------
// .bed code <-> staged code, per byte (4 genotypes).  bed code (hi,lo): 00->g2, 01->NA, 10->g1,
// 11->g0 (src/bed-acc.h:22-37).  staged (hi',lo') = (~hi, hi^lo): g2->10, NA->11, g1->01, g0->00.
__host__ __device__ inline uint32_t bed_to_staged32(uint32_t b) {
  return ((~b) & 0xAAAAAAAAu) | (((b >> 1) ^ b) & 0x55555555u);
}
__host__ __device__ inline uint32_t staged_to_bed32(uint32_t s) {
  return ((~s) & 0xAAAAAAAAu) | ((((~s) >> 1) ^ s) & 0x55555555u);
}

// raw file bytes (column stride n_byte) -> staged copy A (line stride strideA), pads zeroed.
__global__ void k_stage_bed(const uint8_t *__restrict__ raw, int64_t n_byte, int n, int ncols,
                            uint8_t *__restrict__ A, int64_t strideA) {
  int64_t words = strideA / 4;
  int64_t total = (int64_t)ncols * words;
  int tail = n & 3;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t j = t / words, wq = t - j * words;
    const uint8_t *src = raw + j * n_byte + wq * 4;
    uint32_t v = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      int64_t by = wq * 4 + k;
      if (by < n_byte) {
        uint32_t b = bed_to_staged32(src[k]) & 0xFFu;
        if (by == n_byte - 1 && tail) b &= (1u << (2 * tail)) - 1u;
        v |= b << (8 * k);
      }
    }
    reinterpret_cast<uint32_t *>(A + j * strideA)[wq] = v;
  }
}

// FBM.code256 raw bytes (n x m, column-major) -> staged copy A.  map[256]: staged code per byte.
__global__ void k_stage_fbm(const uint8_t *__restrict__ raw, int n, int ncols, const uint8_t *__restrict__ map,
                            uint8_t *__restrict__ A, int64_t strideA) {
  int64_t words = strideA / 4;
  int64_t total = (int64_t)ncols * words;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t j = t / words, wq = t - j * words;
    uint32_t v = 0;
#pragma unroll
    for (int p = 0; p < 16; p++) {
      int64_t i = wq * 16 + p;
      if (i < n) v |= (uint32_t)map[raw[j * (int64_t)n + i]] << (2 * p);
    }
    reinterpret_cast<uint32_t *>(A + j * strideA)[wq] = v;
  }
}

// staged copy A -> .bed bytes (pad slots written as 00 like PLINK).
__global__ void k_export_bed(const uint8_t *__restrict__ A, int64_t strideA, int64_t n_byte, int n, int ncols,
                             uint8_t *__restrict__ out) {
  int64_t total = (int64_t)ncols * n_byte;
  int tail = n & 3;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t j = t / n_byte, by = t - j * n_byte;
    uint32_t b = staged_to_bed32(A[j * strideA + by]) & 0xFFu;
    if (by == n_byte - 1 && tail) b &= (1u << (2 * tail)) - 1u;
    out[t] = (uint8_t)b;
  }
}

// ---------------------------------------------------------------------------------------------
// synthetic generator (SURVEY.md section 8d).  Mirrored bit for bit by tests/synth_ref.py.
__host__ __device__ inline uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void k_synth(uint8_t *__restrict__ A, int64_t strideA, int n, int ncols, uint64_t seed,
                        int64_t col_offset, uint32_t na_thr) {
  int64_t words = strideA / 4;
  int64_t total = (int64_t)ncols * words;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    int64_t j = t / words, wq = t - j * words;
    uint64_t kj = mix64(seed ^ mix64((uint64_t)(col_offset + j)));
    double maf = 0.02 + 0.48 * ((double)(kj >> 11) * (1.0 / 9007199254740992.0));
    uint32_t thr = (uint32_t)(maf * 16777216.0);
    uint32_t v = 0;
#pragma unroll 4
    for (int p = 0; p < 16; p++) {
      int64_t i = wq * 16 + p;
      if (i < n) {
        uint64_t hs = mix64(kj + (uint64_t)i * 0xD1342543DE82EF95ull);
        uint32_t g = ((uint32_t)(hs & 0xFFFFFFu) < thr) + ((uint32_t)((hs >> 24) & 0xFFFFFFu) < thr);
        if ((uint32_t)((hs >> 48) & 0xFFFFu) < na_thr) g = 3;
        v |= g << (2 * p);
      }
    }
    reinterpret_cast<uint32_t *>(A + j * strideA)[wq] = v;
  }
}


// LD-structured variant (SURVEY.md section 8d, "AR(1) haplotypes within blocks"): same per-(sample, SNP) hash as
// k_synth, but the two 24-bit allele uniforms of a haplotype are COPIED from the previous SNP with probability rho
// (a second hash decides, 16 bits per haplotype) unless the SNP starts a block of `ldblock` global columns.  Two
// neighbouring SNPs that share the uniform carry alleles [u < maf_j] and [u < maf_j'], i.e. r close to 1 for similar
// allele frequencies: real windows of correlated variants for the clumping / r2-threshold paths.  Integer
// arithmetic only, so a CPU twin reproduces the matrix bit for bit; rho = 0 is exactly k_synth.
// One thread = 16 samples x one block of columns, walking the block in order with the 32 states in registers.
__global__ void k_synth_ld(uint8_t *__restrict__ A, int64_t strideA, int n, int ncols, uint64_t seed,
                           int64_t col_offset, uint32_t na_thr, uint32_t rho_thr, int ldblock) {
  const int64_t words = strideA / 4;
  const int64_t gb0 = col_offset / ldblock;                              // first global block touched
  const int64_t nblk = (col_offset + ncols + ldblock - 1) / ldblock - gb0;
  const int64_t total = nblk * words;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = t / words, wq = t - b * words;
    const int64_t g0 = (gb0 + b) * ldblock;
    int64_t g1 = g0 + ldblock;
    if (g1 > col_offset + ncols) g1 = col_offset + ncols;
    uint32_t u0[16], u1[16];
#pragma unroll
    for (int p = 0; p < 16; p++) u0[p] = u1[p] = 0;
    for (int64_t gj = g0; gj < g1; gj++) {
      const uint64_t kj = mix64(seed ^ mix64((uint64_t)gj));
      const double maf = 0.02 + 0.48 * ((double)(kj >> 11) * (1.0 / 9007199254740992.0));
      const uint32_t thr = (uint32_t)(maf * 16777216.0);
      const bool first = gj == g0;
      uint32_t v = 0;
#pragma unroll
      for (int p = 0; p < 16; p++) {
        const int64_t i = wq * 16 + p;
        const uint64_t hs = mix64(kj + (uint64_t)i * 0xD1342543DE82EF95ull);
        const uint64_t h2 = mix64(hs ^ 0xA5A5A5A5A5A5A5A5ull);
        const bool c0 = !first && (uint32_t)(h2 & 0xFFFFu) < rho_thr;
        const bool c1 = !first && (uint32_t)((h2 >> 16) & 0xFFFFu) < rho_thr;
        if (!c0) u0[p] = (uint32_t)(hs & 0xFFFFFFu);
        if (!c1) u1[p] = (uint32_t)((hs >> 24) & 0xFFFFFFu);
        uint32_t g = (u0[p] < thr) + (u1[p] < thr);
        if ((uint32_t)((hs >> 48) & 0xFFFFu) < na_thr) g = 3;
        if (i < n) v |= g << (2 * p);
      }
      if (gj >= col_offset) reinterpret_cast<uint32_t *>(A + (gj - col_offset) * strideA)[wq] = v;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// copy A -> copy B (2-bit transpose).  Tile: 128 SNP lines x 128 B (512 samples) in, 512 sample
// lines x 32 B (128 SNPs) out.  One thread per sample of the tile.
__global__ void __launch_bounds__(512) k_transpose(const uint8_t *__restrict__ A, int64_t strideA, int n, int m,
                                                   uint8_t *__restrict__ B, int64_t strideB) {
  __shared__ uint32_t tile[128][33];  // [snp][word], +1 pad
  int64_t snp0 = (int64_t)blockIdx.x * 128;
  int64_t byte0 = (int64_t)blockIdx.y * 128;  // sample byte offset in A lines
  int tid = threadIdx.x;
  // load: 128 lines x 32 words
  for (int e = tid; e < 128 * 32; e += 512) {
    int l = e >> 5, wq = e & 31;
    int64_t j = snp0 + l;
    uint32_t v = 0;
    if (j < m && byte0 + wq * 4 < strideA) v = reinterpret_cast<const uint32_t *>(A + j * strideA + byte0)[wq];
    tile[l][wq] = v;
  }
  __syncthreads();
  int64_t i = byte0 * 4 + tid;  // sample
  if (i >= n) return;
  int wq = tid >> 4, sh = 2 * (tid & 15);
  uint32_t outw[8];
#pragma unroll
  for (int ow = 0; ow < 8; ow++) {
    uint32_t v = 0;
#pragma unroll
    for (int p = 0; p < 16; p++) v |= ((tile[ow * 16 + p][wq] >> sh) & 3u) << (2 * p);
    outw[ow] = v;
  }
  uint4 *dst = reinterpret_cast<uint4 *>(B + i * strideB + snp0 / 4);
  dst[0] = make_uint4(outw[0], outw[1], outw[2], outw[3]);
  dst[1] = make_uint4(outw[4], outw[5], outw[6], outw[7]);
}

// per-line counts of codes {0,1,2,3} over the first L codes of each line (pads are code 0 and are
// subtracted through L), plus the has-NA flag.  One warp per line.
__global__ void k_line_counts(const uint8_t *__restrict__ P, int64_t stride, int nlines, int L,
                              int32_t *__restrict__ cnt, uint8_t *__restrict__ na) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  int nw = (gridDim.x * blockDim.x) >> 5;
  int64_t nvec = ((int64_t)(L + 3) / 4 + 15) / 16;  // uint4 per line actually holding data
  for (int l = warp; l < nlines; l += nw) {
    const uint4 *src = reinterpret_cast<const uint4 *>(P + (int64_t)l * stride);
    int c1 = 0, c2 = 0, c3 = 0;
    for (int64_t v = lane; v < nvec; v += 32) {
      uint4 q = __ldg(src + v);
      uint32_t ws[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        uint32_t lo = ws[k] & 0x55555555u, hi = (ws[k] >> 1) & 0x55555555u;
        c3 += __popc(lo & hi);
        c1 += __popc(lo & ~hi);
        c2 += __popc(hi & ~lo);
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      c1 += __shfl_xor_sync(0xffffffffu, c1, o);
      c2 += __shfl_xor_sync(0xffffffffu, c2, o);
      c3 += __shfl_xor_sync(0xffffffffu, c3, o);
    }
    if (lane == 0) {
      cnt[4 * (int64_t)l + 0] = L - c1 - c2 - c3;
      cnt[4 * (int64_t)l + 1] = c1;
      cnt[4 * (int64_t)l + 2] = c2;
      cnt[4 * (int64_t)l + 3] = c3;
      na[l] = c3 > 0;
    }
  }
}

__global__ void k_any_nonzero(const uint8_t *__restrict__ f, int64_t n, int *__restrict__ out) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int any = 0;
  for (; t < n; t += (int64_t)gridDim.x * blockDim.x) any |= f[t];
  if (__any_sync(0xffffffffu, any) && (threadIdx.x & 31) == 0) atomicOr(out, 1);
}

static int grid_for(int64_t work, int block) {
  int64_t g = (work + block - 1) / block;
  if (g < 1) g = 1;
  if (g > 148 * 32) g = 148 * 32;
  return (int)g;
}

static int alloc_handle(int n, int m, int device, bsg_bed **out) {
  if (n <= 0 || m <= 0) return fail(BSG_ERR_ARG, "n and m must be positive.");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(BSG_ERR_CUDA, "No CUDA device available (%s): libbsgpu has no CPU fallback.",
                e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(BSG_ERR_ARG, "device %d out of range (0..%d).", device, ndev - 1);
  BSG_CUDA(cudaSetDevice(device));
  bsg_bed *h = new bsg_bed();
  h->device = device;
  h->n = n;
  h->m = m;
  h->n_byte = ((int64_t)n + 3) / 4;
  h->strideA = round_up(h->n_byte, 128);
  h->strideB = round_up(((int64_t)m + 3) / 4, 128);
  cudaError_t e1 = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  cudaError_t e2 = cudaEventCreate(&h->ev0);
  cudaError_t e3 = cudaEventCreate(&h->ev1);
  if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
    delete h;
    return fail(BSG_ERR_CUDA, "cannot create stream/events");
  }
  e = cudaMalloc(&h->A, (size_t)h->strideA * m);
  if (e != cudaSuccess) {
    double gb = (double)h->strideA * m / 1e9;
    cudaGetLastError();
    bsg_close(h);
    return fail(BSG_ERR_ALLOC, "cannot allocate %.2f GB of HBM for the packed genotypes (%s).", gb,
                cudaGetErrorString(e));
  }
  for (int k = 0; k < 256; k++) h->code256[k] = 0;
  *out = h;
  return BSG_OK;
}

int stage_finish(bsg_bed *h) {
  cudaStream_t s = h->stream;
  // counts + NA flags on copy A
  BSG_CUDA(cudaMalloc(&h->cntA, (size_t)h->m * 4 * sizeof(int32_t)));
  BSG_CUDA(cudaMalloc(&h->naA, (size_t)h->m));
  k_line_counts<<<grid_for((int64_t)h->m * 32, 256), 256, 0, s>>>(h->A, h->strideA, h->m, h->n, h->cntA, h->naA);
  count_launch();
  int *d_any = nullptr;
  BSG_CUDA(cudaMalloc(&d_any, sizeof(int)));
  BSG_CUDA(cudaMemsetAsync(d_any, 0, sizeof(int), s));
  k_any_nonzero<<<grid_for(h->m, 256), 256, 0, s>>>(h->naA, h->m, d_any);
  count_launch();
  BSG_CUDA(cudaMemcpyAsync(&h->has_na, d_any, sizeof(int), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaStreamSynchronize(s));
  cudaFree(d_any);

  // Layout policy: the SNP-major copy serves every kernel at full speed (X.y included, k_pmvT), so AUTO stages it
  // alone -- half the HBM footprint, no transpose at open.  The sample-major copy is built when asked for
  // (BSG_LAYOUT_SAMPLE_MAJOR) or on first use by the GRM tiles (build_copy_B).
  int want = h->layouts;
  if (want == BSG_LAYOUT_AUTO) want = BSG_LAYOUT_SNP_MAJOR;
  want |= BSG_LAYOUT_SNP_MAJOR;
  h->layouts = BSG_LAYOUT_SNP_MAJOR;
  if (want & BSG_LAYOUT_SAMPLE_MAJOR) BSG_TRY(build_copy_B(h));
  BSG_CUDA(cudaStreamSynchronize(s));
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

// the 2-bit transpose (line i = sample i) with its per-line counts and missing-value flags
int build_copy_B(bsg_bed *h) {
  if (h->B) return BSG_OK;
  cudaStream_t s = h->stream;
  uint8_t *B = nullptr, *naB = nullptr;
  int32_t *cntB = nullptr;
  cudaError_t e = cudaMalloc(&B, (size_t)h->strideB * h->n);
  if (e == cudaSuccess) e = cudaMalloc(&cntB, (size_t)h->n * 4 * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMalloc(&naB, (size_t)h->n);
  if (e == cudaSuccess) e = cudaMemsetAsync(B, 0, (size_t)h->strideB * h->n, s);
  if (e == cudaSuccess) {
    dim3 grid((unsigned)((h->m + 127) / 128), (unsigned)((h->strideA + 127) / 128));
    k_transpose<<<grid, 512, 0, s>>>(h->A, h->strideA, h->n, h->m, B, h->strideB);
    k_line_counts<<<grid_for((int64_t)h->n * 32, 256), 256, 0, s>>>(B, h->strideB, h->n, h->m, cntB, naB);
    count_launch(2);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {  // all or nothing: a half-built copy must never be visible to the kernels
    cudaGetLastError();
    cudaFree(B);
    cudaFree(cntB);
    cudaFree(naB);
    return fail(BSG_ERR_ALLOC, "cannot build the sample-major copy (%.2f GB): %s.", (double)h->strideB * h->n / 1e9,
                cudaGetErrorString(e));
  }
  h->B = B;
  h->cntB = cntB;
  h->naB = naB;
  h->layouts |= BSG_LAYOUT_SAMPLE_MAJOR;
  return BSG_OK;
}

int upload_index(bsg_bed *h, const int *ind, int len, int limit, DevBuf &buf, const int **dev) {
  *dev = nullptr;
  if (!ind) return BSG_OK;
  std::vector<int> z((size_t)(len > 0 ? len : 1));
  for (int i = 0; i < len; i++) {
    long long v = (long long)ind[i] - 1;
    if (v < 0 || v >= limit) return fail(BSG_ERR_BOUNDS, "Tested subscript out of bounds (%d not in 1..%d).", ind[i], limit);
    z[i] = (int)v;
  }
  BSG_TRY(buf.ensure((size_t)(len > 0 ? len : 1) * sizeof(int)));
  BSG_CUDA(cudaMemcpyAsync(buf.p, z.data(), (size_t)len * sizeof(int), cudaMemcpyHostToDevice, h->stream));
  BSG_CUDA(cudaStreamSynchronize(h->stream));  // z goes out of scope
  *dev = buf.as<int>();
  return BSG_OK;
}

}  // namespace bsg

using namespace bsg;

// =============================================================================================
extern "C" {

const char *bsg_last_error(void) { return g_err.c_str(); }
int bsg_version(void) { return 100; }
int64_t bsg_launch_count(void) { return (int64_t)g_launches.load(); }

int bsg_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int bsg_open_bed(const char *path, int n, int m, int col_begin, int col_end, int device, int layouts,
                 bsg_bed **out) {
  if (!out || !path) return fail(BSG_ERR_ARG, "null argument");
  *out = nullptr;
  // --- the reference's checks, in the reference's order (src/bed-acc-xptr.cpp:16-34) ---
  FILE *f = fopen(path, "rb");
  if (!f) return fail(BSG_ERR_IO, "Error when mapping file:\n  %s.\n", strerror(errno));
  unsigned char hdr[3] = {0, 0, 0};
  size_t got = fread(hdr, 1, 3, f);
  struct stat st;
  if (fstat(fileno(f), &st) != 0) {
    fclose(f);
    return fail(BSG_ERR_IO, "Error when mapping file:\n  %s.\n", strerror(errno));
  }
  if (got < 2 || !(hdr[0] == 0x6C && hdr[1] == 0x1B)) {
    fclose(f);
    return fail(BSG_ERR_MAGIC, "File is not a binary PED file.");
  }
  if (got < 3 || hdr[2] != 0x01) {
    fclose(f);
    return fail(BSG_ERR_MODE, "Variant-major is the only mode supported.");
  }
  int64_t n_byte = ((int64_t)n + 3) / 4;
  if (n <= 0 || m <= 0 || 3 + n_byte * (int64_t)m != (int64_t)st.st_size) {
    fclose(f);
    return fail(BSG_ERR_SIZE, "n or p does not match the dimensions of the file.");
  }
  if (col_begin < 0 || col_end > m || col_begin >= col_end) {
    fclose(f);
    return fail(BSG_ERR_ARG, "column range [%d, %d) is not inside [0, %d).", col_begin, col_end, m);
  }
  int mloc = col_end - col_begin;
  bsg_bed *h = nullptr;
  int rc = alloc_handle(n, mloc, device, &h);
  if (rc) {
    fclose(f);
    return rc;
  }
  h->layouts = layouts;
  // --- stream the column range through a pinned double buffer ---
  const size_t CH = (size_t)64 << 20;
  int64_t cols_per = (int64_t)(CH / (size_t)n_byte);
  if (cols_per < 1) cols_per = 1;
  if (cols_per > mloc) cols_per = mloc;
  size_t chunk_bytes = (size_t)cols_per * n_byte;
  uint8_t *pin[2] = {nullptr, nullptr}, *draw[2] = {nullptr, nullptr};
  cudaEvent_t done[2] = {nullptr, nullptr};
  cudaError_t ce = cudaSuccess;
  for (int b = 0; b < 2 && ce == cudaSuccess; b++) {
    ce = cudaMallocHost(&pin[b], chunk_bytes);
    if (ce == cudaSuccess) ce = cudaMalloc(&draw[b], chunk_bytes);
    if (ce == cudaSuccess) ce = cudaEventCreate(&done[b]);
  }
  rc = BSG_OK;
  if (ce != cudaSuccess) rc = cuda_fail(ce, "staging buffers");
  if (!rc && fseeko(f, (off_t)(3 + n_byte * (int64_t)col_begin), SEEK_SET) != 0) rc = fail(BSG_ERR_IO, "seek failed");
  int64_t j0 = 0;
  int b = 0;
  while (!rc && j0 < mloc) {
    int64_t nc = cols_per < mloc - j0 ? cols_per : mloc - j0;
    cudaEventSynchronize(done[b]);
    size_t want = (size_t)nc * n_byte;
    if (fread(pin[b], 1, want, f) != want) {
      rc = fail(BSG_ERR_IO, "short read on %s", path);
      break;
    }
    ce = cudaMemcpyAsync(draw[b], pin[b], want, cudaMemcpyHostToDevice, h->stream);
    if (ce != cudaSuccess) { rc = cuda_fail(ce, "H2D"); break; }
    k_stage_bed<<<grid_for(nc * (h->strideA / 4), 256), 256, 0, h->stream>>>(draw[b], n_byte, n, (int)nc,
                                                                           h->A + j0 * h->strideA, h->strideA);
    count_launch();
    cudaEventRecord(done[b], h->stream);
    j0 += nc;
    b ^= 1;
  }
  fclose(f);
  cudaStreamSynchronize(h->stream);
  for (int k = 0; k < 2; k++) {
    if (pin[k]) cudaFreeHost(pin[k]);
    if (draw[k]) cudaFree(draw[k]);
    if (done[k]) cudaEventDestroy(done[k]);
  }
  if (!rc) {
    ce = cudaGetLastError();
    if (ce != cudaSuccess) rc = cuda_fail(ce, "staging");
  }
  if (!rc) rc = stage_finish(h);
  if (rc) {
    bsg_close(h);
    return rc;
  }
  *out = h;
  return BSG_OK;
}

int bsg_open_packed(const uint8_t *packed, int n, int m, int device, int layouts, bsg_bed **out) {
  if (!out || !packed) return fail(BSG_ERR_ARG, "null argument");
  *out = nullptr;
  bsg_bed *h = nullptr;
  BSG_TRY(alloc_handle(n, m, device, &h));
  h->layouts = layouts;
  uint8_t *draw = nullptr;
  size_t bytes = (size_t)h->n_byte * m;
  cudaError_t ce = cudaMalloc(&draw, bytes);
  if (ce == cudaSuccess) ce = cudaMemcpy(draw, packed, bytes, cudaMemcpyHostToDevice);
  int rc = BSG_OK;
  if (ce != cudaSuccess) rc = cuda_fail(ce, "upload packed");
  if (!rc) {
    k_stage_bed<<<grid_for((int64_t)m * (h->strideA / 4), 256), 256, 0, h->stream>>>(draw, h->n_byte, n, m, h->A,
                                                                                     h->strideA);
    count_launch();
    cudaStreamSynchronize(h->stream);
  }
  if (draw) cudaFree(draw);
  if (!rc) rc = stage_finish(h);
  if (rc) {
    bsg_close(h);
    return rc;
  }
  *out = h;
  return BSG_OK;
}

int bsg_open_synth(int n, int m, uint64_t seed, double na_rate, int64_t col_offset, int device, int layouts,
                   bsg_bed **out) {
  if (!out) return fail(BSG_ERR_ARG, "null argument");
  *out = nullptr;
  if (!(na_rate >= 0 && na_rate < 1)) return fail(BSG_ERR_ARG, "na_rate must be in [0, 1).");
  bsg_bed *h = nullptr;
  BSG_TRY(alloc_handle(n, m, device, &h));
  h->layouts = layouts;
  uint32_t na_thr = (uint32_t)(na_rate * 65536.0);
  k_synth<<<grid_for((int64_t)m * (h->strideA / 4), 256), 256, 0, h->stream>>>(h->A, h->strideA, n, m, seed, col_offset,
                                                                               na_thr);
  count_launch();
  int rc = stage_finish(h);
  if (rc) {
    bsg_close(h);
    return rc;
  }
  *out = h;
  return BSG_OK;
}


int bsg_open_synth_ld(int n, int m, uint64_t seed, double na_rate, int64_t col_offset, double rho, int ld_block,
                      int device, int layouts, bsg_bed **out) {
  if (!out) return fail(BSG_ERR_ARG, "null argument");
  *out = nullptr;
  if (!(na_rate >= 0 && na_rate < 1)) return fail(BSG_ERR_ARG, "na_rate must be in [0, 1).");
  if (!(rho >= 0 && rho < 1) || ld_block < 1 || col_offset < 0) return fail(BSG_ERR_ARG, "rho must be in [0, 1), ld_block >= 1.");
  bsg_bed *h = nullptr;
  BSG_TRY(alloc_handle(n, m, device, &h));
  h->layouts = layouts;
  const uint32_t na_thr = (uint32_t)(na_rate * 65536.0), rho_thr = (uint32_t)(rho * 65536.0);
  const int64_t nblk = (col_offset + m + ld_block - 1) / ld_block - col_offset / ld_block;
  k_synth_ld<<<grid_for(nblk * (h->strideA / 4), 128), 128, 0, h->stream>>>(h->A, h->strideA, n, m, seed, col_offset, na_thr,
                                                                           rho_thr, ld_block);
  count_launch();
  int rc = stage_finish(h);
  if (rc) {
    bsg_close(h);
    return rc;
  }
  *out = h;
  return BSG_OK;
}

int bsg_open_fbm256(const uint8_t *bytes, int n, int m, const double *code256, int device, int layouts,
                    bsg_bed **out) {
  if (!out || !bytes || !code256) return fail(BSG_ERR_ARG, "null argument");
  *out = nullptr;
  uint8_t map[256];
  bool generic = false;  // a code other than 0 / 1 / 2 / NA (dosages, CODE_DOSAGE): the handle keeps the bytes, fp64 kernels
  for (int k = 0; k < 256; k++) {
    double v = code256[k];
    if (v != v) map[k] = 3;
    else if (v == 0.0) map[k] = 0;
    else if (v == 1.0) map[k] = 1;
    else if (v == 2.0) map[k] = 2;
    else {
      map[k] = 3;
      generic = true;
    }
  }
  bsg_bed *h = nullptr;
  BSG_TRY(alloc_handle(n, m, device, &h));
  h->kind = BSG_KIND_FBM;
  h->layouts = layouts;
  memcpy(h->code256, code256, 256 * sizeof(double));
  uint8_t *draw = nullptr, *dmap = nullptr;
  size_t nb = (size_t)n * m;
  cudaError_t ce = cudaMalloc(&draw, nb);
  if (ce == cudaSuccess) ce = cudaMalloc(&dmap, 256);
  if (ce == cudaSuccess) ce = cudaMemcpy(draw, bytes, nb, cudaMemcpyHostToDevice);
  if (ce == cudaSuccess) ce = cudaMemcpy(dmap, map, 256, cudaMemcpyHostToDevice);
  int rc = BSG_OK;
  if (ce != cudaSuccess) rc = cuda_fail(ce, "upload FBM");
  if (!rc) {
    k_stage_fbm<<<grid_for((int64_t)m * (h->strideA / 4), 256), 256, 0, h->stream>>>(draw, n, m, dmap, h->A, h->strideA);
    count_launch();
    cudaStreamSynchronize(h->stream);
  }
  // Centi-dosage table (every non-NA code within 1e-9 of a multiple of 1/100 in [0, 2.54], one fp64 value per value byte,
  // not only 0 / 1 / 2 / NA -- CODE_DOSAGE, R/bigSNP-class.R:13): the code bytes are re-encoded into value bytes
  // rint(100 x), NA -> 255, that the integer tensor pipe multiplies as they stand (bsg_pmv8.cu).  The table is then
  // indexed by value byte, so the fp64 kernels of bsg_generic.cu see the same value per element as before.
  uint8_t vbyte[256];
  const bool centi = generic && dosage_value_bytes(code256, vbyte);
  double table[256];
  memcpy(table, code256, sizeof table);
  if (centi && !rc) {
    for (int k = 0; k < 256; k++) table[k] = 0.0;
    table[255] = NAN;
    for (int k = 0; k < 256; k++) table[vbyte[k]] = code256[k];
    ce = cudaMemcpy(dmap, vbyte, 256, cudaMemcpyHostToDevice);
    rc = ce != cudaSuccess ? cuda_fail(ce, "upload value bytes") : dosage_stage(h, draw, dmap);
  }
  if (generic && !rc) {  // keep the code bytes and the table: bsg_generic.cu reads code256[byte] like SubBMCode256Acc does
    h->fbm_generic = 1;
    if (!centi) {
      h->raw = draw;
      h->raw_stride = n;
      draw = nullptr;
    }
    double both[512];
    for (int k = 0; k < 256; k++) {
      both[k] = table[k];
      both[256 + k] = (table[k] != table[k]) ? 3.0 : table[k];  // code[is_na(code)] = 3 (src/corr.cpp:115)
    }
    ce = cudaMalloc((void **)&h->d_code, sizeof both);
    if (ce == cudaSuccess) ce = cudaMemcpy(h->d_code, both, sizeof both, cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "upload code256");
  }
  if (draw) cudaFree(draw);
  if (dmap) cudaFree(dmap);
  if (!rc) rc = stage_finish(h);
  if (rc) {
    bsg_close(h);
    return rc;
  }
  *out = h;
  return BSG_OK;
}

void bsg_close(bsg_bed *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->cv) {
    bsg_view_destroy(h->cv);
    h->cv = nullptr;
  }
  void *ptrs[] = {h->A, h->B, h->cntA, h->cntB, h->naA, h->naB, h->raw, h->d_code, h->ellCnt[0], h->ellCnt[1], h->ellEnt[0],
                  h->ellEnt[1], h->ellOff[0], h->ellOff[1], h->ellOut[0], h->ellOut[1]};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  DevBuf *bufs[] = {&h->w_idx_row, &h->w_idx_col, &h->w_center, &h->w_scale, &h->w_x, &h->w_out, &h->w_tmp0,
                    &h->w_tmp1, &h->w_tmp2, &h->w_tmp3, &h->w_part, &h->w_dig1, &h->w_dig2, &h->w_misc};
  for (DevBuf *b : bufs) b->release();
  for (DevBuf &b : h->w_proj) b.release();
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (cudaEvent_t &e : h->copy_ev)
    if (e) cudaEventDestroy(e);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

int bsg_nrow(const bsg_bed *h) { return h ? h->n : 0; }
int bsg_ncol(const bsg_bed *h) { return h ? h->m : 0; }
int bsg_layouts(const bsg_bed *h) { return h ? h->layouts : 0; }
int bsg_has_na(const bsg_bed *h) { return h ? h->has_na : 0; }
int64_t bsg_packed_bytes(const bsg_bed *h) { return h ? h->n_byte * (int64_t)h->m : 0; }

int bsg_export_packed(const bsg_bed *h, uint8_t *out) {
  if (!h || !out) return fail(BSG_ERR_ARG, "null argument");
  BSG_PACKED_ONLY(h, "The 2-bit export");
  BSG_TRY(bind_device(h));
  uint8_t *d = nullptr;
  size_t bytes = (size_t)h->n_byte * h->m;
  BSG_CUDA(cudaMalloc(&d, bytes));
  k_export_bed<<<grid_for((int64_t)bytes, 256), 256, 0, h->stream>>>(h->A, h->strideA, h->n_byte, h->n, h->m, d);
  count_launch();
  cudaError_t e = cudaMemcpyAsync(out, d, bytes, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(d);
  if (e != cudaSuccess) return cuda_fail(e, "export");
  return BSG_OK;
}

void bsg_free(void *ptr) { free(ptr); }

}  // extern "C"
