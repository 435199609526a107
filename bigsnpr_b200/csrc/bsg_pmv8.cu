// bsg_pmv8.cu -- X.y and Xt.y over "centi-dosage" FBM.code256 matrices on the integer tensor pipe.
//
// bigsnpr's dosage tables (CODE_DOSAGE, R/bigSNP-class.R:13: what snp_readBGEN and snp_fastImputeSimple(G, "mean2")
// return) code values that are all multiples of 1/100 in [0, 2].  A code is therefore staged as its VALUE byte
// v = rint(100 x) (255 = missing), which is the u8 A operand of mma.sync.m16n8k32.u8.s8.s32 as it stands, and
//     X~ y  =  sum_j (v_ij / 100 - c_j) / s_j y_j  =  sum_j (v_ij - 100 c_j) / (100 s_j) y_j
// is the algebra the 2-bit kernels already run (bsg_pmv.cu) with center' = 100 c, scale' = 100 s and no missing-value
// plane: same 61-bit quantisation of the vector, same digit blocks, exact integer partials, same fp64 finish kernels.
//   * Xt.y: k_pmv8 below.  Lines = SNP columns, contraction along the samples of a line, one producer warp filling the
//     digit ring (k_prep2 / k_digits layout, unchanged) and consumer lanes streaming 32-byte sectors of their lines.
//   * X.y: k_pmvT<.., BYTES = true> (bsg_pmv.cu), the SNP-major transposing kernel with one IMMA per transposed word.
// Roofline: one pass reads n x m bytes (4x the 2-bit matrix); the IMMA count per byte is a quarter of the 2-bit loops'.
//
// Missing values follow fp64 arithmetic on code256[byte] (bigstatsr's products over an FBM.code256 propagate NA_real_),
// not bedAccScaled's "NA -> 0": an output entry whose row / column meets a selected missing value is NaN.  The integer
// kernels multiply the byte 255 like any other value; the host-vector forms then overwrite the affected entries
// (dosage_mark_na, runs only when a selected column has a missing value); the device-vector forms, which cannot look
// at their result, return an all-NaN vector (include/bsgpu.h).
//
// Contents: k_pmv8 and its launcher; staging of the value bytes; the missing-value marks; the PCA projection of a
// dosage matrix (prod_and_rowSumsSq2); bsg_code256_kind.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "bsg_internal.cuh"
#include "bsg_pmv_shared.cuh"

namespace bsg {
namespace pmv8 {
using namespace pmv;

constexpr int CW = 8;                 // consumer warps per CTA, 16 lines each
constexpr int GROUP = CW * 16;        // lines per work item
constexpr int R = 4;                  // register ring: half-chunks (256 bytes of a line) in flight per warp
constexpr int CHUNK = 512;            // bytes of a line per digit block (= pmv::CODES elements)
constexpr int SMEM8 = STAGES * DIG + 128;
constexpr int MAX_CHUNKS8 = 128;      // 65,536 samples per item: 254 x 128 x 2^16 < 2^31 (int32 accumulators)

__device__ __forceinline__ void ldg256(uint32_t (&w)[16], int o, const uint8_t *p) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[o]), "=r"(w[o + 1]), "=r"(w[o + 2]), "=r"(w[o + 3]), "=r"(w[o + 4]), "=r"(w[o + 5]), "=r"(w[o + 6]),
                 "=r"(w[o + 7])
               : "l"(p));
}

// 4 x 4 byte transpose: t[c] byte r = x[r] byte c
__device__ __forceinline__ void tr4(uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t (&t)[4]) {
  const uint32_t a = prmt(x0, x1, 0x5140), b = prmt(x2, x3, 0x5140);
  const uint32_t c = prmt(x0, x1, 0x7362), d = prmt(x2, x3, 0x7362);
  t[0] = prmt(a, b, 0x5410);
  t[1] = prmt(a, b, 0x7632);
  t[2] = prmt(c, d, 0x5410);
  t[3] = prmt(c, d, 0x7632);
}

// Xt.y: lines = SNP columns (value bytes along the samples).  The digit block of a 512-byte chunk has k_pmv's layout: the
// 16-byte unit (w, slice g, lane q) holds the digits of elements u + 4 r + c at byte 4 c + r, u = 64 q + 16 w (w < 4) or
// 256 + 64 q + 16 (w - 4).  Lane (g, q) of a warp owns lines g and g + 8 of its 16 and bytes [64 q, 64 q + 64) of each
// half-chunk (one 32-byte sector per load); the 4 words of unit w transposed are the A registers c = 0..3 (elements
// u + 4 r + c), which pair with the digit registers d.x .. d.w as they are.
__global__ void __launch_bounds__((CW + 1) * 32, 1) k_pmv8(const Args a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_base + STAGES * DIG;  // full[s] at +8s, empty[s] at +8(STAGES+s)
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(bar_base + 8 * s, 1);
      mbar_init(bar_base + 8 * (STAGES + s), CW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int ngroups = a.nlines_pad / GROUP;
  const int nitems = ngroups * a.ksplit;
  int stage = 0;
  uint32_t phase = 0;

  if (warp == CW) {
    // producer: one bulk copy of the 4 KB digit block per chunk
    if (lane == 0) {
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int ks = item % a.ksplit;
        const int c0 = ks * a.chunks_per_split, c1 = min(a.nchunks, c0 + a.chunks_per_split);
        for (int c = c0; c < c1; c++) {
          const uint32_t full = bar_base + 8 * stage, empty = bar_base + 8 * (STAGES + stage);
          mbar_wait(empty, phase ^ 1);
          mbar_expect_tx(full, DIG);
          bulk_g2s(smem_base + stage * DIG, a.dig1 + (int64_t)c * DIG, DIG, full);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
    return;
  }

  const int g = lane >> 2, q = lane & 3;
  for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
    const int group = item / a.ksplit, ks = item - group * a.ksplit;
    const int c0 = ks * a.chunks_per_split, c1 = min(a.nchunks, c0 + a.chunks_per_split);
    const int la = min(group * GROUP + warp * 16 + g, a.nlines - 1), lb = min(group * GROUP + warp * 16 + g + 8, a.nlines - 1);
    const uint8_t *pa = a.P + (int64_t)(a.lines ? a.lines[la] : la) * a.stride + 64 * q;
    const uint8_t *pb = a.P + (int64_t)(a.lines ? a.lines[lb] : lb) * a.stride + 64 * q;
    int acc[2][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
    // ring[k]: half-chunk t0 + k (+ j R) of lines g ([0..15]) and g + 8 ([16..31]); t even = first half of a chunk
    uint32_t ring[R][2][16];
    const int t0 = 2 * c0, t1 = 2 * c1;
#pragma unroll
    for (int k = 0; k < R; k++) {
      if (t0 + k < t1) {
        const int64_t off = (int64_t)((t0 + k) >> 1) * CHUNK + (k & 1) * 256;
        ldg256(ring[k][0], 0, pa + off);
        ldg256(ring[k][0], 8, pa + off + 32);
        ldg256(ring[k][1], 0, pb + off);
        ldg256(ring[k][1], 8, pb + off + 32);
      }
    }
    for (int t = t0; t < t1; t += R) {
#pragma unroll
      for (int par = 0; par < R; par++) {
        if (par > 0 && t + par >= t1) break;  // t1 - t0 is even: the loop never stops inside a chunk
        const int h = par & 1;
        if (h == 0) mbar_wait(bar_base + 8 * stage, phase);
        const uint32_t dbase = smem_base + stage * DIG + (g * 4 + q) * 16 + h * 2048;
#pragma unroll
        for (int w = 0; w < 4; w++) {
          const uint4 d = lds128(dbase + w * 512);
          uint32_t A[4], B[4];
          tr4(ring[par][0][4 * w], ring[par][0][4 * w + 1], ring[par][0][4 * w + 2], ring[par][0][4 * w + 3], A);
          tr4(ring[par][1][4 * w], ring[par][1][4 * w + 1], ring[par][1][4 * w + 2], ring[par][1][4 * w + 3], B);
          mma_u8s8(acc[0], A[0], B[0], A[1], B[1], d.x, d.y);
          mma_u8s8(acc[1], A[2], B[2], A[3], B[3], d.z, d.w);
        }
        if (t + par + R < t1) {
          const int64_t off = (int64_t)((t + par + R) >> 1) * CHUNK + h * 256;
          ldg256(ring[par][0], 0, pa + off);
          ldg256(ring[par][0], 8, pa + off + 32);
          ldg256(ring[par][1], 0, pb + off);
          ldg256(ring[par][1], 8, pb + off + 32);
        }
        if (h == 1) {
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_base + 8 * (STAGES + stage));
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
    // D rows = lines g / g + 8, columns = digit slices 2q, 2q + 1; k-splits of a line add up exactly in integers
#pragma unroll
    for (int hrow = 0; hrow < 2; hrow++) {
      const int row = group * GROUP + warp * 16 + g + 8 * hrow;
      unsigned long long *dst = reinterpret_cast<unsigned long long *>(a.part) + (int64_t)row * 16 + 2 * q;
      const long long vx = (long long)acc[0][2 * hrow] + acc[1][2 * hrow];
      const long long vy = (long long)acc[0][2 * hrow + 1] + acc[1][2 * hrow + 1];
      if (vx) atomicAdd(dst, (unsigned long long)vx);
      if (vy) atomicAdd(dst + 1, (unsigned long long)vy);
    }
  }
}

// code bytes (n x m, column-major) -> value bytes on lines of `stride` bytes (zero padding) + missing values per line
__global__ void k_value_bytes(const uint8_t *__restrict__ codes, int n, int m, const uint8_t *__restrict__ vbyte,
                              uint8_t *__restrict__ raw, int64_t stride, int *__restrict__ na_cnt) {
  const int64_t words = stride / 4, total = (int64_t)m * words;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = t / words, w = t - j * words;
    uint32_t out = 0;
    int na = 0;
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int64_t i = 4 * w + r;
      const uint32_t v = i < n ? vbyte[codes[j * n + i]] : 0u;
      na += v == 255u;
      out |= v << (8 * r);
    }
    reinterpret_cast<uint32_t *>(raw + j * stride)[w] = out;
    if (na) atomicAdd(na_cnt + j, na);
  }
}

// one warp per selected column holding a missing value: cprod -> out[t] = NaN when a selected row of column t is
// missing; prod -> out[i] = NaN for every selected row i missing in column t
__global__ void k_mark_na(const uint8_t *__restrict__ raw, int64_t stride, const int *__restrict__ col,
                          const int *__restrict__ pos, int npos, const int *__restrict__ row, int nr, int cprod,
                          double *__restrict__ out) {
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nw = (gridDim.x * blockDim.x) >> 5;
  for (int p = wid; p < npos; p += nw) {
    const int t = pos[p];
    const uint8_t *line = raw + (int64_t)(col ? col[t] : t) * stride;
    bool hit = false;
    for (int i = lane; i < nr; i += 32) {
      if (line[row ? row[i] : i] == 255) {
        hit = true;
        if (!cprod) out[i] = nan("");
      }
    }
    if (cprod && __any_sync(0xffffffffu, hit) && lane == 0) out[t] = nan("");
  }
}

__global__ void k_times100(double *__restrict__ c, double *__restrict__ s, int len) {
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < len; k += gridDim.x * blockDim.x) {
    c[k] *= 100.0;
    s[k] *= 100.0;
  }
}

}  // namespace pmv8

bool dosage_value_bytes(const double *code256, uint8_t vbyte[256]) {
  double val[255];
  bool seen[255] = {false};
  bool other = false;  // a code that is not 0 / 1 / 2 / NA: hard-call tables keep the 2-bit path
  for (int k = 0; k < 256; k++) {
    const double x = code256[k];
    if (x != x) {
      vbyte[k] = 255;
      continue;
    }
    if (x != 0.0 && x != 1.0 && x != 2.0) other = true;
    const double r = rint(100.0 * x);
    if (!(fabs(100.0 * x - r) <= 1e-9) || r < 0 || r > 254) return false;
    const int v = (int)r;
    if (seen[v] && memcmp(&val[v], &x, sizeof x) != 0) return false;  // one value byte, one fp64 value
    seen[v] = true;
    val[v] = x;
    vbyte[k] = (uint8_t)v;
  }
  return other;
}

int dosage_stage(bsg_bed *h, const uint8_t *d_codes, const uint8_t *d_vbyte) {
  const int n = h->n, m = h->m;
  h->raw_stride = round_up(n, pmv8::CHUNK);
  BSG_CUDA(cudaMalloc(&h->raw, (size_t)h->raw_stride * m));
  int *d_cnt = nullptr;
  BSG_CUDA(cudaMalloc(&d_cnt, (size_t)m * sizeof(int)));
  cudaError_t e = cudaMemsetAsync(d_cnt, 0, (size_t)m * sizeof(int), h->stream);
  if (e == cudaSuccess) {
    const int64_t work = (int64_t)m * (h->raw_stride / 4);
    const int grid = (int)std::min<int64_t>((work + 255) / 256, 148 * 32);
    pmv8::k_value_bytes<<<grid, 256, 0, h->stream>>>(d_codes, n, m, d_vbyte, h->raw, h->raw_stride, d_cnt);
    count_launch();
    h->na_line.resize(m);
    e = cudaMemcpyAsync(h->na_line.data(), d_cnt, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, h->stream);
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(d_cnt);
  if (e != cudaSuccess) return cuda_fail(e, "value-byte staging");
  h->dosage = 1;
  return BSG_OK;
}

int dosage_view_scaling(bsg_view *v, cudaStream_t s) {
  if (v->nc == 0) return BSG_OK;
  pmv8::k_times100<<<std::min(1184, (v->nc + 255) / 256), 256, 0, s>>>(v->d_center, v->d_scale, v->nc);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

int run_pmv8(bsg_view *v, const uint8_t *dig, pmv::Args *out, cudaStream_t s) {
  using namespace pmv8;
  bsg_bed *h = v->h;
  Args a{};
  a.P = h->raw;
  a.stride = h->raw_stride;
  a.lines = v->d_col;
  a.nlines = v->nc;
  a.nlines_pad = (int)round_up(v->nc, GROUP);
  a.nchunks = (int)(h->raw_stride / CHUNK);
  const int ngroups = a.nlines_pad / GROUP;
  int ks = (24 * 148 + ngroups - 1) / ngroups;
  ks = std::min(ks, std::max(1, a.nchunks / 8));
  ks = std::max(ks, (a.nchunks + MAX_CHUNKS8 - 1) / MAX_CHUNKS8);
  ks = std::max(ks, 1);
  a.chunks_per_split = (a.nchunks + ks - 1) / ks;
  a.ksplit = (a.nchunks + a.chunks_per_split - 1) / a.chunks_per_split;
  a.dig1 = dig;
  BSG_TRY(v->s_part.ensure((size_t)a.nlines_pad * 16 * sizeof(long long)));
  a.part = v->s_part.as<long long>();
  BSG_CUDA(cudaMemsetAsync(a.part, 0, (size_t)a.nlines_pad * 16 * sizeof(long long), s));
  *out = a;
  if (v->nc == 0) return BSG_OK;
  static unsigned attr_done = 0;  // one bit per device
  if (!(attr_done >> (h->device & 31) & 1u)) {
    BSG_CUDA(cudaFuncSetAttribute(k_pmv8, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM8));
    attr_done |= 1u << (h->device & 31);
  }
  int nsm = 148;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, h->device);
  k_pmv8<<<std::min(ngroups * a.ksplit, nsm), (CW + 1) * 32, SMEM8, s>>>(a);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

int dosage_mark_na(bsg_view *v, bool cprod, double *d_out, cudaStream_t s) {
  if (!v->any_na || v->nr == 0) return BSG_OK;
  const int grid = std::min(148 * 8, (v->n_na_pos * 32 + 255) / 256);
  pmv8::k_mark_na<<<grid, 256, 0, s>>>(v->h->raw, v->h->raw_stride, v->d_col, v->d_na_pos, v->n_na_pos, v->d_row, v->nr,
                                       cprod ? 1 : 0, d_out);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

}  // namespace bsg

// ---- PCA projection (prod_and_rowSumsSq2, src/project-utils.cpp:12-43) -------------------------------------------------
namespace bsg {
namespace pmv8 {
constexpr int RSS_COLS = 2048;  // columns per partial sum of the row sums of squares

// part[split][i] = sum over the split's columns j of ((v - 100 c_j) / (100 s_j))^2, NaN for a missing value; one thread
// per selected row, columns in order (deterministic), lanes read consecutive rows of a line
__global__ void k_rowsumsq8(const uint8_t *__restrict__ raw, int64_t stride, const int *__restrict__ row, int nr,
                            const int *__restrict__ col, int nc, const double *__restrict__ c100,
                            const double *__restrict__ s100, double *__restrict__ part) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nr) return;
  const int r = row ? row[i] : i;
  const int j0 = blockIdx.y * RSS_COLS, j1 = min(nc, j0 + RSS_COLS);
  double acc = 0;
  for (int j = j0; j < j1; j++) {
    const uint8_t v = raw[(int64_t)(col ? col[j] : j) * stride + r];
    const double x = v == 255 ? nan("") : (v - c100[j]) / s100[j];
    acc += x * x;
  }
  part[(int64_t)blockIdx.y * nr + i] = acc;
}

__global__ void k_sum_parts(const double *__restrict__ part, int nsplit, int nr, double *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nr) return;
  double acc = 0;
  for (int s = 0; s < nsplit; s++) acc += part[(int64_t)s * nr + i];
  out[i] = acc;
}
}  // namespace pmv8

int dosage_prod_and_rowsumssq(bsg_view *v, const double *V, int K, double *XV, double *rowSumsSq) {
  bsg_bed *h = v->h;
  cudaStream_t s = h->stream;
  const int nr = v->nr, nc = v->nc;
  if (nr == 0) return BSG_OK;
  const int nsplit = std::max(1, (nc + pmv8::RSS_COLS - 1) / pmv8::RSS_COLS);
  BSG_TRY(h->w_proj[0].ensure(std::max<size_t>(1, (size_t)nc * K) * sizeof(double)));
  BSG_TRY(h->w_proj[1].ensure(std::max<size_t>(1, (size_t)nr * K) * sizeof(double)));
  BSG_TRY(h->w_proj[2].ensure(((size_t)nsplit + 1) * nr * sizeof(double)));
  double *dV = h->w_proj[0].as<double>(), *dXV = h->w_proj[1].as<double>(), *dpart = h->w_proj[2].as<double>();
  double *drss = dpart + (size_t)nsplit * nr;
  if ((size_t)nc * K) BSG_CUDA(cudaMemcpyAsync(dV, V, (size_t)nc * K * sizeof(double), cudaMemcpyHostToDevice, s));
  for (int k = 0; k < K; k++) {  // X~ V column by column, missing values marked as in the host-vector products
    BSG_TRY(view_prodvec_comm(v, dV + (size_t)k * nc, dXV + (size_t)k * nr, s, nullptr));
    BSG_TRY(dosage_mark_na(v, false, dXV + (size_t)k * nr, s));
  }
  if (nc > 0) {
    pmv8::k_rowsumsq8<<<dim3((nr + 255) / 256, nsplit), 256, 0, s>>>(h->raw, h->raw_stride, v->d_row, nr, v->d_col, nc,
                                                                     v->d_center, v->d_scale, dpart);
    pmv8::k_sum_parts<<<(nr + 255) / 256, 256, 0, s>>>(dpart, nsplit, nr, drss);
    count_launch(2);
  } else {
    BSG_CUDA(cudaMemsetAsync(drss, 0, (size_t)nr * sizeof(double), s));
  }
  BSG_CUDA(cudaGetLastError());
  if (K > 0) BSG_CUDA(cudaMemcpyAsync(XV, dXV, (size_t)nr * K * sizeof(double), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaMemcpyAsync(rowSumsSq, drss, (size_t)nr * sizeof(double), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaStreamSynchronize(s));
  return BSG_OK;
}

}  // namespace bsg

extern "C" int bsg_code256_kind(const double *code256) {
  if (!code256) return -bsg::fail(BSG_ERR_ARG, "null argument");
  bool hard = true;
  for (int k = 0; k < 256; k++) {
    const double x = code256[k];
    if (x == x && x != 0.0 && x != 1.0 && x != 2.0) hard = false;
  }
  uint8_t vbyte[256];
  return hard ? 0 : (bsg::dosage_value_bytes(code256, vbyte) ? 1 : 2);
}
