// bsg_la.cu -- the two dense consumers of the packed matvecs.
//
//   bsg_randomsvd   bed_randomSVD (R/autoSVD.R:205-219) -> bigstatsr::big_randomSVD -> RSpectra::svds
//                   [unvendored].  RSpectra runs an implicitly restarted Lanczos iteration on the smaller Gram
//                   operator (A A^T or A^T A), calling back into R twice per step.  Here the whole iteration
//                   stays on the device: thick-restart Lanczos (the explicit form of implicit restarting with
//                   exact shifts) with full re-orthogonalisation, ncv = max(2k+1, 20), the same stopping
//                   rule as ARPACK/Spectra (|Ritz residual| <= tol * max(eps^(2/3), |theta|)), operator =
//                   bsg_view_{c,}prodvec_dev.  Only ncv+1 doubles cross PCIe per step.
//   bsg_tcrossprod  bed_tcrossprodSelf (R/bed-tcrossprodSelf.R:21-52): K = sum_blocks X~_b X~_b^T as ONE weighted
//                   integer Gram product: the per-SNP weights 1/s^2, c/s^2, c^2/s^2 are quantised to base-64 digit
//                   slices folded into the B bytes, the 128 x 128 tiles run on tcgen05 / TMEM (bsg_gram5.cu,
//                   k_wgram5) or on the register-IMMA kernel below (k_wgram), the centering terms come from two
//                   matvecs.  The sample-major copy is built on demand.  Fallback (degenerate scaling, no room for
//                   that copy): device decode of column blocks + cuBLAS DSYRK.
//                   bsg_tcrossprod_dev leaves K in the caller's device buffer (sharded GRM: one all-reduce).
#include <cublas_v2.h>
#include <math.h>
#include <cmath>
#include <string.h>

#include <algorithm>
#include <vector>

#include "bsg_gram.cuh"
#include "bsg_internal.cuh"

namespace bsg {

// ---- small deterministic vector kernels --------------------------------------------------------
// h[j] = <V[:, j], w>, one block per column, fixed-shape tree
__global__ void k_dots(const double *__restrict__ V, int64_t ld, int ncols, const double *__restrict__ w, int N,
                       double *__restrict__ h) {
  __shared__ double sh[32];
  const int j = blockIdx.x;
  if (j >= ncols) return;
  const double *v = V + (int64_t)j * ld;
  double acc = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) acc += v[i] * w[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) t += sh[k];
    h[j] = t;
  }
}

// two-stage deterministic version for long vectors: part[j * nsplit + b] = partial dot of block b
__global__ void k_dots_part(const double *__restrict__ V, int64_t ld, int ncols, const double *__restrict__ w, int N,
                            int nsplit, double *__restrict__ part) {
  __shared__ double sh[32];
  const int j = blockIdx.y, b = blockIdx.x;
  const double *v = V + (int64_t)j * ld;
  const int chunk = (N + nsplit - 1) / nsplit;
  const int i0 = b * chunk, i1 = min(N, i0 + chunk);
  double acc = 0;
  for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) acc += v[i] * w[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) t += sh[k];
    part[(int64_t)j * nsplit + b] = t;
  }
}
__global__ void k_dots_final(const double *__restrict__ part, int ncols, int nsplit, double *__restrict__ h) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= ncols) return;
  double t = 0;
  for (int b = 0; b < nsplit; b++) t += part[(int64_t)j * nsplit + b];
  h[j] = t;
}

// w[i] -= sum_j V[i, j] * h[j]
__global__ void k_axpys(const double *__restrict__ V, int64_t ld, int ncols, const double *__restrict__ h, int N,
                        double *__restrict__ w) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  double acc = 0;
  for (int j = 0; j < ncols; j++) acc += V[(int64_t)j * ld + i] * h[j];
  w[i] -= acc;
}

// out[:, c] = sum_j V[:, j] * S[j, c]   (S is ncv x kk column-major on device)
__global__ void k_combine(const double *__restrict__ V, int64_t ld, int ncv, const double *__restrict__ S, int lds,
                          int kk, int N, double *__restrict__ out, int64_t ldo) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int c = blockIdx.y;
  if (i >= N || c >= kk) return;
  double acc = 0;
  for (int j = 0; j < ncv; j++) acc += V[(int64_t)j * ld + i] * S[(int64_t)c * lds + j];
  out[(int64_t)c * ldo + i] = acc;
}

__global__ void k_scale_copy(const double *__restrict__ src, double alpha, int N, double *__restrict__ dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) dst[i] = src[i] * alpha;
}

__global__ void k_init_vec(int N, uint64_t seed, double *__restrict__ v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  uint64_t x = seed + 0x9E3779B97F4A7C15ull * (uint64_t)(i + 1);
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  x ^= x >> 31;
  v[i] = ((double)(x >> 11) * (1.0 / 9007199254740992.0)) - 0.5;
}

// cyclic Jacobi eigen-decomposition of a small symmetric matrix (column-major n x n); eigenvalues in w,
// eigenvectors in the columns of Z; sorted descending.
static void jacobi_eigh(std::vector<double> A, int n, std::vector<double> &w, std::vector<double> &Z) {
  Z.assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; i++) Z[(size_t)i * n + i] = 1.0;
  auto a = [&](int i, int j) -> double & { return A[(size_t)j * n + i]; };
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0, diag = 0;
    for (int j = 0; j < n; j++)
      for (int i = 0; i < n; i++) (i == j ? diag : off) += a(i, j) * a(i, j);
    if (off <= 1e-30 * (diag + 1e-300)) break;
    for (int p = 0; p < n - 1; p++)
      for (int q = p + 1; q < n; q++) {
        double apq = a(p, q);
        if (fabs(apq) < 1e-300) continue;
        double theta = (a(q, q) - a(p, p)) / (2.0 * apq);
        double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < n; k++) {
          double akp = a(k, p), akq = a(k, q);
          a(k, p) = c * akp - s * akq;
          a(k, q) = s * akp + c * akq;
        }
        for (int k = 0; k < n; k++) {
          double apk = a(p, k), aqk = a(q, k);
          a(p, k) = c * apk - s * aqk;
          a(q, k) = s * apk + c * aqk;
        }
        for (int k = 0; k < n; k++) {
          double zkp = Z[(size_t)p * n + k], zkq = Z[(size_t)q * n + k];
          Z[(size_t)p * n + k] = c * zkp - s * zkq;
          Z[(size_t)q * n + k] = s * zkp + c * zkq;
        }
      }
  }
  std::vector<int> ord(n);
  for (int i = 0; i < n; i++) ord[i] = i;
  std::sort(ord.begin(), ord.end(), [&](int x, int y) { return a(x, x) > a(y, y); });
  w.resize(n);
  std::vector<double> Z2((size_t)n * n);
  for (int c = 0; c < n; c++) {
    w[c] = a(ord[c], ord[c]);
    memcpy(&Z2[(size_t)c * n], &Z[(size_t)ord[c] * n], n * sizeof(double));
  }
  Z.swap(Z2);
}


// ---------------------------------------------------------------------------------------------------
// Weighted integer Gram on the tensor pipe:  K += scale * sum_k fA(code(i,k)) * fB(code(j,k)) * d_k
// with d_k one base-64 digit (0..63) of a non-negative per-k weight.  The digit is folded into the B bytes
// ((x & 1) ? d : 0) | ((x & 2) ? 2d : 0), so the products stay exact in int32; slices are combined in fp64.
// ---------------------------------------------------------------------------------------------------
namespace wgram {
using namespace gram;

enum { WP_AA = 0, WP_AN = 1, WP_NA = 2, WP_NN = 3 };

struct WTile {
  int i0, j0;   // first A line (TM block), first B line (TN block)
  int mode;     // 0: lines without missing values -> product aa only; 1: aa, an, na, nn
};

struct WArgs {
  const uint8_t *P;
  int64_t stride;
  int nlines, nchunks, nslices;
  const uint8_t *dig[3];   // weight digits of W1, W2' = -W2, W3: [nslices][nchunks * 256] in fragment order
  double scale[3][10];     // 64^t * 2^-e per weight and slice
  const WTile *tiles;
  double *K;               // n x n column-major, pre-zeroed; tile (i0, j0) writes K[i, j] for i >= j only
  int64_t ldk;
};

struct WFrag {
  uint4 a[4], b[4];
};

// NA-indicator plane: bit 2p set iff code p is missing
__device__ __forceinline__ uint32_t plane_n(uint32_t w) { return w & (w >> 1) & 0x55555555u; }

template <int PROD, bool RAW>
__device__ __forceinline__ void wfrag_mma(const WFrag &f, const uint8_t *dp, int (&acc)[2][4][4]) {
  const uint32_t *aw[4] = {&f.a[0].x, &f.a[1].x, &f.a[2].x, &f.a[3].x};
  const uint32_t *bw[4] = {&f.b[0].x, &f.b[1].x, &f.b[2].x, &f.b[3].x};
  constexpr bool A_IS_N = (PROD == WP_NA || PROD == WP_NN), B_IS_N = (PROD == WP_AN || PROD == WP_NN);
#pragma unroll
  for (int w = 0; w < 4; w++) {
    const uint4 dq = ldg128(dp + w * 16);  // digits of this word (L1-resident, shared by the 8 lanes of equal q)
    const uint32_t dcls[4] = {dq.x, dq.y, dq.z, dq.w};  // digits of class c: byte r <-> code 4r + c
    uint32_t wa[4], wb[4];
#pragma unroll
    for (int l = 0; l < 4; l++) {
      wa[l] = A_IS_N ? plane_n(aw[l][w]) : (RAW ? aw[l][w] : plane_word<PL_A>(aw[l][w]));
      wb[l] = B_IS_N ? plane_n(bw[l][w]) : (RAW ? bw[l][w] : plane_word<PL_A>(bw[l][w]));
    }
#pragma unroll
    for (int cp = 0; cp < 2; cp++) {
      const int s0 = 4 * cp, s1 = 4 * cp + 2;
      const uint32_t d0 = dcls[2 * cp], d1 = dcls[2 * cp + 1];
      uint32_t b0[4], b1[4];
#pragma unroll
      for (int nt = 0; nt < 4; nt++) {
        const uint32_t x0 = wb[nt] >> s0, x1 = wb[nt] >> s1;
        const uint32_t m0 = (x0 & 0x01010101u) * 0xFFu, m1 = (x1 & 0x01010101u) * 0xFFu;
        if (B_IS_N) {
          b0[nt] = m0 & d0;
          b1[nt] = m1 & d1;
        } else {
          const uint32_t h0 = ((x0 >> 1) & 0x01010101u) * 0xFFu, h1 = ((x1 >> 1) & 0x01010101u) * 0xFFu;
          b0[nt] = (m0 & d0) | (h0 & (d0 << 1));
          b1[nt] = (m1 & d1) | (h1 & (d1 << 1));
        }
      }
#pragma unroll
      for (int mt = 0; mt < 2; mt++) {
        const uint32_t a0 = (wa[2 * mt] >> s0) & 0x03030303u, a1 = (wa[2 * mt + 1] >> s0) & 0x03030303u;
        const uint32_t a2 = (wa[2 * mt] >> s1) & 0x03030303u, a3 = (wa[2 * mt + 1] >> s1) & 0x03030303u;
#pragma unroll
        for (int nt = 0; nt < 4; nt++) mma_u8u8(acc[mt][nt], a0, a1, a2, a3, b0[nt], b1[nt]);
      }
    }
  }
}

template <int PROD, bool RAW>
__device__ __forceinline__ void wgram_product(const uint8_t *const (&pa)[4], const uint8_t *const (&pb)[4],
                                              const uint8_t *dig, int nchunks, int q, int (&acc)[2][4][4]) {
#pragma unroll
  for (int mt = 0; mt < 2; mt++)
#pragma unroll
    for (int nt = 0; nt < 4; nt++)
#pragma unroll
      for (int k = 0; k < 4; k++) acc[mt][nt][k] = 0;
  WFrag f0, f1;
  auto load = [&](WFrag &f, int c) {
    const int64_t off = (int64_t)c * CHUNK;
#pragma unroll
    for (int l = 0; l < 4; l++) f.a[l] = ldg128(pa[l] + off);
#pragma unroll
    for (int l = 0; l < 4; l++) f.b[l] = ldg128(pb[l] + off);
  };
  const uint8_t *dq = dig + (int64_t)q * 64;  // [chunk][q][w][16]
  load(f0, 0);
  for (int c = 0; c < nchunks; c += 2) {
    if (c + 1 < nchunks) load(f1, c + 1);
    wfrag_mma<PROD, RAW>(f0, dq + (int64_t)c * 256, acc);
    if (c + 2 < nchunks) load(f0, c + 2);
    if (c + 1 < nchunks) wfrag_mma<PROD, RAW>(f1, dq + (int64_t)(c + 1) * 256, acc);
  }
}

__global__ void __launch_bounds__(THREADS, 1) k_wgram(const WArgs a) {
  const WTile t = a.tiles[blockIdx.x];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int wm = warp >> 1, wn = warp & 1;
  // this warp's 32 x 32 block lies strictly above the diagonal -> nothing to do (K is filled for i >= j)
  if (t.i0 + wm * 32 + 31 < t.j0 + wn * 32) return;
  const uint8_t *pa[4], *pb[4];
#pragma unroll
  for (int l = 0; l < 4; l++) {
    int la = t.i0 + wm * 32 + (l >> 1) * 16 + g + 8 * (l & 1);
    int lb = t.j0 + wn * 32 + l * 8 + g;
    la = min(la, a.nlines - 1);
    lb = min(lb, a.nlines - 1);
    pa[l] = a.P + (int64_t)la * a.stride + 16 * q;
    pb[l] = a.P + (int64_t)lb * a.stride + 16 * q;
  }
  int acc[2][4][4];
  const int64_t dstride = (int64_t)a.nchunks * 256;
  // K is pre-zeroed and every (i, j) of the tile is owned by one thread: accumulate in place, slice by slice
  auto fold = [&](double sc) {
#pragma unroll
    for (int mt = 0; mt < 2; mt++)
#pragma unroll
      for (int nt = 0; nt < 4; nt++)
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const int i = t.i0 + wm * 32 + mt * 16 + g + 8 * (k >> 1);
          const int j = t.j0 + wn * 32 + nt * 8 + 2 * q + (k & 1);
          if (i < a.nlines && j < a.nlines && i >= j) a.K[(int64_t)j * a.ldk + i] += sc * (double)acc[mt][nt][k];
        }
  };
  for (int sl = a.nslices - 1; sl >= 0; sl--) {
    if (t.mode == 0) {
      wgram_product<WP_AA, true>(pa, pb, a.dig[0] + sl * dstride, a.nchunks, q, acc);
      fold(a.scale[0][sl]);
    } else {
      wgram_product<WP_AA, false>(pa, pb, a.dig[0] + sl * dstride, a.nchunks, q, acc);
      fold(a.scale[0][sl]);
      wgram_product<WP_AN, false>(pa, pb, a.dig[1] + sl * dstride, a.nchunks, q, acc);
      fold(a.scale[1][sl]);
      wgram_product<WP_NA, false>(pa, pb, a.dig[1] + sl * dstride, a.nchunks, q, acc);
      fold(a.scale[1][sl]);
      wgram_product<WP_NN, false>(pa, pb, a.dig[2] + sl * dstride, a.nchunks, q, acc);
      fold(a.scale[2][sl]);
    }
  }
}

// weight digits in fragment order: byte ((chunk*4 + q)*4 + w)*16 + c*4 + r  <->  k = chunk*256 + (4q+w)*16 + 4r + c
__global__ void k_weight_digits(const double *__restrict__ W, int len, int nchunks, int nslices, int e, int dbits,
                                uint8_t *__restrict__ dig) {
  int64_t total = (int64_t)nchunks * 256;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int byte = (int)(t & 15), unit = (int)((t >> 4) & 15), chunk = (int)(t >> 8);
    const int c = byte >> 2, r = byte & 3, w = unit & 3, q = unit >> 2;
    const int64_t k = (int64_t)chunk * 256 + (4 * q + w) * 16 + 4 * r + c;
    unsigned long long v = 0;
    if (k < len) v = (unsigned long long)__double2ll_rn(scalbn(W[k], e));
    for (int sl = 0; sl < nslices; sl++) {
      dig[(int64_t)sl * total + t] = (uint8_t)(v & ((1ull << dbits) - 1ull));
      v >>= dbits;
    }
  }
}

// lower triangle + vector terms -> full symmetric K:  K_ij += r_i + r_j + cst - q_i - q_j
__global__ void k_grm_finish(double *__restrict__ K, int64_t ld, int n, const double *__restrict__ r,
                             const double *__restrict__ qv, double cst) {
  int64_t total = (int64_t)n * n;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(t / n), i = (int)(t - (int64_t)j * n);
    if (i < j) continue;
    double v = K[(int64_t)j * ld + i] + r[i] + r[j] + cst;
    if (qv) v -= qv[i] + qv[j];
    K[(int64_t)j * ld + i] = v;
    K[(int64_t)i * ld + j] = v;
  }
}

// u = 1/s, t = -c/s:  W1 = u^2, W2' = -u t = c/s^2 (>= 0 for c >= 0), W3 = t^2 ; w2 = u t (signed, for the vector term)
__global__ void k_grm_weights(const double *__restrict__ center, const double *__restrict__ scale, int len,
                              double *__restrict__ W1, double *__restrict__ W2p, double *__restrict__ W3,
                              double *__restrict__ w2, double *__restrict__ stats /* max1,max2,max3,sumW3,bad */) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  double m1 = 0, m2 = 0, m3 = 0, s3 = 0;
  int bad = 0;
  if (k < len) {
    const double u = 1.0 / scale[k], tt = -center[k] / scale[k];
    const double a = u * u, b = -(u * tt), c = tt * tt;
    W1[k] = a; W2p[k] = b; W3[k] = c; w2[k] = u * tt;
    if (!isfinite(a) || !isfinite(b) || !isfinite(c) || b < 0) bad = 1;
    m1 = a; m2 = b; m3 = c; s3 = c;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    m1 = fmax(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    m2 = fmax(m2, __shfl_xor_sync(0xffffffffu, m2, o));
    m3 = fmax(m3, __shfl_xor_sync(0xffffffffu, m3, o));
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(reinterpret_cast<unsigned long long *>(&stats[0]), (unsigned long long)__double_as_longlong(m1));
    atomicMax(reinterpret_cast<unsigned long long *>(&stats[1]), (unsigned long long)__double_as_longlong(m2));
    atomicMax(reinterpret_cast<unsigned long long *>(&stats[2]), (unsigned long long)__double_as_longlong(m3));
    if (bad) atomicMax(reinterpret_cast<unsigned long long *>(&stats[4]), (unsigned long long)__double_as_longlong(1.0));
  }
}

}  // namespace wgram

static thread_local int g_last_nconv = -1;  // converged Ritz values of the last bsg_randomsvd* call on this thread

// ---- device-side bookkeeping of the recurrence: no host round trip between two operator applications ----------------
// column j of the projected matrix T gets the Gram-Schmidt coefficients (two passes: set, then add)
__global__ void k_tcol(const double *__restrict__ hcoef, int cnt, double *__restrict__ tcol, int add) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < cnt) tcol[i] = add ? tcol[i] + hcoef[i] : hcoef[i];
}
// scal[0] = |w| (the next off-diagonal entry, kept as beta of the last step), scal[1] = 1 / |w| (0 if w == 0)
__global__ void k_norm_step(const double *__restrict__ h0, double *__restrict__ T, int ncv, int j, double *__restrict__ scal) {
  const double nrm = sqrt(h0[0]);
  scal[0] = nrm;
  scal[1] = nrm > 0 ? 1.0 / nrm : 0.0;
  if (j >= 0 && j + 1 < ncv) T[(size_t)(j + 1) * ncv + j] = nrm;
}
__global__ void k_scale_copy_p(const double *__restrict__ src, const double *__restrict__ alpha, int N, double *__restrict__ dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) dst[i] = src[i] * alpha[0];
}

struct SvdWork {
  double *V = nullptr, *w = nullptr, *tmp = nullptr, *h = nullptr, *S = nullptr, *Y = nullptr, *part = nullptr, *T = nullptr,
         *scal = nullptr, *other = nullptr;
  void release() {
    void *p[] = {V, w, tmp, h, S, Y, part, T, scal, other};
    for (void *q : p)
      if (q) cudaFree(q);
    V = w = tmp = h = S = Y = part = T = scal = other = nullptr;
  }
};


// Thick-restart Lanczos on the Gram operator of X~ (see the header of this file), written over a LIST of column shards:
// one replica of the recurrence per shard / device, all fed the same bits (the fused X.y + all-reduce sums in rank order), so
// the replicas stay identical and only shard 0's projected matrix is read back -- once per restart, which is the only host
// synchronisation of the iteration.  One shard without communicator = the single-GPU bed_randomSVD.
int lanczos_svd(std::vector<SvdShard> &sh, const int *ind_row, int nr, int ncol_total, int k, double tol, int maxit, double *d,
                double *u, int *niter, int *nops, double *z_dev, bsg_reduce_cb reduce_cb, void *cb_ctx) {
  const int G = (int)sh.size();
  if (G < 1 || !d) return fail(BSG_ERR_ARG, "null argument");
  if (!ind_row) nr = sh[0].h->n;
  const bool sharded = G > 1 || sh[0].comm != nullptr || reduce_cb != nullptr;
  const int mtot = sharded ? ncol_total : sh[0].nc;
  if (k < 1 || k > std::min(nr, mtot)) return fail(BSG_ERR_ARG, "k must be in 1..min(n, m).");
  if (tol <= 0) tol = 1e-4;
  if (maxit <= 0) maxit = 1000;

  struct Rep {  // one replica
    bsg_view *view = nullptr;
    SvdWork W;
    double *wv = nullptr;
    cudaStream_t s = nullptr;
    std::vector<double> cen, sca;
  };
  std::vector<Rep> rep(G);
  struct Cleanup {
    std::vector<Rep> &r;
    std::vector<SvdShard> &sh;
    ~Cleanup() {
      for (size_t g = 0; g < r.size(); g++) {
        cudaSetDevice(sh[g].h->device);
        cudaStreamSynchronize(r[g].s);
        if (r[g].view) bsg_view_destroy(r[g].view);
        r[g].W.release();
      }
    }
  } cleanup{rep, sh};

  // ---- scaling: default bed_scaleBinom (R/binom-scaling.R:133-142), same fp64 formulas on the same integers
  for (int g = 0; g < G; g++) {
    bsg_bed *h = sh[g].h;
    BSG_TRY(bind_device(h));
    rep[g].s = h->stream;
    const int nc = sh[g].nc;
    rep[g].cen.resize(std::max(nc, 1));
    rep[g].sca.resize(std::max(nc, 1));
    if (sh[g].center && sh[g].scale) {
      memcpy(rep[g].cen.data(), sh[g].center, (size_t)nc * sizeof(double));
      memcpy(rep[g].sca.data(), sh[g].scale, (size_t)nc * sizeof(double));
    } else if (h->dosage) {
      return fail(BSG_ERR_ARG, "bed_scaleBinom needs hard calls: pass center and scale for a dosage FBM.code256 "
                               "(snp_scaleBinom, or the mean and sd of each column).");
    } else if (nc > 0) {
      std::vector<double> sumX(nc), denoX(nc);
      std::vector<int> nona(nc);
      int n_bad = 0;
      BSG_TRY(bsg_colstats(h, ind_row, nr, sh[g].ind_col, nc, sumX.data(), denoX.data(), nona.data(), &n_bad));
      for (int j = 0; j < nc; j++) {
        double af = sumX[j] / (2.0 * (double)nona[j]);
        rep[g].cen[j] = 2.0 * af;
        rep[g].sca[j] = sqrt(2.0 * af * (1.0 - af));
      }
    }
    for (int j = 0; j < nc; j++) {
      const int64_t row = sh[g].v_pos ? sh[g].v_pos[j] : j;
      if (sh[g].center_out) sh[g].center_out[row] = rep[g].cen[j];
      if (sh[g].scale_out) sh[g].scale_out[row] = rep[g].sca[j];
    }
    BSG_TRY(bsg_view_create(h, ind_row, nr, sh[g].ind_col, nc, rep[g].cen.data(), rep[g].sca.data(), &rep[g].view));
  }

  // operator side: the smaller Gram matrix; a sharded matrix always iterates on the sample side
  const bool row_side = sharded ? true : (nr <= sh[0].nc);
  const int N = row_side ? nr : sh[0].nc;
  int ncv = std::max(2 * k + 1, 20);
  ncv = std::min(ncv, std::min(nr, mtot));
  if (ncv <= k) ncv = std::min(k + 1, std::min(nr, mtot));
  const bool full_space = ncv <= k;  // degenerate: k == min(n, m)
  const int64_t ld = N;
  const int NSPLIT = 32, TB = 256;
  auto gblocks = [&](int len) { return (len + TB - 1) / TB; };

  for (int g = 0; g < G; g++) {
    BSG_TRY(bind_device(sh[g].h));
    SvdWork &W = rep[g].W;
    const int Mo = row_side ? sh[g].nc : nr;
    BSG_CUDA(cudaMalloc((void **)&W.V, (size_t)ld * (ncv + 1) * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.tmp, (size_t)std::max(Mo, 1) * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.other, (size_t)std::max(Mo, 1) * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.h, (size_t)(ncv + 2) * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.S, (size_t)ncv * ncv * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.Y, (size_t)ld * ncv * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.part, (size_t)(ncv + 2) * NSPLIT * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.T, (size_t)ncv * ncv * sizeof(double)));
    BSG_CUDA(cudaMalloc((void **)&W.scal, 4 * sizeof(double)));
    BSG_CUDA(cudaMemsetAsync(W.T, 0, (size_t)ncv * ncv * sizeof(double), rep[g].s));
    if (reduce_cb && z_dev && g == 0) {
      rep[g].wv = z_dev;  // the caller's buffer: results are reduced across ranks by the callback
    } else {
      BSG_CUDA(cudaMalloc((void **)&W.w, (size_t)N * sizeof(double)));
      rep[g].wv = W.w;
    }
  }

  int ops = 0;
  // every step below is enqueued on all replicas before the host moves on: the fused reductions of the replicas meet on
  // the devices, never on the host
  auto dots = [&](int g, const double *Vp, int cnt, const double *wp) {  // W.h[j] = <V[:, j], w>, deterministic
    SvdWork &W = rep[g].W;
    dim3 grd(NSPLIT, cnt);
    k_dots_part<<<grd, 256, 0, rep[g].s>>>(Vp, ld, cnt, wp, N, NSPLIT, W.part);
    k_dots_final<<<(cnt + 63) / 64, 64, 0, rep[g].s>>>(W.part, cnt, NSPLIT, W.h);
    count_launch(2);
  };
  auto apply = [&](int col) -> int {  // wv = H V[:, col]
    for (int g = 0; g < G; g++) {
      BSG_TRY(bind_device(sh[g].h));
      SvdWork &W = rep[g].W;
      cudaStream_t s = rep[g].s;
      const double *x = W.V + (int64_t)col * ld;
      if (row_side) {
        if (sh[g].nc > 0) BSG_TRY(bsg_view_cprodvec_dev(rep[g].view, x, W.tmp, s));
        BSG_TRY(view_prodvec_comm(rep[g].view, W.tmp, rep[g].wv, s, sh[g].comm));
      } else {
        BSG_TRY(bsg_view_prodvec_dev(rep[g].view, x, W.tmp, s));
        BSG_TRY(bsg_view_cprodvec_dev(rep[g].view, W.tmp, rep[g].wv, s));
      }
      if (reduce_cb) {
        BSG_CUDA(cudaStreamSynchronize(s));
        reduce_cb(cb_ctx);
      }
    }
    ops++;
    return BSG_OK;
  };
  // orthogonalise wv against V[:, 0..cnt) (classical Gram-Schmidt, applied twice); coefficients -> column j of T, norm -> scal
  auto orth = [&](int cnt, int j) -> int {
    for (int g = 0; g < G; g++) {
      BSG_TRY(bind_device(sh[g].h));
      SvdWork &W = rep[g].W;
      cudaStream_t s = rep[g].s;
      for (int pass = 0; pass < 2 && cnt > 0; pass++) {
        dots(g, W.V, cnt, rep[g].wv);
        k_axpys<<<gblocks(N), TB, 0, s>>>(W.V, ld, cnt, W.h, N, rep[g].wv);
        if (j >= 0) k_tcol<<<(cnt + 63) / 64, 64, 0, s>>>(W.h, cnt, W.T + (size_t)j * ncv, pass);
        count_launch(j >= 0 ? 2 : 1);
      }
      dots(g, rep[g].wv, 1, rep[g].wv);
      k_norm_step<<<1, 1, 0, s>>>(W.h, W.T, ncv, j, W.scal);
      count_launch();
    }
    return BSG_OK;
  };
  auto next_vec = [&](int dst_col) -> int {
    for (int g = 0; g < G; g++) {
      BSG_TRY(bind_device(sh[g].h));
      k_scale_copy_p<<<gblocks(N), TB, 0, rep[g].s>>>(rep[g].wv, rep[g].W.scal + 1, N, rep[g].W.V + (int64_t)dst_col * ld);
      count_launch();
    }
    BSG_CUDA(cudaGetLastError());
    return BSG_OK;
  };

  // ---- start vector
  for (int g = 0; g < G; g++) {
    BSG_TRY(bind_device(sh[g].h));
    k_init_vec<<<gblocks(N), TB, 0, rep[g].s>>>(N, 0x5EEDull, rep[g].wv);
    count_launch();
  }
  BSG_TRY(orth(0, -1));
  BSG_TRY(next_vec(0));

  std::vector<double> T((size_t)ncv * ncv, 0.0), Td((size_t)ncv * ncv), theta, Sm;
  int have = 0;      // number of basis vectors whose T column is complete
  int iters = 0, nconv = 0;
  double beta_last = 0;
  for (;;) {
    // ---- extend the Krylov basis to ncv vectors: nothing but kernel launches
    for (int j = have; j < ncv; j++) {
      BSG_TRY(apply(j));
      BSG_TRY(orth(j + 1, j));
      BSG_TRY(next_vec(j + 1));  // next basis vector (also kept as the residual vector V[:, ncv] after the last step)
    }
    // ---- the projected matrix of replica 0 (all replicas hold the same bits): the one synchronisation per restart
    {
      BSG_TRY(bind_device(sh[0].h));
      double sc2[2];
      BSG_CUDA(cudaMemcpyAsync(Td.data(), rep[0].W.T, (size_t)ncv * ncv * sizeof(double), cudaMemcpyDeviceToHost, rep[0].s));
      BSG_CUDA(cudaMemcpyAsync(sc2, rep[0].W.scal, 2 * sizeof(double), cudaMemcpyDeviceToHost, rep[0].s));
      BSG_CUDA(cudaStreamSynchronize(rep[0].s));
      beta_last = sc2[0];
      bool finite = std::isfinite(beta_last);
      for (int j = have; j < ncv; j++)
        for (int i = 0; i <= j; i++) {
          const double t = Td[(size_t)j * ncv + i];
          finite = finite && std::isfinite(t);
          T[(size_t)j * ncv + i] = t;
          T[(size_t)i * ncv + j] = t;
        }
      // the device-vector products turn a zero / non-finite scale or center into an all-NaN result (include/bsgpu.h):
      // stop here instead of iterating on NaNs (RSpectra fails on such an operator too)
      if (!finite)
        return fail(BSG_ERR_ARG, "non-finite values in the scaled matrix-vector products (zero or non-finite scale / center?).");
    }
    have = ncv;
    // ---- Ritz pairs of the projected matrix
    jacobi_eigh(T, ncv, theta, Sm);
    const double eps23 = pow(2.220446049250313e-16, 2.0 / 3.0);
    nconv = 0;
    for (int i = 0; i < k; i++) {
      double res = fabs(beta_last * Sm[(size_t)i * ncv + (ncv - 1)]);
      if (res <= tol * std::max(eps23, fabs(theta[i]))) nconv++;
    }
    iters++;
    if (nconv >= k || iters >= maxit || full_space || ncv >= N) break;
    // ---- thick restart: keep nkeep Ritz vectors + the residual direction
    int nkeep = k + std::min(nconv, (ncv - k) / 2);
    if (nkeep == 1 && ncv > 3) nkeep = ncv / 2;
    nkeep = std::min(nkeep, ncv - 1);
    std::fill(T.begin(), T.end(), 0.0);
    for (int i = 0; i < nkeep; i++) {
      T[(size_t)i * ncv + i] = theta[i];
      double b = beta_last * Sm[(size_t)i * ncv + (ncv - 1)];
      T[(size_t)nkeep * ncv + i] = b;
      T[(size_t)i * ncv + nkeep] = b;
    }
    for (int g = 0; g < G; g++) {
      BSG_TRY(bind_device(sh[g].h));
      SvdWork &W = rep[g].W;
      cudaStream_t s = rep[g].s;
      BSG_CUDA(cudaMemcpyAsync(W.S, Sm.data(), (size_t)ncv * ncv * sizeof(double), cudaMemcpyHostToDevice, s));
      BSG_CUDA(cudaMemcpyAsync(W.T, T.data(), (size_t)ncv * ncv * sizeof(double), cudaMemcpyHostToDevice, s));
      dim3 grid(gblocks(N), nkeep);
      k_combine<<<grid, TB, 0, s>>>(W.V, ld, ncv, W.S, ncv, nkeep, N, W.Y, ld);
      count_launch();
      BSG_CUDA(cudaMemcpyAsync(W.V, W.Y, (size_t)ld * nkeep * sizeof(double), cudaMemcpyDeviceToDevice, s));
      BSG_CUDA(cudaMemcpyAsync(W.V + (int64_t)nkeep * ld, W.V + (int64_t)ncv * ld, (size_t)N * sizeof(double),
                               cudaMemcpyDeviceToDevice, s));
    }
    have = nkeep;
  }

  // ---- singular triplets
  std::vector<double> side((size_t)N * k);
  for (int c = 0; c < k; c++) d[c] = sqrt(std::max(theta[c], 0.0));
  std::vector<std::vector<double>> other(G);
  for (int g = 0; g < G; g++) {
    BSG_TRY(bind_device(sh[g].h));
    SvdWork &W = rep[g].W;
    cudaStream_t s = rep[g].s;
    const int Mo = row_side ? sh[g].nc : nr;
    BSG_CUDA(cudaMemcpyAsync(W.S, Sm.data(), (size_t)ncv * ncv * sizeof(double), cudaMemcpyHostToDevice, s));
    dim3 grid(gblocks(N), k);
    k_combine<<<grid, TB, 0, s>>>(W.V, ld, ncv, W.S, ncv, k, N, W.Y, ld);
    count_launch();
    if (g == 0) BSG_CUDA(cudaMemcpyAsync(side.data(), W.Y, (size_t)N * k * sizeof(double), cudaMemcpyDeviceToHost, s));
    other[g].resize((size_t)std::max(Mo, 1) * k);
    for (int c = 0; c < k && Mo > 0; c++) {
      BSG_TRY(row_side ? bsg_view_cprodvec_dev(rep[g].view, W.Y + (int64_t)c * ld, W.tmp, s)
                       : bsg_view_prodvec_dev(rep[g].view, W.Y + (int64_t)c * ld, W.tmp, s));
      k_scale_copy<<<gblocks(Mo), TB, 0, s>>>(W.tmp, d[c] > 0 ? 1.0 / d[c] : 0.0, Mo, W.other);
      count_launch();
      BSG_CUDA(cudaMemcpyAsync(other[g].data() + (size_t)c * Mo, W.other, (size_t)Mo * sizeof(double), cudaMemcpyDeviceToHost, s));
      BSG_CUDA(cudaStreamSynchronize(s));  // W.other is reused by the next column
    }
  }
  for (int g = 0; g < G; g++) {
    BSG_TRY(bind_device(sh[g].h));
    BSG_CUDA(cudaStreamSynchronize(rep[g].s));
  }
  // deterministic sign: the entry of largest magnitude of each left vector (row side) is positive
  for (int c = 0; c < k; c++) {
    const double *us = row_side ? side.data() + (size_t)c * N : other[0].data() + (size_t)c * nr;
    const int len = row_side ? N : nr;
    double best = 0;
    for (int i = 0; i < len; i++)
      if (fabs(us[i]) > fabs(best)) best = us[i];
    if (best < 0) {
      for (int i = 0; i < N; i++) side[(size_t)c * N + i] = -side[(size_t)c * N + i];
      for (int g = 0; g < G; g++) {
        const int Mo = row_side ? sh[g].nc : nr;
        for (int i = 0; i < Mo; i++) other[g][(size_t)c * Mo + i] = -other[g][(size_t)c * Mo + i];
      }
    }
  }
  if (row_side) {
    if (u) memcpy(u, side.data(), (size_t)nr * k * sizeof(double));
    for (int g = 0; g < G; g++) {
      if (!sh[g].v_out) continue;
      const int Mo = sh[g].nc;
      for (int c = 0; c < k; c++)
        for (int j = 0; j < Mo; j++) {
          const int64_t row = sh[g].v_pos ? sh[g].v_pos[j] : j;
          sh[g].v_out[(size_t)c * sh[g].v_ld + row] = other[g][(size_t)c * Mo + j];
        }
    }
  } else {
    if (u) memcpy(u, other[0].data(), (size_t)nr * k * sizeof(double));
    if (sh[0].v_out)
      for (int c = 0; c < k; c++)
        for (int j = 0; j < N; j++) {
          const int64_t row = sh[0].v_pos ? sh[0].v_pos[j] : j;
          sh[0].v_out[(size_t)c * sh[0].v_ld + row] = side[(size_t)c * N + j];
        }
  }
  if (niter) *niter = iters;
  if (nops) *nops = ops;
  g_last_nconv = (full_space || ncv >= N) ? k : nconv;  // the full space is exact
  return BSG_OK;
}

}  // namespace bsg

using namespace bsg;

extern "C" {

// RSpectra::svds (behind big_randomSVD) warns when fewer than k values converged within maxit; the count of the last
// call on this thread is exposed so the host wrapper can do the same
int bsg_randomsvd_nconv(void) { return g_last_nconv; }

// Callback form kept for hosts that bring their own collective: `z_dev` (nr doubles) holds the n-vector of partial
// products; after every local A (A^T x) the library synchronises its stream and calls reduce_cb(ctx), which must sum z_dev
// across ranks and return once the sum is visible.  The communicator form (bsg_randomsvd_comm) needs neither.
int bsg_randomsvd_ex(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                     const double *scale, int k, double tol, int maxit, double *d, double *u, double *v,
                     double *center_out, double *scale_out, int *niter, int *nops, double *z_dev,
                     bsg_reduce_cb reduce_cb, void *ctx, int ncol_total) {
  if (!h || !d) return fail(BSG_ERR_ARG, "null argument");
  if (!ind_col) nc = h->m;
  std::vector<SvdShard> sh(1);
  sh[0] = SvdShard{h, ind_col, nc, center, scale, nullptr, v, nc, nullptr, center_out, scale_out};
  return lanczos_svd(sh, ind_row, nr, ncol_total, k, tol, maxit, d, u, niter, nops, z_dev, reduce_cb, ctx);
}

int bsg_randomsvd(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                  const double *scale, int k, double tol, int maxit, double *d, double *u, double *v,
                  double *center_out, double *scale_out, int *niter, int *nops) {
  return bsg_randomsvd_ex(h, ind_row, nr, ind_col, nc, center, scale, k, tol, maxit, d, u, v, center_out, scale_out,
                          niter, nops, nullptr, nullptr, nullptr, 0);
}

// ---------------------------------------------------------------------------------------------------
// fp64 path: device decode of column blocks + cuBLAS DSYRK.  Used when no sample-major copy is resident or the
// scaling is degenerate (zero / negative scale, negative center, non-finite weights).
__global__ void k_mirror_lower(double *K, int n) {  // K[j, i] (upper) = K[i, j] (lower), column-major
  const int64_t total = (int64_t)n * n;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(t % n), j = (int)(t / n);
    if (i > j) K[(int64_t)i * n + j] = K[t];
  }
}

// K (host) and / or K_dev (caller's device buffer, nr x nr) receive the result
static int tcrossprod_dsyrk(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                            const double *scale, double *K, double *K_dev) {
  cudaStream_t s = h->stream;
  const int *d_row = nullptr, *d_col = nullptr;
  BSG_TRY(upload_index(h, ind_row, nr, h->n, h->w_idx_row, &d_row));
  std::vector<int> iota;
  if (!ind_col) {  // column blocks are addressed through an explicit list
    iota.resize(nc);
    for (int j = 0; j < nc; j++) iota[j] = j + 1;
    ind_col = iota.data();
  }
  BSG_TRY(upload_index(h, ind_col, nc, h->m, h->w_idx_col, &d_col));
  size_t nn = (size_t)std::max(nc, 1);
  BSG_TRY(h->w_center.ensure(nn * sizeof(double)));
  BSG_TRY(h->w_scale.ensure(nn * sizeof(double)));
  BSG_CUDA(cudaMemcpyAsync(h->w_center.p, center, (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, s));
  BSG_CUDA(cudaMemcpyAsync(h->w_scale.p, scale, (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, s));
  // block of columns sized to ~1 GB of decoded doubles
  int blk = (int)std::max<int64_t>(64, std::min<int64_t>(nc > 0 ? nc : 1, ((int64_t)1 << 27) / std::max(nr, 1)));
  double *dK = K_dev, *dX = nullptr;
  if (!K_dev) BSG_CUDA(cudaMalloc((void **)&dK, (size_t)std::max(nr, 1) * std::max(nr, 1) * sizeof(double)));
  cudaError_t e = cudaMalloc((void **)&dX, (size_t)std::max(nr, 1) * blk * sizeof(double));
  if (e != cudaSuccess) {
    if (!K_dev) cudaFree(dK);
    return cuda_fail(e, "GRM block");
  }
  cublasHandle_t cb = nullptr;
  if (cublasCreate(&cb) != CUBLAS_STATUS_SUCCESS) {
    if (!K_dev) cudaFree(dK);
    cudaFree(dX);
    return fail(BSG_ERR_CUDA, "cublasCreate failed");
  }
  cublasSetStream(cb, s);
  cudaMemsetAsync(dK, 0, (size_t)nr * nr * sizeof(double), s);
  int rc = BSG_OK;
  const double one = 1.0;
  for (int j0 = 0; j0 < nc && !rc; j0 += blk) {
    int b = std::min(blk, nc - j0);
    rc = read_dense_scaled(h, d_row, nr, d_col + j0, b, h->w_center.as<double>() + j0, h->w_scale.as<double>() + j0,
                           dX, s);
    if (!rc && nr > 0 &&
        cublasDsyrk(cb, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_N, nr, b, &one, dX, nr, &one, dK, nr) != CUBLAS_STATUS_SUCCESS)
      rc = fail(BSG_ERR_CUDA, "cublasDsyrk failed");
  }
  if (!rc && nr > 0) {
    k_mirror_lower<<<(int)std::min<int64_t>(((int64_t)nr * nr + 255) / 256, 148 * 32), 256, 0, s>>>(dK, nr);
    count_launch();
    cudaError_t e2 = cudaGetLastError();
    if (K) prefault_pages(K, (size_t)nr * nr * sizeof(double));
    if (e2 == cudaSuccess && K) e2 = cudaMemcpyAsync(K, dK, (size_t)nr * nr * sizeof(double), cudaMemcpyDeviceToHost, s);
    if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(s);
    if (e2 != cudaSuccess) rc = cuda_fail(e2, "GRM download");
  }
  cublasDestroy(cb);
  if (!K_dev) cudaFree(dK);
  cudaFree(dX);
  return rc;
}


}  // extern "C"

struct DevPtrs {
  std::vector<void *> p;
  ~DevPtrs() {
    for (void *q : p)
      if (q) cudaFree(q);
  }
  template <class T>
  int alloc(T **out, size_t count) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, (count ? count : 1) * sizeof(T));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(GRM)");
    p.push_back(q);
    *out = (T *)q;
    return BSG_OK;
  }
};

extern "C" {

}  // extern "C"

static int tcrossprod_impl(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                           const double *scale, double *K, double *K_dev) {
  if (!h || (!K && !K_dev)) return fail(BSG_ERR_ARG, "null argument");
  BSG_PACKED_ONLY(h, "The Gram product");
  if (!center || !scale) return fail(BSG_ERR_DIM, "Incompatibility between dimensions.");
  BSG_TRY(bind_device(h));
  if (!ind_row) nr = h->n;
  if (!ind_col) nc = h->m;
  // Weight digits: base 128 (7 bits; the B byte code * digit <= 2 * 127 still fits u8 and a whole sweep of up to 4.2 M
  // columns fits the int32 accumulator: 2 * 254 * m < 2^31), 4 slices = 28 bits of each per-SNP weight -> K agrees with
  // the fp64 reference to ~1e-9, three orders inside the 1e-6 contract.  BSG_GRM_SLICES changes the count.
  static int force_dsyrk = -1, nslices = 4;
  if (force_dsyrk < 0) {
    const char *ev = getenv("BSG_GRM_DSYRK");
    force_dsyrk = (ev && ev[0] == '1') ? 1 : 0;
    const char *es = getenv("BSG_GRM_SLICES");
    if (es) nslices = std::min(9, std::max(2, atoi(es)));
  }
  if (!force_dsyrk && !h->B && nr > 0 && nc > 0 && build_copy_B(h) != BSG_OK) cudaGetLastError();  // no room: fp64 path
  if (force_dsyrk || !h->B || nr == 0 || nc == 0) return tcrossprod_dsyrk(h, ind_row, nr, ind_col, nc, center, scale, K, K_dev);
  using namespace wgram;
  cudaStream_t s = h->stream;
  DevPtrs mem;
  // ---- weights
  double *d_c = nullptr, *d_s = nullptr, *W1 = nullptr, *W2p = nullptr, *W3 = nullptr, *w2 = nullptr, *d_stats = nullptr;
  BSG_TRY(mem.alloc(&d_c, nc));
  BSG_TRY(mem.alloc(&d_s, nc));
  BSG_TRY(mem.alloc(&W1, nc));
  BSG_TRY(mem.alloc(&W2p, nc));
  BSG_TRY(mem.alloc(&W3, nc));
  BSG_TRY(mem.alloc(&w2, nc));
  BSG_TRY(mem.alloc(&d_stats, 8));
  BSG_CUDA(cudaMemcpyAsync(d_c, center, (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, s));
  BSG_CUDA(cudaMemcpyAsync(d_s, scale, (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, s));
  BSG_CUDA(cudaMemsetAsync(d_stats, 0, 8 * sizeof(double), s));
  k_grm_weights<<<(nc + 255) / 256, 256, 0, s>>>(d_c, d_s, nc, W1, W2p, W3, w2, d_stats);
  count_launch();
  double stats[8];
  std::vector<double> hW3(nc);
  BSG_CUDA(cudaMemcpyAsync(stats, d_stats, sizeof stats, cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaMemcpyAsync(hW3.data(), W3, (size_t)nc * sizeof(double), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaStreamSynchronize(s));
  if (stats[4] != 0.0) return tcrossprod_dsyrk(h, ind_row, nr, ind_col, nc, center, scale, K, K_dev);
  double sumW3 = 0;
  for (int j = 0; j < nc; j++) sumW3 += hW3[j];

  // ---- the sub-matrix X[ind_row, ind_col] as dense sample-major lines
  const bool ident = (!ind_row || [&] { if (nr != h->n) return false; for (int i = 0; i < nr; i++) if (ind_row[i] != i + 1) return false; return true; }()) &&
                     (!ind_col || [&] { if (nc != h->m) return false; for (int j = 0; j < nc; j++) if (ind_col[j] != j + 1) return false; return true; }());
  const uint8_t *P = h->B;
  int64_t stride = h->strideB;
  uint8_t *d_na = nullptr;
  BSG_TRY(mem.alloc(&d_na, nr));
  if (!ident) {
    const int *d_row = nullptr, *d_col = nullptr;
    BSG_TRY(upload_index(h, ind_row, nr, h->n, h->w_idx_row, &d_row));
    BSG_TRY(upload_index(h, ind_col, nc, h->m, h->w_idx_col, &d_col));
    stride = round_up(((int64_t)nc + 3) / 4, CHUNK);
    uint8_t *Pc = nullptr;
    BSG_TRY(mem.alloc(&Pc, (size_t)stride * nr));
    // sub-matrix of the sample-major copy: lines = selected samples, codes = selected SNPs
    BSG_TRY(compact_lines(h->B, h->strideB, d_col, nc, d_row, nr, Pc, stride, s));
    int32_t *d_cnt = nullptr;
    BSG_TRY(mem.alloc(&d_cnt, (size_t)nr * 4));
    BSG_TRY(line_counts(Pc, stride, nr, nc, d_cnt, d_na, s));
    P = Pc;
  } else {
    BSG_CUDA(cudaMemcpyAsync(d_na, h->naB, (size_t)nr, cudaMemcpyDeviceToDevice, s));
  }
  std::vector<uint8_t> na(nr);
  BSG_CUDA(cudaMemcpyAsync(na.data(), d_na, (size_t)nr, cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaStreamSynchronize(s));
  const int nchunks = (int)(stride / CHUNK);

  double *dK = K_dev;
  if (!K_dev) BSG_TRY(mem.alloc(&dK, (size_t)nr * nr));
  BSG_CUDA(cudaMemsetAsync(dK, 0, (size_t)nr * nr * sizeof(double), s));
  if (gramt_enabled() && nslices <= 4) {
    // TMA-fed 2-CTA tcgen05 tiles over operands expanded once to uint8 (bsg_gramt.cu): all digit slices in one pass
    const double *Ws3[3] = {W1, W2p, W3};
    const double wmax[3] = {stats[0], stats[1], stats[2]};
    BSG_TRY(gramt_grm(P, stride, nr, nc, Ws3, wmax, na.data(), nslices, dK, nr, h->device, s));
  } else {
  // ---- weight digits (base 64, nslices digits) in fragment order
  WArgs a;
  a.P = P;
  a.stride = stride;
  a.nlines = nr;
  a.nchunks = nchunks;
  a.nslices = nslices;
  const double *Ws[3] = {W1, W2p, W3};
  const int dbits = nc <= 4000000 ? 7 : 6;  // longer sweeps keep the int32 head-room with 6-bit digits (2 * 126 * m < 2^31 up to 8.5 M)
  for (int wv = 0; wv < 3; wv++) {
    uint8_t *dg = nullptr;
    BSG_TRY(mem.alloc(&dg, (size_t)nslices * nchunks * 256));
    int ex = 0;
    if (stats[wv] > 0) frexp(stats[wv], &ex);
    const int e = dbits * nslices - 1 - ex;
    k_weight_digits<<<(int)std::min<int64_t>(((int64_t)nchunks * 256 + 255) / 256, 148 * 16), 256, 0, s>>>(Ws[wv], nc, nchunks,
                                                                                                        nslices, e, dbits, dg);
    count_launch();
    a.dig[wv] = dg;
    for (int sl = 0; sl < nslices; sl++) a.scale[wv][sl] = ldexp(1.0, dbits * sl - e);
  }

  // ---- tiles of the lower triangle
  static int use_t5 = -1;
  if (use_t5 < 0) {
    const char *ev = getenv("BSG_GRM_TCGEN05");
    use_t5 = (ev && ev[0] == '0') ? 0 : 1;
  }
  const int TNv = use_t5 ? 128 : TN;
  const int njb = (nr + TNv - 1) / TNv;
  std::vector<uint8_t> na_jb(njb, 0);
  for (int i = 0; i < nr; i++) na_jb[i / TNv] |= na[i];
  if (use_t5) {
    // 128 x 128 tiles on tcgen05 / TMEM (bsg_gram5.cu); digits are laid out 16 bytes per packed word, in order
    std::vector<int> trip;
    for (int i0 = 0; i0 < nr; i0 += 128) {
      const bool na_i = na_jb[i0 / 128] != 0;
      for (int j0 = 0; j0 <= i0; j0 += 128) {
        trip.push_back(i0);
        trip.push_back(j0);
        trip.push_back((na_i || na_jb[j0 / 128]) ? 1 : 0);
      }
    }
    const uint8_t *digs[3] = {a.dig[0], a.dig[1], a.dig[2]};
    BSG_TRY(wgram5_launch(P, stride, nr, nslices, digs, (int64_t)nchunks * 256, a.scale, trip.data(), (int)(trip.size() / 3),
                          dK, nr, s));
  } else {
    std::vector<WTile> tiles;
    for (int i0 = 0; i0 < nr; i0 += TM) {
      bool na_i = false;
      for (int b = i0 / TN; b <= std::min(nr - 1, i0 + TM - 1) / TN; b++) na_i |= na_jb[b] != 0;
      for (int j0 = 0; j0 <= std::min(nr - 1, i0 + TM - 1); j0 += TN)
        tiles.push_back(WTile{i0, j0, (na_i || na_jb[j0 / TN]) ? 1 : 0});
    }
    WTile *d_tiles = nullptr;
    BSG_TRY(mem.alloc(&d_tiles, tiles.size()));
    BSG_CUDA(cudaMemcpyAsync(d_tiles, tiles.data(), tiles.size() * sizeof(WTile), cudaMemcpyHostToDevice, s));
    a.tiles = d_tiles;
    a.K = dK;
    a.ldk = nr;
    k_wgram<<<(unsigned)tiles.size(), THREADS, 0, s>>>(a);
    count_launch();
    BSG_CUDA(cudaGetLastError());
    BSG_CUDA(cudaStreamSynchronize(s));
  }

  }

  // ---- vector terms through the matvec engine:  r = A w2 ;  q = N w3 = (X~_{c=1,s=1} w3) - A w3 + sum(w3)
  double *d_r = nullptr, *d_q = nullptr, *d_t1 = nullptr;
  BSG_TRY(mem.alloc(&d_r, nr));
  bsg_view *v0 = nullptr;
  BSG_TRY(bsg_view_create(h, ind_row, nr, ind_col, nc, nullptr, nullptr, &v0));
  int rc = bsg_view_prodvec_dev(v0, w2, d_r, s);
  bool any_na = false;
  for (int i = 0; i < nr && !any_na; i++) any_na = na[i] != 0;
  if (!rc && any_na) {
    rc = mem.alloc(&d_q, nr);
    if (!rc) rc = mem.alloc(&d_t1, nr);
    std::vector<double> ones(nc, 1.0);
    bsg_view *v1 = nullptr;
    if (!rc) rc = bsg_view_prodvec_dev(v0, W3, d_t1, s);  // A w3
    if (!rc) rc = bsg_view_create(h, ind_row, nr, ind_col, nc, ones.data(), ones.data(), &v1);
    if (!rc) rc = bsg_view_prodvec_dev(v1, W3, d_q, s);   // A w3 - sum_nonNA w3
    if (!rc) {
      cudaStreamSynchronize(s);
      std::vector<double> hq(nr), ht(nr);
      cudaMemcpy(hq.data(), d_q, (size_t)nr * sizeof(double), cudaMemcpyDeviceToHost);
      cudaMemcpy(ht.data(), d_t1, (size_t)nr * sizeof(double), cudaMemcpyDeviceToHost);
      for (int i = 0; i < nr; i++) hq[i] = hq[i] - ht[i] + sumW3;
      cudaMemcpy(d_q, hq.data(), (size_t)nr * sizeof(double), cudaMemcpyHostToDevice);
    }
    if (v1) {
      cudaStreamSynchronize(s);
      bsg_view_destroy(v1);
    }
  }
  if (!rc) {
    k_grm_finish<<<(int)std::min<int64_t>(((int64_t)nr * nr + 255) / 256, 148 * 32), 256, 0, s>>>(dK, nr, nr, d_r, d_q, sumW3);
    count_launch();
    cudaError_t e2 = cudaGetLastError();
    if (K) prefault_pages(K, (size_t)nr * nr * sizeof(double));  // 800 MB at configs[3], while the device still computes
    if (e2 == cudaSuccess && K) e2 = cudaMemcpyAsync(K, dK, (size_t)nr * nr * sizeof(double), cudaMemcpyDeviceToHost, s);
    if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(s);
    if (e2 != cudaSuccess) rc = cuda_fail(e2, "GRM download");
  }
  cudaStreamSynchronize(s);
  bsg_view_destroy(v0);
  return rc;
}

extern "C" {

int bsg_tcrossprod(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                   const double *scale, double *K) {
  if (!K) return fail(BSG_ERR_ARG, "null argument");
  return tcrossprod_impl(h, ind_row, nr, ind_col, nc, center, scale, K, nullptr);
}

int bsg_tcrossprod_dev(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                       const double *scale, double *K_dev) {
  if (!K_dev) return fail(BSG_ERR_ARG, "null argument");
  return tcrossprod_impl(h, ind_row, nr, ind_col, nc, center, scale, nullptr, K_dev);
}

}  // extern "C"
