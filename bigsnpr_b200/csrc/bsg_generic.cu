// bsg_generic.cu -- fp64 fallback for FBM.code256 objects whose 256 code values are not the hard calls 0 / 1 / 2 / NA
// (dosages, R/bigSNP-class.R:13 CODE_DOSAGE; SURVEY.md section 8f row 3).  The packed 2-bit engine is exact only for hard
// calls, so such handles keep the n x m code bytes in HBM and the snp_* entry points of the path read code256[byte] per
// element exactly like bigstatsr's SubBMCode256Acc does in the reference:
//   snp_colstats   src/colstats.cpp:8-35      (no missing-value handling: NA poisons the column)
//   corMat / ld_scores on an FBM   src/corr.cpp:32-93,113-118, src/ld-scores.cpp:25-75,93-96   (code[is_na(code)] = 3)
//   clumping_chr   src/clumping.cpp:60-75
//   multLinReg     src/multLinReg.cpp:8-60
// One warp per column / pair, lanes over the samples, fixed-shape shuffle reductions (deterministic).  Sums of non-integer
// values are rounded in a different order than the reference's sequential loop: results agree to ~1e-13 relative, the
// contract for floating-point output is 1e-6.  HBM-bound byte streaming; a fallback, not a tuned path.
#include <math.h>

#include <algorithm>

#include "bsg_internal.cuh"

namespace bsg {
namespace gen {

__device__ __forceinline__ double wsum(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void k_colstats(const uint8_t *__restrict__ raw, int64_t n_tot, const double *__restrict__ code,
                           const int *__restrict__ rows, int nr, const int *__restrict__ cols, int nc,
                           double *__restrict__ sumX, double *__restrict__ denoX) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, nw = (gridDim.x * blockDim.x) >> 5;
  for (int j = warp; j < nc; j += nw) {
    const uint8_t *col = raw + (int64_t)(cols ? cols[j] : j) * n_tot;
    double xs = 0, xx = 0;
    for (int i = lane; i < nr; i += 32) {
      const double x = code[col[rows ? rows[i] : i]];
      xs += x;
      xx += x * x;
    }
    xs = wsum(xs);
    xx = wsum(xx);
    if (lane == 0) {
      sumX[j] = xs;
      denoX[j] = xx - xs * xs / nr;
    }
  }
}

// pair o of the band: j0 by binary search on boff, j = j0 - 1 - (o - boff[j0])
template <int KIND>
__global__ void k_pairs(const uint8_t *__restrict__ raw, int64_t n_tot, const double *__restrict__ code3,
                        const double *__restrict__ code, const int *__restrict__ rows, int nr, const int *__restrict__ cols,
                        int nc, const int *__restrict__ wlen, const long long *__restrict__ boff, long long total,
                        const double *__restrict__ thr, double *__restrict__ band, uint8_t *__restrict__ keep,
                        const double *__restrict__ sumX, const double *__restrict__ denoX, double thr_r2) {
  const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5, nw = ((long long)gridDim.x * blockDim.x) >> 5;
  const int lane = threadIdx.x & 31;
  for (long long o = warp; o < total; o += nw) {
    int lo = 0, hi = nc - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (boff[mid] <= o) lo = mid; else hi = mid - 1;
    }
    const int j0 = lo, j = j0 - 1 - (int)(o - boff[j0]);
    const uint8_t *cx = raw + (int64_t)(cols ? cols[j0] : j0) * n_tot, *cy = raw + (int64_t)(cols ? cols[j] : j) * n_tot;
    if (KIND == 3) {
      // xySum with the accessor's values (NA_real for a missing code: the sum and r2 are NA, never > thr)
      double xy = 0;
      for (int i = lane; i < nr; i += 32) {
        const int r = rows ? rows[i] : i;
        xy += code[cx[r]] * code[cy[r]];
      }
      xy = wsum(xy);
      if (lane == 0) {
        const double num = xy - sumX[j] * sumX[j0] / nr;
        const double r2 = num * num / (denoX[j] * denoX[j0]);
        keep[o] = (r2 > thr_r2) ? 1 : 0;  // false for NaN
      }
      continue;
    }
    // pairwise-complete sums (src/corr.cpp:52-75): x = column j0, y = column j, value 3 = missing
    double nona = 0, xs = 0, xx = 0, ys = 0, yy = 0, xy = 0;
    for (int i = lane; i < nr; i += 32) {
      const int r = rows ? rows[i] : i;
      const double x = code3[cx[r]], y = code3[cy[r]];
      if (x != 3 && y != 3) {
        nona += 1;
        xs += x;
        xx += x * x;
        ys += y;
        yy += y * y;
        xy += x * y;
      }
    }
    nona = wsum(nona); xs = wsum(xs); xx = wsum(xx); ys = wsum(ys); yy = wsum(yy); xy = wsum(xy);
    if (lane == 0) {
      const double num = xy - xs * ys / nona;
      const double deno_x = xx - xs * xs / nona, deno_y = yy - ys * ys / nona;
      if (KIND == 1) {
        band[o] = num * num / (deno_x * deno_y);
      } else {
        double r = num / sqrt(deno_x * deno_y);
        const int nn = (int)nona;
        const bool kp = isnan(r) || fabs(r) > thr[nn > 0 ? nn - 1 : 0];
        if (r > 1) r = 1; else if (r < -1) r = -1;
        band[o] = r;
        keep[o] = kp;
      }
    }
  }
}

// t-scores of the regression of every column on each column of U (src/multLinReg.cpp:24-55); out is nc x K column-major
__global__ void k_multlinreg(const uint8_t *__restrict__ raw, int64_t n_tot, const double *__restrict__ code3,
                             const int *__restrict__ rows, int nr, const int *__restrict__ cols, int nc,
                             const double *__restrict__ U, int K, double *__restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, nw = (gridDim.x * blockDim.x) >> 5;
  for (int j = warp; j < nc; j += nw) {
    const uint8_t *col = raw + (int64_t)(cols ? cols[j] : j) * n_tot;
    double nona = 0, xs = 0, xx = 0;
    for (int i = lane; i < nr; i += 32) {
      const double x = code3[col[rows ? rows[i] : i]];
      if (x != 3) {
        nona += 1;
        xs += x;
        xx += x * x;
      }
    }
    nona = wsum(nona); xs = wsum(xs); xx = wsum(xx);
    const double deno_x = xx - xs * xs / nona;
    for (int k = 0; k < K; k++) {
      double xy = 0, ys = 0, yy = 0;
      for (int i = lane; i < nr; i += 32) {
        const double x = code3[col[rows ? rows[i] : i]];
        if (x != 3) {
          const double y = U[(int64_t)k * nr + i];
          xy += x * y;
          ys += y;
          yy += y * y;
        }
      }
      xy = wsum(xy); ys = wsum(ys); yy = wsum(yy);
      if (lane == 0) {
        const double num = xy - xs * ys / nona, deno_y = yy - ys * ys / nona;
        const double deno = deno_x * deno_y - num * num;
        out[(int64_t)k * nc + j] = (deno == 0 || nona < 2) ? nan("") : num * sqrt((nona - 2) / deno);
      }
    }
  }
}

static int grid_warps(long long items) { return (int)std::max<long long>(1, std::min<long long>((items * 32 + 255) / 256, 148 * 16)); }

}  // namespace gen

int generic_colstats(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, double *d_sumX, double *d_denoX,
                     cudaStream_t s) {
  if (nc <= 0) return BSG_OK;
  gen::k_colstats<<<gen::grid_warps(nc), 256, 0, s>>>(h->raw, h->raw_stride, h->d_code, d_row, nr, d_col, nc, d_sumX, d_denoX);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

int generic_pairs(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, int kind, const int *d_wlen,
                  const long long *d_boff, long long total, const double *d_thr, double *d_band, uint8_t *d_keep,
                  const double *d_sumX, const double *d_denoX, double thr_r2, cudaStream_t s) {
  if (total <= 0) return BSG_OK;
  const int grid = gen::grid_warps(total);
  const double *c3 = h->d_code + 256;
  if (kind == 0)
    gen::k_pairs<0><<<grid, 256, 0, s>>>(h->raw, h->raw_stride, c3, h->d_code, d_row, nr, d_col, nc, d_wlen, d_boff, total, d_thr, d_band, d_keep, d_sumX, d_denoX, thr_r2);
  else if (kind == 1)
    gen::k_pairs<1><<<grid, 256, 0, s>>>(h->raw, h->raw_stride, c3, h->d_code, d_row, nr, d_col, nc, d_wlen, d_boff, total, d_thr, d_band, d_keep, d_sumX, d_denoX, thr_r2);
  else
    gen::k_pairs<3><<<grid, 256, 0, s>>>(h->raw, h->raw_stride, c3, h->d_code, d_row, nr, d_col, nc, d_wlen, d_boff, total, d_thr, d_band, d_keep, d_sumX, d_denoX, thr_r2);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

int generic_multlinreg(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, const double *d_U, int K,
                       double *d_out, cudaStream_t s) {
  if (nc <= 0 || K <= 0) return BSG_OK;
  gen::k_multlinreg<<<gen::grid_warps(nc), 256, 0, s>>>(h->raw, h->raw_stride, h->d_code + 256, d_row, nr, d_col, nc, d_U, K, d_out);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

}  // namespace bsg
