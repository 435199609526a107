// bsg_pmv.cu -- X.y and Xt.y over the packed genotypes: bed_pMatVec4 / bed_cpMatVec4
// (src/bed-prod-vec.cpp:15-54, :59-97) re-designed for sm_100a.
//
// Why not one-thread-per-genotype: at 2 bits per genotype the HBM roofline is 4 genotypes per byte
// (2.6e13 genotypes/s at the measured 6.57 TB/s), more than the SIMT pipes can issue as
// extract + table lookup + DFMA (SURVEY.md section 7 "Hard parts").  So the per-genotype multiply-add is
// moved to the integer tensor pipe and made EXACT:
//
//   * the vector is quantised once per call to 61-bit fixed point, Q_k = rint(y_k * 2^e) with
//     |Q_k| < 2^60, and split into 8 signed base-256 digits (int8).  Digit s of every element is
//     column s of an int8 "B" operand with N = 8.
//   * the staged 2-bit code of a genotype is its value (0/1/2, 3 = missing), so masking a packed
//     32-bit word with 0x03030303 / 0x30303030 (and the same after >> 2) yields four uint8 "A"
//     fragments holding 16 genotypes with NO unpack arithmetic beyond 1 shift + 4 ANDs: the fields
//     left in place at bit 4 are simply worth 16x and accumulate in a second accumulator.
//   * mma.sync.m16n8k32.u8.s8.s32 accumulates sum_k code_k * digit_k exactly in int32; the 8 slices
//     are recombined in fp64 only at the very end.  A second plane ([code == 3]) gives the sum of
//     the vector over missing entries, which turns "NA -> 0 after centering" into algebra:
//         sum_i (g-c)/s * y_i  over non-missing  =  (R - 3N - c (Y - N)) / s,
//         R = sum code*y, N = sum [NA]*y, Y = sum y.
//   * integer partial sums make the result independent of the work split and of the GPU count.
//
// Data movement (measured on B200, tools/ubench.cu): cp.async.bulk costs ~55 cycles per copy whatever
// its size, so 128-byte per-line copies cap at 0.7 TB/s; IMMA.16832 sustains one per 2.4 cycles per SM.
// Hence: the packed genotypes never touch shared memory -- each consumer lane streams its own fragment
// bytes with ld.global.nc.L1::no_allocate.v4 (every warp-level load covers 8 lines x 64 contiguous
// bytes = full sectors) through a 4-slot register ring (3 half-stages in flight per warp); only the
// 4 KB digit block of each 512-code chunk goes through a shared-memory ring, filled by one bulk copy
// per stage from a producer warp (mbarrier full/empty).
//
// Contents, in order: k_pmv (lines = contraction-contiguous: Xt.y on the SNP-major copy, X.y on the sample-major
// copy); vector preparation and finish kernels; k_pmvT / k_pmvT2 (X.y straight from the SNP-major copy: the
// contraction runs across lines, bytes are transposed in registers; T2 = raw + flag plane in one pass); the sparse
// missing-value lists; views and the C-ABI entry points (bsg_prodvec / bsg_cprodvec / bsg_view_*); the planes API
// behind bsg_prod_and_rowsumssq, bsg_multlinreg and the by-row counts.
#include <algorithm>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cub/device/device_scan.cuh>

#include "bsg_internal.cuh"
#include "bsg_pmv_shared.cuh"

namespace bsg {
namespace pmv {

// Fragment bytes of one lane for one 16-line sub-tile and one 128-byte chunk: lines g (a*) and g+8 (b*),
// bytes [16q, 16q+16) (lo) and [64+16q, 64+16q+16) (hi) of the chunk.
struct Slot {
  uint4 alo, ahi, blo, bhi;
};

__device__ __forceinline__ void slot_load(Slot &s, const uint8_t *pa, const uint8_t *pb, int64_t off) {
  s.alo = ldg_stream(pa + off);
  s.ahi = ldg_stream(pa + off + 64);
  s.blo = ldg_stream(pb + off);
  s.bhi = ldg_stream(pb + off + 64);
}

// Second plane of the packed codes, one bit per code at the low bit of its 2-bit field: MODE 1 / 2 = missing
// value flag (code 3: both bits set), MODE 3 = the high bit alone (codes 2 and 3; sums of squares need it).
template <int MODE>
__device__ __forceinline__ uint32_t plane2(uint32_t x) {
  return MODE == 3 ? (x >> 1) : (x & (x >> 1));
}

// One chunk of the warp's 32 lines (two 16-line sub-tiles t0 / t1).  Word w of the lane (w < 4: lo bytes,
// w >= 4: hi bytes) holds 16 codes of each of its 4 lines; d = digits of slice g for those 16 codes (one
// LDS.128 per word, shared by both sub-tiles), register c <-> codes 4r+c (r = byte of the register).
// The four MMAs of a word go to four different accumulators: independent chains for the tensor pipe.
template <int MODE, bool PRE>
__device__ __forceinline__ void chunk_mma(const Slot &t0, const Slot &t1, uint32_t dig_addr, int (&acc1)[2][4],
                                          int (&acc16)[2][4], int (&accn1)[2][4], int (&accn16)[2][4]) {
  const uint32_t wA0[8] = {t0.alo.x, t0.alo.y, t0.alo.z, t0.alo.w, t0.ahi.x, t0.ahi.y, t0.ahi.z, t0.ahi.w};
  const uint32_t wB0[8] = {t0.blo.x, t0.blo.y, t0.blo.z, t0.blo.w, t0.bhi.x, t0.bhi.y, t0.bhi.z, t0.bhi.w};
  const uint32_t wA1[8] = {t1.alo.x, t1.alo.y, t1.alo.z, t1.alo.w, t1.ahi.x, t1.ahi.y, t1.ahi.z, t1.ahi.w};
  const uint32_t wB1[8] = {t1.blo.x, t1.blo.y, t1.blo.z, t1.blo.w, t1.bhi.x, t1.bhi.y, t1.bhi.z, t1.bhi.w};
  uint4 dpre[8];
  if (PRE) {
#pragma unroll
    for (int w = 0; w < 8; w++) dpre[w] = lds128(dig_addr + w * 512);
  }
#pragma unroll
  for (int w = 0; w < 8; w++) {
    const uint4 d = PRE ? dpre[w] : lds128(dig_addr + w * 512);
    const uint32_t a0 = wA0[w], b0 = wB0[w], a1 = wA1[w], b1 = wB1[w];
    const uint32_t a0t = a0 >> 2, b0t = b0 >> 2, a1t = a1 >> 2, b1t = b1 >> 2;
    // codes 4r (x1) and 4r+1 (x1) | codes 4r+2 (x16) and 4r+3 (x16)
    mma_u8s8(acc1[0], a0 & 0x03030303u, b0 & 0x03030303u, a0t & 0x03030303u, b0t & 0x03030303u, d.x, d.y);
    mma_u8s8(acc1[1], a1 & 0x03030303u, b1 & 0x03030303u, a1t & 0x03030303u, b1t & 0x03030303u, d.x, d.y);
    mma_u8s8(acc16[0], a0 & 0x30303030u, b0 & 0x30303030u, a0t & 0x30303030u, b0t & 0x30303030u, d.z, d.w);
    mma_u8s8(acc16[1], a1 & 0x30303030u, b1 & 0x30303030u, a1t & 0x30303030u, b1t & 0x30303030u, d.z, d.w);
    if (MODE != 0) {
      uint4 dn = d;
      if (MODE >= 2) dn = lds128(dig_addr + DIG + w * 512);
      // bit 2p of x & (x >> 1) is set iff code p == 3
      const uint32_t a0n = plane2<MODE>(a0), b0n = plane2<MODE>(b0), a0nt = plane2<MODE>(a0t), b0nt = plane2<MODE>(b0t);
      const uint32_t a1n = plane2<MODE>(a1), b1n = plane2<MODE>(b1), a1nt = plane2<MODE>(a1t), b1nt = plane2<MODE>(b1t);
      mma_u8s8(accn1[0], a0n & 0x01010101u, b0n & 0x01010101u, a0nt & 0x01010101u, b0nt & 0x01010101u, dn.x, dn.y);
      mma_u8s8(accn1[1], a1n & 0x01010101u, b1n & 0x01010101u, a1nt & 0x01010101u, b1nt & 0x01010101u, dn.x, dn.y);
      mma_u8s8(accn16[0], a0n & 0x10101010u, b0n & 0x10101010u, a0nt & 0x10101010u, b0nt & 0x10101010u, dn.z, dn.w);
      mma_u8s8(accn16[1], a1n & 0x10101010u, b1n & 0x10101010u, a1nt & 0x10101010u, b1nt & 0x10101010u, dn.z, dn.w);
    }
  }
}

// One 16-line sub-tile x one chunk with digits already in registers (STRUCT 0: sub-tiles in sequence,
// the slot is refilled as soon as its own MMAs are issued).
template <int MODE>
__device__ __forceinline__ void tile_mma(const Slot &sl, const uint4 (&b1)[8], uint32_t dig2_addr, int (&acc1)[4],
                                         int (&acc16)[4], int (&accn1)[4], int (&accn16)[4]) {
  const uint32_t wA[8] = {sl.alo.x, sl.alo.y, sl.alo.z, sl.alo.w, sl.ahi.x, sl.ahi.y, sl.ahi.z, sl.ahi.w};
  const uint32_t wB[8] = {sl.blo.x, sl.blo.y, sl.blo.z, sl.blo.w, sl.bhi.x, sl.bhi.y, sl.bhi.z, sl.bhi.w};
#pragma unroll
  for (int w = 0; w < 8; w++) {
    const uint32_t a = wA[w], bq = wB[w];
    const uint32_t at = a >> 2, bt = bq >> 2;
    mma_u8s8(acc1, a & 0x03030303u, bq & 0x03030303u, at & 0x03030303u, bt & 0x03030303u, b1[w].x, b1[w].y);
    mma_u8s8(acc16, a & 0x30303030u, bq & 0x30303030u, at & 0x30303030u, bt & 0x30303030u, b1[w].z, b1[w].w);
    if (MODE != 0) {
      uint4 d = b1[w];
      if (MODE >= 2) d = lds128(dig2_addr + w * 512);
      const uint32_t an = plane2<MODE>(a), bn = plane2<MODE>(bq);
      const uint32_t ant = plane2<MODE>(at), bnt = plane2<MODE>(bt);
      mma_u8s8(accn1, an & 0x01010101u, bn & 0x01010101u, ant & 0x01010101u, bnt & 0x01010101u, d.x, d.y);
      mma_u8s8(accn16, an & 0x10101010u, bn & 0x10101010u, ant & 0x10101010u, bnt & 0x10101010u, d.z, d.w);
    }
  }
}

// STRUCT 0: digits preloaded, sub-tiles in sequence, early refill.  1: digits just in time, both sub-tiles
// interleaved per word (4 independent MMA chains).  2: digits preloaded, interleaved.
template <int MODE, int CW, int R, int STRUCT>
__global__ void __launch_bounds__((CW + 1) * 32, 1) k_pmv(const Args a) {
  constexpr int GROUP = CW * 32;
  extern __shared__ __align__(128) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_base + STAGES * STAGE_BYTES;  // full[s] at +8s, empty[s] at +8(STAGES+s)

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
  constexpr bool two_dig = MODE >= 2;
  const uint32_t stage_tx = DIG + (two_dig ? DIG : 0);

  int stage = 0;
  uint32_t phase = 0;

  if (warp == CW) {
    // ============ producer warp: one bulk copy of the digit block(s) per chunk ============
    if (lane == 0) {
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int group = item / a.ksplit, ks = item - group * a.ksplit;
        const int c0 = ks * a.chunks_per_split;
        const int c1 = min(a.nchunks, c0 + a.chunks_per_split);
        for (int c = c0; c < c1; c++) {
          const uint32_t full = bar_base + 8 * stage, empty = bar_base + 8 * (STAGES + stage);
          mbar_wait(empty, phase ^ 1);
          mbar_expect_tx(full, stage_tx);
          const uint32_t dst = smem_base + stage * STAGE_BYTES;
          bulk_g2s(dst, a.dig1 + (int64_t)c * DIG, DIG, full);
          if (two_dig) bulk_g2s(dst + DIG, a.dig2 + (int64_t)c * DIG, DIG, full);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else {
    // ============ consumer warps: LDG.128 register ring -> IMMA ===========================
    const int g = lane >> 2, q = lane & 3;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
      const int group = item / a.ksplit, ks = item - group * a.ksplit;
      const int c0 = ks * a.chunks_per_split;
      const int c1 = min(a.nchunks, c0 + a.chunks_per_split);
      // line pointers of this lane: sub-tile u, lines g and g+8, pre-offset by the lane's 16 q bytes
      const uint8_t *pA[2], *pB[2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        int la = min(group * GROUP + warp * 32 + u * 16 + g, a.nlines - 1);
        int lb = min(group * GROUP + warp * 32 + u * 16 + g + 8, a.nlines - 1);
        const int pa = a.lines ? a.lines[la] : la, pb = a.lines ? a.lines[lb] : lb;
        pA[u] = a.P + (int64_t)pa * a.stride + 16 * q;
        pB[u] = a.P + (int64_t)pb * a.stride + 16 * q;
      }
      // does any of this warp's 32 lines hold a missing value?  (warp-uniform)
      bool tile_na = false;
      if (MODE == 3) {
        tile_na = true;  // the high-bit plane is populated everywhere
      } else if (MODE != 0) {
        if (a.na_flags) {
          int l = min(group * GROUP + warp * 32 + lane, a.nlines - 1);
          const int phys = a.lines ? a.lines[l] : l;
          tile_na = __any_sync(0xffffffffu, a.na_flags[phys] != 0);
        } else {
          tile_na = true;
        }
      }
      int acc1[2][4], acc16[2][4], accn1[2][4], accn16[2][4];
#pragma unroll
      for (int u = 0; u < 2; u++)
#pragma unroll
        for (int k = 0; k < 4; k++) acc1[u][k] = acc16[u][k] = accn1[u][k] = accn16[u][k] = 0;

      // register ring: ring[k][u] = fragment bytes of chunk (c0 + j*R + k), sub-tile u; R chunks resident,
      // each slot is refilled for chunk + R right after its MMAs are issued (2R - 1 slots in flight)
      Slot ring[R][2];
#pragma unroll
      for (int k = 0; k < R; k++) {
        ring[k][0] = ring[k][1] =
            Slot{make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
        if (c0 + k < c1) {
          slot_load(ring[k][0], pA[0], pB[0], (int64_t)(c0 + k) * SEG);
          slot_load(ring[k][1], pA[1], pB[1], (int64_t)(c0 + k) * SEG);
        }
      }

      for (int c = c0; c < c1; c += R) {
#pragma unroll
        for (int par = 0; par < R; par++) {
          if (par > 0 && c + par >= c1) break;
          const uint32_t full = bar_base + 8 * stage, empty = bar_base + 8 * (STAGES + stage);
          mbar_wait(full, phase);
          const uint32_t dbase = smem_base + stage * STAGE_BYTES + (g * 4 + q) * 16;
          const int64_t next = (int64_t)(c + par + R) * SEG;
          const bool more = (c + par + R) < c1;
          if (STRUCT == 0) {
            uint4 b1[8];
#pragma unroll
            for (int w = 0; w < 8; w++) b1[w] = lds128(dbase + w * 512);
#pragma unroll
            for (int u = 0; u < 2; u++) {
              if (MODE != 0 && tile_na)
                tile_mma<MODE>(ring[par][u], b1, dbase + DIG, acc1[u], acc16[u], accn1[u], accn16[u]);
              else
                tile_mma<0>(ring[par][u], b1, 0, acc1[u], acc16[u], accn1[u], accn16[u]);
              if (more) slot_load(ring[par][u], pA[u], pB[u], next);
            }
          } else {
            if (MODE != 0 && tile_na)
              chunk_mma<MODE, STRUCT == 2>(ring[par][0], ring[par][1], dbase, acc1, acc16, accn1, accn16);
            else
              chunk_mma<0, STRUCT == 2>(ring[par][0], ring[par][1], dbase, acc1, acc16, accn1, accn16);
            if (more) {
              slot_load(ring[par][0], pA[0], pB[0], next);
              slot_load(ring[par][1], pA[1], pB[1], next);
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(empty);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
      // ---- item epilogue: exact recombination of the x1 / x16 accumulators, 16 B stores ----
#pragma unroll
      for (int u = 0; u < 2; u++) {
#pragma unroll
        for (int hrow = 0; hrow < 2; hrow++) {
          const int row = group * GROUP + warp * 32 + u * 16 + g + 8 * hrow;
          // integer adds commute: the k-splits of a line accumulate in any order to the same exact sum
          unsigned long long *dst = reinterpret_cast<unsigned long long *>(a.part) + (int64_t)row * 16 + 2 * q;
          long long vx = (long long)acc1[u][2 * hrow] + (long long)(acc16[u][2 * hrow] >> 4);
          long long vy = (long long)acc1[u][2 * hrow + 1] + (long long)(acc16[u][2 * hrow + 1] >> 4);
          atomicAdd(dst, (unsigned long long)vx);
          atomicAdd(dst + 1, (unsigned long long)vy);
          if (MODE != 0) {
            long long nx = (long long)accn1[u][2 * hrow] + (long long)(accn16[u][2 * hrow] >> 4);
            long long ny = (long long)accn1[u][2 * hrow + 1] + (long long)(accn16[u][2 * hrow + 1] >> 4);
            atomicAdd(dst + 8, (unsigned long long)nx);
            atomicAdd(dst + 9, (unsigned long long)ny);
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// vector preparation: max |v| + finiteness, quantisation, digit layout, exact sums
// ---------------------------------------------------------------------------------------------

// mode 0: v0 = x                      (Xt.y, identity scaling handled in finish)
// mode 1: v0 = x / s, v1 = (c - 3) * x / s   (X.y with scaling)
// mode 2: v0 = x, v1 = second vector passed in the `center` slot   (two independent planes, bsg_pmv planes API)
__device__ __forceinline__ void make_vals(int mode, const double *x, const double *center, const double *scale, int k,
                                          double &v0, double &v1) {
  if (mode == 0) {
    v0 = x[k];
    v1 = 0;
  } else if (mode == 2) {
    v0 = x[k];
    v1 = center[k];
  } else {
    double z = x[k] / scale[k];
    v0 = z;
    v1 = (center[k] - 3.0) * z;
  }
}

__global__ void k_scal_reset(Scal *sc) {
  sc->maxabs[0] = sc->maxabs[1] = 0;
  sc->nonfinite = 0;
  sc->e[0] = sc->e[1] = 0;
  sc->Y = 0;
  sc->C = 0;
  sc->sum_hi = sc->sum_lo = 0;
}

__global__ void k_maxabs(int mode, const double *__restrict__ x, const double *__restrict__ center,
                         const double *__restrict__ scale, int len, Scal *sc) {
  double m0 = 0, m1 = 0;
  int bad = 0;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < len; k += gridDim.x * blockDim.x) {
    double v0, v1;
    make_vals(mode, x, center, scale, k, v0, v1);
    if (!isfinite(v0) || !isfinite(v1)) bad = 1;
    m0 = fmax(m0, fabs(v0));
    m1 = fmax(m1, fabs(v1));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    m0 = fmax(m0, __shfl_xor_sync(0xffffffffu, m0, o));
    m1 = fmax(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    // non-negative doubles order like their bit patterns
    atomicMax(reinterpret_cast<unsigned long long *>(&sc->maxabs[0]), (unsigned long long)__double_as_longlong(m0));
    atomicMax(reinterpret_cast<unsigned long long *>(&sc->maxabs[1]), (unsigned long long)__double_as_longlong(m1));
    if (bad) atomicOr(&sc->nonfinite, 1);
  }
}

// e = 60 - exponent(maxabs) - headroom_bits, so that |sum of <= 2^headroom quantised values| < 2^60
__global__ void k_pick_exp(Scal *sc, int headroom_bits) {
  for (int p = 0; p < 2; p++) {
    double m = sc->maxabs[p];
    int ex = 0;
    if (m > 0 && isfinite(m)) {
      frexp(m, &ex);
      sc->e[p] = 60 - ex - headroom_bits;
    } else {
      sc->e[p] = 0;
    }
  }
}

// Q[idx ? idx[k] : k] (+)= rint(v * 2^e).  With idx the destination is pre-zeroed and duplicates add
// up in integers (order independent) -- the scatter side of `ind.row` / `ind.col` multisets.
__global__ void k_quantise(int mode, const double *__restrict__ x, const double *__restrict__ center,
                           const double *__restrict__ scale, int len, const int *__restrict__ idx, const Scal *sc,
                           long long *__restrict__ Q0, long long *__restrict__ Q1) {
  const int e0 = sc->e[0], e1 = sc->e[1];
  const bool bad = sc->nonfinite != 0;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < len; k += gridDim.x * blockDim.x) {
    double v0, v1;
    make_vals(mode, x, center, scale, k, v0, v1);
    long long q0 = bad ? 0 : __double2ll_rn(scalbn(v0, e0));
    long long q1 = (bad || !Q1) ? 0 : __double2ll_rn(scalbn(v1, e1));
    if (idx) {
      atomicAdd(reinterpret_cast<unsigned long long *>(Q0 + idx[k]), (unsigned long long)q0);
      if (Q1) atomicAdd(reinterpret_cast<unsigned long long *>(Q1 + idx[k]), (unsigned long long)q1);
    } else {
      Q0[k] = q0;
      if (Q1) Q1[k] = q1;
    }
  }
}

// digits: one thread per 16-byte unit (chunk, w, s, q) -> 16 int8 digits of slice s for the 16 codes of
// word w of lane q (bytes 16q + 4w of the chunk for w < 4, bytes 64 + 16q + 4(w-4) for w >= 4), i.e. codes
// t = (w < 4 ? 64 q + 16 w : 256 + 64 q + 16 (w - 4)) + 4 r + c, stored at byte c*4 + r  (see tile_stage).
__global__ void k_digits(const long long *__restrict__ Q, int len, int nchunks, uint8_t *__restrict__ dig) {
  int64_t total = (int64_t)nchunks * 256;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    int chunk = (int)(t >> 8), unit = (int)(t & 255);
    int q = unit & 3, s = (unit >> 2) & 7, w = unit >> 5;
    uint32_t out[4] = {0, 0, 0, 0};
#pragma unroll
    for (int c = 0; c < 4; c++) {
#pragma unroll
      for (int r = 0; r < 4; r++) {
        int64_t k = (int64_t)chunk * CODES + (w < 4 ? 64 * q + 16 * w : 256 + 64 * q + 16 * (w - 4)) + 4 * r + c;
        long long v = k < len ? Q[k] : 0;
        // signed base-256 digit s: peel s digits
        int d = 0;
        for (int i = 0; i <= s; i++) {
          d = (int)(signed char)(v & 0xFF);
          v = (v - d) >> 8;
        }
        out[c] |= (uint32_t)(d & 0xFF) << (8 * r);
      }
    }
    reinterpret_cast<uint4 *>(dig)[t] = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// e = 60 - exponent(maxabs) - headroom_bits  ->  |sum of <= 2^hb quantised values| < 2^60
__device__ __forceinline__ int pick_e(double m, int hb) {
  int ex = 0;
  if (m > 0 && isfinite(m)) {
    frexp(m, &ex);
    return 60 - ex - hb;
  }
  return 0;
}

// Fused preparation, direct (identity index) path -- pass 1: max |v0|, max |v1|, finiteness and, for X.y with
// scaling, the per-block partials of C = sum_k c_k z_k.  Fixed grid of SUMCZ_BLOCKS blocks.
__global__ void k_prep1(int mode, const double *__restrict__ x, const double *__restrict__ center,
                        const double *__restrict__ scale, int len, int hb, Scal *sc) {
  __shared__ double sh[32];
  double m0 = 0, m1 = 0, cz = 0;
  int bad = 0;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < len; k += gridDim.x * blockDim.x) {
    double v0, v1;
    make_vals(mode, x, center, scale, k, v0, v1);
    if (!isfinite(v0) || !isfinite(v1)) bad = 1;
    m0 = fmax(m0, fabs(v0));
    m1 = fmax(m1, fabs(v1));
    if (mode == 1) cz += center[k] * v0;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    m0 = fmax(m0, __shfl_xor_sync(0xffffffffu, m0, o));
    m1 = fmax(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
    cz += __shfl_xor_sync(0xffffffffu, cz, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(reinterpret_cast<unsigned long long *>(&sc->maxabs[0]), (unsigned long long)__double_as_longlong(m0));
    atomicMax(reinterpret_cast<unsigned long long *>(&sc->maxabs[1]), (unsigned long long)__double_as_longlong(m1));
    if (bad) atomicOr(&sc->nonfinite, 1);
    sh[threadIdx.x >> 5] = cz;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += sh[w];
    sc->cpart[blockIdx.x] = t;
    if (blockIdx.x == 0) sc->hb = hb;
  }
}

// pass 2: quantise and lay out the digits straight from the input vector (no Q array).  One thread per
// 16-byte unit (chunk, w, s, q) as in k_digits; with two planes the thread writes both units.  want_sum: the
// slice-0 threads also accumulate the exact integer sum of Q (Xt.y needs Y = sum y).
__global__ void k_prep2(int mode, const double *__restrict__ x, const double *__restrict__ center,
                        const double *__restrict__ scale, int len, int nchunks, Scal *sc, uint8_t *__restrict__ dig1,
                        uint8_t *__restrict__ dig2, int want_sum, long long *__restrict__ qout = nullptr) {
  const int e0 = pick_e(sc->maxabs[0], sc->hb), e1 = pick_e(sc->maxabs[1], sc->hb);
  const bool bad = sc->nonfinite != 0;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    sc->e[0] = e0;
    sc->e[1] = e1;
  }
  long long hi = 0, lo = 0;
  // 2^e as a double when it is a normal number (always, unless the vector is denormal-small or huge)
  const bool fast0 = e0 > -1000 && e0 < 1000, fast1 = e1 > -1000 && e1 < 1000;
  const double f0 = fast0 ? scalbn(1.0, e0) : 0.0, f1 = fast1 ? scalbn(1.0, e1) : 0.0;
  int64_t total = (int64_t)nchunks * 32;  // (chunk, w, q)
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int chunk = (int)(t >> 5), wq = (int)(t & 31);
    const int q = wq & 3, w = wq >> 2;
    uint32_t o1[8][4], o2[8][4];
#pragma unroll
    for (int sl = 0; sl < 8; sl++)
#pragma unroll
      for (int c = 0; c < 4; c++) o1[sl][c] = o2[sl][c] = 0;
#pragma unroll
    for (int c = 0; c < 4; c++) {
#pragma unroll
      for (int r = 0; r < 4; r++) {
        int64_t k = (int64_t)chunk * CODES + (w < 4 ? 64 * q + 16 * w : 256 + 64 * q + 16 * (w - 4)) + 4 * r + c;
        long long qa = 0, qb = 0;
        if (k < len && !bad) {
          double v0, v1;
          make_vals(mode, x, center, scale, (int)k, v0, v1);
          qa = __double2ll_rn(fast0 ? v0 * f0 : scalbn(v0, e0));
          if (dig2) qb = __double2ll_rn(fast1 ? v1 * f1 : scalbn(v1, e1));
        }
        if (want_sum) {
          hi += qa >> 32;
          lo += (long long)(unsigned int)(qa & 0xFFFFFFFFll);
        }
        if (qout && k < len) qout[k] = qa;  // the quantised raw-plane vector (sparse missing-value correction)
#pragma unroll
        for (int sl = 0; sl < 8; sl++) {
          int d = (int)(signed char)(qa & 0xFF);
          qa = (qa - d) >> 8;
          o1[sl][c] |= (uint32_t)(d & 0xFF) << (8 * r);
          if (dig2) {
            int d2 = (int)(signed char)(qb & 0xFF);
            qb = (qb - d2) >> 8;
            o2[sl][c] |= (uint32_t)(d2 & 0xFF) << (8 * r);
          }
        }
      }
    }
#pragma unroll
    for (int sl = 0; sl < 8; sl++) {
      const int64_t unit = (int64_t)chunk * 256 + (w * 8 + sl) * 4 + q;
      reinterpret_cast<uint4 *>(dig1)[unit] = make_uint4(o1[sl][0], o1[sl][1], o1[sl][2], o1[sl][3]);
      if (dig2) reinterpret_cast<uint4 *>(dig2)[unit] = make_uint4(o2[sl][0], o2[sl][1], o2[sl][2], o2[sl][3]);
    }
  }
  if (want_sum) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      hi += __shfl_xor_sync(0xffffffffu, hi, o);
      lo += __shfl_xor_sync(0xffffffffu, lo, o);
    }
    if ((threadIdx.x & 31) == 0 && (hi | lo)) {
      atomicAdd(reinterpret_cast<unsigned long long *>(&sc->sum_hi), (unsigned long long)hi);
      atomicAdd(reinterpret_cast<unsigned long long *>(&sc->sum_lo), (unsigned long long)lo);
    }
  }
}

// exact integer sum of Q (split in 32-bit halves, integer atomics: order independent); Y is formed from
// (sum_hi, sum_lo) in the finish kernel.
__global__ void k_sum_q(const long long *__restrict__ Q, int len, Scal *sc) {
  long long hi = 0, lo = 0;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < len; k += gridDim.x * blockDim.x) {
    long long v = Q[k];
    hi += v >> 32;
    lo += (long long)(unsigned int)(v & 0xFFFFFFFFll);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    hi += __shfl_xor_sync(0xffffffffu, hi, o);
    lo += __shfl_xor_sync(0xffffffffu, lo, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(reinterpret_cast<unsigned long long *>(&sc->sum_hi), (unsigned long long)hi);
    atomicAdd(reinterpret_cast<unsigned long long *>(&sc->sum_lo), (unsigned long long)lo);
  }
}

// C = sum_k c_k * (x_k / s_k): per-block partial sums with a fixed-shape tree, written to cpart[block];
// the finish kernel adds the SUMCZ_BLOCKS partials in index order -> deterministic.
__global__ void k_sum_cz(const double *__restrict__ x, const double *__restrict__ center,
                         const double *__restrict__ scale, int len, double *__restrict__ cpart) {
  __shared__ double sh[32];
  double acc = 0;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < len; k += gridDim.x * blockDim.x)
    acc += center[k] * (x[k] / scale[k]);
#pragma unroll
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += sh[w];
    cpart[blockIdx.x] = t;
  }
}

// Xt.y:  out_j = ((R - 3N) - c_j (Y - N)) / s_j        (bedAccScaled semantics, src/bed-acc.h:98-111)
__global__ void k_finish_cprod(const long long *__restrict__ part, int ksplit, int64_t nlines_pad, int nlines,
                               const Scal *sc, const double *__restrict__ center, const double *__restrict__ scale,
                               int use_na, double *__restrict__ out) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nlines) return;
  if (sc->nonfinite) {
    out[j] = nan("");
    return;
  }
  const int e = sc->e[0];
  double G = combine8(part, j, 1, use_na ? -3 : 0, e);  // R - 3N, exact
  double N = use_na ? combine8(part, j, 0, 1, e) : 0.0;
  if (center) {
    const double Y = scalbn((double)sc->sum_hi, 32 - e) + scalbn((double)sc->sum_lo, -e);
    out[j] = (G - center[j] * (Y - N)) / scale[j];
  } else {
    out[j] = G;
  }
}

// X.y:  full_l = R + Nw - C   with Nw the NA-plane sum against w = (c - 3) z;  without scaling
// full_l = R - 3 N.   out[i] = full[gather[i]].
__global__ void k_finish_prod(const long long *__restrict__ part, int ksplit, int64_t nlines_pad, int nlines,
                              const Scal *sc, int has_scaling, int use_na, double *__restrict__ full) {
  int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlines) return;
  full[l] = finish_prod_value(part, l, sc, has_scaling, use_na);
}

// planes API:  full_l = cR * R_l + cP * P_l + add0,  R = raw-plane sum against vector 1 (exponent e[0]),
// P = second-plane sum against vector 2 (e[1]);  optional second output fullB_l = cRb * R_l + cPb * P_l.
__global__ void k_finish_planes(const long long *__restrict__ part, int nlines, const Scal *sc, int have_p, int p_same,
                                double cR, double cP, double add0, double *__restrict__ full, double cRb, double cPb,
                                double *__restrict__ fullB) {
  int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlines) return;
  if (sc->nonfinite) {
    full[l] = nan("");
    if (fullB) fullB[l] = nan("");
    return;
  }
  const double R = combine8(part, l, 1, 0, sc->e[0]);
  const double P = have_p ? combine8(part, l, 0, 1, sc->e[p_same ? 0 : 1]) : 0.0;
  full[l] = (cR * R + cP * P) + add0;
  if (fullB) fullB[l] = cRb * R + cPb * P;
}

__global__ void k_gather(const double *__restrict__ full, const int *__restrict__ idx, int len, double *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < len) out[i] = full[idx[i]];
}

// CUDA-event timing of k_pmv on the launching stream: a ring of event pairs, read back lazily
constexpr int EV_POOL = 128;
static cudaEvent_t g_ev0[EV_POOL], g_ev1[EV_POOL];
static bool g_ev_ready = false;
static bool g_timing = false;
static int g_ev_n = 0;  // launches recorded since the last reset (ring overwrites beyond EV_POOL)

static int launch_cap(int64_t work, int block, int cap) {
  int64_t g = (work + block - 1) / block;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

static int launch_cap_pub_impl(int64_t work) { return launch_cap(work, 256, 148 * 16); }

static int hb_bits(int maxmult) {
  int b = 0;
  while ((1 << b) < maxmult) b++;
  return b;
}

// shared launcher of the tensor-pipe kernel + scratch sizing
static int run_pmv(bsg_view *v, const uint8_t *P, int64_t stride, int L, const int *lines, int nlines,
                   const uint8_t *dig1, const uint8_t *dig2, const uint8_t *na_flags, int use_na, Args *out_args,
                   cudaStream_t s, bool plane_hi = false) {
  // variant: BSG_PMV_VARIANT = "<consumer warps>x<ring chunks>" (tuning knob; default chosen from measurements)
  static int var_cw = 0, var_r = 0, var_s = 0;
  if (!var_cw) {
    var_cw = 11;  // measured on B200 (profiles/r01_pmv_variants.md): 11x3s1 1.066 ms, 11x2s0 1.075, 15x2s1 1.078
    var_r = 3;
    var_s = 1;
    const char *ev = getenv("BSG_PMV_VARIANT");
    int cw = 0, r = 0, st = 0;
    if (ev && sscanf(ev, "%dx%ds%d", &cw, &r, &st) >= 2) {
      if ((cw == 11 || cw == 15) && (r == 2 || r == 3) && st >= 0 && st <= 2) {
        var_cw = cw;
        var_r = r;
        var_s = st;
      }
    }
  }
  const int GROUP = var_cw * 32;
  Args a;
  a.P = P;
  a.stride = stride;
  a.lines = lines;
  a.nlines = nlines;
  a.nlines_pad = (int)round_up(nlines, GROUP);
  a.nchunks = (int)(round_up(((int64_t)L + 3) / 4, SEG) / SEG);
  int ngroups = a.nlines_pad / GROUP;
  int target_items = 24 * 148;
  int ks = (target_items + ngroups - 1) / ngroups;
  int ks_max = std::max(1, a.nchunks / 16);
  int ks_min = (a.nchunks + MAX_CHUNKS_PER_ITEM - 1) / MAX_CHUNKS_PER_ITEM;
  ks = std::min(ks, ks_max);
  ks = std::max(ks, ks_min);
  ks = std::max(ks, 1);
  a.chunks_per_split = (a.nchunks + ks - 1) / ks;
  a.ksplit = (a.nchunks + a.chunks_per_split - 1) / a.chunks_per_split;
  a.dig1 = dig1;
  a.dig2 = dig2;
  a.na_flags = na_flags;
  a.use_na = use_na;
  BSG_TRY(v->s_part.ensure((size_t)a.nlines_pad * 16 * sizeof(long long)));
  a.part = v->s_part.as<long long>();
  BSG_CUDA(cudaMemsetAsync(a.part, 0, (size_t)a.nlines_pad * 16 * sizeof(long long), s));
  const int mode = plane_hi ? 3 : (!use_na ? 0 : (dig2 ? 2 : 1));
  if (plane_hi && !dig2) return fail(BSG_ERR_ARG, "high-bit plane needs its own digits");
  void (*kern)(const Args) = nullptr;
#define PMV_PICK(CWv, Rv, Sv)                                                                   \
  if (var_cw == CWv && var_r == Rv && var_s == Sv)                                              \
    kern = mode == 0 ? k_pmv<0, CWv, Rv, Sv>                                                    \
                     : (mode == 1 ? k_pmv<1, CWv, Rv, Sv> : (mode == 2 ? k_pmv<2, CWv, Rv, Sv> : k_pmv<3, CWv, Rv, Sv>));
  PMV_PICK(11, 2, 0)
  PMV_PICK(11, 2, 1)
  PMV_PICK(11, 2, 2)
  PMV_PICK(11, 3, 0)
  PMV_PICK(11, 3, 1)
  PMV_PICK(15, 2, 1)
#undef PMV_PICK
  if (!kern) return fail(BSG_ERR_ARG, "unknown k_pmv variant");
  BSG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  int nsm = 148;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, v->h->device);
  int nitems = ngroups * a.ksplit;
  int grid = std::min(nitems, nsm);
  if (g_timing) cudaEventRecord(g_ev0[g_ev_n % EV_POOL], s);
  kern<<<grid, (var_cw + 1) * 32, SMEM_BYTES, s>>>(a);
  if (g_timing) {
    cudaEventRecord(g_ev1[g_ev_n % EV_POOL], s);
    g_ev_n++;
  }
  count_launch();
  BSG_CUDA(cudaGetLastError());
  *out_args = a;
  return BSG_OK;
}

}  // namespace pmv

// =============================================================================================
// k_pmvT: X.y straight from the SNP-major copy (no sample-major copy needed).
//
// The contraction now runs ACROSS lines (SNPs) while the bytes of a line run along samples, so the IMMA k index
// has to be assembled from 4 different lines.  A CTA owns TBYTES sample-bytes (4 TBYTES samples) of every line,
// 64 bytes per warp, and walks a range of lines 32 at a time: every warp stages its own 32 x 64 B strip with
// cp.async into a private multi-stage ring (no block barrier in the loop), laid out so the fragment reads are
// conflict free; every thread reads one 32-bit word from 4 consecutive lines and transposes the 4 x 4 bytes with
// 8 PRMTs.  A transposed word holds, for 4 lines, the
// byte of 4 samples: masking the 2-bit fields gives the A fragments of 4 IMMAs (sample 4b + c, c = 0..3; field c
// enters as 4^c x code, removed by an exact shift in the epilogue).  B = the 8 signed base-256 digits
// of the quantised vector, 32 lines per step, laid out [step][slice][32] so a B register is one aligned word.
// Per warp and step: 16 IMMAs over 32 lines x 64 bytes; accumulators: 4 (byte) x 4 (field) x 4 registers.
// Missing values / the high-bit plane: k_pmvT2 below does the raw and the flag plane in one pass.
// =============================================================================================
namespace pmvt {
using namespace pmv;
constexpr int TLINES = 32, TBYTES = 512, TWARPS = 8, TSTAGES = 6;
constexpr int WSTAGE_BYTES = TLINES * 64;                  // one warp's strip of a step: 32 lines x 64 B
constexpr int TSMEM = TWARPS * TSTAGES * WSTAGE_BYTES;     // 96 KB -> 2 CTAs per SM
constexpr int MAX_LINES_PER_ITEM = 1 << 16;                // 64 x 3 x 128 x 2^16 < 2^31; value bytes: 254 x 128 x 2^16 < 2^31

struct TArgs {
  const uint8_t *P;
  int64_t stride;
  const int *lines;   // physical line of selected column t (null = identity)
  int nlines;
  const uint8_t *dig; // [steps][8][32]
  int lines_per_split, ksplit, nblocks, n;
  long long *part;    // [n][16]
};

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// BYTES: the lines hold one value byte per sample (centi-dosage FBM handles, bsg_pmv8.cu) instead of four 2-bit codes; a
// transposed word is then directly the A fragment of ONE IMMA (4 lines x 1 sample), no field masks, no 4^c to undo.
template <int PLANE, bool LINES, bool BYTES = false>
__global__ void __launch_bounds__(TWARPS * 32, 2) k_pmvT(const TArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, q = lane & 3;
  const int blk = blockIdx.x % a.nblocks, ks = blockIdx.x / a.nblocks;
  const int64_t byte0 = (int64_t)blk * TBYTES + 64 * warp;  // this warp's 64 sample-bytes of every line
  const int l0 = ks * a.lines_per_split, l1 = min(a.nlines, l0 + a.lines_per_split);
  const int nsteps = (l1 - l0 + TLINES - 1) / TLINES;
  // Every warp runs its own cp.async pipeline over its own strip (no block-level barrier in the loop):
  // TSTAGES stages of 32 lines x 64 B.  Word (row = 16 hf + 4 qq + r, column wc = 8 sl + gg) of a stage lives at
  // word offset ((((r 2 + hf) 2 + sl) 4 + qq) 8 + gg): the 32 lanes of one fragment read (fixed r, hf, sl) hit 32
  // consecutive words, and a 16-byte granule (4 consecutive gg of one row) stays contiguous for cp.async.
  const uint32_t wbase = smem_u32(smem) + warp * (TSTAGES * WSTAGE_BYTES);

  // loader role of the lane: rows 8 i + (lane >> 2), granule lane & 3.  Out-of-range rows / byte columns are
  // clamped to valid memory instead of predicated: their digits are zero, resp. their samples are never stored.
  const int lrow = lane >> 2, lch = lane & 3;
  const int64_t colb = (byte0 + 16 * lch < a.stride) ? byte0 + 16 * lch : 0;
  uint32_t dst_off[4];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int row = 8 * i + lrow;
    const int hf = row >> 4, qq = (row >> 2) & 3, r = row & 3, sl = lch >> 1, hc = lch & 1;
    dst_off[i] = (uint32_t)((((((r * 2 + hf) * 2 + sl) * 4 + qq) * 8) + 4 * hc) * 4);
  }
  const int full_steps = (l1 - l0) / TLINES;  // steps whose 32 lines all exist
  const int64_t stride8 = 8 * a.stride;
  // general issue: any step, clamped rows, optional line list
  auto issue = [&](int step, int stage) {
    const uint32_t dst = wbase + stage * WSTAGE_BYTES;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int t = min(l0 + step * TLINES + 8 * i + lrow, l1 - 1);
      const int phys = LINES ? a.lines[t] : t;
      cp_async16(dst + dst_off[i], a.P + colb + (int64_t)phys * a.stride, 16);
    }
  };

  int acc[4][4][4];
#pragma unroll
  for (int j = 0; j < 4; j++)
#pragma unroll
    for (int c = 0; c < 4; c++)
#pragma unroll
      for (int k = 0; k < 4; k++) acc[j][c][k] = 0;

#pragma unroll
  for (int st = 0; st < TSTAGES - 1; st++) {
    if (st < nsteps) issue(st, st);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  // B registers of the step: slice g, lines 4q..4q+3 and 16+4q..16+4q+3
  const uint8_t *dg = a.dig + (int64_t)(l0 / TLINES) * 256 + g * 32 + 4 * q;
  uint32_t nb0 = 0, nb1 = 0;
  if (nsteps > 0) {
    nb0 = *reinterpret_cast<const uint32_t *>(dg);
    nb1 = *reinterpret_cast<const uint32_t *>(dg + 16);
  }
  const uint32_t rd_base = wbase + (uint32_t)((q * 8 + g) * 4);  // + ((r 2 + hf) 2 + sl) * 128 bytes

  auto compute = [&](uint32_t st_base, uint32_t b0, uint32_t b1) {
    uint32_t W[2][2][4];  // [slot g / g+8][lines lo / hi][byte]
#pragma unroll
    for (int sl = 0; sl < 2; sl++)
#pragma unroll
      for (int hf = 0; hf < 2; hf++) {
        const uint32_t ad = st_base + (hf * 2 + sl) * 128;
        const uint32_t x0 = lds32(ad), x1 = lds32(ad + 512), x2 = lds32(ad + 1024), x3 = lds32(ad + 1536);
        const uint32_t t0 = prmt(x0, x1, 0x5140), t1 = prmt(x2, x3, 0x5140);
        const uint32_t t2 = prmt(x0, x1, 0x7362), t3 = prmt(x2, x3, 0x7362);
        W[sl][hf][0] = prmt(t0, t1, 0x5410);
        W[sl][hf][1] = prmt(t0, t1, 0x7632);
        W[sl][hf][2] = prmt(t2, t3, 0x5410);
        W[sl][hf][3] = prmt(t2, t3, 0x7632);
      }
#pragma unroll
    for (int j = 0; j < 4; j++) {
      uint32_t wa = W[0][0][j], wb = W[1][0][j], wc2 = W[0][1][j], wd = W[1][1][j];
      if (PLANE == 1) {  // missing-value flag at the low bit of each 2-bit field
        wa = wa & (wa >> 1) & 0x55555555u;
        wb = wb & (wb >> 1) & 0x55555555u;
        wc2 = wc2 & (wc2 >> 1) & 0x55555555u;
        wd = wd & (wd >> 1) & 0x55555555u;
      } else if (PLANE == 2) {  // high bit of the code (codes 2 and 3), for the sums of squares
        wa = (wa >> 1) & 0x55555555u;
        wb = (wb >> 1) & 0x55555555u;
        wc2 = (wc2 >> 1) & 0x55555555u;
        wd = (wd >> 1) & 0x55555555u;
      }
      if (BYTES) {
        mma_u8s8(acc[j][0], wa, wb, wc2, wd, b0, b1);
        continue;
      }
      // field c of every byte enters as 4^c x code (exact, undone in the epilogue): no shifts in the loop
      mma_u8s8(acc[j][0], wa & 0x03030303u, wb & 0x03030303u, wc2 & 0x03030303u, wd & 0x03030303u, b0, b1);
      mma_u8s8(acc[j][1], wa & 0x0C0C0C0Cu, wb & 0x0C0C0C0Cu, wc2 & 0x0C0C0C0Cu, wd & 0x0C0C0C0Cu, b0, b1);
      mma_u8s8(acc[j][2], wa & 0x30303030u, wb & 0x30303030u, wc2 & 0x30303030u, wd & 0x30303030u, b0, b1);
      mma_u8s8(acc[j][3], wa & 0xC0C0C0C0u, wb & 0xC0C0C0C0u, wc2 & 0xC0C0C0C0u, wd & 0xC0C0C0C0u, b0, b1);
    }
  };

  int step = 0;
  uint32_t rd_stage = 0, wr_stage = (TSTAGES - 1) * WSTAGE_BYTES;  // byte offsets of the stage read / refilled
  const uint8_t *dgn = dg + 256;
  // main loop (identity line order): the refilled step is entirely in range -> running pointers, no branches
  if (!LINES) {
    const int main_end = min(nsteps, full_steps - (TSTAGES - 1));
    const uint8_t *psrc = a.P + colb + (int64_t)(l0 + (TSTAGES - 1) * TLINES + lrow) * a.stride;
    for (; step < main_end; step++) {
      asm volatile("cp.async.wait_group %0;" ::"n"(TSTAGES - 2) : "memory");
      __syncwarp();
      {
        const uint32_t dst = wbase + wr_stage;
        cp_async16(dst + dst_off[0], psrc, 16);
        cp_async16(dst + dst_off[1], psrc + stride8, 16);
        cp_async16(dst + dst_off[2], psrc + 2 * stride8, 16);
        cp_async16(dst + dst_off[3], psrc + 3 * stride8, 16);
        asm volatile("cp.async.commit_group;" ::: "memory");
        psrc += 4 * stride8;
      }
      const uint32_t b0 = nb0, b1 = nb1;
      nb0 = *reinterpret_cast<const uint32_t *>(dgn);  // main_end < nsteps: the next step exists
      nb1 = *reinterpret_cast<const uint32_t *>(dgn + 16);
      dgn += 256;
      compute(rd_base + rd_stage, b0, b1);
      rd_stage = rd_stage + WSTAGE_BYTES == TSTAGES * WSTAGE_BYTES ? 0 : rd_stage + WSTAGE_BYTES;
      wr_stage = wr_stage + WSTAGE_BYTES == TSTAGES * WSTAGE_BYTES ? 0 : wr_stage + WSTAGE_BYTES;
    }
  }
  for (; step < nsteps; step++) {
    asm volatile("cp.async.wait_group %0;" ::"n"(TSTAGES - 2) : "memory");
    __syncwarp();
    {
      const int nxt = step + TSTAGES - 1;
      if (nxt < nsteps) issue(nxt, (int)(wr_stage / WSTAGE_BYTES));
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    const uint32_t b0 = nb0, b1 = nb1;
    if (step + 1 < nsteps) {
      nb0 = *reinterpret_cast<const uint32_t *>(dgn);
      nb1 = *reinterpret_cast<const uint32_t *>(dgn + 16);
      dgn += 256;
    }
    compute(rd_base + rd_stage, b0, b1);
    rd_stage = rd_stage + WSTAGE_BYTES == TSTAGES * WSTAGE_BYTES ? 0 : rd_stage + WSTAGE_BYTES;
    wr_stage = wr_stage + WSTAGE_BYTES == TSTAGES * WSTAGE_BYTES ? 0 : wr_stage + WSTAGE_BYTES;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  // epilogue: D rows = samples (slot g / g + 8), D columns = slices 2q, 2q + 1
#pragma unroll
  for (int j = 0; j < 4; j++)
#pragma unroll
    for (int c = 0; c < (BYTES ? 1 : 4); c++)
#pragma unroll
      for (int sl = 0; sl < 2; sl++) {
        const int64_t sample = BYTES ? byte0 + 4 * (8 * sl + g) + j : 4 * (byte0 + 4 * (8 * sl + g) + j) + c;
        if (sample < a.n) {
          unsigned long long *dst = reinterpret_cast<unsigned long long *>(a.part) + sample * 16 + (PLANE ? 8 : 0) + 2 * q;
          long long v0 = acc[j][c][2 * sl], v1 = acc[j][c][2 * sl + 1];
          v0 >>= 2 * c;
          v1 >>= 2 * c;
          if (v0) atomicAdd(dst, (unsigned long long)v0);
          if (v1) atomicAdd(dst + 1, (unsigned long long)v1);
        }
      }
}

// Two planes in one pass: the raw codes against `dig` and a flag plane (PL 1 = missing value, 2 = high bit)
// against `dig2`.  Same scheme as k_pmvT with 32-byte strips per warp, so the two accumulator sets (2 x 32
// registers) fit: rows g / g + 8 of an IMMA are bytes u and u + 2 of the lane's word column.
constexpr int W2STAGE_BYTES = TLINES * 32;                 // 1 KB per warp and stage
constexpr int T2BYTES = TWARPS * 32;                       // sample-bytes of a line per CTA
constexpr int T2SMEM = TWARPS * TSTAGES * W2STAGE_BYTES;   // 48 KB

template <int PL, bool LINES>
__global__ void __launch_bounds__(TWARPS * 32, 2) k_pmvT2(const TArgs a, const uint8_t *__restrict__ dig2) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, q = lane & 3;
  const int blk = blockIdx.x % a.nblocks, ks = blockIdx.x / a.nblocks;
  const int64_t byte0 = (int64_t)blk * T2BYTES + 32 * warp;
  const int l0 = ks * a.lines_per_split, l1 = min(a.nlines, l0 + a.lines_per_split);
  const int nsteps = (l1 - l0 + TLINES - 1) / TLINES;
  const uint32_t wbase = smem_u32(smem) + warp * (TSTAGES * W2STAGE_BYTES);
  // loader role: rows 16 i + (lane >> 1), granule lane & 1; stage layout: word (row = 16 hf + 4 qq + r, column gg)
  // at word offset (((r 2 + hf) 4 + qq) 8 + gg)
  const int lrow = lane >> 1, lch = lane & 1;
  const int64_t colb = (byte0 + 16 * lch < a.stride) ? byte0 + 16 * lch : 0;
  uint32_t dst_off[2];
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const int row = 16 * i + lrow;
    const int hf = row >> 4, qq = (row >> 2) & 3, r = row & 3;
    dst_off[i] = (uint32_t)(((((r * 2 + hf) * 4 + qq) * 8) + 4 * lch) * 4);
  }
  const int full_steps = (l1 - l0) / TLINES;
  const int64_t stride16 = 16 * a.stride;
  auto issue = [&](int step, int stage) {
    const uint32_t dst = wbase + stage * W2STAGE_BYTES;
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int t = min(l0 + step * TLINES + 16 * i + lrow, l1 - 1);
      const int phys = LINES ? a.lines[t] : t;
      cp_async16(dst + dst_off[i], a.P + colb + (int64_t)phys * a.stride, 16);
    }
  };
  int acc[2][2][4][4];  // [plane][unit][field][fragment]
#pragma unroll
  for (int p = 0; p < 2; p++)
#pragma unroll
    for (int u = 0; u < 2; u++)
#pragma unroll
      for (int c = 0; c < 4; c++)
#pragma unroll
        for (int k = 0; k < 4; k++) acc[p][u][c][k] = 0;
#pragma unroll
  for (int st = 0; st < TSTAGES - 1; st++) {
    if (st < nsteps) issue(st, st);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  const int64_t doff = (int64_t)(l0 / TLINES) * 256 + g * 32 + 4 * q;
  const uint8_t *dg = a.dig + doff, *dp = dig2 + doff;
  uint32_t nb0 = 0, nb1 = 0, np0 = 0, np1 = 0;
  if (nsteps > 0) {
    nb0 = *reinterpret_cast<const uint32_t *>(dg);
    nb1 = *reinterpret_cast<const uint32_t *>(dg + 16);
    np0 = *reinterpret_cast<const uint32_t *>(dp);
    np1 = *reinterpret_cast<const uint32_t *>(dp + 16);
  }
  const uint32_t rd_base = wbase + (uint32_t)((q * 8 + g) * 4);

  auto compute = [&](uint32_t st_base, uint32_t b0, uint32_t b1, uint32_t p0, uint32_t p1) {
    uint32_t W[2][4];  // [lines lo / hi][byte]
#pragma unroll
    for (int hf = 0; hf < 2; hf++) {
      const uint32_t ad = st_base + hf * 128;
      const uint32_t x0 = lds32(ad), x1 = lds32(ad + 256), x2 = lds32(ad + 512), x3 = lds32(ad + 768);
      const uint32_t t0 = prmt(x0, x1, 0x5140), t1 = prmt(x2, x3, 0x5140);
      const uint32_t t2 = prmt(x0, x1, 0x7362), t3 = prmt(x2, x3, 0x7362);
      W[hf][0] = prmt(t0, t1, 0x5410);
      W[hf][1] = prmt(t0, t1, 0x7632);
      W[hf][2] = prmt(t2, t3, 0x5410);
      W[hf][3] = prmt(t2, t3, 0x7632);
    }
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const uint32_t wa = W[0][u], wb = W[0][u + 2], wc2 = W[1][u], wd = W[1][u + 2];
      mma_u8s8(acc[0][u][0], wa & 0x03030303u, wb & 0x03030303u, wc2 & 0x03030303u, wd & 0x03030303u, b0, b1);
      mma_u8s8(acc[0][u][1], wa & 0x0C0C0C0Cu, wb & 0x0C0C0C0Cu, wc2 & 0x0C0C0C0Cu, wd & 0x0C0C0C0Cu, b0, b1);
      mma_u8s8(acc[0][u][2], wa & 0x30303030u, wb & 0x30303030u, wc2 & 0x30303030u, wd & 0x30303030u, b0, b1);
      mma_u8s8(acc[0][u][3], wa & 0xC0C0C0C0u, wb & 0xC0C0C0C0u, wc2 & 0xC0C0C0C0u, wd & 0xC0C0C0C0u, b0, b1);
      // flag plane: one bit per field at the field's low bit
      const uint32_t fa = PL == 1 ? (wa & (wa >> 1)) : (wa >> 1), fb = PL == 1 ? (wb & (wb >> 1)) : (wb >> 1);
      const uint32_t fc = PL == 1 ? (wc2 & (wc2 >> 1)) : (wc2 >> 1), fd = PL == 1 ? (wd & (wd >> 1)) : (wd >> 1);
      mma_u8s8(acc[1][u][0], fa & 0x01010101u, fb & 0x01010101u, fc & 0x01010101u, fd & 0x01010101u, p0, p1);
      mma_u8s8(acc[1][u][1], fa & 0x04040404u, fb & 0x04040404u, fc & 0x04040404u, fd & 0x04040404u, p0, p1);
      mma_u8s8(acc[1][u][2], fa & 0x10101010u, fb & 0x10101010u, fc & 0x10101010u, fd & 0x10101010u, p0, p1);
      mma_u8s8(acc[1][u][3], fa & 0x40404040u, fb & 0x40404040u, fc & 0x40404040u, fd & 0x40404040u, p0, p1);
    }
  };

  int step = 0;
  uint32_t rd_stage = 0, wr_stage = (TSTAGES - 1) * W2STAGE_BYTES;
  int64_t dnext = 256;
  if (!LINES) {
    const int main_end = min(nsteps, full_steps - (TSTAGES - 1));
    const uint8_t *psrc = a.P + colb + (int64_t)(l0 + (TSTAGES - 1) * TLINES + lrow) * a.stride;
    for (; step < main_end; step++) {
      asm volatile("cp.async.wait_group %0;" ::"n"(TSTAGES - 2) : "memory");
      __syncwarp();
      {
        const uint32_t dst = wbase + wr_stage;
        cp_async16(dst + dst_off[0], psrc, 16);
        cp_async16(dst + dst_off[1], psrc + stride16, 16);
        asm volatile("cp.async.commit_group;" ::: "memory");
        psrc += 2 * stride16;
      }
      const uint32_t b0 = nb0, b1 = nb1, p0 = np0, p1 = np1;
      nb0 = *reinterpret_cast<const uint32_t *>(dg + dnext);
      nb1 = *reinterpret_cast<const uint32_t *>(dg + dnext + 16);
      np0 = *reinterpret_cast<const uint32_t *>(dp + dnext);
      np1 = *reinterpret_cast<const uint32_t *>(dp + dnext + 16);
      dnext += 256;
      compute(rd_base + rd_stage, b0, b1, p0, p1);
      rd_stage = rd_stage + W2STAGE_BYTES == TSTAGES * W2STAGE_BYTES ? 0 : rd_stage + W2STAGE_BYTES;
      wr_stage = wr_stage + W2STAGE_BYTES == TSTAGES * W2STAGE_BYTES ? 0 : wr_stage + W2STAGE_BYTES;
    }
  }
  for (; step < nsteps; step++) {
    asm volatile("cp.async.wait_group %0;" ::"n"(TSTAGES - 2) : "memory");
    __syncwarp();
    {
      const int nxt = step + TSTAGES - 1;
      if (nxt < nsteps) issue(nxt, (int)(wr_stage / W2STAGE_BYTES));
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    const uint32_t b0 = nb0, b1 = nb1, p0 = np0, p1 = np1;
    if (step + 1 < nsteps) {
      nb0 = *reinterpret_cast<const uint32_t *>(dg + dnext);
      nb1 = *reinterpret_cast<const uint32_t *>(dg + dnext + 16);
      np0 = *reinterpret_cast<const uint32_t *>(dp + dnext);
      np1 = *reinterpret_cast<const uint32_t *>(dp + dnext + 16);
      dnext += 256;
    }
    compute(rd_base + rd_stage, b0, b1, p0, p1);
    rd_stage = rd_stage + W2STAGE_BYTES == TSTAGES * W2STAGE_BYTES ? 0 : rd_stage + W2STAGE_BYTES;
    wr_stage = wr_stage + W2STAGE_BYTES == TSTAGES * W2STAGE_BYTES ? 0 : wr_stage + W2STAGE_BYTES;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
  for (int p = 0; p < 2; p++)
#pragma unroll
    for (int u = 0; u < 2; u++)
#pragma unroll
      for (int c = 0; c < 4; c++)
#pragma unroll
        for (int sl = 0; sl < 2; sl++) {
          const int64_t sample = 4 * (byte0 + 4 * g + u + 2 * sl) + c;
          if (sample < a.n) {
            unsigned long long *dst = reinterpret_cast<unsigned long long *>(a.part) + sample * 16 + 8 * p + 2 * q;
            long long v0 = acc[p][u][c][2 * sl], v1 = acc[p][u][c][2 * sl + 1];
            v0 >>= 2 * c;
            v1 >>= 2 * c;
            if (v0) atomicAdd(dst, (unsigned long long)v0);
            if (v1) atomicAdd(dst + 1, (unsigned long long)v1);
          }
        }
}

// digits of the quantised vector(s) in step order: dig[(t / 32) * 256 + slice * 32 + (t % 32)]
__global__ void k_quantT(int mode, const double *__restrict__ x, const double *__restrict__ center,
                         const double *__restrict__ scale, int len, int len_pad, const pmv::Scal *sc,
                         uint8_t *__restrict__ dig1, uint8_t *__restrict__ dig2, const int *__restrict__ lines = nullptr,
                         long long *__restrict__ qna_full = nullptr, int na_second = 0, pmv::Scal *pick = nullptr) {
  // pick: the exponents are derived here from the maxima k_prep1 left in *sc (and published for the finish kernels)
  const int e0 = pick ? pmv::pick_e(sc->maxabs[0], sc->hb) : sc->e[0], e1 = pick ? pmv::pick_e(sc->maxabs[1], sc->hb) : sc->e[1];
  if (pick && blockIdx.x == 0 && threadIdx.x == 0) {
    pick->e[0] = e0;
    pick->e[1] = e1;
  }
  const bool bad = sc->nonfinite != 0;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < len_pad; t += gridDim.x * blockDim.x) {
    long long q0 = 0, q1 = 0;
    if (t < len && !bad) {
      double v0, v1;
      pmv::make_vals(mode, x, center, scale, t, v0, v1);
      q0 = __double2ll_rn(scalbn(v0, e0));
      if (dig2 || na_second) q1 = __double2ll_rn(scalbn(v1, e1));
      if (qna_full)  // missing-value vector by physical line (duplicates of a column add up)
        atomicAdd(reinterpret_cast<unsigned long long *>(qna_full + (lines ? lines[t] : t)),
                  (unsigned long long)(na_second ? q1 : q0));
    }
    const int64_t base = (int64_t)(t >> 5) * 256 + (t & 31);
#pragma unroll
    for (int sl = 0; sl < 8; sl++) {
      int d = (int)(signed char)(q0 & 0xFF);
      q0 = (q0 - d) >> 8;
      dig1[base + sl * 32] = (uint8_t)d;
      if (dig2) {
        int d2 = (int)(signed char)(q1 & 0xFF);
        q1 = (q1 - d2) >> 8;
        dig2[base + sl * 32] = (uint8_t)d2;
      }
    }
  }
}

// ---- two vectors per pass (PCA projection, bsg_prod_and_rowsumssq) ---------------------------------------------------
// An IMMA always produces 8 columns; with the full 61-bit fixed point all 8 are digit slices of ONE vector.  For the K
// columns of a projection the vectors are quantised to 30 bits instead (4 signed base-256 digits, |Q| < 2^30 relative to
// the largest entry of the vector: ~1e-9 of the result, three orders inside the 1e-6 contract) and TWO vectors share a
// pass: columns 0..3 = vector 1, 4..7 = vector 2.  Same kernels, same bytes read, twice the vectors.
__global__ void k_pick_exp_pair(pmv::Scal *sc, int headroom_bits) {
  const int v = threadIdx.x >> 1, p = threadIdx.x & 1;  // 4 threads: (vector, plane)
  if (threadIdx.x >= 4) return;
  const double m = sc[v].maxabs[p];
  int ex = 0;
  if (m > 0 && isfinite(m)) {
    frexp(m, &ex);
    sc[v].e[p] = 30 - ex - headroom_bits;  // |Q| < 2^30 fits 4 signed base-256 digits (max 127 * (2^32 - 1) / 255)
  } else {
    sc[v].e[p] = 0;
  }
}

// dig[(t / 32) * 256 + slice * 32 + (t % 32)], slices 0..3 = vector 1, 4..7 = vector 2; dig2 = the (c - 3) z plane
__global__ void k_quantT_pair(int mode, const double *__restrict__ xa, const double *__restrict__ xb,
                              const double *__restrict__ center, const double *__restrict__ scale, int len, int len_pad,
                              const pmv::Scal *sc, uint8_t *__restrict__ dig1, uint8_t *__restrict__ dig2) {
  const int e0a = sc[0].e[0], e1a = sc[0].e[1], e0b = sc[1].e[0], e1b = sc[1].e[1];
  const bool bada = sc[0].nonfinite != 0, badb = sc[1].nonfinite != 0;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < len_pad; t += gridDim.x * blockDim.x) {
    long long q[2][2] = {{0, 0}, {0, 0}};  // [vector][plane]
    if (t < len) {
      double v0, v1;
      if (!bada) {
        pmv::make_vals(mode, xa, center, scale, t, v0, v1);
        q[0][0] = __double2ll_rn(scalbn(v0, e0a));
        if (dig2) q[0][1] = __double2ll_rn(scalbn(v1, e1a));
      }
      if (xb && !badb) {
        pmv::make_vals(mode, xb, center, scale, t, v0, v1);
        q[1][0] = __double2ll_rn(scalbn(v0, e0b));
        if (dig2) q[1][1] = __double2ll_rn(scalbn(v1, e1b));
      }
    }
    const int64_t base = (int64_t)(t >> 5) * 256 + (t & 31);
#pragma unroll
    for (int vv = 0; vv < 2; vv++)
#pragma unroll
      for (int sl = 0; sl < 4; sl++) {
        int d = (int)(signed char)(q[vv][0] & 0xFF);
        q[vv][0] = (q[vv][0] - d) >> 8;
        dig1[base + (4 * vv + sl) * 32] = (uint8_t)d;
        if (dig2) {
          int d2 = (int)(signed char)(q[vv][1] & 0xFF);
          q[vv][1] = (q[vv][1] - d2) >> 8;
          dig2[base + (4 * vv + sl) * 32] = (uint8_t)d2;
        }
      }
  }
}

// (raw-plane * c0 + NA-plane * c1) over the 4 slices of vector vv
__device__ __forceinline__ double combine4(const long long *__restrict__ part, int64_t line, int vv, int c0, int c1, int e) {
  const long long *p = part + line * 16 + 4 * vv;
  double acc = 0;
#pragma unroll
  for (int s = 3; s >= 0; s--) {
    long long v = 0;
    if (c0) v += c0 * p[s];
    if (c1) v += c1 * p[8 + s];
    acc += scalbn((double)v, 8 * s - e);
  }
  return acc;
}

__global__ void k_finish_prod_pair(const long long *__restrict__ part, int nlines, const pmv::Scal *sc, int has_scaling,
                                   int use_na, double *__restrict__ out1, double *__restrict__ out2) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlines) return;
#pragma unroll
  for (int vv = 0; vv < 2; vv++) {
    double *out = vv ? out2 : out1;
    if (!out) continue;
    double r;
    if (sc[vv].nonfinite) {
      r = nan("");
    } else if (has_scaling) {
      double C = 0;
      for (int b = 0; b < pmv::SUMCZ_BLOCKS; b++) C += sc[vv].cpart[b];
      const double R = combine4(part, l, vv, 1, 0, sc[vv].e[0]);
      const double Nw = use_na ? combine4(part, l, vv, 0, 1, sc[vv].e[1]) : 0.0;
      r = (R + Nw) - C;
    } else {
      r = combine4(part, l, vv, 1, use_na ? -3 : 0, sc[vv].e[0]);
    }
    out[l] = r;
  }
}

// Two vectors per pass through k_pmv (lines = SNP columns, vectors over the samples: multLinReg).  Digit layout of
// k_digits, slices 0..3 = 30-bit vector 1 (Qa), 4..7 = vector 2 (Qb).
__global__ void k_digits_pair(const long long *__restrict__ Qa, const long long *__restrict__ Qb, int len, int nchunks,
                              uint8_t *__restrict__ dig) {
  const int64_t total = (int64_t)nchunks * 256;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int chunk = (int)(t >> 8), unit = (int)(t & 255);
    const int q = unit & 3, s = (unit >> 2) & 7, w = unit >> 5;
    const long long *Q = s < 4 ? Qa : Qb;
    const int sd = s & 3;
    uint32_t out[4] = {0, 0, 0, 0};
#pragma unroll
    for (int c = 0; c < 4; c++) {
#pragma unroll
      for (int r = 0; r < 4; r++) {
        const int64_t k = (int64_t)chunk * pmv::CODES + (w < 4 ? 64 * q + 16 * w : 256 + 64 * q + 16 * (w - 4)) + 4 * r + c;
        long long v = (Q && k < len) ? Q[k] : 0;
        int d = 0;
        for (int i = 0; i <= sd; i++) {
          d = (int)(signed char)(v & 0xFF);
          v = (v - d) >> 8;
        }
        out[c] |= (uint32_t)(d & 0xFF) << (8 * r);
      }
    }
    reinterpret_cast<uint4 *>(dig)[t] = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// per vector vv:  out_l = cR R_l + cP P_l,  outB_l = cRb R_l + cPb P_l   (R raw-plane sum, P missing-value plane sum of
// the SAME vector: one digit block serves both planes)
struct PairCoef {
  double cR, cP, cRb, cPb;
  double *out, *outB;
};
__global__ void k_finish_planes_pair(const long long *__restrict__ part, int nlines, const pmv::Scal *sc, int have_p,
                                     PairCoef ca, PairCoef cb) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= nlines) return;
#pragma unroll
  for (int vv = 0; vv < 2; vv++) {
    const PairCoef &c = vv ? cb : ca;
    if (!c.out) continue;
    if (sc[vv].nonfinite) {
      c.out[l] = nan("");
      if (c.outB) c.outB[l] = nan("");
      continue;
    }
    const double R = combine4(part, l, vv, 1, 0, sc[vv].e[0]);
    const double P = have_p ? combine4(part, l, vv, 0, 1, sc[vv].e[0]) : 0.0;
    c.out[l] = c.cR * R + c.cP * P;
    if (c.outB) c.outB[l] = c.cRb * R + c.cPb * P;
  }
}
}  // namespace pmvt


static int launch_cap_pub(int64_t work) { return pmv::launch_cap_pub_impl(work); }

// =============================================================================================
// views
// =============================================================================================
static int dev_copy(void **dst, const void *src, size_t bytes, cudaStream_t s) {
  BSG_CUDA(cudaMalloc(dst, bytes ? bytes : 16));
  if (bytes) BSG_CUDA(cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, s));
  return BSG_OK;
}

static bool is_identity(const int *ind, int len, int limit) {
  if (!ind) return true;
  if (len != limit) return false;
  for (int i = 0; i < len; i++)
    if (ind[i] != i + 1) return false;
  return true;
}

static int max_mult(std::vector<int> z) {
  if (z.empty()) return 1;
  std::sort(z.begin(), z.end());
  int best = 1, run = 1;
  for (size_t i = 1; i < z.size(); i++) {
    run = (z[i] == z[i - 1]) ? run + 1 : 1;
    best = std::max(best, run);
  }
  return best;
}

}  // namespace bsg

using namespace bsg;

extern "C" {

int bsg_view_create(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                    const double *scale, bsg_view **out) {
  if (!h || !out) return fail(BSG_ERR_ARG, "null argument");
  *out = nullptr;
  if (!h->dosage) BSG_PACKED_ONLY(h, "The packed matrix-vector engine");
  BSG_TRY(bind_device(h));
  if (!ind_row) nr = h->n;
  if (!ind_col) nc = h->m;
  if (nr < 0 || nc < 0) return fail(BSG_ERR_ARG, "negative length");
  if ((center == nullptr) != (scale == nullptr)) return fail(BSG_ERR_ARG, "center and scale must be given together");
  bsg_view *v = new bsg_view();
  v->h = h;
  v->nr = nr;
  v->nc = nc;
  v->row_identity = is_identity(ind_row, nr, h->n);
  v->col_identity = is_identity(ind_col, nc, h->m);
  v->has_scaling = center != nullptr;
  if (center) {
    // center = 0, scale = 1 (the reference's defaults, R/bed-mult-vec.R:23-24): identity scaling, which takes
    // the path whose missing-value correction cancels exactly in integers
    bool ident = true;
    for (int j = 0; j < nc && ident; j++) ident = center[j] == 0.0 && scale[j] == 1.0;
    if (ident) v->has_scaling = 0;
  }
  // value bytes are 100 x the dosage: the scaling is always applied, as (100 c, 100 s), default (0, 100)
  std::vector<double> dos_c, dos_s;
  if (h->dosage) {
    v->has_scaling = 1;
    dos_c.assign(std::max(nc, 1), 0.0);
    dos_s.assign(std::max(nc, 1), 1.0);
    if (center) {
      std::copy(center, center + nc, dos_c.begin());
      std::copy(scale, scale + nc, dos_s.begin());
    }
    center = dos_c.data();
    scale = dos_s.data();
  }
  cudaStream_t s = h->stream;
  int rc = BSG_OK;
  std::vector<int> zr, zc, uniq, gat;
  if (!v->row_identity) {
    zr.resize(nr);
    for (int i = 0; i < nr && !rc; i++) {
      long long t = (long long)ind_row[i] - 1;
      if (t < 0 || t >= h->n) rc = fail(BSG_ERR_BOUNDS, "Tested subscript out of bounds (row %d not in 1..%d).", ind_row[i], h->n);
      zr[i] = (int)t;
    }
    if (!rc) {
      v->row_maxmult = max_mult(zr);
      uniq = zr;
      std::sort(uniq.begin(), uniq.end());
      uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
      gat.resize(nr);
      for (int i = 0; i < nr; i++) gat[i] = (int)(std::lower_bound(uniq.begin(), uniq.end(), zr[i]) - uniq.begin());
      v->nru = (int)uniq.size();
      rc = dev_copy((void **)&v->d_row, zr.data(), (size_t)nr * sizeof(int), s);
      if (!rc) rc = dev_copy((void **)&v->d_rows_unique, uniq.data(), uniq.size() * sizeof(int), s);
      if (!rc) rc = dev_copy((void **)&v->d_row_gather, gat.data(), (size_t)nr * sizeof(int), s);
    }
  } else {
    v->nru = h->n;
  }
  if (!rc && !v->col_identity) {
    zc.resize(nc);
    for (int j = 0; j < nc && !rc; j++) {
      long long t = (long long)ind_col[j] - 1;
      if (t < 0 || t >= h->m) rc = fail(BSG_ERR_BOUNDS, "Tested subscript out of bounds (column %d not in 1..%d).", ind_col[j], h->m);
      zc[j] = (int)t;
    }
    if (!rc) {
      v->col_maxmult = max_mult(zc);
      rc = dev_copy((void **)&v->d_col, zc.data(), (size_t)nc * sizeof(int), s);
    }
  }
  if (!rc && v->has_scaling) {
    rc = dev_copy((void **)&v->d_center, center, (size_t)nc * sizeof(double), s);
    if (!rc) rc = dev_copy((void **)&v->d_scale, scale, (size_t)nc * sizeof(double), s);
  }
  std::vector<int> na_pos;
  if (!rc && h->dosage) {
    rc = dosage_view_scaling(v, s);
    for (int j = 0; j < nc && !rc; j++)
      if (h->na_line[v->col_identity ? j : zc[j]] > 0) na_pos.push_back(j);
    v->n_na_pos = (int)na_pos.size();
    v->any_na = v->n_na_pos > 0;
    if (!rc && v->any_na) rc = dev_copy((void **)&v->d_na_pos, na_pos.data(), na_pos.size() * sizeof(int), s);
  }
  if (!rc) rc = v->s_scal.ensure(2 * sizeof(pmv::Scal));  // the second block serves the two-vectors-per-pass mode
  cudaError_t e = cudaStreamSynchronize(s);  // host vectors go out of scope
  if (!rc && e != cudaSuccess) rc = cuda_fail(e, "view upload");
  if (rc) {
    bsg_view_destroy(v);
    return rc;
  }
  *out = v;
  return BSG_OK;
}

void bsg_view_destroy(bsg_view *v) {
  if (!v) return;
  cudaSetDevice(v->h->device);
  cudaStreamSynchronize(v->h->stream);
  void *ptrs[] = {v->d_row, v->d_col, v->d_center, v->d_scale, v->d_rows_unique, v->d_row_gather, v->d_na_pos};
  for (void *p : ptrs)
    if (p) cudaFree(p);
  DevBuf *bufs[] = {&v->s_vec0, &v->s_vec1, &v->s_vec2, &v->s_q0, &v->s_q1, &v->s_dig1,
                    &v->s_dig2, &v->s_part, &v->s_scal, &v->s_full};
  for (DevBuf *b : bufs) b->release();
  delete v;
}

}  // extern "C"

__global__ void k_fill(double *x, int len, double v) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x) x[i] = v;
}

// device-vector forms on a centi-dosage view with a selected missing value: the whole output is NaN (bsgpu.h)
static int dosage_na_fill(bsg_view *v, double *out_dev, int len, cudaStream_t s) {
  if (!v->h->dosage || !v->any_na || len == 0) return BSG_OK;
  k_fill<<<std::min(1184, (len + 255) / 256), 256, 0, s>>>(out_dev, len, nan(""));
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

// t(X~) x : lines = SNP columns of copy A (value bytes on a centi-dosage handle), contraction over samples
static int cprodvec_dev(bsg_view *v, const double *x_dev, double *out_dev, cudaStream_t s) {
  if (!v || !x_dev || !out_dev) return fail(BSG_ERR_ARG, "null argument");
  bsg_bed *h = v->h;
  BSG_TRY(bind_device(h));
  if (v->nc == 0) return BSG_OK;
  using namespace pmv;
  Scal *sc = v->s_scal.as<Scal>();
  const int n = h->n;
  int nchunks = (int)((h->dosage ? h->raw_stride : h->strideA * 4) / CODES);
  BSG_TRY(v->s_q0.ensure((size_t)n * sizeof(long long)));
  BSG_TRY(v->s_dig1.ensure((size_t)nchunks * DIG));
  long long *Q = v->s_q0.as<long long>();
  const int hb = hb_bits(v->row_maxmult);
  // few missing values: the kernel runs in its no-missing mode and the N plane comes from the per-SNP lists
  const bool lists = !h->dosage && h->has_na && na_ell_ready(h);
  if (v->row_identity) {
    // direct path: memset + 2 kernels
    BSG_CUDA(cudaMemsetAsync(sc, 0, sizeof(Scal), s));
    k_prep1<<<SUMCZ_BLOCKS, 256, 0, s>>>(0, x_dev, nullptr, nullptr, v->nr, hb, sc);
    k_prep2<<<launch_cap((int64_t)nchunks * 32, 128, 1184), 128, 0, s>>>(0, x_dev, nullptr, nullptr, n, nchunks, sc,
                                                                          v->s_dig1.as<uint8_t>(), nullptr, 1,
                                                                          lists ? Q : nullptr);
    count_launch(2);
  } else {
    k_scal_reset<<<1, 1, 0, s>>>(sc);
    k_maxabs<<<launch_cap(v->nr, 256, 592), 256, 0, s>>>(0, x_dev, nullptr, nullptr, v->nr, sc);
    k_pick_exp<<<1, 1, 0, s>>>(sc, hb);
    BSG_CUDA(cudaMemsetAsync(Q, 0, (size_t)n * sizeof(long long), s));
    k_quantise<<<launch_cap(v->nr, 256, 592), 256, 0, s>>>(0, x_dev, nullptr, nullptr, v->nr, v->d_row, sc, Q, nullptr);
    k_digits<<<launch_cap((int64_t)nchunks * 256, 256, 1184), 256, 0, s>>>(Q, n, nchunks, v->s_dig1.as<uint8_t>());
    k_sum_q<<<launch_cap(n, 256, 296), 256, 0, s>>>(Q, n, sc);
    count_launch(6);
  }
  Args a;
  if (h->dosage)
    BSG_TRY(run_pmv8(v, v->s_dig1.as<uint8_t>(), &a, s));
  else
    BSG_TRY(run_pmv(v, h->A, h->strideA, n, v->d_col, v->nc, v->s_dig1.as<uint8_t>(), nullptr, h->naA,
                    lists ? 0 : h->has_na, &a, s));
  if (lists) BSG_TRY(na_ell_correction(h, 1, v->d_col, v->nc, Q, a.part, s));
  k_finish_cprod<<<(v->nc + 255) / 256, 256, 0, s>>>(a.part, a.ksplit, a.nlines_pad, v->nc, sc, v->d_center, v->d_scale,
                                                      h->has_na && !h->dosage, out_dev);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

extern "C" {

int bsg_view_cprodvec_dev(bsg_view *v, const double *x_dev, double *out_dev, void *stream) {
  // NULL = the legacy default stream (what the header documents and what torch's default stream is): work is then
  // ordered with the caller's kernels and collectives, not on the handle's private non-blocking stream
  cudaStream_t s = stream ? (cudaStream_t)stream : cudaStreamLegacy;
  BSG_TRY(cprodvec_dev(v, x_dev, out_dev, s));
  return dosage_na_fill(v, out_dev, v->nc, s);
}

// Launcher of k_pmvT: raw plane with `dig_raw`, then (plane != 0) the flag plane (1 = missing value, 2 = high bit)
// with `dig_plane`, both accumulating into part[n][16] (zeroed here).  Lines = the view's selected columns.
static int run_pmvT(bsg_view *v, const uint8_t *dig_raw, int plane, const uint8_t *dig_plane, long long **part_out,
                    cudaStream_t s) {
  using namespace pmv;
  using namespace pmvt;
  bsg_bed *h = v->h;
  const int n = h->n, nc = v->nc;
  const int nsteps = (nc + TLINES - 1) / TLINES;
  BSG_TRY(v->s_part.ensure((size_t)std::max(n, 1) * 16 * sizeof(long long)));
  long long *part = v->s_part.as<long long>();
  *part_out = part;
  BSG_CUDA(cudaMemsetAsync(part, 0, (size_t)n * 16 * sizeof(long long), s));
  if (nc == 0 || n == 0) return BSG_OK;
  TArgs a;
  a.P = h->dosage ? h->raw : h->A;
  a.stride = h->dosage ? h->raw_stride : h->strideA;
  a.lines = v->d_col;
  a.nlines = nc;
  a.n = n;
  a.part = part;
  if (h->dosage && plane) return fail(BSG_ERR_ARG, "value-byte lines have no flag plane");
  const int64_t nbytes = h->dosage ? (int64_t)n : ((int64_t)n + 3) / 4;
  a.nblocks = (int)((nbytes + TBYTES - 1) / TBYTES);
  int nsm = 148;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, h->device);
  // items = nblocks x ksplit CTAs, 2 resident per SM: fill whole waves (4 of them) so no tail wave runs nearly empty
  static int waves = 0;
  if (!waves) {
    const char *ev = getenv("BSG_PMVT_WAVES");
    waves = ev ? std::max(1, std::min(64, atoi(ev))) : 4;
  }
  // k-split: the grid (nblocks x ksplit CTAs, 2 resident per SM) should fill WHOLE waves -- 3.2 waves cost as much as 4
  // (measured on the configs[4] 1/8 shard: 238 blocks x 4 splits = 952 CTAs over 296 slots, 0.79 instead of 0.89 of the HBM
  // peak).  Among the admissible counts pick the one whose last wave is fullest, preferring >= `waves` waves.
  auto pick_ks = [&](int nblocks) {
    const int slots = 2 * nsm;
    const int lo = std::max(1, (nc + MAX_LINES_PER_ITEM - 1) / MAX_LINES_PER_ITEM);  // int32 accumulator head-room
    const int hi = std::max(lo, std::min(std::max(1, nsteps / 32), std::max(lo, (4 * waves * slots) / std::max(nblocks, 1))));
    static int force_ks = -1;
    if (force_ks < 0) {
      const char *ev = getenv("BSG_PMVT_KS");
      force_ks = ev ? std::max(0, atoi(ev)) : 0;
    }
    if (force_ks > 0) return std::max(lo, force_ks);
    int best = lo;
    double best_score = -1;
    for (int ks = lo; ks <= hi; ks++) {
      const double ctas = (double)nblocks * ks, nwav = ceil(ctas / slots);
      double score = ctas / (nwav * slots);             // occupancy of the waves
      // every split adds a pipeline ramp and n x 8 integer atomics: worth ~1000 lines of streaming (sweeps on the
      // configs[4] 1/8 shard and on configs[1], profiles/r02_results.md)
      const double lines = (double)nc / ks;
      score *= lines / (lines + 1000.0);
      if (nwav < waves) score *= 0.9 + 0.1 * nwav / waves;  // very few waves: tail imbalance shows
      if (score > best_score + 1e-9) {
        best_score = score;
        best = ks;
      }
    }
    return best;
  };
  int ks = pick_ks(a.nblocks);
  a.lines_per_split = (int)round_up((nc + ks - 1) / ks, TLINES);
  a.ksplit = (nc + a.lines_per_split - 1) / a.lines_per_split;
  static unsigned attr_done = 0;  // one bit per device: function attributes are per device
  if (!(attr_done >> (h->device & 31) & 1u)) {
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TSMEM));
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TSMEM));
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT<0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TSMEM));
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT<0, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TSMEM));
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT2<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2SMEM));
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT2<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2SMEM));
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT2<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2SMEM));
    BSG_CUDA(cudaFuncSetAttribute(k_pmvT2<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, T2SMEM));
    attr_done |= 1u << (h->device & 31);
  }
  const int thr = TWARPS * 32;
  const bool lines = a.lines != nullptr;
  a.dig = dig_raw;
  if (g_timing) cudaEventRecord(g_ev0[g_ev_n % EV_POOL], s);
  if (!plane) {
    const int grid = a.nblocks * a.ksplit;
    if (h->dosage && lines)
      k_pmvT<0, true, true><<<grid, thr, TSMEM, s>>>(a);
    else if (h->dosage)
      k_pmvT<0, false, true><<<grid, thr, TSMEM, s>>>(a);
    else if (lines)
      k_pmvT<0, true><<<grid, thr, TSMEM, s>>>(a);
    else
      k_pmvT<0, false><<<grid, thr, TSMEM, s>>>(a);
  } else {
    // both planes in one pass: 32-byte strips per warp, twice the sample blocks
    a.nblocks = (int)((nbytes + T2BYTES - 1) / T2BYTES);
    const int ks2 = pick_ks(a.nblocks);
    a.lines_per_split = (int)round_up((nc + ks2 - 1) / ks2, TLINES);
    a.ksplit = (nc + a.lines_per_split - 1) / a.lines_per_split;
    const int grid = a.nblocks * a.ksplit;
    if (plane == 1) {
      if (lines)
        k_pmvT2<1, true><<<grid, thr, T2SMEM, s>>>(a, dig_plane);
      else
        k_pmvT2<1, false><<<grid, thr, T2SMEM, s>>>(a, dig_plane);
    } else {
      if (lines)
        k_pmvT2<2, true><<<grid, thr, T2SMEM, s>>>(a, dig_plane);
      else
        k_pmvT2<2, false><<<grid, thr, T2SMEM, s>>>(a, dig_plane);
    }
  }
  if (g_timing) {
    cudaEventRecord(g_ev1[g_ev_n % EV_POOL], s);
    g_ev_n++;
  }
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

// digit blocks of one or two vectors over the selected columns, in k_pmvT's step order
static int prep_T(bsg_view *v, int mode, const double *x, const double *p1, const double *p2, bool two, cudaStream_t s,
                  long long *qna_full = nullptr, int na_second = 0) {
  using namespace pmv;
  using namespace pmvt;
  Scal *sc = v->s_scal.as<Scal>();
  const int nc = v->nc;
  const int nsteps = (nc + TLINES - 1) / TLINES;
  BSG_TRY(v->s_dig1.ensure((size_t)std::max(nsteps, 1) * 256));
  if (two) BSG_TRY(v->s_dig2.ensure((size_t)std::max(nsteps, 1) * 256));
  // memset + 2 kernels: maxima, finiteness and (mode 1) the block partials of C = sum c z in one pass over the vector,
  // then quantisation + digits with the exponents picked per block from the maxima
  BSG_CUDA(cudaMemsetAsync(sc, 0, sizeof(Scal), s));
  k_prep1<<<SUMCZ_BLOCKS, 256, 0, s>>>(mode, x, p1, p2, nc, 0, sc);
  k_quantT<<<launch_cap((int64_t)std::max(nsteps, 1) * TLINES, 256, 1184), 256, 0, s>>>(
      mode, x, p1, p2, nc, nsteps * TLINES, sc, v->s_dig1.as<uint8_t>(), two ? v->s_dig2.as<uint8_t>() : nullptr, v->d_col,
      qna_full, na_second, sc);
  count_launch(2);
  return BSG_OK;
}

// X~ x from the SNP-major copy alone (k_pmvT): lines = selected SNP columns in selection order (duplicates are
// just repeated lines), all n samples are produced and the requested rows gathered at the end.
static int prodvec_T(bsg_view *v, const double *x_dev, double *out_dev, cudaStream_t s, bsg_comm *comm) {
  using namespace pmv;
  bsg_bed *h = v->h;
  Scal *sc = v->s_scal.as<Scal>();
  const int n = h->n, nc = v->nc;
  const int mode = v->has_scaling ? 1 : 0;
  const bool na = h->has_na && !h->dosage;  // value bytes: missing values are marked after the product (bsg_pmv8.cu)
  const bool lists = na && na_ell_ready(h);  // few missing values: per-sample lists instead of the flag plane
  const bool two = v->has_scaling && na && !lists;
  long long *qna = nullptr;
  if (lists) {  // the missing-value vector ((c - 3) z with scaling, else y) by physical SNP
    BSG_TRY(v->s_q1.ensure((size_t)h->m * sizeof(long long)));
    qna = v->s_q1.as<long long>();
    BSG_CUDA(cudaMemsetAsync(qna, 0, (size_t)h->m * sizeof(long long), s));
  }
  BSG_TRY(prep_T(v, mode, x_dev, v->d_center, v->d_scale, two, s, qna, v->has_scaling ? 1 : 0));  // incl. the partials of C
  long long *part = nullptr;
  BSG_TRY(run_pmvT(v, v->s_dig1.as<uint8_t>(), (na && !lists) ? 1 : 0,
                   two ? v->s_dig2.as<uint8_t>() : v->s_dig1.as<uint8_t>(), &part, s));
  if (lists) BSG_TRY(na_ell_correction(h, 0, nullptr, n, qna, part, s));
  double *full = out_dev;
  if (!v->row_identity) {
    BSG_TRY(v->s_full.ensure((size_t)n * sizeof(double)));
    full = v->s_full.as<double>();
  }
  if (comm && v->row_identity)  // epilogue fused with the sum over the column shards (NVLink peer memory, bsg_comm.cu)
    return comm_finish_prod_allreduce(comm, part, n, sc, v->has_scaling, h->has_na, out_dev, s);
  if (n > 0) {
    k_finish_prod<<<(n + 255) / 256, 256, 0, s>>>(part, 1, n, n, sc, v->has_scaling, na, full);
    count_launch();
  }
  if (!v->row_identity && v->nr > 0) {
    k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(full, v->d_row, v->nr, out_dev);
    count_launch();
  }
  BSG_CUDA(cudaGetLastError());
  if (comm) return comm_allreduce_oneshot(comm, out_dev, v->nr, s);
  return BSG_OK;
}

// X~ [xa | xb] from the SNP-major copy in ONE pass over the matrix (two vectors, 4 + 4 digit slices; see k_quantT_pair).
// xb / outb may be null (odd count).  Outputs in the caller's row order.
static int prodvec_T_pair(bsg_view *v, const double *xa, const double *xb, double *outa, double *outb, cudaStream_t s) {
  using namespace pmv;
  using namespace pmvt;
  bsg_bed *h = v->h;
  Scal *sc = v->s_scal.as<Scal>();
  const int n = h->n, nc = v->nc;
  const int mode = v->has_scaling ? 1 : 0;
  const bool two = v->has_scaling && h->has_na;  // the NA plane has its own digits ((c - 3) z); else it reuses the raw ones
  const int nsteps = (nc + TLINES - 1) / TLINES;
  BSG_TRY(v->s_dig1.ensure((size_t)std::max(nsteps, 1) * 256));
  if (two) BSG_TRY(v->s_dig2.ensure((size_t)std::max(nsteps, 1) * 256));
  for (int vv = 0; vv < 2; vv++) {
    const double *x = vv ? xb : xa;
    k_scal_reset<<<1, 1, 0, s>>>(sc + vv);
    count_launch();
    if (!x) continue;
    k_maxabs<<<launch_cap(nc, 256, 592), 256, 0, s>>>(mode, x, v->d_center, v->d_scale, nc, sc + vv);
    if (v->has_scaling) k_sum_cz<<<SUMCZ_BLOCKS, 256, 0, s>>>(x, v->d_center, v->d_scale, nc, sc[vv].cpart);
    count_launch(v->has_scaling ? 2 : 1);
  }
  k_pick_exp_pair<<<1, 32, 0, s>>>(sc, 0);
  k_quantT_pair<<<launch_cap((int64_t)std::max(nsteps, 1) * TLINES, 256, 1184), 256, 0, s>>>(
      mode, xa, xb, v->d_center, v->d_scale, nc, nsteps * TLINES, sc, v->s_dig1.as<uint8_t>(),
      two ? v->s_dig2.as<uint8_t>() : nullptr);
  count_launch(2);
  long long *part = nullptr;
  BSG_TRY(run_pmvT(v, v->s_dig1.as<uint8_t>(), h->has_na ? 1 : 0, two ? v->s_dig2.as<uint8_t>() : v->s_dig1.as<uint8_t>(),
                   &part, s));
  double *fa = outa, *fb = outb;
  if (!v->row_identity) {
    BSG_TRY(v->s_full.ensure((size_t)n * 2 * sizeof(double)));
    fa = v->s_full.as<double>();
    fb = outb ? fa + n : nullptr;
  }
  if (n > 0) {
    k_finish_prod_pair<<<(n + 255) / 256, 256, 0, s>>>(part, n, sc, v->has_scaling, h->has_na, fa, fb);
    count_launch();
  }
  if (!v->row_identity && v->nr > 0) {
    k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(fa, v->d_row, v->nr, outa);
    if (outb) k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(fb, v->d_row, v->nr, outb);
    count_launch(outb ? 2 : 1);
  }
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

static int g_force_t = -1;  // 1: X-side products use the SNP-major kernel even when the sample-major copy is resident
static bool use_T(const bsg_bed *h) {
  if (g_force_t < 0) {
    const char *ev = getenv("BSG_PMVT");
    g_force_t = (ev && ev[0] == '1') ? 1 : 0;
  }
  // with missing values the fused SNP-major kernel (k_pmvT2, 1.68 ms at cfg2) is ahead of the sample-major
  // kernel's NA mode (1.81 ms); without, the sample-major kernel keeps a 1-3 % edge when its copy is resident
  return !h->B || g_force_t == 1 || h->has_na || h->dosage;
}

}  // extern "C"

// X~ x : lines = samples of copy B, contraction over SNP columns.  comm != null: the result is summed over the column
// shards of the communicator (every rank receives the full n-vector).
int bsg::view_prodvec_comm(bsg_view *v, const double *x_dev, double *out_dev, cudaStream_t s, bsg_comm *comm) {
  if (!v || !x_dev || !out_dev) return fail(BSG_ERR_ARG, "null argument");
  bsg_bed *h = v->h;
  BSG_TRY(bind_device(h));
  if (v->nr == 0) return BSG_OK;
  if (h->dosage && comm) return fail(BSG_ERR_ARG, "centi-dosage handles have no column-sharded form");
  if (use_T(h)) return prodvec_T(v, x_dev, out_dev, s, comm);  // transposing kernel over the SNP-major copy
  using namespace pmv;
  Scal *sc = v->s_scal.as<Scal>();
  const int m = h->m;
  int nchunks = (int)(h->strideB / SEG);
  const int mode = v->has_scaling ? 1 : 0;
  const bool two = v->has_scaling && h->has_na;
  BSG_TRY(v->s_q0.ensure((size_t)m * sizeof(long long)));
  BSG_TRY(v->s_dig1.ensure((size_t)nchunks * DIG));
  if (two) {
    BSG_TRY(v->s_q1.ensure((size_t)m * sizeof(long long)));
    BSG_TRY(v->s_dig2.ensure((size_t)nchunks * DIG));
  }
  long long *Q0 = v->s_q0.as<long long>();
  long long *Q1 = two ? v->s_q1.as<long long>() : nullptr;
  const int hb = hb_bits(v->col_maxmult);
  if (v->col_identity) {
    BSG_CUDA(cudaMemsetAsync(sc, 0, sizeof(Scal), s));
    k_prep1<<<SUMCZ_BLOCKS, 256, 0, s>>>(mode, x_dev, v->d_center, v->d_scale, v->nc, hb, sc);
    k_prep2<<<launch_cap((int64_t)nchunks * 32, 128, 1184), 128, 0, s>>>(
        mode, x_dev, v->d_center, v->d_scale, m, nchunks, sc, v->s_dig1.as<uint8_t>(),
        two ? v->s_dig2.as<uint8_t>() : nullptr, 0);
    count_launch(2);
  } else {
    k_scal_reset<<<1, 1, 0, s>>>(sc);
    k_maxabs<<<launch_cap(v->nc, 256, 592), 256, 0, s>>>(mode, x_dev, v->d_center, v->d_scale, v->nc, sc);
    k_pick_exp<<<1, 1, 0, s>>>(sc, hb);
    BSG_CUDA(cudaMemsetAsync(Q0, 0, (size_t)m * sizeof(long long), s));
    if (Q1) BSG_CUDA(cudaMemsetAsync(Q1, 0, (size_t)m * sizeof(long long), s));
    k_quantise<<<launch_cap(v->nc, 256, 592), 256, 0, s>>>(mode, x_dev, v->d_center, v->d_scale, v->nc, v->d_col, sc, Q0, Q1);
    k_digits<<<launch_cap((int64_t)nchunks * 256, 256, 1184), 256, 0, s>>>(Q0, m, nchunks, v->s_dig1.as<uint8_t>());
    if (Q1) k_digits<<<launch_cap((int64_t)nchunks * 256, 256, 1184), 256, 0, s>>>(Q1, m, nchunks, v->s_dig2.as<uint8_t>());
    if (v->has_scaling) k_sum_cz<<<SUMCZ_BLOCKS, 256, 0, s>>>(x_dev, v->d_center, v->d_scale, v->nc, sc->cpart);
    count_launch(5 + (Q1 ? 1 : 0) + (v->has_scaling ? 1 : 0));
  }
  Args a;
  const int nlines = v->row_identity ? h->n : v->nru;
  BSG_TRY(run_pmv(v, h->B, h->strideB, m, v->d_rows_unique, nlines, v->s_dig1.as<uint8_t>(),
                  two ? v->s_dig2.as<uint8_t>() : nullptr, h->naB, h->has_na, &a, s));
  double *full = out_dev;
  if (!v->row_identity) {
    BSG_TRY(v->s_full.ensure((size_t)nlines * sizeof(double)));
    full = v->s_full.as<double>();
  }
  if (comm && v->row_identity)
    return comm_finish_prod_allreduce(comm, a.part, nlines, sc, v->has_scaling, h->has_na, out_dev, s);
  k_finish_prod<<<(nlines + 255) / 256, 256, 0, s>>>(a.part, a.ksplit, a.nlines_pad, nlines, sc, v->has_scaling,
                                                     h->has_na, full);
  count_launch();
  if (!v->row_identity) {
    k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(full, v->d_row_gather, v->nr, out_dev);
    count_launch();
  }
  BSG_CUDA(cudaGetLastError());
  if (comm) return comm_allreduce_oneshot(comm, out_dev, v->nr, s);
  return BSG_OK;
}

extern "C" {

int bsg_view_prodvec_dev(bsg_view *v, const double *x_dev, double *out_dev, void *stream) {
  // NULL = the legacy default stream (what the header documents and what torch's default stream is): work is then
  // ordered with the caller's kernels and collectives, not on the handle's private non-blocking stream
  cudaStream_t s = stream ? (cudaStream_t)stream : cudaStreamLegacy;
  BSG_TRY(view_prodvec_comm(v, x_dev, out_dev, s, nullptr));
  return v->nr ? dosage_na_fill(v, out_dev, v->nr, s) : BSG_OK;
}

// host-vector front ends: H2D of x, the product, D2H of the result; non-finite input falls back to the
// accessor kernel, which propagates Inf / NaN exactly like the reference's table arithmetic.
static int view_host_call(bsg_view *v, const double *x, double *out, bool cprod) {
  if (!v || !x || !out) return fail(BSG_ERR_ARG, "null argument");
  bsg_bed *h = v->h;
  BSG_TRY(bind_device(h));
  cudaStream_t s = h->stream;
  const int nin = cprod ? v->nr : v->nc, nout = cprod ? v->nc : v->nr;
  BSG_TRY(v->s_vec0.ensure((size_t)std::max(nin, 1) * sizeof(double)));
  BSG_TRY(v->s_vec1.ensure((size_t)std::max(nout, 1) * sizeof(double)));
  double *dx = v->s_vec0.as<double>(), *dout = v->s_vec1.as<double>();
  BSG_CUDA(cudaMemcpyAsync(dx, x, (size_t)nin * sizeof(double), cudaMemcpyHostToDevice, s));
  BSG_TRY(cprod ? cprodvec_dev(v, dx, dout, s) : view_prodvec_comm(v, dx, dout, s, nullptr));
  if (h->dosage) BSG_TRY(dosage_mark_na(v, cprod, dout, s));
  int bad = 0;
  if (nout > 0)  // every product path (copy A or copy B) raises the flag on non-finite input
    BSG_CUDA(cudaMemcpyAsync(&bad, &v->s_scal.as<pmv::Scal>()->nonfinite, sizeof(int), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaMemcpyAsync(out, dout, (size_t)nout * sizeof(double), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaStreamSynchronize(s));
  if (bad && !h->dosage) {  // (a centi-dosage handle keeps the finish kernels' all-NaN output)
    BSG_TRY(cprod ? simple_cprodvec(h, v->d_row, v->nr, v->d_col, v->nc, v->d_center, v->d_scale, dx, dout, s)
                  : simple_prodvec(h, v->d_row, v->nr, v->d_col, v->nc, v->d_center, v->d_scale, dx, dout, s));
    BSG_CUDA(cudaMemcpyAsync(out, dout, (size_t)nout * sizeof(double), cudaMemcpyDeviceToHost, s));
    BSG_CUDA(cudaStreamSynchronize(s));
  }
  return BSG_OK;
}

int bsg_view_prodvec(bsg_view *v, const double *x, double *out) { return view_host_call(v, x, out, false); }
int bsg_view_cprodvec(bsg_view *v, const double *x, double *out) { return view_host_call(v, x, out, true); }

// The 9-argument drop-in calls (the .Call twins).  The reference rebuilds its accessor on every call
// (src/bed-prod-vec.cpp:22-23); here the accessor state lives in a view cached on the handle: it is
// reused while the index vectors are unchanged (compared by content), and only center / scale / x are
// re-uploaded, so a Lanczos loop calling through the old interface does no per-call allocation.
// Strided sample of (center, scale): every element when nc <= 2048, else 2048 evenly spaced ones of each + the last.  A
// different scaling differs (practically) everywhere, so address + length + this sample identify "the same vectors as in
// the previous call" -- what a Lanczos loop through the old interface passes ~1,000 times (R/autoSVD.R:216-218).
// It is OPT-IN (bsg_set_scaling_reuse(1) or BSG_SCALING_REUSE=1): a vector edited in place at a position the sample
// does not cover would go unnoticed, and the reference re-reads center / scale on every call.  Default: upload every call.
static int g_scaling_reuse = -1;
static void scaling_sample(const double *center, const double *scale, int nc, std::vector<double> &out) {
  out.clear();
  if (!center || !scale || nc <= 0) return;
  const int ns = std::min(nc, 2048);
  out.reserve(2 * (size_t)ns + 2);
  for (int t = 0; t < ns; t++) {
    const size_t j = (size_t)((int64_t)t * nc / ns);
    out.push_back(center[j]);
    out.push_back(scale[j]);
  }
  out.push_back(center[nc - 1]);
  out.push_back(scale[nc - 1]);
}

static int cached_view(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                       const double *scale, bsg_view **out) {
  if (!h) return fail(BSG_ERR_ARG, "null handle");
  if (!ind_row) nr = h->n;
  if (!ind_col) nc = h->m;
  if (nr < 0 || nc < 0) return fail(BSG_ERR_ARG, "negative length");
  if ((center == nullptr) != (scale == nullptr)) return fail(BSG_ERR_ARG, "center and scale must be given together");
  // the cached view must have device copies of center / scale to refresh (identity scaling keeps none)
  bool hit = h->cv != nullptr && h->cv->nr == nr && h->cv->nc == nc && (h->cv->d_center != nullptr) == (center != nullptr) &&
             (center == nullptr || h->cv->has_scaling != 0);
  if (hit) {
    hit = (ind_row == nullptr) == h->cv_row.empty() || (ind_row && (int)h->cv_row.size() == nr);
    if (hit && ind_row) hit = (int)h->cv_row.size() == nr && memcmp(h->cv_row.data(), ind_row, (size_t)nr * sizeof(int)) == 0;
    if (hit && !ind_row) hit = h->cv_row.empty();
    if (hit && ind_col) hit = (int)h->cv_col.size() == nc && memcmp(h->cv_col.data(), ind_col, (size_t)nc * sizeof(int)) == 0;
    if (hit && !ind_col) hit = h->cv_col.empty();
  }
  if (!hit) {
    if (h->cv) bsg_view_destroy(h->cv);
    h->cv = nullptr;
    bsg_view *v = nullptr;
    BSG_TRY(bsg_view_create(h, ind_row, nr, ind_col, nc, center, scale, &v));
    h->cv = v;
    h->cv_row.assign(ind_row ? ind_row : nullptr, ind_row ? ind_row + nr : nullptr);
    h->cv_col.assign(ind_col ? ind_col : nullptr, ind_col ? ind_col + nc : nullptr);
    h->cv_center_ptr = center;
    h->cv_scale_ptr = scale;
    scaling_sample(center, scale, nc, h->cv_scal_sample);
  } else if (center) {
    BSG_TRY(bind_device(h));
    if (g_scaling_reuse < 0) {
      const char *ev = getenv("BSG_SCALING_REUSE");
      g_scaling_reuse = (ev && ev[0] == '1') ? 1 : 0;
    }
    std::vector<double> smp;
    scaling_sample(center, scale, nc, smp);
    const bool same = g_scaling_reuse == 1 && center == h->cv_center_ptr && scale == h->cv_scale_ptr &&
                      smp.size() == h->cv_scal_sample.size() &&
                      memcmp(smp.data(), h->cv_scal_sample.data(), smp.size() * sizeof(double)) == 0;
    if (!same) {
      BSG_CUDA(cudaMemcpyAsync(h->cv->d_center, center, (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      BSG_CUDA(cudaMemcpyAsync(h->cv->d_scale, scale, (size_t)nc * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      if (h->dosage) BSG_TRY(dosage_view_scaling(h->cv, h->stream));
      h->cv_center_ptr = center;
      h->cv_scale_ptr = scale;
      h->cv_scal_sample.swap(smp);
    }
  }
  *out = h->cv;
  return BSG_OK;
}

int bsg_prodvec(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                const double *scale, const double *x, double *out) {
  bsg_view *v = nullptr;
  BSG_TRY(cached_view(h, ind_row, nr, ind_col, nc, center, scale, &v));
  return bsg_view_prodvec(v, x, out);
}

int bsg_cprodvec(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                 const double *scale, const double *x, double *out) {
  bsg_view *v = nullptr;
  BSG_TRY(cached_view(h, ind_row, nr, ind_col, nc, center, scale, &v));
  return bsg_view_cprodvec(v, x, out);
}

}  // extern "C"

// =============================================================================================
// planes API: the two integer plane sums of the tensor-pipe kernel against caller-chosen vectors.
//   dir 0: lines = samples (copy B), vectors run over the selected SNP columns   (X-side sums)
//   dir 1: lines = SNP columns (copy A), vectors run over the selected samples   (Xt-side sums)
//   R_l = sum_t code(l, t) x1[t]   (code 3 for a missing value)
//   P_l = sum_t plane(l, t) x2[t]  plane = missing-value flag (PLANE_NA) or high bit of the code (PLANE_HI)
// out = cR R + cP P + add0, outB = cRb R + cPb P (optional), both in the caller's index order.
// =============================================================================================
namespace bsg {
enum { PLANE_NONE = 0, PLANE_NA = 1, PLANE_HI = 2 };
struct PlaneOut {
  double cR, cP, add0;
  double *out;
  double cRb, cPb;
  double *outB;
};

static int view_planes_dev(bsg_view *v, int dir, const double *x1, const double *x2, int plane, const PlaneOut &o,
                           cudaStream_t s) {
  using namespace pmv;
  bsg_bed *h = v->h;
  if (plane == PLANE_NA && !h->has_na) plane = PLANE_NONE;
  const bool same = plane == PLANE_NA && x2 == x1;          // one digit block serves both planes
  const bool two = plane != PLANE_NONE && !same;
  Scal *sc = v->s_scal.as<Scal>();
  if (dir == 0 && use_T(h)) {
    // X-side sums from the SNP-major copy: raw-plane launch + flag-plane launch of k_pmvT
    BSG_TRY(prep_T(v, two ? 2 : 0, x1, x2, nullptr, two, s));
    long long *part = nullptr;
    BSG_TRY(run_pmvT(v, v->s_dig1.as<uint8_t>(), plane == PLANE_NONE ? 0 : (plane == PLANE_NA ? 1 : 2),
                     two ? v->s_dig2.as<uint8_t>() : v->s_dig1.as<uint8_t>(), &part, s));
    const int n = h->n;
    const bool gather = !v->row_identity;
    double *full = o.out, *fullB = o.outB;
    if (gather) {
      BSG_TRY(v->s_full.ensure((size_t)n * 2 * sizeof(double)));
      full = v->s_full.as<double>();
      fullB = o.outB ? full + n : nullptr;
    }
    k_finish_planes<<<(n + 255) / 256, 256, 0, s>>>(part, n, sc, plane != PLANE_NONE, same ? 1 : 0, o.cR, o.cP, o.add0, full,
                                                    o.cRb, o.cPb, fullB);
    count_launch();
    if (gather && v->nr > 0) {
      k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(full, v->d_row, v->nr, o.out);
      if (o.outB) k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(fullB, v->d_row, v->nr, o.outB);
      count_launch(o.outB ? 2 : 1);
    }
    BSG_CUDA(cudaGetLastError());
    return BSG_OK;
  }
  const int L = dir == 0 ? h->m : h->n;                      // contraction length in the staged copy
  const int len = dir == 0 ? v->nc : v->nr;                  // vector length (selection order)
  const int *idx = dir == 0 ? v->d_col : v->d_row;
  const bool ident = dir == 0 ? v->col_identity : v->row_identity;
  const int hb = hb_bits(dir == 0 ? v->col_maxmult : v->row_maxmult);
  const int64_t stride = dir == 0 ? h->strideB : h->strideA;
  const int nchunks = (int)(stride / SEG);
  const int mode = two ? 2 : 0;
  BSG_TRY(v->s_dig1.ensure((size_t)nchunks * DIG));
  if (two) BSG_TRY(v->s_dig2.ensure((size_t)nchunks * DIG));
  uint8_t *dig1 = v->s_dig1.as<uint8_t>(), *dig2 = two ? v->s_dig2.as<uint8_t>() : nullptr;
  if (ident) {
    BSG_CUDA(cudaMemsetAsync(sc, 0, sizeof(Scal), s));
    k_prep1<<<SUMCZ_BLOCKS, 256, 0, s>>>(mode, x1, x2, nullptr, len, hb, sc);
    k_prep2<<<launch_cap((int64_t)nchunks * 32, 128, 1184), 128, 0, s>>>(mode, x1, x2, nullptr, L, nchunks, sc, dig1, dig2, 0);
    count_launch(2);
  } else {
    BSG_TRY(v->s_q0.ensure((size_t)L * sizeof(long long)));
    long long *Q0 = v->s_q0.as<long long>(), *Q1 = nullptr;
    if (two) {
      BSG_TRY(v->s_q1.ensure((size_t)L * sizeof(long long)));
      Q1 = v->s_q1.as<long long>();
    }
    k_scal_reset<<<1, 1, 0, s>>>(sc);
    k_maxabs<<<launch_cap(len, 256, 592), 256, 0, s>>>(mode, x1, x2, nullptr, len, sc);
    k_pick_exp<<<1, 1, 0, s>>>(sc, hb);
    BSG_CUDA(cudaMemsetAsync(Q0, 0, (size_t)L * sizeof(long long), s));
    if (Q1) BSG_CUDA(cudaMemsetAsync(Q1, 0, (size_t)L * sizeof(long long), s));
    k_quantise<<<launch_cap(len, 256, 592), 256, 0, s>>>(mode, x1, x2, nullptr, len, idx, sc, Q0, Q1);
    k_digits<<<launch_cap((int64_t)nchunks * 256, 256, 1184), 256, 0, s>>>(Q0, L, nchunks, dig1);
    if (Q1) k_digits<<<launch_cap((int64_t)nchunks * 256, 256, 1184), 256, 0, s>>>(Q1, L, nchunks, dig2);
    count_launch(5 + (Q1 ? 1 : 0));
  }
  Args a;
  int nlines;
  if (dir == 0) {
    nlines = v->row_identity ? h->n : v->nru;
    BSG_TRY(run_pmv(v, h->B, stride, L, v->d_rows_unique, nlines, dig1, dig2, h->naB, plane != PLANE_NONE, &a, s,
                    plane == PLANE_HI));
  } else {
    nlines = v->nc;
    BSG_TRY(run_pmv(v, h->A, stride, L, v->d_col, nlines, dig1, dig2, h->naA, plane != PLANE_NONE, &a, s,
                    plane == PLANE_HI));
  }
  const bool gather = dir == 0 && !v->row_identity;
  double *full = o.out, *fullB = o.outB;
  if (gather) {
    BSG_TRY(v->s_full.ensure((size_t)nlines * 2 * sizeof(double)));
    full = v->s_full.as<double>();
    fullB = o.outB ? full + nlines : nullptr;
  }
  k_finish_planes<<<(nlines + 255) / 256, 256, 0, s>>>(a.part, nlines, sc, plane != PLANE_NONE, same ? 1 : 0, o.cR, o.cP,
                                                       o.add0, full, o.cRb, o.cPb, fullB);
  count_launch();
  if (gather) {
    k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(full, v->d_row_gather, v->nr, o.out);
    if (o.outB) k_gather<<<(v->nr + 255) / 256, 256, 0, s>>>(fullB, v->d_row_gather, v->nr, o.outB);
    count_launch(o.outB ? 2 : 1);
  }
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}


// Xt-side plane sums of TWO vectors in one pass over the SNP-major copy (30-bit fixed point each, see k_pick_exp_pair):
// per vector R_l = sum_t code(l, t) x[t] and, with plane == PLANE_NA, N_l = sum_t [missing(l, t)] x[t].
static int view_planes_pair_dev(bsg_view *v, const double *xa, const double *xb, int plane, const pmvt::PairCoef &ca,
                                const pmvt::PairCoef &cb, cudaStream_t s) {
  using namespace pmv;
  bsg_bed *h = v->h;
  if (plane == PLANE_NA && !h->has_na) plane = PLANE_NONE;
  Scal *sc = v->s_scal.as<Scal>();
  const int L = h->n, len = v->nr;
  const int hb = hb_bits(v->row_maxmult);
  const int64_t stride = h->strideA;
  const int nchunks = (int)(stride / SEG);
  BSG_TRY(v->s_dig1.ensure((size_t)nchunks * DIG));
  BSG_TRY(v->s_q0.ensure((size_t)L * sizeof(long long)));
  BSG_TRY(v->s_q1.ensure((size_t)L * sizeof(long long)));
  uint8_t *dig1 = v->s_dig1.as<uint8_t>();
  long long *Q0 = v->s_q0.as<long long>(), *Q1 = v->s_q1.as<long long>();
  const int *idx = v->row_identity ? nullptr : v->d_row;
  k_scal_reset<<<1, 1, 0, s>>>(sc);
  k_scal_reset<<<1, 1, 0, s>>>(sc + 1);
  k_maxabs<<<launch_cap(len, 256, 592), 256, 0, s>>>(0, xa, nullptr, nullptr, len, sc);
  if (xb) k_maxabs<<<launch_cap(len, 256, 592), 256, 0, s>>>(0, xb, nullptr, nullptr, len, sc + 1);
  pmvt::k_pick_exp_pair<<<1, 32, 0, s>>>(sc, hb);
  if (idx) {
    BSG_CUDA(cudaMemsetAsync(Q0, 0, (size_t)L * sizeof(long long), s));
    BSG_CUDA(cudaMemsetAsync(Q1, 0, (size_t)L * sizeof(long long), s));
  }
  k_quantise<<<launch_cap(len, 256, 592), 256, 0, s>>>(0, xa, nullptr, nullptr, len, idx, sc, Q0, nullptr);
  if (xb) k_quantise<<<launch_cap(len, 256, 592), 256, 0, s>>>(0, xb, nullptr, nullptr, len, idx, sc + 1, Q1, nullptr);
  pmvt::k_digits_pair<<<launch_cap((int64_t)nchunks * 256, 256, 1184), 256, 0, s>>>(Q0, xb ? Q1 : nullptr, idx ? L : len, nchunks,
                                                                                  dig1);
  count_launch(6 + (xb ? 2 : 0));
  Args a;
  const int nlines = v->nc;
  BSG_TRY(run_pmv(v, h->A, stride, L, v->d_col, nlines, dig1, nullptr, h->naA, plane != PLANE_NONE, &a, s, false));
  pmvt::k_finish_planes_pair<<<(nlines + 255) / 256, 256, 0, s>>>(a.part, nlines, sc, plane != PLANE_NONE, ca, cb);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}

// per selected column: a = (1 - 2c)/s^2, w = 1/s^2, nv = (5 - 6c + c^2)/s^2 and block partials of T = sum c^2/s^2
__global__ void k_rss_weights(const double *__restrict__ center, const double *__restrict__ scale, int nc,
                              double *__restrict__ a, double *__restrict__ w, double *__restrict__ nv,
                              double *__restrict__ tpart) {
  __shared__ double sh[32];
  double t = 0;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nc; j += gridDim.x * blockDim.x) {
    const double c = center ? center[j] : 0.0, sc = scale ? scale[j] : 1.0;
    const double w0 = 1.0 / (sc * sc);
    w[j] = w0;
    a[j] = (1.0 - 2.0 * c) * w0;
    nv[j] = (5.0 - 6.0 * c + c * c) * w0;
    t += c * c * w0;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = t;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tt = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) tt += sh[k];
    tpart[blockIdx.x] = tt;
  }
}

__global__ void k_rss_final(int nr, const double *__restrict__ t1, const double *__restrict__ t2,
                            const double *__restrict__ tpart, int nparts, double *__restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nr) return;
  double T = 0;
  for (int k = 0; k < nparts; k++) T += tpart[k];
  out[i] = (t1[i] + (t2 ? t2[i] : 0.0)) + T;
}

__global__ void k_or_flag(const pmv::Scal *sc, int *flag) {
  if (sc->nonfinite) *flag = 1;
}

__global__ void k_square(const double *__restrict__ x, int64_t len, double *__restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = x[i] * x[i];
}

// t-scores of multLinReg (src/multLinReg.cpp:44-51) from exact column counts and the plane sums:
//   xySum = R - 3N,  ySum = Y - N(u),  yySum = YY - N(u^2);  tscores[j + nc k]
__global__ void k_tscores(int nc, int K, const int32_t *__restrict__ cnt4, const double *__restrict__ G,
                          const double *__restrict__ Nu, const double *__restrict__ Nuu, const double *__restrict__ Y,
                          const double *__restrict__ YY, double *__restrict__ out) {
  const int64_t total = (int64_t)nc * K;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(t % nc), k = (int)(t / nc);
    const int c1 = cnt4[4 * j + 1], c2 = cnt4[4 * j + 2];
    const int nona = cnt4[4 * j] + c1 + c2;
    const double xSum = (double)c1 + 2.0 * c2, xxSum = (double)c1 + 4.0 * c2;
    const double xySum = G[t];
    const double ySum = Y[k] - (Nu ? Nu[t] : 0.0), yySum = YY[k] - (Nuu ? Nuu[t] : 0.0);
    const double deno_x = xxSum - xSum * xSum / nona;
    const double num = xySum - xSum * ySum / nona;
    const double deno_y = yySum - ySum * ySum / nona;
    const double deno = deno_x * deno_y - num * num;
    out[t] = (deno == 0 || nona < 2) ? nan("") : num * sqrt((nona - 2) / deno);
  }
}

// work arrays of the two entry points below live on the handle (grow-only): no cudaMalloc / cudaFree per call
struct ProjScratch {
  bsg_bed *h;
  int next = 0;
  template <class T>
  int alloc(T **out, size_t count) {
    if (next >= 8) return fail(BSG_ERR_ARG, "projection scratch exhausted");
    DevBuf &b = h->w_proj[next++];
    BSG_TRY(b.ensure((count ? count : 1) * sizeof(T)));
    *out = b.as<T>();
    return BSG_OK;
  }
};

// bed_row_counts_cpp (src/bed-fun.cpp:72-98) from three linear functionals of the all-ones vector over the selected
// columns: R = c1 + 2 c2 + 3 c3 (raw codes), N = c3 (missing flag), H = c2 + c3 (high bit).  Sums of exactly
// representable integers: the counts are exact.
__global__ void k_counts_from_planes(int nr, int nc, const double *__restrict__ R, const double *__restrict__ N,
                                     const double *__restrict__ H, int32_t *__restrict__ out4) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nr) return;
  const long long r = llrint(R[i]), c3 = llrint(N[i]), hh = llrint(H[i]);
  const long long c2 = hh - c3, c1 = r - 2 * c2 - 3 * c3;
  out4[4 * i + 0] = (int32_t)(nc - c1 - c2 - c3);
  out4[4 * i + 1] = (int32_t)c1;
  out4[4 * i + 2] = (int32_t)c2;
  out4[4 * i + 3] = (int32_t)c3;
}

int row_counts_planes(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, int32_t *d_out4) {
  bsg_view *v = nullptr;
  BSG_TRY(cached_view(h, ind_row, nr, ind_col, nc, nullptr, nullptr, &v));
  cudaStream_t s = h->stream;
  ProjScratch mem{h};
  double *ones = nullptr, *rows = nullptr;
  BSG_TRY(mem.alloc(&ones, (size_t)v->nc));
  BSG_TRY(mem.alloc(&rows, 3 * (size_t)v->nr));
  double *R = rows, *N = rows + v->nr, *H = rows + 2 * (size_t)v->nr;
  k_fill<<<launch_cap_pub(v->nc), 256, 0, s>>>(ones, v->nc, 1.0);
  count_launch();
  PlaneOut o1{1.0, 0.0, 0.0, R, 0.0, 1.0, N};
  BSG_TRY(view_planes_dev(v, 0, ones, ones, PLANE_NA, o1, s));
  PlaneOut o2{0.0, 1.0, 0.0, H, 0, 0, nullptr};
  BSG_TRY(view_planes_dev(v, 0, ones, ones, PLANE_HI, o2, s));
  k_counts_from_planes<<<(v->nr + 255) / 256, 256, 0, s>>>(v->nr, v->nc, R, N, H, d_out4);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  return BSG_OK;
}
}  // namespace bsg

extern "C" {

// prod_and_rowSumsSq (src/bed-fun.cpp:103-133): XV = X~ V (nr x K) and rowSumsSq_i = sum_j X~_ij^2.
// XV is K applications of the X.y engine; the sums of squares come from two more passes over the same bytes:
//   sum_j [x present] ((x - c)/s)^2 = R(a) + 2 H(w) - N(nv) + T
// with x^2 = code + 2 hi - 5 na for the staged codes, a = (1 - 2c)/s^2, w = 1/s^2, nv = (5 - 6c + c^2)/s^2,
// T = sum_j c^2/s^2, and R / H / N the raw, high-bit and missing-value plane sums.
int bsg_prod_and_rowsumssq(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                           const double *scale, const double *V, int K, double *XV, double *rowSumsSq) {
  if (!h || !XV || !rowSumsSq || (!V && K > 0)) return fail(BSG_ERR_ARG, "null argument");
  if (!center || !scale) return fail(BSG_ERR_DIM, "Incompatibility between dimensions.");
  if (K < 0) return fail(BSG_ERR_ARG, "negative length");
  if (!h->dosage) BSG_PACKED_ONLY(h, "prod_and_rowSumsSq");
  bsg_view *v = nullptr;
  BSG_TRY(cached_view(h, ind_row, nr, ind_col, nc, center, scale, &v));
  if (h->dosage) return dosage_prod_and_rowsumssq(v, V, K, XV, rowSumsSq);  // prod_and_rowSumsSq2 (bsg_pmv8.cu)
  nr = v->nr;
  nc = v->nc;
  cudaStream_t s = h->stream;
  ProjScratch mem{h};
  const int NP = 64;
  double *dV = nullptr, *dXV = nullptr, *d_rows = nullptr, *d_cols = nullptr;
  BSG_TRY(mem.alloc(&dV, (size_t)nc * K));
  BSG_TRY(mem.alloc(&dXV, (size_t)nr * K));
  BSG_TRY(mem.alloc(&d_rows, 3 * (size_t)nr));            // rowSumsSq | pass 1 | pass 2
  BSG_TRY(mem.alloc(&d_cols, 3 * (size_t)nc + NP + 2));   // a | w | nv | partials of T | flag
  double *d_rs = d_rows;
  if (nr == 0) return BSG_OK;
  if (nc == 0) {
    BSG_CUDA(cudaStreamSynchronize(s));
    memset(XV, 0, (size_t)nr * K * sizeof(double));
    memset(rowSumsSq, 0, (size_t)nr * sizeof(double));
    return BSG_OK;
  }
  // V (nc x K doubles, configs[1]: 40 MB, usually pageable R memory) goes up in pieces of two columns on a second stream:
  // the host stages piece p + 1 while the kernels of piece p run, instead of 3-4 ms of upload in front of everything
  if (!h->copy_stream) BSG_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (cudaEvent_t &e : h->copy_ev)
    if (!e) BSG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  BSG_CUDA(cudaEventRecord(h->copy_ev[7], s));  // dV may still be read by work enqueued earlier on s
  BSG_CUDA(cudaStreamWaitEvent(h->copy_stream, h->copy_ev[7], 0));
  auto upload = [&](int k0, int k1) -> int {  // columns [k0, k1) of V; afterwards s waits for them
    BSG_CUDA(cudaMemcpyAsync(dV + (size_t)k0 * nc, V + (size_t)k0 * nc, (size_t)(k1 - k0) * nc * sizeof(double),
                             cudaMemcpyHostToDevice, h->copy_stream));
    cudaEvent_t ev = h->copy_ev[(k0 / 2) % 7];
    BSG_CUDA(cudaEventRecord(ev, h->copy_stream));
    BSG_CUDA(cudaStreamWaitEvent(s, ev, 0));
    return BSG_OK;
  };
  int *d_bad = reinterpret_cast<int *>(d_cols + 3 * (size_t)nc + NP);  // any pass saw a non-finite quantity
  BSG_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), s));
  static int pair_mode = -1;
  if (pair_mode < 0) {
    const char *ev = getenv("BSG_PROJ_PAIR");
    pair_mode = (ev && ev[0] == '0') ? 0 : 1;
  }
  if (pair_mode && K >= 2) {
    // two columns of V per pass over the matrix (30-bit fixed point per vector, see k_quantT_pair)
    for (int k = 0; k < K; k += 2) {
      const bool both = k + 1 < K;
      BSG_TRY(upload(k, std::min(K, k + 2)));
      BSG_TRY(prodvec_T_pair(v, dV + (size_t)k * nc, both ? dV + (size_t)(k + 1) * nc : nullptr, dXV + (size_t)k * nr,
                             both ? dXV + (size_t)(k + 1) * nr : nullptr, s));
      k_or_flag<<<1, 1, 0, s>>>(v->s_scal.as<pmv::Scal>(), d_bad);
      k_or_flag<<<1, 1, 0, s>>>(v->s_scal.as<pmv::Scal>() + 1, d_bad);
      count_launch(2);
    }
  } else {
    if (K > 0) BSG_TRY(upload(0, K));
    for (int k = 0; k < K; k++) {
      BSG_TRY(bsg_view_prodvec_dev(v, dV + (size_t)k * nc, dXV + (size_t)k * nr, s));
      k_or_flag<<<1, 1, 0, s>>>(v->s_scal.as<pmv::Scal>(), d_bad);
      count_launch();
    }
  }
  bool need_simple = false;
  {
    double *d_a = d_cols, *d_w = d_cols + nc, *d_n = d_cols + 2 * (size_t)nc, *d_tp = d_cols + 3 * (size_t)nc;
    double *d_t1 = d_rows + nr, *d_t2 = nullptr;
    k_rss_weights<<<NP, 256, 0, s>>>(v->d_center, v->d_scale, nc, d_a, d_w, d_n, d_tp);
    count_launch();
    PlaneOut o1{1.0, 2.0, 0.0, d_t1, 0, 0, nullptr};
    BSG_TRY(view_planes_dev(v, 0, d_a, d_w, PLANE_HI, o1, s));
    if (h->has_na) {
      d_t2 = d_rows + 2 * (size_t)nr;
      PlaneOut o2{0.0, -1.0, 0.0, d_t2, 0, 0, nullptr};
      BSG_TRY(view_planes_dev(v, 0, d_n, d_n, PLANE_NA, o2, s));
    }
    k_rss_final<<<(nr + 255) / 256, 256, 0, s>>>(nr, d_t1, d_t2, d_tp, NP, d_rs);
    count_launch();
    k_or_flag<<<1, 1, 0, s>>>(v->s_scal.as<pmv::Scal>(), d_bad);
    count_launch();
    int bad = 0;  // zero / non-finite scale: the table arithmetic of the accessor kernels gives the reference's Inf / NaN
    BSG_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, s));
    BSG_CUDA(cudaStreamSynchronize(s));
    if (bad) {
      need_simple = true;
      for (int k = 0; k < K; k++)
        BSG_TRY(simple_prodvec(h, v->d_row, nr, v->d_col, nc, v->d_center, v->d_scale, dV + (size_t)k * nc,
                               dXV + (size_t)k * nr, s));
    }
  }
  if (need_simple) BSG_TRY(simple_rowsumssq(h, v->d_row, nr, v->d_col, nc, v->d_center, v->d_scale, d_rs, s));
  BSG_CUDA(cudaMemcpyAsync(XV, dXV, (size_t)nr * K * sizeof(double), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaMemcpyAsync(rowSumsSq, d_rs, (size_t)nr * sizeof(double), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaStreamSynchronize(s));
  return BSG_OK;
}

// multLinReg (src/multLinReg.cpp:8-88): t-scores of genotype ~ U[, k] per SNP over the samples where the
// genotype is present.  U is nr x K column-major, tscores nc x K column-major, NA_REAL is written as NaN.
int bsg_multlinreg(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *U, int K,
                   double *tscores) {
  if (!h || !tscores || (!U && K > 0)) return fail(BSG_ERR_ARG, "null argument");
  if (K < 0) return fail(BSG_ERR_ARG, "negative length");
  if (h->fbm_generic) {  // dosage FBM: literal fp64 sums over code256[byte] (bsg_generic.cu)
    BSG_TRY(bind_device(h));
    if (!ind_row) nr = h->n;
    if (!ind_col) nc = h->m;
    if (nc == 0 || K == 0) return BSG_OK;
    cudaStream_t gs = h->stream;
    const int *d_row = nullptr, *d_col = nullptr;
    BSG_TRY(upload_index(h, ind_row, nr, h->n, h->w_idx_row, &d_row));
    BSG_TRY(upload_index(h, ind_col, nc, h->m, h->w_idx_col, &d_col));
    BSG_TRY(h->w_tmp1.ensure((size_t)std::max(nr, 1) * K * sizeof(double)));
    BSG_TRY(h->w_tmp2.ensure((size_t)nc * K * sizeof(double)));
    BSG_CUDA(cudaMemcpyAsync(h->w_tmp1.p, U, (size_t)nr * K * sizeof(double), cudaMemcpyHostToDevice, gs));
    BSG_TRY(generic_multlinreg(h, d_row, nr, d_col, nc, h->w_tmp1.as<double>(), K, h->w_tmp2.as<double>(), gs));
    BSG_CUDA(cudaMemcpyAsync(tscores, h->w_tmp2.p, (size_t)nc * K * sizeof(double), cudaMemcpyDeviceToHost, gs));
    BSG_CUDA(cudaStreamSynchronize(gs));
    return BSG_OK;
  }
  bsg_view *v = nullptr;
  BSG_TRY(cached_view(h, ind_row, nr, ind_col, nc, nullptr, nullptr, &v));
  nr = v->nr;
  nc = v->nc;
  if (nc == 0 || K == 0) return BSG_OK;
  cudaStream_t s = h->stream;
  ProjScratch mem{h};
  double *dU, *dUU = nullptr, *dG, *dNu = nullptr, *dNuu = nullptr, *dY, *dOut;
  BSG_TRY(mem.alloc(&dU, (size_t)nr * K));
  BSG_TRY(mem.alloc(&dG, (size_t)nc * K));
  BSG_TRY(mem.alloc(&dOut, (size_t)nc * K));
  BSG_TRY(mem.alloc(&dY, 2 * (size_t)K));
  std::vector<double> ysum(2 * (size_t)K, 0.0);
  for (int k = 0; k < K; k++) {
    double y = 0, yy = 0;
    for (int i = 0; i < nr; i++) {
      const double u = U[(size_t)k * nr + i];
      y += u;
      yy += u * u;
    }
    ysum[k] = y;
    ysum[K + k] = yy;
  }
  BSG_CUDA(cudaMemcpyAsync(dU, U, (size_t)nr * K * sizeof(double), cudaMemcpyHostToDevice, s));
  BSG_CUDA(cudaMemcpyAsync(dY, ysum.data(), 2 * (size_t)K * sizeof(double), cudaMemcpyHostToDevice, s));
  const bool na = h->has_na != 0;
  if (na) {
    BSG_TRY(mem.alloc(&dUU, (size_t)nr * K));
    BSG_TRY(mem.alloc(&dNu, (size_t)nc * K));
    BSG_TRY(mem.alloc(&dNuu, (size_t)nc * K));
    k_square<<<launch_cap_pub((int64_t)nr * K), 256, 0, s>>>(dU, (int64_t)nr * K, dUU);
    count_launch();
  }
  static int pair_mode = -1;
  if (pair_mode < 0) {
    const char *ev = getenv("BSG_MLR_PAIR");
    pair_mode = (ev && ev[0] == '0') ? 0 : 1;
  }
  if (pair_mode && K >= 2) {
    // two columns of U per pass over the matrix (30-bit fixed point per vector: ~1e-9 of the sums).  The t-scores of a pair
    // are evaluated right after its passes and fetched (nc x 2 doubles into usually pageable, untouched host memory: the
    // fetch blocks the host) while the passes of the NEXT pair run.
    BSG_CUDA(cudaStreamSynchronize(s));  // the counts helper stages its index upload from host memory
    int32_t *d_cnt0 = nullptr;
    BSG_TRY(col_counts_dev(h, ind_row, nr, ind_col, nc, &d_cnt0));
    if (!h->copy_stream) BSG_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (cudaEvent_t &e : h->copy_ev)
      if (!e) BSG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    auto fetch = [&](int k0) -> int {
      const int k1 = std::min(K, k0 + 2);
      BSG_CUDA(cudaStreamWaitEvent(h->copy_stream, h->copy_ev[(k0 / 2) % 7], 0));
      BSG_CUDA(cudaMemcpyAsync(tscores + (size_t)k0 * nc, dOut + (size_t)k0 * nc, (size_t)(k1 - k0) * nc * sizeof(double),
                               cudaMemcpyDeviceToHost, h->copy_stream));
      return BSG_OK;
    };
    for (int k = 0; k < K; k += 2) {
      const bool both = k + 1 < K;
      const double *ua = dU + (size_t)k * nr, *ub = both ? dU + (size_t)(k + 1) * nr : nullptr;
      pmvt::PairCoef ca{1.0, na ? -3.0 : 0.0, 0.0, 1.0, dG + (size_t)k * nc, na ? dNu + (size_t)k * nc : nullptr};
      pmvt::PairCoef cb{1.0, na ? -3.0 : 0.0, 0.0, 1.0, both ? dG + (size_t)(k + 1) * nc : nullptr,
                        (na && both) ? dNu + (size_t)(k + 1) * nc : nullptr};
      BSG_TRY(view_planes_pair_dev(v, ua, ub, na ? PLANE_NA : PLANE_NONE, ca, cb, s));
      if (na) {
        const double *uua = dUU + (size_t)k * nr, *uub = both ? dUU + (size_t)(k + 1) * nr : nullptr;
        pmvt::PairCoef da{0.0, 1.0, 0.0, 0.0, dNuu + (size_t)k * nc, nullptr};
        pmvt::PairCoef db{0.0, 1.0, 0.0, 0.0, both ? dNuu + (size_t)(k + 1) * nc : nullptr, nullptr};
        BSG_TRY(view_planes_pair_dev(v, uua, uub, PLANE_NA, da, db, s));
      }
      const int kp = both ? 2 : 1;
      k_tscores<<<launch_cap_pub((int64_t)nc * kp), 256, 0, s>>>(nc, kp, d_cnt0, dG + (size_t)k * nc, na ? dNu + (size_t)k * nc : nullptr,
                                                                na ? dNuu + (size_t)k * nc : nullptr, dY + k, dY + K + k,
                                                                dOut + (size_t)k * nc);
      count_launch();
      BSG_CUDA(cudaEventRecord(h->copy_ev[(k / 2) % 7], s));
      if (k >= 2) BSG_TRY(fetch(k - 2));
    }
    BSG_TRY(fetch(((K - 1) / 2) * 2));
    BSG_CUDA(cudaGetLastError());
    BSG_CUDA(cudaStreamSynchronize(h->copy_stream));
    BSG_CUDA(cudaStreamSynchronize(s));
    return BSG_OK;
  } else {
    for (int k = 0; k < K; k++) {
      const double *u = dU + (size_t)k * nr;
      PlaneOut o1{1.0, na ? -3.0 : 0.0, 0.0, dG + (size_t)k * nc, 0.0, 1.0, na ? dNu + (size_t)k * nc : nullptr};
      BSG_TRY(view_planes_dev(v, 1, u, u, na ? PLANE_NA : PLANE_NONE, o1, s));
      if (na) {
        const double *uu = dUU + (size_t)k * nr;
        PlaneOut o2{0.0, 1.0, 0.0, dNuu + (size_t)k * nc, 0, 0, nullptr};
        BSG_TRY(view_planes_dev(v, 1, uu, uu, PLANE_NA, o2, s));
      }
    }
  }
  BSG_CUDA(cudaStreamSynchronize(s));  // the counts helper stages its index upload from host memory
  int32_t *d_cnt = nullptr;
  BSG_TRY(col_counts_dev(h, ind_row, nr, ind_col, nc, &d_cnt));
  k_tscores<<<launch_cap_pub((int64_t)nc * K), 256, 0, s>>>(nc, K, d_cnt, dG, dNu, dNuu, dY, dY + K, dOut);
  count_launch();
  BSG_CUDA(cudaGetLastError());
  BSG_CUDA(cudaMemcpyAsync(tscores, dOut, (size_t)nc * K * sizeof(double), cudaMemcpyDeviceToHost, s));
  BSG_CUDA(cudaStreamSynchronize(s));
  return BSG_OK;
}

// 0: automatic (sample-major kernel when that copy is resident, else the SNP-major kernel); 1: always the
// SNP-major kernel (k_pmvT) for the X-side products.  Process-wide; for tests and measurements.
// 1: the 9-argument calls skip the upload of center / scale when address, length and a strided sample of the values equal
// those of the previous call on the handle (see scaling_sample); 0 (default): always upload.  Process-wide.
int bsg_set_scaling_reuse(int on) {
  if (on != 0 && on != 1) return fail(BSG_ERR_ARG, "on must be 0 or 1");
  g_scaling_reuse = on;
  return BSG_OK;
}

int bsg_set_prodvec_path(int path) {
  if (path != 0 && path != 1) return fail(BSG_ERR_ARG, "path must be 0 or 1");
  g_force_t = path;
  return BSG_OK;
}

double bsg_last_kernel_ms(void) {
  using namespace pmv;
  if (!g_ev_ready || g_ev_n == 0) return 0.0;
  float ms = 0;
  int k = (g_ev_n - 1) % EV_POOL;
  if (cudaEventElapsedTime(&ms, g_ev0[k], g_ev1[k]) != cudaSuccess) {
    cudaGetLastError();
    return 0.0;
  }
  return (double)ms;
}

// enable (and reset) / disable CUDA-event timing of the tensor-pipe kernel; events are recorded on the
// launching stream around every k_pmv launch.
int bsg_set_kernel_timing(int on) {
  using namespace pmv;
  if (on && !g_ev_ready) {
    for (int k = 0; k < EV_POOL; k++) {
      BSG_CUDA(cudaEventCreate(&g_ev0[k]));
      BSG_CUDA(cudaEventCreate(&g_ev1[k]));
    }
    g_ev_ready = true;
  }
  g_timing = on != 0;
  g_ev_n = 0;
  return BSG_OK;
}

// launches timed since the last bsg_set_kernel_timing(1) and their summed device time (ms).  Call after
// synchronising the stream(s).  At most the last 128 launches are kept.
int bsg_kernel_time_stats(int *count, double *total_ms) {
  using namespace pmv;
  int n = g_ev_n < EV_POOL ? g_ev_n : EV_POOL;
  double tot = 0;
  for (int k = 0; k < n; k++) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, g_ev0[k], g_ev1[k]) != cudaSuccess) {
      cudaGetLastError();
      return fail(BSG_ERR_CUDA, "kernel timing events not complete: synchronise first");
    }
    tot += ms;
  }
  if (count) *count = n;
  if (total_ms) *total_ms = tot;
  return BSG_OK;
}

}  // extern "C"
