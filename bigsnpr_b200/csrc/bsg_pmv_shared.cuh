// bsg_pmv_shared.cuh -- device-side pieces of the matvecs shared between bsg_pmv.cu (2-bit kernels, plain finish kernels),
// bsg_pmv8.cu (value-byte kernel) and bsg_comm.cu (finish fused with the all-reduce over NVLink peer memory).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bsg {
namespace pmv {

constexpr int SUMCZ_BLOCKS = 128;

constexpr int SEG = 128;              // bytes per line per stage = 512 codes
constexpr int CODES = 512;            // codes per line per stage
constexpr int DIG = 4096;             // digit bytes per stage per plane (512 codes x 8 slices)
constexpr int STAGES = 6;
constexpr int STAGE_BYTES = 2 * DIG;  // raw-plane digits + NA-plane digits
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 128;
// Variants <CW consumer warps, R chunks of register ring per warp>; lines per work item = 32 * CW.
// Register file: (CW + 1) warps share 4 SMSPs of 16 K registers -> cap 255 regs for 8 warps, 168 for 9..12.
constexpr int MAX_CHUNKS_PER_ITEM = 512;  // 262144 codes: |acc16| <= 262144*48*128 < 2^31

struct Args {
  const uint8_t *P;
  int64_t stride;
  const int *lines;      // physical line per logical line (null = identity)
  int nlines;
  int nlines_pad;        // multiple of the group size (32 * consumer warps)
  int nchunks;           // 128-byte chunks per line
  int chunks_per_split;
  int ksplit;
  const uint8_t *dig1;   // [nchunks][DIG]
  const uint8_t *dig2;   // NA-plane digits (null = same as dig1)
  const uint8_t *na_flags;  // per physical line (null = assume missing values anywhere)
  int use_na;            // 0: matrix has no missing value, skip the NA plane
  long long *part;       // [nlines_pad][16] zeroed accumulators: 8 raw-plane slices, 8 NA-plane slices
};

struct Scal {          // device-resident scalars of one call
  double maxabs[2];    // [0] raw-plane vector, [1] NA-plane vector
  int nonfinite;
  int e[2];            // Q = rint(v * 2^e); written by the scatter path, derived from maxabs on the direct path
  int hb;              // headroom bits (log2 of the largest index multiplicity)
  double Y;            // sum of the (scattered) vector, for Xt.y
  double C;            // (unused, kept for layout)
  long long sum_hi, sum_lo;
  double cpart[128];   // per-block partials of sum_k c_k z_k (X.y), added in index order by the finish kernel
};

// ---- PTX wrappers of the tensor-pipe matvec kernels (k_pmv, k_pmvT: bsg_pmv.cu; k_pmv8: bsg_pmv8.cu) ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void mma_u8s8(int (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                         uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k32.row.col.s32.u8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

__device__ __forceinline__ uint4 ldg_stream(const uint8_t *p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p));
  return v;
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
  return r;
}

// (raw-plane * c0 + NA-plane * c1) per digit slice, exact in integers, then one top-down fp64 sum of the 8
// scaled slice totals.
__device__ __forceinline__ double combine8(const long long *__restrict__ part, int64_t line, int c0, int c1, int e) {
  const long long *p = part + line * 16;
  double acc = 0;
#pragma unroll
  for (int s = 7; s >= 0; s--) {
    long long v = 0;
    if (c0) v += c0 * p[s];
    if (c1) v += c1 * p[8 + s];
    acc += scalbn((double)v, 8 * s - e);
  }
  return acc;
}

// X.y:  full_l = R + Nw - C   with Nw the NA-plane sum against w = (c - 3) z;  without scaling full_l = R - 3 N.
__device__ __forceinline__ double finish_prod_value(const long long *__restrict__ part, int64_t l, const Scal *sc,
                                                    int has_scaling, int use_na) {
  if (sc->nonfinite) return nan("");
  if (has_scaling) {
    double C = 0;
    for (int b = 0; b < SUMCZ_BLOCKS; b++) C += sc->cpart[b];
    double R = combine8(part, l, 1, 0, sc->e[0]);
    double Nw = use_na ? combine8(part, l, 0, 1, sc->e[1]) : 0.0;
    return (R + Nw) - C;
  }
  return combine8(part, l, 1, use_na ? -3 : 0, sc->e[0]);  // R - 3N, exact
}

}  // namespace pmv
}  // namespace bsg
