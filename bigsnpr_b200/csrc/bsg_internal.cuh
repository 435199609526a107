// bsg_internal.cuh -- shared declarations of libbsgpu (not part of the public ABI).
//
// HBM layout of a staged genotype matrix (see DESIGN.md "Data layout"):
//   * "staged code": 2 bits per genotype, value = genotype for 0/1/2 and 3 for missing.  It is a
//     bijective recode of the .bed code of the reference (src/bed-acc.h:22-37: 00->2, 01->NA,
//     10->1, 11->0), done once at staging, so that the packed value IS the number the kernels
//     multiply with.  Padding slots (samples >= n of the last byte, bytes up to the line stride)
//     hold code 0: they add nothing to any sum and are never missing.
//   * copy A (SNP-major): line j = SNP column j, n codes, lowest bits = first sample -- the .bed
//     orientation.  Line stride = round_up(ceil(n/4), 128) bytes.
//   * copy B (sample-major), optional: line i = sample i, m codes.  Line stride = round_up(ceil(m/4), 128).
//     Built on request or on first use by the GRM; every other kernel runs from copy A alone.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "bsgpu.h"

#define BSG_KIND_BED 0
#define BSG_KIND_FBM 1

namespace bsg {

extern thread_local std::string g_err;
int fail(int code, const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);
void count_launch(int n = 1);

#define BSG_CUDA(call)                                   \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return bsg::cuda_fail(e__, #call); \
  } while (0)

#define BSG_TRY(call)        \
  do {                       \
    int rc__ = (call);       \
    if (rc__) return rc__;   \
  } while (0)

inline int64_t round_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

// growable device scratch buffer
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes);
  void release();
  template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

}  // namespace bsg

#define BSG_MAX_PEERS 16

// One rank's end of a group of GPUs that exchange data through each other's memory over NVLink / NVSwitch (peer access
// inside one process, CUDA IPC between processes).  Region layout (same on every rank):
//   [0, 1024)        push flags: flag[q] = last epoch whose data rank q has finished writing into THIS region
//   [1024, 2048)     barrier flags, same convention
//   [2048, 2112)     block counter of the fused kernels (+ padding)
//   [4096, ...)      slots: 2 parities x world x slot_elems doubles; slot (p, q) receives rank q's vector of epoch parity p
struct bsg_comm {
  int rank = 0, world = 1, device = 0;
  size_t slot_elems = 0;
  uint8_t *region = nullptr;
  size_t region_bytes = 0;
  uint8_t *peer[BSG_MAX_PEERS] = {nullptr};  // peer[q]: rank q's region mapped into this device's address space
  bool peer_ipc[BSG_MAX_PEERS] = {false};    // opened with cudaIpcOpenMemHandle (to be closed)
  unsigned long long epoch = 0, bar_epoch = 0;
  int *d_err = nullptr;                      // set by a kernel whose wait timed out
  bool connected = false;
};

struct bsg_bed {
  int kind = BSG_KIND_BED;
  int device = 0;
  int n = 0, m = 0;          // samples, SNP columns held by this handle
  int64_t n_byte = 0;        // ceil(n/4): bytes per column in the .bed file
  int64_t strideA = 0, strideB = 0;
  uint8_t *A = nullptr;      // m lines of strideA bytes
  uint8_t *B = nullptr;      // n lines of strideB bytes (may be null)
  int layouts = 0;
  int has_na = 0;
  int32_t *cntA = nullptr;   // [m][4] counts of codes 0,1,2,3 per SNP over all n samples
  int32_t *cntB = nullptr;   // [n][4] counts per sample over all m SNPs (only with copy B)
  uint8_t *naA = nullptr;    // [m] 1 if the SNP line has a missing value
  uint8_t *naB = nullptr;    // [n]
  // missing-value positions as blocked-ELL lists (bsg_naell.cu), built on first use; side 0: lines = samples, 1: lines = SNPs
  uint16_t *ellCnt[2] = {nullptr, nullptr}, *ellEnt[2] = {nullptr, nullptr};
  long long *ellOff[2] = {nullptr, nullptr}, *ellOut[2] = {nullptr, nullptr};
  int ellChunks[2] = {0, 0}, ellGroups[2] = {0, 0};
  int64_t na_nnz = 0;
  int na_ell = 0;            // 0 not tried yet, 1 resident, -1 not used (rate too high, no memory, disabled)
  double code256[256];       // FBM handles: value of each raw byte code (bigstatsr code256)
  int fbm_generic = 0;       // FBM whose codes are not {0,1,2,NA} (dosages ...): served by the fp64 kernels of bsg_generic.cu
  uint8_t *raw = nullptr;    // generic FBM: the n x m code bytes, column-major, line j at raw + j * raw_stride
  int64_t raw_stride = 0;    // n, or round_up(n, 512) with zero padding for a centi-dosage handle
  double *d_code = nullptr;  // generic FBM: byte value on the device [0,256) and the same with NA -> 3 [256,512)
  // centi-dosage FBM (every code a multiple of 1/100 in [0, 2.54], bsg_core.cu): raw holds VALUE bytes rint(100 x), 255 =
  // missing, and d_code is indexed by value byte; the matvecs run on the integer tensor pipe (bsg_pmv8.cu)
  int dosage = 0;
  std::vector<int> na_line;  // centi-dosage: missing values per SNP line over all n samples
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaStream_t copy_stream = nullptr;  // created on first use: host -> device uploads that run under the kernels of `stream`
  cudaEvent_t copy_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  // view cached for the 9-argument drop-in matvec calls (bsg_prodvec / bsg_cprodvec)
  struct bsg_view *cv = nullptr;
  std::vector<int> cv_row, cv_col;
  // fingerprint of the center / scale vectors last uploaded into the cached view (address, length, strided sample of the
  // values): an unchanged scaling is not uploaded again by the next 9-argument call
  const double *cv_center_ptr = nullptr, *cv_scale_ptr = nullptr;
  std::vector<double> cv_scal_sample;
  // scratch reused across calls
  bsg::DevBuf w_idx_row, w_idx_col, w_center, w_scale, w_x, w_out, w_tmp0, w_tmp1, w_tmp2, w_tmp3,
      w_part, w_dig1, w_dig2, w_misc;
  bsg::DevBuf w_proj[8];  // projection / multLinReg work arrays (grow-only, reused across calls)
};

namespace bsg {

// ---- bsg_core.cu -----------------------------------------------------------------------------
int stage_finish(bsg_bed *h);  // counts and NA flags from copy A; copy B only when requested
int build_copy_B(bsg_bed *h);  // sample-major copy on demand (no-op when resident)
int bind_device(const bsg_bed *h);
void prefault_pages(void *p, size_t bytes);  // parallel first touch of a host output buffer (bsg_core.cu)
cudaError_t pool_alloc(void **p, size_t bytes, int device, cudaStream_t s);  // stream-ordered pool, freed with cudaFree

// ---- index helpers (bsg_core.cu) -------------------------------------------------------------
// validates 1-based host indices against `limit` (src/bed-acc.h:64-65) and uploads them 0-based.
// ind == NULL -> identity of length `len` is implied, *dev = nullptr.
int upload_index(bsg_bed *h, const int *ind, int len, int limit, DevBuf &buf, const int **dev);

// ---- bsg_simple.cu: generic accessor-style kernels (any index multiset) ----------------------
int simple_prodvec(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, const double *d_center,
                   const double *d_scale, const double *d_x, double *d_out, cudaStream_t s);
int simple_cprodvec(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, const double *d_center,
                    const double *d_scale, const double *d_x, double *d_out, cudaStream_t s);
int counts_cols(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, int32_t *d_out4, cudaStream_t s);
int counts_rows(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, int32_t *d_out4, cudaStream_t s);
int read_dense(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, int na_val, int *d_out, cudaStream_t s);
int read_bytes(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, uint8_t *d_out, cudaStream_t s);
int pack_bed(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, uint8_t *d_out, cudaStream_t s);
int read_dense_scaled(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, const double *d_center,
                      const double *d_scale, double *d_out, cudaStream_t s);

// ---- bsg_pmv.cu: 4 x nr code counts per sample from the plane sums of the X-side kernels (device array)
int row_counts_planes(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, int32_t *d_out4);

// ---- bsg_stats.cu: 4 x nc code counts of (ind_row, ind_col) on the device (h->w_tmp0), on h->stream
int col_counts_dev(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, int32_t **d_out);
int simple_rowsumssq(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, const double *d_center,
                     const double *d_scale, double *d_out, cudaStream_t s);

// ---- bsg_cor.cu: dense sub-matrix of a packed matrix, per-line code counts ------------------------
int compact_lines(const uint8_t *src, int64_t src_stride, const int *code_idx, int ncodes, const int *line_idx,
                  int nlines, uint8_t *out, int64_t out_stride, cudaStream_t s);
int line_counts(const uint8_t *P, int64_t stride, int nlines, int L, int32_t *cnt, uint8_t *na, cudaStream_t s);

// ---- bsg_gram5.cu: 128 x 128 integer Gram tiles on tcgen05 / TMEM (tiles = gram::Tile array on the device)
int gram5_launch(const uint8_t *P, int64_t stride, int nlines, int64_t line_bytes, const void *d_tiles, int ntiles,
                 int *d_sums, bool any_clean, bool any_na, cudaStream_t s);

// weighted Gram for the GRM on tcgen05: tiles = (i0, j0, mode) int triplets on the host, K pre-zeroed, fills i >= j
int wgram5_launch(const uint8_t *P, int64_t stride, int nlines, int nslices, const uint8_t *const dig[3],
                  int64_t dig_stride, const double (*scale)[10], const int *h_tiles, int ntiles, double *K,
                  int64_t ldk, cudaStream_t s);

// ---- bsg_naell.cu: missing values of the matvecs as blocked-ELL lists gathered from shared memory -------------------
bool na_ell_ready(bsg_bed *h);
int na_ell_correction(bsg_bed *h, int side, const int *lines, int nlines, const long long *Q, long long *part, cudaStream_t s);

// ---- bsg_generic.cu: fp64 fallback for FBM.code256 handles whose codes are not 0 / 1 / 2 / NA (dosages) --------------
#define BSG_PACKED_ONLY(h, what)                                                                                          \
  do {                                                                                                                    \
    if ((h)->fbm_generic)                                                                                                 \
      return bsg::fail(BSG_ERR_TYPE, "%s needs hard calls (codes 0 / 1 / 2 / NA); this FBM.code256 holds other values "    \
                                     "(dosages): snp_colstats, snp_cor, snp_ld_scores, snp_clumping and snp_pcadapt are served " \
                                     "by the fp64 kernels, the packed engine is not.", what);                             \
  } while (0)
int generic_colstats(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, double *d_sumX, double *d_denoX,
                     cudaStream_t s);
// pair statistics of the windowed correlations straight from the code bytes; kind 0: r + keep (threshold), 1: r^2,
// 3: clumping_chr conflict flag (src/clumping.cpp:66-73) with the caller's sumX / denoX
int generic_pairs(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, int kind, const int *d_wlen,
                  const long long *d_boff, long long total, const double *d_thr, double *d_band, uint8_t *d_keep,
                  const double *d_sumX, const double *d_denoX, double thr_r2, cudaStream_t s);
int generic_multlinreg(bsg_bed *h, const int *d_row, int nr, const int *d_col, int nc, const double *d_U, int K,
                       double *d_out, cudaStream_t s);

// ---- bsg_pmv8.cu: centi-dosage handles (value bytes) ----------------------------------------------------------------
// code table -> value byte per code (255 = NA); false when the table is not centi-dosage (see bsg_open_fbm256)
bool dosage_value_bytes(const double *code256, uint8_t vbyte[256]);
// value bytes with a zero-padded line stride + missing values per line, from the n x m code bytes on the device
int dosage_stage(bsg_bed *h, const uint8_t *d_codes, const uint8_t *d_vbyte);
// Xt.y on the value bytes: lines = SNP columns, contraction over all n samples (pmv::Args: dig1 = k_prep2 / k_digits
// layout, part zeroed here); the NA plane is never used
namespace pmv { struct Args; }
int run_pmv8(bsg_view *v, const uint8_t *dig, pmv::Args *out, cudaStream_t s);
// view scaling of a centi-dosage handle: d_center, d_scale (uploaded as c, s) -> 100 c, 100 s
int dosage_view_scaling(bsg_view *v, cudaStream_t s);
// host-vector forms: out[t] = NaN for every output entry whose row / column meets a selected missing value
int dosage_mark_na(bsg_view *v, bool cprod, double *d_out, cudaStream_t s);
// prod_and_rowSumsSq2 on a centi-dosage view (host V / XV / rowSumsSq, synchronous)
int dosage_prod_and_rowsumssq(bsg_view *v, const double *V, int K, double *XV, double *rowSumsSq);

// ---- bsg_gramt.cu: integer Gram tiles fed by TMA, 2-CTA tcgen05 MMAs (GRM and windowed correlations) ----------
namespace gram { struct Tile; }
bool gramt_enabled();  // BSG_GRAM_TMA=0 selects the round-1 kernels (in-kernel expansion) for cross-checks
int gramt_grm(const uint8_t *P, int64_t stride, int nr, int nc, const double *const Ws[3], const double wmax[3],
              const uint8_t *na, int nslices, double *K, int64_t ldk, int device, cudaStream_t s);
int gramt_cor(const uint8_t *M, int64_t stride, int nlines, const gram::Tile *tiles, int ntiles, int *d_sums, int device,
              cudaStream_t s, bool *done);

// ---- bsg_pmv.cu: packed matrix x vector on the integer tensor pipe ----------------------------
struct PmvPlan;  // opaque, owned by a view
namespace pmv { struct Scal; }
// X~ x enqueued on `s`; with a communicator the partial n-vectors of the column shards are summed (fused epilogue)
int view_prodvec_comm(bsg_view *v, const double *x_dev, double *out_dev, cudaStream_t s, bsg_comm *comm);

// ---- bsg_la.cu: the Lanczos driver over one or several column shards (one replica of the recurrence per shard) ----
struct SvdShard {
  bsg_bed *h;
  const int *ind_col;              // local 1-based columns of this shard (null = all)
  int nc;
  const double *center, *scale;    // per local column, or null (bed_scaleBinom computed on the device)
  bsg_comm *comm;                  // null: single shard
  double *v_out;                   // host, receives this shard's rows of v (null: not wanted)
  int64_t v_ld;                    // leading dimension of v_out
  const int *v_pos;                // row of v_out per local column (null: 0..nc-1)
  double *center_out, *scale_out;  // optional, indexed like the rows of v_out
};
int lanczos_svd(std::vector<SvdShard> &sh, const int *ind_row, int nr, int ncol_total, int k, double tol, int maxit, double *d,
                double *u, int *niter, int *nops, double *z_dev, bsg_reduce_cb reduce_cb, void *cb_ctx);

// ---- bsg_comm.cu: collectives over NVLink peer memory ------------------------------------------------
// epilogue of X.y (integer slice sums -> fp64) fused with the all-reduce over the shards: one kernel
int comm_finish_prod_allreduce(bsg_comm *c, const long long *part, int nlines, const pmv::Scal *sc, int has_scaling,
                               int use_na, double *out_dev, cudaStream_t s);
// in-place sum of `count` doubles over the ranks (one-shot: push to every peer, sum in rank order)
int comm_allreduce_oneshot(bsg_comm *c, double *buf_dev, int64_t count, cudaStream_t s);
}  // namespace bsg

struct bsg_view {
  bsg_bed *h = nullptr;
  int nr = 0, nc = 0;
  int row_identity = 1, col_identity = 1;
  int row_maxmult = 1, col_maxmult = 1;
  int has_scaling = 0;       // center/scale given (else 0 / 1); always 1 on a centi-dosage handle
  int any_na = 0;            // centi-dosage: a selected SNP column holds a missing value
  int *d_na_pos = nullptr;   // centi-dosage: positions (in ind_col) of the selected columns holding a missing value
  int n_na_pos = 0;
  // device arrays (owned)
  int *d_row = nullptr;      // [nr] 0-based rows (null if identity)
  int *d_col = nullptr;      // [nc] 0-based cols (null if identity)
  double *d_center = nullptr, *d_scale = nullptr;  // [nc] (null if !has_scaling); 100 c, 100 s on a centi-dosage handle
  // prodvec over copy B: distinct rows to compute and the gather map back to ind_row order
  int *d_rows_unique = nullptr;  // [nru] sorted distinct rows (null if identity)
  int *d_row_gather = nullptr;   // [nr] position of each requested row in d_rows_unique
  int nru = 0;
  // scratch owned by the view (so device-pointer calls are allocation free)
  bsg::DevBuf s_vec0, s_vec1, s_vec2, s_q0, s_q1, s_dig1, s_dig2, s_part, s_scal, s_full;
};
