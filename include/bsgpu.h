/*
 * bsgpu.h -- C ABI of libbsgpu, the B200 (sm_100a) engine for bigsnpr's packed-genotype hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no R / torch types.  Every entry point
 * replaces one `.Call` target of privefl/bigsnpr 1.12.21 (file:line under /root/reference cited per
 * function); the R-side shim that binds them under the original `_bigsnpr_*` names is r_shim/ and
 * is documented in INTEGRATION.md.
 *
 * Conventions (kept from the reference so the shim is a pass-through):
 *   - ind_row / ind_col are 1-based int32 (R integer vectors); duplicates and any order are allowed
 *     (src/bed-acc.h:64-65).  NULL means "all rows" / "all columns" (rows_along / cols_along).
 *   - matrices are column-major; vectors are double (REALSXP) or int32 (INTSXP).
 *   - all pointers are HOST pointers unless the name ends in _dev.
 *   - every function returns 0 on success, else a BSG_ERR_* code; bsg_last_error() returns the message
 *     (the text the reference raises, e.g. "Incompatibility between dimensions.").
 *   - `ncores` of the reference is accepted by the shim and ignored: the GPU path has no thread knob.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     BSG_ERR_CUDA.
 */
#ifndef BSGPU_H
#define BSGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSG_OK 0
#define BSG_ERR_DIM 1     /* "Incompatibility between dimensions."  src/bed-acc.h:95-96 */
#define BSG_ERR_BOUNDS 2  /* subscript out of bounds                  src/bed-acc.h:64-65 */
#define BSG_ERR_MAGIC 3   /* "File is not a binary PED file."         src/bed-acc-xptr.cpp:21-22 */
#define BSG_ERR_MODE 4    /* "Variant-major is the only mode supported."  src/bed-acc-xptr.cpp:29-30 */
#define BSG_ERR_SIZE 5    /* "n or p does not match the dimensions of the file."  :33-34 */
#define BSG_ERR_IO 6      /* "Error when mapping file"                 src/bed-acc-xptr.cpp:19 */
#define BSG_ERR_ALLOC 7
#define BSG_ERR_CUDA 8
#define BSG_ERR_ARG 9
#define BSG_ERR_TYPE 10   /* "Unknown object type."                    src/corr.cpp:124 */

/* layouts kept resident in HBM (bit mask) */
#define BSG_LAYOUT_SNP_MAJOR 1    /* variant-major, the .bed orientation: serves every entry point at full speed */
#define BSG_LAYOUT_SAMPLE_MAJOR 2 /* also keep the 2-bit transpose (what the GRM tiles read; X.y 1-3 % faster on it) */
#define BSG_LAYOUT_AUTO 0         /* SNP-major only; the transpose is built on first use by bsg_tcrossprod */

typedef struct bsg_bed bsg_bed;   /* replaces class bed + XPtr<bed>: src/bed-acc.h:18-48, src/bed-acc-xptr.cpp:40-55 */
typedef struct bsg_comm bsg_comm;   /* one rank's end of a GPU group exchanging data over NVLink peer memory (no reference twin: the
                                       reference has no multi-device path; SURVEY.md section 8e) */
typedef struct bsg_group bsg_group; /* several GPUs driven by ONE host process: column shards of one matrix + their communicators */
typedef struct bsg_view bsg_view; /* replaces bedAccScaled: (ind_row, ind_col, center, scale) resident on device, src/bed-acc.h:86-115 */

const char *bsg_last_error(void);
int bsg_version(void);
int bsg_device_count(void);

/* ---- handles ------------------------------------------------------------------------------ */
/* bedXPtr(path, n, p): src/bed-acc-xptr.cpp:14-55.  Validates the header and size exactly as the
 * reference, then stages the packed bytes to HBM once (columns [col_begin, col_end), 0-based; pass
 * 0, m for the whole file -- the range is how SNP columns are sharded across GPUs / ranks). */
int bsg_open_bed(const char *path, int n, int m, int col_begin, int col_end, int device, int layouts,
                 bsg_bed **out);
/* same, from packed bytes in host memory (m * ceil(n/4) bytes, .bed bit layout, no header) */
int bsg_open_packed(const uint8_t *packed, int n, int m, int device, int layouts, bsg_bed **out);
/* synthetic .bed generated on the device (SURVEY.md section 8d): per-SNP maf ~ U(0.02,0.5),
 * g ~ Binomial(2, maf), missing with probability na_rate; counter-based RNG keyed by (seed, global
 * column = col_offset + j), so column shards of one matrix are reproducible on any rank. */
int bsg_open_synth(int n, int m, uint64_t seed, double na_rate, int64_t col_offset, int device,
                   int layouts, bsg_bed **out);
/* LD-structured variant of the generator (SURVEY.md section 8d, AR(1)-like haplotype blocks): within every block of
 * `ld_block` consecutive global columns a haplotype's allele uniform is copied from the previous SNP with probability
 * `rho`, so neighbouring SNPs are correlated (r2 well above 0) and the clumping / r2-threshold paths have something to
 * prune.  rho = 0 reproduces bsg_open_synth bit for bit.  Same (seed, global column) keying: shards are reproducible. */
int bsg_open_synth_ld(int n, int m, uint64_t seed, double na_rate, int64_t col_offset, double rho, int ld_block,
                      int device, int layouts, bsg_bed **out);
/* FBM.code256 (bigstatsr, R/bigSNP-class.R:7,13): n x m bytes column-major + 256 doubles.  Codes
 * that round to 0/1/2/NA are repacked to 2 bits at staging and share every kernel (snp_* twins:
 * src/colstats.cpp:8-35, src/corr.cpp:113-118, src/ld-scores.cpp:93-96).  Other tables (dosages) are served by
 * fp64 kernels over the code bytes (snp_colstats, cor, LD, clumping, multLinReg); among them a "centi-dosage"
 * table -- every non-NA code within 1e-9 of v / 100, v in 0..254, one fp64 value per v (CODE_DOSAGE) -- is
 * staged as value bytes v (NA -> 255) and also serves bsg_prodvec, bsg_cprodvec, the views, bsg_randomsvd (with
 * the caller's center / scale) and bsg_prod_and_rowsumssq on the integer tensor pipe.  On such a handle the
 * products follow fp64 arithmetic over code256[byte]: an output entry whose row / column meets a selected missing
 * value is NaN (host-vector forms), the _dev forms return an all-NaN vector when a selected column holds one. */
int bsg_open_fbm256(const uint8_t *bytes, int n, int m, const double *code256, int device, int layouts,
                    bsg_bed **out);
/* the path bsg_open_fbm256 gives a code table: 0 = hard calls (2-bit engine), 1 = centi-dosage (value bytes: fp64
 * statistics + the tensor-pipe products above), 2 = other values (fp64 statistics only); -BSG_ERR_ARG for NULL */
int bsg_code256_kind(const double *code256);
void bsg_close(bsg_bed *h);
int bsg_nrow(const bsg_bed *h);
int bsg_ncol(const bsg_bed *h);
int bsg_layouts(const bsg_bed *h);
int bsg_has_na(const bsg_bed *h);
/* bytes of packed genotypes one full pass reads (ceil(n/4) * m): the roofline numerator */
int64_t bsg_packed_bytes(const bsg_bed *h);
/* copy the staged matrix back in .bed bit layout (m * ceil(n/4) bytes): round-trip check */
int bsg_export_packed(const bsg_bed *h, uint8_t *out);

/* ---- X.y and Xt.y ---------------------------------------------------------------------------- */
/* The accessor state of a call (index vectors, center, scale) is cached on the handle: a following call with the same
 * index vectors (compared by content) re-uses it; center / scale are uploaded with every call, like the reference
 * re-reads them (src/bed-prod-vec.cpp:22-23).  bsg_set_scaling_reuse(1) (or BSG_SCALING_REUSE=1) lets a call skip that
 * upload when address, length and a strided sample of 2,048 values of each vector equal the previous call's -- the shape
 * of big_randomSVD's closures (R/autoSVD.R:216-218: ~1,000 calls with identical scaling vectors).  Opt-in because a vector
 * edited in place at an unsampled position would go unnoticed. */
int bsg_set_scaling_reuse(int on);
/* bed_pMatVec4: src/bed-prod-vec.cpp:15-54.  out[nr] = X~[ind_row, ind_col] %*% x[nc] */
int bsg_prodvec(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                const double *center, const double *scale, const double *x, double *out);
/* bed_cpMatVec4: src/bed-prod-vec.cpp:59-97.  out[nc] = t(X~[ind_row, ind_col]) %*% x[nr] */
int bsg_cprodvec(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                 const double *center, const double *scale, const double *x, double *out);

/* views: the accessor state of bedAccScaled kept on the device across calls (what big_randomSVD's
 * closures re-create on every operator call in the reference, R/autoSVD.R:216-218) */
int bsg_view_create(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                    const double *center, const double *scale, bsg_view **out);
void bsg_view_destroy(bsg_view *v);
int bsg_view_prodvec(bsg_view *v, const double *x, double *out);   /* host vectors */
int bsg_view_cprodvec(bsg_view *v, const double *x, double *out);  /* host vectors */
/* device-resident vectors, enqueued on `stream` (a cudaStream_t; NULL = the legacy default stream, i.e. ordered with
 * everything the caller enqueued on stream 0 -- torch's default stream included); no sync.
 * Non-finite input: the host-vector forms above reproduce the reference's per-element Inf / NaN propagation (a zero scale
 * makes only that column's Xt.y entry NaN, src/bed-acc.h:98-111) by re-running through the accessor kernels.  The _dev
 * forms cannot look at their result: ANY non-finite x, center or 1/scale entry makes the WHOLE output NaN.  The SVD
 * drivers built on them return BSG_ERR_ARG in that case instead of iterating on NaNs. */
int bsg_view_prodvec_dev(bsg_view *v, const double *x_dev, double *out_dev, void *stream);
int bsg_view_cprodvec_dev(bsg_view *v, const double *x_dev, double *out_dev, void *stream);

/* ---- column / row statistics ------------------------------------------------------------------ */
/* bed_colstats: src/bed-fun.cpp:9-46.  n_bad = count behind the ">50% missing values" warning */
int bsg_colstats(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, double *sumX,
                 double *denoX, int *nb_nona_col, int *n_bad);
/* bed_col_counts_cpp / bed_row_counts_cpp: src/bed-fun.cpp:51-69, :72-98.  out is 4 x nc (4 x nr) */
int bsg_col_counts(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, int *out);
int bsg_row_counts(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, int *out);
/* snp_colstats: src/colstats.cpp:8-35 (FBM.code256 handles; NA handling as the reference: none) */
int bsg_snp_colstats(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, double *sumX,
                     double *denoX);

/* ---- dense decode ------------------------------------------------------------------------------ */
/* read_bed: src/bed-mat-acc.cpp:8-26 (NA -> na_val; R passes NA_INTEGER) */
int bsg_read_bed(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, int na_val,
                 int *out);
/* read_bed_scaled: src/bed-mat-acc.cpp:30-49 */
int bsg_read_bed_scaled(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                        const double *center, const double *scale, double *out);

/* ---- windowed correlations ---------------------------------------------------------------------- */
/* corMat: src/corr.cpp:11-97,102-126.  CSC pieces: p[nc+1], *i (0-based rows, ascending, diagonal
 * last), *x; the caller releases *i and *x with bsg_free.  thr has nr entries, pos has nc. */
int bsg_cor(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, double size,
            const double *thr, const double *pos, int fill_diag, int64_t *p, int **i, double **x);
/* ld_scores: src/ld-scores.cpp:11-78,83-105 */
int bsg_ld_scores(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, double size,
                  const double *pos, double *out);
void bsg_free(void *ptr);
/* bed_clumping_chr: src/clumping-bed.cpp:11-91.  ordInd = 1-based positions (within ind_col) by decreasing
 * priority; center / scale / pos per selected column; keep[nc] receives 0 / 1.  Pair statistics come from the same
 * Gram tiles as bsg_cor; the greedy sweep in rank order (the sequential part of the algorithm) runs on the host. */
int bsg_clumping_chr(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                     const double *scale, const int *ordInd, const double *pos, double size, double thr,
                     int *keep);

/* ---- FBM.code256 <-> .bed conversion (SURVEY.md section 8f row 3) ----------------------------------- */
/* _bigsnpr_readbina2: src/read-plink.cpp:61-80 (snp_readBed2, R/read-plink.R:72-111).  out = nr x nc bytes column-major, the
 * FBM.code256 codes 0 / 1 / 2 / 3 (NA) of X[ind_row, ind_col] -- what the reference writes into the .bk file. */
int bsg_readbina2(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, unsigned char *out);
/* _bigsnpr_writebina: src/write-plink.cpp:13-52 (snp_writeBed, R/write-plink.R:15-45).  Writes X[ind_row, ind_col] of a
 * bed- or FBM-staged handle as a PLINK .bed: magic bytes, then ceil(nr/4) bytes per column, byte for byte the
 * reference's output (unused slots of a column's last byte hold genotype 0). */
int bsg_writebina(bsg_bed *h, const char *path, const int *ind_row, int nr, const int *ind_col, int nc);

/* Which kernel serves the X-side products (bsg_prodvec, bsg_view_prodvec*, XV and row sums of squares):
 * 0 = automatic -- the sample-major kernel when that copy is resident, else the SNP-major kernel (k_pmvT), which
 * needs only the copy every handle has; 1 = always the SNP-major kernel.  Process-wide; no reference twin
 * (bed_prodVec has one code path, src/bed-prod-vec.cpp:15-54). */
int bsg_set_prodvec_path(int path);

/* ---- PCA projection / pcadapt (SURVEY.md section 8f row 2) ------------------------------------------- */
/* _bigsnpr_prod_and_rowSumsSq: src/bed-fun.cpp:103-133 (R: part_prod, R/bed-projectPCA.R:45-58).
 * V is nc x K column-major; XV (nr x K column-major) = X~ V and rowSumsSq[nr] = sum_j X~_ij^2 with the
 * bedAccScaled semantics (missing value -> 0).  center / scale length nc, else
 * "Incompatibility between dimensions."  On a centi-dosage FBM.code256 handle: _bigsnpr_prod_and_rowSumsSq2,
 * src/project-utils.cpp:12-43 (snp_projectSelfPCA), x = (code256[byte] - c) / s, a missing value makes its row NaN. */
int bsg_prod_and_rowsumssq(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                           const double *center, const double *scale, const double *V, int K,
                           double *XV, double *rowSumsSq);
/* _bigsnpr_multLinReg: src/multLinReg.cpp:8-88 (R: pcadapt0, R/pcadapt.R:3-27).  U is nr x K column-major;
 * tscores is nc x K column-major (the reference returns transpose(res)); NA_REAL is written as NaN.
 * Works on .bed handles and on FBM.code256 handles alike (the reference dispatches on the class, :72-92). */
int bsg_multlinreg(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *U, int K,
                   double *tscores);

/* _bigsnpr_clumping_chr: src/clumping.cpp:10-91 (snp_clumping on an FBM.code256, R/clumping.R:93-137).  Same
 * greedy sweep; the statistic is r2 = (xySum - sumX_j sumX_j0 / n)^2 / (denoX_j denoX_j0) with the caller's
 * snp_colstats vectors and no missing-value handling (a missing genotype never prunes, like the reference's NA). */
int bsg_clumping_chr_fbm(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc, const double *sumX,
                         const double *denoX, const int *ordInd, const double *pos, double size, double thr,
                         int *keep);

/* _bigsnpr_impute: src/impute-simple.cpp:10-73 (snp_fastImputeSimple, R/impute.R:189-203).  Imputes the n x m
 * CODE_012 bytes in place (any byte other than 0 / 1 / 2 is missing), streamed through `device` in column blocks.
 * method 1 mode (writes 4..6), 2 mean0 (4 + round(mean)), 3 mean2 (7 + round(100 mean), a CODE_DOSAGE code), 4 random
 * (4 + two Bernoulli(af) draws from a counter-based generator keyed by (seed, column, row); the reference uses R's
 * rbinom).  Rounding is R's fround(x, 0): half to even.  *n_all_missing (may be NULL) = columns without any non-missing
 * value: left unchanged by methods 2-4 (undefined in the reference), filled with 4 by the mode. */
int bsg_impute(uint8_t *bytes, int n, int m, int method, uint64_t seed, int device, int *n_all_missing);

/* ---- Gram product --------------------------------------------------------------------------------- */
/* bed_tcrossprodSelf's block loop collapsed into one call: R/bed-tcrossprodSelf.R:38-49 +
 * src/bed-mat-acc.cpp:30-49.  K is nr x nr; center/scale are the per-column scaling (length nc). */
int bsg_tcrossprod(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                   const double *center, const double *scale, double *K);
/* Same product, result left in the caller's DEVICE buffer K_dev (nr x nr doubles, full symmetric matrix) so
 * column shards can be summed in place by one all-reduce (SURVEY.md section 8e: GRM row). */
int bsg_tcrossprod_dev(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                       const double *center, const double *scale, double *K_dev);

/* ---- truncated SVD ----------------------------------------------------------------------------------- */
/* bed_randomSVD: R/autoSVD.R:205-219 -> bigstatsr::big_randomSVD -> RSpectra::svds.  The Lanczos
 * iteration runs on the device over the two products above.  center/scale NULL = bed_scaleBinom
 * (R/binom-scaling.R:133-142) computed on the device and returned in center_out/scale_out; a centi-dosage FBM.code256
 * handle needs the caller's center/scale (snp_scaleBinom), NULL is refused with BSG_ERR_ARG.
 * d[k], u[nr x k], v[nc x k] column-major. */
int bsg_randomsvd(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                  const double *center, const double *scale, int k, double tol, int maxit, double *d,
                  double *u, double *v, double *center_out, double *scale_out, int *niter, int *nops);

/* Ritz values that met the stopping rule in the last bsg_randomsvd / bsg_randomsvd_ex call of this thread (k when it
 * converged; fewer when `maxit` restarts were not enough -- RSpectra::svds warns in that case and so does the host
 * wrapper); -1 before any call. */
int bsg_randomsvd_nconv(void);

/* Same iteration for a matrix whose SNP columns are sharded over several handles (one per GPU / rank):
 * every rank calls it with its own shard and the same (ind_row, k, tol).  z_dev is a device buffer of nr
 * doubles owned by the caller; after each local A (A^T x) the library synchronises its stream and calls
 * reduce_cb(ctx), which must sum z_dev over the ranks (NCCL all-reduce) and return when the sum is visible
 * to the device.  ncol_total = number of columns of the whole matrix.  u is replicated, v is this rank's
 * rows. */
typedef void (*bsg_reduce_cb)(void *ctx);
int bsg_randomsvd_ex(bsg_bed *h, const int *ind_row, int nr, const int *ind_col, int nc,
                     const double *center, const double *scale, int k, double tol, int maxit, double *d,
                     double *u, double *v, double *center_out, double *scale_out, int *niter, int *nops,
                     double *z_dev, bsg_reduce_cb reduce_cb, void *ctx, int ncol_total);

/* ---- several GPUs (SURVEY.md section 8e; the reference has no multi-device path) ---------------------------------------
 * SNP columns are sharded contiguously over the GPUs (shard g = columns [g*m/G, (g+1)*m/G), first m % G shards one longer).
 * X.y ends in a sum of partial n-vectors over the shards, done INSIDE the product's epilogue kernel over NVLink peer memory;
 * Xt.y, column statistics and v need no exchange; Gram partials are summed by a two-shot all-reduce over peer memory.
 *
 * (1) one host process driving all GPUs -- what an R session is: bsg_group_*.  ind_col is a GLOBAL 1-based multiset. */
int bsg_group_open_bed(const char *path, int n, int m, const int *devices, int ndev, int layouts, bsg_group **out);
int bsg_group_open_synth(int n, int m, uint64_t seed, double na_rate, double ld_rho, int ld_block, const int *devices,
                         int ndev, int layouts, bsg_group **out);
void bsg_group_close(bsg_group *g);
int bsg_group_ndev(const bsg_group *g);
int bsg_group_nrow(const bsg_group *g);
int bsg_group_ncol(const bsg_group *g);
bsg_bed *bsg_group_shard(bsg_group *g, int i);          /* the per-device handle (statistics, counts, decode per shard) */
int bsg_group_shard_begin(const bsg_group *g, int i);   /* first global column (0-based) of shard i; i = ndev gives m */
/* bed_pMatVec4 / bed_cpMatVec4 (src/bed-prod-vec.cpp:15-54, :59-97) over the shards, host vectors, the 9-argument form */
int bsg_group_prodvec(bsg_group *g, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                      const double *scale, const double *x, double *out);
int bsg_group_cprodvec(bsg_group *g, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                       const double *scale, const double *x, double *out);
/* bed_randomSVD (R/autoSVD.R:205-219) over the shards: u[nr x k], v[nc x k] in the caller's column order */
int bsg_group_randomsvd(bsg_group *g, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                        const double *scale, int k, double tol, int maxit, double *d, double *u, double *v,
                        double *center_out, double *scale_out, int *niter, int *nops);
/* bed_tcrossprodSelf (R/bed-tcrossprodSelf.R:21-52) over the shards: K[nr x nr] on the host */
int bsg_group_tcrossprod(bsg_group *g, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                         const double *scale, double *K);

/* (2) one process per GPU (torchrun): every rank creates its end of the communicator (the 64-byte CUDA IPC handle of its
 * region comes back in handle64), the ranks exchange the handles by any means (torch.distributed all_gather) and connect.
 * max_elems = longest vector that will be reduced (n).  After that no host-side exchange happens on the data path. */
int bsg_comm_create(int rank, int world, int device, int64_t max_elems, bsg_comm **out, unsigned char *handle64);
int bsg_comm_connect(bsg_comm *c, const unsigned char *handles /* world x 64 bytes in rank order */);
void bsg_comm_destroy(bsg_comm *c);
int bsg_comm_rank(const bsg_comm *c);
int bsg_comm_world(const bsg_comm *c);
int bsg_comm_check(bsg_comm *c); /* error if a wait inside a collective timed out (a peer never arrived) */
/* in-place sum of count doubles over the ranks, enqueued on `stream`; same bits on every rank */
int bsg_comm_allreduce_dev(bsg_comm *c, double *buf_dev, int64_t count, void *stream);
/* X~ x over this rank's column shard with the sum over the ranks fused into the epilogue kernel: out_dev = full n-vector */
int bsg_view_prodvec_allreduce_dev(bsg_view *v, bsg_comm *c, const double *x_dev, double *out_dev, void *stream);
/* bed_randomSVD on a column-sharded matrix, every rank passing its shard: u, d replicated, v = this rank's rows */
int bsg_randomsvd_comm(bsg_bed *h, bsg_comm *c, const int *ind_row, int nr, const int *ind_col, int nc, const double *center,
                       const double *scale, int ncol_total, int k, double tol, int maxit, double *d, double *u, double *v,
                       double *center_out, double *scale_out, int *niter, int *nops);

/* ---- instrumentation --------------------------------------------------------------------------------- */
/* kernels launched by this library since load (the bench's gpu_launches claim) */
int64_t bsg_launch_count(void);
/* CUDA-event timing of the matvecs' dominant kernel (k_pmv), recorded on the launching stream:
 * enable with bsg_set_kernel_timing(1); after a stream synchronise bsg_last_kernel_ms() is the device
 * time of the last launch. */
int bsg_set_kernel_timing(int on);
double bsg_last_kernel_ms(void);
/* number of k_pmv launches timed since bsg_set_kernel_timing(1) (at most the last 128) and their summed
 * device time in ms; call after synchronising */
int bsg_kernel_time_stats(int *count, double *total_ms);

#ifdef __cplusplus
}
#endif
#endif /* BSGPU_H */
