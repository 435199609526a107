/*
 * bigsnpr_shim.c -- the R side of the drop-in boundary (see INTEGRATION.md).
 *
 * Replaces, inside the bigsnpr package, the generated src/RcppExports.cpp entries of the hot path and the
 * C++ files behind them (src/bed-acc-xptr.cpp, src/bed-prod-vec.cpp, src/bed-fun.cpp, src/bed-mat-acc.cpp,
 * src/corr.cpp, src/ld-scores.cpp, src/colstats.cpp).  Every function keeps the registered name and arity
 * of the reference (src/RcppExports.cpp:597-640), pulls plain pointers out of the SEXPs and calls libbsgpu
 * (include/bsgpu.h).  R's own wrappers (R/RcppExports.R, R/bed-mult-vec.R, R/binom-scaling.R, R/corr.R,
 * R/ld-scores.R) run unchanged.  `ncores` is accepted and ignored.
 *
 * Build (inside the package, needs R headers -- not available in the CUDA build image, so this file is
 * not compiled there):   PKG_LIBS = -L<dir> -lbsgpu     PKG_CPPFLAGS = -I<repo>/include
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Random.h>
#include <R_ext/Rdynload.h>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "bsgpu.h"

static void chk(int rc) {
  if (rc) Rf_error("%s", bsg_last_error()); /* same texts as the reference, e.g. "Incompatibility between dimensions." */
}

/* obj$name for RefClass objects / environments (active bindings are evaluated, R/bed-class.R:105-110) */
static SEXP field(SEXP obj, const char *name) {
  SEXP call = PROTECT(Rf_lang3(Rf_install("$"), obj, Rf_mkString(name)));
  SEXP val = Rf_eval(call, R_GlobalEnv);
  UNPROTECT(1);
  return val;
}

static void bed_finalizer(SEXP xp) {
  bsg_bed *h = (bsg_bed *)R_ExternalPtrAddr(xp);
  if (h) bsg_close(h);
  R_ClearExternalPtr(xp);
}

static int gpu_device(void) {
  /* options(bigsnpr.gpu.device = k), default 0 */
  SEXP o = Rf_GetOption1(Rf_install("bigsnpr.gpu.device"));
  return (o == R_NilValue) ? 0 : Rf_asInteger(o);
}

/* options(bigsnpr.gpu.scaling.reuse = TRUE): an unchanged center / scale pair (same R vectors as in the previous call,
 * the pattern of big_randomSVD's closures) is not uploaded again -- include/bsgpu.h, bsg_set_scaling_reuse.  Default off. */
static void apply_scaling_option(void) {
  SEXP o = Rf_GetOption1(Rf_install("bigsnpr.gpu.scaling.reuse"));
  chk(bsg_set_scaling_reuse((o == R_NilValue) ? 0 : (Rf_asInteger(o) != 0)));
}

/* _bigsnpr_bedXPtr(path, n, p): src/bed-acc-xptr.cpp:40-55.  Validation + staging to HBM. */
SEXP _bigsnpr_bedXPtr(SEXP path, SEXP n, SEXP p) {
  bsg_bed *h = NULL;
  int m = Rf_asInteger(p);
  chk(bsg_open_bed(CHAR(STRING_ELT(path, 0)), Rf_asInteger(n), m, 0, m, gpu_device(), BSG_LAYOUT_AUTO, &h));
  SEXP xp = PROTECT(R_MakeExternalPtr(h, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(xp, bed_finalizer, TRUE);
  UNPROTECT(1);
  return xp;
}

static bsg_bed *handle_of(SEXP obj_bed) {
  SEXP xp = field(obj_bed, "address"); /* lazily re-opens in PSOCK workers, R/bed-class.R:187-192 */
  bsg_bed *h = (bsg_bed *)R_ExternalPtrAddr(xp);
  if (!h) Rf_error("external pointer is not valid");
  return h;
}

/* _bigsnpr_bed_pMatVec4: src/bed-prod-vec.cpp:15-54 */
SEXP _bigsnpr_bed_pMatVec4(SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP x, SEXP ncores) {
  bsg_bed *h = handle_of(obj_bed);
  apply_scaling_option();
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col);
  if (LENGTH(center) != nc || LENGTH(scale) != nc) Rf_error("Incompatibility between dimensions.");
  SEXP out = PROTECT(Rf_allocVector(REALSXP, nr));
  chk(bsg_prodvec(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), REAL(x), REAL(out)));
  UNPROTECT(1);
  return out;
}

/* _bigsnpr_bed_cpMatVec4: src/bed-prod-vec.cpp:59-97 */
SEXP _bigsnpr_bed_cpMatVec4(SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP x, SEXP ncores) {
  bsg_bed *h = handle_of(obj_bed);
  apply_scaling_option();
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col);
  if (LENGTH(center) != nc || LENGTH(scale) != nc) Rf_error("Incompatibility between dimensions.");
  SEXP out = PROTECT(Rf_allocVector(REALSXP, nc));
  chk(bsg_cprodvec(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), REAL(x), REAL(out)));
  UNPROTECT(1);
  return out;
}

/* _bigsnpr_bed_colstats: src/bed-fun.cpp:9-46 -> list(sumX, denoX, nb_nona_col) + the >50% warning */
SEXP _bigsnpr_bed_colstats(SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP ncores) {
  bsg_bed *h = handle_of(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), n_bad = 0;
  SEXP sumX = PROTECT(Rf_allocVector(REALSXP, nc)), denoX = PROTECT(Rf_allocVector(REALSXP, nc));
  SEXP nona = PROTECT(Rf_allocVector(INTSXP, nc));
  chk(bsg_colstats(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(sumX), REAL(denoX), INTEGER(nona), &n_bad));
  if (n_bad > 0) Rf_warning("%d variants have >50%% missing values.", n_bad);
  SEXP res = PROTECT(Rf_allocVector(VECSXP, 3)), nm = PROTECT(Rf_allocVector(STRSXP, 3));
  SET_VECTOR_ELT(res, 0, sumX); SET_VECTOR_ELT(res, 1, denoX); SET_VECTOR_ELT(res, 2, nona);
  SET_STRING_ELT(nm, 0, Rf_mkChar("sumX")); SET_STRING_ELT(nm, 1, Rf_mkChar("denoX"));
  SET_STRING_ELT(nm, 2, Rf_mkChar("nb_nona_col"));
  Rf_setAttrib(res, R_NamesSymbol, nm);
  UNPROTECT(5);
  return res;
}

/* _bigsnpr_bed_col_counts_cpp / _bigsnpr_bed_row_counts_cpp: src/bed-fun.cpp:51-69, :72-98 */
static SEXP counts(SEXP obj_bed, SEXP ind_row, SEXP ind_col, int byrow) {
  bsg_bed *h = handle_of(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), k = byrow ? nr : nc;
  SEXP res = PROTECT(Rf_allocMatrix(INTSXP, 4, k));
  chk((byrow ? bsg_row_counts : bsg_col_counts)(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, INTEGER(res)));
  UNPROTECT(1);
  return res;
}
SEXP _bigsnpr_bed_col_counts_cpp(SEXP o, SEXP r, SEXP c, SEXP ncores) { return counts(o, r, c, 0); }
SEXP _bigsnpr_bed_row_counts_cpp(SEXP o, SEXP r, SEXP c, SEXP ncores) { return counts(o, r, c, 1); }

/* _bigsnpr_read_bed: src/bed-mat-acc.cpp:8-26 */
SEXP _bigsnpr_read_bed(SEXP obj_bed, SEXP ind_row, SEXP ind_col) {
  bsg_bed *h = handle_of(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col);
  SEXP res = PROTECT(Rf_allocMatrix(INTSXP, nr, nc));
  chk(bsg_read_bed(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, NA_INTEGER, INTEGER(res)));
  UNPROTECT(1);
  return res;
}

/* _bigsnpr_read_bed_scaled: src/bed-mat-acc.cpp:30-49 */
SEXP _bigsnpr_read_bed_scaled(SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale) {
  bsg_bed *h = handle_of(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col);
  if (LENGTH(center) != nc || LENGTH(scale) != nc) Rf_error("Incompatibility between dimensions.");
  SEXP res = PROTECT(Rf_allocMatrix(REALSXP, nr, nc));
  chk(bsg_read_bed_scaled(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), REAL(res)));
  UNPROTECT(1);
  return res;
}

/* bigstatsr's FBM objects (RefClass environments) expose `$backingfile` (the .bk file: nrow x ncol elements of the FBM's
 * type, column-major, no header), `$nrow`, `$ncol` and, for FBM.code256, `$code256`.  The shim maps that file itself
 * (the reference reaches the same bytes through bigstatsr's C++ accessor, src/corr.cpp:113-118), so it depends on no
 * bigstatsr header or symbol.  Writable maps serve the in-place outputs of the reference: the integer FBM `keep` of the
 * clumping routines (R/clumping.R:115, R/bed-clumping.R:51) and the FBM.code256 filled by readbina2. */
static void *fbm_map(SEXP obj, size_t elt_size, int writable, size_t *bytes_out) {
  SEXP bf = field(obj, "backingfile");
  if (TYPEOF(bf) != STRSXP || LENGTH(bf) < 1) Rf_error("object has no backing file");
  const char *path = CHAR(STRING_ELT(bf, 0));
  size_t want = (size_t)Rf_asInteger(field(obj, "nrow")) * (size_t)Rf_asInteger(field(obj, "ncol")) * elt_size;
  int fd = open(path, writable ? O_RDWR : O_RDONLY);
  if (fd < 0) Rf_error("Error when mapping file:\n  %s.\n", path);
  struct stat st;
  if (fstat(fd, &st) != 0 || (size_t)st.st_size < want) {
    close(fd);
    Rf_error("Inconsistency between size of backingfile and dimensions.");
  }
  void *p = want ? mmap(NULL, want, writable ? (PROT_READ | PROT_WRITE) : PROT_READ, MAP_SHARED, fd, 0) : NULL;
  close(fd);
  if (want && p == MAP_FAILED) Rf_error("Error when mapping file:\n  %s.\n", path);
  *bytes_out = want;
  return p;
}
static void fbm_unmap(void *p, size_t bytes, int writable) {
  if (!p || !bytes) return;
  if (writable) msync(p, bytes, MS_SYNC); /* R reads the result through its own mapping of the same file */
  munmap(p, bytes);
}

/* FBM.code256 objects (snp_cor / snp_ld_scores / snp_colstats / snp_clumping / snp_pcadapt / snp_writeBed): the n x m
 * bytes are staged to HBM once per object; the handle is cached in the environment (variable ".bsg"). */
static bsg_bed *fbm_handle_of(SEXP obj) {
  SEXP cached = Rf_findVarInFrame(obj, Rf_install(".bsg"));
  if (cached != R_UnboundValue && TYPEOF(cached) == EXTPTRSXP && R_ExternalPtrAddr(cached))
    return (bsg_bed *)R_ExternalPtrAddr(cached);
  int n = Rf_asInteger(field(obj, "nrow")), m = Rf_asInteger(field(obj, "ncol"));
  SEXP code = PROTECT(Rf_coerceVector(field(obj, "code256"), REALSXP));
  if (LENGTH(code) != 256) Rf_error("'code256' must have 256 values.");
  size_t bytes = 0;
  void *raw = fbm_map(obj, 1, 0, &bytes);
  bsg_bed *h = NULL;
  int rc = bsg_open_fbm256((const uint8_t *)raw, n, m, REAL(code), gpu_device(), BSG_LAYOUT_SNP_MAJOR, &h);
  fbm_unmap(raw, bytes, 0);
  chk(rc);
  SEXP xp = PROTECT(R_MakeExternalPtr(h, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(xp, bed_finalizer, TRUE);
  Rf_defineVar(Rf_install(".bsg"), xp, obj);
  UNPROTECT(2);
  return h;
}

static int has_field(SEXP obj, const char *name) { return Rf_findVarInFrame(obj, Rf_install(name)) != R_UnboundValue; }

/* dispatch of src/corr.cpp:113-125: "code256" -> FBM, "bedfile" -> bed, else "Unknown object type." */
static bsg_bed *any_handle(SEXP obj) {
  if (has_field(obj, "code256")) return fbm_handle_of(obj);
  if (has_field(obj, "bedfile")) return handle_of(obj);
  Rf_error("Unknown object type.");
  return NULL;
}

/* _bigsnpr_snp_colstats: src/colstats.cpp:8-35 */
SEXP _bigsnpr_snp_colstats(SEXP BM, SEXP rowInd, SEXP colInd, SEXP ncores) {
  bsg_bed *h = fbm_handle_of(BM);
  int nr = LENGTH(rowInd), nc = LENGTH(colInd);
  SEXP sumX = PROTECT(Rf_allocVector(REALSXP, nc)), denoX = PROTECT(Rf_allocVector(REALSXP, nc));
  chk(bsg_snp_colstats(h, INTEGER(rowInd), nr, INTEGER(colInd), nc, REAL(sumX), REAL(denoX)));
  SEXP res = PROTECT(Rf_allocVector(VECSXP, 2)), nm = PROTECT(Rf_allocVector(STRSXP, 2));
  SET_VECTOR_ELT(res, 0, sumX); SET_VECTOR_ELT(res, 1, denoX);
  SET_STRING_ELT(nm, 0, Rf_mkChar("sumX")); SET_STRING_ELT(nm, 1, Rf_mkChar("denoX"));
  Rf_setAttrib(res, R_NamesSymbol, nm);
  UNPROTECT(4);
  return res;
}

/* _bigsnpr_corMat: src/corr.cpp:102-126 -> list of m lists {i, x} (R/corr.R:43-47 assembles the dsCMatrix) */
SEXP _bigsnpr_corMat(SEXP obj, SEXP rowInd, SEXP colInd, SEXP size, SEXP thr, SEXP pos, SEXP fill_diag, SEXP ncores) {
  int nr = LENGTH(rowInd), nc = LENGTH(colInd);
  if (LENGTH(pos) != nc) Rf_error("Incompatibility between dimensions.");
  bsg_bed *h = any_handle(obj);
  int64_t *p = (int64_t *)R_alloc((size_t)nc + 1, sizeof(int64_t));
  int *ci = NULL;
  double *cx = NULL;
  chk(bsg_cor(h, INTEGER(rowInd), nr, INTEGER(colInd), nc, Rf_asReal(size), REAL(thr), REAL(pos), Rf_asLogical(fill_diag),
              p, &ci, &cx));
  SEXP res = PROTECT(Rf_allocVector(VECSXP, nc));
  SEXP nm = PROTECT(Rf_allocVector(STRSXP, 2));
  SET_STRING_ELT(nm, 0, Rf_mkChar("i")); SET_STRING_ELT(nm, 1, Rf_mkChar("x"));
  for (int j = 0; j < nc; j++) {
    int len = (int)(p[j + 1] - p[j]);
    SEXP el = PROTECT(Rf_allocVector(VECSXP, 2)), vi = PROTECT(Rf_allocVector(INTSXP, len));
    SEXP vx = PROTECT(Rf_allocVector(REALSXP, len));
    for (int k = 0; k < len; k++) { INTEGER(vi)[k] = ci[p[j] + k]; REAL(vx)[k] = cx[p[j] + k]; }
    SET_VECTOR_ELT(el, 0, vi); SET_VECTOR_ELT(el, 1, vx);
    Rf_setAttrib(el, R_NamesSymbol, nm);
    SET_VECTOR_ELT(res, j, el);
    UNPROTECT(3);
  }
  bsg_free(ci); bsg_free(cx);
  UNPROTECT(2);
  return res;
}

/* _bigsnpr_ld_scores: src/ld-scores.cpp:83-105 */
SEXP _bigsnpr_ld_scores(SEXP obj, SEXP rowInd, SEXP colInd, SEXP size, SEXP pos, SEXP ncores) {
  int nr = LENGTH(rowInd), nc = LENGTH(colInd);
  if (LENGTH(pos) != nc) Rf_error("Incompatibility between dimensions.");
  bsg_bed *h = any_handle(obj);
  SEXP out = PROTECT(Rf_allocVector(REALSXP, nc));
  chk(bsg_ld_scores(h, INTEGER(rowInd), nr, INTEGER(colInd), nc, Rf_asReal(size), REAL(pos), REAL(out)));
  UNPROTECT(1);
  return out;
}

/* _bigsnpr_bed_clumping_chr: src/clumping-bed.cpp:11-91 (12 arguments).  BM2 is the 1 x nc integer FBM `keep`
 * (R/bed-clumping.R:51), written in place through its backing file; rankInd is implied by ordInd. */
SEXP _bigsnpr_bed_clumping_chr(SEXP obj_bed, SEXP BM2, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP ordInd,
                               SEXP rankInd, SEXP pos, SEXP size, SEXP thr, SEXP ncores) {
  bsg_bed *h = handle_of(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col);
  if (LENGTH(center) != nc || LENGTH(scale) != nc || LENGTH(pos) != nc || LENGTH(ordInd) != nc)
    Rf_error("Incompatibility between dimensions.");
  size_t bytes = 0;
  int *keep = (int *)fbm_map(BM2, sizeof(int), 1, &bytes);
  if (bytes < (size_t)nc * sizeof(int)) { fbm_unmap(keep, bytes, 1); Rf_error("Incompatibility between dimensions."); }
  int rc = bsg_clumping_chr(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), INTEGER(ordInd), REAL(pos),
                            Rf_asReal(size), Rf_asReal(thr), keep);
  fbm_unmap(keep, bytes, 1);
  chk(rc);
  return R_NilValue;
}

/* _bigsnpr_clumping_chr: src/clumping.cpp:10-91 (12 arguments; BM is the FBM.code256 environment, src/clumping.cpp:24-25) */
SEXP _bigsnpr_clumping_chr(SEXP BM, SEXP BM2, SEXP rowInd, SEXP colInd, SEXP ordInd, SEXP rankInd, SEXP pos, SEXP sumX,
                           SEXP denoX, SEXP size, SEXP thr, SEXP ncores) {
  bsg_bed *h = fbm_handle_of(BM);
  int nr = LENGTH(rowInd), nc = LENGTH(colInd);
  if (LENGTH(sumX) != nc || LENGTH(denoX) != nc || LENGTH(pos) != nc || LENGTH(ordInd) != nc)
    Rf_error("Incompatibility between dimensions.");
  size_t bytes = 0;
  int *keep = (int *)fbm_map(BM2, sizeof(int), 1, &bytes);
  if (bytes < (size_t)nc * sizeof(int)) { fbm_unmap(keep, bytes, 1); Rf_error("Incompatibility between dimensions."); }
  int rc = bsg_clumping_chr_fbm(h, INTEGER(rowInd), nr, INTEGER(colInd), nc, REAL(sumX), REAL(denoX), INTEGER(ordInd), REAL(pos),
                                Rf_asReal(size), Rf_asReal(thr), keep);
  fbm_unmap(keep, bytes, 1);
  chk(rc);
  return R_NilValue;
}

/* _bigsnpr_readbina2: src/read-plink.cpp:61-80 (5 arguments; BM is the destination FBM.code256, filled in place; the R
 * wrapper creates it with exactly length(ind_row) x length(ind_col) bytes, R/read-plink.R:93-100) */
SEXP _bigsnpr_readbina2(SEXP BM, SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP ncores) {
  bsg_bed *h = handle_of(obj_bed);
  size_t bytes = 0, want = (size_t)LENGTH(ind_row) * (size_t)LENGTH(ind_col);
  unsigned char *dst = (unsigned char *)fbm_map(BM, 1, 1, &bytes);
  if (bytes != want) { fbm_unmap(dst, bytes, 1); Rf_error("Incompatibility between dimensions."); }
  int rc = bsg_readbina2(h, INTEGER(ind_row), LENGTH(ind_row), INTEGER(ind_col), LENGTH(ind_col), dst);
  fbm_unmap(dst, bytes, 1);
  chk(rc);
  return R_NilValue;
}

/* _bigsnpr_writebina: src/write-plink.cpp:13-52 (5 arguments; BM is the FBM.code256 of the bigSNP, src/write-plink.cpp:19-20;
 * `tab` = getInverseCode() is implied by the library) */
SEXP _bigsnpr_writebina(SEXP filename, SEXP BM, SEXP tab, SEXP rowInd, SEXP colInd) {
  bsg_bed *h = fbm_handle_of(BM);
  chk(bsg_writebina(h, CHAR(STRING_ELT(filename, 0)), INTEGER(rowInd), LENGTH(rowInd), INTEGER(colInd), LENGTH(colInd)));
  return R_NilValue;
}

/* _bigsnpr_prod_and_rowSumsSq: src/bed-fun.cpp:103-133 (6 arguments) -> list(XV, rowSumsSq) */
SEXP _bigsnpr_prod_and_rowSumsSq(SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP V) {
  bsg_bed *h = handle_of(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), K = Rf_ncols(V);
  if (LENGTH(center) != nc || LENGTH(scale) != nc || Rf_nrows(V) != nc) Rf_error("Incompatibility between dimensions.");
  SEXP XV = PROTECT(Rf_allocMatrix(REALSXP, nr, K)), rss = PROTECT(Rf_allocVector(REALSXP, nr));
  chk(bsg_prod_and_rowsumssq(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), REAL(V), K, REAL(XV),
                             REAL(rss)));
  SEXP res = PROTECT(Rf_allocVector(VECSXP, 2));
  SET_VECTOR_ELT(res, 0, XV);
  SET_VECTOR_ELT(res, 1, rss);
  UNPROTECT(3);
  return res;
}

/* _bigsnpr_prod_and_rowSumsSq2: src/project-utils.cpp:12-43 (6 arguments; snp_projectSelfPCA, R/bed-projectPCA.R:229-270)
 * -> list(XV, rowSumsSq) on an FBM.code256 environment (centi-dosage codes: include/bsgpu.h) */
SEXP _bigsnpr_prod_and_rowSumsSq2(SEXP BM, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP V) {
  bsg_bed *h = fbm_handle_of(BM);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), K = Rf_ncols(V);
  if (LENGTH(center) != nc || LENGTH(scale) != nc || Rf_nrows(V) != nc) Rf_error("Incompatibility between dimensions.");
  SEXP XV = PROTECT(Rf_allocMatrix(REALSXP, nr, K)), rss = PROTECT(Rf_allocVector(REALSXP, nr));
  chk(bsg_prod_and_rowsumssq(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), REAL(V), K, REAL(XV),
                             REAL(rss)));
  for (R_xlen_t i = 0; i < XLENGTH(XV); i++)
    if (ISNAN(REAL(XV)[i])) REAL(XV)[i] = NA_REAL; /* a missing dosage: NA_real_ like bigstatsr's accessor */
  for (int i = 0; i < nr; i++)
    if (ISNAN(REAL(rss)[i])) REAL(rss)[i] = NA_REAL;
  SEXP res = PROTECT(Rf_allocVector(VECSXP, 2));
  SET_VECTOR_ELT(res, 0, XV);
  SET_VECTOR_ELT(res, 1, rss);
  UNPROTECT(3);
  return res;
}

/* _bigsnpr_impute: src/impute-simple.cpp:10-73 (3 arguments; snp_fastImputeSimple, R/impute.R:189-203).  The bytes of the
 * FBM.code256 are imputed in place through a shared writable mapping of its backing file; the seed of the random method
 * comes from R's RNG (set.seed reproduces it).  A staged copy of the object is dropped: its bytes changed. */
SEXP _bigsnpr_impute(SEXP BM, SEXP method, SEXP ncores) {
  int n = Rf_asInteger(field(BM, "nrow")), m = Rf_asInteger(field(BM, "ncol")), meth = Rf_asInteger(method), n_all = 0;
  GetRNGstate();
  const uint64_t seed = ((uint64_t)(unif_rand() * 4294967296.0) << 32) | (uint64_t)(unif_rand() * 4294967296.0);
  PutRNGstate();
  size_t bytes = 0;
  uint8_t *p = (uint8_t *)fbm_map(BM, 1, 1, &bytes);
  int rc = bsg_impute(p, n, m, meth, seed, gpu_device(), &n_all);
  fbm_unmap(p, bytes, 1);
  Rf_defineVar(Rf_install(".bsg"), R_NilValue, BM);
  chk(rc);
  return R_NilValue;
}

/* _bigsnpr_multLinReg: src/multLinReg.cpp:64-88 (5 arguments; `obj` is a bed or an FBM.code256 environment) */
SEXP _bigsnpr_multLinReg(SEXP obj, SEXP ind_row, SEXP ind_col, SEXP U, SEXP ncores) {
  bsg_bed *h = any_handle(obj); /* src/multLinReg.cpp:72-78: FBM.code256 or bed, else "Unknown object type." */
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), K = Rf_ncols(U);
  if (Rf_nrows(U) != nr) Rf_error("Incompatibility between dimensions.");
  SEXP t = PROTECT(Rf_allocMatrix(REALSXP, nc, K));
  chk(bsg_multlinreg(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(U), K, REAL(t)));
  for (R_xlen_t i = 0; i < XLENGTH(t); i++)
    if (ISNAN(REAL(t)[i])) REAL(t)[i] = NA_REAL; /* the library writes NaN where the reference writes NA_REAL */
  UNPROTECT(1);
  return t;
}

/* new entry points: R/bed-tcrossprodSelf.R's block loop and R/autoSVD.R's bed_randomSVD collapse to one call each */
SEXP _bigsnpr_bed_tcrossprod_gpu(SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale) {
  bsg_bed *h = handle_of(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col);
  SEXP K = PROTECT(Rf_allocMatrix(REALSXP, nr, nr));
  chk(bsg_tcrossprod(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), REAL(K)));
  UNPROTECT(1);
  return K;
}

/* obj_bed: a bed environment, or an FBM.code256 one with centi-dosage codes and the caller's center / scale (bed_scaleBinom
 * needs hard calls) */
SEXP _bigsnpr_bed_randomSVD_gpu(SEXP obj_bed, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP k, SEXP tol) {
  bsg_bed *h = any_handle(obj_bed);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), kk = Rf_asInteger(k), niter = 0, nops = 0;
  SEXP d = PROTECT(Rf_allocVector(REALSXP, kk)), u = PROTECT(Rf_allocMatrix(REALSXP, nr, kk));
  SEXP v = PROTECT(Rf_allocMatrix(REALSXP, nc, kk));
  SEXP co = PROTECT(Rf_allocVector(REALSXP, nc)), so = PROTECT(Rf_allocVector(REALSXP, nc));
  const double *cen = (center == R_NilValue) ? NULL : REAL(center), *sca = (scale == R_NilValue) ? NULL : REAL(scale);
  chk(bsg_randomsvd(h, INTEGER(ind_row), nr, INTEGER(ind_col), nc, cen, sca, kk, Rf_asReal(tol), 1000, REAL(d), REAL(u),
                    REAL(v), REAL(co), REAL(so), &niter, &nops));
  const char *names[] = {"d", "u", "v", "niter", "nops", "center", "scale", ""};
  SEXP res = PROTECT(Rf_mkNamed(VECSXP, names));
  SET_VECTOR_ELT(res, 0, d); SET_VECTOR_ELT(res, 1, u); SET_VECTOR_ELT(res, 2, v);
  SET_VECTOR_ELT(res, 3, Rf_ScalarInteger(niter)); SET_VECTOR_ELT(res, 4, Rf_ScalarInteger(nops));
  SET_VECTOR_ELT(res, 5, co); SET_VECTOR_ELT(res, 6, so);
  Rf_setAttrib(res, R_ClassSymbol, Rf_mkString("big_SVD"));
  UNPROTECT(6);
  return res;
}

/* ---- several GPUs from the one R process (SURVEY.md section 8e): options(bigsnpr.gpu.devices = c(0, 1, ...)) --------------
 * A group handle shards the file's SNP columns over the listed devices; the two new symbols mirror the single-GPU ones. */
static void group_finalizer(SEXP xp) {
  bsg_group *g = (bsg_group *)R_ExternalPtrAddr(xp);
  if (g) bsg_group_close(g);
  R_ClearExternalPtr(xp);
}
SEXP _bigsnpr_bed_group_gpu(SEXP path, SEXP n, SEXP p, SEXP devices) {
  bsg_group *g = NULL;
  chk(bsg_group_open_bed(CHAR(STRING_ELT(path, 0)), Rf_asInteger(n), Rf_asInteger(p), INTEGER(devices), LENGTH(devices),
                         BSG_LAYOUT_AUTO, &g));
  SEXP xp = PROTECT(R_MakeExternalPtr(g, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(xp, group_finalizer, TRUE);
  UNPROTECT(1);
  return xp;
}
static bsg_group *group_of(SEXP xp) {
  bsg_group *g = (TYPEOF(xp) == EXTPTRSXP) ? (bsg_group *)R_ExternalPtrAddr(xp) : NULL;
  if (!g) Rf_error("external pointer is not valid");
  return g;
}
SEXP _bigsnpr_group_pMatVec4_gpu(SEXP grp, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP x, SEXP transpose) {
  bsg_group *g = group_of(grp);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), tr = Rf_asLogical(transpose);
  if (LENGTH(center) != nc || LENGTH(scale) != nc || LENGTH(x) != (tr ? nr : nc)) Rf_error("Incompatibility between dimensions.");
  SEXP out = PROTECT(Rf_allocVector(REALSXP, tr ? nc : nr));
  chk((tr ? bsg_group_cprodvec : bsg_group_prodvec)(g, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale),
                                                    REAL(x), REAL(out)));
  UNPROTECT(1);
  return out;
}
SEXP _bigsnpr_group_randomSVD_gpu(SEXP grp, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale, SEXP k, SEXP tol) {
  bsg_group *g = group_of(grp);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col), kk = Rf_asInteger(k), niter = 0, nops = 0;
  SEXP d = PROTECT(Rf_allocVector(REALSXP, kk)), u = PROTECT(Rf_allocMatrix(REALSXP, nr, kk));
  SEXP v = PROTECT(Rf_allocMatrix(REALSXP, nc, kk));
  SEXP co = PROTECT(Rf_allocVector(REALSXP, nc)), so = PROTECT(Rf_allocVector(REALSXP, nc));
  const double *cen = (center == R_NilValue) ? NULL : REAL(center), *sca = (scale == R_NilValue) ? NULL : REAL(scale);
  chk(bsg_group_randomsvd(g, INTEGER(ind_row), nr, INTEGER(ind_col), nc, cen, sca, kk, Rf_asReal(tol), 1000, REAL(d), REAL(u),
                          REAL(v), REAL(co), REAL(so), &niter, &nops));
  const char *names[] = {"d", "u", "v", "niter", "nops", "center", "scale", ""};
  SEXP res = PROTECT(Rf_mkNamed(VECSXP, names));
  SET_VECTOR_ELT(res, 0, d); SET_VECTOR_ELT(res, 1, u); SET_VECTOR_ELT(res, 2, v);
  SET_VECTOR_ELT(res, 3, Rf_ScalarInteger(niter)); SET_VECTOR_ELT(res, 4, Rf_ScalarInteger(nops));
  SET_VECTOR_ELT(res, 5, co); SET_VECTOR_ELT(res, 6, so);
  Rf_setAttrib(res, R_ClassSymbol, Rf_mkString("big_SVD"));
  UNPROTECT(6);
  return res;
}
SEXP _bigsnpr_group_tcrossprod_gpu(SEXP grp, SEXP ind_row, SEXP ind_col, SEXP center, SEXP scale) {
  bsg_group *g = group_of(grp);
  int nr = LENGTH(ind_row), nc = LENGTH(ind_col);
  if (LENGTH(center) != nc || LENGTH(scale) != nc) Rf_error("Incompatibility between dimensions.");
  SEXP K = PROTECT(Rf_allocMatrix(REALSXP, nr, nr));
  chk(bsg_group_tcrossprod(g, INTEGER(ind_row), nr, INTEGER(ind_col), nc, REAL(center), REAL(scale), REAL(K)));
  UNPROTECT(1);
  return K;
}

/* registration: same table shape as src/RcppExports.cpp:597-640 (only the hot-path rows shown; the other
 * entries of the reference stay as generated) */
static const R_CallMethodDef CallEntries[] = {
    {"_bigsnpr_bedXPtr", (DL_FUNC)&_bigsnpr_bedXPtr, 3},
    {"_bigsnpr_bed_colstats", (DL_FUNC)&_bigsnpr_bed_colstats, 4},
    {"_bigsnpr_bed_col_counts_cpp", (DL_FUNC)&_bigsnpr_bed_col_counts_cpp, 4},
    {"_bigsnpr_bed_row_counts_cpp", (DL_FUNC)&_bigsnpr_bed_row_counts_cpp, 4},
    {"_bigsnpr_read_bed", (DL_FUNC)&_bigsnpr_read_bed, 3},
    {"_bigsnpr_read_bed_scaled", (DL_FUNC)&_bigsnpr_read_bed_scaled, 5},
    {"_bigsnpr_bed_pMatVec4", (DL_FUNC)&_bigsnpr_bed_pMatVec4, 7},
    {"_bigsnpr_bed_cpMatVec4", (DL_FUNC)&_bigsnpr_bed_cpMatVec4, 7},
    {"_bigsnpr_snp_colstats", (DL_FUNC)&_bigsnpr_snp_colstats, 4},
    {"_bigsnpr_corMat", (DL_FUNC)&_bigsnpr_corMat, 8},
    {"_bigsnpr_ld_scores", (DL_FUNC)&_bigsnpr_ld_scores, 6},
    {"_bigsnpr_bed_clumping_chr", (DL_FUNC)&_bigsnpr_bed_clumping_chr, 12},
    {"_bigsnpr_clumping_chr", (DL_FUNC)&_bigsnpr_clumping_chr, 12},
    {"_bigsnpr_readbina2", (DL_FUNC)&_bigsnpr_readbina2, 5},
    {"_bigsnpr_writebina", (DL_FUNC)&_bigsnpr_writebina, 5},
    {"_bigsnpr_prod_and_rowSumsSq", (DL_FUNC)&_bigsnpr_prod_and_rowSumsSq, 6},
    {"_bigsnpr_multLinReg", (DL_FUNC)&_bigsnpr_multLinReg, 5},
    {"_bigsnpr_prod_and_rowSumsSq2", (DL_FUNC)&_bigsnpr_prod_and_rowSumsSq2, 6},
    {"_bigsnpr_impute", (DL_FUNC)&_bigsnpr_impute, 3},
    {"_bigsnpr_bed_tcrossprod_gpu", (DL_FUNC)&_bigsnpr_bed_tcrossprod_gpu, 5},
    {"_bigsnpr_bed_randomSVD_gpu", (DL_FUNC)&_bigsnpr_bed_randomSVD_gpu, 7},
    {"_bigsnpr_bed_group_gpu", (DL_FUNC)&_bigsnpr_bed_group_gpu, 4},
    {"_bigsnpr_group_pMatVec4_gpu", (DL_FUNC)&_bigsnpr_group_pMatVec4_gpu, 7},
    {"_bigsnpr_group_randomSVD_gpu", (DL_FUNC)&_bigsnpr_group_randomSVD_gpu, 7},
    {"_bigsnpr_group_tcrossprod_gpu", (DL_FUNC)&_bigsnpr_group_tcrossprod_gpu, 5},
    {NULL, NULL, 0}};

void R_init_bigsnpr_hotpath(DllInfo *dll) {
  /* in the package this table is merged into R_init_bigsnpr (src/RcppExports.cpp:637-640) */
  R_registerRoutines(dll, NULL, CallEntries, NULL, NULL);
  R_useDynamicSymbols(dll, FALSE);
}
