"""CPU oracle for the bigsnpr hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package ``bigsnpr_b200`` never does.

Two layers:

* thin ctypes wrappers over ``oracle/_build/libbsg_oracle.so`` (``bsg_oracle.c``: literal scalar C
  restatement of the reference's C++ loops, each function citing the reference file:line);
* NumPy restatements of the reference's *R-level* glue (thresholds of ``cor0``, ``bed_scaleBinom``,
  ``bed_MAF``, the ``bed_tcrossprodSelf`` block loop, ``getCode`` / ``getInverseCode``), again citing
  file:line under ``/root/reference``.

Index conventions follow R: ``ind_row`` / ``ind_col`` are **1-based** int32 arrays.

Parity pin: ``tests/test_oracle.py`` checks this oracle against the reference's own fixtures
(``example.bed``, ``example-missing.bed``, ``example.ld``; SURVEY.md section 8c).  The reference cannot be
built here (no R / Rcpp / bigstatsr), so there is no ``oracle/_ref``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libbsg_oracle.so")

ERR_MSG = {
    1: "Incompatibility between dimensions.",
    2: "Tested subscript out of bounds.",
    3: "File is not a binary PED file.",
    4: "Variant-major is the only mode supported.",
    5: "n or p does not match the dimensions of the file.",
    6: "Error when mapping file.",
    7: "allocation failure",
}


class OracleError(RuntimeError):
    pass


def stale() -> bool:
    src = os.path.join(_HERE, "bsg_oracle.c")
    return (not os.path.exists(_SO)) or os.path.getmtime(_SO) < os.path.getmtime(src)


def build(force: bool = False) -> str:
    """Compile ``bsg_oracle.c`` (gcc -O2 -fopenmp) if the shared object is missing or stale."""
    if force or stale():
        subprocess.check_call(["make", "-s", "-C", _HERE])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.orc_max_threads.restype = C.c_int
    return _lib


def max_threads() -> int:
    return int(lib().orc_max_threads())


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _chk(rc):
    if rc:
        raise OracleError(ERR_MSG.get(rc, "error %d" % rc))


class OracleBed:
    """Host-side ``bed`` handle of the oracle (reference: src/bed-acc.h:18-48, src/bed-acc-xptr.cpp:14-34)."""

    def __init__(self, path: str, n: int | None = None, m: int | None = None):
        self.bedfile = path
        if n is None or m is None:
            pre = path[:-4]
            n = sum(1 for _ in open(pre + ".fam"))
            m = sum(1 for _ in open(pre + ".bim"))
        self.nrow, self.ncol = int(n), int(m)
        _chk(lib().orc_bed_validate(path.encode(), C.c_int(self.nrow), C.c_int(self.ncol)))
        raw = np.fromfile(path, dtype=np.uint8)
        self.bytes = np.ascontiguousarray(raw[3:])
        self.n_byte = (self.nrow + 3) // 4

    @classmethod
    def from_packed(cls, packed: np.ndarray, n: int, m: int) -> "OracleBed":
        """Wrap an in-memory packed matrix (m x ceil(n/4) bytes, no header)."""
        self = cls.__new__(cls)
        self.bedfile = "<memory>"
        self.nrow, self.ncol = int(n), int(m)
        self.n_byte = (n + 3) // 4
        self.bytes = np.ascontiguousarray(packed, dtype=np.uint8).reshape(-1)
        assert self.bytes.size == self.n_byte * m
        return self

    def rows_along(self):
        return np.arange(1, self.nrow + 1, dtype=np.int32)

    def cols_along(self):
        return np.arange(1, self.ncol + 1, dtype=np.int32)


def _defaults(obj, ind_row, ind_col):
    ind_row = obj.rows_along() if ind_row is None else _i32(ind_row)
    ind_col = obj.cols_along() if ind_col is None else _i32(ind_col)
    return ind_row, ind_col


# ----------------------------------------------------------------------------------------------
# C-level entry points (the .Call layer of the reference)
# ----------------------------------------------------------------------------------------------
def bed_pMatVec4(obj, ind_row, ind_col, center, scale, x, ncores=1):
    """src/bed-prod-vec.cpp:15-54."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    center, scale, x = _f64(center), _f64(scale), _f64(x)
    if center.size != ind_col.size or scale.size != ind_col.size:
        raise OracleError(ERR_MSG[1])
    out = np.empty(ind_row.size, dtype=np.float64)
    _chk(lib().orc_pMatVec4(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(ind_row, C.c_int),
                            ind_row.size, _p(ind_col, C.c_int), ind_col.size, _p(center, C.c_double),
                            _p(scale, C.c_double), _p(x, C.c_double), int(ncores), _p(out, C.c_double)))
    return out


def bed_cpMatVec4(obj, ind_row, ind_col, center, scale, x, ncores=1):
    """src/bed-prod-vec.cpp:59-97."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    center, scale, x = _f64(center), _f64(scale), _f64(x)
    if center.size != ind_col.size or scale.size != ind_col.size:
        raise OracleError(ERR_MSG[1])
    out = np.empty(ind_col.size, dtype=np.float64)
    _chk(lib().orc_cpMatVec4(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(ind_row, C.c_int),
                             ind_row.size, _p(ind_col, C.c_int), ind_col.size, _p(center, C.c_double),
                             _p(scale, C.c_double), _p(x, C.c_double), int(ncores), _p(out, C.c_double)))
    return out


def bed_colstats(obj, ind_row, ind_col, ncores=1):
    """src/bed-fun.cpp:9-46 -> dict(sumX, denoX, nb_nona_col, n_bad)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    m = ind_col.size
    sumX, denoX = np.empty(m), np.empty(m)
    nb = np.empty(m, dtype=np.int32)
    n_bad = C.c_int(0)
    with np.errstate(all="ignore"):
        _chk(lib().orc_bed_colstats(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(ind_row, C.c_int),
                                    ind_row.size, _p(ind_col, C.c_int), m, int(ncores),
                                    _p(sumX, C.c_double), _p(denoX, C.c_double), _p(nb, C.c_int),
                                    C.byref(n_bad)))
    return {"sumX": sumX, "denoX": denoX, "nb_nona_col": nb, "n_bad": n_bad.value}


def bed_col_counts_cpp(obj, ind_row, ind_col, ncores=1):
    """src/bed-fun.cpp:51-69 -> int32 (4, nc)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    res = np.zeros((ind_col.size, 4), dtype=np.int32)
    _chk(lib().orc_bed_col_counts(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(ind_row, C.c_int),
                                  ind_row.size, _p(ind_col, C.c_int), ind_col.size, int(ncores),
                                  _p(res, C.c_int)))
    return res.T


def bed_row_counts_cpp(obj, ind_row, ind_col, ncores=1):
    """src/bed-fun.cpp:72-98 -> int32 (4, nr)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    res = np.zeros((ind_row.size, 4), dtype=np.int32)
    _chk(lib().orc_bed_row_counts(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(ind_row, C.c_int),
                                  ind_row.size, _p(ind_col, C.c_int), ind_col.size, int(ncores),
                                  _p(res, C.c_int)))
    return res.T


NA_INTEGER = -2147483648


def read_bed(obj, ind_row, ind_col, na_val=NA_INTEGER):
    """src/bed-mat-acc.cpp:8-26 -> int32 (nr, nc), NA -> NA_INTEGER."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    res = np.empty((ind_col.size, ind_row.size), dtype=np.int32)
    _chk(lib().orc_read_bed(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(ind_row, C.c_int),
                            ind_row.size, _p(ind_col, C.c_int), ind_col.size, int(na_val),
                            _p(res, C.c_int)))
    return res.T


def read_bed_scaled(obj, ind_row, ind_col, center, scale):
    """src/bed-mat-acc.cpp:30-49 -> float64 (nr, nc)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    center, scale = _f64(center), _f64(scale)
    if center.size != ind_col.size or scale.size != ind_col.size:
        raise OracleError(ERR_MSG[1])
    res = np.empty((ind_col.size, ind_row.size), dtype=np.float64)
    with np.errstate(all="ignore"):
        _chk(lib().orc_read_bed_scaled(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol,
                                       _p(ind_row, C.c_int), ind_row.size, _p(ind_col, C.c_int),
                                       ind_col.size, _p(center, C.c_double), _p(scale, C.c_double),
                                       _p(res, C.c_double)))
    return res.T


def prod_and_rowSumsSq(obj, ind_row, ind_col, center, scale, V):
    """src/bed-fun.cpp:103-133 -> (XV (nr, K), rowSumsSq (nr))."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    center, scale = _f64(center), _f64(scale)
    V = np.asfortranarray(V, dtype=np.float64)
    if V.shape[0] != ind_col.size:
        raise OracleError(ERR_MSG[1])
    K = V.shape[1]
    XV = np.zeros((ind_row.size, K), dtype=np.float64, order="F")
    rss = np.zeros(ind_row.size, dtype=np.float64)
    _chk(lib().orc_prod_and_rowSumsSq(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol,
                                      _p(ind_row, C.c_int), ind_row.size, _p(ind_col, C.c_int),
                                      ind_col.size, _p(center, C.c_double), _p(scale, C.c_double),
                                      _p(V, C.c_double), K, _p(XV, C.c_double), _p(rss, C.c_double)))
    return XV, rss


class OracleFBM:
    """Minimal FBM.code256: n x m bytes column-major + 256 doubles ([bigstatsr], R/bigSNP-class.R:7,13)."""

    def __init__(self, bytes_nm: np.ndarray, code256=None):
        a = np.asfortranarray(bytes_nm, dtype=np.uint8)
        self.nrow, self.ncol = a.shape
        self.bytes = a
        if code256 is None:  # CODE_012 = c(0, 1, 2, rep(NA, 253))
            code256 = np.full(256, np.nan)
            code256[:3] = [0, 1, 2]
        self.code256 = _f64(code256)

    def rows_along(self):
        return np.arange(1, self.nrow + 1, dtype=np.int32)

    def cols_along(self):
        return np.arange(1, self.ncol + 1, dtype=np.int32)


def snp_colstats(fbm, ind_row, ind_col, ncores=1):
    """src/colstats.cpp:8-35."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    m = ind_col.size
    sumX, denoX = np.empty(m), np.empty(m)
    _chk(lib().orc_snp_colstats(_p(fbm.bytes, C.c_uint8), fbm.nrow, fbm.ncol, _p(fbm.code256, C.c_double),
                                _p(ind_row, C.c_int), ind_row.size, _p(ind_col, C.c_int), m, int(ncores),
                                _p(sumX, C.c_double), _p(denoX, C.c_double)))
    return {"sumX": sumX, "denoX": denoX}


def _kind_args(obj):
    if isinstance(obj, OracleFBM):
        return 1, _p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(obj.code256, C.c_double)
    return 0, _p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, None


def corMat(obj, rowInd, colInd, size, thr, pos, fill_diag=True, ncores=1):
    """src/corr.cpp:11-97,102-126 -> CSC pieces (p int64 (nc+1), i int32, x float64)."""
    rowInd, colInd = _i32(rowInd), _i32(colInd)
    thr, pos = _f64(thr), _f64(pos)
    if pos.size != colInd.size:
        raise OracleError(ERR_MSG[1])
    kind, mat, n, m, code = _kind_args(obj)
    p = np.zeros(colInd.size + 1, dtype=np.int64)
    pi = C.POINTER(C.c_int)()
    px = C.POINTER(C.c_double)()
    with np.errstate(all="ignore"):
        _chk(lib().orc_corMat(kind, mat, n, m, code, _p(rowInd, C.c_int), rowInd.size,
                              _p(colInd, C.c_int), colInd.size, C.c_double(size), _p(thr, C.c_double),
                              _p(pos, C.c_double), int(bool(fill_diag)), int(ncores),
                              _p(p, C.c_longlong), C.byref(pi), C.byref(px)))
    nnz = int(p[-1])
    i = np.ctypeslib.as_array(pi, shape=(max(nnz, 1),))[:nnz].copy()
    x = np.ctypeslib.as_array(px, shape=(max(nnz, 1),))[:nnz].copy()
    lib().orc_free(pi)
    lib().orc_free(px)
    return p, i, x


def multLinReg(obj, ind_row, ind_col, U, ncores=1):
    """src/multLinReg.cpp:8-88 -> t-scores (nc, K); NA_REAL is NaN."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    U = np.asfortranarray(np.asarray(U, dtype=np.float64).reshape(len(U), -1))
    if U.shape[0] != ind_row.size:
        raise OracleError(ERR_MSG[1])
    kind, mat, n, m, code = _kind_args(obj)
    K = U.shape[1]
    out = np.zeros((ind_col.size, K), dtype=np.float64, order="F")
    with np.errstate(all="ignore"):
        _chk(lib().orc_multLinReg(kind, mat, n, m, code, _p(ind_row, C.c_int), ind_row.size, _p(ind_col, C.c_int),
                                  ind_col.size, _p(U, C.c_double), K, int(ncores), _p(out, C.c_double)))
    return out


def ld_scores(obj, rowInd, colInd, size, pos, ncores=1):
    """src/ld-scores.cpp:11-78,83-105."""
    rowInd, colInd = _i32(rowInd), _i32(colInd)
    pos = _f64(pos)
    if pos.size != colInd.size:
        raise OracleError(ERR_MSG[1])
    kind, mat, n, m, code = _kind_args(obj)
    res = np.empty(colInd.size, dtype=np.float64)
    _chk(lib().orc_ld_scores(kind, mat, n, m, code, _p(rowInd, C.c_int), rowInd.size,
                             _p(colInd, C.c_int), colInd.size, C.c_double(size), _p(pos, C.c_double),
                             int(ncores), _p(res, C.c_double)))
    return res


# ----------------------------------------------------------------------------------------------
# R-level glue of the reference, restated in NumPy
# ----------------------------------------------------------------------------------------------
def getCode(NA_VAL=3):
    """R/utils.R:21-31 (== src/bed-acc.h:22-37): uint8 (4, 256) decode table."""
    out = np.empty(4 * 256, dtype=np.int32)
    lib().orc_get_code(int(NA_VAL), _p(out, C.c_int))
    return out.reshape(256, 4).T.copy()


def getInverseCode():
    """R/utils.R:35-45: byte for each (g0, g1, g2, g3) in {0,1,2,3(NA)}^4 -> array [4,4,4,4]."""
    geno = getCode()
    r = np.zeros((4, 4, 4, 4), dtype=np.uint8)
    for b in range(256):
        g = geno[:, b]
        r[g[0], g[1], g[2], g[3]] = b
    return r


def write_bed_bytes(G: np.ndarray) -> np.ndarray:
    """src/write-plink.cpp:29-47: pack an (n, m) matrix of {0,1,2,3=NA} into m x ceil(n/4) bytes.

    Trailing slots of the last byte are written as genotype 0 (code 11), as the reference does.
    """
    G = np.asarray(G)
    n, m = G.shape
    nb = (n + 3) // 4
    tab = getInverseCode()
    Gp = np.zeros((4 * nb, m), dtype=np.int64)
    Gp[:n] = G
    Gq = Gp.reshape(nb, 4, m)
    by = tab[Gq[:, 0], Gq[:, 1], Gq[:, 2], Gq[:, 3]]  # (nb, m)
    return np.ascontiguousarray(by.T)


def write_bed(path: str, G: np.ndarray, chrom=None, pos=None):
    """Write bed/bim/fam like snp_writeBed (R/write-plink.R:14-45) for a fake bigSNP (R/fake.R:27-54)."""
    n, m = G.shape
    by = write_bed_bytes(G)
    with open(path, "wb") as f:
        f.write(bytes([108, 27, 1]))
        f.write(by.tobytes())
    pre = path[:-4]
    chrom = np.ones(m, dtype=int) if chrom is None else chrom
    pos = 1000 * np.arange(1, m + 1) if pos is None else pos
    with open(pre + ".bim", "w") as f:
        for j in range(m):
            f.write("%d\tsnp_%d\t0\t%d\tC\tT\n" % (chrom[j], j + 1, pos[j]))
    with open(pre + ".fam", "w") as f:
        for i in range(n):
            f.write("fam_%d\tind_%d\t0\t0\t0\t-9\n" % (i + 1, i + 1))
    return path


def bed_prodVec(obj, y_col, ind_row=None, ind_col=None, center=None, scale=None, ncores=1):
    """R/bed-mult-vec.R:58-75."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    y_col = _f64(y_col)
    if y_col.size != ind_col.size:
        raise OracleError(ERR_MSG[1])
    center = np.zeros(ind_col.size) if center is None else _f64(center)
    scale = np.ones(ind_col.size) if scale is None else _f64(scale)
    return bed_pMatVec4(obj, ind_row, ind_col, center, scale, y_col, ncores)


def bed_cprodVec(obj, y_row, ind_row=None, ind_col=None, center=None, scale=None, ncores=1):
    """R/bed-mult-vec.R:20-37."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    y_row = _f64(y_row)
    if y_row.size != ind_row.size:
        raise OracleError(ERR_MSG[1])
    center = np.zeros(ind_col.size) if center is None else _f64(center)
    scale = np.ones(ind_col.size) if scale is None else _f64(scale)
    return bed_cpMatVec4(obj, ind_row, ind_col, center, scale, y_row, ncores)


def bed_scaleBinom(obj, ind_row=None, ind_col=None, ncores=1):
    """R/binom-scaling.R:133-142."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    st = bed_colstats(obj, ind_row, ind_col, ncores)
    with np.errstate(all="ignore"):
        af = st["sumX"] / (2 * st["nb_nona_col"])
        return {"center": 2 * af, "scale": np.sqrt(2 * af * (1 - af))}


def bed_counts(obj, ind_row=None, ind_col=None, byrow=False, ncores=1):
    """R/binom-scaling.R:166-178."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    f = bed_row_counts_cpp if byrow else bed_col_counts_cpp
    return f(obj, ind_row, ind_col, ncores)


def bed_MAF(obj, ind_row=None, ind_col=None, ncores=1):
    """R/binom-scaling.R:203-222."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    counts = bed_counts(obj, ind_row, ind_col, False, ncores).astype(np.int64)
    ac = counts[1] + 2 * counts[2]
    nb_nona = ind_row.size - counts[3]
    with np.errstate(all="ignore"):
        af = ac / (2 * nb_nona)
    return {"ac": ac, "mac": np.minimum(ac, 2 * nb_nona - ac), "af": af,
            "maf": np.minimum(af, 1 - af), "N": nb_nona}


def snp_scaleBinom(fbm, ind_row=None, ind_col=None, nploidy=2, ncores=1):
    """R/binom-scaling.R:62-77."""
    ind_row, ind_col = _defaults(fbm, ind_row, ind_col)
    af = snp_colstats(fbm, ind_row, ind_col, ncores)["sumX"] / (ind_row.size * nploidy)
    with np.errstate(all="ignore"):
        return {"center": nploidy * af, "scale": np.sqrt(nploidy * af * (1 - af))}


def cor_thresholds(n_row: int, alpha: float = 1.0, thr_r2: float = 0.0) -> np.ndarray:
    """R/corr.R:17-23,29: THR[k] = q / sqrt(k - 2 + q^2), q = qt(alpha/2, k-2, upper); pmax(THR, sqrt(thr_r2)).

    R's pmax(NaN, x) is NaN, kept here (entries k = 1, 2).
    """
    from scipy import stats

    k = np.arange(1, n_row + 1, dtype=np.float64)
    with np.errstate(all="ignore"):
        q = stats.t.isf(alpha / 2, df=k - 2)
        thr = q / np.sqrt(k - 2 + q * q)
        out = np.where(np.isnan(thr), np.nan, np.maximum(thr, np.sqrt(thr_r2)))
    return out


def cor0(obj, ind_row=None, ind_col=None, size=500, alpha=1.0, thr_r2=0.0, fill_diag=True,
         infos_pos=None, ncores=1):
    """R/corr.R:3-57 (snp_cor / bed_cor) -> CSC (p, i, x) of the upper-triangular dsCMatrix."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    if infos_pos is None:
        infos_pos = 1000.0 * np.arange(1, ind_col.size + 1)
    infos_pos = _f64(infos_pos)
    if infos_pos.size != ind_col.size:
        raise OracleError(ERR_MSG[1])
    if np.any(np.diff(infos_pos) < 0):
        raise OracleError("'infos.pos' is not sorted.")
    thr = cor_thresholds(ind_row.size, alpha, thr_r2)
    return corMat(obj, ind_row, ind_col, size * 1000.0, thr, infos_pos, fill_diag, ncores)


def ld0(obj, ind_row=None, ind_col=None, size=500, infos_pos=None, ncores=1):
    """R/ld-scores.R:3-22 (snp_ld_scores / bed_ld_scores)."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    if infos_pos is None:
        infos_pos = 1000.0 * np.arange(1, ind_col.size + 1)
    return ld_scores(obj, ind_row, ind_col, size * 1000.0, _f64(infos_pos), ncores)


def bed_tcrossprodSelf(obj, fun_scaling=bed_scaleBinom, ind_row=None, ind_col=None, block_size=1000):
    """R/bed-tcrossprodSelf.R:21-52: K = sum over column blocks of X~_b X~_b^T, scaling per block."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    n, m = ind_row.size, ind_col.size
    K = np.zeros((n, n))
    center, scale = np.zeros(m), np.zeros(m)
    for lo in range(0, m, block_size):  # CutBySize(m, block.size)
        ind = slice(lo, min(lo + block_size, m))
        ms = fun_scaling(obj, ind_row, ind_col[ind])
        center[ind], scale[ind] = ms["center"], ms["scale"]
        tmp = read_bed_scaled(obj, ind_row, ind_col[ind], ms["center"], ms["scale"])
        K += tmp @ tmp.T  # big_increment(K, tcrossprod(tmp))
    return K, center, scale


def bed_randomSVD(obj, fun_scaling=bed_scaleBinom, ind_row=None, ind_col=None, k=10):
    """R/autoSVD.R:205-219.  The Lanczos driver is bigstatsr::big_randomSVD -> RSpectra::svds
    [unvendored]; the oracle computes the same truncated SVD densely (LAPACK) on the scaled matrix,
    which is what the reference's own test pins it to (tests/testthat/test-2-bed-clumping-SVD.R:76-79:
    d == sqrt(eigen(K)) to 1.5e-8)."""
    ind_row, ind_col = _defaults(obj, ind_row, ind_col)
    ms = fun_scaling(obj, ind_row, ind_col)
    X = read_bed_scaled(obj, ind_row, ind_col, ms["center"], ms["scale"])
    u, d, vt = np.linalg.svd(X, full_matrices=False)
    return {"d": d[:k], "u": u[:, :k], "v": vt[:k].T, "center": ms["center"], "scale": ms["scale"]}


def read_bim(bedfile):
    """chromosome (as str) and physical position columns of the .bim (NAMES.MAP, R/utils.R:50-51)."""
    chrom, pos = [], []
    with open(bedfile[:-4] + ".bim") as f:
        for line in f:
            p = line.split()
            chrom.append(p[0])
            pos.append(float(p[3]))
    return np.array(chrom), np.array(pos)


def bed_clumping_chr(obj, ind_row, ind_col, center, scale, ordInd, rankInd, pos, size, thr):
    """src/clumping-bed.cpp:11-91 -> keep (int32 0/1 per column of ind_col)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    keep = np.full(ind_col.size, -1, dtype=np.int32)
    center, scale, pos = _f64(center), _f64(scale), _f64(pos)
    ordInd, rankInd = _i32(ordInd), _i32(rankInd)
    with np.errstate(all="ignore"):
        _chk(lib().orc_bed_clumping_chr(_p(obj.bytes, C.c_uint8), obj.nrow, obj.ncol, _p(ind_row, C.c_int),
                                        ind_row.size, _p(ind_col, C.c_int), ind_col.size, _p(center, C.c_double),
                                        _p(scale, C.c_double), _p(ordInd, C.c_int), _p(rankInd, C.c_int),
                                        _p(pos, C.c_double), C.c_double(size), C.c_double(thr), _p(keep, C.c_int)))
    return keep


def bed_clumping(obj, ind_row=None, S=None, thr_r2=0.2, size=None, exclude=None, infos_chr=None, infos_pos=None,
                 clump_chr=bed_clumping_chr):
    """R/bed-clumping.R:7-74 (bed_clumping + bedClumpingChr) -> sorted 1-based indices of the kept variants."""
    if size is None:
        size = 100 / thr_r2
    if infos_chr is None or infos_pos is None:
        infos_chr, infos_pos = read_bim(obj.bedfile)
    ind_row = obj.rows_along() if ind_row is None else _i32(ind_row)
    m = obj.ncol
    noexcl = np.setdiff1d(np.arange(1, m + 1), np.asarray([] if exclude is None else exclude, dtype=np.int64))
    kept = []
    for chrom in sorted(set(infos_chr[noexcl - 1].tolist())):  # split(ind.noexcl, infos.chr[ind.noexcl])
        ind_chr = noexcl[infos_chr[noexcl - 1] == chrom].astype(np.int32)
        st = bed_colstats(obj, ind_row, ind_chr)
        with np.errstate(all="ignore"):
            center = st["sumX"] / st["nb_nona_col"]
            scale = np.sqrt(st["denoX"])
        S_chr = np.minimum(st["sumX"], 2 * st["nb_nona_col"] - st["sumX"]) if S is None else np.asarray(S)[ind_chr - 1]
        ordv = np.argsort(-np.asarray(S_chr, dtype=np.float64), kind="stable") + 1  # order(S.chr, decreasing = TRUE)
        rank = np.empty_like(ordv)
        rank[ordv - 1] = np.arange(1, ordv.size + 1)  # match(seq_along(ord), ord)
        pos_chr = infos_pos[ind_chr - 1]
        if np.any(np.diff(pos_chr) < 0):
            raise OracleError("'pos.chr' is not sorted.")
        keep = clump_chr(obj, ind_row, ind_chr, center, scale, ordv, rank, pos_chr, size * 1000.0, thr_r2)
        assert np.all((keep == 0) | (keep == 1))
        kept.append(ind_chr[keep == 1])
    return np.sort(np.concatenate(kept)) if kept else np.zeros(0, dtype=np.int32)


def clumping_chr(G, rowInd, colInd, ordInd, rankInd, pos, sumX, denoX, size, thr):
    """src/clumping.cpp:10-91 -> keep (int32 0/1 per column of colInd); G is an OracleFBM (or OracleBed)."""
    rowInd, colInd = _i32(rowInd), _i32(colInd)
    keep = np.full(colInd.size, -1, dtype=np.int32)
    pos, sumX, denoX = _f64(pos), _f64(sumX), _f64(denoX)
    ordInd, rankInd = _i32(ordInd), _i32(rankInd)
    kind, mat, n, m, code = _kind_args(G)
    with np.errstate(all="ignore"):
        _chk(lib().orc_clumping_chr(kind, mat, n, m, code, _p(rowInd, C.c_int), rowInd.size, _p(colInd, C.c_int),
                                    colInd.size, _p(ordInd, C.c_int), _p(rankInd, C.c_int), _p(pos, C.c_double),
                                    _p(sumX, C.c_double), _p(denoX, C.c_double), C.c_double(size), C.c_double(thr),
                                    _p(keep, C.c_int)))
    return keep


def snp_clumping(G, infos_chr, ind_row=None, S=None, thr_r2=0.2, size=None, infos_pos=None, exclude=None,
                 clump_chr=clumping_chr):
    """R/clumping.R:62-137 (snp_clumping + clumpingChr) -> sorted 1-based indices of the kept variants."""
    if size is None:
        size = 100 / thr_r2
    infos_chr = np.asarray(infos_chr)
    m = G.ncol
    if infos_chr.size != m:
        raise OracleError(ERR_MSG[1])
    ind_row = np.arange(1, G.nrow + 1, dtype=np.int32) if ind_row is None else _i32(ind_row)
    noexcl = np.setdiff1d(np.arange(1, m + 1), np.asarray([] if exclude is None else exclude, dtype=np.int64))
    kept = []
    for chrom in sorted(set(infos_chr[noexcl - 1].tolist())):
        ind_chr = noexcl[infos_chr[noexcl - 1] == chrom].astype(np.int32)
        st = snp_colstats(G, ind_row, ind_chr)
        n = ind_row.size
        if S is None:
            af = st["sumX"] / (2 * n)
            S_chr = np.minimum(af, 1 - af)
        else:
            S_chr = np.asarray(S)[ind_chr - 1]
        ordv = np.argsort(-np.asarray(S_chr, dtype=np.float64), kind="stable") + 1
        rank = np.empty_like(ordv)
        rank[ordv - 1] = np.arange(1, ordv.size + 1)
        if infos_pos is None:
            pos_chr, sz = np.arange(1, ind_chr.size + 1, dtype=np.float64), float(size)
        else:
            pos_chr, sz = _f64(np.asarray(infos_pos)[ind_chr - 1]), size * 1000.0
            if np.any(np.diff(pos_chr) < 0):
                raise OracleError("'pos.chr' is not sorted.")
        keep = clump_chr(G, ind_row, ind_chr, ordv, rank, pos_chr, st["sumX"], st["denoX"], sz, thr_r2)
        assert np.all((keep == 0) | (keep == 1))
        kept.append(ind_chr[keep == 1])
    return np.sort(np.concatenate(kept)) if kept else np.zeros(0, dtype=np.int32)


def synth_bed(n, m, seed=20250924, na_rate=0.0, col_offset=0, ld_rho=0.0, ld_block=50) -> "OracleBed":
    """CPU twin of the device synthetic generator (same counter-based RNG), as an OracleBed.  ld_rho > 0: the
    LD-structured variant (haplotype blocks of ld_block SNPs, allele uniforms copied with probability ld_rho)."""
    nb = (n + 3) // 4
    out = np.zeros(nb * m, dtype=np.uint8)
    if ld_rho > 0:
        f = lib().orc_synth_packed_ld
        f.restype = None
        f.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_longlong, C.c_double, C.c_int, C.POINTER(C.c_uint8)]
        f(int(n), int(m), int(seed), float(na_rate), int(col_offset), float(ld_rho), int(ld_block), _p(out, C.c_uint8))
        return OracleBed.from_packed(out, n, m)
    f = lib().orc_synth_packed
    f.restype = None
    f.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_longlong, C.POINTER(C.c_uint8)]
    f(int(n), int(m), int(seed), float(na_rate), int(col_offset), _p(out, C.c_uint8))
    return OracleBed.from_packed(out, n, m)


def decode_dense(obj) -> np.ndarray:
    """Vectorised NumPy twin of the accessor: full (n, m) uint8 matrix with NA = 3."""
    code = getCode().astype(np.uint8)  # (4, 256)
    by = obj.bytes.reshape(obj.ncol, obj.n_byte)
    dec = code[:, by]  # (4, m, n_byte)
    full = dec.transpose(2, 0, 1).reshape(4 * obj.n_byte, obj.ncol)
    return full[: obj.nrow]
