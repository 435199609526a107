"""Host-side mirror of the reference's R interface for the packed-genotype hot path.

R is not available in the build image, so the host side above the C ABI (include/bsgpu.h) is Python,
mirroring the reference's operator interface: same function names, argument meaning (1-based
``ind_row`` / ``ind_col``, ``center`` / ``scale`` per selected column, ``ncores`` accepted and ignored)
and error behaviour, so the parity tests read like the reference's testthat files.  Reference:

    bed()/bed_light          R/bed-class.R:65-134,176-208      -> class Bed
    bed_prodVec / cprodVec   R/bed-mult-vec.R:58-75 / :20-37
    bed_counts / bed_MAF / bed_scaleBinom   R/binom-scaling.R:166-178 / :203-222 / :133-142
    obj.bed[i, j]            R/bed-mat-acc.R:21-38 (read_bed)
    bed_cor / snp_cor        R/corr.R:3-57,95-132
    bed_ld_scores / snp_ld_scores  R/ld-scores.R:3-72
    bed_tcrossprodSelf       R/bed-tcrossprodSelf.R:21-52
    bed_randomSVD            R/autoSVD.R:205-219
    bed_autoSVD              R/autoSVD.R:226-339 (control flow; outlier statistic pluggable, see the docstring)
    prod_and_rowSumsSq / bed_projectSelfPCA   src/bed-fun.cpp:103-133, R/bed-projectPCA.R:45-58,196-227
    multLinReg / bed_pcadapt / snp_pcadapt    src/multLinReg.cpp:8-88, R/pcadapt.R:3-27,61-81
    readbina2 / snp_readBed2, writebina / snp_writeBed   src/read-plink.cpp:61-80, src/write-plink.cpp:13-52

Everything computes on the GPU through libbsgpu; there is no CPU path here.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import BsgError, check, lib

ERROR_DIM = "Incompatibility between dimensions."
NA_INTEGER = -2147483648

LAYOUT_AUTO, LAYOUT_SNP_MAJOR, LAYOUT_SAMPLE_MAJOR = 0, 1, 2

# FBM.code256 code tables (R/bigSNP-class.R:7,13, R/impute.R:9).  A table whose non-NA codes are multiples of 1/100 in
# [0, 2.54] with one value per multiple, and not only 0 / 1 / 2 (CODE_DOSAGE), is staged as value bytes: bed_prodVec,
# bed_cprodVec, View and bed_randomSVD then run on the integer tensor pipe.  CODE_012 / CODE_IMPUTE_PRED keep the
# 2-bit path.
CODE_012 = np.array([0.0, 1.0, 2.0] + [np.nan] * 253)
CODE_DOSAGE = np.concatenate([[0.0, 1.0, 2.0, np.nan, 0.0, 1.0, 2.0], 0 + np.arange(201) * 0.01, np.full(48, np.nan)])
CODE_IMPUTE_PRED = np.array([0.0, 1.0, 2.0, np.nan, 0.0, 1.0, 2.0] + [np.nan] * 249)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _pi(a):
    return None if a is None else a.ctypes.data_as(_lib.c_int_p)


def _pd(a):
    return None if a is None else a.ctypes.data_as(_lib.c_dbl_p)


def _count_lines(path):
    n = 0
    with open(path, "rb") as f:
        for _ in f:
            n += 1
    return n


class Bed:
    """A PLINK .bed staged in HBM: the ``bed`` RefClass of the reference (R/bed-class.R:65-134).

    ``Bed(bedfile)`` reads n from the .fam and m from the .bim like ``$nrow`` / ``$ncol`` do, validates
    the file exactly like ``bedXPtr`` (src/bed-acc-xptr.cpp:14-34) and stages the packed bytes once.
    ``col_range=(begin, end)`` (0-based, half open) stages only a column shard (multi-GPU).
    """

    def __init__(self, bedfile=None, nrow=None, ncol=None, device=0, layouts=LAYOUT_AUTO, col_range=None,
                 _handle=None, _shape=None):
        self._h = None
        self.bedfile = None
        if _handle is not None:
            self._h = _handle
            self.nrow, self.ncol = _shape
            self.bedfile = "<device>"
            return
        bedfile = os.path.expanduser(bedfile)
        self.bedfile = bedfile
        pre = bedfile[:-4] if bedfile.endswith(".bed") else bedfile
        for f in (bedfile, pre + ".bim", pre + ".fam"):
            if (nrow is None or ncol is None) and not os.path.exists(f):
                raise FileNotFoundError("File '%s' doesn't exist." % f)
        n = _count_lines(pre + ".fam") if nrow is None else int(nrow)
        m = _count_lines(pre + ".bim") if ncol is None else int(ncol)
        b, e = (0, m) if col_range is None else col_range
        h = C.c_void_p()
        check(lib().bsg_open_bed(bedfile.encode(), n, m, int(b), int(e), int(device), int(layouts), C.byref(h)))
        self._h = h
        self.nrow, self.ncol = n, int(e) - int(b)
        self.col_offset = int(b)

    # --- alternative constructors -----------------------------------------------------------
    @classmethod
    def from_packed(cls, packed, n, m, device=0, layouts=LAYOUT_AUTO):
        packed = np.ascontiguousarray(packed, dtype=np.uint8).reshape(-1)
        if packed.size != ((n + 3) // 4) * m:
            raise BsgError(5, "n or p does not match the dimensions of the file.")
        h = C.c_void_p()
        check(lib().bsg_open_packed(packed.ctypes.data_as(_lib.c_u8_p), int(n), int(m), int(device), int(layouts),
                                    C.byref(h)))
        return cls(_handle=h, _shape=(int(n), int(m)))

    @classmethod
    def synthetic(cls, n, m, seed=20250924, na_rate=0.0, col_offset=0, device=0, layouts=LAYOUT_AUTO, ld_rho=0.0,
                  ld_block=50):
        """Synthetic matrix generated on the device (SURVEY.md section 8d).  ld_rho > 0: haplotype blocks of `ld_block`
        SNPs whose alleles are copied from the previous SNP with probability ld_rho (correlated neighbours)."""
        h = C.c_void_p()
        if ld_rho > 0:
            check(lib().bsg_open_synth_ld(int(n), int(m), int(seed), float(na_rate), int(col_offset), float(ld_rho),
                                          int(ld_block), int(device), int(layouts), C.byref(h)))
        else:
            check(lib().bsg_open_synth(int(n), int(m), int(seed), float(na_rate), int(col_offset), int(device),
                                       int(layouts), C.byref(h)))
        return cls(_handle=h, _shape=(int(n), int(m)))

    @classmethod
    def from_fbm(cls, bytes_nm, code256=None, device=0, layouts=LAYOUT_AUTO):
        """FBM.code256 twin (snp_* functions): n x m raw bytes + the 256-entry code (default CODE_012)."""
        a = np.asfortranarray(bytes_nm, dtype=np.uint8)
        n, m = a.shape
        if code256 is None:
            code256 = np.full(256, np.nan)
            code256[:3] = [0, 1, 2]
        code256 = _f64(code256)
        h = C.c_void_p()
        check(lib().bsg_open_fbm256(a.ctypes.data_as(_lib.c_u8_p), n, m, _pd(code256), int(device), int(layouts),
                                    C.byref(h)))
        return cls(_handle=h, _shape=(n, m))

    # --- RefClass surface -------------------------------------------------------------------------
    @property
    def address(self):
        return self._h

    @property
    def light(self):
        return self

    @property
    def shape(self):
        return (self.nrow, self.ncol)

    def __len__(self):
        return self.nrow * self.ncol

    def __repr__(self):
        return "A 'bed' object with %d samples and %d variants." % (self.nrow, self.ncol)

    def rows_along(self):
        return np.arange(1, self.nrow + 1, dtype=np.int32)

    def cols_along(self):
        return np.arange(1, self.ncol + 1, dtype=np.int32)

    @property
    def map(self):
        """`$map` of the RefClass (R/bed-class.R:87-93): chromosome (str) and physical.pos read lazily from the .bim."""
        if getattr(self, "_map", None) is None:
            if not self.bedfile or self.bedfile.startswith("<"):
                raise ValueError("this handle has no .bim file: pass infos_chr / infos_pos")
            chrom, pos = [], []
            with open(self.bedfile[:-4] + ".bim") as f:
                for line in f:
                    p = line.split()
                    chrom.append(p[0])
                    pos.append(float(p[3]))
            off = getattr(self, "col_offset", 0)
            self._map = {"chromosome": np.array(chrom)[off:off + self.ncol],
                         "physical.pos": np.array(pos)[off:off + self.ncol]}
        return self._map

    @property
    def has_na(self):
        return bool(lib().bsg_has_na(self._h))

    @property
    def layouts(self):
        return int(lib().bsg_layouts(self._h))

    @property
    def packed_bytes(self):
        return int(lib().bsg_packed_bytes(self._h))

    def export_packed(self):
        out = np.empty(((self.nrow + 3) // 4) * self.ncol, dtype=np.uint8)
        check(lib().bsg_export_packed(self._h, out.ctypes.data_as(_lib.c_u8_p)))
        return out

    def close(self):
        if self._h is not None:
            lib().bsg_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # obj.bed[i, j]  (R/bed-mat-acc.R:21-38; 1-based like R, NA -> NA_INTEGER)
    def __getitem__(self, key):
        i, j = key
        ind_row = self.rows_along() if i is None or (isinstance(i, slice) and i == slice(None)) else _i32(np.atleast_1d(i))
        ind_col = self.cols_along() if j is None or (isinstance(j, slice) and j == slice(None)) else _i32(np.atleast_1d(j))
        return read_bed(self, ind_row, ind_col)


class Group:
    """One matrix sharded by SNP columns over several GPUs driven by THIS process (bsg_group, SURVEY.md section 8e) -- the
    multi-GPU form an R session uses.  `ind_col` is global and 1-based like everywhere else; the library buckets it by
    owning device.  X.y ends in a sum over the devices done inside the epilogue kernel over NVLink peer memory."""

    def __init__(self, _handle):
        self._g = _handle
        L = lib()
        self.nrow, self.ncol, self.ndev = int(L.bsg_group_nrow(_handle)), int(L.bsg_group_ncol(_handle)), int(L.bsg_group_ndev(_handle))

    @classmethod
    def open(cls, bedfile, devices, nrow=None, ncol=None, layouts=LAYOUT_AUTO):
        bedfile = os.path.expanduser(bedfile)
        pre = bedfile[:-4] if bedfile.endswith(".bed") else bedfile
        n = _count_lines(pre + ".fam") if nrow is None else int(nrow)
        m = _count_lines(pre + ".bim") if ncol is None else int(ncol)
        dv = _i32(devices)
        g = C.c_void_p()
        check(lib().bsg_group_open_bed(bedfile.encode(), n, m, _pi(dv), dv.size, int(layouts), C.byref(g)))
        return cls(g)

    @classmethod
    def synthetic(cls, n, m, devices, seed=20250924, na_rate=0.0, ld_rho=0.0, ld_block=50, layouts=LAYOUT_AUTO):
        dv = _i32(devices)
        g = C.c_void_p()
        check(lib().bsg_group_open_synth(int(n), int(m), int(seed), float(na_rate), float(ld_rho), int(ld_block), _pi(dv),
                                         dv.size, int(layouts), C.byref(g)))
        return cls(g)

    def shard(self, i):
        """The per-device handle as a (non-owning) Bed plus its first global column (0-based)."""
        h = lib().bsg_group_shard(self._g, int(i))
        b0, b1 = lib().bsg_group_shard_begin(self._g, int(i)), lib().bsg_group_shard_begin(self._g, int(i) + 1)
        b = Bed(_handle=C.c_void_p(h), _shape=(self.nrow, b1 - b0))
        b.close = lambda: None  # owned by the group
        return b, b0

    def rows_along(self):
        return np.arange(1, self.nrow + 1, dtype=np.int32)

    def cols_along(self):
        return np.arange(1, self.ncol + 1, dtype=np.int32)

    def _args(self, ind_row, ind_col, center, scale):
        ir = None if ind_row is ... else _i32(ind_row)
        ic = None if ind_col is ... else _i32(ind_col)
        nr = self.nrow if ir is None else ir.size
        nc = self.ncol if ic is None else ic.size
        if (center is None) != (scale is None):
            raise ValueError("center and scale must be given together")
        if center is not None:
            center, scale = _f64(center), _f64(scale)
            if center.size != nc or scale.size != nc:
                raise ValueError(ERROR_DIM)
        return ir, nr, ic, nc, center, scale

    def prodVec(self, y_col, ind_row=..., ind_col=..., center=None, scale=None):
        ir, nr, ic, nc, center, scale = self._args(ind_row, ind_col, center, scale)
        y_col = _f64(y_col)
        if y_col.size != nc:
            raise ValueError(ERROR_DIM)
        out = np.empty(nr)
        check(lib().bsg_group_prodvec(self._g, _pi(ir), nr, _pi(ic), nc, _pd(center), _pd(scale), _pd(y_col), _pd(out)))
        return out

    def cprodVec(self, y_row, ind_row=..., ind_col=..., center=None, scale=None):
        ir, nr, ic, nc, center, scale = self._args(ind_row, ind_col, center, scale)
        y_row = _f64(y_row)
        if y_row.size != nr:
            raise ValueError(ERROR_DIM)
        out = np.empty(nc)
        check(lib().bsg_group_cprodvec(self._g, _pi(ir), nr, _pi(ic), nc, _pd(center), _pd(scale), _pd(y_row), _pd(out)))
        return out

    def randomSVD(self, ind_row=..., ind_col=..., center=None, scale=None, k=10, tol=1e-4, maxit=1000):
        """bed_randomSVD (binomial scaling computed per shard when center / scale are not given)."""
        ir, nr, ic, nc, center, scale = self._args(ind_row, ind_col, center, scale)
        d, u, v = np.empty(k), np.empty((k, nr)), np.empty((k, nc))
        c_out, s_out = np.empty(nc), np.empty(nc)
        niter, nops = C.c_int(0), C.c_int(0)
        check(lib().bsg_group_randomsvd(self._g, _pi(ir), nr, _pi(ic), nc, _pd(center), _pd(scale), int(k), float(tol),
                                        int(maxit), _pd(d), _pd(u), _pd(v), _pd(c_out), _pd(s_out), C.byref(niter),
                                        C.byref(nops)))
        return {"d": d, "u": u.T, "v": v.T, "niter": niter.value, "nops": nops.value, "center": c_out, "scale": s_out}

    def tcrossprodSelf(self, center, scale, ind_row=..., ind_col=...):
        ir, nr, ic, nc, center, scale = self._args(ind_row, ind_col, center, scale)
        K = np.empty((nr, nr))
        check(lib().bsg_group_tcrossprod(self._g, _pi(ir), nr, _pi(ic), nc, _pd(center), _pd(scale), _pd(K)))
        return K

    def scaleBinom(self, ind_row=...):
        """bed_scaleBinom over all columns: per-shard statistics concatenated (a gather, SURVEY.md section 8e)."""
        cs, ss = [], []
        for i in range(self.ndev):
            b, _ = self.shard(i)
            sc = bed_scaleBinom(b, ind_row)
            cs.append(sc["center"])
            ss.append(sc["scale"])
        return {"center": np.concatenate(cs), "scale": np.concatenate(ss)}

    def close(self):
        if self._g is not None:
            lib().bsg_group_close(self._g)
            self._g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bed(bedfile, **kw):
    """Wrapper constructor (R/bed-class.R:146)."""
    return Bed(bedfile, **kw)


def _assert_bed(obj):
    if not isinstance(obj, Bed):
        raise TypeError("'obj.bed' is not of class 'bed' or 'bed_light'.")


def _ind(obj, ind_row, ind_col):
    if ind_row is None:
        raise ValueError("'ind.row' can't be `NULL`.")
    if ind_col is None:
        raise ValueError("'ind.col' can't be `NULL`.")
    return _i32(ind_row), _i32(ind_col)


def _dflt(obj, ind_row, ind_col):
    return (obj.rows_along() if ind_row is ... else ind_row), (obj.cols_along() if ind_col is ... else ind_col)


def _assert_lengths(a, b):
    if len(a) != len(b):
        raise ValueError(ERROR_DIM)


class View:
    """Device-resident accessor state (ind.row, ind.col, center, scale): bsg_view."""

    def __init__(self, obj, ind_row=..., ind_col=..., center=None, scale=None):
        _assert_bed(obj)
        ind_row, ind_col = _dflt(obj, ind_row, ind_col)
        ind_row, ind_col = _ind(obj, ind_row, ind_col)
        self.obj = obj
        self.nr, self.nc = ind_row.size, ind_col.size
        if (center is None) != (scale is None):
            raise ValueError("center and scale must be given together")
        if center is not None:
            center, scale = _f64(center), _f64(scale)
            _assert_lengths(center, ind_col)
            _assert_lengths(scale, ind_col)
        v = C.c_void_p()
        check(lib().bsg_view_create(obj._h, _pi(ind_row), self.nr, _pi(ind_col), self.nc, _pd(center), _pd(scale),
                                    C.byref(v)))
        self._v = v

    def prodvec(self, y_col):
        y_col = _f64(y_col)
        if y_col.size != self.nc:
            raise ValueError(ERROR_DIM)
        out = np.empty(self.nr)
        check(lib().bsg_view_prodvec(self._v, _pd(y_col), _pd(out)))
        return out

    def cprodvec(self, y_row):
        y_row = _f64(y_row)
        if y_row.size != self.nr:
            raise ValueError(ERROR_DIM)
        out = np.empty(self.nc)
        check(lib().bsg_view_cprodvec(self._v, _pd(y_row), _pd(out)))
        return out

    def prodvec_dev(self, x_ptr, out_ptr, stream=0):
        check(lib().bsg_view_prodvec_dev(self._v, int(x_ptr), int(out_ptr), int(stream) or None))

    def cprodvec_dev(self, x_ptr, out_ptr, stream=0):
        check(lib().bsg_view_cprodvec_dev(self._v, int(x_ptr), int(out_ptr), int(stream) or None))

    def close(self):
        if self._v is not None:
            lib().bsg_view_destroy(self._v)
            self._v = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bed_prodVec(obj_bed, y_col, ind_row=..., ind_col=..., center=None, scale=None, ncores=1):
    """Product between a "bed" object and a vector (R/bed-mult-vec.R:58-75)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    y_col = _f64(y_col)
    _assert_lengths(y_col, ind_col)
    center = np.zeros(ind_col.size) if center is None else _f64(center)
    _assert_lengths(center, ind_col)
    scale = np.ones(ind_col.size) if scale is None else _f64(scale)
    _assert_lengths(scale, ind_col)
    out = np.empty(ind_row.size)
    check(lib().bsg_prodvec(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, _pd(center),
                            _pd(scale), _pd(y_col), _pd(out)))
    return out


def bed_cprodVec(obj_bed, y_row, ind_row=..., ind_col=..., center=None, scale=None, ncores=1):
    """Cross-product between a "bed" object and a vector (R/bed-mult-vec.R:20-37)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    y_row = _f64(y_row)
    _assert_lengths(y_row, ind_row)
    center = np.zeros(ind_col.size) if center is None else _f64(center)
    _assert_lengths(center, ind_col)
    scale = np.ones(ind_col.size) if scale is None else _f64(scale)
    _assert_lengths(scale, ind_col)
    out = np.empty(ind_col.size)
    check(lib().bsg_cprodvec(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, _pd(center),
                             _pd(scale), _pd(y_row), _pd(out)))
    return out


def bed_colstats(obj_bed, ind_row=..., ind_col=..., ncores=1):
    """src/bed-fun.cpp:9-46 -> dict(sumX, denoX, nb_nona_col); warns like the reference (:40-41)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    m = ind_col.size
    sumX, denoX, nb = np.empty(m), np.empty(m), np.empty(m, dtype=np.int32)
    n_bad = C.c_int(0)
    check(lib().bsg_colstats(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), m, _pd(sumX), _pd(denoX), _pi(nb),
                             C.byref(n_bad)))
    if n_bad.value > 0:
        import warnings

        warnings.warn("%d variants have >50%% missing values." % n_bad.value)
    return {"sumX": sumX, "denoX": denoX, "nb_nona_col": nb}


def bed_scaleBinom(obj_bed, ind_row=..., ind_col=..., ncores=1):
    """Binomial(2, p) scaling (R/binom-scaling.R:133-142)."""
    st = bed_colstats(obj_bed, ind_row, ind_col, ncores)
    with np.errstate(all="ignore"):
        af = st["sumX"] / (2 * st["nb_nona_col"])
        return {"center": 2 * af, "scale": np.sqrt(2 * af * (1 - af))}


def bed_counts(obj_bed, ind_row=..., ind_col=..., byrow=False, ncores=1):
    """Counts of 0s, 1s, 2s and NAs by variant (or by individual): R/binom-scaling.R:166-178 -> (4, k)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    k = ind_row.size if byrow else ind_col.size
    res = np.zeros((k, 4), dtype=np.int32)
    f = lib().bsg_row_counts if byrow else lib().bsg_col_counts
    check(f(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, _pi(res)))
    return res.T


def bed_MAF(obj_bed, ind_row=..., ind_col=..., ncores=1):
    """Allele frequencies (R/binom-scaling.R:203-222)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    counts = bed_counts(obj_bed, ind_row, ind_col, False, ncores).astype(np.int64)
    ac = counts[1] + 2 * counts[2]
    nb_nona = ind_row.size - counts[3]
    with np.errstate(all="ignore"):
        af = ac / (2 * nb_nona)
    return {"ac": ac, "mac": np.minimum(ac, 2 * nb_nona - ac), "af": af, "maf": np.minimum(af, 1 - af), "N": nb_nona}


def snp_colstats(G, ind_row=..., ind_col=..., ncores=1):
    """src/colstats.cpp:8-35 on an FBM-backed handle."""
    ind_row, ind_col = _ind(G, *_dflt(G, ind_row, ind_col))
    m = ind_col.size
    sumX, denoX = np.empty(m), np.empty(m)
    check(lib().bsg_snp_colstats(G._h, _pi(ind_row), ind_row.size, _pi(ind_col), m, _pd(sumX), _pd(denoX)))
    return {"sumX": sumX, "denoX": denoX}


def snp_scaleBinom(nploidy=2):
    """R/binom-scaling.R:62-77: returns the scaling function."""

    def f(X, ind_row=..., ind_col=..., ncores=1):
        ind_row2, _ = _dflt(X, ind_row, ind_col)
        af = snp_colstats(X, ind_row, ind_col, ncores)["sumX"] / (len(ind_row2) * nploidy)
        with np.errstate(all="ignore"):
            return {"center": nploidy * af, "scale": np.sqrt(nploidy * af * (1 - af))}

    return f


def snp_MAF(G, ind_row=..., ind_col=..., nploidy=2, ncores=1):
    """R/binom-scaling.R:94-106."""
    ind_row2, _ = _dflt(G, ind_row, ind_col)
    af = snp_colstats(G, ind_row, ind_col, ncores)["sumX"] / (len(ind_row2) * nploidy)
    return np.minimum(af, 1 - af)


def read_bed(obj_bed, ind_row, ind_col, na_val=NA_INTEGER):
    """src/bed-mat-acc.cpp:8-26 -> int32 (nr, nc)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    res = np.empty((ind_col.size, ind_row.size), dtype=np.int32)
    check(lib().bsg_read_bed(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, int(na_val), _pi(res)))
    return res.T


def read_bed_scaled(obj_bed, ind_row, ind_col, center, scale):
    """src/bed-mat-acc.cpp:30-49 -> float64 (nr, nc)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    center, scale = _f64(center), _f64(scale)
    if center.size != ind_col.size or scale.size != ind_col.size:
        raise ValueError(ERROR_DIM)
    res = np.empty((ind_col.size, ind_row.size), dtype=np.float64)
    check(lib().bsg_read_bed_scaled(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, _pd(center),
                                    _pd(scale), _pd(res)))
    return res.T


def cor_thresholds(n_row, alpha=1.0, thr_r2=0.0):
    """R/corr.R:17-23,29: THR = q / sqrt(k - 2 + q^2) with q = qt(alpha/2, k-2, upper); pmax with sqrt(thr_r2)."""
    from scipy import stats

    k = np.arange(1, n_row + 1, dtype=np.float64)
    with np.errstate(all="ignore"):
        q = stats.t.isf(alpha / 2, df=k - 2)
        thr = q / np.sqrt(k - 2 + q * q)
        return np.where(np.isnan(thr), np.nan, np.maximum(thr, np.sqrt(thr_r2)))


def corMat(obj, rowInd, colInd, size, thr, pos, fill_diag=True, ncores=1):
    """src/corr.cpp:102-126 -> CSC pieces (p, i, x); i 0-based ascending, diagonal last."""
    rowInd, colInd = _i32(rowInd), _i32(colInd)
    thr, pos = _f64(thr), _f64(pos)
    if pos.size != colInd.size:
        raise ValueError(ERROR_DIM)
    if thr.size != rowInd.size:
        raise ValueError(ERROR_DIM)
    p = np.zeros(colInd.size + 1, dtype=np.int64)
    pi, px = _lib.c_int_p(), _lib.c_dbl_p()
    check(lib().bsg_cor(obj._h, _pi(rowInd), rowInd.size, _pi(colInd), colInd.size, float(size), _pd(thr), _pd(pos),
                        int(bool(fill_diag)), p.ctypes.data_as(_lib.c_i64_p), C.byref(pi), C.byref(px)))
    nnz = int(p[-1])
    return p, _adopt(pi, C.c_int32, np.int32, nnz), _adopt(px, C.c_double, np.float64, nnz)


class _CBuffer:
    """Owner of an array the library allocated: released with bsg_free when the last numpy view is gone."""

    def __init__(self, ptr):
        self._ptr = ptr

    def __del__(self):
        try:
            lib().bsg_free(self._ptr)
        except Exception:  # interpreter shutdown
            pass


def _adopt(ptr, ctype, dtype, count):
    """numpy array over a library-owned buffer WITHOUT a copy (configs[2]'s CSC arrays are 1.2 GB: a copy doubles the
    host time of the call); the buffer lives as long as the array or any view of it."""
    owner = _CBuffer(C.cast(ptr, C.c_void_p))
    if count <= 0:
        return np.zeros(0, dtype=dtype)
    buf = (ctype * count).from_address(C.addressof(ptr.contents))
    buf._owner = owner
    return np.frombuffer(buf, dtype=dtype, count=count)


def _cor0(obj, ind_row, ind_col, size, alpha, thr_r2, fill_diag, infos_pos, ncores):
    ind_row, ind_col = _ind(obj, *_dflt(obj, ind_row, ind_col))
    if infos_pos is None:
        infos_pos = 1000.0 * np.arange(1, ind_col.size + 1)
    infos_pos = _f64(infos_pos)
    _assert_lengths(infos_pos, ind_col)
    if np.any(np.diff(infos_pos) < 0):
        raise ValueError("'infos.pos' is not sorted.")
    thr = cor_thresholds(ind_row.size, alpha, thr_r2)
    p, i, x = corMat(obj, ind_row, ind_col, size * 1000.0, thr, infos_pos, fill_diag, ncores)
    if np.isnan(x).any():
        import warnings

        warnings.warn("NA or NaN values in the resulting correlation matrix.")
    return p, i, x


def bed_cor(obj_bed, ind_row=..., ind_col=..., size=500, alpha=1.0, thr_r2=0.0, fill_diag=True, infos_pos=None, ncores=1):
    """Correlation matrix (R/corr.R:116-132): CSC (p, i, x) of the upper-triangular dsCMatrix."""
    _assert_bed(obj_bed)
    return _cor0(obj_bed, ind_row, ind_col, size, alpha, thr_r2, fill_diag, infos_pos, ncores)


snp_cor = bed_cor  # R/corr.R:95-110 (FBM-backed handles share the packed kernels)


def bed_ld_scores(obj_bed, ind_row=..., ind_col=..., size=500, infos_pos=None, ncores=1):
    """LD scores (R/ld-scores.R:59-72)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    if infos_pos is None:
        infos_pos = 1000.0 * np.arange(1, ind_col.size + 1)
    infos_pos = _f64(infos_pos)
    _assert_lengths(infos_pos, ind_col)
    if np.any(np.diff(infos_pos) < 0):
        raise ValueError("'infos.pos' is not sorted.")
    out = np.empty(ind_col.size)
    check(lib().bsg_ld_scores(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, float(size) * 1000.0,
                              _pd(infos_pos), _pd(out)))
    return out


snp_ld_scores = bed_ld_scores


def bed_tcrossprodSelf(obj_bed, fun_scaling=bed_scaleBinom, ind_row=..., ind_col=..., block_size=None):
    """tcrossprod / GRM (R/bed-tcrossprodSelf.R:21-52).  The R block loop is one C-ABI call; ``block_size``
    is accepted for signature compatibility.  Returns (K, center, scale)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    ms = fun_scaling(obj_bed, ind_row=ind_row, ind_col=ind_col)
    center, scale = _f64(ms["center"]), _f64(ms["scale"])
    n = ind_row.size
    K = np.empty((n, n))
    check(lib().bsg_tcrossprod(obj_bed._h, _pi(ind_row), n, _pi(ind_col), ind_col.size, _pd(center), _pd(scale), _pd(K)))
    return K, center, scale


def bed_randomSVD(obj_bed, fun_scaling=bed_scaleBinom, ind_row=..., ind_col=..., k=10, tol=1e-4, verbose=False,
                  ncores=1, maxit=1000):
    """Randomized partial SVD (R/autoSVD.R:205-219) -> dict(d, u, v, niter, nops, center, scale)."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    n, m = ind_row.size, ind_col.size
    center = scale = None
    if fun_scaling is not bed_scaleBinom:
        ms = fun_scaling(obj_bed, ind_row=ind_row, ind_col=ind_col)
        center, scale = _f64(ms["center"]), _f64(ms["scale"])
    d = np.empty(k)
    u = np.empty((k, n))
    v = np.empty((k, m))
    c_out, s_out = np.empty(m), np.empty(m)
    niter, nops = C.c_int(0), C.c_int(0)
    check(lib().bsg_randomsvd(obj_bed._h, _pi(ind_row), n, _pi(ind_col), m, _pd(center), _pd(scale), int(k), float(tol),
                              int(maxit), _pd(d), _pd(u), _pd(v), _pd(c_out), _pd(s_out), C.byref(niter), C.byref(nops)))
    nconv = int(lib().bsg_randomsvd_nconv())
    if 0 <= nconv < k:  # RSpectra::svds behind big_randomSVD: "only %d singular values converged"
        import warnings

        warnings.warn("only %d singular values converged after %d restarts (maxit = %d)." % (nconv, niter.value, maxit))
    return {"d": d, "u": u.T, "v": v.T, "niter": niter.value, "nops": nops.value, "center": c_out, "scale": s_out}


def _get_intervals(x, n=2):
    """R/autoSVD.R:4-12: regroup consecutive integers (runs of at least n) into [start, stop] rows."""
    x = np.asarray(x, dtype=np.int64)
    out, i = [], 0
    while i < x.size:
        j = i
        while j + 1 < x.size and x[j + 1] - x[j] == 1:
            j += 1
        if j - i + 1 >= max(n, 2):  # rle(diff(x)): a run needs at least one unit step, singletons never count
            out.append((int(x[i]), int(x[j])))
        i = j + 1
    return out


def _outlier_callable(outlier_fun, roll_size, alpha_tukey):
    """"default": the reference's detector (OGK distance -> rolling mean -> adjusted Tukey fence, outliers.py);
    None: never flag a variant (the loop stops after the first SVD); a callable is used as is."""
    if outlier_fun == "default":
        from .outliers import autosvd_outlier_fun

        return autosvd_outlier_fun(roll_size, alpha_tukey)
    return outlier_fun


def snp_autoSVD(G, infos_chr, infos_pos=None, ind_row=..., ind_col=..., fun_scaling=None, thr_r2=0.2, size=None, k=10,
                roll_size=50, int_min_size=20, alpha_tukey=0.05, min_mac=10, min_maf=0.02, max_iter=5, ncores=1,
                verbose=False, outlier_fun="default"):
    """R/autoSVD.R:67-186: the FBM.code256 twin of bed_autoSVD (snp_MAF -> snp_clumping -> randomSVD loop); `G` is a
    handle staged from an FBM (Bed.from_fbm).  Same remark on the outlier statistic as bed_autoSVD."""
    outlier_fun = _outlier_callable(outlier_fun, roll_size, alpha_tukey)
    infos_chr = np.asarray(infos_chr)
    _assert_lengths(infos_chr, G.cols_along())
    if infos_pos is not None:
        _assert_lengths(infos_pos, infos_chr)
    return _auto_svd(G, infos_chr, None if infos_pos is None else _f64(infos_pos), ind_row, ind_col,
                     fun_scaling or snp_scaleBinom(), thr_r2, size, k, int_min_size, min_mac, min_maf, max_iter, ncores,
                     verbose, outlier_fun, fbm=True)


def bed_autoSVD(obj_bed, ind_row=..., ind_col=..., fun_scaling=bed_scaleBinom, thr_r2=0.2, size=None, k=10,
                roll_size=50, int_min_size=20, alpha_tukey=0.05, min_mac=10, min_maf=0.02, max_iter=5, ncores=1,
                verbose=False, outlier_fun="default"):
    """Truncated SVD while limiting LD (R/autoSVD.R:226-339): MAC / MAF filter (bed_MAF) -> clumping on MAC
    (bed_clumping) -> bed_randomSVD, then up to `max_iter` rounds of outlier-variant removal, same arguments and defaults
    as the reference (roll.size = 50, int.min.size = 20, alpha.tukey = 0.05).

    The engine steps (counts, clumping, SVD) run on the GPU.  The outlier statistic (R/autoSVD.R:295-302) is host-side
    code on the (m x k) loadings: the default restates bigutilsr's dist_ogk / rollmean / tukey_mc_up from their published
    algorithms (bigsnpr_b200/outliers.py -- bigutilsr is un-vendored, so this step's numbers are NOT pinned against the
    reference; every engine step is).  ``outlier_fun`` may also be a callable ``(v, infos_chr_keep) -> 0-based indices
    into the kept variants`` or None (no pruning).  Returns the SVD dict plus ``subset`` (1-based kept columns) and
    ``lrldr`` (list of (chr, start, stop, iter))."""
    _assert_bed(obj_bed)
    outlier_fun = _outlier_callable(outlier_fun, roll_size, alpha_tukey)
    return _auto_svd(obj_bed, obj_bed.map["chromosome"], obj_bed.map["physical.pos"], ind_row, ind_col, fun_scaling, thr_r2,
                     size, k, int_min_size, min_mac, min_maf, max_iter, ncores, verbose, outlier_fun, fbm=False)


def _auto_svd(obj_bed, infos_chr, infos_pos, ind_row, ind_col, fun_scaling, thr_r2, size, k, int_min_size, min_mac, min_maf,
              max_iter, ncores, verbose, outlier_fun, fbm):
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    if size is None and thr_r2 is not None and not np.isnan(thr_r2):
        size = 100 / thr_r2
    say = print if verbose else (lambda *a, **k: None)
    if not (min_mac > 0 and min_maf > 0):
        raise ValueError("You cannot use variants with no variation; set min.mac > 0 and min.maf > 0.")
    try:
        info = bed_MAF(obj_bed, ind_row, ind_col, ncores)
        nok = (info["mac"] < min_mac) | (info["maf"] < min_maf)
    except BsgError:
        if not fbm:
            raise
        # dosage FBM.code256 (no hard-call counts): the reference's own filter, R/autoSVD.R:95-97
        maf = snp_MAF(obj_bed, ind_row, ind_col, ncores=ncores)
        nok = maf < max(min_maf, min_mac / (2 * ind_row.size))
    say("Discarding %d variant%s with MAC < %s or MAF < %s." % (nok.sum(), "s" if nok.sum() > 1 else "", min_mac, min_maf))
    ind_keep = ind_col[~nok]
    if thr_r2 is None or np.isnan(thr_r2):
        say("Skipping clumping.")
    else:
        excl = np.setdiff1d(obj_bed.cols_along(), ind_keep)
        if fbm:
            ind_keep = snp_clumping(obj_bed, infos_chr, ind_row=ind_row, exclude=excl, thr_r2=thr_r2, size=size,
                                    infos_pos=infos_pos, ncores=ncores)
        else:
            ind_keep = bed_clumping(obj_bed, ind_row=ind_row, exclude=excl, thr_r2=thr_r2, size=size, ncores=ncores,
                                    infos_chr=infos_chr, infos_pos=infos_pos)
        say("Phase of clumping (on MAC) at r^2 > %s.. keep %d variants." % (thr_r2, ind_keep.size))
    it, lrldr = 0, []
    while True:
        it += 1
        svd = bed_randomSVD(obj_bed, fun_scaling=fun_scaling, ind_row=ind_row, ind_col=ind_keep, k=k, ncores=ncores)
        if it > max_iter:
            say("Maximum number of iterations reached.")
            break
        excl = np.zeros(0, dtype=np.int64) if outlier_fun is None else np.asarray(
            outlier_fun(svd["v"], infos_chr[ind_keep - 1]), dtype=np.int64)
        say("%d outlier variant%s detected.." % (excl.size, "s" if excl.size > 1 else ""))
        if excl.size == 0:
            say("Converged!")
            break
        for a, b in _get_intervals(np.sort(excl) + 1, n=int_min_size):
            seq = np.arange(a, b + 1) - 1
            chrs = infos_chr[ind_keep[seq] - 1]
            vals, cnts = np.unique(chrs, return_counts=True)
            ch = vals[np.argmax(cnts)]
            in_chr = chrs == ch
            if infos_pos is not None:
                rng_pos = infos_pos[ind_keep[seq[in_chr]] - 1]
                lrldr.append((ch, float(rng_pos.min()), float(rng_pos.max()), it))
        ind_keep = np.delete(ind_keep, excl)
    svd = dict(svd)
    svd["subset"] = ind_keep
    svd["lrldr"] = sorted(lrldr)
    return svd


def clumping_chr(G, rowInd, colInd, ordInd, rankInd, pos, sumX, denoX, size, thr, ncores=1):
    """src/clumping.cpp:10-91 (FBM.code256 handle) -> keep (int32 0/1 per column of colInd)."""
    rowInd, colInd, ordInd = _i32(rowInd), _i32(colInd), _i32(ordInd)
    pos, sumX, denoX = _f64(pos), _f64(sumX), _f64(denoX)
    for v in (pos, sumX, denoX, ordInd):
        if v.size != colInd.size:
            raise ValueError(ERROR_DIM)
    keep = np.full(colInd.size, -1, dtype=np.int32)
    check(lib().bsg_clumping_chr_fbm(G._h, _pi(rowInd), rowInd.size, _pi(colInd), colInd.size, _pd(sumX), _pd(denoX),
                                     _pi(ordInd), _pd(pos), float(size), float(thr), _pi(keep)))
    return keep


def snp_clumping(G, infos_chr, ind_row=..., S=None, thr_r2=0.2, size=None, infos_pos=None, exclude=None, ncores=1):
    """LD clumping on an FBM.code256 handle (R/clumping.R:62-137): sorted 1-based indices of the variants kept."""
    _assert_bed(G)
    infos_chr = np.asarray(infos_chr)
    _assert_lengths(infos_chr, G.cols_along())
    if infos_pos is not None:
        _assert_lengths(infos_pos, infos_chr)
    if S is not None:
        _assert_lengths(S, infos_chr)
    ind_row = G.rows_along() if ind_row is ... else _i32(ind_row)
    if size is None:
        size = 100 / thr_r2
    m = G.ncol
    noexcl = np.setdiff1d(np.arange(1, m + 1), np.asarray([] if exclude is None else exclude, dtype=np.int64))
    kept = []
    for chrom in sorted(set(infos_chr[noexcl - 1].tolist())):
        ind_chr = noexcl[infos_chr[noexcl - 1] == chrom].astype(np.int32)
        st = snp_colstats(G, ind_row, ind_chr, ncores)
        n = ind_row.size
        if S is None:
            af = st["sumX"] / (2 * n)
            S_chr = np.minimum(af, 1 - af)
        else:
            S_chr = np.asarray(S)[ind_chr - 1]
        ordv = (np.argsort(-np.asarray(S_chr, dtype=np.float64), kind="stable") + 1).astype(np.int32)
        if infos_pos is None:
            pos_chr, sz = np.arange(1, ind_chr.size + 1, dtype=np.float64), float(size)
        else:
            pos_chr, sz = _f64(np.asarray(infos_pos)[ind_chr - 1]), size * 1000.0
            if np.any(np.diff(pos_chr) < 0):
                raise ValueError("'pos.chr' is not sorted.")
        keep = clumping_chr(G, ind_row, ind_chr, ordv, None, pos_chr, st["sumX"], st["denoX"], sz, thr_r2, ncores)
        if not np.all((keep == 0) | (keep == 1)):
            raise RuntimeError("clumping left undecided variants")
        kept.append(ind_chr[keep == 1])
    return np.sort(np.concatenate(kept)) if kept else np.zeros(0, dtype=np.int32)


def prod_and_rowSumsSq(obj_bed, ind_row, ind_col, center, scale, V):
    """src/bed-fun.cpp:103-133 -> (XV (nr, K), rowSumsSq (nr)); V has one row per selected column (:116)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    center, scale = _f64(center), _f64(scale)
    V = np.asarray(V, dtype=np.float64)
    V = np.asfortranarray(V.reshape(V.shape[0], -1))
    if center.size != ind_col.size or scale.size != ind_col.size or V.shape[0] != ind_col.size:
        raise ValueError(ERROR_DIM)
    K = V.shape[1]
    XV = np.empty((ind_row.size, K), dtype=np.float64, order="F")
    rss = np.empty(ind_row.size, dtype=np.float64)
    check(lib().bsg_prod_and_rowsumssq(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, _pd(center),
                                       _pd(scale), V.ctypes.data_as(_lib.c_dbl_p), K,
                                       XV.ctypes.data_as(_lib.c_dbl_p), _pd(rss)))
    return XV, rss


def bed_projectSelfPCA(obj_svd, obj_bed, ind_row, ind_col=None, ncores=1):
    """R/bed-projectPCA.R:196-227: project the samples `ind_row` of the same file on the PCs of `obj_svd`
    (dict with v, d, center, scale).  Returns obj.svd.ref, simple_proj (= XV) and X_norm (row sums of squares);
    the OADP correction is bigutilsr::pca_OADP_proj2 applied to (XV, X_norm, d) on the host (un-vendored R code)."""
    _assert_bed(obj_bed)
    v = np.asarray(obj_svd["v"], dtype=np.float64)
    if ind_col is None:
        ind_col = obj_svd.get("subset", None)
    if ind_col is None:
        raise ValueError("'ind.col' can't be `NULL`.")
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    _assert_lengths(np.arange(v.shape[0]), ind_col)
    XV, x_norm = prod_and_rowSumsSq(obj_bed, ind_row, ind_col, obj_svd["center"], obj_svd["scale"], v)
    return {"obj.svd.ref": obj_svd, "simple_proj": XV, "X_norm": x_norm}


def snp_projectSelfPCA(obj_svd, G, ind_row, ind_col=None, ncores=1):
    """R/bed-projectPCA.R:229-270: bed_projectSelfPCA for the FBM.code256 `G` (a handle from Bed.from_fbm) that the SVD
    was computed on; the products are prod_and_rowSumsSq2 (src/project-utils.cpp:12-43), served on a centi-dosage
    handle (CODE_DOSAGE): x = (code256[byte] - center) / scale, a missing value makes its row of XV and X_norm NaN."""
    return bed_projectSelfPCA(obj_svd, G, ind_row, ind_col, ncores)


_IMPUTE_METHODS = ("mode", "mean0", "mean2", "random")


def snp_fastImputeSimple(G_bytes, method="mode", code256=CODE_012, seed=None, device=0, ncores=1):
    """R/impute.R:189-203 (-> src/impute-simple.cpp:10-73): imputes the missing values of the n x m FBM.code256 bytes
    ``G_bytes`` (numpy uint8, column-major) IN PLACE on the GPU and returns the code table of the result, like
    ``Gna$copy(code = ...)``: CODE_DOSAGE for "mean2", CODE_IMPUTE_PRED otherwise.  "random" draws from a counter-based
    generator keyed by (seed, column, row) instead of R's rbinom (``seed`` None: a fresh one).  A column with no
    non-missing value is left unchanged by "mean0" / "mean2" / "random" (the reference casts NaN to a byte there), with a
    warning."""
    import warnings

    if not np.array_equal(np.asarray(code256, dtype=np.float64), CODE_012, equal_nan=True):
        raise ValueError("identical(Gna$code256, CODE_012) is not TRUE")
    if isinstance(method, str) and method == "zero":
        warnings.warn('Using \'method = "zero"\' is deprecated. Using $copy() instead..')
        return np.array([0.0, 1.0, 2.0, 0.0] + [np.nan] * 252)
    if method not in _IMPUTE_METHODS:
        raise ValueError("'arg' should be one of " + ", ".join('"%s"' % m for m in _IMPUTE_METHODS))
    if not (isinstance(G_bytes, np.ndarray) and G_bytes.dtype == np.uint8 and G_bytes.ndim == 2
            and G_bytes.flags.f_contiguous and G_bytes.flags.writeable):
        raise TypeError("G_bytes must be a writeable column-major (n, m) uint8 array: it is imputed in place")
    n, m = G_bytes.shape
    k = _IMPUTE_METHODS.index(method) + 1
    if seed is None:
        seed = int(np.random.default_rng().integers(0, 2**63))
    n_all = C.c_int(0)
    check(lib().bsg_impute(G_bytes.ctypes.data_as(_lib.c_u8_p), int(n), int(m), k, int(seed) & (2**64 - 1), int(device),
                           C.byref(n_all)))
    if n_all.value > 0 and k > 1:
        warnings.warn("%d columns have no non-missing value: left unchanged." % n_all.value)
    return CODE_DOSAGE.copy() if k == 3 else CODE_IMPUTE_PRED.copy()


def multLinReg(obj, ind_row, ind_col, U, ncores=1):
    """src/multLinReg.cpp:64-88 -> t-scores (nc, K), NaN where the reference gives NA."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    U = np.asarray(U, dtype=np.float64)
    U = np.asfortranarray(U.reshape(U.shape[0], -1))
    if U.shape[0] != ind_row.size:
        raise ValueError(ERROR_DIM)
    K = U.shape[1]
    out = np.empty((ind_col.size, K), dtype=np.float64, order="F")
    check(lib().bsg_multlinreg(obj._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size,
                               U.ctypes.data_as(_lib.c_dbl_p), K, out.ctypes.data_as(_lib.c_dbl_p)))
    return out


def bed_pcadapt(obj_bed, U_row, ind_row=..., ind_col=..., ncores=1):
    """R/pcadapt.R:3-27,73-81 up to the t-scores: the Mahalanobis distance (bigutilsr::dist_ogk) and the genomic
    control that follow are host-side R code on the (nc x K) matrix returned here.  K == 1 returns the reference's
    score (t - median(t))^2 directly."""
    _assert_bed(obj_bed)
    ind_row, ind_col = _ind(obj_bed, *_dflt(obj_bed, ind_row, ind_col))
    U = np.asarray(U_row, dtype=np.float64)
    U = U.reshape(U.shape[0], -1)
    _assert_lengths(np.arange(U.shape[0]), ind_row)
    t = multLinReg(obj_bed, ind_row, ind_col, U, ncores)
    if U.shape[1] == 1:
        return {"tscores": t, "score": (t[:, 0] - np.median(t[:, 0])) ** 2}
    return {"tscores": t}


snp_pcadapt = bed_pcadapt  # R/pcadapt.R:61-68 (FBM.code256 handles share the packed kernels)


def readbina2(obj_bed, ind_row, ind_col, ncores=1):
    """src/read-plink.cpp:61-80 -> the FBM.code256 bytes (nr, nc) uint8 with codes 0 / 1 / 2 / 3 (NA)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    out = np.empty((ind_row.size, ind_col.size), dtype=np.uint8, order="F")
    check(lib().bsg_readbina2(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size,
                              out.ctypes.data_as(C.POINTER(C.c_uint8))))
    return out


def snp_readBed2(bedfile, backingfile=None, ind_row=..., ind_col=..., ncores=1):
    """R/read-plink.R:72-111: fill an FBM.code256 (code CODE_012) from a .bed.  Returns dict(genotypes = (nr, nc) uint8
    codes, map = the selected .bim rows, backingfile); with `backingfile` the bytes are also written to
    `<backingfile>.bk` (column-major, the FBM layout), refusing to overwrite like assert_noexist."""
    obj = bed(bedfile)
    try:
        ind_row, ind_col = _ind(obj, *_dflt(obj, ind_row, ind_col))
        G = readbina2(obj, ind_row, ind_col, ncores)
        bim = {k: np.asarray(v)[ind_col - 1] for k, v in obj.map.items()}
    finally:
        obj.close()
    bk = None
    if backingfile is not None:
        bk = os.path.expanduser(backingfile) + ".bk"
        if os.path.exists(bk):
            raise FileExistsError("File '%s' already exists." % bk)
        G.T.tofile(bk)  # column-major on disk
    return {"genotypes": G, "map": bim, "backingfile": bk}


def writebina(filename, obj, ind_row, ind_col):
    """src/write-plink.cpp:13-52: X[ind_row, ind_col] of a staged handle as a .bed file (the reference's bytes)."""
    ind_row, ind_col = _i32(ind_row), _i32(ind_col)
    check(lib().bsg_writebina(obj._h, os.fsencode(filename), _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size))


def snp_writeBed(G, bedfile, ind_row=..., ind_col=...):
    """R/write-plink.R:15-45 for the genotype part: write `bedfile` from a handle (bed- or FBM.code256-staged).
    The .bim / .fam tables are plain-text host data of the caller's bigSNP and are not produced here."""
    if os.path.exists(bedfile):
        raise FileExistsError("File '%s' already exists." % bedfile)
    os.makedirs(os.path.dirname(os.path.abspath(bedfile)), exist_ok=True)
    ind_row, ind_col = _ind(G, *_dflt(G, ind_row, ind_col))
    writebina(os.path.expanduser(bedfile), G, ind_row, ind_col)
    return bedfile


def bed_clumping_chr(obj_bed, ind_row, ind_col, center, scale, ordInd, rankInd, pos, size, thr, ncores=1):
    """src/clumping-bed.cpp:11-91 -> keep (int32 0/1 per column of ind_col).  rankInd is implied by ordInd."""
    ind_row, ind_col, ordInd = _i32(ind_row), _i32(ind_col), _i32(ordInd)
    center, scale, pos = _f64(center), _f64(scale), _f64(pos)
    for v in (center, scale, pos, ordInd):
        if v.size != ind_col.size:
            raise ValueError(ERROR_DIM)
    keep = np.full(ind_col.size, -1, dtype=np.int32)
    check(lib().bsg_clumping_chr(obj_bed._h, _pi(ind_row), ind_row.size, _pi(ind_col), ind_col.size, _pd(center),
                                 _pd(scale), _pi(ordInd), _pd(pos), float(size), float(thr), _pi(keep)))
    return keep


def bed_clumping(obj_bed, ind_row=..., S=None, thr_r2=0.2, size=None, exclude=None, ncores=1, infos_chr=None,
                 infos_pos=None):
    """LD clumping on a bed object (R/bed-clumping.R:7-74): sorted 1-based indices of the variants kept."""
    _assert_bed(obj_bed)
    if ind_row is None:
        raise ValueError("'ind.row' can't be `NULL`.")
    ind_row = obj_bed.rows_along() if ind_row is ... else _i32(ind_row)
    if size is None:
        size = 100 / thr_r2
    if infos_chr is None:
        infos_chr = obj_bed.map["chromosome"]
    if infos_pos is None:
        infos_pos = obj_bed.map["physical.pos"]
    infos_chr, infos_pos = np.asarray(infos_chr), _f64(infos_pos)
    m = obj_bed.ncol
    if S is not None:
        _assert_lengths(infos_chr, S)
    noexcl = np.setdiff1d(np.arange(1, m + 1), np.asarray([] if exclude is None else exclude, dtype=np.int64))
    kept = []
    for chrom in sorted(set(infos_chr[noexcl - 1].tolist())):
        ind_chr = noexcl[infos_chr[noexcl - 1] == chrom].astype(np.int32)
        st = bed_colstats(obj_bed, ind_row, ind_chr, ncores)
        with np.errstate(all="ignore"):
            center = st["sumX"] / st["nb_nona_col"]
            scale = np.sqrt(st["denoX"])
        S_chr = np.minimum(st["sumX"], 2 * st["nb_nona_col"] - st["sumX"]) if S is None else np.asarray(S)[ind_chr - 1]
        ordv = (np.argsort(-np.asarray(S_chr, dtype=np.float64), kind="stable") + 1).astype(np.int32)
        pos_chr = infos_pos[ind_chr - 1]
        if np.any(np.diff(pos_chr) < 0):
            raise ValueError("'pos.chr' is not sorted.")
        keep = bed_clumping_chr(obj_bed, ind_row, ind_chr, center, scale, ordv, None, pos_chr, size * 1000.0, thr_r2, ncores)
        if not np.all((keep == 0) | (keep == 1)):
            raise RuntimeError("clumping left undecided variants")
        kept.append(ind_chr[keep == 1])
    return np.sort(np.concatenate(kept)) if kept else np.zeros(0, dtype=np.int32)
