"""bigsnpr_b200 -- B200-native (sm_100a) engine for bigsnpr's packed-genotype hot path.

The product is the C-ABI CUDA library ``libbsgpu.so`` (include/bsgpu.h).  This package is its Python host
side: a mirror of the reference's R functions (``api``), the loader (``_lib``) and the in-tree build
(``build``).  Importing the package does not load CUDA; the first call does, and fails loudly if the
extension is missing -- there is no CPU fallback.
"""
from .api import (  # noqa: F401
    CODE_012, CODE_DOSAGE, CODE_IMPUTE_PRED, ERROR_DIM, LAYOUT_AUTO, LAYOUT_SAMPLE_MAJOR, LAYOUT_SNP_MAJOR, NA_INTEGER, Bed, BsgError, Group, View, bed, bed_MAF,
    bed_clumping, bed_clumping_chr, bed_colstats, bed_pcadapt, bed_projectSelfPCA, multLinReg, prod_and_rowSumsSq,
    snp_pcadapt, bed_autoSVD, snp_autoSVD, clumping_chr, snp_clumping, readbina2, snp_readBed2, snp_writeBed, writebina, bed_cor, bed_counts, bed_cprodVec, bed_ld_scores, bed_prodVec, bed_randomSVD, bed_scaleBinom,
    bed_tcrossprodSelf, corMat, cor_thresholds, read_bed, read_bed_scaled, snp_MAF, snp_colstats, snp_cor,
    snp_ld_scores, snp_scaleBinom, snp_fastImputeSimple, snp_projectSelfPCA)

__all__ = [n for n in dir() if not n.startswith("_")]
