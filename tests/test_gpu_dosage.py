"""Centi-dosage FBM.code256 matrices (CODE_DOSAGE, R/bigSNP-class.R:13) on the integer tensor pipe: X.y, Xt.y and
bed_randomSVD against dense fp64 restatements of bigstatsr's products over code256[byte] (bigstatsr is not vendored in
the reference tree: its big_prodVec / big_cprodVec compute ((code256[X] - center) / scale) %*% y in fp64, so a missing
value propagates NA_real_ to every output entry it touches).

Bar: 1e-12 of the largest output entry; the products are exact integer sums of the 61-bit quantised vector, the
references are accumulated in extended precision."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import bigsnpr_b200 as b

    from bigsnpr_b200 import build

    build.build()
    return b


def dosage_bytes(rng, n, m, na_rate=0.0):
    """n x m CODE_DOSAGE code bytes: mostly dosages (codes 7..207), some hard calls (0..2, imputed 4..6)."""
    G = (7 + rng.integers(0, 201, size=(n, m))).astype(np.uint8)
    hard = rng.random(size=(n, m)) < 0.05
    G[hard] = rng.choice(np.array([0, 1, 2, 4, 5, 6], dtype=np.uint8), size=int(hard.sum()))
    if na_rate > 0:
        na = rng.random(size=(n, m)) < na_rate
        G[na] = rng.choice(np.array([3, 208, 255], dtype=np.uint8), size=int(na.sum()))
    return np.asfortranarray(G)


def ref_prod(code, G, y, ir, ic, center, scale, cprod):
    """((code[G[ir, ic]] - center) / scale) %*% y (or its transpose), fp64 elements, extended-precision sums."""
    out = np.empty(ic.size if cprod else ir.size, dtype=np.longdouble)
    yl = y.astype(np.longdouble)
    step = 4096
    if cprod:
        out[:] = 0
        for a in range(0, ir.size, step):
            X = (code[G[np.ix_(ir[a:a + step] - 1, ic - 1)]] - center) / scale
            out += yl[a:a + step] @ X.astype(np.longdouble)
    else:
        for a in range(0, ir.size, step):
            X = (code[G[np.ix_(ir[a:a + step] - 1, ic - 1)]] - center) / scale
            out[a:a + step] = X.astype(np.longdouble) @ yl
    return out.astype(np.float64)


def _close(got, want, tol=1e-12):
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    if ok.any():
        err = np.max(np.abs(got[ok] - want[ok])) / max(np.max(np.abs(want[ok])), 1e-300)
        assert err <= tol, err


def test_code_tables_select_the_path(B, rng):
    n, m = 300, 40
    G = dosage_bytes(rng, n, m)
    y = rng.normal(size=m)
    # CODE_DOSAGE: value bytes, the products are served
    g = B.Bed.from_fbm(G, code256=B.CODE_DOSAGE)
    _close(B.bed_prodVec(g, y), ref_prod(B.CODE_DOSAGE, G, y, np.arange(1, n + 1), np.arange(1, m + 1), 0.0, 1.0, False))
    with pytest.raises(B.BsgError, match="needs hard calls"):
        B.bed_counts(g)
    g.close()
    # not multiples of 1/100: generic fp64 handle, the products are refused as before
    lin = B.Bed.from_fbm(G, code256=np.linspace(0, 2, 256))
    with pytest.raises(B.BsgError, match="needs hard calls"):
        B.bed_prodVec(lin, y)
    lin.close()
    # CODE_IMPUTE_PRED output (codes 4..6 = 0/1/2, no NA): the 2-bit path, no missing value
    Gi = np.asfortranarray(rng.choice(np.array([0, 1, 2, 4, 5, 6], dtype=np.uint8), size=(n, m)))
    gi = B.Bed.from_fbm(Gi, code256=B.CODE_IMPUTE_PRED)
    assert not gi.has_na
    assert np.array_equal(B.bed_counts(gi)[:3].sum(axis=0), np.full(m, n))
    gi.close()


@pytest.mark.parametrize("scaled", [False, True])
def test_dosage_products_index_multisets(B, rng, scaled):
    n, m = 1537, 611
    G = dosage_bytes(rng, n, m)
    code = B.CODE_DOSAGE
    g = B.Bed.from_fbm(G, code256=code)
    for ir, ic in ((np.arange(1, n + 1), np.arange(1, m + 1)),
                   (rng.integers(1, n + 1, size=900), rng.integers(1, m + 1, size=1300)),
                   (np.sort(rng.choice(n, 1000, replace=False)) + 1, rng.integers(1, m + 1, size=200))):
        ir, ic = ir.astype(np.int32), ic.astype(np.int32)
        c = rng.uniform(0.2, 1.8, size=ic.size) if scaled else None
        s = rng.uniform(0.3, 0.9, size=ic.size) if scaled else None
        y_col, y_row = rng.normal(size=ic.size), rng.normal(size=ir.size)
        c0, s0 = (c, s) if scaled else (0.0, 1.0)
        _close(B.bed_prodVec(g, y_col, ir, ic, c, s), ref_prod(code, G, y_col, ir, ic, c0, s0, False))
        _close(B.bed_cprodVec(g, y_row, ir, ic, c, s), ref_prod(code, G, y_row, ir, ic, c0, s0, True))
    g.close()


@pytest.mark.parametrize("shape", [(150_000, 2_048), (2_048, 150_000)])
def test_dosage_products_split_shapes(B, shape):
    rng = np.random.default_rng(7)
    n, m = shape
    G = dosage_bytes(rng, n, m)
    code = B.CODE_DOSAGE
    g = B.Bed.from_fbm(G, code256=code)
    ir, ic = np.arange(1, n + 1, dtype=np.int32), np.arange(1, m + 1, dtype=np.int32)
    c, s = rng.uniform(0.5, 1.5, size=m), rng.uniform(0.4, 0.8, size=m)
    y_col, y_row = rng.normal(size=m), rng.normal(size=n)
    _close(B.bed_prodVec(g, y_col, ir, ic, c, s), ref_prod(code, G, y_col, ir, ic, c, s, False))
    _close(B.bed_cprodVec(g, y_row, ir, ic, c, s), ref_prod(code, G, y_row, ir, ic, c, s, True))
    g.close()


def test_dosage_missing_values(B, rng):
    torch = pytest.importorskip("torch")
    n, m = 2000, 700
    G = dosage_bytes(rng, n, m, na_rate=0.01)
    G[:, :100] = np.where(np.isnan(B.CODE_DOSAGE[G[:, :100]]), 107, G[:, :100])  # 100 complete columns
    code = B.CODE_DOSAGE
    g = B.Bed.from_fbm(G, code256=code)
    ir = rng.integers(1, n + 1, size=1500).astype(np.int32)
    for ic in (rng.integers(1, m + 1, size=400).astype(np.int32), np.arange(1, 101, dtype=np.int32)):
        c, s = rng.uniform(0.5, 1.5, size=ic.size), rng.uniform(0.4, 0.8, size=ic.size)
        y_col, y_row = rng.normal(size=ic.size), rng.normal(size=ir.size)
        a, a0 = B.bed_prodVec(g, y_col, ir, ic, c, s), ref_prod(code, G, y_col, ir, ic, c, s, False)
        b, b0 = B.bed_cprodVec(g, y_row, ir, ic, c, s), ref_prod(code, G, y_row, ir, ic, c, s, True)
        _close(a, a0)
        _close(b, b0)
        v = B.View(g, ir, ic, c, s)
        xd, yd = torch.tensor(y_col, device="cuda"), torch.tensor(y_row, device="cuda")
        od, pd = torch.empty(ir.size, dtype=torch.float64, device="cuda"), torch.empty(ic.size, dtype=torch.float64, device="cuda")
        v.prodvec_dev(xd.data_ptr(), od.data_ptr())
        v.cprodvec_dev(yd.data_ptr(), pd.data_ptr())
        torch.cuda.synchronize()
        if np.isnan(a0).any():  # device-vector forms: any selected missing value makes the whole output NaN
            assert torch.isnan(od).all() and torch.isnan(pd).all()
        else:
            _close(od.cpu().numpy(), a0)
            _close(pd.cpu().numpy(), b0)
        v.close()
    assert np.isnan(a0).sum() == 0  # the complete columns
    g.close()


def test_dosage_randomSVD(B, rng):
    n, m = 1200, 500
    # rank-structured dosages so that the leading singular values are separated
    lat = rng.normal(size=(n, 4)) @ rng.normal(size=(4, m))
    p = 1 / (1 + np.exp(-0.7 * lat))
    G = np.asfortranarray((7 + np.clip(np.rint(200 * p), 0, 200)).astype(np.uint8))
    code = B.CODE_DOSAGE
    g = B.Bed.from_fbm(G, code256=code)
    scal = B.snp_scaleBinom()
    svd = B.bed_randomSVD(g, fun_scaling=scal, k=6, tol=1e-10)
    ms = scal(g)
    X = (code[G] - ms["center"]) / ms["scale"]
    d0 = np.linalg.svd(X, compute_uv=False)[:6]
    assert np.max(np.abs(svd["d"] - d0) / d0[0]) < 1e-7
    with pytest.raises(B.BsgError, match="snp_scaleBinom"):
        B.bed_randomSVD(g, k=3)
    # a selected missing value: the drivers refuse instead of iterating on NaN
    G2 = G.copy()
    G2[5, 7] = 3
    g2 = B.Bed.from_fbm(G2, code256=code)
    with pytest.raises(B.BsgError):
        B.bed_randomSVD(g2, fun_scaling=lambda X, **kw: ms, k=3)
    g2.close()
    # the FBM twin of autoSVD runs end to end on a dosage handle
    res = B.snp_autoSVD(g, np.ones(m, dtype=int), k=4, outlier_fun=None)
    sub = res["subset"]
    Xs = (code[G[:, sub - 1]] - res["center"]) / res["scale"]
    d1 = np.linalg.svd(Xs, compute_uv=False)[:4]
    assert np.max(np.abs(res["d"] - d1) / d1[0]) < 1e-6
    g.close()


# ---- snp_fastImputeSimple ------------------------------------------------------------------------------------------
def _example_missing_bytes(oracle):
    import os

    o = oracle.OracleBed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example-missing.bed"))
    X = oracle.read_bed(o, np.arange(1, o.nrow + 1), np.arange(1, o.ncol + 1), na_val=3)
    return np.asfortranarray(X.astype(np.uint8))


def test_impute_matches_host_twin(B, oracle):
    from tests.impute_ref import impute

    rng = np.random.default_rng(3)
    big = np.asfortranarray(rng.choice(np.array([0, 1, 2], dtype=np.uint8), p=[0.5, 0.35, 0.15], size=(20_000, 5_000)))
    big[rng.random(size=big.shape) < 0.02] = 3
    big[:, 17] = 3  # an all-missing column
    for G in (_example_missing_bytes(oracle), big):
        for k, method in enumerate(("mode", "mean0", "mean2", "random"), start=1):
            got = G.copy(order="F")
            with pytest.warns(UserWarning) if (k > 1 and G is big) else _nullcontext():
                code = B.snp_fastImputeSimple(got, method, seed=99)
            want, _ = impute(G, k, seed=99)
            assert np.array_equal(got, want), method
            assert np.array_equal(code, B.CODE_DOSAGE if k == 3 else B.CODE_IMPUTE_PRED, equal_nan=True)
    with pytest.raises(ValueError, match="should be one of"):
        B.snp_fastImputeSimple(big.copy(order="F"), "mean")
    with pytest.warns(UserWarning, match="deprecated"):
        z = B.snp_fastImputeSimple(big, "zero")
    assert z[3] == 0


class _nullcontext:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def test_impute_random_chisq(B, oracle):
    """test-3-fastImpute.R:132-138: the imputed values at G[c(18, 72), 400] over 500 seeds follow Binomial(2, p)."""
    from scipy import stats

    G = _example_missing_bytes(oracle)
    vals = []
    for seed in range(500):
        Gi = G.copy(order="F")
        B.snp_fastImputeSimple(Gi, "random", seed=seed)
        vals += list(Gi[[17, 71], 399] - 4)
    col = G[:, 399]
    p = col[col <= 2].mean() / 2
    prob = np.array([(1 - p) ** 2, 2 * p * (1 - p), p ** 2])
    obs = np.bincount(vals, minlength=3)
    assert stats.chisquare(obs, prob * obs.sum()).pvalue > 1e-4


def test_imputed_mode_is_hard_calls_and_autosvd_matches_bed(B, oracle, tmp_path):
    G = _example_missing_bytes(oracle)
    B.snp_fastImputeSimple(G, "mode")
    g = B.Bed.from_fbm(G, code256=B.CODE_IMPUTE_PRED)
    assert not g.has_na  # codes 4..6 land on the 2-bit path without missing values
    import os
    import shutil

    n, m = G.shape
    path = str(tmp_path / "imputed")
    B.snp_writeBed(g, path + ".bed")
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example-missing")
    shutil.copy(golden + ".bim", path + ".bim")
    shutil.copy(golden + ".fam", path + ".fam")
    bd = B.Bed(path + ".bed")
    a = B.snp_autoSVD(g, bd.map["chromosome"], bd.map["physical.pos"], k=5, outlier_fun=None)
    b = B.bed_autoSVD(bd, k=5, outlier_fun=None)
    assert np.array_equal(a["subset"], b["subset"])
    assert np.allclose(a["d"], b["d"], rtol=1e-8)
    g.close()
    bd.close()


def test_autosvd_on_mean2_imputed_ld_matrix(B, oracle):
    n, m = 2_000, 3_000
    h = B.Bed.synthetic(n, m, seed=41, na_rate=0.01, ld_rho=0.8)
    G = np.asfortranarray(B.readbina2(h, np.arange(1, n + 1), np.arange(1, m + 1)))
    h.close()
    code = B.snp_fastImputeSimple(G, "mean2", seed=1)
    g = B.Bed.from_fbm(G, code256=code)
    chrom = np.ones(m, dtype=int)
    res = B.snp_autoSVD(g, chrom, k=5, outlier_fun=None)
    # R/autoSVD.R:95-117: MAF filter, then clumping of the rest -- restated on the oracle's literal loops
    o = oracle.OracleFBM(G, code256=code)
    ir, ic = np.arange(1, n + 1, dtype=np.int32), np.arange(1, m + 1, dtype=np.int32)
    af = oracle.snp_colstats(o, ir, ic)["sumX"] / (2 * n)
    excl = ic[np.minimum(af, 1 - af) < max(0.02, 10 / (2 * n))]
    keep0 = oracle.snp_clumping(o, chrom, ind_row=ir, exclude=excl, thr_r2=0.2, size=500)
    sub = res["subset"]
    assert sub.size < m and np.array_equal(np.sort(sub), np.sort(keep0))
    Xs = (code[G[:, sub - 1]] - res["center"]) / res["scale"]
    d0 = np.linalg.svd(Xs, compute_uv=False)[:5]
    assert np.max(np.abs(res["d"] - d0) / d0[0]) < 1e-7
    g.close()


# ---- snp_projectSelfPCA / prod_and_rowSumsSq2 -------------------------------------------------------------------------
def test_dosage_projection(B, rng):
    n, m, K = 1500, 800, 4
    G = dosage_bytes(rng, n, m, na_rate=0.0005)
    code = B.CODE_DOSAGE
    g = B.Bed.from_fbm(G, code256=code)
    ir = rng.integers(1, n + 1, size=700).astype(np.int32)
    ic = np.sort(rng.choice(m, 500, replace=False)).astype(np.int32) + 1
    c, s = rng.uniform(0.5, 1.5, size=ic.size), rng.uniform(0.4, 0.8, size=ic.size)
    V = rng.normal(size=(ic.size, K))
    XV, rss = B.prod_and_rowSumsSq(g, ir, ic, c, s, V)
    # src/project-utils.cpp:32-40 restated: x = (code256[byte] - c) / s, XV += x V, rowSumsSq += x^2
    X = (code[G[np.ix_(ir - 1, ic - 1)]] - c) / s
    XV0 = (X.astype(np.longdouble) @ V.astype(np.longdouble)).astype(np.float64)
    rss0 = (X.astype(np.longdouble) ** 2).sum(axis=1).astype(np.float64)
    assert np.isnan(rss0).any() and not np.isnan(rss0).all()
    for k in range(K):
        _close(XV[:, k], XV0[:, k])
    _close(rss, rss0)
    svd = {"v": V, "d": np.ones(K), "center": c, "scale": s}
    pr = B.snp_projectSelfPCA(svd, g, ir, ic)
    assert np.array_equal(pr["simple_proj"], XV, equal_nan=True) and np.array_equal(pr["X_norm"], rss, equal_nan=True)
    g.close()


# ---- the R shim (.Call on FBM.code256 environments) -------------------------------------------------------------------
from tests.test_gpu_shim import R  # noqa: E402,F401  (the shim built against the minimal R API, as in test_gpu_shim.py)


def _lcg_seed(state):
    """(seed, next state): the seed _bigsnpr_impute draws from R's RNG (two unif_rand), restated for the stand-in RNG of
    tests/stubs/R_ext/Random.h."""
    M = (1 << 64) - 1
    out = []
    for _ in range(2):
        state = (state * 6364136223846793005 + 1442695040888963407) & M
        out.append(int(((state >> 11) * (1.0 / 9007199254740992.0)) * 4294967296.0))
    return (out[0] << 32) | out[1], state


def test_shim_impute_and_projection(B, R, oracle, tmp_path):
    from tests.impute_ref import impute

    G = _example_missing_bytes(oracle)
    n, m = G.shape
    state = 20251017  # the stand-in RNG's start state; this shim build has made no draw before
    for k in (1, 2, 3, 4):
        bk = tmp_path / ("geno%d.bk" % k)
        G.T.tofile(bk)
        fbm = R.env(backingfile=R.s(str(bk)), nrow=R.ints([n]), ncol=R.ints([m]), code256=R.reals(B.CODE_012))
        R.call("_bigsnpr_impute", fbm, R.ints([k]), R.ints([1]))
        seed, state = _lcg_seed(state)
        got = np.fromfile(bk, dtype=np.uint8).reshape(m, n).T
        want, _ = impute(G, k, seed=seed)
        assert np.array_equal(got, want), k
    with pytest.raises(RuntimeError, match="should be 1, 2, 3, or 4"):
        R.call("_bigsnpr_impute", fbm, R.ints([5]), R.ints([1]))
    # prod_and_rowSumsSq2 on the mean2-imputed dosages (code CODE_DOSAGE), src/project-utils.cpp:32-40
    G3 = np.fromfile(tmp_path / "geno3.bk", dtype=np.uint8).reshape(m, n).T
    dos = R.env(backingfile=R.s(str(tmp_path / "geno3.bk")), nrow=R.ints([n]), ncol=R.ints([m]),
                code256=R.reals(B.CODE_DOSAGE))
    rng = np.random.default_rng(5)
    ir = rng.integers(1, n + 1, size=300).astype(np.int32)
    ic = np.sort(rng.choice(m, 400, replace=False)).astype(np.int32) + 1
    c, s = rng.uniform(0.2, 1.5, size=ic.size), rng.uniform(0.3, 0.9, size=ic.size)
    V = rng.normal(size=(ic.size, 3))
    res = R.call("_bigsnpr_prod_and_rowSumsSq2", dos, R.ints(ir), R.ints(ic), R.reals(c), R.reals(s), R.mat(V))
    XV, rss = R.vec(R.L.minir_list_get(res, 0)), R.vec(R.L.minir_list_get(res, 1))
    X = (B.CODE_DOSAGE[G3[np.ix_(ir - 1, ic - 1)]] - c) / s
    _close(XV.reshape(ir.size, 3)[:, 0], (X.astype(np.longdouble) @ V[:, 0].astype(np.longdouble)).astype(np.float64))
    _close(rss, (X.astype(np.longdouble) ** 2).sum(axis=1).astype(np.float64))
    # bed_randomSVD on the FBM environment with the caller's scaling
    svd = R.call("_bigsnpr_bed_randomSVD_gpu", dos, R.ints(np.arange(1, n + 1)), R.ints(ic), R.reals(c), R.reals(s),
                 R.ints([3]), R.reals([1e-8]))
    Xf = (B.CODE_DOSAGE[G3[:, ic - 1]] - c) / s
    d0 = np.linalg.svd(Xf, compute_uv=False)[:3]
    assert np.max(np.abs(R.vec(R.named(svd, "d")) - d0) / d0[0]) < 1e-7
