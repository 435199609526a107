"""Host restatement of snp_fastImputeSimple (src/impute-simple.cpp:10-73) with the random method's counter-based
generator of bigsnpr_b200/csrc/bsg_impute.cu mirrored bit for bit.  Test infrastructure only."""
import numpy as np

from tests.synth_ref import mix64

DOMAIN = np.uint64(0x696D707574650000)
ROW_MUL = np.uint64(0xD1342543DE82EF95)


def fround0(x):
    """R's fround(x, 0): round half to even (nearbyint)."""
    return float(np.rint(x))


def random_draws(seed, j, rows, af):
    """4 + two Bernoulli(af) draws for the given 0-based rows of global column j."""
    thr = int(np.rint(af * 4294967296.0))
    kj = mix64((np.uint64(seed) ^ DOMAIN) ^ mix64(np.uint64(j)))
    with np.errstate(over="ignore"):
        h = mix64(kj + np.asarray(rows, dtype=np.uint64) * ROW_MUL)
    lo = (h & np.uint64(0xFFFFFFFF)) < np.uint64(thr)
    hi = (h >> np.uint64(32)) < np.uint64(thr)
    return (4 + lo.astype(np.uint8) + hi.astype(np.uint8)).astype(np.uint8)


def impute(G, method, seed=0):
    """Imputed copy of the (n, m) uint8 CODE_012 bytes and the number of all-missing columns; method 1..4 as in
    src/impute-simple.cpp (mode, mean0, mean2, random)."""
    G = np.array(G, dtype=np.uint8, order="F", copy=True)
    n = G.shape[0]
    n_all = 0
    for j in range(G.shape[1]):
        col = G[:, j]
        na = col > 2
        if not na.any():
            continue
        c1, c2 = int((col == 1).sum()), int((col == 2).sum())
        c = n - int(na.sum())
        if c == 0:
            n_all += 1
        if method == 1:
            c0 = c - (c1 + c2)
            imputed = 0
            if c1 > c0:
                imputed = 1
            if imputed == 0 and c2 > c0:
                imputed = 2
            if imputed == 1 and c2 > c1:
                imputed = 2
            col[na] = imputed + 4
        elif c == 0:
            continue
        elif method == 2:
            col[na] = int(fround0((c1 + 2.0 * c2) / c)) + 4
        elif method == 3:
            col[na] = int(fround0(100 * ((c1 + 2.0 * c2) / c))) + 7
        else:
            col[na] = random_draws(seed, j, np.nonzero(na)[0], (0.5 * c1 + c2) / c)
    return G, n_all
