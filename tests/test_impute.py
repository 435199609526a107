"""snp_fastImputeSimple restated on the host (tests/impute_ref.py) against the reference's own pins on
example-missing.bed (tests/testthat/test-3-fastImpute.R:111-142, test-7-OpenMP.R:274-287) and the rounding rule."""
import os

import numpy as np

from tests.impute_ref import fround0, impute, random_draws

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CODE_IMPUTE_PRED = np.array([0.0, 1.0, 2.0, np.nan, 0.0, 1.0, 2.0] + [np.nan] * 249)
CODE_DOSAGE = np.concatenate([[0.0, 1.0, 2.0, np.nan, 0.0, 1.0, 2.0], np.arange(201) * 0.01, np.full(48, np.nan)])


def _example_missing(oracle):
    o = oracle.OracleBed(os.path.join(GOLDEN, "example-missing.bed"))
    X = oracle.read_bed(o, np.arange(1, o.nrow + 1), np.arange(1, o.ncol + 1), na_val=3)
    return np.asfortranarray(X.astype(np.uint8))


def test_reference_pins_on_example_missing(oracle):
    G = _example_missing(oracle)
    assert np.all(G[[17, 71], 399] == 3)  # G[c(18, 72), 400] is NA
    G2, _ = impute(G, 2)
    assert np.array_equal(CODE_IMPUTE_PRED[G2[[17, 71], 399]], [1.0, 1.0])
    G3, _ = impute(G, 3)
    assert np.array_equal(CODE_DOSAGE[G3[[17, 71], 399]], [1.01, 1.01])
    G4, _ = impute(G, 1)
    assert np.array_equal(CODE_IMPUTE_PRED[G4[[3, 11], 0]], [0.0, 0.0])
    assert np.array_equal(CODE_IMPUTE_PRED[G4[[17, 71], 399]], [1.0, 1.0])
    for method in (1, 2, 3, 4):  # no missing value left (test-7-OpenMP.R:274-287)
        Gi, n_all = impute(G, method, seed=3)
        code = CODE_DOSAGE if method == 3 else CODE_IMPUTE_PRED
        assert n_all == 0 and not np.isnan(code[Gi]).any()
        assert np.array_equal(Gi[G <= 2], G[G <= 2])


def test_fround_ties_to_even():
    assert fround0(0.5) == 0.0 and fround0(1.5) == 2.0 and fround0(2.5) == 2.0
    # a column with c1 = 1, c = 2: mean = 0.5 -> 0 (mean0); 100 * mean = 50 (mean2, no tie) -> 0.50
    G = np.asfortranarray(np.array([[0], [1], [3]], dtype=np.uint8))
    assert impute(G, 2)[0][2, 0] == 4
    assert CODE_DOSAGE[impute(G, 3)[0][2, 0]] == 0.5
    G = np.asfortranarray(np.array([[1], [2], [3]], dtype=np.uint8))  # mean 1.5 -> 2
    assert impute(G, 2)[0][2, 0] == 6


def test_mode_tie_order_and_all_missing():
    cols = [[0, 1, 3], [1, 2, 3], [0, 2, 3], [0, 1, 2, 3], [3, 3, 3]]
    n = max(len(c) for c in cols)
    G = np.full((n, len(cols)), 3, dtype=np.uint8, order="F")
    for j, c in enumerate(cols):
        G[:len(c), j] = c
    out, n_all = impute(G, 1)
    # c0 = c1 -> 0; c1 = c2 (> c0) -> 1; c0 = c2 -> 0; all equal -> 0; all missing -> 4
    assert list(out[n - 1]) == [4, 5, 4, 4, 4] and n_all == 1
    for method in (2, 3, 4):
        out, n_all = impute(G, method, seed=1)
        assert np.all(out[:, 4] == 3) and n_all == 1


def test_random_draws_follow_binomial():
    rows = np.arange(200_000)
    for af in (0.0, 0.1, 0.37, 1.0):
        d = random_draws(11, 5, rows, af) - 4
        if af in (0.0, 1.0):
            assert np.all(d == 2 * af)
            continue
        freq = np.bincount(d, minlength=3) / rows.size
        want = np.array([(1 - af) ** 2, 2 * af * (1 - af), af ** 2])
        assert np.max(np.abs(freq - want)) < 5e-3
    a, b = random_draws(11, 5, rows[:64], 0.4), random_draws(12, 5, rows[:64], 0.4)
    assert not np.array_equal(a, b) and np.array_equal(a, random_draws(11, 5, rows[:64], 0.4))
