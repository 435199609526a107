"""Which path an FBM.code256 table is staged on (bsg_code256_kind, the rule of bsg_open_fbm256): hard calls keep the 2-bit
engine, centi-dosage tables (every non-NA code a multiple of 1/100 in [0, 2.54], one value per multiple) get the value-byte
products, anything else the fp64 statistics only.  Host code: no GPU needed."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def kind():
    from bigsnpr_b200 import _lib, build

    build.build()
    L = _lib.lib()
    return lambda code: L.bsg_code256_kind(np.ascontiguousarray(code, dtype=np.float64).ctypes.data_as(_lib.c_dbl_p))


def test_reference_tables(kind):
    import bigsnpr_b200 as B

    assert kind(B.CODE_012) == 0
    assert kind(B.CODE_IMPUTE_PRED) == 0
    assert kind(B.CODE_DOSAGE) == 1
    assert kind(np.linspace(0, 2, 256)) == 2


def test_code_dosage_is_r_seq():
    """CODE_DOSAGE restates R's seq(0, 2, by = 0.01) = 0 + i * 0.01: within 1.5e-14 of i / 100, codes 1, 5, 107 all 1.0."""
    import bigsnpr_b200 as B

    d = B.CODE_DOSAGE[7:208]
    assert np.max(np.abs(100 * d - np.arange(201))) < 1.5e-14
    assert B.CODE_DOSAGE[1] == B.CODE_DOSAGE[5] == B.CODE_DOSAGE[107] == 1.0
    assert np.isnan(B.CODE_DOSAGE[3]) and np.isnan(B.CODE_DOSAGE[208:]).all()


def test_qualification_rule(kind):
    code = np.full(256, np.nan)
    code[:201] = np.arange(201) / 100.0
    assert kind(code) == 1
    c = code.copy()
    c[0] = 2.55  # value byte 255 is reserved for NA
    assert kind(c) == 2
    c = code.copy()
    c[250] = 0.5 + 1e-6  # not within 1e-9 of a multiple of 1/100
    assert kind(c) == 2
    c = code.copy()
    c[250] = np.nextafter(0.5, 1)  # same value byte as code 50, different fp64 value
    assert kind(c) == 2
    c = code.copy()
    c[250] = -0.01
    assert kind(c) == 2
    c = np.full(256, np.nan)
    c[:3] = [0, 1, 2]
    c[10] = 2.54
    assert kind(c) == 1
    assert kind(np.zeros(256)) == 0
