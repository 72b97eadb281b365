"""poseidon_254 hash suite (SURVEY.md 8f-4, first slice): circomlib's public known answers through the Python oracle and through the
product's host permutation (8-limb Montgomery arithmetic), then the device kernels against the oracle."""
import ctypes as C

import numpy as np
import pytest

from oracle import poseidon254 as O254


def _host_permute(vals):
    from zktls_b200 import lib
    from zktls_b200._lib import check
    a = np.concatenate([O254.to_digest(v) for v in vals])
    o = np.zeros(24, np.uint32)
    check(lib().zkb_poseidon254_permute_host(a.ctypes.data_as(C.POINTER(C.c_uint32)), o.ctypes.data_as(C.POINTER(C.c_uint32))))
    return [sum(int(o[8 * i + q]) << (32 * q) for q in range(8)) for i in range(3)]


def test_oracle_reproduces_circomlib_known_answers():
    for (a, b), want in O254.KAT.items():
        assert O254.permute([0, a, b])[0] == want
    assert O254.RC[0] == 0x0EE9A592BA9A9518D05986D656F40C2114C4993C11BB29938D21D47304CD8E6E          # circomlib C[0] for t = 3
    assert O254.MDS[0][0] == 0x109B7F411BA0E4C9B2B70CAF5C36A7B194BE7C11AD24378BFEDB68592BA8118B       # circomlib M[0][0]


def test_product_host_permutation_reproduces_the_known_answers_and_the_oracle():
    for (a, b), want in O254.KAT.items():
        assert _host_permute([0, a, b])[0] == want
    rng = np.random.default_rng(254)
    for _ in range(5):
        vals = [int.from_bytes(rng.bytes(32), "little") % O254.P for _ in range(3)]
        assert _host_permute(vals) == O254.permute(vals)
    # edge values: 0, p - 1, and a 256-bit word above p (reduced on input: 2^256 - 1 takes five subtractions of p)
    assert _host_permute([0, O254.P - 1, 1]) == O254.permute([0, O254.P - 1, 1])
    assert _host_permute([0, (1 << 256) - 1, 1]) == O254.permute([0, ((1 << 256) - 1) % O254.P, 1])


@pytest.fixture(scope="module")
def hal():
    from zktls_b200.hal import B200Hal
    h = B200Hal(0)
    yield h
    h.close()


@pytest.mark.gpu
def test_hash_fold_and_merkle_build_match_oracle(hal):
    rng = np.random.default_rng(1)
    rows = 64
    leaves = np.concatenate([O254.to_digest(int.from_bytes(rng.bytes(32), "little") % O254.P) for _ in range(rows)])
    nodes0 = np.concatenate([np.zeros(rows * 8, np.uint32), leaves])
    d = hal.copy_from_digest(nodes0)
    hal.p254_hash_fold(d, rows, rows // 2)
    assert np.array_equal(d.to_numpy(), O254.hash_fold(nodes0, rows, rows // 2))
    d = hal.copy_from_digest(nodes0)
    hal.p254_merkle_build(d, rows)
    got, want = d.to_numpy().reshape(-1, 8), O254.merkle_build(nodes0, rows).reshape(-1, 8)
    assert np.array_equal(got[1:], want[1:])
    # the 2-to-1 hash of the known-answer inputs, through the device kernel
    pair = np.concatenate([np.zeros(16, np.uint32), O254.to_digest(1), O254.to_digest(2)])
    d = hal.copy_from_digest(pair)
    hal.p254_hash_fold(d, 2, 1)
    assert O254.from_digest(d.to_numpy().reshape(-1, 8)[1]) == O254.KAT[(1, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", [(5, 0), (7, 1), (33, 8), (20, 9), (16, 16), (9, 17), (64, 40)])
def test_hash_rows_matches_oracle_under_the_provisional_packing(hal, rows, cols):
    m = np.random.default_rng(rows * 100 + cols).integers(0, O254.BABYBEAR, size=rows * cols, dtype=np.uint32)
    out = hal.alloc_digest(rows)
    hal.p254_hash_rows(out, hal.copy_from_elem(m) if cols else hal.alloc_elem(4))
    assert np.array_equal(out.to_numpy(), O254.hash_rows(m, rows, cols))
