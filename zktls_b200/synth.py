"""Synthetic segment traces for the SYN circuit family (SURVEY.md 8d, config 2).

Trace A: i.i.d. uniform field elements (throughput + bit-exactness; the constraints do not hold).
Trace B: a witness that satisfies the SYN constraints, so the seal verifies.
All arrays are column-major (cols x n) uint32 Montgomery words, as the prover expects.
"""
import numpy as np

from .circuit import ZK_ROWS

P = 2013265921
_P64 = np.uint64(P)


def encode(x):
    return ((np.asarray(x, dtype=np.uint64) % _P64) << np.uint64(32)) % _P64


def decode(w):
    rinv = np.uint64(pow(1 << 32, -1, P))
    return (np.asarray(w, dtype=np.uint64) * rinv) % _P64


def _mul(a, b):
    return (a * b) % _P64


def splitmix_fp(seed, count):
    """uniform canonical values < P from splitmix64 with rejection (deterministic across hosts)."""
    out = np.empty(count, dtype=np.uint64)
    filled, ctr = 0, np.uint64(0)
    with np.errstate(over="ignore"):
        while filled < count:
            need = int((count - filled) * 1.1) + 16
            z = (np.uint64(seed) + (ctr + np.arange(1, need + 1, dtype=np.uint64)) * np.uint64(0x9E3779B97F4A7C15))
            ctr += np.uint64(need)
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            z = z ^ (z >> np.uint64(31))
            v = z >> np.uint64(33)              # 31 bits
            v = v[v < _P64][: count - filled]
            out[filled: filled + v.size] = v
            filled += v.size
    return out


def trace_a(shape, po2, seed):
    """(io, code, data, accum) of uniform Montgomery words; io is out_size words."""
    n = 1 << po2
    io = splitmix_fp(seed * 4 + 0, shape["out_size"]).astype(np.uint32)
    code = splitmix_fp(seed * 4 + 1, shape["code_cols"] * n).astype(np.uint32)
    data = splitmix_fp(seed * 4 + 2, shape["data_cols"] * n).astype(np.uint32)
    accum = splitmix_fp(seed * 4 + 3, shape["accum_cols"] * n).astype(np.uint32)
    return io, code, data, accum


def trace_b_code_data(shape, po2, seed, code=None):
    """Valid code + data columns (canonical values) and io.  Returns (io_mont, code_canon, data_canon).  code: a canonical code trace
    of an earlier call to reuse (several segments of one program), else generated from the seed."""
    n = 1 << po2
    C, D = shape["code_cols"], shape["data_cols"]
    io = splitmix_fp(seed * 4 + 0, shape["out_size"])
    if code is None:
        code = splitmix_fp(seed * 4 + 1, C * n).reshape(C, n)
        sel = np.zeros(n, dtype=np.uint64)
        sel[1: n - ZK_ROWS] = 1
        code[0] = sel
    data = splitmix_fp(seed * 4 + 2, D * n).reshape(D, n)
    kidx = 1 + (np.arange(D) % (C - 1))
    for i in range(1, n - ZK_ROWS):
        data[:, i] = (_mul(data[:, i - 1], data[:, i - 1]) + code[kidx, i]) % _P64
    return encode(io).astype(np.uint32), code, data


def trace_b_accum(shape, po2, seed, code, data, io_mont, mix_mont):
    """accum columns (canonical) from code/data (canonical) and the prover's `mix` globals (Montgomery words)."""
    n = 1 << po2
    A, D, M, O = shape["accum_cols"], shape["data_cols"], shape["mix_size"], shape["out_size"]
    mix = decode(mix_mont); out = decode(io_mont)
    accum = splitmix_fp(seed * 4 + 3, A * n).reshape(A, n)
    live = code[0].astype(bool)
    prev = lambda col: np.roll(col, 1)
    for j in range(A):
        if j % 2 == 0:
            v = (_mul(np.full(n, mix[j % M], dtype=np.uint64), data[j % D]) + prev(data[(j + 1) % D])) % _P64
        else:
            v = (_mul(prev(accum[j - 1]), accum[j - 1]) + mix[j % M] + out[j % O]) % _P64
        accum[j][live] = v[live]
    return accum


def to_mont(canon_matrix):
    return encode(canon_matrix).astype(np.uint32).ravel()
