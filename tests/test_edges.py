"""Boundary field values and offset sub-buffer views, for every device operator.

The parity suites draw their inputs uniformly from [0, P) and run on whole pool allocations.  The lazy-range arguments of the hot
kernels (NTT butterflies on [0, 2P) with Shoup twiddles, Poseidon2's lazy partial rounds, the unreduced 64-bit accumulators fixed up
once per two products, the 8-limb poseidon_254 input reduction) break on inputs that turn up with probability ~1/P under uniform
draws: a result that is exactly zero (which a lazy form can store as P), operands all at P-1 (the accumulator maximum), a 256-bit
word of at least p.  Callers also hand operators views at arbitrary element offsets (`Buffer.slice`, the Rust shim's `as_device_ptr`).

Here every operator runs on edge patterns (all zero, all P-1, constant columns, alternating 0 / P-1, deltas at both ends, edge words
mixed into random words) and on GUARDED views: the operand sits at word offset `off` inside an allocation padded with a non-canonical
sentinel, so a read outside the view is a wrong result and a write outside it is a changed guard word, not a fault.  Entry points
that require 16-byte alignment run at off = 4 and must reject off = 1 before launching.  Every Fp / Fp4 output is checked canonical.
The CPU part pins the two oracles against each other on the same patterns."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle2 as O2
from oracle import poseidon254 as O254
from zktls_b200 import circuit

P = 2013265921
ONE = 0x0FFFFFFE                   # Montgomery word of 1
MONE = P - ONE                     # Montgomery word of -1
EDGE_WORDS = [0, 1, 2, P - 2, P - 1, ONE, MONE, (P - 1) // 2, (P + 1) // 2, 1 << 27, (1 << 27) + 1, 1 << 30]
EDGE_VALUES = [int(v) for v in O2.enc([0, 1, P - 1, 2])]
EDGES = np.array(sorted(set(EDGE_WORDS + EDGE_VALUES)), dtype=np.uint32)
PATTERNS = ["zero", "pm1", "const", "alt", "delta", "mixed"]
SENTINEL = 0xDEADBEEF              # > P: never a valid word
G = 64                             # guard words on each side (256 bytes: the view at off = 0 keeps the pool's alignment)
SMALL = dict(accum_cols=4, code_cols=3, data_cols=6, mix_size=5, out_size=4)
MID = dict(accum_cols=7, code_cols=5, data_cols=33, mix_size=20, out_size=32)
REDUCED = dict(accum_cols=6, code_cols=6, data_cols=12, mix_size=5, out_size=4, majors=3, fanout=(2, 2, 2), leaf_constraints=12)


def pattern(kind, count, n, seed=0):
    """count columns of n Montgomery words each (column-major, like every trace and coefficient batch)"""
    rng = np.random.default_rng(seed)
    x = np.zeros((count, n), dtype=np.uint32)
    if kind == "pm1":
        x[:] = P - 1
    elif kind == "const":
        x[:] = rng.choice(EDGES, size=count)[:, None]
    elif kind == "alt":
        x[:, 1::2] = P - 1
    elif kind == "delta":
        x[:, 0] = P - 1
        x[:, -1] = ONE
    elif kind == "mixed":
        x[:] = rng.integers(0, P, size=(count, n), dtype=np.uint32)
        hit = rng.random((count, n)) < 0.25
        x[hit] = rng.choice(EDGES, size=int(hit.sum()))
    else:
        assert kind == "zero", kind
    return x.ravel()


def neg(w):
    """-x on Montgomery words"""
    w = np.asarray(w, dtype=np.uint64)
    return ((P - w) % P).astype(np.uint32)


def assert_canonical(arr, what="output"):
    arr = np.asarray(arr)
    bad = np.nonzero(arr >= P)[0]
    assert bad.size == 0, f"{what}: {bad.size} non-canonical words, first at {bad[:5]}: {[hex(int(arr[i])) for i in bad[:5]]}"


def eq(got, want, what="output"):
    got, want = np.asarray(got, dtype=np.uint32).ravel(), np.asarray(want, dtype=np.uint32).ravel()
    assert got.size == want.size, f"{what}: {got.size} words, want {want.size}"
    diff = np.nonzero(got != want)[0]
    assert diff.size == 0, f"{what}: {diff.size} words differ, first at {diff[:5]}: got {got[diff[:3]]}, want {want[diff[:3]]}"


# ---- guarded views ------------------------------------------------------------------------------------------------------
class View:
    """`data` placed at word offset G + off of a sentinel-filled allocation; `.buf` is the Buffer view (elements of `words` u32)."""

    def __init__(self, hal, data, off, words=1):
        from zktls_b200.hal import Buffer
        self.data = np.ascontiguousarray(data, dtype=np.uint32).ravel()
        self.off, self.n = off, self.data.size
        host = np.full(self.n + 2 * G, SENTINEL, np.uint32)
        host[G + off: G + off + self.n] = self.data
        self.base = hal.copy_from_elem(host)
        self.buf = Buffer(hal, self.base.ptr + 4 * (G + off), self.n // words, words, owner=self.base)

    def read(self, what="view"):
        """the view's words; fails if any guard word changed"""
        full = self.base.to_numpy()
        lo, hi = full[: G + self.off], full[G + self.off + self.n:]
        assert (lo == SENTINEL).all() and (hi == SENTINEL).all(), \
            f"{what}: write outside the view (guard words changed at {np.nonzero(lo != SENTINEL)[0]} before / {np.nonzero(hi != SENTINEL)[0]} after)"
        return full[G + self.off: G + self.off + self.n]

    def unchanged(self, what="input"):
        eq(self.read(what), self.data, what + " (must be left unchanged)")


ANY_OFFSETS = [0, 1, 3, 4]


def _deep_tap_circuit():
    from test_prover_parity import _deep_tap_circuit as f
    return f()


def _grand_product_circuit():
    from test_accumulate import _grand_product_circuit as f
    return f()


# ===================================================================== CPU: the oracles agree at the edges ===================
@pytest.mark.parametrize("kind", PATTERNS)
def test_oracles_agree_on_edge_patterns(oracle, kind):
    """oracle2 (canonical-value numpy) against the C++ oracle (Montgomery words), on every operator both implement"""
    O = oracle
    for po2, count, eb in ((1, 2, 2), (4, 3, 2), (9, 2, 0), (10, 1, 2)):
        x = pattern(kind, count, 1 << po2, 10 + po2)
        eq(O2.batch_interpolate_ntt(x, count, po2), O.batch_interpolate_ntt(x, count, po2), "interpolate")
        eq(O2.zk_shift(x, count, po2), O.zk_shift(x, count, po2), "zk_shift")
        eq(O2.batch_expand_into_evaluate_ntt(x, count, po2, eb), O.batch_expand_into_evaluate_ntt(x, count, po2, eb), "LDE")
    for rows, cols in ((5, 1), (9, 16), (4, 17), (3, 224)):
        m = pattern(kind, cols, rows, cols)
        eq(O2.hash_rows(m, rows, cols), O.hash_rows(m, rows, cols), "hash_rows")
    leaves = pattern(kind, 1, 64 * 8, 5)
    nodes = np.concatenate([np.zeros(64 * 8, np.uint32), leaves])
    eq(O2.merkle_build_words(nodes, 64)[8:], O.merkle_build(nodes, 64)[8:], "merkle_build")
    coeffs = pattern(kind, 2, 1 << 8, 6)
    xs = np.concatenate([[ONE, 0, 0, 0], [MONE, 0, 0, 0], [0, 0, 0, 0], [P - 1] * 4]).astype(np.uint32)
    which = np.array([0, 1, 0, 1], np.uint32)
    eq(O2.batch_evaluate_any(coeffs, 2, 8, which, xs), O.batch_evaluate_any(coeffs, 2, 8, which, xs), "batch_evaluate_any")
    fin = pattern(kind, 4, 16 * 3, 7)
    for mix in ([0, 0, 0, 0], [ONE, 0, 0, 0], [P - 1] * 4):
        eq(O2.fri_fold(fin, np.array(mix, np.uint32), 3), O.fri_fold(fin, np.array(mix, np.uint32), 3), "fri_fold")
    p = pattern(kind, 1, 4 * 65, 8)
    for z in ([0, 0, 0, 0], [ONE, 0, 0, 0], [P - 1] * 4):
        z = np.array(z, np.uint32)
        q2, r2 = O2.poly_divide_words(p, z)
        q1, r1 = O.poly_divide(p, z)
        eq(q2, q1, "poly_divide quotient"); eq(r2, r1, "poly_divide remainder")
    inp, count, input_size = pattern(kind, 301, 5, 9), 5, 301
    out0 = pattern(kind, 2 * count, 4, 10)
    combos = np.zeros(input_size, np.uint32); combos[::3] = 1
    for ms, mx in (([P - 1] * 4, [ONE, 0, 0, 0]), ([P - 1] * 4, [P - 1] * 4)):
        ms, mx = np.array(ms, np.uint32), np.array(mx, np.uint32)
        eq(O2.mix_poly_coeffs(out0, ms, mx, inp, combos, input_size, count), O.mix_poly_coeffs(out0, ms, mx, inp, combos, input_size, count), "mix_poly_coeffs")
    s = pattern(kind, 64, 4 * 3, 11)
    eq(O2.eltwise_sum_extelem(s, 3, 64), O.eltwise_sum_extelem(s, 3, 64), "eltwise_sum_extelem")
    pp = pattern(kind, 1, 4 * 300, 12)
    eq(O2.prefix_products(pp), O.prefix_products(pp), "prefix_products")
    b = circuit.syn_circuit(**MID); blob = b.blob(); po2 = 6; dom = 4 << po2
    accum, code, data = (pattern(kind, n, dom, 13 + n) for n in b.group_size)
    g = pattern(kind, 1, b.mix_size + b.out_size + 4, 14)
    mix, out, pm = g[: b.mix_size], g[b.mix_size: b.mix_size + b.out_size], g[-4:]
    eq(O2.eval_check(blob, accum, code, data, mix, out, pm, po2), O.eval_check(blob, accum, code, data, mix, out, pm, po2), "eval_check MID")


@pytest.mark.parametrize("po2,eb", [(1, 2), (5, 0), (8, 2), (12, 2)])
def test_lde_of_x_is_the_root_of_unity_powers(oracle, po2, eb):
    """the closed form the full-size GPU test relies on: the LDE of the single coefficient x^1 (bit-reversed input: index rev(1) = n / 2)
    is w^0, w^1, ... in natural order, w the primitive 2^(po2 + eb)-th root of unity -- pinned against both oracles"""
    n = 1 << po2
    x = np.zeros(n, np.uint32); x[n // 2 if n > 1 else 0] = ONE
    want = O2.enc(O2._powers(O2.rou(po2 + eb), n << eb))
    eq(oracle.batch_expand_into_evaluate_ntt(x, 1, po2, eb), want, "C++ oracle")
    eq(O2.batch_expand_into_evaluate_ntt(x, 1, po2, eb), want, "oracle2")


NONCANONICAL_254 = [O254.P, O254.P + 1, 2 * O254.P, (1 << 256) - 1]
EDGE_254 = [0, 1, O254.P - 1, 1 << 253] + NONCANONICAL_254


def _host_permute(vals):
    from zktls_b200 import lib
    from zktls_b200._lib import check
    a = np.concatenate([O254.to_digest(v) for v in vals])
    o = np.zeros(24, np.uint32)
    check(lib().zkb_poseidon254_permute_host(a.ctypes.data_as(C.POINTER(C.c_uint32)), o.ctypes.data_as(C.POINTER(C.c_uint32))))
    return [sum(int(o[8 * i + q]) << (32 * q) for q in range(8)) for i in range(3)]


@pytest.mark.parametrize("word", NONCANONICAL_254, ids=["p", "p+1", "2p", "2^256-1"])
def test_p254_host_permutation_reduces_noncanonical_words(word):
    """a 256-bit input word >= p is reduced mod p on input (2^256 - 1 takes five subtractions)"""
    for vals in ([word, 1, 2], [0, word, O254.P - 1], [word, word, word]):
        assert _host_permute(vals) == O254.permute([v % O254.P for v in vals])


# ===================================================================== GPU ====================================================
@pytest.fixture(scope="module")
def hal():
    from zktls_b200.hal import B200Hal
    h = B200Hal(0)
    yield h
    h.close()


# ---- NTT family ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", PATTERNS)
@pytest.mark.parametrize("po2", [1, 4, 12, 13, 16])
def test_ntt_family_on_edge_patterns(hal, oracle, po2, kind):
    """interpolate, interpolate + zk_shift, and the LDE (expand bits 0 and 2) on 16-byte-aligned views at word offset 4;
    po2 12 is one contiguous pass, 13 and 16 two passes"""
    count, n = 2, 1 << po2
    x = pattern(kind, count, n, 100 + po2)
    coeffs = oracle.batch_interpolate_ntt(x, count, po2)
    for fn, want in ((hal.batch_interpolate_ntt, coeffs), (hal.batch_interpolate_ntt_zk_shift, oracle.zk_shift(coeffs, count, po2))):
        v = View(hal, x, 4)
        fn(v.buf, count)
        got = v.read(fn.__name__)
        assert_canonical(got, fn.__name__)
        eq(got, want, fn.__name__)
    c = pattern(kind, count, n, 200 + po2)
    for eb in (0, 2):
        src, out = View(hal, c, 4), View(hal, np.zeros(count << (po2 + eb), np.uint32), 4)
        hal.batch_expand_into_evaluate_ntt(out.buf, src.buf, count, eb)
        got = out.read("LDE")
        assert_canonical(got, f"LDE eb={eb}")
        eq(got, oracle.batch_expand_into_evaluate_ntt(c, count, po2, eb), f"LDE eb={eb}")
        src.unchanged("LDE input")


@pytest.mark.gpu
@pytest.mark.parametrize("po2", [23, 24])
def test_three_pass_ntts_closed_forms(hal, po2):
    """one column in the three-pass plans, where the oracle would take minutes: the interpolant of a constant is that constant at
    position 0 and EXACT zeros elsewhere (n - 1 cancellations), with and without zk_shift; the LDE of [c, 0, ...] is the constant c;
    the LDE of x^1 is the sequence of root-of-unity powers (order pinned by test_lde_of_x_is_the_root_of_unity_powers)"""
    n = 1 << po2
    for c, shift in ((MONE, False), (P - 1, True)):
        b = hal.copy_from_elem(np.full(n, c, np.uint32))
        (hal.batch_interpolate_ntt_zk_shift if shift else hal.batch_interpolate_ntt)(b, 1)
        got = b.to_numpy()
        assert_canonical(got, "interpolant")
        assert int(got[0]) == c and not got[1:].any(), f"interpolant of a constant: {np.count_nonzero(got[1:])} non-zero words after position 0"
        del b
    eb = 2
    x = np.zeros(n, np.uint32); x[0] = P - 1
    out = hal.alloc_elem(n << eb)
    hal.batch_expand_into_evaluate_ntt(out, hal.copy_from_elem(x), 1, eb)
    got = out.to_numpy()
    assert_canonical(got, "LDE of a constant")
    assert (got == P - 1).all(), "LDE of a constant"
    x[0] = 0; x[n // 2] = ONE
    hal.batch_expand_into_evaluate_ntt(out, hal.copy_from_elem(x), 1, eb)
    got = out.to_numpy()
    assert_canonical(got, "LDE of x")
    eq(got, O2.enc(O2._powers(O2.rou(po2 + eb), n << eb)), "LDE of x")


@pytest.mark.gpu
@pytest.mark.parametrize("off", ANY_OFFSETS)
def test_unaligned_elementwise_ops_stay_inside_their_views(hal, oracle, off):
    """operators with scalar accesses accept any offset: zk_shift, batch_expand, batch_bit_reverse (both kernels: po2 9 and 12),
    eltwise add / copy / zeroize, gather_sample / gather_rows, scatter"""
    for po2 in (9, 12):
        count = 3
        x = pattern("mixed", count, 1 << po2, po2)
        v = View(hal, x, off); hal.zk_shift(v.buf, count)
        got = v.read("zk_shift"); assert_canonical(got, "zk_shift"); eq(got, oracle.zk_shift(x, count, po2), "zk_shift")
        v = View(hal, x, off); hal.batch_bit_reverse(v.buf, count)
        eq(v.read("bit_reverse"), oracle.batch_bit_reverse(x, count, po2), "bit_reverse")
        src, out = View(hal, x, off), View(hal, np.zeros(count << (po2 + 2), np.uint32), (off + 1) % 4)
        hal.batch_expand(out.buf, src.buf, count)
        eq(out.read("batch_expand"), oracle.batch_expand(x, count, po2, 2), "batch_expand"); src.unchanged("batch_expand input")
    n = 1001
    a, b = pattern("alt", 1, n), neg(pattern("alt", 1, n))       # a + (-a): exact zeros and P-1 + 1
    b[::3] = 1
    va, vb, vo = View(hal, a, off), View(hal, b, (off + 3) % 4), View(hal, pattern("mixed", 1, n, 1), off)
    hal.eltwise_add_elem(vo.buf, va.buf, vb.buf)
    got = vo.read("eltwise_add"); assert_canonical(got, "eltwise_add"); eq(got, oracle.eltwise_add_elem(a, b), "eltwise_add")
    va.unchanged("eltwise_add a"); vb.unchanged("eltwise_add b")
    hal.eltwise_copy_elem(vo.buf, va.buf)
    eq(vo.read("eltwise_copy"), a, "eltwise_copy")
    z = pattern("mixed", 1, n, 2); z[::5] = 0xFFFFFFFF
    vz = View(hal, z, off); hal.eltwise_zeroize_elem(vz.buf)
    eq(vz.read("zeroize"), oracle.eltwise_zeroize_elem(z), "zeroize")
    s = pattern("mixed", 1, n, 3)
    vs, vg = View(hal, s, off), View(hal, np.zeros(50, np.uint32), (off + 1) % 4)
    hal.gather_sample(vg.buf, vs.buf, 3, 50, 20)
    eq(vg.read("gather_sample"), oracle.gather_sample(s, 3, 50, 20), "gather_sample")
    idx = np.array([0, 19, 7, 19], np.uint32)
    vr = View(hal, np.zeros(idx.size * 50, np.uint32), off)
    hal.gather_rows(vr.buf, vs.buf, idx, 50, 20)
    eq(vr.read("gather_rows"), np.concatenate([oracle.gather_sample(s, int(i), 50, 20) for i in idx]), "gather_rows")
    vs.unchanged("gather source")
    index = np.array([0, 2, 2, 5], np.uint32); offsets = np.array([0, n - 1, 7, 500, 8], np.uint32); values = EDGES[:5].copy()
    vi = View(hal, s, off)
    hal.scatter(vi.buf, index, offsets, values)
    eq(vi.read("scatter"), oracle.scatter(s, index, offsets, values), "scatter")


@pytest.mark.gpu
def test_aligned_entry_points_reject_a_misaligned_view(hal):
    """the entry points whose kernels make 16-byte accesses check the pointer before launching: a view at word offset 1 is an error"""
    from zktls_b200.hal import Buffer, ZkbError
    base = hal.alloc_elem(4 * 4096 + 64)
    el = Buffer(hal, base.ptr + 4, 4096, 1, owner=base)        # 4-byte aligned only
    e4 = Buffer(hal, base.ptr + 4, 256, 4, owner=base)
    dg = Buffer(hal, base.ptr + 4, 64, 8, owner=base)
    good = hal.alloc_elem(4096)
    calls = {
        "batch_interpolate_ntt": lambda: hal.batch_interpolate_ntt(el, 2),
        "batch_interpolate_ntt_zk_shift": lambda: hal.batch_interpolate_ntt_zk_shift(el, 2),
        "batch_evaluate_ntt": lambda: hal.batch_evaluate_ntt(el, 2, 2),
        "expand_into_evaluate out": lambda: hal.batch_expand_into_evaluate_ntt(el, hal.alloc_elem(1024), 1, 2),
        "expand_into_evaluate in": lambda: hal.batch_expand_into_evaluate_ntt(good, el.slice(0, 1024), 1, 2),
        "hash_rows out": lambda: hal.hash_rows(dg, good),
        "hash_fold": lambda: hal.hash_fold(dg, 32, 16),
        "merkle_build": lambda: hal.merkle_build(dg, 32),
        "p254_hash_fold": lambda: hal.p254_hash_fold(dg, 32, 16),
        "p254_merkle_build": lambda: hal.p254_merkle_build(dg, 32),
        "eltwise_sum_extelem in": lambda: hal.eltwise_sum_extelem(hal.alloc_elem(4 * 64), e4),
        "mix_poly_coeffs out": lambda: hal.mix_poly_coeffs(e4, [ONE, 0, 0, 0], [ONE, 0, 0, 0], good.slice(0, 256), hal.copy_from_u32(np.zeros(1, np.uint32)), 1, 256),
        "batch_evaluate_any xs": lambda: hal.batch_evaluate_any(good, 1, hal.copy_from_u32(np.zeros(2, np.uint32)), e4.slice(0, 2), hal.alloc_extelem(2)),
        "batch_evaluate_any out": lambda: hal.batch_evaluate_any(good, 1, hal.copy_from_u32(np.zeros(2, np.uint32)), hal.alloc_extelem(2), e4.slice(0, 2)),
        "poly_divide": lambda: hal.poly_divide(e4, [ONE, 0, 0, 0]),
        "combos_divide": lambda: hal.combos_divide(e4, 128, [0], [ONE, 0, 0, 0]),
        "prefix_products": lambda: hal.prefix_products(e4),
    }
    before = base.to_numpy()
    for name, call in calls.items():
        with pytest.raises(ZkbError, match="aligned"):
            call()
        hal.sync()
    eq(base.to_numpy(), before, "a rejected call wrote to its buffer")


# ---- hashing ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["zero", "pm1", "mixed"])
@pytest.mark.parametrize("cols", [1, 15, 16, 17, 224])
def test_hash_rows_edges(hal, oracle, cols, kind):
    """all-zero and all-(P-1) rows and edge-mixed rows; the matrix at every word offset, the digests at a 16-byte-aligned offset"""
    rows = 64 if cols == 224 else 300
    m = pattern(kind, cols, rows, cols)
    want = oracle.hash_rows(m, rows, cols)
    for off in ANY_OFFSETS:
        vm, vo = View(hal, m, off), View(hal, np.zeros(rows * 8, np.uint32), 4, words=8)
        hal.hash_rows(vo.buf, vm.buf)
        got = vo.read("digests")
        assert_canonical(got, "digests")
        eq(got, want, f"hash_rows off={off}")
        vm.unchanged("matrix")


@pytest.mark.gpu
@pytest.mark.parametrize("leaf", [0, P - 1, ONE])
@pytest.mark.parametrize("rows", [4096, 8192])
def test_merkle_build_and_fold_saturated_leaves(hal, oracle, rows, leaf):
    """leaves of all-(P-1) words and all-zero words: the warp-cooperative tops and k_merkle_tail_coop see saturated lanes"""
    nodes = np.zeros(2 * rows * 8, np.uint32)
    nodes[rows * 8:] = leaf
    want = oracle.merkle_build(nodes, rows)
    v = View(hal, nodes, 4, words=8)
    hal.merkle_build(v.buf, rows)
    got = v.read("merkle_build")[8:]
    assert_canonical(got, "nodes")
    eq(got, want[8:], "merkle_build")
    v = View(hal, nodes, 4, words=8)
    size = rows
    while size > 1:
        hal.hash_fold(v.buf, size, size // 2)
        size //= 2
    eq(v.read("hash_fold")[8:], want[8:], "hash_fold levels")


@pytest.mark.gpu
def test_p254_hash_fold_and_merkle_build_reduce_noncanonical_leaves(hal):
    """leaves 0, 1, p - 1, 2^253 and the non-canonical words p, p + 1, 2p, 2^256 - 1 (five subtractions) against the oracle, whose
    from_digest reduces mod p"""
    rows = len(EDGE_254)
    leaves = np.concatenate([O254.to_digest(x) for x in EDGE_254])
    nodes = np.concatenate([np.zeros(rows * 8, np.uint32), leaves])
    v = View(hal, nodes, 4, words=8)
    hal.p254_hash_fold(v.buf, rows, rows // 2)
    eq(v.read("p254_hash_fold"), O254.hash_fold(nodes, rows, rows // 2), "p254_hash_fold")
    v = View(hal, nodes, 4, words=8)
    hal.p254_merkle_build(v.buf, rows)
    got, want = v.read("p254_merkle_build").reshape(-1, 8), O254.merkle_build(nodes, rows).reshape(-1, 8)
    eq(got[1:], want[1:], "p254_merkle_build")
    for d in got[1:rows]:
        assert O254.from_digest(d) == sum(int(w) << (32 * i) for i, w in enumerate(d)), "a digest the suite produced must be canonical"


@pytest.mark.gpu
@pytest.mark.parametrize("cols", [7, 8, 9, 16, 17])
def test_p254_hash_rows_saturated_lanes(hal, cols):
    """every BabyBear value P - 1 (the 31-bit lanes straddle the 32-bit limbs) and edge-mixed rows, at every word offset"""
    rows = 40
    for kind, m in (("pm1-value", np.full(rows * cols, MONE, np.uint32)), ("pm1-word", np.full(rows * cols, P - 1, np.uint32)),
                    ("mixed", pattern("mixed", cols, rows, cols))):
        want = O254.hash_rows(m, rows, cols)
        for off in ANY_OFFSETS:
            vm, vo = View(hal, m, off), View(hal, np.zeros(rows * 8, np.uint32), (off + 1) % 4, words=8)
            hal.p254_hash_rows(vo.buf, vm.buf)
            eq(vo.read("p254 digests"), want, f"p254_hash_rows {kind} off={off}")
            vm.unchanged("matrix")


# ---- mixing / DEEP / FRI ---------------------------------------------------------------------------------------------------
MIX_CASES = {          # input, mix_start, mix, out0
    "max": (lambda n: np.full(n, P - 1, np.uint32), [P - 1] * 4, [ONE, 0, 0, 0], lambda n: np.full(n, P - 1, np.uint32)),   # every product (P-1)^2
    "pm1": (lambda n: np.full(n, P - 1, np.uint32), [P - 1] * 4, [P - 1] * 4, lambda n: np.full(n, P - 1, np.uint32)),
    "mixed": (lambda n: pattern("mixed", 1, n, 3), [MONE, 0, P - 1, 1], [ONE, 1, 0, P - 1], lambda n: pattern("mixed", 1, n, 4)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MIX_CASES))
@pytest.mark.parametrize("count,off", [(4096, 0), (4096, 1), (4096, 3), (4097, 0), (4096, 4)])
def test_mix_poly_coeffs_longest_accumulator_chains(hal, oracle, count, off, case):
    """301 columns on ONE combo (the longest accumulator chain; 256 + 45 hits: an odd tail), and 3 combos with odd hit counts.
    count % 4 == 0 on an aligned input runs k_mix_poly_coeffs4; count 4097 or an offset input runs k_mix_poly_coeffs"""
    inp_f, ms, mx, out_f = MIX_CASES[case]
    ms, mx = np.array(ms, np.uint32), np.array(mx, np.uint32)
    for input_size, combos in ((301, np.zeros(301, np.uint32)), (47, (np.arange(47) % 3).astype(np.uint32))):
        n_combos = int(combos.max()) + 1
        inp, out0 = inp_f(input_size * count), out_f(4 * n_combos * count)
        vi, vo = View(hal, inp, off), View(hal, out0, 4, words=4)
        hal.mix_poly_coeffs(vo.buf, ms, mx, vi.buf, hal.copy_from_u32(combos), input_size, count)
        got = vo.read("mix out")
        assert_canonical(got, "mix_poly_coeffs")
        eq(got, oracle.mix_poly_coeffs(out0, ms, mx, inp, combos, input_size, count), f"mix_poly_coeffs {input_size} columns")
        vi.unchanged("mix input")


def _f4_words(c):
    return np.array([c, 0, 0, 0], np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("po2,n_eval", [(10, 8), (15, 8), (18, 8), (18, 256)])
def test_batch_evaluate_any_closed_forms(hal, oracle, po2, n_eval):
    """coefficients all P-1 and edge-mixed: at x = 1 the sum, at x = -1 the alternating sum (zero for a constant polynomial), at x = 0
    the constant coefficient.  po2 10: a partial slab; 15 and 18 with 8 points: full 64-step slabs; 18 with 256 points: 256 steps"""
    n = 1 << po2
    coeffs = np.concatenate([np.full(n, P - 1, np.uint32), pattern("mixed", 1, n, po2)])
    canon = O2.dec(coeffs).reshape(2, n)
    sign = np.where(np.arange(n) % 2 == 0, 1, P - 1).astype(np.uint64)
    closed = {ONE: [int(c.sum() % P) for c in canon], MONE: [int((c * sign % P).sum() % P) for c in canon], 0: [int(c[0]) for c in canon]}
    pts = [ONE, MONE, 0]
    which = (np.arange(n_eval) // 3 % 2).astype(np.uint32)
    xs = np.concatenate([_f4_words(pts[j % 3]) for j in range(n_eval)])
    want = np.concatenate([O2.enc([closed[pts[j % 3]][int(which[j])], 0, 0, 0]) for j in range(n_eval)])
    assert want[4:8].tolist() == [0, 0, 0, 0]           # (P-1) * (1 - 1 + 1 - ...) at x = -1 is exactly zero
    for off in ANY_OFFSETS:
        vc = View(hal, coeffs, off)
        out = hal.alloc_extelem(n_eval)
        hal.batch_evaluate_any(vc.buf, 2, hal.copy_from_u32(which), hal.copy_from_extelem(xs), out)
        got = out.to_numpy()
        assert_canonical(got, "batch_evaluate_any")
        eq(got, want, f"batch_evaluate_any off={off}")
        vc.unchanged("coeffs")
    if po2 <= 15:
        eq(got, oracle.batch_evaluate_any(coeffs, 2, po2, which, xs), "vs oracle")


def _times_x_minus_z(q, z):
    """(x - z) * q for canonical Fp4 coefficient rows q (low first) -> one more row"""
    m = q.shape[0]
    p = np.zeros((m + 1, 4), dtype=np.uint64)
    p[1:] = q
    if m:
        p[:m] = (p[:m] + P - O2.f4mul(q, z)) % P
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 8, 9, 64, 65, 8 * 64 + 1])
def test_poly_divide_exact_quotients(hal, oracle, n):
    """p = (x - z) q: the remainder is exactly [0, 0, 0, 0] and the quotient is q, around DIV_CHUNK = 8 and the serial cut-off at 64;
    z = 0, z = 1, z all P-1, z random; q all P-1 and edge-mixed"""
    zs = [_f4_words(0), _f4_words(ONE), np.full(4, P - 1, np.uint32), pattern("mixed", 1, 4, n)]
    for kind in ("pm1", "mixed"):
        for zi, z in enumerate(zs):
            q = O2.dec(pattern(kind, 1, 4 * (n - 1), 10 * n + zi)).reshape(-1, 4)
            p = O2.enc(_times_x_minus_z(q, O2.dec(z))).ravel()
            v = View(hal, p, 4, words=4)
            rem = hal.poly_divide(v.buf, z)
            got = v.read("poly_divide")
            assert_canonical(got, "quotient"); assert_canonical(rem, "remainder")
            assert rem.tolist() == [0, 0, 0, 0], f"remainder {rem} (z #{zi}, {kind})"
            eq(got, np.concatenate([O2.enc(q).ravel(), np.zeros(4, np.uint32)]), f"quotient (z #{zi}, {kind})")
            qo, ro = oracle.poly_divide(p, z)
            eq(got, qo, "vs oracle")
    # combos_divide: three polynomials, each divided by the root it was built with
    q3 = [O2.dec(pattern("mixed", 1, 4 * (n - 1), 7 * n + k)).reshape(-1, 4) for k in range(3)]
    combos = np.concatenate([O2.enc(_times_x_minus_z(q3[k], O2.dec(zs[k]))).ravel() for k in range(3)])
    v = View(hal, combos, 4, words=4)
    rems = hal.combos_divide(v.buf, n, [2, 0, 1], np.concatenate([zs[2], zs[0], zs[1]]))
    assert not rems.any(), f"remainders {rems}"
    eq(v.read("combos_divide"), np.concatenate([np.concatenate([O2.enc(q).ravel(), np.zeros(4, np.uint32)]) for q in q3]), "combos_divide")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [200, 257, 5000, 1 << 14])
def test_prefix_products_zeros_and_saturation(hal, oracle, n):
    """zero elements at positions 0, 63, 64, 255, 256 and the last (PP_CHUNK = 64, serial cut-off 256), all -1, all P-1 words"""
    base = pattern("mixed", 1, 4 * n, n).reshape(n, 4)
    cases = {"mone": np.tile(_f4_words(MONE), n), "pm1": np.full(4 * n, P - 1, np.uint32)}
    for pos in (0, 63, 64, 255, 256, n - 1):
        if pos < n:
            x = base.copy(); x[pos] = 0
            cases[f"zero@{pos}"] = x.ravel()
    for name, x in cases.items():
        v = View(hal, x, 4, words=4)
        hal.prefix_products(v.buf)
        got = v.read("prefix_products")
        assert_canonical(got, name)
        eq(got, oracle.prefix_products(x), f"prefix_products {name}")


@pytest.mark.gpu
@pytest.mark.parametrize("off", ANY_OFFSETS)
def test_fri_fold_and_sum_extelem_cancellations(hal, oracle, off):
    """mix = 0 and mix = 1 with inputs all P-1; inputs whose sums cancel to exactly zero (a + (P - a)); to_add = 64.
    fri_fold in / out and the sum's output at every word offset; the sum's Fp4 input at offset 4"""
    m = 1000
    cancel = pattern("mixed", 4 * 8, m, 1).reshape(4, 8, m)
    cancel = np.stack([cancel, neg(cancel)], axis=2).reshape(-1)          # rows 2k and 2k + 1 of each component cancel
    for x in (np.full(64 * m, P - 1, np.uint32), cancel):
        for mix in (_f4_words(0), _f4_words(ONE), np.full(4, P - 1, np.uint32)):
            vi, vo = View(hal, x, off), View(hal, np.zeros(4 * m, np.uint32), (off + 3) % 4)
            hal.fri_fold(vo.buf, vi.buf, mix)
            got = vo.read("fri_fold")
            assert_canonical(got, "fri_fold")
            want = oracle.fri_fold(x, mix, m)
            eq(got, want, "fri_fold")
            vi.unchanged("fri_fold input")
    assert not oracle.fri_fold(cancel, _f4_words(ONE), m).any()
    count, to_add = 777, 64
    half = pattern("mixed", to_add // 2, 4 * count, 2)
    for x in (np.full(to_add * 4 * count, P - 1, np.uint32), np.concatenate([half, neg(half)])):
        vi, vo = View(hal, x, 4, words=4), View(hal, np.zeros(4 * count, np.uint32), off)
        hal.eltwise_sum_extelem(vo.buf, vi.buf)
        got = vo.read("sum_extelem")
        assert_canonical(got, "eltwise_sum_extelem")
        eq(got, oracle.eltwise_sum_extelem(x, count, to_add), "eltwise_sum_extelem")
    assert not got.any(), "sums that cancel must be exactly zero"


# ---- eval_check / accumulate ------------------------------------------------------------------------------------------------
EC_CIRCUITS = {"MID": lambda: circuit.syn_circuit(**MID), "deep": _deep_tap_circuit, "heavy": lambda: circuit.syn_heavy_circuit(**REDUCED)}
EC_FORMS = {"staged": {}, "register": {"ZKB_EC_STAGED": "0"}, "vm": {"ZKB_EVAL_CHECK": "vm"}, "compact": {"ZKB_EC_FORM": "compact"},
            "flat": {"ZKB_EC_FORM": "flat"}}


def _ec_inputs(b, kind, po2):
    dom = 4 << po2
    fill = 0 if kind == "zero" else P - 1
    accum, code, data = (np.full(n * dom, fill, np.uint32) for n in b.group_size)
    mix, out = np.full(b.mix_size, fill, np.uint32), np.full(b.out_size, fill, np.uint32)
    pm = np.array([ONE, 5, 0, 7], np.uint32) if kind == "zero" else np.full(4, P - 1, np.uint32)
    return accum, code, data, mix, out, pm


def _ec_run(hal, b, ins, po2, off):
    accum, code, data, mix, out, pm = ins
    views = [View(hal, g, off) for g in (accum, code, data)]
    chk = View(hal, np.zeros(16 << po2, np.uint32), off)
    hal.eval_check(chk.buf, b.blob(), *(v.buf for v in views), mix, out, pm, po2)
    for v, name in zip(views, ("accum", "code", "data")):
        v.unchanged(name)
    return chk.read("check")


@pytest.mark.gpu
@pytest.mark.parametrize("form", [pytest.param(f, marks=pytest.mark.slow) if f == "flat" else f for f in EC_FORMS])
@pytest.mark.parametrize("name", list(EC_CIRCUITS))
def test_eval_check_zero_and_saturated_traces(hal, oracle, name, form, monkeypatch):
    """all-zero traces and globals (no check word may be stored as P), and all-(P-1) traces with poly_mix, mix and out all P-1, in
    every form of the JIT and in the device interpreter"""
    for k, v in EC_FORMS[form].items():
        monkeypatch.setenv(k, v)
    b = EC_CIRCUITS[name]()
    po2 = 8
    for kind in ("zero", "pm1"):
        ins = _ec_inputs(b, kind, po2)
        got = _ec_run(hal, b, ins, po2, 0)
        assert_canonical(got, f"check ({kind})")
        eq(got, oracle.eval_check(b.blob(), *ins, po2), f"eval_check {kind}")
        assert kind != "zero" or not got.any(), "zero traces satisfy every constraint: the check polynomial is zero"


@pytest.mark.gpu
@pytest.mark.parametrize("off", [1, 4])
@pytest.mark.parametrize("name", list(EC_CIRCUITS))
def test_eval_check_on_offset_views(hal, oracle, name, off):
    """traces and check buffer as views: at offset 4 the aligned forms run, at offset 1 the register form or (heavy) the interpreter"""
    b = EC_CIRCUITS[name]()
    po2 = 8
    dom = 4 << po2
    rng = np.random.default_rng(off)
    ins = tuple(pattern("mixed", n, dom, int(rng.integers(1 << 30))) for n in b.group_size) + \
        (pattern("mixed", 1, b.mix_size, 1), pattern("mixed", 1, b.out_size, 2), pattern("mixed", 1, 4, 3))
    got = _ec_run(hal, b, ins, po2, off)
    assert_canonical(got, "check")
    eq(got, oracle.eval_check(b.blob(), *ins, po2), f"eval_check off={off}")


@pytest.mark.gpu
def test_heavy_eval_check_on_an_unaligned_view_runs_the_interpreter(oracle, monkeypatch, tmp_path):
    """a heavy circuit on a view that is not 16-byte aligned cannot take the compact / flat form (16-byte column copies); it must go to
    the device interpreter and never compile the straight-line register form (tens of minutes of ptxas at rv32im size).  A context of
    its own, so that no register form compiled earlier in this module sits in the in-memory kernel cache; an empty on-disk cache, so
    that a compile would leave a .zkbj file behind."""
    from zktls_b200.hal import B200Hal
    monkeypatch.setenv("ZKB_EC_FORM", "compact")
    monkeypatch.setenv("ZKB_CACHE_DIR", str(tmp_path))
    b = circuit.syn_heavy_circuit(**REDUCED)
    po2 = 7
    ins = tuple(pattern("mixed", n, 4 << po2, n) for n in b.group_size) + \
        (pattern("mixed", 1, b.mix_size, 1), pattern("mixed", 1, b.out_size, 2), pattern("mixed", 1, 4, 3))
    h = B200Hal(0)
    try:
        got = _ec_run(h, b, ins, po2, 1)
    finally:
        h.close()
    eq(got, oracle.eval_check(b.blob(), *ins, po2), "heavy eval_check on an unaligned view")
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".zkbj")], "a kernel was compiled for the unaligned heavy circuit"


@pytest.mark.gpu
@pytest.mark.parametrize("off", ANY_OFFSETS)
def test_accumulate_saturated_and_zero_products(hal, oracle, off):
    """SYN SMALL with code, data, mix and io all P-1; the grand-product circuit with zero factors in its product column (mix[0] = -1
    cancels the +1 of column 0 where data[0] is zero, mix[1] = 0 zeroes column 3); all groups as views at `off`"""
    po2 = 9
    n = 1 << po2
    b = circuit.syn_circuit(**SMALL); blob = b.blob()
    accum, code, data = (np.full(c * n, P - 1, np.uint32) for c in b.group_size)
    mix, io = np.full(b.mix_size, P - 1, np.uint32), np.full(b.out_size, P - 1, np.uint32)
    gp = _grand_product_circuit()
    rng = np.random.default_rng(off)
    g_accum, g_code, g_data = (pattern("mixed", c, n, c) for c in gp.group_size)
    g_code[:n] = O2.enc(rng.integers(0, 2, size=n))
    g_data[:n][rng.random(n) < 0.3] = 0
    for blob_, ins in ((blob, (accum, code, data, mix, io)), (gp.blob(), (g_accum, g_code, g_data, O2.enc([P - 1, 0]), pattern("mixed", 1, 2, 5)))):
        a, c, d, mx, o = ins
        va, vc, vd = View(hal, a, off), View(hal, c, (off + 1) % 4), View(hal, d, (off + 2) % 4)
        hal.accumulate(blob_, va.buf, vc.buf, vd.buf, mx, o, po2)
        got = va.read("accum")
        assert_canonical(got, "accum")
        eq(got, oracle.accumulate(blob_, a, c, d, mx, o, po2), "accumulate")
        vc.unchanged("code"); vd.unchanged("data")


# ---- whole seals -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fill", [0, P - 1], ids=["zero", "pm1"])
@pytest.mark.parametrize("shape,po2", [(SMALL, 10), (circuit.SYN280, 11)], ids=["SMALL", "SYN280"])
def test_seal_of_constant_traces(hal, oracle, shape, po2, fill):
    """all-zero and all-(P-1) traces through the whole prover: every column interpolates to a constant (n - 1 exact zeros)"""
    from zktls_b200.prover import SegmentProver
    blob = circuit.syn_circuit(**shape).blob()
    n = 1 << po2
    io = np.full(shape["out_size"], fill, np.uint32)
    code, data, accum = (np.full(shape[k] * n, fill, np.uint32) for k in ("code_cols", "data_cols", "accum_cols"))
    gp = SegmentProver(hal, blob)
    seal = gp.prove(po2, io, code, data, accum)
    roots = gp.roots()
    gp.close()
    op = oracle.Prover(blob)
    op.begin(po2, io, code, data)
    seal_o = op.finish(accum)
    eq(roots, op.roots(), "Merkle / FRI roots")
    assert_canonical(seal, "seal")
    eq(seal, seal_o, "seal")
