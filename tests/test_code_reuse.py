"""A prover keeps the last code-group commitment it completed and reuses it when the next segment's code trace is equal to it,
word for word (csrc/prover.cu, commit_code).  Whatever a prover committed before, every seal and root must be the one the CPU
oracle (or a fresh prover) gives for the same inputs: on every trace path, across a change of po2, and for a code trace that
differs from the retained one in a single word of a buffer the caller rewrote in place."""
import numpy as np
import pytest

from zktls_b200 import circuit, synth

pytestmark = pytest.mark.gpu

P = 2013265921
SMALL = dict(accum_cols=4, code_cols=3, data_cols=6, mix_size=5, out_size=4)


@pytest.fixture(scope="module")
def hal():
    from zktls_b200.hal import B200Hal
    h = B200Hal(0)
    yield h
    h.close()


def oracle_proof(oracle, blob, po2, io, code, data, accum):
    op = oracle.Prover(blob)
    op.begin(po2, io, code, data)
    return op.finish(accum), op.roots()


def one_word_changed(code, at):
    out = code.copy()
    out[at] = (int(out[at]) + 1) % P
    return out


def assert_proof(gp, seal, want, what):
    assert np.array_equal(seal, want[0]), f"seal differs: {what}"
    assert np.array_equal(gp.roots(), want[1]), f"roots differ: {what}"


@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "misaligned_view"])
@pytest.mark.parametrize("where", ["first_column", "last_word"])
def test_a_a_b_a_in_one_device_buffer_rewritten_in_place(hal, oracle, where, offset):
    """B differs from A in one word; the code buffer is the same pointer every time (at a 4-byte offset in the misaligned case)."""
    from zktls_b200.prover import SegmentProver
    po2 = 10
    n = 1 << po2
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code_a, data, accum = synth.trace_a(SMALL, po2, 301)
    code_b = one_word_changed(code_a, n // 2 if where == "first_column" else code_a.size - 1)
    want = {"A": oracle_proof(oracle, blob, po2, io, code_a, data, accum), "B": oracle_proof(oracle, blob, po2, io, code_b, data, accum)}
    d_code = hal.alloc_elem(code_a.size + offset).slice(offset, code_a.size)
    d_data, d_accum = hal.copy_from_elem(data), hal.copy_from_elem(accum)
    gp = SegmentProver(hal, blob)
    for i, k in enumerate("AABA"):
        d_code.copy_from(code_a if k == "A" else code_b)
        assert_proof(gp, gp.prove(po2, io, d_code, d_data, d_accum), want[k], f"segment {i} ({k})")
    gp.close()


def test_po2_change_and_back_on_the_host_pointer_path(hal, oracle):
    from zktls_b200.prover import SegmentProver
    blob = circuit.syn_circuit(**SMALL).blob()
    traces = {po2: synth.trace_a(SMALL, po2, 400 + po2) for po2 in (9, 10)}
    want = {po2: oracle_proof(oracle, blob, po2, *t) for po2, t in traces.items()}
    gp = SegmentProver(hal, blob)
    for i, po2 in enumerate((10, 10, 9, 9, 10)):
        assert_proof(gp, gp.prove(po2, *traces[po2]), want[po2], f"segment {i} (po2 {po2})")
    gp.close()


def test_split_begin_finish_path_and_the_reused_seal_verifies(hal, oracle):
    """A satisfying witness through begin() / finish(), from host arrays and then from device buffers: the mix, the seal and the
    roots of the second (reused) segment are the oracle's, and zkb_verify_segment accepts it with the control ID of its own code root."""
    from zktls_b200.prover import SegmentProver, verify_segment, control_id
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code, data = synth.trace_b_code_data(SMALL, po2, 55)
    code_m, data_m = synth.to_mont(code), synth.to_mont(data)
    op = oracle.Prover(blob)
    mix_o = op.begin(po2, io, code_m, data_m)
    accum_m = synth.to_mont(synth.trace_b_accum(SMALL, po2, 55, code, data, io, mix_o))
    want = (op.finish(accum_m), op.roots())
    gp = SegmentProver(hal, blob)
    for i, (c, d, a) in enumerate(((code_m, data_m, accum_m), tuple(hal.copy_from_elem(t) for t in (code_m, data_m, accum_m)))):
        assert np.array_equal(gp.begin(po2, io, c, d), mix_o), f"mix of segment {i}"
        seal = gp.finish(a)
        assert_proof(gp, seal, want, f"segment {i}")
    assert verify_segment(blob, seal, control_id(po2, gp.roots()[0]))[0] == po2
    gp.close()


def test_staged_path_a_a_b_a(hal, oracle):
    """Double-buffered staging: the code trace of each segment lands in a different staging slot."""
    from zktls_b200.prover import SegmentProver
    po2 = 9
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code_a, data, accum = synth.trace_a(SMALL, po2, 500)
    code_b = one_word_changed(code_a, 7)
    want = {"A": oracle_proof(oracle, blob, po2, io, code_a, data, accum), "B": oracle_proof(oracle, blob, po2, io, code_b, data, accum)}
    seq = "AABA"
    gp = SegmentProver(hal, blob)
    gp.stage(po2, code_a, data, accum)
    for i, k in enumerate(seq):
        if i + 1 < len(seq):
            gp.stage(po2, code_a if seq[i + 1] == "A" else code_b, data, accum)
        assert_proof(gp, gp.prove_staged(io), want[k], f"segment {i} ({k})")
    gp.close()


def test_staged_path_with_device_accumulate_a_a_b_a(hal, oracle):
    """No accum trace staged: the witness program reads the staged code trace, so a reused code commitment must not change it."""
    from zktls_b200.prover import SegmentProver
    po2 = 9
    n = 1 << po2
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code, data = synth.trace_b_code_data(SMALL, po2, 66)
    code_a, data_m = synth.to_mont(code), synth.to_mont(data)
    code_b = one_word_changed(code_a, code_a.size - 1)
    want = {}
    for k, c in (("A", code_a), ("B", code_b)):
        op = oracle.Prover(blob)
        mix = op.begin(po2, io, c, data_m)
        acc = oracle.accumulate(blob, np.zeros(SMALL["accum_cols"] * n, np.uint32), c, data_m, mix, io, po2)
        want[k] = (op.finish(acc), op.roots())
    seq = "AABA"
    gp = SegmentProver(hal, blob)
    gp.stage(po2, code_a, data_m)
    for i, k in enumerate(seq):
        if i + 1 < len(seq):
            gp.stage(po2, code_a if seq[i + 1] == "A" else code_b, data_m)
        assert_proof(gp, gp.prove_staged(io), want[k], f"segment {i} ({k})")
    gp.close()


def test_second_identical_segment_launches_fewer_kernels(hal):
    from zktls_b200.prover import SegmentProver
    po2 = 12
    blob = circuit.syn_circuit(**circuit.SYN280).blob()
    io, code, data, accum = synth.trace_a(circuit.SYN280, po2, 600)
    gp = SegmentProver(hal, blob)
    l0 = hal.kernel_launches()
    s1 = gp.prove(po2, io, code, data, accum)
    l1 = hal.kernel_launches()
    s2 = gp.prove(po2, io, code, data, accum)
    l2 = hal.kernel_launches()
    gp.close()
    assert np.array_equal(s1, s2)
    assert l2 - l1 < l1 - l0, f"first segment {l1 - l0} launches, second {l2 - l1}"


@pytest.mark.slow
def test_two_full_size_segments_on_one_prover_give_identical_seals(hal):
    """The benchmark segment (SYN-280, 2^20 cycles, device-resident traces) twice on one prover: the second reuses the code group."""
    import torch
    from zktls_b200.hal import Buffer
    from zktls_b200.prover import SegmentProver
    shape, po2 = circuit.SYN280, 20
    n = 1 << po2
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(0xC0DE)
    ts = [torch.randint(0, P, (shape[k] * n,), device=dev, dtype=torch.int64, generator=g).to(torch.int32) for k in ("code_cols", "data_cols", "accum_cols")]
    torch.cuda.synchronize()          # the ctx has its own stream
    bufs = [Buffer(hal, t.data_ptr(), t.numel(), 1, owner=t) for t in ts]
    io = np.arange(shape["out_size"], dtype=np.uint32)
    gp = SegmentProver(hal, circuit.syn_circuit(**shape).blob())
    l0 = hal.kernel_launches()
    s1, r1 = gp.prove(po2, io, *bufs), gp.roots()
    l1 = hal.kernel_launches()
    s2, r2 = gp.prove(po2, io, *bufs), gp.roots()
    l2 = hal.kernel_launches()
    gp.close()
    assert s1.size == 67489
    assert np.array_equal(s1, s2) and np.array_equal(r1, r2)
    assert l2 - l1 < l1 - l0
