"""A program (zkb_program) commits a circuit's code trace once per po2 on the device and returns its control ID; provers that use it
prove segments from that commitment given only their data and accum traces (csrc/prover.cu, Program).  Every control ID must be the
code root the CPU oracle commits, and every seal and root the oracle's: on every trace path, across provers and ctxs sharing one
program, after the caller's handle is closed, and interleaved with segments that pass their code trace."""
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


def assert_proof(gp, seal, want, what):
    assert np.array_equal(seal, want[0]), f"seal differs: {what}"
    assert np.array_equal(gp.roots(), want[1]), f"roots differ: {what}"


def trace_b_proof(oracle, blob, po2, seed):
    """A satisfying witness (Montgomery words) and the oracle's mix, seal and roots for it."""
    io, code, data = synth.trace_b_code_data(SMALL, po2, seed)
    code_m, data_m = synth.to_mont(code), synth.to_mont(data)
    op = oracle.Prover(blob)
    mix = op.begin(po2, io, code_m, data_m)
    accum_m = synth.to_mont(synth.trace_b_accum(SMALL, po2, seed, code, data, io, mix))
    return (io, code_m, data_m, accum_m), mix, (op.finish(accum_m), op.roots())


@pytest.mark.parametrize("source", ["host", "device", "device_view_at_4_bytes"])
def test_control_ids_are_the_oracle_code_roots(hal, oracle, source):
    from zktls_b200.prover import Program, control_id
    blob = circuit.syn_circuit(**SMALL).blob()
    prog = Program(hal, blob)
    want = {}
    for po2 in (10, 6, 9):          # not ascending: control_ids() sorts
        io, code, data, accum = synth.trace_a(SMALL, po2, 700 + po2)
        want[po2] = control_id(po2, oracle_proof(oracle, blob, po2, io, code, data, accum)[1][0])
        if source == "host":
            arg = code
        elif source == "device":
            arg = hal.copy_from_elem(code)
        else:
            arg = hal.alloc_elem(code.size + 1).slice(1, code.size)
            arg.copy_from(code)
        assert np.array_equal(prog.commit(po2, arg), want[po2]), f"po2 {po2}"
    ids = prog.control_ids()
    assert ids.shape == (3, 9) and ids.dtype == np.uint32
    assert np.array_equal(ids, np.stack([want[k] for k in (6, 9, 10)]))
    prog.close()


@pytest.mark.parametrize("side", ["device", "host"])
def test_prove_from_the_program_matches_the_oracle(hal, oracle, side):
    from zktls_b200.prover import Program, SegmentProver
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code, data, accum = synth.trace_a(SMALL, po2, 801)
    want = oracle_proof(oracle, blob, po2, io, code, data, accum)
    prog = Program(hal, blob)
    prog.commit(po2, code)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    d, a = (hal.copy_from_elem(data), hal.copy_from_elem(accum)) if side == "device" else (data, accum)
    for i in range(2):
        assert_proof(gp, gp.prove(po2, io, None, d, a), want, f"segment {i}")
    gp.close(); prog.close()


def test_begin_finish_from_the_program_verifies_against_its_control_ids_alone(hal, oracle):
    from zktls_b200.prover import Program, SegmentProver, verify_segment
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    (io, code_m, data_m, accum_m), mix_o, want = trace_b_proof(oracle, blob, po2, 55)
    prog = Program(hal, blob)
    prog.commit(po2, code_m)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    for i, (d, a) in enumerate(((data_m, accum_m), (hal.copy_from_elem(data_m), hal.copy_from_elem(accum_m)))):
        assert np.array_equal(gp.begin(po2, io, None, d), mix_o), f"mix of segment {i}"
        seal = gp.finish(a)
        assert_proof(gp, seal, want, f"segment {i}")
    assert verify_segment(blob, seal, prog.control_ids())[0] == po2
    gp.close(); prog.close()


def test_staged_path_from_the_program_with_an_accum_trace(hal, oracle):
    from zktls_b200.prover import Program, SegmentProver
    po2 = 9
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code, _, _ = synth.trace_a(SMALL, po2, 900)
    segs = [synth.trace_a(SMALL, po2, 901 + k)[2:] for k in range(3)]          # per-segment data and accum, one code trace
    want = [oracle_proof(oracle, blob, po2, io, code, d, a) for d, a in segs]
    prog = Program(hal, blob)
    prog.commit(po2, code)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    gp.stage(po2, None, *segs[0])
    for k in range(len(segs)):
        if k + 1 < len(segs):
            gp.stage(po2, None, *segs[k + 1])
        assert_proof(gp, gp.prove_staged(io), want[k], f"segment {k}")
    gp.close(); prog.close()


def test_staged_path_from_the_program_with_device_accumulate(hal, oracle):
    """No code and no accum trace staged: the witness program reads the program's copy of the code trace."""
    from zktls_b200.prover import Program, SegmentProver
    po2 = 9
    n = 1 << po2
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code, data = synth.trace_b_code_data(SMALL, po2, 66)
    code_m = synth.to_mont(code)
    datas = [synth.to_mont(data), synth.to_mont(synth.trace_b_code_data(SMALL, po2, 67)[2])]
    want = []
    for d in datas:
        op = oracle.Prover(blob)
        mix = op.begin(po2, io, code_m, d)
        acc = oracle.accumulate(blob, np.zeros(SMALL["accum_cols"] * n, np.uint32), code_m, d, mix, io, po2)
        want.append((op.finish(acc), op.roots()))
    prog = Program(hal, blob)
    prog.commit(po2, code_m)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    seq = [0, 1, 0]
    gp.stage(po2, None, datas[seq[0]])
    for i, k in enumerate(seq):
        if i + 1 < len(seq):
            gp.stage(po2, None, datas[seq[i + 1]])
        assert_proof(gp, gp.prove_staged(io), want[k], f"segment {i}")
    gp.close(); prog.close()


def test_one_program_two_po2_alternating(hal, oracle):
    from zktls_b200.prover import Program, SegmentProver
    blob = circuit.syn_circuit(**SMALL).blob()
    traces = {po2: synth.trace_a(SMALL, po2, 1000 + po2) for po2 in (9, 10)}
    want = {po2: oracle_proof(oracle, blob, po2, *t) for po2, t in traces.items()}
    prog = Program(hal, blob)
    for po2, (_, code, _, _) in traces.items():
        prog.commit(po2, code)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    for i, po2 in enumerate((10, 9, 10)):
        io, _, data, accum = traces[po2]
        assert_proof(gp, gp.prove(po2, io, None, data, accum), want[po2], f"segment {i} (po2 {po2})")
    gp.close(); prog.close()


def test_program_segments_neither_read_nor_change_the_provers_own_code_cache(hal, oracle):
    """program(A), trace(B), program(A), trace(B) on one prover, B one word away from A: the second B is a hit in the prover's own
    cache, and neither program segment may see B's commitment."""
    from zktls_b200.prover import Program, SegmentProver
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code_a, data, accum = synth.trace_a(SMALL, po2, 1100)
    code_b = code_a.copy()
    code_b[5] = (int(code_b[5]) + 1) % P
    want = {"A": oracle_proof(oracle, blob, po2, io, code_a, data, accum), "B": oracle_proof(oracle, blob, po2, io, code_b, data, accum)}
    prog = Program(hal, blob)
    prog.commit(po2, code_a)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    for i, k in enumerate("ABAB"):
        assert_proof(gp, gp.prove(po2, io, None if k == "A" else code_b, data, accum), want[k], f"segment {i} ({k})")
    gp.close(); prog.close()


def test_two_ctxs_share_one_program(hal, oracle):
    from zktls_b200.hal import B200Hal
    from zktls_b200.prover import Program, SegmentProver
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    io_a, code, data_a, accum_a = synth.trace_a(SMALL, po2, 1200)
    io_b, _, data_b, accum_b = synth.trace_a(SMALL, po2, 1201)
    want_a = oracle_proof(oracle, blob, po2, io_a, code, data_a, accum_a)
    want_b = oracle_proof(oracle, blob, po2, io_b, code, data_b, accum_b)
    hal_b = B200Hal(0)
    prog = Program(hal, blob)
    prog.commit(po2, code)
    ga, gb = SegmentProver(hal, blob), SegmentProver(hal_b, blob)
    ga.use_program(prog); gb.use_program(prog)
    d_data_b, d_accum_b = hal_b.copy_from_elem(data_b), hal_b.copy_from_elem(accum_b)
    ga.begin(po2, io_a, None, data_a)
    gb.begin(po2, io_b, None, d_data_b)
    assert_proof(ga, ga.finish(accum_a), want_a, "prover A")
    assert_proof(gb, gb.finish(d_accum_b), want_b, "prover B")
    ga.close(); gb.close(); prog.close()
    del d_data_b, d_accum_b
    hal_b.close()


def test_prover_keeps_a_closed_program_alive_until_it_detaches(hal, oracle):
    """The program outlives the ctx it was made with and the caller's handle; detaching makes code=None an error again."""
    from zktls_b200.hal import B200Hal
    from zktls_b200.prover import Program, SegmentProver
    from zktls_b200._lib import ZkbError
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code, data, accum = synth.trace_a(SMALL, po2, 1300)
    want = oracle_proof(oracle, blob, po2, io, code, data, accum)
    tmp = B200Hal(0)
    prog = Program(tmp, blob)
    prog.commit(po2, code)
    tmp.close()
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    prog.close()
    assert_proof(gp, gp.prove(po2, io, None, data, accum), want, "after the handle was closed")
    gp.use_program(None)
    with pytest.raises(ZkbError, match="null argument"):
        gp.prove(po2, io, None, data, accum)
    with pytest.raises(ValueError):
        gp.use_program(prog)
    gp.close()


def test_errors_are_strings_and_the_prover_stays_usable(hal, oracle):
    from zktls_b200.prover import Program, SegmentProver
    from zktls_b200._lib import ZkbError
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    io, code, data, accum = synth.trace_a(SMALL, po2, 1400)
    want = oracle_proof(oracle, blob, po2, io, code, data, accum)
    io9, _, data9, accum9 = synth.trace_a(SMALL, 9, 1401)
    prog = Program(hal, blob)
    prog.commit(po2, code)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    assert_proof(gp, gp.prove(po2, io, None, data, accum), want, "first segment")

    def still_usable(what):
        assert_proof(gp, gp.prove(po2, io, None, data, accum), want, f"after: {what}")

    with pytest.raises(ZkbError, match="po2 9"):
        gp.prove(9, io9, None, data9, accum9)
    assert_proof(gp, gp.seal(), want, "the refused segment touched the transcript")
    still_usable("no commitment at po2 9 (prove)")
    with pytest.raises(ZkbError, match="po2 9"):
        gp.stage(9, None, data9, accum9)
    gp.stage(po2, None, data, accum)
    assert_proof(gp, gp.prove_staged(io), want, "staged after a refused stage")
    still_usable("no commitment at po2 9 (stage)")
    other = Program(hal, circuit.syn_circuit(**dict(SMALL, data_cols=7)).blob())
    with pytest.raises(ZkbError, match="circuit blob"):
        gp.use_program(other)
    other.close()
    still_usable("a program of another circuit")
    with pytest.raises(ZkbError, match="already"):
        prog.commit(po2, code)
    still_usable("the same po2 committed twice")
    for bad in (5, 25):
        with pytest.raises(ZkbError, match="out of range"):
            prog.commit(bad, np.zeros(SMALL["code_cols"] << min(bad, 10), np.uint32))
    still_usable("a po2 outside [6, 24]")
    assert prog.control_ids().shape == (1, 9)
    gp.close(); prog.close()


def test_a_seal_of_another_code_trace_is_rejected_against_the_programs_control_ids(hal, oracle):
    from zktls_b200.prover import Program, SegmentProver, verify_segment, seal_code_root
    from zktls_b200._lib import ZkbError
    po2 = 10
    blob = circuit.syn_circuit(**SMALL).blob()
    (_, code_m, _, _), _, _ = trace_b_proof(oracle, blob, po2, 55)
    (io, other_code, data_m, accum_m), _, want = trace_b_proof(oracle, blob, po2, 56)      # also satisfies the constraints
    prog = Program(hal, blob)
    prog.commit(po2, code_m)
    gp = SegmentProver(hal, blob)
    seal = gp.prove(po2, io, other_code, data_m, accum_m)
    assert_proof(gp, seal, want, "trace segment")
    assert seal_code_root(blob, seal)[0] == po2          # every other check passes
    with pytest.raises(ZkbError):
        verify_segment(blob, seal, prog.control_ids())
    gp.close(); prog.close()


def test_program_segment_launches_fewer_kernels(hal):
    """Against the first trace segment (full commit) and against a hit in the prover's own cache (k_differ does not run)."""
    from zktls_b200.prover import Program, SegmentProver
    po2 = 12
    blob = circuit.syn_circuit(**circuit.SYN280).blob()
    io, code, data, accum = synth.trace_a(circuit.SYN280, po2, 600)
    prog = Program(hal, blob)
    prog.commit(po2, code)
    gp = SegmentProver(hal, blob)
    l0 = hal.kernel_launches()
    s1 = gp.prove(po2, io, code, data, accum)
    l1 = hal.kernel_launches()
    s2 = gp.prove(po2, io, code, data, accum)
    l2 = hal.kernel_launches()
    gp.use_program(prog)
    s3 = gp.prove(po2, io, None, data, accum)
    l3 = hal.kernel_launches()
    gp.close(); prog.close()
    assert np.array_equal(s1, s2) and np.array_equal(s1, s3)
    first, hit, program = l1 - l0, l2 - l1, l3 - l2
    assert program < first and program <= hit - 1, f"first {first}, cache hit {hit}, program {program} launches"


@pytest.mark.slow
def test_full_size_program_segment_equals_the_trace_segment(hal):
    """The benchmark segment (SYN-280, 2^20 cycles, device-resident traces): the control ID is the code root of the trace proof, and
    the program seal is the trace seal."""
    import torch
    from zktls_b200.hal import Buffer
    from zktls_b200.prover import Program, SegmentProver, control_id
    shape, po2 = circuit.SYN280, 20
    n = 1 << po2
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(0xC0DE)
    ts = [torch.randint(0, P, (shape[k] * n,), device=dev, dtype=torch.int64, generator=g).to(torch.int32) for k in ("code_cols", "data_cols", "accum_cols")]
    torch.cuda.synchronize()          # the ctx has its own stream
    bufs = [Buffer(hal, t.data_ptr(), t.numel(), 1, owner=t) for t in ts]
    io = np.arange(shape["out_size"], dtype=np.uint32)
    blob = circuit.syn_circuit(**shape).blob()
    gp = SegmentProver(hal, blob)
    s1, r1 = gp.prove(po2, io, *bufs), gp.roots()
    prog = Program(hal, blob)
    assert np.array_equal(prog.commit(po2, bufs[0]), control_id(po2, r1[0]))
    gp.use_program(prog)
    s2, r2 = gp.prove(po2, io, None, *bufs[1:]), gp.roots()
    gp.close(); prog.close()
    assert s1.size == 67489
    assert np.array_equal(s1, s2) and np.array_equal(r1, r2)
