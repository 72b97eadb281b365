"""A session (zkb_session) proves a queue of segments on one or more devices with its own worker threads, one program per device and the
staged pipeline (csrc/session.cpp).  Every seal must be the CPU oracle's for that ticket's own inputs: whatever the number of provers
in flight, the order tickets are waited in, the mix of host and device accum, the number of devices and host threads, and segments that
fail around it.  Freeing a session with work outstanding must return and leave no thread behind."""
import os
import threading

import numpy as np
import pytest

from zktls_b200 import circuit, synth

pytestmark = pytest.mark.gpu

P = 2013265921
SMALL = dict(accum_cols=4, code_cols=3, data_cols=6, mix_size=5, out_size=4)
BLOB = circuit.syn_circuit(**SMALL).blob()


@pytest.fixture(scope="module")
def hal():
    from zktls_b200.hal import B200Hal
    h = B200Hal(0)
    yield h
    h.close()


def code_trace(po2):
    """The one code trace of every segment at po2."""
    return synth.trace_a(SMALL, po2, 7000 + po2)[1]


_seals = {}


def segment(oracle, po2, k, device_accum=False):
    """Segment k at po2: its own io, data (and accum unless device_accum), and the oracle's seal for them."""
    key = (po2, k, device_accum)
    io, _, data, accum = synth.trace_a(SMALL, po2, 8000 + 64 * po2 + k)
    if key not in _seals:
        code = code_trace(po2)
        op = oracle.Prover(BLOB)
        mix = op.begin(po2, io, code, data)
        if device_accum:
            accum = oracle.accumulate(BLOB, np.zeros(SMALL["accum_cols"] << po2, np.uint32), code, data, mix, io, po2)
        _seals[key] = op.finish(accum)
    return io, data, None if device_accum else accum, _seals[key]


def session(devices=(0,), inflight=2, po2s=(9, 10), blob=BLOB):
    from zktls_b200.prover import Session
    s = Session(blob, devices=None if devices is None else list(devices), inflight=inflight)
    for po2 in po2s:
        s.commit(po2, code_trace(po2))
    return s


@pytest.mark.parametrize("inflight", [1, 2, 3])
def test_interleaved_po2_waited_in_reverse_order(oracle, inflight):
    s = session(inflight=inflight)
    segs = [(9 if k % 2 == 0 else 10, k) for k in range(12)]
    tickets = []
    for po2, k in segs:
        io, data, accum, _ = segment(oracle, po2, k)
        tickets.append(s.submit(po2, io, data, accum))
    assert tickets == sorted(tickets) and len(set(tickets)) == len(tickets)
    for (po2, k), t in reversed(list(zip(segs, tickets))):
        assert np.array_equal(s.wait(t), segment(oracle, po2, k)[3]), f"segment {k} (po2 {po2}, ticket {t})"
    s.close()


def test_device_and_host_accum_in_one_session(oracle):
    s = session(inflight=2, po2s=(9,))
    jobs = [(k, k % 2 == 1) for k in range(6)]
    tickets = [s.submit(9, *segment(oracle, 9, k, dev)[:3]) for k, dev in jobs]
    for (k, dev), t in zip(jobs, tickets):
        assert np.array_equal(s.wait(t), segment(oracle, 9, k, dev)[3]), f"segment {k} ({'device' if dev else 'host'} accum)"
    s.close()


def test_control_ids_and_every_seal_verifies(hal, oracle):
    """Satisfying witnesses (trace B: one code trace per po2, each segment its own io and data, accum from the witness program), so every
    seal verifies against the session's control IDs."""
    from zktls_b200.prover import Program, control_id, verify_segment
    s = session(inflight=2, po2s=())
    prog = Program(hal, BLOB)
    codes, segs = {}, []
    for po2 in (10, 9):          # not ascending: control_ids() sorts
        n = 1 << po2
        codes[po2] = synth.trace_b_code_data(SMALL, po2, 7100 + po2)[1]
        code_m = synth.to_mont(codes[po2])
        for k in range(2):
            io, _, data = synth.trace_b_code_data(SMALL, po2, 7200 + 16 * po2 + k, code=codes[po2])
            data_m = synth.to_mont(data)
            op = oracle.Prover(BLOB)
            mix = op.begin(po2, io, code_m, data_m)
            accum = oracle.accumulate(BLOB, np.zeros(SMALL["accum_cols"] * n, np.uint32), code_m, data_m, mix, io, po2)
            segs.append((po2, io, data_m, op.finish(accum), control_id(po2, op.roots()[0])))
        want = segs[-1][4]
        assert np.array_equal(s.commit(po2, code_m), want), f"po2 {po2}"
        assert np.array_equal(prog.commit(po2, code_m), want), f"po2 {po2} (Program)"
    ids = s.control_ids()
    assert ids.shape == (2, 9) and list(ids[:, 0]) == [9, 10]
    assert np.array_equal(ids, prog.control_ids())
    prog.close()
    tickets = [s.submit(po2, io, data_m) for po2, io, data_m, _, _ in segs]
    for (po2, _, _, want_seal, _), t in zip(segs, tickets):
        seal = s.wait(t)
        assert np.array_equal(seal, want_seal), f"po2 {po2}"
        assert verify_segment(BLOB, seal, ids)[0] == po2
    s.close()


def test_every_visible_device(oracle):
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs two or more devices")
    inflight = 2
    s = session(devices=None, inflight=inflight, po2s=(9,))
    jobs = [(k, k % 3 == 0) for k in range(3 * ndev * inflight)]
    tickets = [s.submit(9, *segment(oracle, 9, k, dev)[:3]) for k, dev in jobs]
    for (k, dev), t in zip(jobs, tickets):
        assert np.array_equal(s.wait(t), segment(oracle, 9, k, dev)[3]), f"segment {k}"
    s.close()


def test_refusals_at_submit_commit_and_wait(oracle):
    from zktls_b200._lib import ZkbError
    s = session(inflight=1, po2s=(9,))
    io, data, accum, want = segment(oracle, 9, 0)
    with pytest.raises(ZkbError, match="po2 10"):
        s.submit(10, io, data, accum)
    with pytest.raises(ZkbError, match="already"):
        s.commit(9, code_trace(9))
    with pytest.raises(ZkbError, match="null data"):
        s.submit(9, io, None, accum)
    with pytest.raises(ZkbError, match="unknown"):
        s.wait(12345)
    t = s.submit(9, io, data, accum)
    assert np.array_equal(s.wait(t), want)
    with pytest.raises(ZkbError, match="released"):
        s.wait(t)
    assert s.control_ids().shape == (1, 9)
    s.close()
    b = circuit.syn_circuit(**SMALL)
    b.wsteps = []
    s = session(inflight=1, po2s=(9,), blob=b.blob())
    with pytest.raises(ZkbError, match="no witness program"):
        s.submit(9, io, data)
    s.close()


@pytest.mark.parametrize("inflight", [1, 2])
def test_an_io_word_out_of_range_fails_only_its_own_ticket(oracle, inflight):
    """With one worker the segment after the bad one is prefetched onto the prover that fails: it must be staged again, not failed."""
    from zktls_b200._lib import ZkbError
    s = session(inflight=inflight, po2s=(9,))
    ks = [0, 1, "bad", 2, 3, 4]
    tickets = []
    for k in ks:
        if k == "bad":
            io, data, accum, _ = segment(oracle, 9, 5)
            io = io.copy(); io[1] = P
        else:
            io, data, accum, _ = segment(oracle, 9, k)
        tickets.append(s.submit(9, io, data, accum))
    for k, t in zip(ks, tickets):
        if k == "bad":
            with pytest.raises(ZkbError, match="io word"):
                s.wait(t)
        else:
            assert np.array_equal(s.wait(t), segment(oracle, 9, k)[3]), f"segment {k}"
    s.close()


def test_close_with_tickets_outstanding_leaves_no_thread(oracle):
    def threads():
        return len(os.listdir("/proc/self/task"))

    io, data, accum, want = segment(oracle, 9, 0)
    s = session(inflight=3, po2s=(9,))          # the device's runtime threads exist after the first session
    assert np.array_equal(s.wait(s.submit(9, io, data, accum)), want)
    s.close()
    before = threads()
    s = session(inflight=3, po2s=(9,))
    assert threads() > before
    for k in range(6):
        s.submit(9, *segment(oracle, 9, k)[:3])
    s.close()
    assert threads() == before
    s = session(inflight=3, po2s=(9,))
    assert np.array_equal(s.wait(s.submit(9, io, data, accum)), want)
    s.close()


def test_four_host_threads_submit_and_wait_on_one_session(oracle):
    s = session(inflight=3)
    jobs = {w: [(9 if (w + j) % 2 else 10, 4 * w + j, j == 1) for j in range(3)] for w in range(4)}
    for w in jobs:
        for po2, k, dev in jobs[w]:
            segment(oracle, po2, k, dev)         # oracle seals before the threads start
    bad = []

    def work(w):
        try:
            tickets = [s.submit(po2, *segment(oracle, po2, k, dev)[:3]) for po2, k, dev in jobs[w]]
            for (po2, k, dev), t in zip(jobs[w], tickets):
                if not np.array_equal(s.wait(t), segment(oracle, po2, k, dev)[3]):
                    bad.append((w, k))
        except Exception as e:      # noqa: BLE001
            bad.append((w, repr(e)))

    ths = [threading.Thread(target=work, args=(w,)) for w in jobs]
    for th in ths: th.start()
    for th in ths: th.join()
    s.close()
    assert not bad, bad


@pytest.mark.slow
def test_full_size_session_with_device_accum(oracle):
    """Six SYN-280 2^20 segments (pageable host traces, accum computed on the device): the first seal is the oracle's, and every seal is
    the seal of a staged SegmentProver proof of the same inputs from a Program."""
    from zktls_b200.hal import B200Hal
    from zktls_b200.prover import Program, SegmentProver, Session
    shape, po2 = circuit.SYN280, 20
    n = 1 << po2
    blob = circuit.syn_circuit(**shape).blob()
    rng = np.random.default_rng(0x5E55)
    code = rng.integers(0, P, size=shape["code_cols"] * n, dtype=np.uint32)
    datas = [rng.integers(0, P, size=shape["data_cols"] * n, dtype=np.uint32) for _ in range(3)]
    ios = [rng.integers(0, P, size=shape["out_size"], dtype=np.uint32) for _ in range(6)]
    s = Session(blob, devices=[0], inflight=3)
    s.commit(po2, code)
    tickets = [s.submit(po2, io, datas[k % 3]) for k, io in enumerate(ios)]
    seals = [s.wait(t) for t in tickets]
    s.close()

    hal = B200Hal(0)
    prog = Program(hal, blob)
    prog.commit(po2, code)
    gp = SegmentProver(hal, blob)
    gp.use_program(prog)
    for k, io in enumerate(ios):
        gp.stage(po2, None, datas[k % 3])
        assert np.array_equal(seals[k], gp.prove_staged(io)), f"segment {k}"
    gp.close(); prog.close(); hal.close()

    op = oracle.Prover(blob)
    mix = op.begin(po2, ios[0], code, datas[0])
    accum = oracle.accumulate(blob, np.zeros(shape["accum_cols"] * n, np.uint32), code, datas[0], mix, ios[0], po2)
    assert np.array_equal(seals[0], op.finish(accum))
    assert seals[0].size == 67489
