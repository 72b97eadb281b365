"""Host-side mirror of the segment prover over the libzkb200 C-ABI.

`SegmentProver` corresponds to risc0-zkp `prove::Prover` driven by the circuit crate's `prove_segment` (SURVEY.md
App. D.2): begin() commits `code` and `data` and returns the Fiat-Shamir `mix` globals the caller's accumulate step
needs; finish() commits `accum` and finalizes; prove() is the one-shot form.  Traces may be numpy arrays (host) or
`hal.Buffer`s (device).  `Program` commits a circuit's code trace once per po2 on a device; a prover that uses it takes
code=None and proves from that commitment.  `Session` proves a queue of segments on every device from one object.
"""
import ctypes as C
import threading

import numpy as np

from ._lib import lib, check
from .hal import B200Hal, Buffer, _hp, _sz


def _trace_arg(t):
    if isinstance(t, Buffer):
        return C.c_void_p(t.ptr), True
    arr = np.ascontiguousarray(t, dtype=np.uint32)
    return arr, False


def _trace_args(*traces):
    """(arrays / pointers to keep alive, C pointers, on_device) for the traces given; None is a NULL pointer.  The traces given must
    all be host arrays or all be device buffers."""
    args = [None if t is None else _trace_arg(t) for t in traces]
    sides = {a[1] for a in args if a is not None}
    assert len(sides) <= 1, "the traces given must all be host arrays or all be device buffers"
    dev = sides.pop() if sides else False
    return args, [C.c_void_p(None) if a is None else SegmentProver._ptr(a[0], dev) for a in args], dev


class Program:
    """A circuit's code commitments on one device, one per po2 (zkb_program): commit() commits a code trace once and returns its
    control ID; any number of SegmentProvers on the device prove from it after use_program(), given code=None."""

    def __init__(self, hal: B200Hal, circuit_blob):
        self.blob = np.ascontiguousarray(circuit_blob, dtype=np.uint32)
        self.h = C.c_void_p()
        check(lib().zkb_program_new(hal.ctx, _hp(self.blob), _sz(self.blob.size), C.byref(self.h)))

    def commit(self, po2, code):
        """Commits `code` (numpy array or hal.Buffer) at po2; returns the control ID (po2, code root[8]) as 9 words."""
        _, (c,), dev = _trace_args(code)
        out = np.zeros(9, np.uint32)
        check(lib().zkb_program_commit(self.h, C.c_int(po2), c, C.c_int(int(dev)), _hp(out)))
        return out

    def control_ids(self):
        """(k, 9) array of every committed (po2, code root), ascending po2: the table verify_segment takes."""
        n = C.c_size_t(); check(lib().zkb_program_control_ids(self.h, C.byref(n), None))
        out = np.zeros((n.value, 9), np.uint32)
        check(lib().zkb_program_control_ids(self.h, C.byref(n), _hp(out)))
        return out[: n.value]

    def close(self):
        """Releases this handle; provers that use the program keep it alive."""
        if self.h:
            check(lib().zkb_program_free(self.h)); self.h = C.c_void_p()


class Session:
    """The continuation segments of one session on one or more devices (zkb_session): `inflight` staged provers per device, one Program
    per device, one queue.  commit() the code trace once per po2, submit() each segment's io and host traces (numpy arrays, ideally over
    pinned memory) for a ticket, wait() for its seal.  submit and wait may be called from several threads.  devices=None: every visible
    device."""

    def __init__(self, circuit_blob, devices=None, inflight=3):
        self.blob = np.ascontiguousarray(circuit_blob, dtype=np.uint32)
        devs = None if devices is None else np.ascontiguousarray(devices, dtype=np.int32)
        self.h = C.c_void_p()
        self._keep, self._lock = {}, threading.Lock()      # ticket -> the traces the library reads until its seal is collected
        check(lib().zkb_session_new(_hp(self.blob), _sz(self.blob.size), None if devs is None else devs.ctypes.data_as(C.POINTER(C.c_int)),
                                    _sz(0 if devs is None else devs.size), C.c_int(inflight), C.byref(self.h)))

    def commit(self, po2, code):
        """Commits the host code trace at po2 on every device of the session; returns the control ID (po2, code root[8])."""
        code = np.ascontiguousarray(code, dtype=np.uint32)
        out = np.zeros(9, np.uint32)
        check(lib().zkb_session_commit(self.h, C.c_int(po2), code.ctypes.data_as(C.c_void_p), _hp(out)))
        return out

    def control_ids(self):
        """(k, 9) array of every committed (po2, code root), ascending po2: the table verify_segment takes."""
        n = C.c_size_t(); check(lib().zkb_session_control_ids(self.h, C.byref(n), None))
        out = np.zeros((n.value, 9), np.uint32)
        check(lib().zkb_session_control_ids(self.h, C.byref(n), _hp(out)))
        return out[: n.value]

    def submit(self, po2, io, data, accum=None):
        """Queues one segment and returns its ticket.  accum=None: the circuit's witness program computes the accum group on the device.
        The arrays are kept alive until wait() or close()."""
        io = np.ascontiguousarray(io, dtype=np.uint32)
        arrs = [None if t is None else np.ascontiguousarray(t, dtype=np.uint32) for t in (data, accum)]
        ptrs = [C.c_void_p(None) if a is None else a.ctypes.data_as(C.c_void_p) for a in arrs]
        t = C.c_uint64()
        with self._lock:          # the ticket is recorded before another thread can wait for it
            check(lib().zkb_session_submit(self.h, C.c_int(po2), _hp(io), *ptrs, C.byref(t)))
            self._keep[t.value] = arrs
        return t.value

    def wait(self, ticket):
        """Blocks until the ticket's segment is proven; returns its seal, or raises the segment's own error.  Releases the ticket."""
        try:
            n = C.c_size_t(); check(lib().zkb_session_wait(self.h, C.c_uint64(ticket), None, C.byref(n)))
            s = np.zeros(n.value, np.uint32)
            check(lib().zkb_session_wait(self.h, C.c_uint64(ticket), _hp(s), C.byref(n)))
            return s
        finally:
            with self._lock:
                self._keep.pop(ticket, None)

    def close(self):
        """Fails the segments whose proof has not started, waits for the ones in progress, and frees the workers and programs."""
        if self.h:
            check(lib().zkb_session_free(self.h)); self.h = C.c_void_p()
            self._keep.clear()


class SegmentProver:
    def __init__(self, hal: B200Hal, circuit_blob):
        self.hal = hal
        self.blob = np.ascontiguousarray(circuit_blob, dtype=np.uint32)
        self.mix_size = int(self.blob[4])
        self.h = C.c_void_p()
        check(lib().zkb_prover_new(hal.ctx, _hp(self.blob), _sz(self.blob.size), C.byref(self.h)))

    def close(self):
        if self.h:
            check(lib().zkb_prover_free(self.h)); self.h = C.c_void_p()

    @staticmethod
    def _ptr(a, dev):
        return a if dev else a.ctypes.data_as(C.c_void_p)

    def use_program(self, program):
        """Attaches a Program (None detaches): code=None then proves from its commitment at the segment's po2."""
        if program is not None and not program.h:
            raise ValueError("the program is closed")
        check(lib().zkb_prover_set_program(self.h, program.h if program is not None else None))

    def begin(self, po2, io, code, data):
        io = np.ascontiguousarray(io, dtype=np.uint32)
        _, (c, d), dev = _trace_args(code, data)
        mix = np.zeros(max(self.mix_size, 1), np.uint32)
        check(lib().zkb_prover_segment_begin(self.h, C.c_int(po2), _hp(io), c, d, C.c_int(int(dev)), _hp(mix)))
        return mix[: self.mix_size]

    def finish(self, accum):
        a, ad = _trace_arg(accum)
        check(lib().zkb_prover_segment_finish(self.h, self._ptr(a, ad), C.c_int(int(ad))))
        return self.seal()

    def prove(self, po2, io, code, data, accum):
        io = np.ascontiguousarray(io, dtype=np.uint32)
        _, (c, d, a), dev = _trace_args(code, data, accum)
        check(lib().zkb_prove_segment(self.h, C.c_int(po2), _hp(io), c, d, a, C.c_int(int(dev))))
        return self.seal()

    def stage(self, po2, code, data, accum=None):
        """Starts the asynchronous upload of one segment's host traces (numpy arrays, ideally over pinned memory) into a
        staging slot; returns immediately.  The arrays must stay alive and unmodified until the matching prove_staged().
        accum=None: the accum group is computed on the device by the circuit's witness program (CircuitHal::accumulate) inside
        prove_staged and never uploaded.  code=None: the attached Program's commitment at po2 is used, and no code is uploaded."""
        arrs = [None if t is None else np.ascontiguousarray(t, dtype=np.uint32) for t in (code, data, accum)]
        check(lib().zkb_prover_stage_traces(self.h, C.c_int(po2), *[C.c_void_p(None) if a is None else a.ctypes.data_as(C.c_void_p) for a in arrs]))
        self._staged = getattr(self, "_staged", []) + [arrs]      # only a staged segment: a refused one must not shift the queue

    def stage_wait(self):
        check(lib().zkb_prover_stage_wait(self.h))

    def prove_staged(self, io):
        io = np.ascontiguousarray(io, dtype=np.uint32)
        check(lib().zkb_prove_staged(self.h, _hp(io)))
        self._staged.pop(0)
        return self.seal()

    def seal(self):
        n = C.c_size_t(); check(lib().zkb_prover_seal_words(self.h, C.byref(n)))
        s = np.zeros(n.value, np.uint32); check(lib().zkb_prover_seal_copy(self.h, _hp(s))); return s

    def roots(self):
        n = C.c_size_t(); check(lib().zkb_prover_root_count(self.h, C.byref(n)))
        r = np.zeros(n.value * 8, np.uint32); check(lib().zkb_prover_roots_copy(self.h, _hp(r))); return r.reshape(n.value, 8)


def control_id(po2, code_root):
    """One control-ID entry (po2, code root[8]) for verify_segment: the Merkle root of the code group identifies the program
    (risc0-zkp `check_code(po2, root)`); `code_root` is `roots()[0]` of a prover that committed the genuine code trace.
    `Program.commit(po2, code)` computes the same entry from the code trace alone, without proving a segment, and
    `Program.control_ids()` gives the whole table."""
    return np.concatenate([np.array([po2], np.uint32), np.ascontiguousarray(code_root, dtype=np.uint32).ravel()[:8]])


def verify_segment(circuit_blob, seal, control_ids):
    """Raises ZkbError unless `seal` verifies AND its code root is one of `control_ids` (array of 9-word entries, see
    control_id()).  Returns (po2, code_root)."""
    blob = np.ascontiguousarray(circuit_blob, dtype=np.uint32); seal = np.ascontiguousarray(seal, dtype=np.uint32)
    ids = np.ascontiguousarray(control_ids, dtype=np.uint32).ravel()
    if ids.size == 0 or ids.size % 9:
        raise ValueError("control_ids must hold 9-word entries (po2, code root[8])")
    out = np.zeros(9, np.uint32)
    check(lib().zkb_verify_segment(_hp(blob), _sz(blob.size), _hp(seal), _sz(seal.size), _hp(ids), _sz(ids.size // 9), _hp(out)))
    return int(out[0]), out[1:].copy()


def seal_code_root(circuit_blob, seal):
    """(po2, code root) a seal commits to, with every other check of verify_segment applied -- for building a control-ID table
    from a trusted seal; NOT a verification of the program."""
    blob = np.ascontiguousarray(circuit_blob, dtype=np.uint32); seal = np.ascontiguousarray(seal, dtype=np.uint32)
    out = np.zeros(9, np.uint32)
    check(lib().zkb_verify_segment(_hp(blob), _sz(blob.size), _hp(seal), _sz(seal.size), None, _sz(0), _hp(out)))
    return int(out[0]), out[1:].copy()
