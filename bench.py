#!/usr/bin/env python
"""Benchmark of the B200 proving backend on BASELINE.json's metric: segments proven/sec (2^20 cycles).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py ... --dump-outputs DIR      also writes the last timed step's seal and roots as DIR/seal.npy, DIR/roots.npy

A "step" proves ONE synthetic 2^20-cycle segment of the SYN-280 circuit (BASELINE.json configs[1]; SURVEY.md 8d):
iNTT + zk-shift, x4 coset LDE, Poseidon2 row hashing + Merkle commit for the code/data/accum/check groups,
eval_check, DEEP evaluation + mixing + on-device division, three FRI rounds and the 50 queries -- the whole
`prove_segment` transcript, ending with the seal on the host.

  value  = segments/s with the three trace groups already resident in HBM when the timed region starts
  e2e    = the same through the reference-facing C-ABI call with HOST (pinned) trace buffers: the 1.17 GB host->device
           copy and the seal read-back are inside the timed region
  roofline = live CUDA-event timing of the dominant kernel (Poseidon2 hash_rows over the data group's 224 x 2^22 LDE
           matrix).  The kernel is bound by the INT32 multiplier ("fmaheavy") pipe, so `bound` is "int32": achieved =
           multiplier-pipe slots of its multiplications per second, peak = 64 lanes x SMs x the observed SM clock; the
           mandated HBM figures (algorithmic bytes / time against MEASURED_PEAKS.json) are the `hbm` sub-object, and
           `traffic` is the kernel's dram bytes from this round's ncu --set full capture (profiles/)
  cpu_baseline = the CPU oracle (C++ restatement of CpuHal, OpenMP) proving ONE full 2^20-cycle segment on this box's
           host cores (measured, ~35 s on 16 threads)
  --impl reference = the same oracle prover, every timed step a real 2^20-cycle segment, steps capped by --ref-budget-s
  --workload synheavy = a SECONDARY line: the same segment under the rv32im-shaped SYN-HEAVY constraint system

Segments are independent (continuations), so N GPUs prove N segments per step with no data-path collective
("scaling": "weak"); the only collectives are the timing barrier / max-reduce.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

ORIG_AFFINITY = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
METRIC = "segments proven/sec (2^20 cycles)"
UNIT = "segments/s"
PO2 = 20
P = 2013265921
# Multiplier-pipe ("fmaheavy") model of sm_100a, fitted to ncu (profiles/r1_v_hash_ncu_raw.txt: sm__pipe_fmaheavy_cycles_active
# 88.5 % = 7327 model slots / 8279 slot-times per permutation; tools/sass_hist.py reproduces the 7327 from the SASS): the pipe has
# 16 lanes per SM sub-partition (64 per SM); IMAD / IMAD.IADD occupy one slot, IMAD.WIDE / IMAD.HI two.
FMAHEAVY_LANES_PER_SM = 64
SLOTS_MONT, SLOTS_SHOUP = 5, 4                      # Montgomery product = WIDE + IMAD + HI; Shoup product = HI + 2 IMAD
SLOTS_PER_PERMUTATION = 852 * SLOTS_MONT + 504 * SLOTS_SHOUP      # 6276: the multiplications alone (SURVEY 8d: 1356 modmul)
SLOTS_PER_BUTTERFLY = SLOTS_SHOUP                   # Shoup twiddle product; the add / sub run on the ALU pipe


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons for one GPU.  Started before the warm-up so that nvidia-smi is already
    streaming when the timed region begins; stop(t0, t1) keeps only the samples whose host time falls inside [t0, t1]."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 or ts > t1 + 0.05:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1]); power.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power) if power else None}


_TRACES = {}


def cpu_baseline(sample_po2, threads=None):
    """The oracle prover (restated CpuHal) on a SYN-280 segment of 2^sample_po2 cycles, all host threads."""
    from zktls_b200 import circuit, synth
    from oracle import oracle as O
    # all host cores, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1 to its workers) and wherever the GPU arm
    # pinned this process
    if ORIG_AFFINITY:
        os.sched_setaffinity(0, ORIG_AFFINITY)
    O.lib().orc_set_num_threads(int(threads) if threads else (len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()))
    cores = O.lib().orc_num_threads()
    blob = circuit.syn_circuit(**circuit.SYN280).blob()
    if sample_po2 not in _TRACES:                      # generated once per size (1.17 GB at 2^20), outside every timed region
        _TRACES.clear()
        _TRACES[sample_po2] = synth.trace_a(circuit.SYN280, sample_po2, 0xB200)
    io, code, data, accum = _TRACES[sample_po2]
    t0 = time.time()
    pr = O.Prover(blob)
    pr.begin(sample_po2, io, code, data)
    pr.finish(accum)
    dt = time.time() - t0
    return dt, cores, pr


def dump_outputs(out_dir, arrays, rank=0):
    """--dump-outputs: every array as <out_dir>/<name>.npy in float64 (exact for u32 words), so that two builds can be compared
    output for output; ranks other than 0 add _rank<r> to the name."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + (f"_rank{rank}" if rank else "") + ".npy"), np.asarray(a, dtype=np.float64))


def reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path.  The Rust crates cannot be built here (no
    cargo, source un-vendored), so this is the oracle port (oracle/, C++/OpenMP restatement of CpuHal) on all host threads.
    Every timed step proves one REAL SYN-280 segment of 2^20 cycles (no extrapolation): `value` = segments / measured seconds.
    A full segment takes 20-40 s on 16 host cores, so --ref-budget-s S can cap the timed steps at a wall-clock budget (at least
    one step): `steps` is what was timed, `steps_requested` what the command line asked.  Without it every requested step runs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    po2 = args.po2
    warm = []
    for _ in range(min(args.warmup, 1)):
        warm.append(cpu_baseline(min(po2, 14))[0])             # untimed: loads the library, spins up the OpenMP team
    times, cores = [], 0
    t_start = time.time()
    while len(times) < args.steps:
        dt, cores, pr = cpu_baseline(po2)
        times.append(dt)
        if args.ref_budget_s is not None and (time.time() - t_start) + dt > args.ref_budget_s:      # the next step would not fit
            break
    ms = 1000.0 * sum(times) / len(times)
    value = 1000.0 / ms
    sample = (f"{len(times)} full SYN-280 segment(s) of 2^{po2} cycles proven by the oracle prover (C++/OpenMP restatement of CpuHal), "
              f"{', '.join(f'{t:.1f}' for t in times)} s each; measured, not extrapolated")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times), "steps_requested": args.steps,
            "warmup": min(args.warmup, 1), "warmup_requested": args.warmup, "warmup_what": "one 2^14-cycle segment (library load + OpenMP team), untimed",
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (BabyBear Montgomery)", "data": "synthetic",
            "config": workload_config(po2),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "steps_capped_by": None if len(times) >= args.steps else f"--ref-budget-s {args.ref_budget_s:.0f} (a full CPU segment proof takes {ms / 1000:.0f} s)"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"seal": pr.seal(), "roots": pr.roots()})
    print(json.dumps(line), flush=True)


def workload_config(po2=PO2):
    """identical in both arms (the driver compares the two `config` objects)"""
    name = "syn280-segment-po2-20" if po2 == PO2 else f"DEBUG po2={po2} (not the benchmark config)"
    return {"workload": name + ": one synthetic 2^20-cycle rv32im-shaped segment (BASELINE.json configs[1]): iNTT+zk-shift, x4 LDE, "
                        "Poseidon2 Merkle commit of code/data/accum/check, eval_check, DEEP + mix + divide, 3 FRI rounds, 50 queries; seal on host",
            "po2": po2, "columns": {"accum": 40, "code": 16, "data": 224, "check": 16}, "trace": "A (uniform field elements, seeded)",
            "l2": "inputs (1.17 GB trace, 4.7 GB LDE) exceed the 126 MB L2, no flush needed", "parallelism": "segment-parallel, one process per GPU, no data-path collective"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--po2", type=int, default=PO2, help="debug only: any value other than 20 is not the benchmark config")
    ap.add_argument("--cpu-sample-po2", type=int, default=0, help="cpu_baseline leg of the GPU arm: prove a 2^k-cycle segment instead of the full 2^20 one (debug)")
    ap.add_argument("--ref-budget-s", type=float, default=None, help="--impl reference: wall-clock budget that may cut the timed full-size CPU segment proofs short of --steps (at least one is run)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inflight", type=int, default=3, help="segments proven concurrently per GPU (one host thread + stream each)")
    ap.add_argument("--breakdown", action="store_true", help="per-operator timings to stderr")
    ap.add_argument("--workload", default="syn280", choices=["syn280", "synheavy"],
                    help="syn280 = the benchmark segment (BASELINE configs[1]); synheavy = the SAME segment shape with the rv32im-shaped SYN-HEAVY "
                         "constraint system (22 k constraints, 117 k steps): a SECONDARY, eval_check-weighted line, not the headline")
    ap.add_argument("--session-segments", type=int, default=64, help="segments of the synthetic TLS session timed for the 'e2e TLS prove s' metric (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the seal and roots of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        reference_arm(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from zktls_b200 import circuit
    from zktls_b200.hal import B200Hal
    from zktls_b200.prover import SegmentProver

    rank = int(os.environ.get("RANK", "0")); local_rank = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 backend has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from zktls_b200.shard import bind_rank_to_gpu_numa_node
    numa = bind_rank_to_gpu_numa_node(local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's version banner (NCCL_DEBUG=VERSION from the environment or from
        # /etc/nccl.conf) is printed to stdout when the first communicator is created, so (i) ask for WARN unless the user
        # wants more, and (ii) point fd 1 at stderr while the communicator comes up
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    po2 = args.po2
    n = 1 << po2
    shape = circuit.SYN280
    heavy = args.workload == "synheavy"
    blob = (circuit.syn_heavy_circuit() if heavy else circuit.syn_circuit(**shape)).blob()
    # `inflight` segments are proven concurrently per GPU, each by its own host thread + ctx (stream) + prover: one segment's
    # latency-bound stretches (Merkle tree tops, FRI rounds, Fiat-Shamir round trips) are filled by the other's kernels
    # (SURVEY.md 8e: ">= 2 segments in flight per GPU").  A ctx is used by one thread at a time, as the C-ABI requires.
    inflight = max(1, args.inflight)
    hals = [B200Hal(local_rank) for _ in range(inflight)]
    provers = [SegmentProver(h, blob) for h in hals]
    hal, prover = hals[0], provers[0]

    # synthetic trace, generated on the device (uniform field elements), seeded per rank
    g = torch.Generator(device=dev); g.manual_seed(0xB2000000 + rank)
    def rand_fp(count):
        return torch.randint(0, P, (count,), device=dev, dtype=torch.int64, generator=g).to(torch.int32)   # < 2^31: same bits as u32
    d_code, d_data, d_accum = rand_fp(shape["code_cols"] * n), rand_fp(shape["data_cols"] * n), rand_fp(shape["accum_cols"] * n)
    io = np.random.default_rng(rank).integers(0, P, size=shape["out_size"], dtype=np.uint32)
    from zktls_b200.hal import Buffer
    bufs = [[Buffer(h, t.data_ptr(), t.numel(), 1, owner=t) for t in (d_code, d_data, d_accum)] for h in hals]
    # pinned host copies for the end-to-end arm
    h_code, h_data, h_accum = (t.cpu().pin_memory() for t in (d_code, d_data, d_accum))
    h_np = [t.numpy().view(np.uint32) for t in (h_code, h_data, h_accum)]
    trace_bytes = sum(t.numel() * 4 for t in (d_code, d_data, d_accum))
    torch.cuda.synchronize()

    def run_workers(fn, k):
        """segments 0..k-1 over the `inflight` workers (worker w takes w, w + inflight, ...); returns the last seal a worker produced"""
        out, errs = [None] * inflight, []
        def work(w):
            try:
                out[w] = fn(w, len(range(w, k, inflight)))
            except Exception as e:      # noqa: BLE001
                errs.append(e)
                for ev in first_up:     # nobody may wait for a worker that died
                    ev.set()
        ths = [threading.Thread(target=work, args=(w,)) for w in range(1, inflight)]
        for th in ths: th.start()
        work(0)
        for th in ths: th.join()
        if errs:
            raise errs[0]
        return next((o for o in out if o is not None), None)

    def device_worker(w, k):
        s = None
        for _ in range(k):
            s = provers[w].prove(po2, io, *bufs[w])
        return s

    class SegmentQueue:
        """k segments handed to whichever worker asks next (a session's continuation segments are a queue, not a static split:
        the tail is then one segment, not one round of `inflight`)."""
        def __init__(self, k):
            self.left, self.lock = k, threading.Lock()
        def take(self):
            with self.lock:
                if self.left <= 0:
                    return False
                self.left -= 1
                return True

    def host_worker(w, queue, h_accum="host"):
        """Segments from HOST (pinned) buffers through the C-ABI, double-buffered: the 1.17 GB upload of the worker's next segment
        runs on the copy stream while the current one is proven.  Every segment's host->device copy and seal read-back happen
        inside this call.  A proof starts as soon as its 64 MB code group has landed (per-group upload events inside
        zkb_prove_staged); the data / accum uploads run behind the first commits.  Uploads of all provers of a device share ONE
        FIFO copy stream, so they are served in the order they are asked for, each at the full link rate: at start-up every worker
        stages its FIRST segment (in worker order) before anyone stages a second one -- otherwise worker 0's prefetch would sit in
        the queue in front of the other workers' first segments (measured: 169 ms of pipeline fill per rank instead of ~60)."""
        s = None
        have = queue.take()
        if w > 0:
            first_up[w - 1].wait()
        acc = h_np[2] if h_accum == "host" else None          # None: the accum group is computed on the device (CircuitHal::accumulate)
        if have:
            provers[w].stage(po2, h_np[0], h_np[1], acc)
        first_up[w].set()
        for ev in first_up:
            ev.wait()
        while have:
            ta = time.time()
            nxt = queue.take()
            if nxt:
                provers[w].stage(po2, h_np[0], h_np[1], acc)
            tb = time.time()
            s = provers[w].prove_staged(io)
            if timeline is not None:
                timeline.append((w, round((ta - timeline_t0[0]) * 1e3, 2), round((tb - timeline_t0[0]) * 1e3, 2), round((time.time() - timeline_t0[0]) * 1e3, 2)))
            have = nxt
        return s

    class SessionQueue:
        """bench-side adapter of shard.SharedSegmentQueue (one queue over all ranks; no data moves between ranks)"""
        def __init__(self, total, name):
            from zktls_b200.shard import SharedSegmentQueue
            self.q = SharedSegmentQueue(total, name)
        def take(self):
            return self.q.take() is not None

    def run_host(k, queue=None, h_accum="host"):
        q = queue or SegmentQueue(k)
        out = run_workers(lambda w, _k: host_worker(w, q, h_accum), inflight)       # one call per worker; the queue decides who proves what
        return out

    first_up = [threading.Event() for _ in range(inflight)]
    # ZKB_BENCH_TIMELINE=<prefix>: every rank writes <prefix>_rank<r>.json with (worker, take, prove start, prove end) in ms per segment of
    # the end-to-end arm and of the session (diagnostic; list.append is the only work added to the timed region)
    timeline, timeline_t0, timelines = ([] if os.environ.get("ZKB_BENCH_TIMELINE") else None), [0.0], {}

    # ---- device-resident arm -----------------------------------------------------------------------------------------
    sampler = ClockSampler(local_rank); sampler.start()
    seal = run_workers(device_worker, args.warmup * inflight)          # every worker warms up `warmup` times
    barrier()
    l0 = sum(h.kernel_launches() for h in hals)
    hal.timer_start(); t0 = time.time()           # event on worker 0's stream; every prove call returns with its seal on the host,
    seal = run_workers(device_worker, args.steps)  # so when the workers have joined all device work of the K steps is complete
    ms_dev = hal.timer_stop()
    barrier()
    t1 = time.time()
    wall = t1 - t0
    roots = prover.roots()          # worker 0 proves the first timed segment, and `seal` is its last one
    launches = sum(h.kernel_launches() for h in hals) - l0
    clocks = sampler.stop(t0, t1)
    t = torch.tensor([ms_dev], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = world * args.steps / (ms_total / 1000.0)

    # ---- end-to-end arm: host buffers through the C-ABI prove call ------------------------------------------------------
    first_up = [threading.Event() for _ in range(inflight)]
    seal_h = run_host(min(args.warmup, 2) * inflight)
    barrier()
    first_up = [threading.Event() for _ in range(inflight)]
    if timeline is not None:
        timeline.clear(); timeline_t0[0] = time.time()
    hal.timer_start()
    seal_h = run_host(args.steps)
    ms_e2e = hal.timer_stop()
    if timeline is not None:
        timelines["e2e"] = sorted(timeline, key=lambda r: r[1])
    barrier()
    t = torch.tensor([ms_e2e], device=dev, dtype=torch.float64)
    e2e_per_rank = [ms_e2e]
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        e2e_per_rank = [float(x.item()) for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps / (float(t.item()) / 1000.0)
    numa_all = [numa]
    if world > 1:
        numa_all = [None] * world
        dist.all_gather_object(numa_all, numa)
    assert np.array_equal(seal, seal_h), "device-resident and host-buffer paths disagree"

    # ---- the same with the accum group computed on the device (SURVEY 8f-3): code + data are uploaded, CircuitHal::accumulate (the
    # circuit blob's witness program) runs between the data commit and the accum commit as in the reference's prove_segment, the accum
    # trace (14 % of the bytes) never crosses the host link.  A different accum trace than Trace A's, so a SECONDARY number.
    e2e_dev_accum = None
    if not heavy and timeline is None:
        try:
            first_up = [threading.Event() for _ in range(inflight)]
            run_host(inflight, h_accum="device")
            barrier()
            first_up = [threading.Event() for _ in range(inflight)]
            hal.timer_start()
            run_host(args.steps, h_accum="device")
            ms_da = hal.timer_stop()
            barrier()
            t = torch.tensor([ms_da], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_dev_accum = {"value": world * args.steps / (float(t.item()) / 1000.0), "unit": UNIT, "h2d_bytes_per_step": int((d_code.numel() + d_data.numel()) * 4),
                             "what": "secondary: code + data groups from pinned host memory, accum group computed on the device by the circuit's witness program inside zkb_prove_staged"}
        except Exception as e:      # noqa: BLE001  (every rank raises or none: the circuit is the same everywhere)
            e2e_dev_accum = {"unavailable": str(e)[:200]}

    # ---- BASELINE metric "e2e TLS prove s": one TLS session = S continuation segments (SURVEY.md 8d config 4: S = 64 for a
    # 64 KB AES-128-GCM response), segment i -> rank i mod N, every segment uploaded from pinned host memory and its seal read back
    session = None
    if args.session_segments > 0:
        from zktls_b200.shard import segments_for_rank
        mine = len(segments_for_rank(args.session_segments, rank, world))
        first_up = [threading.Event() for _ in range(inflight)]
        sq, sharing = None, "static: segment i -> rank i mod N"
        if world > 1:
            try:
                sq = SessionQueue(args.session_segments, "session0"); sharing = "dynamic: one queue over all ranks (c10d store counter)"
            except Exception:      # noqa: BLE001  (no default store: keep the static split)
                sq = None
        barrier()
        hal.timer_start(); ts0 = time.time()
        if timeline is not None:
            timeline.clear(); timeline_t0[0] = time.time()
        run_host(mine, sq)
        ms_sess = hal.timer_stop()
        if timeline is not None:
            timelines["session"] = sorted(timeline, key=lambda r: r[1])
        barrier()
        t = torch.tensor([ms_sess], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        session = {"segments": args.session_segments, "seconds": float(t.item()) / 1000.0, "wall_s_rank0": time.time() - ts0, "sharing": sharing,
                   "what": "synthetic stand-in for one recorded TLS session: S independent SYN-280 2^20-cycle segments, segment-parallel over the ranks, host traces in / seals out"}

    if timeline is not None:
        with open(f"{os.environ['ZKB_BENCH_TIMELINE']}_rank{rank}.json", "w") as f:
            json.dump({"rank": rank, "columns": ["worker", "take_ms", "prove_start_ms", "prove_end_ms"], **timelines}, f)

    # ---- roofline of the dominant kernel (hash_rows over the data group's LDE matrix), live CUDA events -----------------
    roof = None
    if rank == 0:
        peaks, peak_kind = load_peaks()
        sm_mhz = clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0          # the clock observed during the timed region
        slot_peak = FMAHEAVY_LANES_PER_SM * hal.device_info()["sm_count"] * sm_mhz * 1e6      # multiplier-pipe issue slots per second
        rows, cols = 4 * n, shape["data_cols"]
        mat = hal.alloc_elem(rows * cols)           # contents irrelevant for timing; zero-initialised
        dig = hal.alloc_digest(rows)
        for _ in range(3):
            hal.hash_rows(dig, mat)
        reps = 5
        hal.timer_start()
        for _ in range(reps):
            hal.hash_rows(dig, mat)
        ms = hal.timer_stop() / reps
        alg_bytes = 4 * rows * cols + 32 * rows
        hbm_achieved = alg_bytes / (ms * 1e-3) / 1e9
        perms = rows * ((cols + 15) // 16)
        slots = perms * SLOTS_PER_PERMUTATION / (ms * 1e-3)
        traffic, traffic_src, ncu_pipes, stale = None, None, None, None
        import glob
        tpaths = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_hash_rows_traffic.json")))     # dram__bytes_read.sum + dram__bytes_write.sum of this kernel, one ncu --set full capture per round
        tpath = tpaths[-1] if tpaths else ""
        if po2 == PO2 and tpath:
            with open(tpath) as f:
                tj = json.load(f)
            traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
            ncu_pipes = {k: tj[k] for k in ("sm__pipe_fmaheavy_cycles_active_pct", "sm__pipe_alu_cycles_active_pct", "smsp__issue_active_pct") if k in tj}
            if tj.get("duration_ms"):               # the capture is of another build if its kernel time is far from today's
                stale = abs(tj["duration_ms"] - ms) / ms > 0.10
        roof = {"bound": "int32", "kernel": "k_hash_rows (Poseidon2, 224 cols x 2^22 rows)",
                "achieved": slots / 1e12, "peak": slot_peak / 1e12, "unit": "T multiplier-pipe slots/s", "frac": slots / slot_peak,
                "what": "Poseidon2 is bound by the INT32 multiplier (fmaheavy) pipe, not HBM (SURVEY.md 8d).  achieved = permutations/s x 6276 slots "
                        "(852 Montgomery products x 5 + 504 Shoup products x 4: the multiplications alone); peak = 64 lanes/SM x SMs x the SM clock "
                        "observed in the timed region.  Slot costs (IMAD 1, IMAD.WIDE / IMAD.HI 2) are fitted to ncu's sm__pipe_fmaheavy_cycles_active.",
                "sm_mhz": sm_mhz, "permutations_per_s": perms / (ms * 1e-3), "modmul_per_s": 1356 * perms / (ms * 1e-3), "ms_per_launch": ms,
                "traffic": traffic, "traffic_source": traffic_src, "traffic_stale": stale, "ncu_pipe_utilisation": ncu_pipes,
                "hbm": {"bound": "hbm", "achieved": hbm_achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_achieved / peaks["hbm_gbs"],
                        "algorithmic_bytes": alg_bytes, "peak_source": peak_kind}}
        del mat, dig
        # NTT roofline lines (BASELINE metric "NTT GB/s"): iNTT + zk-shift and x4 LDE over the data group's 224 columns of 2^20
        ntt_cols = 224
        buf = hal.alloc_elem(ntt_cols * n); big = hal.alloc_elem(ntt_cols * 4 * n)
        for _ in range(2):
            hal.batch_interpolate_ntt_zk_shift(buf, ntt_cols); hal.batch_expand_into_evaluate_ntt(big, buf, ntt_cols, 2)
        hal.timer_start()
        for _ in range(reps):
            hal.batch_interpolate_ntt_zk_shift(buf, ntt_cols)
        ms_i = hal.timer_stop() / reps
        hal.timer_start()
        for _ in range(reps):
            hal.batch_expand_into_evaluate_ntt(big, buf, ntt_cols, 2)
        ms_l = hal.timer_stop() / reps
        mm_i = ntt_cols * (n // 2) * po2 + ntt_cols * n            # butterflies + inter-pass twiddle / scale multiplications
        mm_l = ntt_cols * 2 * n * po2 + ntt_cols * 4 * n
        def ntt_line(ms_, alg, mm):
            return {"cols": ntt_cols, "po2": po2, "ms": ms_, "GBps": alg / (ms_ * 1e-3) / 1e9, "hbm_frac": alg / (ms_ * 1e-3) / 1e9 / peaks["hbm_gbs"],
                    "int32_frac": mm * SLOTS_PER_BUTTERFLY / (ms_ * 1e-3) / slot_peak}
        roof["ntt"] = {"intt_zk_shift": ntt_line(ms_i, 8 * n * ntt_cols, mm_i), "lde_x4": ntt_line(ms_l, 20 * n * ntt_cols, mm_l),
                       "note": "NTT GB/s on algorithmic bytes (8 n c / 20 n c); int32_frac = butterflies x 4 multiplier-pipe slots (one Shoup twiddle product) "
                               "against the same hardware slot peak: above n ~ 2^12 the transform is bound by that pipe, not by HBM"}
        del buf, big

    # ---- CPU baseline (rank 0, N = 1 only): ONE full 2^20 segment, measured -----------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not heavy:
        sample_po2 = args.cpu_sample_po2 or po2
        dt, cores, _ = cpu_baseline(sample_po2)
        scale = 1 << (po2 - sample_po2)
        cpu = {"value": 1.0 / (dt * scale), "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"oracle prover (C++/OpenMP restatement of CpuHal) on one SYN-280 segment of 2^{sample_po2} cycles: {dt:.2f} s"
                         + ("; the full benchmark segment, measured" if scale == 1 else f", x{scale} for 2^{po2} (DEBUG sample)")}

    ec = None
    if rank == 0 and heavy:      # eval_check alone over the 2^22-point domain, CUDA events
        dom = 4 * n
        bufs_ec = [hal.alloc_elem(shape[k] * dom) for k in ("accum_cols", "code_cols", "data_cols")]
        chk = hal.alloc_elem(4 * dom)
        gl_m, gl_o, pm = np.arange(1, 1 + shape["mix_size"], dtype=np.uint32), np.arange(1, 1 + shape["out_size"], dtype=np.uint32), np.arange(3, 7, dtype=np.uint32)
        for _ in range(2):
            hal.eval_check(chk, blob, *bufs_ec, gl_m, gl_o, pm, po2)
        hal.timer_start()
        for _ in range(3):
            hal.eval_check(chk, blob, *bufs_ec, gl_m, gl_o, pm, po2)
        ms_ec = hal.timer_stop() / 3
        n_eqz = int((blob[16 + 3 * int(blob[6]):].reshape(-1, 4)[:, 0] == circuit.OP_AND_EQZ).sum())
        ec = {"kernel": "zkb_ec (compact form: all tapped columns resident per 128-point tile, one loop body per expression shape, terms as operand records)", "ms": ms_ec, "constraints": n_eqz, "steps": int(blob[7]),
              "domain_points": dom, "constraint_evaluations_per_s": n_eqz * dom / (ms_ec * 1e-3),
              "multiplier_slots_per_point": n_eqz * (4 * 2 + 5), "note": "per constraint: 4 IMAD.WIDE accumulations (8 slots) + ~1 Montgomery product (5 slots) on the multiplier pipe"}
        del bufs_ec, chk

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (BabyBear Montgomery)", "data": "synthetic",
                "config": workload_config(po2), "segments_in_flight_per_gpu": inflight, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": trace_bytes, "d2h_bytes_per_step": int(seal.size * 4),
                        "pipeline": "zkb_prover_stage_traces + zkb_prove_staged: pinned host traces, upload of segment k+1 overlaps the proof of segment k",
                        "per_rank_ms_per_step": [round(x / args.steps, 3) for x in e2e_per_rank],
                        "host_numa_binding_per_rank": numa_all, "device_accumulate": e2e_dev_accum},
                "gpu_launches": int(launches), "tls_session": session,
                "config5_estimate": {"what": "BASELINE configs[4] (64 sessions -> succinct receipts), SEGMENT STAGE ONLY, extrapolated from the measured end-to-end rate "
                                             "(SURVEY.md 8d: 64 x 40 SYN-280 segments; lift / join need the recursion circuit, which is not built)",
                                     "segments": 2560, "estimated_seconds": 2560.0 / e2e_value, "sessions_per_hour": e2e_value * 3600.0 / 40.0}, "roofline": roof, "cpu_baseline": cpu, "wall_s": wall, "seal_words": int(seal.size)}
        if heavy:
            line["config"]["workload"] = "SECONDARY synheavy280-segment-po2-20: the benchmark segment's shape (280 columns, 2^20 cycles, Trace A) under the SYN-HEAVY " \
                                         "constraint system (rv32im-shaped: 22 k constraints / 117 k PolyExtSteps, AndCond depth 4, taps back 0..4, 5 combos) -- eval_check-weighted companion of the headline"
            line["eval_check"] = ec
        print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"seal": seal, "roots": roots}, rank)
    for pr in provers:
        pr.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
