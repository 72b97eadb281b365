"""K SYN-280 segments of 2^po2 cycles that share one code trace and differ in their data trace and io words, staged from pinned host
memory with the accum group computed on the device, `--inflight` provers per GPU.  Two arms, run alternately in the same command:

    session  one zkb_session (Session): the library's worker threads, queue and ordering rules; the caller only submits and waits
    threads  Python threads over staged SegmentProvers sharing one Program: tools/program_session.py's program mode (worker w takes
             w, w + inflight, ...; each stages its next segment before it proves the current one)

Each run makes fresh provers, commits the code trace (not timed), proves one warm-up segment per prover and then times the K segments.
`--devices all` adds session runs over every visible GPU in this one process.  Writes <out>/session_api.json (and prints it): segments/s
per run, whether every seal of every run equals the same segment's seal in the first run, and the GPUs' names and power limits read in
the same command.

    python tools/session_api.py --out /tmp/session_api [--devices all]
"""
import argparse, hashlib, json, os, subprocess, sys, threading, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from zktls_b200 import circuit
from zktls_b200.hal import B200Hal
from zktls_b200.prover import Program, SegmentProver, Session

ap = argparse.ArgumentParser()
ap.add_argument("--segments", type=int, default=64)
ap.add_argument("--po2", type=int, default=20)
ap.add_argument("--inflight", type=int, default=3)
ap.add_argument("--data-traces", type=int, default=6, help="distinct pinned data traces; segment k uses k mod this (and its own io words)")
ap.add_argument("--repeats", type=int, default=2, help="runs per arm, alternating session / threads")
ap.add_argument("--device", type=int, default=0)
ap.add_argument("--devices", choices=["one", "all"], default="one", help="all: also run the session over every visible GPU")
ap.add_argument("--out", required=True)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("session_api.py measures on a CUDA device; none is visible")

P = 2013265921
shape, po2, n = circuit.SYN280, a.po2, 1 << a.po2
blob = circuit.syn_circuit(**shape).blob()
dev = torch.device("cuda", a.device)
g = torch.Generator(device=dev); g.manual_seed(0xB2000004)


def pinned_trace(cols):
    t = torch.randint(0, P, (cols * n,), device=dev, dtype=torch.int64, generator=g).to(torch.int32).cpu().pin_memory()
    return t, t.numpy().view(np.uint32)


keep = []
code = pinned_trace(shape["code_cols"]); keep.append(code[0]); code = code[1]
datas = []
for _ in range(a.data_traces):
    t, v = pinned_trace(shape["data_cols"]); keep.append(t); datas.append(v)
ios = [np.random.default_rng(3000 + k).integers(0, P, size=shape["out_size"], dtype=np.uint32) for k in range(a.segments)]
torch.cuda.synchronize()


def digest(seal):
    return hashlib.sha256(seal.tobytes()).hexdigest()


def run_session(devices):
    s = Session(blob, devices=devices, inflight=a.inflight)
    s.commit(po2, code)
    warm = [s.submit(po2, ios[0], datas[0]) for _ in range(a.inflight * len(devices))]
    for t in warm:
        s.wait(t)
    t0 = time.time()
    tickets = [s.submit(po2, ios[k], datas[k % a.data_traces]) for k in range(a.segments)]
    seals = [digest(s.wait(t)) for t in tickets]
    wall = time.time() - t0
    s.close()
    return wall, seals


def run_threads():
    hals = [B200Hal(a.device) for _ in range(a.inflight)]
    provers = [SegmentProver(h, blob) for h in hals]
    prog = Program(hals[0], blob)
    prog.commit(po2, code)
    for p in provers:
        p.use_program(prog)
    prog.close()
    ths = [threading.Thread(target=lambda p: (p.stage(po2, None, datas[0]), p.prove_staged(ios[0])), args=(p,)) for p in provers]
    for th in ths: th.start()
    for th in ths: th.join()
    seals, errs = {}, []

    def work(w):
        try:
            mine = list(range(w, a.segments, a.inflight))
            if mine:
                provers[w].stage(po2, None, datas[mine[0] % a.data_traces])
            for i, k in enumerate(mine):
                if i + 1 < len(mine):
                    provers[w].stage(po2, None, datas[mine[i + 1] % a.data_traces])
                seals[k] = digest(provers[w].prove_staged(ios[k]))
        except Exception as e:      # noqa: BLE001
            errs.append(e)

    t0 = time.time()
    ths = [threading.Thread(target=work, args=(w,)) for w in range(a.inflight)]
    for th in ths: th.start()
    for th in ths: th.join()
    wall = time.time() - t0
    if errs:
        raise errs[0]
    for p in provers: p.close()
    for h in hals: h.close()
    return wall, [seals[k] for k in range(a.segments)]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(a.device), "device_count": torch.cuda.device_count(),
            "nvidia_smi_index_name_power_limit_max_sm_clock": (q.stdout.strip() or q.stderr.strip()).splitlines()}


runs, ref = [], None
same = True
arms = [("session", lambda: run_session([a.device])), ("threads", run_threads)]
if a.devices == "all":
    arms.append(("session_all_devices", lambda: run_session(list(range(torch.cuda.device_count())))))
for r in range(a.repeats):
    for arm, fn in arms:
        wall, seals = fn()
        ref = ref or seals
        same = same and seals == ref
        runs.append({"arm": arm, "wall_s": wall, "segments_per_s": a.segments / wall})
        print(json.dumps(runs[-1]), flush=True)
out = {
    "workload": f"{a.segments} SYN-280 segments of 2^{po2} cycles, one code trace, {a.data_traces} distinct data traces + per-segment io, "
                f"staged from pinned host memory, accum computed on the device, {a.inflight} provers in flight per GPU",
    "gpu": gpu_identity(),
    "runs": runs,
    "segments_per_s": {arm: [r["segments_per_s"] for r in runs if r["arm"] == arm] for arm, _ in arms},
    "seals_equal_across_arms_and_runs": same,
}
os.makedirs(a.out, exist_ok=True)
with open(os.path.join(a.out, "session_api.json"), "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out), flush=True)
