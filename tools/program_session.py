"""One GPU, `--inflight` provers on the staged path (pinned host traces, device-side `accumulate`), K SYN-280 segments of 2^po2 cycles
that share one code trace and differ in their data trace and io words.  Two modes, run alternately with fresh provers each time:

    trace    the code trace is staged for every segment; each prover's own retained commitment is hit from its second segment on
    program  one shared zkb_program holds the code commitment; segments stage only their data trace (code=None)

Writes <out>/program_session.json (and prints it): segments/s per run, host->device bytes per segment (from shapes), device memory in
use after warm-up (cudaMemGetInfo, minus what was in use before the first prover was made), whether every seal of one mode equals the
seal of the same segment in the other, and the GPU's name and power limit read in the same run.

    python tools/program_session.py --out /tmp/program_session
"""
import argparse, hashlib, json, os, subprocess, sys, threading, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from zktls_b200 import circuit
from zktls_b200.hal import B200Hal
from zktls_b200.prover import Program, SegmentProver

ap = argparse.ArgumentParser()
ap.add_argument("--segments", type=int, default=24)
ap.add_argument("--po2", type=int, default=20)
ap.add_argument("--inflight", type=int, default=3)
ap.add_argument("--data-traces", type=int, default=6, help="distinct pinned data traces; segment k uses k mod this (and its own io words)")
ap.add_argument("--repeats", type=int, default=2, help="runs per mode, alternating trace / program")
ap.add_argument("--device", type=int, default=0)
ap.add_argument("--out", required=True)
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("program_session.py measures on a CUDA device; none is visible")

P = 2013265921
shape, po2, n = circuit.SYN280, a.po2, 1 << a.po2
blob = circuit.syn_circuit(**shape).blob()
torch.cuda.set_device(a.device)
dev = torch.device("cuda", a.device)
g = torch.Generator(device=dev); g.manual_seed(0xB2000003)


def pinned_trace(cols):
    t = torch.randint(0, P, (cols * n,), device=dev, dtype=torch.int64, generator=g).to(torch.int32).cpu().pin_memory()
    return t, t.numpy().view(np.uint32)


keep = []
code = pinned_trace(shape["code_cols"]); keep.append(code[0]); code = code[1]
datas = []
for _ in range(a.data_traces):
    t, v = pinned_trace(shape["data_cols"]); keep.append(t); datas.append(v)
ios = [np.random.default_rng(2000 + k).integers(0, P, size=shape["out_size"], dtype=np.uint32) for k in range(a.segments)]
torch.cuda.synchronize()


def mem_used():
    free, total = torch.cuda.mem_get_info(a.device)
    return total - free


def run(mode):
    """One run of `mode`: fresh ctxs and provers, one warm-up segment per prover, then the K timed segments (worker w takes w, w +
    inflight, ...; each stages its next segment before it proves the current one).  Returns (stats, sha256 of every seal)."""
    hals = [B200Hal(a.device) for _ in range(a.inflight)]
    provers = [SegmentProver(h, blob) for h in hals]
    prog, commit_s = None, None
    if mode == "program":
        prog = Program(hals[0], blob)
        t0 = time.time(); prog.commit(po2, code); commit_s = time.time() - t0
        for p in provers:
            p.use_program(prog)
        prog.close()                   # the provers hold it
    code_arg = code if mode == "trace" else None
    ths = [threading.Thread(target=lambda p: (p.stage(po2, code_arg, datas[0]), p.prove_staged(ios[0])), args=(p,)) for p in provers]
    for th in ths: th.start()
    for th in ths: th.join()
    torch.cuda.synchronize()
    mem = mem_used()
    seals, errs = {}, []

    def work(w):
        try:
            mine = list(range(w, a.segments, a.inflight))
            if mine:
                provers[w].stage(po2, code_arg, datas[mine[0] % a.data_traces])
            for i, k in enumerate(mine):
                if i + 1 < len(mine):
                    provers[w].stage(po2, code_arg, datas[mine[i + 1] % a.data_traces])
                seals[k] = hashlib.sha256(provers[w].prove_staged(ios[k]).tobytes()).hexdigest()
        except Exception as e:      # noqa: BLE001
            errs.append(e)

    t0 = time.time()
    ths = [threading.Thread(target=work, args=(w,)) for w in range(a.inflight)]
    for th in ths: th.start()
    for th in ths: th.join()
    torch.cuda.synchronize()
    wall = time.time() - t0
    if errs:
        raise errs[0]
    for p in provers: p.close()
    for h in hals: h.close()
    stats = {"mode": mode, "wall_s": wall, "segments_per_s": a.segments / wall, "device_mem_in_use_after_warmup_bytes": mem - base_mem}
    if commit_s is not None:
        stats["program_commit_s"] = commit_s
    return stats, [seals[k] for k in range(a.segments)]


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "-i", str(a.device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(a.device), "nvidia_smi_name_power_limit_max_sm_clock": q.stdout.strip() or q.stderr.strip()}


base_mem = mem_used()
runs, seals = [], {"trace": [], "program": []}
for r in range(a.repeats):
    for mode in ("trace", "program"):
        st, s = run(mode)
        runs.append(st); seals[mode].append(s)
ref = seals["trace"][0]
cols = {k: shape[k] for k in ("code_cols", "data_cols", "accum_cols")}
word_bytes = 4 * n
commit_bytes = 4 * (cols["code_cols"] * n * (1 + 1 + 4) + 2 * 4 * n * 8)          # trace copy, coefficients, LDE matrix, Merkle nodes
out = {
    "workload": f"{a.segments} SYN-280 segments of 2^{po2} cycles, one code trace, {a.data_traces} distinct data traces + per-segment io, "
                f"staged from pinned host memory, accum computed on the device, {a.inflight} provers in flight on one GPU",
    "gpu": gpu_identity(),
    "runs": runs,
    "segments_per_s": {m: [r["segments_per_s"] for r in runs if r["mode"] == m] for m in ("trace", "program")},
    "h2d_bytes_per_segment": {"trace": (cols["code_cols"] + cols["data_cols"]) * word_bytes, "program": cols["data_cols"] * word_bytes,
                              "difference": cols["code_cols"] * word_bytes},
    "device_mem_in_use_after_warmup_bytes": {m: [r["device_mem_in_use_after_warmup_bytes"] for r in runs if r["mode"] == m] for m in ("trace", "program")},
    "expected_mem_difference_bytes": {"retained_commitments": (a.inflight - 1) * commit_bytes,
                                      "staging_code_slots": a.inflight * 2 * cols["code_cols"] * word_bytes},
    "seals_equal_across_modes_and_runs": all(s == ref for m in seals for s in seals[m]),
}
os.makedirs(a.out, exist_ok=True)
with open(os.path.join(a.out, "program_session.json"), "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out), flush=True)
