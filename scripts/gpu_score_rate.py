"""Scoring given tokens: b200rwkv_infer_score against what a shim has to do without it.

Workload: a v6-3b-shaped model at V = 65536, max_batch 8, token_chunk_size 128; one request = 8 slots x 512 scored tokens
(one Choose request with 8 choices of 512 tokens, crates/ai00-core/src/run.rs:936-983).  Two paths, alternated in one run:
  (a) infer_score: SCORE entries, log-probabilities computed on the device, 8 x 512 f32 back to the host;
  (b) infer(OPTION_FULL) into pinned host memory, then the host normalisation of run.rs:731-747 (exp of the whole row, sum,
      p[target] / sum, ln) at each target.
Reports wall time per request (every call ends in a device synchronise), bytes copied device -> host (from shapes), the
agreement of the two paths, and, in a separate profiled pass (torch.profiler, CUDA activities), the device time of
score_rows_kernel against all kernels of an (a) request.  The card's name and power limit are read in the same run.
usage: gpu_score_rate.py [out_dir (default: a new temporary directory)] [reps]"""
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ai00_server_b200 import capi, runtime, synth  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else tempfile.mkdtemp(prefix="score_rate_")    # JSON result + profiler trace
REPS = int(sys.argv[2]) if len(sys.argv) > 2 else 5
NS, NT, CHUNK, PRESET = 8, 512, 128, "v6-3b"


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as ex:          # the measurement stands without it, but says so
        return {"error": str(ex)}


def main():
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures on the GPU only")
    os.makedirs(OUT, exist_ok=True)
    shp = synth.PRESETS[PRESET]
    assert shp.V == 65536, shp
    m = runtime.Model(synth.make_st(PRESET, 0), max_batch=NS, token_chunk_size=CHUNK)
    V = m.info["num_vocab"]
    rng = np.random.default_rng(0)
    toks = rng.integers(1, V, (NS, NT)).astype(np.uint32)
    flat = toks.reshape(-1)
    slots, ntok = np.arange(NS, dtype=np.int32), np.full(NS, NT, np.int32)
    zero = m.state.init()
    L = capi.lib()

    # pinned host buffer for path (b): every row of every token
    nrows = NS * NT
    p = C.c_void_p()
    capi.check(L.b200rwkv_host_alloc(nrows * V * 4, C.byref(p)))
    host = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=(nrows, V))
    logp = np.empty(nrows, np.float32)
    rows_out = np.zeros(NS, np.int32)

    def reset():
        for s in range(NS):
            m.state.load(zero, s)

    def path_a():
        opt = np.full(NS, capi.OPTION_SCORE, np.int32)
        t0 = time.perf_counter()
        capi.check(L.b200rwkv_infer_score(m._h, NS, capi.ptr(slots), capi.ptr(ntok), capi.ptr(flat), capi.ptr(opt), None, 0,
                                          capi.ptr(rows_out), capi.ptr(logp), logp.size), m._h)
        return time.perf_counter() - t0, logp.reshape(NS, NT)[:, 1:].copy()

    def path_b():
        opt = np.full(NS, capi.OPTION_FULL, np.int32)
        t0 = time.perf_counter()
        capi.check(L.b200rwkv_infer(m._h, NS, capi.ptr(slots), capi.ptr(ntok), capi.ptr(flat), capi.ptr(opt), p, host.size,
                                    capi.ptr(rows_out)), m._h)
        t1 = time.perf_counter()
        out = np.empty((NS, NT - 1), np.float32)
        for s in range(NS):                                   # run.rs:739-742, one entry's rows at a time
            r = host[s * NT: s * NT + NT - 1]
            e = np.exp(r)
            out[s] = np.log(e[np.arange(NT - 1), toks[s, 1:]] / e.sum(axis=1, dtype=np.float32))
        return time.perf_counter() - t0, out, t1 - t0

    reset(); path_a()                                         # warm-up: graphs of every step shape, buffers
    reset(); path_b()
    ta, tb, tb_dev = [], [], []
    for _ in range(REPS):                                     # alternated
        reset(); t, la = path_a(); ta.append(t)
        reset(); t, lb, td = path_b(); tb.append(t); tb_dev.append(td)
    finite = np.isfinite(lb)
    diff = float(np.abs(la[finite] - lb[finite]).max())

    # separate pass: device time of the score kernel within one (a) request
    from torch.profiler import ProfilerActivity, profile
    reset()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t_prof, _ = path_a()
    score_us, total_us, nscore, nkern = 0.0, 0.0, 0, 0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        dur = ev.time_range.elapsed_us()
        if "memcpy" in ev.name.lower() or "memset" in ev.name.lower():
            continue
        total_us += dur; nkern += 1
        if "score_rows_kernel" in ev.name:
            score_us += dur; nscore += 1
    prof.export_chrome_trace(os.path.join(OUT, "score_rate_trace.json"))

    res = {
        "card": card(),
        "model": PRESET, "num_vocab": V, "slots": NS, "tokens_per_slot": NT, "token_chunk_size": CHUNK, "reps": REPS,
        "a_infer_score_ms": {"median": 1e3 * float(np.median(ta)), "min": 1e3 * min(ta), "max": 1e3 * max(ta)},
        "b_full_rows_plus_host_ms": {"median": 1e3 * float(np.median(tb)), "min": 1e3 * min(tb), "max": 1e3 * max(tb)},
        "b_infer_call_alone_ms": {"median": 1e3 * float(np.median(tb_dev))},
        "d2h_bytes": {"a": NS * NT * 4, "b": nrows * V * 4},
        "max_abs_logp_diff_a_vs_b": diff,
        "profiled_pass": {"score_kernel_us": score_us, "score_launches": nscore, "all_kernels_us": total_us, "kernels": nkern,
                          "score_share_of_kernel_time": (score_us / total_us) if total_us else None,
                          "score_share_of_call_wall": (score_us * 1e-6 / t_prof) if t_prof else None,
                          "call_wall_ms_under_profiler": 1e3 * t_prof},
    }
    print(json.dumps(res, indent=1))
    print(f"written to {OUT}", file=sys.stderr)
    with open(os.path.join(OUT, "score_rate.json"), "w") as f:
        json.dump(res, f, indent=1)
    L.b200rwkv_host_free(p)
    m.close()


if __name__ == "__main__":
    main()
