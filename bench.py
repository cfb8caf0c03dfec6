#!/usr/bin/env python
"""bench.py — decode tokens/s of the RWKV hot path on B200 (BASELINE.json metric).

A "step" is one decode step of the whole model for every slot of the batch (one token per
slot): the per-layer WKV recurrence + token shift + GroupNorm, all projections and the head.
Workload at N=1: configs[2] of BASELINE.json, RWKV-6-World-7B shape, fp16 weights, batch 16,
slots primed with a 128-token synthetic prompt (random-init weights of that architecture,
there are no checkpoints offline).

  value     tokens/s with token ids staged in HBM and logits left in HBM (CUDA events around
            `steps` graph replays, b200rwkv_bench_decode)
  e2e       the same metric through the reference-facing call (Runtime.infer ->
            b200rwkv_infer): token ids copied H2D and all logits rows copied D2H every step
  roofline  projection-GEMM kernel: algorithmic weight bytes per step / summed GEMM launch
            durations (CUDA events on the engine's stream, un-graphed profiling pass)
  cpu_baseline / --impl reference
            the C/OpenMP oracle (oracle/rwkv_ref.c) on the host cores, same weights/tokens
            (the reference's own web-rwkv+lavapipe path cannot be built here: no Rust, no Vulkan)

--dump-outputs DIR writes what the timed path computed in its last step as DIR/<name>.npy (f32), so two builds can be
compared output for output on identical seeded inputs: decode -> `logits` [batch, vocab] and `state` [batch, L, N+2, C],
prefill -> `state` of every sequence.  An array over its share of DUMP_BYTES is replaced by a fixed seeded sample of its
flattened elements.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json: the headline metric is quoted on configs[2] (7B, batch 16); configs[1] and [3] are the secondary lines
MODEL_NAMES = {"v6-7b": "RWKV-6-World-7B", "v6-3b": "RWKV-6-World-3B", "v6-1b6": "RWKV-6-World-1.6B", "v7-2b9": "RWKV-7-World-2.9B"}
PRESET = os.environ.get("B200RWKV_BENCH_PRESET", "v6-7b")
BATCH = int(os.environ.get("B200RWKV_BENCH_BATCH", "16"))
PROMPT = int(os.environ.get("B200RWKV_BENCH_PROMPT", "128"))


def metric_name(preset: str, batch: int) -> str:
    return f"decode tokens/s {MODEL_NAMES.get(preset, preset)} fp16 batch={batch}"


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_tokens(n_steps: int, batch: int, vocab: int):
    rng = np.random.default_rng(1234)                      # SURVEY.md §8(d)
    return rng.integers(1, min(vocab, 65530), size=(batch, n_steps), dtype=np.int64)


DUMP_BYTES = 48 << 20          # all of --dump-outputs together, .npy headers aside


def dump_outputs(path: str, arrays: dict) -> None:
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, np.float32)
        if a.nbytes > share:
            a = a.reshape(-1)[np.unique(np.random.default_rng(0).integers(0, a.size, share // a.itemsize))]
        np.save(os.path.join(path, f"{name}.npy"), a)


def last_step_outputs(model, slots) -> dict:
    """Logits row and state of every slot after the model's most recent step, through device snapshots (untimed)."""
    logits = np.empty((len(slots), model.info["num_vocab"]), np.float32)
    state = None
    for i, s in enumerate(slots):
        snap = model.state.read(s)
        st, logits[i] = model.state.snapshot_back(snap, with_logits=True)
        snap.free()
        if state is None:
            state = np.empty((len(slots),) + st.shape, np.float32)
        state[i] = st
    return {"logits": logits, "state": state}


def host_threads() -> int:
    """Threads the CPU arms use: the physical cores inside this process' affinity mask and cgroup CPU quota (measured on
    the GPU box: 128 OpenMP threads on its 64 cores run the same step 18x slower than 64).  Never taken from
    OMP_NUM_THREADS: torchrun exports OMP_NUM_THREADS=1 to its workers."""
    if os.environ.get("B200RWKV_CPU_THREADS"):
        return max(1, int(os.environ["B200RWKV_CPU_THREADS"]))
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        # SMT present -> one thread per core = half of the usable logical CPUs.  (The absolute core count virtualised hosts
        # report is not trusted: the GPU box says 16 cores / 128 logical CPUs, where 64 threads measured fastest.)
        import psutil
        phys, logical = psutil.cpu_count(logical=False), psutil.cpu_count(logical=True)
        if phys and logical and logical > phys:
            n = max(1, n // 2)
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def cpu_arm(weights, batch: int, steps: int, warmup: int, toks_bt: np.ndarray, budget_s: float = 1e9):
    """Times the C/OpenMP oracle on the host cores: up to `steps` decode steps of the same workload (stops early once
    `budget_s` seconds of timed work are spent).  Returns tokens/s, ms/step, threads, steps timed."""
    os.environ.setdefault("OMP_PROC_BIND", "false")
    from ai00_server_b200 import build
    from oracle import ref_c
    if not os.path.exists(ref_c.LIB_PATH):
        build.build_oracle()
    rc = ref_c.RefC(weights, "f16")
    rc.set_num_threads(host_threads())             # explicit: the inherited OMP_NUM_THREADS is not ours (torchrun sets 1)
    st = rc.state_init(batch)
    for i in range(warmup):
        rc.decode_step(toks_bt[:, i % toks_bt.shape[1]], st)
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        rc.decode_step(toks_bt[:, (warmup + i) % toks_bt.shape[1]], st)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return batch * done / dt, dt / done * 1e3, rc.num_threads(), done


def prefill_main(args):
    """cfg 5 (BASELINE.json configs[4]): `seqs` prompts of `seq_len` tokens through the embeddings route's path -- prefill with
    no logits, then State::back of every slot (run.rs:984-989 returns the backed state as the embedding).  A "step" is one
    pass over all seqs x seq_len tokens."""
    import torch
    from ai00_server_b200 import capi, runtime, synth
    from oracle import rwkv_numpy as O
    preset = args.preset if args.preset != "v6-7b" or "--preset" in sys.argv else "v6-3b"
    shape = synth.PRESETS[preset]
    B, Tn = args.seqs, args.seq_len
    steps, warm = args.steps, max(3, args.warmup if args.warmup < 8 else 3)
    metric = f"prefill tokens/s {MODEL_NAMES.get(preset, preset)} fp16 {B}x{Tn}-token inputs (embeddings route)"
    st = synth.make_st(shape, 0)
    PASS = 128                                              # tokens per weight pass (the engine's largest step)
    model = runtime.Model(st, max_batch=B, token_chunk_size=PASS, device=0)
    slots = list(range(B))
    rng = np.random.default_rng(1234)
    toks = rng.integers(1, min(shape.V, 65530), size=(B, Tn), dtype=np.int64)
    model.state.load(model.state.init(), 0)
    zero_snap = model.state.read(0)

    def reset():
        for s_ in slots:
            model.state.write(zero_snap, s_)

    for _ in range(warm):                                   # untimed: short passes through the same kernels
        reset()
        model.infer_raw(slots, [16] * B, toks[:, :16].reshape(-1).tolist(), [capi.OPTION_NONE] * B)
    flat = toks.reshape(-1).tolist()
    sampler = ClockSampler(0)
    sampler.start()
    t_dev, t_e2e = [], []
    state_buf = np.empty((B,) + model.state.init().shape, np.float32)
    launches0 = model.launch_count()
    for _ in range(steps):
        reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.infer_raw(slots, [Tn] * B, flat, [capi.OPTION_NONE] * B)         # returns after the last step completed
        t1 = time.perf_counter()
        for s_ in slots:
            state_buf[s_] = model.state.back(s_)
        t2 = time.perf_counter()
        t_dev.append(t1 - t0); t_e2e.append(t2 - t0)
    clocks = sampler.stop()
    launches = model.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"state": state_buf})
    ntok = B * Tn
    dt, de = float(np.mean(t_dev)), float(np.mean(t_e2e))
    checksum = [float(state_buf.astype(np.float64).sum()), float(np.abs(state_buf).astype(np.float64).sum())]
    # parity spot check + CPU baseline (outside the timed region): the first sequences' first tokens against the C oracle
    w = O.parse_st(st)
    from oracle import ref_c
    if not os.path.exists(ref_c.LIB_PATH):
        from ai00_server_b200 import build
        build.build_oracle()
    rc = ref_c.RefC(w, "f16")
    rc.set_num_threads(host_threads())
    rc32 = ref_c.RefC(w, "f32")
    nb, nt = min(B, 4), min(Tn, 24)
    cst, cst32 = rc.state_init(nb), rc32.state_init(nb)
    c0 = time.perf_counter()
    for j in range(nt):
        rc.decode_step(toks[:nb, j], cst)
    cdt = time.perf_counter() - c0
    for j in range(nt):
        rc32.decode_step(toks[:nb, j], cst32)
    reset()
    model.infer_raw(slots[:nb], [nt] * nb, toks[:nb, :nt].reshape(-1).tolist(), [capi.OPTION_NONE] * nb)
    got = [model.state.back(i) for i in range(nb)]
    errs = [float(np.abs(got[i] - cst[i]).max() / np.abs(cst[i]).max()) for i in range(nb)]
    errs32 = [float(np.abs(got[i] - cst32[i]).max() / np.abs(cst32[i]).max()) for i in range(nb)]
    floor = [float(np.abs(cst[i] - cst32[i]).max() / np.abs(cst32[i]).max()) for i in range(nb)]
    # the same tokens one at a time through the decode-shaped kernels: differs from the one-call prefill only in summation order
    reset()
    for j in range(nt):
        model.infer_raw(slots[:nb], [1] * nb, toks[:nb, j].tolist(), [capi.OPTION_NONE] * nb)
    dec_vs_pre = [float(np.abs(model.state.back(i) - got[i]).max() / np.abs(got[i]).max()) for i in range(nb)]
    # where a pass goes: in-situ windows of one 128-slot x 1-token step (the shape every prefill pass has here)
    breakdown = None
    try:
        wins, step_us = model.profile_insitu(slots[:PASS], toks[:PASS, 0].astype(np.uint32), reps=3)
        agg = {}
        for wdw in wins:
            ty = wdw["type"]
            name = "gemm" if ty >= 1000000 else {0: "ln_mix", 2: "wkv", 6: "front_half"}.get(ty, "ln_mix")
            a = agg.setdefault(name, [0.0, 0])
            a[0] += wdw["end_us"] - wdw["start_us"]; a[1] += 1
        breakdown = {"step_us": step_us, "class_us": {k: v[0] for k, v in agg.items()}, "class_launches": {k: v[1] for k, v in agg.items()}}
    except Exception as ex:                                  # profiling is evidence, not the measurement
        breakdown = {"error": str(ex)}
    peaks, peak_src = read_peaks()
    n_pass = -(-ntok // PASS)
    wbytes = 2 * (synth.num_params(shape) - shape.V * shape.C)              # every pass streams all weights but the embedding
    pass_bytes = wbytes + PASS * 2 * shape.L * (shape.H * 64 * 64 + 2 * shape.C) * 4
    flops = 2.0 * (synth.num_params(shape) - 2 * shape.V * shape.C) * ntok  # no head: the route needs no logits
    line = {"metric": metric, "value": ntok / dt, "unit": "tokens/s", "n_gpus": 1, "steps": steps, "warmup": warm,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"{preset} prefill, {B} sequences x {Tn} tokens, no logits, final state of every sequence returned",
                       "preset": preset, "seqs": B, "seq_len": Tn, "tokens_per_pass": PASS,
                       "l2": f"inputs larger than L2 (5.9 GB of weights streamed per {PASS}-token pass), no flush"},
            "clocks": clocks,
            "e2e": {"value": ntok / de, "unit": "tokens/s", "ms_per_step": de * 1e3, "h2d_bytes_per_step": int(ntok * 4 + n_pass * 1800),
                    "d2h_bytes_per_step": int(state_buf.nbytes),
                    "api": "b200rwkv_infer (host token ids, OPTION_NONE) + b200rwkv_state_back of every slot (the embedding, run.rs:984-989)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": f"gemm_kernel<8> ({PASS}-token passes: every pass streams all projection weights once)",
                         "achieved": n_pass * pass_bytes / dt / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": n_pass * pass_bytes / dt / 1e9 / peaks["hbm_gbs"], "traffic": None,
                         "peak_source": f"MEASURED_PEAKS.json ({peak_src})", "passes": n_pass, "bytes_per_pass": int(pass_bytes),
                         "tensor_tflops_achieved": flops / dt / 1e12, "tensor_tflops_peak_sustained": peaks.get("bf16_tflops_sustained"),
                         "note": f"the route turns tensor-bound at >= 280 FLOP/B = ~300 tokens per weight pass; at {PASS} tokens per pass "
                                 "(shared memory: 32 KB weights + 32 KB tokens per stage, TMEM: 256 of 512 columns) it is still bound by "
                                 "streaming the weights, which is what `achieved` measures"},
            "cpu_baseline": {"value": nb * nt / cdt, "unit": "tokens/s", "cores": rc.num_threads(), "kind": "port",
                             "sample": f"first {nt} tokens of the first {nb} sequences, C/OpenMP oracle (token by token)"},
            "pass_breakdown": breakdown,
            "state_checksum": {"sum": checksum[0], "abs_sum": checksum[1]},
            "parity_check": {"what": f"final state of the first {nb} sequences after {nt} tokens (one prefill call), max |d| / max |state|",
                             "vs_oracle_f16_contract": max(errs), "vs_oracle_f32_contract": max(errs32),
                             "oracle_f16_vs_f32_contract": max(floor), "prefill_call_vs_token_by_token_decode": max(dec_vs_pre)}}
    print(json.dumps(line))
    zero_snap.free()
    model.close()


def main():
    global PRESET, BATCH
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 128 decode steps, 4 prefill passes)")
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-steps", type=int, default=int(os.environ.get("B200RWKV_BENCH_CPU_STEPS", "6")))
    ap.add_argument("--preset", default=PRESET, help="model shape: v6-7b (headline), v6-3b, v7-2b9, v6-1b6 (BASELINE.json configs)")
    ap.add_argument("--batch", type=int, default=BATCH, help="concurrent slots, one token per slot per step")
    ap.add_argument("--exact", action="store_true", help="precision 1: f32-exact activations (split hi+lo operands)")
    ap.add_argument("--mode", default="decode", choices=["decode", "prefill"],
                    help="prefill = BASELINE.json configs[4]: the embeddings route's workload (prompts in, final states out)")
    ap.add_argument("--quant", default="none", choices=["none", "int8", "nf4"],
                    help="weight-only quantised projection matrices (the reference's quant_type); not the headline configuration")
    ap.add_argument("--quant-layers", type=int, default=-1, help="the reference's `quant`: first N layers (default: all)")
    ap.add_argument("--seqs", type=int, default=256)
    ap.add_argument("--seq-len", type=int, default=512)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (1-GPU B200 arm)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 4 if args.mode == "prefill" else 128
    assert args.steps >= 1, "--steps must be at least 1"
    args.warmup = max(args.warmup, 3)
    PRESET, BATCH = args.preset, args.batch
    METRIC = metric_name(PRESET, BATCH)
    if args.quant != "none":
        METRIC = METRIC.replace("fp16", {"int8": "Int8", "nf4": "NF4"}[args.quant] + " projections (fp16 elsewhere)")
        assert args.mode == "decode" and not args.exact and args.impl == "b200" and args.gpus == 1, "--quant: 1-GPU decode arm only"
    if args.mode == "prefill":
        return prefill_main(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert not args.dump_outputs or (args.impl == "b200" and world == 1), "--dump-outputs: 1-GPU B200 arm only"

    from ai00_server_b200 import synth
    from oracle import rwkv_numpy as O          # only for parse_st of the cpu arm (checker side)
    shape = synth.PRESETS[PRESET]
    config = {"workload": f"{PRESET} decode, batch {BATCH} slots x 1 token/step, {PROMPT}-token synthetic prompt per slot",
              "preset": PRESET, "batch": BATCH, "prompt_tokens": PROMPT, "parallelism": f"tp{world}",
              "activations": "f32-exact (split f16 hi+lo operands)" if args.exact else "f16 operands",
              "l2": "inputs larger than L2 (14.7 GB of weights streamed per step vs 126 MB L2), no flush"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        st = synth.make_st(shape, 0)
        w = O.parse_st(st)
        warm = max(1, min(args.warmup, 2))
        toks = make_tokens(args.steps + warm, BATCH, shape.V)
        tps, ms, threads, steps = cpu_arm(w, BATCH, args.steps, warm, toks, budget_s=150.0)
        line = {"impl": "reference", "metric": METRIC, "value": tps, "unit": "tokens/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": threads, "kind": "port",
                                 "sample": f"{steps} decode steps of the full workload (requested {args.steps}; bounded to ~150 s), "
                                           "C/OpenMP oracle on the physical host cores; reference web-rwkv/lavapipe path unbuildable here"},
                "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch                                  # plumbing only: device selection + distributed barrier
    from ai00_server_b200 import runtime
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank if world > 1 else 0

    t_build = time.perf_counter()
    st = synth.make_st(shape, 0)
    qlayers = shape.L if args.quant_layers < 0 else min(args.quant_layers, shape.L)
    if args.quant != "none":
        model = runtime.Model(st, max_batch=BATCH, token_chunk_size=64, device=dev, quant=qlayers, quant_type=args.quant)
        config["weights"] = f"first {qlayers} of {shape.L} layers: eight projection matrices in {args.quant} (quantised at load on the GPU)"
    else:
        model = runtime.Model(st, max_batch=BATCH, token_chunk_size=64, device=dev, rank=rank, world=world, exact=args.exact)
    if world > 1:
        from ai00_server_b200 import tp
        tp.connect(model)
    build_s = time.perf_counter() - t_build

    n_steps = args.warmup + args.steps
    toks = make_tokens(PROMPT + 2 * n_steps + 8, BATCH, shape.V)
    slots = list(range(BATCH))
    zero = model.state.init()
    for s in slots:
        model.state.load(zero, s)
    # prime every slot with its prompt (prefill through the same path, untimed)
    model.infer_raw(slots, [PROMPT] * BATCH, toks[:, :PROMPT].reshape(-1).tolist(), [2] * BATCH)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: resident inputs, graph replays, CUDA events ----
    dec = np.ascontiguousarray(toks[:, PROMPT:PROMPT + n_steps].T).astype(np.uint32)       # [steps, B]
    sampler = ClockSampler(dev)
    barrier()
    sampler.start()
    ms, launches = model.bench_decode(slots, dec, args.warmup, args.steps)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step_outputs(model, slots))
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = BATCH * args.steps / (ms * 1e-3)

    # ---- e2e: host tokens in, host logits out, every step, through Runtime.infer ----
    out = np.empty((BATCH, shape.V), np.float32)       # rank 0 receives the gathered full-vocabulary logits
    try:
        tt = torch.from_numpy(out)
        torch.cuda.cudart().cudaHostRegister(tt.data_ptr(), out.nbytes, 0)     # pinned host memory
    except Exception:
        pass
    e2e_steps = args.steps
    dec2 = toks[:, PROMPT + n_steps:PROMPT + n_steps + args.warmup + e2e_steps]
    for i in range(args.warmup):
        model.infer_raw(slots, [1] * BATCH, dec2[:, i].tolist(), [0] * BATCH, out=out)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        model.infer_raw(slots, [1] * BATCH, dec2[:, args.warmup + i].tolist(), [0] * BATCH, out=out)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": BATCH * e2e_steps / e2e_s, "unit": "tokens/s", "ms_per_step": e2e_s / e2e_steps * 1e3,
           "h2d_bytes_per_step": int((8 + 6 * 128 + 3 * BATCH) * 4), "d2h_bytes_per_step": int(out.nbytes),
           "api": "runtime.Model.infer_raw -> b200rwkv_infer (host token ids in, host f32 logits out, wall clock)"}

    # ---- e2e with the GPU sampling front half: logits stay in HBM, <= 128 (id, prob) pairs per slot come back ----
    ids = probs = None
    for i in range(args.warmup):
        model.infer_raw(slots, [1] * BATCH, dec2[:, i].tolist(), [0] * BATCH, keep_on_device=True)
        if rank == 0:
            ids, probs = model.sample_topk(slots, top_k=128)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        model.infer_raw(slots, [1] * BATCH, dec2[:, args.warmup + i].tolist(), [0] * BATCH, keep_on_device=True)
        if rank == 0:
            ids, probs = model.sample_topk(slots, top_k=128)
    barrier()
    e2s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2s], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2s = float(t.item())
    e2e["sampled"] = {"value": BATCH * e2e_steps / e2s, "unit": "tokens/s", "ms_per_step": e2s / e2e_steps * 1e3,
                      "d2h_bytes_per_step": int(BATCH * 128 * 8),
                      "api": "b200rwkv_infer(logits_out = NULL) + b200rwkv_sample_topk(top_k = 128): the reference's nucleus default"}

    # ---- roofline of the dominant kernel (projection GEMM); SPMD under tensor parallelism ----
    # In-situ windows of a graph-replayed step (globaltimer stamps written by the kernels: [wait released, last CTA exit]);
    # consecutive windows cannot overlap, so the class sums are <= the step.  The un-graphed CUDA-event pass is kept beside
    # it (`events_ungraphed`): it over-counts because programmatic dependent launch is off there.
    peaks, peak_src = read_peaks()
    step_ms_dist = np.sort(np.asarray(model.step_ms, np.float64))
    windows, insitu_step_us = model.profile_insitu(slots, dec[0], reps=5)
    prof_ms = np.zeros(4)
    prof_n = np.zeros(4, dtype=np.int64)
    wbytes = 0
    reps = 3
    for i in range(reps + 1):
        m4, n4, wbytes = model.profile_step(slots, dec[i % dec.shape[0]])
        if i == 0:
            continue                       # first un-graphed pass is cold
        prof_ms += np.array(m4)
        prof_n = np.array(n4)
    prof_ms /= reps
    if rank != 0:
        barrier()
        model.close()
        return
    cls = {"gemm": [0.0, 0, 0], "wkv": [0.0, 0, 0], "ln_mix": [0.0, 0, 0], "front_half": [0.0, 0, 0]}
    per_label = {}
    for wdw in windows:
        ty = wdw["type"]
        name = "gemm" if ty >= 1000000 else {0: "ln_mix", 2: "wkv", 6: "front_half"}.get(ty, "ln_mix")
        d = wdw["end_us"] - wdw["start_us"]
        cls[name][0] += d; cls[name][1] += 1; cls[name][2] += wdw["bytes"]
        lab = f"gemm_{ty - 1000000}MiB" if ty >= 1000000 else name
        a = per_label.setdefault(lab, [0.0, 0, 0])
        a[0] += d; a[1] += 1; a[2] += wdw["bytes"]
    gemm_us, gemm_n, gemm_bytes = cls["gemm"]
    gemm_gbs = gemm_bytes / (gemm_us * 1e-6) / 1e9 if gemm_us > 0 else 0.0
    alg_bytes = synth.algorithmic_bytes_per_step(shape, BATCH) / world
    if args.quant != "none":
        C_, F_ = shape.C, shape.F
        mats = ([(C_, C_)] * (5 if shape.version != 7 else 4)) + [(F_, C_), (C_, F_)] + ([(C_, C_)] if shape.version != 7 else [])
        per = (lambda n, k: n * k + n * k // 128 * 4) if args.quant == "int8" else (lambda n, k: n * k // 2 + n * k // 64 * 2)
        alg_bytes += qlayers * sum(per(n, k) - 2 * n * k for n, k in mats)
    traffic = None       # DRAM bytes of the same launches from the committed ncu capture (N = 1 capture of this workload)
    tpath = os.path.join(ROOT, "profiles", "r01_gemm_traffic.json")
    if world == 1 and PRESET == "v6-7b" and BATCH == 16 and args.quant == "none" and os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj["layers"] * sum(x["dram_bytes"] for x in tj["per_layer_gemm_launches"]) + tj["head"]["algorithmic_weight_bytes"]
    windows_sum_us = sum(v[0] for v in cls.values())
    roofline = {"bound": "hbm", "kernel": "gemm_kernel (tcgen05 projection GEMM: every launch of one step, per GPU)",
                "achieved": gemm_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gemm_gbs / peaks["hbm_gbs"],
                "peak_source": f"MEASURED_PEAKS.json ({peak_src})", "traffic": traffic,
                "traffic_note": "per step, summed over the same projection launches as `achieved`: ncu dram read+write bytes of one "
                                "captured layer x 32 + the head's algorithmic bytes (profiles/r01_gemm_traffic.json)",
                "how": "in situ: algorithmic weight bytes of the step's projection launches / sum of their windows [griddepcontrol.wait "
                       "released, last CTA exit] inside a graph-replayed step (globaltimer stamps, mean of 5 replays)",
                "algorithmic_bytes_per_step_gemm": int(gemm_bytes), "gemm_us_per_step": gemm_us, "gemm_launches_per_step": int(gemm_n),
                "class_us_per_step": {k: v[0] for k, v in cls.items()},
                "class_launches_per_step": {k: int(v[1]) for k, v in cls.items()},
                "insitu_step_us": insitu_step_us, "windows_sum_us": windows_sum_us,
                "between_windows_us": insitu_step_us - windows_sum_us,
                "per_launch_class": {k: {"launches": int(v[1]), "avg_us": v[0] / max(v[1], 1),
                                         "gbs": (v[2] / (v[0] * 1e-6) / 1e9) if v[2] and v[0] > 0 else None}
                                     for k, v in sorted(per_label.items())},
                "events_ungraphed": {"gemm_ms": float(prof_ms[0]), "wkv_ms": float(prof_ms[1]), "ln_mix_ms": float(prof_ms[2]),
                                     "other_ms": float(prof_ms[3]), "launches": [int(x) for x in prof_n],
                                     "note": "CUDA events around every launch of an un-graphed step without PDL: upper bounds"},
                "step_algorithmic_bytes": int(alg_bytes),
                "step_achieved_gbs": alg_bytes / (ms_per_step * 1e-3) / 1e9,
                "step_frac": alg_bytes / (ms_per_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "step_ms_p10_p50_p90": [float(np.percentile(step_ms_dist, q)) for q in (10, 50, 90)] if step_ms_dist.size else None}

    # ---- the parity path beside the throughput path: precision 1 (f32-exact activations) on the same workload ----
    exact_rec = None
    if world == 1 and not args.exact and args.quant == "none" and os.environ.get("B200RWKV_BENCH_SKIP_EXACT") != "1":
        m2 = runtime.Model(st, max_batch=BATCH, token_chunk_size=64, device=dev, exact=True)
        for s_ in slots:
            m2.state.load(zero, s_)
        m2.infer_raw(slots, [PROMPT] * BATCH, toks[:, :PROMPT].reshape(-1).tolist(), [2] * BATCH)
        ms2, _ = m2.bench_decode(slots, dec, args.warmup, args.steps)
        exact_rec = {"ms_per_step": ms2 / args.steps, "value": BATCH * args.steps / (ms2 * 1e-3), "unit": "tokens/s",
                     "what": "b200rwkv_create(precision = 1): split f16 hi+lo operands, no activation rounded; logits within 1.6e-4 of the "
                             "f32 oracle at the 7B shape (tests/test_gpu_zfullsize.py, profiles/r02_parity_fullsize.jsonl)"}
        m2.close()

    # ---- cpu baseline (rank 0, N=1 only) ----
    cpu = None
    if world == 1 and args.cpu_steps > 0 and args.quant == "none":
        w = O.parse_st(st)
        ctoks = toks[:, PROMPT:PROMPT + args.cpu_steps + 1]
        tps, cms, threads, _ = cpu_arm(w, BATCH, args.cpu_steps, 1, ctoks, budget_s=30.0)
        cpu = {"value": tps, "unit": "tokens/s", "cores": threads, "kind": "port", "ms_per_step": cms,
               "sample": f"{args.cpu_steps} decode steps of the same workload on the host cores (C/OpenMP oracle, "
                         "f16 weights, f32 math); reference web-rwkv/lavapipe path unbuildable here"}

    line = {"metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "precision1": exact_rec, "build_seconds": build_s}
    print(json.dumps(line))
    barrier()
    model.close()


if __name__ == "__main__":
    main()
