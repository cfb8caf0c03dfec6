"""Host-side mirror of the web-rwkv interface that crates/ai00-core consumes, over the C ABI.

The reference's host code is Rust (crates/ai00-core/src/run.rs, lib.rs) and no Rust toolchain
exists in this image, so the shim that would live in ai00-core is specified in INTEGRATION.md
and mirrored here 1:1 in Python for the parity tests and bench.py: same names, argument
meaning and error behaviour as the trait objects the reference holds:

  RnnOption / RnnInputBatch / RnnInput / RnnOutputBatch   run.rs:25, 1121-1136, 1146
  Runtime.infer(input) -> (input, output)                   run.rs:1143
  State.{init, load, back, read, write}                     run.rs:477, 1099-1107
  softmax(list of [V] tensors)                              run.rs:1179
  Loader.info                                               lib.rs:587
  ModelBuilder(...).build() + Bundle(model, max_batch)      lib.rs:484-497

Every method calls straight into libb200rwkv.so; nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import enum
from dataclasses import dataclass, field

import numpy as np

from . import capi


class RnnOption(enum.IntEnum):
    Last = capi.OPTION_LAST
    Full = capi.OPTION_FULL


@dataclass
class RnnInputBatch:
    tokens: list = field(default_factory=list)
    option: RnnOption = RnnOption.Last


@dataclass
class RnnInput:
    batches: list
    token_chunk_size: int

    def num_token(self) -> int:
        return sum(len(b.tokens) for b in self.batches)


@dataclass
class RnnOutputBatch:
    """`RnnOutputBatch(TensorCpu<f32>)`: [rows, V]; empty when the slot produced nothing."""
    data: np.ndarray

    def is_empty(self) -> bool:
        return self.data.shape[0] == 0


class Loader:
    @staticmethod
    def info(st: np.ndarray) -> dict:
        return capi.info_from_st(st)


def read_state(info: dict, st: np.ndarray) -> np.ndarray:
    """`vN::read_state(&context, &info, reader)` (lib.rs:378-389): `.state` file / state-tuned model -> state tensor."""
    st = np.ascontiguousarray(st, dtype=np.uint8)
    ci = capi.Info(**{k: int(v) for k, v in info.items()})
    out = np.empty((info["num_layer"], info["head_size"] + 2, info["num_emb"]), np.float32)
    capi.check(capi.lib().b200rwkv_read_state(C.byref(ci), capi.ptr(st), st.size, capi.ptr(out)))
    return out


class TensorGpu:
    """Device-side state snapshot handle (`TensorGpu<f32, ReadWrite>` at run.rs:1104-1108)."""

    def __init__(self, model: "Model", snap_id: int):
        self._model, self.id = model, snap_id

    def free(self):
        if self.id:
            capi.check(capi.lib().b200rwkv_state_free(self._model._h, self.id), self._model._h)
            self.id = 0


class State:
    def __init__(self, model: "Model"):
        self._m = model

    def shape(self):
        s = (C.c_int64 * 4)()
        capi.check(capi.lib().b200rwkv_state_shape(self._m._h, C.byref(s)), self._m._h)
        return tuple(s)

    def _numel(self):
        s = self.shape()
        return int(s[0] * s[1] * s[2] * s[3])

    def _np_shape(self):
        c, r, l, _ = self.shape()
        return (int(l), int(r), int(c))        # numpy C-order view of web-rwkv [C, N+2, L, 1]

    def init(self) -> np.ndarray:
        out = np.empty(self._np_shape(), np.float32)
        capi.check(capi.lib().b200rwkv_state_init(self._m._h, capi.ptr(out)), self._m._h)
        return out

    def load(self, tensor: np.ndarray, batch: int) -> None:
        t = np.ascontiguousarray(tensor, dtype=np.float32)
        if t.size != self._numel():
            raise capi.B200Error(capi.ERR_INVALID, "state tensor has the wrong number of elements")
        capi.check(capi.lib().b200rwkv_state_load(self._m._h, batch, capi.ptr(t)), self._m._h)

    def back(self, batch: int) -> np.ndarray:
        out = np.empty(self._np_shape(), np.float32)
        capi.check(capi.lib().b200rwkv_state_back(self._m._h, batch, capi.ptr(out)), self._m._h)
        return out

    def read(self, batch: int) -> TensorGpu:
        sid = C.c_uint64(0)
        capi.check(capi.lib().b200rwkv_state_read(self._m._h, batch, C.byref(sid)), self._m._h)
        return TensorGpu(self._m, sid.value)

    def write(self, tensor: TensorGpu, batch: int) -> None:
        capi.check(capi.lib().b200rwkv_state_write(self._m._h, batch, tensor.id), self._m._h)

    # ---- device-resident cache items (CachedItem {state, output}, run.rs:199-205) ----
    def snapshot_back(self, tensor: TensorGpu, with_logits: bool = False):
        out = np.empty(self._np_shape(), np.float32)
        lg = np.empty(self._m.info["num_vocab"], np.float32) if with_logits else None
        capi.check(capi.lib().b200rwkv_snapshot_back(self._m._h, tensor.id, capi.ptr(out), capi.ptr(lg) if with_logits else None), self._m._h)
        return (out, lg) if with_logits else out

    def snapshot_load(self, tensor: np.ndarray, logits: np.ndarray | None = None) -> TensorGpu:
        t = np.ascontiguousarray(tensor, dtype=np.float32)
        if t.size != self._numel():
            raise capi.B200Error(capi.ERR_INVALID, "state tensor has the wrong number of elements")
        lg = None if logits is None else np.ascontiguousarray(logits, dtype=np.float32)
        sid = C.c_uint64(0)
        capi.check(capi.lib().b200rwkv_snapshot_load(self._m._h, capi.ptr(t), capi.ptr(lg) if lg is not None else None, C.byref(sid)), self._m._h)
        return TensorGpu(self._m, sid.value)

    def cache_stats(self) -> dict:
        n, used, free = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        capi.check(capi.lib().b200rwkv_cache_stats(self._m._h, C.byref(n), C.byref(used), C.byref(free)), self._m._h)
        return {"snapshots": n.value, "bytes_used": used.value, "bytes_free": free.value}


class NucleusSampler:
    """Host back half of the reference's `NucleusSampler` (sampler/nucleus.rs:13-123) over the <= 128 candidates the GPU
    front half returns: same parameters, same penalty state, same arithmetic in f32; `rand` is the uniform draw the
    reference takes from fastrand (nucleus.rs:104), passed in so tests are deterministic."""

    def __init__(self, top_p=0.5, top_k=128, temperature=1.0, presence_penalty=0.3, frequency_penalty=0.3,
                 penalty_decay=0.99654026):
        f = np.float32
        self.top_p, self.top_k, self.temperature = f(top_p), int(top_k), f(temperature)
        self.presence_penalty, self.frequency_penalty, self.penalty_decay = f(presence_penalty), f(frequency_penalty), f(penalty_decay)
        self.penalties: dict[int, np.float32] = {}

    def init(self, model_tokens):                                   # nucleus.rs:50-59
        for index, token in enumerate(reversed(list(model_tokens))):
            pen = self.penalties.pop(int(token), self.presence_penalty)
            pen = np.float32(pen + self.frequency_penalty * np.float32(np.power(self.penalty_decay, np.float32(index))))
            self.penalties[int(token)] = pen

    def sample_candidates(self, ids, probs, rand: float) -> int:   # nucleus.rs:69-123 after the sort / take(top_k)
        f = np.float32
        kept, cum = [], f(0.0)
        for i, x in zip(ids[:self.top_k], probs[:self.top_k]):
            if cum > self.top_p:
                break
            cum = f(cum + x)
            kept.append((int(i), f(np.power(f(x), f(1.0) / self.temperature))))
        total = f(0.0)
        for _, x in kept:
            total = f(total + x)
        token, cum = kept[0][0], f(0.0)
        for i, x in kept:
            cum = f(cum + f(x / total))
            if f(rand) <= cum:
                token = i
                break
        for t in self.penalties:
            self.penalties[t] = f(self.penalties[t] * self.penalty_decay)
        self.penalties[token] = f(self.penalties[token] + self.frequency_penalty) if token in self.penalties else self.presence_penalty
        return token


class Runtime:
    """`Arc<dyn Runtime<Rnn>>`.  `infer` consumes at most `token_chunk_size` tokens of the
    input across slots and returns the remaining input with the per-slot outputs, exactly the
    contract the batching shim loops on (run.rs:1134-1155)."""

    def __init__(self, model: "Model"):
        self._m = model

    def infer(self, inp: RnnInput):
        m = self._m
        budget = max(1, inp.token_chunk_size)
        slots, ntok, opts, toks, takes = [], [], [], [], []
        for b, batch in enumerate(inp.batches):
            if not batch.tokens or budget == 0:
                takes.append(0)
                continue
            take = min(len(batch.tokens), budget)
            budget -= take
            takes.append(take)
            finishes = take == len(batch.tokens)
            slots.append(b)
            ntok.append(take)
            toks.extend(int(t) for t in batch.tokens[:take])
            # Last only yields a row once the slot's tokens are exhausted
            opts.append(int(RnnOption.Full) if batch.option == RnnOption.Full
                        else (int(RnnOption.Last) if finishes else capi.OPTION_NONE))
        rows = m.infer_raw(slots, ntok, toks, opts)
        out = [RnnOutputBatch(np.zeros((0, m.info["num_vocab"]), np.float32)) for _ in inp.batches]
        for s, r in zip(slots, rows):
            out[s] = RnnOutputBatch(r)
        rest = RnnInput([RnnInputBatch(list(b.tokens[t:]), b.option) for b, t in zip(inp.batches, takes)],
                        inp.token_chunk_size)
        return rest, out


class Model:
    """Owns one engine (`ModelBuilder...build_vN()` + `Bundle::new(model, max_batch)` +
    `TokioRuntime::new(bundle)`, lib.rs:484-497)."""

    def __init__(self, st: np.ndarray, max_batch: int = 8, token_chunk_size: int = 128, device: int = 0,
                 precision: int = 0, rank: int = 0, world: int = 1, exact: bool = False, devices=None, lora=None,
                 quant: int = 0, quant_type: int | str = 0):
        """devices: list of CUDA ordinals -> ONE engine object owning all tensor-parallel ranks (b200rwkv_create_ex);
        lora: list of (st_bytes, alpha) blended at load (reference lib.rs:466-485);
        quant / quant_type: the reload request's fields (lib.rs:211-215): the first `quant` layers in "Int8" or "NF4";
        rank / world: one process per GPU instead (b200rwkv_create_tp + tp.connect)."""
        if isinstance(quant_type, str):
            kinds = {"none": capi.QUANT_NONE, "int8": capi.QUANT_INT8, "nf4": capi.QUANT_NF4, "sf4": 3}
            if quant_type.lower() not in kinds:
                raise capi.B200Error(capi.ERR_INVALID, "quant_type must be None, Int8, NF4 or SF4")
            quant_type = kinds[quant_type.lower()]
        quantised = quant > 0 and quant_type != capi.QUANT_NONE
        if exact:
            precision = 1          # `Bundle::<f32>`: f32-exact activations (split hi + lo f16 operands)
        st = np.ascontiguousarray(st, dtype=np.uint8)
        h = C.c_void_p()
        L = capi.lib()
        if devices is not None or lora or quantised:
            if world != 1:
                raise capi.B200Error(capi.ERR_INVALID, "devices / lora / quant go through b200rwkv_create_ex (in-process ranks)")
            opt = capi.Options()
            opt.struct_bytes = C.sizeof(capi.Options)
            opt.max_batch, opt.token_chunk_size, opt.precision = max_batch, token_chunk_size, precision
            devs = list(devices) if devices is not None else [device]
            opt.num_devices = len(devs)
            for i, d in enumerate(devs):
                opt.devices[i] = int(d)
            self._lora_keep = []
            for i, (img, alpha) in enumerate(lora or []):
                img = np.ascontiguousarray(img, dtype=np.uint8)
                self._lora_keep.append(img)
                opt.lora_st[i], opt.lora_len[i], opt.lora_alpha[i] = img.ctypes.data, img.size, float(alpha)
            opt.num_lora = len(lora or [])
            opt.quant_layers, opt.quant_type = (int(quant), int(quant_type)) if quantised else (0, 0)
            capi.check(L.b200rwkv_create_ex(capi.ptr(st), st.size, C.byref(opt), C.byref(h)))
            self._lora_keep = []
        else:
            capi.check(L.b200rwkv_create_tp(capi.ptr(st), st.size, device, max_batch, token_chunk_size, precision,
                                            rank, world, C.byref(h)))
        self._h = h
        self.max_batch, self.token_chunk_size = max_batch, token_chunk_size
        self.rank, self.world = rank, world
        info = capi.Info()
        capi.check(L.b200rwkv_get_info(self._h, C.byref(info)), self._h)
        self.info = info.as_dict()
        self.runtime = Runtime(self)
        self.state = State(self)

    def close(self):
        if self._h:
            capi.lib().b200rwkv_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- raw call: one b200rwkv_infer ----
    def infer_raw(self, slots, ntok, tokens, options, out: np.ndarray | None = None, keep_on_device: bool = False):
        V = self.info["num_vocab"]          # rank 0 receives the gathered full-vocabulary rows
        n = len(slots)
        total = sum(nt if o == capi.OPTION_FULL else (1 if (o == capi.OPTION_LAST and nt > 0) else 0)
                    for nt, o in zip(ntok, options))
        if keep_on_device:                  # logits_out = NULL: rows stay in HBM for sample_topk
            a_slot, a_ntok = np.asarray(slots, np.int32), np.asarray(ntok, np.int32)
            a_tok, a_opt = np.asarray(tokens, np.uint32), np.asarray(options, np.int32)
            a_rows = np.zeros(max(n, 1), np.int32)
            capi.check(capi.lib().b200rwkv_infer(self._h, n, capi.ptr(a_slot), capi.ptr(a_ntok), capi.ptr(a_tok),
                                                 capi.ptr(a_opt), None, 0, capi.ptr(a_rows)), self._h)
            return [int(r) for r in a_rows[:n]]
        if out is None:
            out = np.empty((max(total, 1), V), np.float32)
        a_slot = np.asarray(slots, np.int32)
        a_ntok = np.asarray(ntok, np.int32)
        a_tok = np.asarray(tokens, np.uint32)
        a_opt = np.asarray(options, np.int32)
        a_rows = np.zeros(max(n, 1), np.int32)
        capi.check(capi.lib().b200rwkv_infer(self._h, n, capi.ptr(a_slot), capi.ptr(a_ntok), capi.ptr(a_tok),
                                             capi.ptr(a_opt), capi.ptr(out), out.size, capi.ptr(a_rows)), self._h)
        res, off = [], 0
        for i in range(n):
            r = int(a_rows[i])
            res.append(out[off:off + r])
            off += r
        return res

    # ---- scoring: b200rwkv_infer_score ----
    def infer_score(self, slots, ntok, tokens, options, out: np.ndarray | None = None):
        """One b200rwkv_infer_score call.  Options as infer_raw plus capi.OPTION_SCORE / OPTION_SCORE_KEPT.  Returns (host rows
        per entry -- [rows, V], none for scoring entries --, one f32 log-probability array per scoring entry in entry order)."""
        V = self.info["num_vocab"]
        n = len(slots)
        scoring = (capi.OPTION_SCORE, capi.OPTION_SCORE_KEPT)
        total = sum(nt if o == capi.OPTION_FULL else (1 if (o == capi.OPTION_LAST and nt > 0) else 0) for nt, o in zip(ntok, options))
        nscore = sum(nt for nt, o in zip(ntok, options) if o in scoring)
        if out is None and total > 0:
            out = np.empty((total, V), np.float32)
        logp = np.empty(max(nscore, 1), np.float32)
        a_slot, a_ntok = np.asarray(slots, np.int32), np.asarray(ntok, np.int32)
        a_tok, a_opt = np.asarray(tokens, np.uint32), np.asarray(options, np.int32)
        a_rows = np.zeros(max(n, 1), np.int32)
        capi.check(capi.lib().b200rwkv_infer_score(self._h, n, capi.ptr(a_slot), capi.ptr(a_ntok), capi.ptr(a_tok), capi.ptr(a_opt),
                                                   capi.ptr(out) if out is not None else None, out.size if out is not None else 0,
                                                   capi.ptr(a_rows), capi.ptr(logp), nscore), self._h)
        rows, lps, off, loff = [], [], 0, 0
        for i in range(n):
            r = int(a_rows[i])
            rows.append(out[off:off + r] if r else np.zeros((0, V), np.float32))
            off += r
            if options[i] in scoring:
                lps.append(logp[loff:loff + ntok[i]].copy())
                loff += ntok[i]
        return rows, lps

    def perplexity(self, batch: int, tokens, head: bool) -> float:
        """The reference's `perplexity(batch, tokens, head)` (run.rs:699-755) on the device: -mean ln p of the tokens, fed to
        slot `batch` from its current state.  head = True is `Some(output[tokens[0]])`: the first token is scored against the
        slot's kept row (SCORE_KEPT).  head = False is `None`: like the reference, token 0 is prepended and fed too, and the sum
        of len(tokens) terms is divided by len(tokens) + 1.  The reference's f32 sum of ln p is kept."""
        toks = [int(t) for t in tokens]
        if not toks:
            raise capi.B200Error(capi.ERR_INVALID, "perplexity of an empty token list is undefined (the reference never asks)")
        if head:
            _, (lp,) = self.infer_score([batch], [len(toks)], toks, [capi.OPTION_SCORE_KEPT])
        else:
            toks = [0] + toks
            _, (lp,) = self.infer_score([batch], [len(toks)], toks, [capi.OPTION_SCORE])
            lp = lp[1:]
        s = np.float32(0.0)
        for x in lp:
            s = np.float32(s + x)
        return float(np.float32(-s) / np.float32(len(toks)))

    def choose(self, batch: int, choices, calibrate: bool, init_state: np.ndarray | None = None) -> list[float]:
        """The Choose branch of the reference (run.rs:936-983) on slot `batch`, which holds the prompt's state and kept row:
        ppl per choice (lower is better, empty choices +inf).  calibrate subtracts each choice's no-head perplexity from
        `init_state` (the cached state of the request, default State::init).  The slot's state and kept row are snapshotted
        with State::read and restored with State::write after every choice."""
        backed = self.state.read(batch)
        try:
            ppl = [float("inf")] * len(choices)
            if calibrate:
                init = self.state.init() if init_state is None else init_state
                for i, c in enumerate(choices):
                    if len(c):
                        self.state.load(init, batch)
                        ppl[i] = -self.perplexity(batch, c, head=False)
                self.state.write(backed, batch)
            for i, c in enumerate(choices):
                if len(c):
                    p = self.perplexity(batch, c, head=True)
                    ppl[i] = ppl[i] + p if calibrate else p
                    self.state.write(backed, batch)
        finally:
            backed.free()
        return ppl

    def softmax(self, tensors):
        """`softmax(&context, Vec<TensorCpu<f32>>)`: list of [V] rows in, list out."""
        if not tensors:
            return []
        x = np.ascontiguousarray(np.stack([np.asarray(t, np.float32).reshape(-1) for t in tensors], 0))
        y = np.empty_like(x)
        capi.check(capi.lib().b200rwkv_softmax(self._h, x.shape[0], capi.ptr(x), capi.ptr(y)), self._h)
        return [y[i] for i in range(y.shape[0])]

    def sample_topk(self, slots, penalties=None, bias=None, allow=None, top_k: int = 128):
        """GPU front half of sampling (b200rwkv_sample_topk): for each slot the `top_k` most probable tokens of its last
        logits row after penalties / grammar mask / bias, as (ids [n, top_k] uint32, probs [n, top_k] f32).
        penalties, bias: per-slot dict token -> value (the reference's HashMaps, nucleus.rs:29, run.rs:679);
        allow: optional [n, V] bool array (tokens the formatter allows)."""
        n = len(slots)
        V = self.info["num_vocab"]

        def pack(maps):
            off = np.zeros(n + 1, np.int32)
            toks, vals = [], []
            for i in range(n):
                m = (maps[i] if maps is not None else None) or {}
                toks.extend(int(t) for t in m.keys())
                vals.extend(float(v) for v in m.values())
                off[i + 1] = len(toks)
            return off, np.asarray(toks, np.uint32), np.asarray(vals, np.float32)

        po, pt, pv = pack(penalties)
        bo, bt, bv = pack(bias)
        bits = None
        if allow is not None:
            a = np.asarray(allow, bool).reshape(n, V)
            words = (V + 31) // 32
            padded = np.zeros((n, words * 32), bool)
            padded[:, :V] = a
            bits = np.ascontiguousarray(np.packbits(padded.reshape(n, words, 32), axis=2, bitorder="little").view(np.uint32).reshape(n, words))
        ids = np.empty((n, top_k), np.uint32)
        probs = np.empty((n, top_k), np.float32)
        a_slot = np.asarray(slots, np.int32)
        capi.check(capi.lib().b200rwkv_sample_topk(self._h, n, capi.ptr(a_slot), capi.ptr(po), capi.ptr(pt), capi.ptr(pv),
                                                   capi.ptr(bits) if bits is not None else None, capi.ptr(bo), capi.ptr(bt),
                                                   capi.ptr(bv), top_k, capi.ptr(ids), capi.ptr(probs)), self._h)
        return ids, probs

    def launch_count(self) -> int:
        n = C.c_int64(0)
        capi.check(capi.lib().b200rwkv_launch_count(self._h, C.byref(n)), self._h)
        return n.value

    def keep_hidden(self, enable: bool = True) -> None:
        capi.check(capi.lib().b200rwkv_keep_hidden(self._h, int(enable)), self._h)

    def last_hidden(self, max_rows: int = 64) -> np.ndarray:
        """Residual stream after the last layer per token of the most recent infer call (all tokens after keep_hidden())."""
        Cc = self.info["num_emb"]
        buf = np.empty((max_rows, Cc), np.float32)
        r = capi.lib().b200rwkv_last_hidden(self._h, capi.ptr(buf), buf.size)
        capi.check(r, self._h)
        return buf[:r]

    def debug_read(self, name: str) -> np.ndarray:
        """A named activation buffer of the most recent internal step (b200rwkv_debug_read): [rows, cols] f32, rows as the
        engine reports them (the step's tokens; its output rows for "a_head")."""
        buf = np.empty(128 * 65536, np.float32)
        rows = C.c_int32(0)
        cols = capi.lib().b200rwkv_debug_read(self._h, name.encode(), capi.ptr(buf), buf.size, C.byref(rows))
        capi.check(cols, self._h)
        return buf[: rows.value * cols].reshape(rows.value, cols).copy()

    def debug_plan(self, layer: int, mt: int) -> list[dict]:
        """Projection launches of `layer` (-1: the head) in a step of `mt` token tiles (b200rwkv_debug_plan)."""
        buf = np.zeros(64 * capi.PLAN_INTS, np.int32)
        n = capi.check(capi.lib().b200rwkv_debug_plan(self._h, layer, mt, capi.ptr(buf), buf.size), self._h)
        out = []
        for r in buf[: n * capi.PLAN_INTS].reshape(n, capi.PLAN_INTS):
            segs = [dict(zip(("KB", "tiles", "N", "out_mode", "act"), (int(x) for x in r[8 + 5 * i: 13 + 5 * i]))) for i in range(r[7])]
            out.append(dict(grid_run=int(r[0]), grid=int(r[1]), grid_wide=int(r[2]), total_blocks=int(r[3]), max_contrib=int(r[4]),
                            qtype=int(r[5]), forced=bool(r[6]), segs=segs))
        return out

    def bench_decode(self, slots, tokens: np.ndarray, warmup: int, steps: int, flush_l2: bool = False):
        a_slot = np.asarray(slots, np.int32)
        tok = np.ascontiguousarray(tokens, dtype=np.uint32)
        assert tok.size == (warmup + steps) * len(slots)
        ms = C.c_float(0)
        launches = C.c_int64(0)
        self.step_ms = np.zeros(steps, np.float32)          # CUDA-event time of every timed step (distribution)
        capi.check(capi.lib().b200rwkv_bench_decode(self._h, len(slots), capi.ptr(a_slot), capi.ptr(tok), warmup, steps,
                                                    int(flush_l2), C.byref(ms), C.byref(launches), capi.ptr(self.step_ms)), self._h)
        return ms.value, launches.value

    def profile_insitu(self, slots, tokens, reps: int = 5):
        """Per-launch windows of one graph-replayed decode step (b200rwkv_profile_insitu): list of dicts + step_us."""
        a_slot = np.asarray(slots, np.int32)
        tok = np.ascontiguousarray(tokens, dtype=np.uint32)
        cap = 1024
        n = C.c_int32(0)
        types = np.zeros(cap, np.int32)
        st, en = np.zeros(cap, np.float64), np.zeros(cap, np.float64)
        by = np.zeros(cap, np.int64)
        step = C.c_double(0)
        capi.check(capi.lib().b200rwkv_profile_insitu(self._h, len(slots), capi.ptr(a_slot), capi.ptr(tok), reps, cap, C.byref(n),
                                                      capi.ptr(types), capi.ptr(st), capi.ptr(en), capi.ptr(by), C.byref(step)), self._h)
        k = n.value
        return [{"type": int(types[i]), "start_us": float(st[i]), "end_us": float(en[i]), "bytes": int(by[i])} for i in range(k)], step.value

    def profile_step(self, slots, tokens):
        a_slot = np.asarray(slots, np.int32)
        tok = np.ascontiguousarray(tokens, dtype=np.uint32)
        ms = (C.c_float * 4)()
        ln = (C.c_int32 * 4)()
        wb = C.c_int64(0)
        capi.check(capi.lib().b200rwkv_profile_step(self._h, len(slots), capi.ptr(a_slot), capi.ptr(tok), C.byref(ms),
                                                    C.byref(ln), C.byref(wb)), self._h)
        return list(ms), list(ln), wb.value
