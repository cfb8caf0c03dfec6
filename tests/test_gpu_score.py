"""Scoring given tokens on the device (b200rwkv_infer_score, csrc/sample.cuh score_rows_kernel) and the reference's
perplexity() / Choose restated on it (runtime.Model.perplexity / choose; reference crates/ai00-core/src/run.rs:699-755,
936-983), against float64 log-softmax of the engine's own FULL rows, of the oracle's logits (oracle/score_numpy.py), across
step cuts, mixed entries, chained calls, the f32-activation and Int8 modes, the error cases and tensor parallelism."""
import dataclasses
import math

import numpy as np
import pytest

from ai00_server_b200 import capi, runtime, synth
from oracle import rwkv_numpy as O
from oracle import sampling_numpy as S
from oracle import score_numpy as SC

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3          # the engine's logits against the oracle (test_gpu_parity.py)
STEP_TOL = 5e-4         # the same engine under different step shapes (test_decode_matches_prefill_and_chunking)
SCORE, KEPT, FULL, LAST = capi.OPTION_SCORE, capi.OPTION_SCORE_KEPT, capi.OPTION_FULL, capi.OPTION_LAST


def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.fixture(scope="module")
def models():
    cache = {}

    def get(preset, max_batch=4, chunk=32, exact=False, quant=0, devices=None, **over):
        key = (preset, max_batch, chunk, exact, quant, tuple(devices or ()), tuple(sorted(over.items())))
        if key not in cache:
            shp = dataclasses.replace(synth.PRESETS[preset], **over) if over else synth.PRESETS[preset]
            st = synth.make_st(shp, 0)
            m = runtime.Model(st, max_batch=max_batch, token_chunk_size=chunk, exact=exact, devices=devices,
                              quant=quant, quant_type="int8" if quant else 0)
            cache[key] = (m, st)
        return cache[key]

    yield get
    for m, _ in cache.values():
        m.close()


def targets_logp(rows, toks):
    """float64 log-softmax of each row at the next token: entry j >= 1 of what SCORE returns"""
    return SC.token_logp(rows, toks)[1:]


def full_rows(m, slot, toks, state):
    m.state.load(state, slot)
    return m.infer_raw([slot], [len(toks)], toks, [FULL])[0].copy()


def kept_row(m, slot):
    snap = m.state.read(slot)
    try:
        return m.state.snapshot_back(snap, with_logits=True)[1]
    finally:
        snap.free()


def check_own_rows(m, toks, tol=1e-5):
    """FULL and SCORE calls with the same entry shape from the same state run identical steps: logp equals float64
    log-softmax of the FULL rows at the targets up to the kernel's f32 reduction."""
    zero = m.state.init()
    rows = full_rows(m, 0, toks, zero)
    m.state.load(zero, 0)
    host, (lp,) = m.infer_score([0], [len(toks)], toks, [SCORE])
    assert host[0].shape[0] == 0 and lp.shape == (len(toks),)
    assert math.isnan(lp[0])
    err = np.abs(lp[1:].astype(np.float64) - targets_logp(rows, toks)).max()
    assert err <= tol, err
    return rows, lp


TOKS = [1, 5, 9, 33, 2, 7, 300, 41, 41, 8, 0, 17, 250, 3, 3, 99, 12, 400, 6, 77, 5, 1, 2, 130, 64, 65, 66, 67, 411, 8, 9, 10,
        11, 12, 13, 14, 15]       # 37 tokens: two steps at chunk 32


@pytest.mark.parametrize("preset,over", [("tiny5", {}), ("tiny6", {}), ("tiny7", {}), ("small6", {}), ("small6", {"V": 65536})])
def test_scores_match_the_engines_own_rows(models, preset, over):
    m, _ = models(preset, **over)
    check_own_rows(m, TOKS)


@pytest.mark.parametrize("preset", ["tiny5", "tiny6", "tiny7", "small6"])
def test_scores_match_the_oracle(models, preset):
    """log-softmax moves by at most 2 max|dx|, and the logits are within REL_TOL * max|x| of the oracle's f16 contract."""
    m, st = models(preset)
    orc = O.Oracle(O.parse_st(st), "f16")
    m.state.load(m.state.init(), 1)
    _, (lp,) = m.infer_score([1], [len(TOKS)], TOKS, [SCORE])
    want, _ = orc.run(TOKS, orc.state_init(), full=True)
    bound = 2 * REL_TOL * np.abs(want).max()
    err = np.abs(lp[1:].astype(np.float64) - targets_logp(want, TOKS)).max()
    assert err <= bound, (err, bound)


def test_step_cuts_and_mixed_entries(models):
    """At chunk 8 one call carries SCORE 11, LAST 5, SCORE_KEPT 9, SCORE 1 and SCORE 0 entries with a host logits buffer:
    the packer cuts the scoring runs across steps, so some targets are the first token of the entry's next step."""
    m, _ = models("tiny6", max_batch=6, chunk=8)
    rng = np.random.default_rng(3)
    zero = m.state.init()
    runs = [rng.integers(1, 500, n).tolist() for n in (11, 5, 9, 1, 0)]
    prompt = rng.integers(1, 500, 6).tolist()
    # slot 2 holds a prompt and its kept row; the other slots start from zero
    m.state.load(zero, 2)
    head = m.infer_raw([2], [len(prompt)], prompt, [LAST])[0][0].copy()
    snap2 = m.state.read(2)
    for s in (0, 1, 3, 4):
        m.state.load(zero, s)
    opts = [SCORE, LAST, KEPT, SCORE, SCORE]
    out = np.full((4, m.info["num_vocab"]), np.nan, np.float32)
    host, lps = m.infer_score([0, 1, 2, 3, 4], [len(r) for r in runs], sum(runs, []), opts, out=out)
    assert [h.shape[0] for h in host] == [0, 1, 0, 0, 0]
    assert [lp.shape[0] for lp in lps] == [11, 9, 1, 0]
    # the LAST entry's row against a plain infer of that entry
    m.state.load(zero, 1)
    alone = m.infer_raw([1], [5], runs[1], [LAST])[0][0]
    assert np.abs(host[1][0] - alone).max() <= STEP_TOL * np.abs(alone).max()
    assert host[1][0].argmax() == alone.argmax()
    # every score against solo FULL calls (other step shapes: the chunking bound of the logits, doubled by log-softmax)
    rows0 = full_rows(m, 0, runs[0], zero)
    assert math.isnan(lps[0][0])
    bound = 2 * STEP_TOL * np.abs(rows0).max()
    assert np.abs(lps[0][1:] - targets_logp(rows0, runs[0])).max() <= bound
    m.state.write(snap2, 2)
    rows2 = m.infer_raw([2], [9], runs[2], [FULL])[0].copy()
    want2 = SC.token_logp(rows2, runs[2], head_row=head)
    bound = 2 * STEP_TOL * max(np.abs(rows2).max(), np.abs(head).max())
    assert np.abs(lps[1] - want2).max() <= bound
    assert lps[1][0] == pytest.approx(SC.log_softmax(head)[runs[2][0]], abs=1e-5)      # the kept row itself, unchanged
    assert math.isnan(lps[2][0])
    snap2.free()


def test_chained_calls_equal_one_call_and_leave_the_last_row_kept(models):
    m, _ = models("tiny6")
    rng = np.random.default_rng(7)
    toks = rng.integers(1, 500, size=45).tolist()
    zero = m.state.init()
    rows = full_rows(m, 0, toks, zero)             # 45 tokens at chunk 32: two steps
    m.state.load(zero, 0)
    _, (one,) = m.infer_score([0], [45], toks, [SCORE])
    m.state.load(zero, 1)
    _, (a,) = m.infer_score([1], [7], toks[:7], [SCORE])
    _, (b,) = m.infer_score([1], [23], toks[7:30], [KEPT])
    _, (c,) = m.infer_score([1], [15], toks[30:], [KEPT])
    chained = np.concatenate([a, b, c])
    assert math.isnan(one[0]) and math.isnan(chained[0])
    assert np.abs(one[1:] - chained[1:]).max() <= 2 * STEP_TOL * np.abs(rows).max()
    # the kept row after the one-call score is the last row of a FULL call with the same entry shape, bit for bit
    last = kept_row(m, 0)
    assert np.array_equal(last, rows[-1])
    ids, _ = m.sample_topk([0], top_k=16)
    want, _ = S.sorted_candidates(rows[-1], top_k=16)
    assert np.array_equal(ids[0], want)


@pytest.mark.parametrize("calibrate", [False, True])
def test_choose_matches_the_oracle_and_restores_the_slot(models, calibrate):
    m, st = models("tiny6")
    orc = O.Oracle(O.parse_st(st), "f16")
    rng = np.random.default_rng(5)
    prompt = rng.integers(1, 500, 12).tolist()
    choices = [rng.integers(1, 500, 4).tolist(), [7], [], rng.integers(1, 500, 9).tolist(), [41, 41]]
    m.state.load(m.state.init(), 3)
    m.infer_raw([3], [len(prompt)], prompt, [LAST])
    state_before, row_before = m.state.back(3), kept_row(m, 3)
    got = m.choose(3, choices, calibrate)
    # the slot is what it was: state and kept row
    assert np.array_equal(m.state.back(3), state_before)
    assert np.array_equal(kept_row(m, 3), row_before)
    # the oracle on the same token sequences
    p_logits, p_state = orc.run(prompt, orc.state_init())
    head = p_logits[-1] if p_logits.ndim == 2 else p_logits
    rows_head = [orc.run(c, p_state, full=True)[0] if c else None for c in choices]
    rows_init = [orc.run([0] + c, orc.state_init(), full=True)[0] if c else None for c in choices]
    want = SC.choose(choices, head, rows_head, rows_init, calibrate=calibrate)
    xmax = max([np.abs(head).max()] + [np.abs(r).max() for r in rows_head + rows_init if r is not None])
    bound = 2 * REL_TOL * xmax * (2 if calibrate else 1)       # calibrate: the difference of two perplexities
    assert got[2] == math.inf and want[2] == math.inf
    live = [i for i, c in enumerate(choices) if c]
    assert max(abs(got[i] - want[i]) for i in live) <= bound
    assert min(live, key=lambda i: got[i]) == min(live, key=lambda i: want[i])


def test_perplexity_head_and_no_head(models):
    """runtime.Model.perplexity against oracle/score_numpy.perplexity on the engine's own FULL rows."""
    m, _ = models("small6")
    rng = np.random.default_rng(9)
    prompt, choice = rng.integers(1, 2000, 5).tolist(), rng.integers(1, 2000, 13).tolist()
    zero = m.state.init()
    m.state.load(zero, 2)
    head = m.infer_raw([2], [5], prompt, [LAST])[0][0].copy()
    snap = m.state.read(2)
    rows = m.infer_raw([2], [13], choice, [FULL])[0].copy()
    m.state.write(snap, 2)
    assert m.perplexity(2, choice, head=True) == pytest.approx(SC.perplexity(rows, choice, head), abs=1e-5)
    rows0 = full_rows(m, 2, [0] + choice, zero)
    m.state.load(zero, 2)
    assert m.perplexity(2, choice, head=False) == pytest.approx(SC.perplexity(rows0, choice), abs=1e-5)
    snap.free()


@pytest.mark.parametrize("mode", ["exact", "int8"])
def test_other_modes(models, mode):
    m, _ = models("tiny6", exact=(mode == "exact"), quant=(2 if mode == "int8" else 0))
    check_own_rows(m, TOKS)


def test_vocabulary_not_a_multiple_of_4(models):
    """Rows of odd width take the kernel's scalar path; such an engine keeps no rows, so SCORE_KEPT is unsupported."""
    m, _ = models("tiny6", V=510)
    check_own_rows(m, TOKS)
    m.state.load(m.state.init(), 1)
    m.infer_raw([1], [3], [4, 5, 6], [LAST])
    before = m.state.back(1)
    with pytest.raises(capi.B200Error) as ei:
        m.infer_score([1], [2], [7, 8], [KEPT])
    assert ei.value.code == capi.ERR_UNSUPPORTED
    assert np.array_equal(m.state.back(1), before)


def test_errors_change_no_state(models):
    m, _ = models("tiny6", max_batch=4, chunk=16)
    L = capi.lib()
    m.state.load(m.state.init(), 0)
    m.infer_raw([0], [3], [4, 5, 6], [LAST])
    fresh = runtime.Model(synth.make_st("tiny6", 0), max_batch=2, token_chunk_size=16)
    try:
        fresh.state.load(fresh.state.init(), 1)
        before = fresh.state.back(1)
        with pytest.raises(capi.B200Error) as ei:              # slot 1 has never produced a row
            fresh.infer_score([1], [2], [7, 8], [KEPT])
        assert ei.value.code == capi.ERR_STATE
        assert np.array_equal(fresh.state.back(1), before)
    finally:
        fresh.close()
    state0, row0 = m.state.back(0), kept_row(m, 0)

    def call(opt, logp, cap, fn=L.b200rwkv_infer_score):
        s, n, t, o = (np.asarray(x, d) for x, d in (([0], np.int32), ([4], np.int32), ([9, 10, 11, 12], np.uint32), ([opt], np.int32)))
        rows = np.zeros(1, np.int32)
        args = [m._h, 1, capi.ptr(s), capi.ptr(n), capi.ptr(t), capi.ptr(o), None, 0, capi.ptr(rows)]
        if fn is L.b200rwkv_infer_score:
            args += [capi.ptr(logp) if logp is not None else None, cap]
        return fn(*args)

    buf = np.zeros(4, np.float32)
    assert call(SCORE, None, 4) == capi.ERR_INVALID                  # scoring entries need a logp buffer
    assert call(KEPT, buf, 3) == capi.ERR_INVALID                    # ... of at least their token total
    for opt in (SCORE, KEPT):                                        # b200rwkv_infer does not take the scoring options
        assert call(opt, None, 0, fn=L.b200rwkv_infer) == capi.ERR_INVALID
    assert np.array_equal(m.state.back(0), state0)
    assert np.array_equal(kept_row(m, 0), row0)
    # an accepted call with the exact capacity
    assert call(KEPT, buf, 4) == capi.OK and np.isfinite(buf).all()


@pytest.mark.skipif(_ngpu() < 2, reason="needs at least 2 GPUs")
def test_tensor_parallel_matches_one_gpu(models):
    """In-process ranks: rank 0 reads every rank's vocabulary shard.  The sharded and the single-GPU engine differ in f32
    summation order only."""
    single, _ = models("small6")
    multi, _ = models("small6", devices=[0, 1])
    rng = np.random.default_rng(13)
    prompt, toks = rng.integers(1, 2000, 6).tolist(), rng.integers(1, 2000, 40).tolist()
    res = []
    for m in (single, multi):
        zero = m.state.init()
        for s in (0, 1):
            m.state.load(zero, s)
        m.infer_raw([1], [6], prompt, [LAST], keep_on_device=True)
        rows = full_rows(m, 2, toks, zero)
        _, lps = m.infer_score([0, 1], [40, 40], toks + toks, [SCORE, KEPT])
        res.append((rows, lps))
    (rows, (a0, a1)), (_, (b0, b1)) = res
    bound = 2 * 1e-4 * np.abs(rows).max()
    assert math.isnan(b0[0])
    assert np.abs(a0[1:] - b0[1:]).max() <= bound
    assert np.abs(a1 - b1).max() <= bound
