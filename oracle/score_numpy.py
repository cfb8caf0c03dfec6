"""float64 restatement of the reference's scoring path over given logits rows: `perplexity()` (crates/ai00-core/src/run.rs:
699-755) and the Choose branch that calls it (run.rs:936-983).  The rows are what the model emits; everything after them --
softmax at the next token, the logarithm, the head / no-head bookkeeping, the calibrate sum -- is restated here, so the engine's
b200rwkv_infer_score + runtime.Model.perplexity / choose can be checked against it on the same (or the oracle's) logits.

The reference works in probabilities: p = exp(x[t]) / sum exp(x), then ln p.  Here that is the max-shifted log-softmax in
float64, the same number without the overflow of exp(x) for large logits.
"""
from __future__ import annotations

import numpy as np


def log_softmax(row) -> np.ndarray:
    x = np.asarray(row, np.float64)
    m = x.max()
    return x - m - np.log(np.exp(x - m).sum())


def token_logp(rows, tokens, head_row=None) -> np.ndarray:
    """What b200rwkv_infer_score returns for one entry: rows[j] is the logits row emitted after tokens[j];
    logp[j] = log_softmax(rows[j - 1])[tokens[j]] for j >= 1, logp[0] = log_softmax(head_row)[tokens[0]] (SCORE_KEPT) or NaN
    (SCORE, head_row None).  The last row has no target and is not read."""
    t = [int(x) for x in tokens]
    out = np.full(len(t), np.nan, np.float64)
    if t and head_row is not None:
        out[0] = log_softmax(head_row)[t[0]]
    for j in range(1, len(t)):
        out[j] = log_softmax(rows[j - 1])[t[j]]
    return out


def perplexity(rows, tokens, head_row=None) -> float:
    """run.rs:699-755.  With a head (`Some(output[choice[0]])`): `rows` are the rows of `tokens` fed from the current state,
    head_row is the slot's last row before them, and the mean runs over len(tokens) terms.  Without (`None`): the reference
    feeds [0] + tokens, `rows` are the rows of that sequence, the first token is scored against the row of the prepended 0,
    and the sum of len(tokens) terms is divided by len(tokens) + 1 (the length of the fed sequence)."""
    t = [int(x) for x in tokens]
    if head_row is not None:
        lp = token_logp(rows, t, head_row)
        return float(-lp.sum() / len(t))
    seq = [0] + t
    lp = token_logp(rows, seq)[1:]
    return float(-lp.sum() / len(seq))


def choose(choices, head_row, rows_head, rows_init=None, calibrate: bool = False) -> list[float]:
    """run.rs:936-983: the `ppl` list a Choose request returns (lower is better; empty choices stay +inf).
    rows_head[i]: rows of choices[i] fed from the state after the prompt, whose last row is head_row;
    rows_init[i] (calibrate only): rows of [0] + choices[i] fed from the initial state.
    calibrate: ppl[i] = perplexity(with head) - perplexity(without head, from the initial state)."""
    ppl = [float("inf")] * len(choices)
    if calibrate:
        for i, c in enumerate(choices):
            if len(c):
                ppl[i] = -perplexity(rows_init[i], c)
    for i, c in enumerate(choices):
        if len(c):
            p = perplexity(rows_head[i], c, head_row)
            ppl[i] = ppl[i] + p if calibrate else p
    return ppl
