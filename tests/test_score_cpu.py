"""oracle/score_numpy.py (the float64 restatement of the reference's perplexity() and Choose, run.rs:699-755, 936-983) on
hand-made logits rows, where every expected number is written out by hand.  No GPU."""
import math

import numpy as np
import pytest

from oracle import score_numpy as SC

V = 4


def row(p):
    """logits whose softmax is the probability vector p"""
    return np.log(np.asarray(p, np.float64))


# the row emitted after each fed token: softmax(rows[j]) is the distribution of the token after tokens[j]
P0 = [0.1, 0.2, 0.3, 0.4]
P1 = [0.25, 0.25, 0.25, 0.25]
P2 = [0.7, 0.1, 0.1, 0.1]
HEAD = [0.5, 0.125, 0.125, 0.25]


def test_token_logp_reads_the_row_before_each_token():
    lp = SC.token_logp([row(P0), row(P1), row(P2)], [3, 1, 0])
    assert math.isnan(lp[0])
    np.testing.assert_allclose(lp[1:], [math.log(0.2), math.log(0.25)], rtol=1e-14)
    lp = SC.token_logp([row(P0), row(P1), row(P2)], [3, 1, 0], head_row=row(HEAD))
    np.testing.assert_allclose(lp, [math.log(0.25), math.log(0.2), math.log(0.25)], rtol=1e-14)


def test_head_perplexity_divides_by_the_choice_length():
    # Some(head): p = [head[x0], P0[x1], P1[x2]], mean over len(choice) = 3
    got = SC.perplexity([row(P0), row(P1), row(P2)], [3, 1, 0], head_row=row(HEAD))
    want = -(math.log(0.25) + math.log(0.2) + math.log(0.25)) / 3
    assert got == pytest.approx(want, rel=1e-14)


def test_no_head_perplexity_prepends_token_0_and_divides_by_one_more():
    # None: the fed sequence is [0, 3, 1]; rows are those of 0, 3, 1; p = [P0[3], P1[1]], of length len(choice) = 2,
    # divided by len([0] + choice) = 3 -- the reference's quirk
    got = SC.perplexity([row(P0), row(P1), row(P2)], [3, 1])
    want = -(math.log(0.4) + math.log(0.25)) / 3
    assert got == pytest.approx(want, rel=1e-14)
    assert got != pytest.approx(-(math.log(0.4) + math.log(0.25)) / 2)


def test_choose_without_and_with_calibrate():
    choices = [[3, 1], [], [0]]
    rows_head = [[row(P0), row(P1)], [], [row(P2)]]
    rows_init = [[row(P1), row(P0), row(P2)], [], [row(P2), row(P0)]]
    plain = SC.choose(choices, row(HEAD), rows_head)
    want0 = -(math.log(0.25) + math.log(0.2)) / 2
    want2 = -math.log(0.5) / 1
    assert plain[0] == pytest.approx(want0, rel=1e-14)
    assert plain[1] == math.inf                                 # empty choices are never scored
    assert plain[2] == pytest.approx(want2, rel=1e-14)
    cal = SC.choose(choices, row(HEAD), rows_head, rows_init, calibrate=True)
    none0 = -(math.log(0.25) + math.log(0.2)) / 3               # [0, 3, 1] from the initial state
    none2 = -math.log(0.7) / 2                                  # [0, 0]
    assert cal[0] == pytest.approx(want0 - none0, rel=1e-13)
    assert cal[1] == math.inf
    assert cal[2] == pytest.approx(want2 - none2, rel=1e-13)


def test_a_max_shifted_row_gives_the_same_result():
    rng = np.random.default_rng(0)
    rows = [rng.normal(0, 3, 512) for _ in range(6)]
    toks = rng.integers(0, 512, 6).tolist()
    head = rng.normal(0, 3, 512)
    base = SC.token_logp(rows, toks, head)
    shifted = SC.token_logp([r + 1e4 for r in rows], toks, head - 7e3)    # exp(x) alone would overflow here
    np.testing.assert_allclose(shifted, base, rtol=0, atol=1e-9)
    assert SC.perplexity([r + 1e4 for r in rows], toks) == pytest.approx(SC.perplexity(rows, toks), abs=1e-10)
    # and the log-probabilities are those of a normalised distribution
    assert np.exp(SC.log_softmax(rows[0])).sum() == pytest.approx(1.0, abs=1e-12)
