"""CPU oracle for ONE projection launch: a float64 product of the f16 operands the engine used, with the fused epilogues of
csrc/gemm.cuh restated (bias, the six activations of common.cuh `apply_act`, f16 saturation of `f2h_sat`, the v6 ddlerp
`xx + sx * (mu + y)`), and a comparator whose bound follows from f32 accumulation.

TEST INFRASTRUCTURE ONLY (tests/test_gpu_projections.py, tests/test_projection_compare_cpu.py).

Bound.  Products of two f16 numbers are exact in f32, so an f32 accumulation of K of them differs from the float64 sum by
rounding alone; for any summation order that is statistically ~ sqrt(K) * 2^-24 * sum |x_k| |w_k|.  A projection output y is
accepted when

    |y - y64| <= TAU * sqrt(K) * 2^-24 * (|x| . |w|)          (TAU = 16)

elementwise.  Behind a bias and an activation the interval y64 +- that bound (+ the f32 rounding of the bias add) is pushed
through the activation (its end points: every activation here is monotone or convex near its extremum), plus a few f32 ulps
for evaluating the activation itself.  An f16 (A16) output must lie between the f16 roundings of that interval's ends: it is
the correctly rounded value, or the neighbour only where the exact value sits within the bound of a rounding midpoint.
Dropping one 8-term k chunk, a 128-wide k block, a contributor's partial counted twice or two swapped token rows all exceed
this bound by far (tests/test_projection_compare_cpu.py), while any f32 summation order stays orders of magnitude inside it.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

TAU = 16.0
U32 = 2.0 ** -24
F16_MAX = 65504.0

# csrc/common.cuh `enum Act`, csrc/gemm.cuh `enum OutMode`
ACT_NONE, ACT_TANH, ACT_SIGMOID, ACT_SILU, ACT_RELU2, ACT_EXPNEGEXP, ACT_V7DECAY = range(7)
ACT_NAMES = ("none", "tanh", "sigmoid", "silu", "relu2", "exp(-exp)", "v7decay")
OUT_F32, OUT_A16, OUT_LERP_A16 = range(3)
OUT_NAMES = ("f32", "a16", "lerp_a16")


def _sig(z):
    return 1.0 / (1.0 + np.exp(-z))


def act64(z: np.ndarray, act: int) -> np.ndarray:
    z = np.asarray(z, np.float64)
    with np.errstate(over="ignore"):
        if act == ACT_TANH:
            return np.tanh(z)
        if act == ACT_SIGMOID:
            return _sig(z)
        if act == ACT_SILU:
            return z * _sig(z)
        if act == ACT_RELU2:
            return np.maximum(z, 0.0) ** 2
        if act == ACT_EXPNEGEXP:
            return np.exp(-np.exp(z))
        if act == ACT_V7DECAY:
            return np.exp(-0.606531 * _sig(z))
    return z


def _eval_tol(z: np.ndarray, a: np.ndarray, act: int) -> np.ndarray:
    """Error of evaluating the activation in f32 (CUDA expf / tanhf: <= 2 ulp each): 16 ulps of the result; exp(-exp(z))
    also carries the relative error of the inner exp times exp(z)."""
    if act == ACT_NONE:
        return np.zeros_like(a)
    t = np.abs(a)
    if act == ACT_EXPNEGEXP:
        with np.errstate(over="ignore"):
            t = t * (1.0 + np.exp(z))
    return TAU * U32 * t


def product(x: np.ndarray, w: np.ndarray):
    """y64 = x . w^T and s = |x| . |w|^T in float64.  x [T, K], w [N, K] (both f16-valued)."""
    x = np.asarray(x, np.float64)
    w = np.asarray(w, np.float64)
    return x @ w.T, np.abs(x) @ np.abs(w).T


@dataclass
class Check:
    ok: bool
    worst: float          # f32 outputs: max |got - want| / (bound / TAU), the error in units of sqrt(K) 2^-24 |x|.|w|;
                          # f16 outputs: f16 ulps from the correctly rounded value (a failing element comes first)
    where: tuple          # (token row, output column) of the worst element
    got: float
    want: float

    def __str__(self):
        return f"worst {self.worst:.3g} at {self.where} (got {self.got!r}, want {self.want!r})"


def _interval(x, w, bias, act, K):
    y64, s = product(x, w)
    z = y64 + (0.0 if bias is None else np.asarray(bias, np.float64)[None, :])
    e = TAU * np.sqrt(K) * U32 * s
    if bias is not None:
        e = e + U32 * np.abs(z)                       # the f32 bias add
    a = act64(z, act)
    with np.errstate(over="ignore", invalid="ignore"):
        d = np.maximum(np.abs(act64(z + e, act) - a), np.abs(act64(z - e, act) - a))
    return a, np.nan_to_num(d, posinf=np.inf) + _eval_tol(z, a, act)


def _result(err, bound, got, want) -> Check:
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(err == 0, 0.0, err / np.maximum(bound / TAU, 1e-300))
    i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    return Check(bool(np.all(err <= bound)), float(ratio[i]), tuple(int(v) for v in i), float(got[i]), float(want[i]))


def check_f32(got, x, w, bias=None, act=ACT_NONE) -> Check:
    """An f32 output [T, N] of the projection x [T, K] . w [N, K]^T (+ bias [N], then `act`)."""
    got = np.asarray(got, np.float64)
    K = np.asarray(x).shape[1]
    want, bound = _interval(x, w, bias, act, K)
    assert got.shape == want.shape, (got.shape, want.shape)
    return _result(np.abs(got - want), bound, got, want)


def f16_sat(v: np.ndarray) -> np.ndarray:
    return np.clip(np.asarray(v, np.float64), -F16_MAX, F16_MAX).astype(np.float16).astype(np.float64)


def check_a16(got, x, w, bias=None, act=ACT_NONE, lerp=None, split=False) -> Check:
    """An A16 output [T, N] (f16 operand of the next projection).  lerp = (xx [T, N], sx [T, N], mu [N]): the v6 ddlerp
    epilogue f16(xx + sx * (mu + act(y))).  split: a split-operand step, `got` is hi + lo (an f32 value, not rounded to f16)."""
    got = np.asarray(got, np.float64)
    K = np.asarray(x).shape[1]
    want, bound = _interval(x, w, bias, act, K)
    if lerp is not None:
        xx, sx, mu = (np.asarray(v, np.float64) for v in lerp)
        inner = mu[None, :] + want
        want = xx + sx * inner
        bound = np.abs(sx) * bound + 4 * U32 * (np.abs(xx) + np.abs(sx) * (np.abs(mu[None, :]) + np.abs(inner)))
    assert got.shape == want.shape, (got.shape, want.shape)
    err = np.abs(got - want)
    if split:
        return _result(err, bound + 2.0 ** -21 * np.abs(want), got, want)
    lo, hi = f16_sat(want - bound), f16_sat(want + bound)
    ok = (got >= lo) & (got <= hi)
    # reported: f16 ulps between the output and the correctly rounded exact value (0, or 1 beside a rounding midpoint)
    r = f16_sat(want)
    ulp = np.abs(np.spacing(r.astype(np.float16)).astype(np.float64))
    ulps = np.abs(got - r) / ulp
    i = np.unravel_index(int(np.argmax(np.where(ok, ulps, np.inf))), ulps.shape)
    return Check(bool(np.all(ok)), float(ulps[i]), tuple(int(v) for v in i), float(got[i]), float(want[i]))


def contributors(plan: dict) -> list[tuple[int, int, int]]:
    """Per output tile of one launch (b200rwkv_debug_plan record): (segment, contributors, CTAs whose block range also covers
    another segment's blocks).  The c_first / c_last formulas of gemm_epilogue_role, restated."""
    G, TB = plan["grid_run"], plan["total_blocks"]
    out, blk = [], 0
    bounds = []
    for s in plan["segs"]:
        bounds.append((blk, blk + s["tiles"] * s["KB"]))
        blk += s["tiles"] * s["KB"]
    assert blk == TB, (blk, TB)
    cta_range = lambda c: (c * TB // G, (c + 1) * TB // G)
    for si, s in enumerate(plan["segs"]):
        for t in range(s["tiles"]):
            tb0 = bounds[si][0] + t * s["KB"]
            c_first = ((tb0 + 1) * G - 1) // TB
            c_last = ((tb0 + s["KB"]) * G - 1) // TB
            span = 0
            for c in range(c_first, c_last + 1):
                b0, b1 = cta_range(c)
                span += int(b0 < bounds[si][0] or b1 > bounds[si][1])
            out.append((si, c_last - c_first + 1, span))
    return out
