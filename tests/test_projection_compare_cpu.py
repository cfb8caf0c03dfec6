"""The projection comparator (oracle/projection_numpy.py) is tight enough to catch what a broken stream-K fix-up or tile walk
would produce, and loose enough for any f32 summation order.  Synthetic f16 operands at the two reduction depths of the
flagship models (K = 2560: 3B width; K = 14336: the 7B channel-mix value projection); no GPU."""
import numpy as np
import pytest

from oracle import projection_numpy as P

T, N, BK = 16, 256, 128          # one decode token tile, two 128-row output tiles, 128-wide k blocks


def operands(K, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((T, K)).astype(np.float16)                          # LayerNorm output scale
    w = rng.uniform(-np.sqrt(3 / K), np.sqrt(3 / K), (N, K)).astype(np.float16)  # synth.py's projection init
    return x, w


def f32_sum(x, w, order, chunk=16):
    """f32 accumulation of the exact f16 x f16 products: 16-term chunks summed in f32, chunks added in `order`."""
    prod = (x.astype(np.float32)[:, None, :] * w.astype(np.float32)[None, :, :])       # exact
    parts = prod.reshape(T, N, -1, chunk)
    acc = np.zeros((T, N), np.float32)
    for c in order:
        s = np.zeros((T, N), np.float32)
        for j in range(chunk):
            s = (s + parts[:, :, c, j]).astype(np.float32)
        acc = (acc + s).astype(np.float32)
    return acc


def partial(x, w, k0, k1, rows):
    return (x[:, k0:k1].astype(np.float64) @ w[rows, k0:k1].astype(np.float64).T).astype(np.float32)


@pytest.fixture(scope="module", params=[2560, 14336])
def case(request):
    K = request.param
    x, w = operands(K, K)
    y = f32_sum(x, w, np.random.default_rng(1).permutation(K // 16))
    return K, x, w, y


def test_a_shuffled_f32_sum_passes(case):
    K, x, w, y = case
    c = P.check_f32(y, x, w)
    print(f"K={K}: shuffled f32 sum {c}")
    assert c.ok and c.worst < 0.1 * P.TAU, c


def test_a_dropped_k_block_is_rejected(case):
    K, x, w, y = case
    kb = (K // BK) // 2
    bad = y.copy()
    bad[:, 128:256] -= partial(x, w, kb * BK, (kb + 1) * BK, slice(128, 256))
    c = P.check_f32(bad, x, w)
    print(f"K={K}: dropped k block {c}")
    assert not c.ok


def test_a_dropped_k8_chunk_is_rejected(case):
    K, x, w, y = case
    bad = y.copy()
    bad[:, :128] -= partial(x, w, 8 * 37, 8 * 38, slice(0, 128))
    c = P.check_f32(bad, x, w)
    print(f"K={K}: dropped k8 chunk {c}")
    assert not c.ok


def test_a_partial_counted_twice_is_rejected(case):
    """A tile cut across three CTAs: the middle contributor's partial summed twice by the last arriver."""
    K, x, w, y = case
    kb = K // BK
    bad = y.copy()
    bad[:, 128:256] += partial(x, w, (kb // 3) * BK, (2 * kb // 3) * BK, slice(128, 256))
    c = P.check_f32(bad, x, w)
    print(f"K={K}: partial counted twice {c}")
    assert not c.ok


def test_swapped_token_rows_are_rejected(case):
    K, x, w, y = case
    bad = y.copy()
    bad[[6, 7]] = bad[[7, 6]]
    assert not P.check_f32(bad, x, w).ok


def test_a16_outputs_accept_the_rounded_value_and_reject_a_dropped_chunk(case):
    """Behind tanh into an f16 operand: the correctly rounded f16 of the f32 result passes, the same dropped k8 chunk fails."""
    K, x, w, y = case
    good = np.tanh(y.astype(np.float32)).astype(np.float16).astype(np.float32)
    c = P.check_a16(good, x, w, act=P.ACT_TANH)
    assert c.ok, c
    bad = (y - np.pad(partial(x, w, 8 * 37, 8 * 38, slice(0, 128)), ((0, 0), (0, 128)))).astype(np.float32)
    assert not P.check_a16(np.tanh(bad).astype(np.float16).astype(np.float32), x, w, act=P.ACT_TANH).ok


@pytest.mark.parametrize("act", range(7))
def test_every_activation_accepts_an_f32_evaluation(act):
    """Each activation evaluated in f32 on an f32 accumulation, with a bias, stays inside its propagated bound."""
    x, w = operands(512, act)
    y = f32_sum(x, w, range(512 // 16))
    b = np.random.default_rng(act).uniform(-3, 1, N).astype(np.float16).astype(np.float32)
    z = (y + b).astype(np.float32)
    f = np.float32
    sig = lambda v: f(1) / (f(1) + np.exp(-v))
    got = {P.ACT_NONE: z, P.ACT_TANH: np.tanh(z), P.ACT_SIGMOID: sig(z), P.ACT_SILU: z * sig(z),
           P.ACT_RELU2: np.maximum(z, f(0)) ** 2, P.ACT_EXPNEGEXP: np.exp(-np.exp(z)),
           P.ACT_V7DECAY: np.exp(f(-0.606531) * sig(z))}[act].astype(np.float32)
    c = P.check_f32(got, x, w, bias=b, act=act)
    assert c.ok, (P.ACT_NAMES[act], c)
    assert P.check_a16(got.astype(np.float16).astype(np.float32), x, w, bias=b, act=act).ok


def test_contributors_follow_the_cta_ranges():
    """gemm_epilogue_role's c_first / c_last, restated: 3 tiles of 20 k blocks on 15 CTAs -> 5 contributors each; two
    segments cut by 7 CTAs -> a CTA whose range spans the boundary."""
    plan = dict(grid_run=15, total_blocks=60, segs=[dict(KB=20, tiles=3, N=384, out_mode=0, act=0)])
    assert [c for _, c, _ in P.contributors(plan)] == [5, 5, 5]
    plan = dict(grid_run=7, total_blocks=40, segs=[dict(KB=20, tiles=1, N=128, out_mode=0, act=0)] * 2)
    tiles = P.contributors(plan)
    assert [c for _, c, _ in tiles] == [4, 4] and all(span > 0 for _, _, span in tiles)
    whole = dict(grid_run=2, total_blocks=40, segs=[dict(KB=20, tiles=1, N=128, out_mode=0, act=0)] * 2)
    assert P.contributors(whole) == [(0, 1, 0), (1, 1, 0)]
