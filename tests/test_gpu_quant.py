"""GPU parity tests for the weight-only quantised formats (`quant` / `quant_type` of the reload request, reference
crates/ai00-core/src/lib.rs:211-215, 465, 694-704): the load-time quantisers against oracle/quant_numpy.py bit for bit, and the
engine with quantised layers against the forward-pass oracle running on the SAME dequantised weights (1e-3 relative, argmax
exact).  Every engine call goes through the C ABI."""
import numpy as np
import pytest

from ai00_server_b200 import capi, runtime, synth
from oracle import quant_numpy as Q
from oracle import rwkv_numpy as O

pytestmark = pytest.mark.gpu

REL_TOL = 1e-3


def rel_err(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _matrix(n, k, seed):
    rng = np.random.default_rng(seed)
    w = (rng.standard_normal((n, k)) * 0.05).astype(np.float16)
    w[3, :128] = np.float16(0.125)                 # a constant block: max == min
    w[5, :] = 0                                    # an all-zero row: absmax == 0
    w[7, 128:256] = np.linspace(-1, 1, 128).astype(np.float16)
    w[9, 0] = np.float16(60000.0)                  # a block dominated by one outlier
    w[11, :64] = (Q.NF4_LEVELS[:, None].repeat(4, 1).reshape(-1) * 0.5).astype(np.float16)   # exactly on NF4 levels
    mids = (Q.NF4_LEVELS[:-1] + Q.NF4_LEVELS[1:]) / 2                                        # and near the decision boundaries
    w[12, :15] = mids.astype(np.float16)
    w[12, 15] = 1.0
    return w


@pytest.mark.parametrize("shape", [(200, 384), (128, 128), (1, 256)])
def test_int8_quantiser_is_bit_exact(shape):
    w = _matrix(max(shape[0], 16), max(shape[1], 256), 1)[:shape[0], :shape[1]].copy()
    codes, mn, scale = capi.op_quantize(capi.QUANT_INT8, w)
    q, mn_o, mx_o = Q.quant_int8(w)
    assert (mn.view(np.uint16) == mn_o.view(np.uint16)).all()
    assert (scale.view(np.uint16) == Q.int8_scale(mn_o, mx_o).view(np.uint16)).all()
    assert (codes == q).all()


@pytest.mark.parametrize("shape", [(200, 384), (128, 128), (1, 256)])
def test_nf4_quantiser_is_bit_exact(shape):
    w = _matrix(max(shape[0], 16), max(shape[1], 256), 2)[:shape[0], :shape[1]].copy()
    codes, am = capi.op_quantize(capi.QUANT_NF4, w)
    q, am_o = Q.quant_nf4(w)
    assert (am.view(np.uint16) == am_o.view(np.uint16)).all()
    assert (codes == q).all()


@pytest.fixture(scope="module")
def qmodels():
    cache = {}

    def get(preset, qtype, layers=None, max_batch=4, chunk=128):
        key = (preset, qtype, layers, max_batch, chunk)
        if key not in cache:
            st = synth.make_st(synth.PRESETS[preset], 0)
            w = O.parse_st(st)
            L = synth.PRESETS[preset].L if layers is None else layers
            m = runtime.Model(st, max_batch=max_batch, token_chunk_size=chunk, quant=L, quant_type=qtype)
            orc = O.Oracle(Q.quantize_model(w, L, qtype), "f16")
            cache[key] = (m, orc, w)
        return cache[key]

    yield get
    for m, _, _ in cache.values():
        m.close()


def feed(model, slot, tokens, full=False):
    rows = model.infer_raw([slot], [len(tokens)], list(tokens), [capi.OPTION_FULL if full else capi.OPTION_LAST])
    return rows[0].copy()


@pytest.mark.parametrize("qtype", [capi.QUANT_INT8, capi.QUANT_NF4])
@pytest.mark.parametrize("preset", ["tiny6", "tiny5", "tiny7", "small6"])
def test_quantised_logits_match_oracle(qmodels, preset, qtype):
    m, orc, w = qmodels(preset, qtype)
    toks = [1, 5, 9, 33, 2, 7, 300, 41, 41, 8, 0, 17]
    m.state.load(m.state.init(), 0)
    got = np.stack([feed(m, 0, [t])[0] for t in toks])                    # decode-shaped steps (one token tile)
    want, want_state = orc.run(toks, orc.state_init(), full=True)
    assert rel_err(got, want) <= REL_TOL
    assert (got.argmax(1) == want.argmax(1)).all()
    assert rel_err(m.state.back(0), want_state) <= REL_TOL
    # the format is really in effect: the f16 model answers differently
    plain, _ = O.Oracle(w, "f16").run(toks, orc.state_init(), full=True)
    assert rel_err(want, plain) > (1e-4 if qtype == capi.QUANT_INT8 else 1e-3)
    # and the reference's f32 dequantisation (no rounding of the expanded weight to f16) stays within the same bound
    L = len([k for k in w if k.endswith(".ln1.weight")])
    want32, _ = O.Oracle(Q.quantize_model(w, L, qtype, contract="f32"), "f32").run(toks, orc.state_init(), full=True)
    assert rel_err(got, want32) <= 3 * REL_TOL
    assert (got.argmax(1) == want32.argmax(1)).all()


@pytest.mark.parametrize("qtype", [capi.QUANT_INT8, capi.QUANT_NF4])
@pytest.mark.parametrize("preset", ["tiny6", "tiny7"])
def test_quantised_prefill_shapes(qmodels, preset, qtype):
    """Steps of 2, 4 and 8 token tiles run the quantised projections with the wider token operand."""
    m, orc, _ = qmodels(preset, qtype)
    rng = np.random.default_rng(11)
    for n, slot in ((20, 0), (50, 1), (128, 2), (300, 3)):
        toks = rng.integers(1, 500, size=n).tolist()
        m.state.load(m.state.init(), slot)
        got = feed(m, slot, toks)
        want, want_state = orc.run(toks, orc.state_init())
        assert rel_err(got, want) <= REL_TOL, n
        assert got.argmax() == want.argmax()
        assert rel_err(m.state.back(slot), want_state) <= REL_TOL, n


@pytest.mark.parametrize("qtype", [capi.QUANT_INT8, capi.QUANT_NF4])
def test_only_the_first_layers_are_quantised(qmodels, qtype):
    """`quant = 2` of a 4-layer model (lib.rs:465: `(0..quant).map(|layer| (layer, quant_type))`), batch of ragged slots."""
    m, orc, _ = qmodels("small6", qtype, layers=2)
    seqs = [[3, 4, 5, 6, 7], [100, 200], [9] * 17, [1]]
    for s in range(4):
        m.state.load(m.state.init(), s)
    rows = m.infer_raw([0, 1, 2, 3], [len(x) for x in seqs], [t for x in seqs for t in x], [capi.OPTION_LAST] * 4)
    for s, x in enumerate(seqs):
        want, _ = orc.run(x, orc.state_init())
        assert rel_err(rows[s][0], want[0]) <= REL_TOL
        assert rows[s][0].argmax() == want[0].argmax()


def test_unsupported_quant_requests_fail_loudly():
    st = synth.make_st(synth.PRESETS["tiny6"], 0)
    with pytest.raises(capi.B200Error) as e:
        runtime.Model(st, max_batch=2, token_chunk_size=32, quant=2, quant_type="SF4")
    assert e.value.code == capi.ERR_UNSUPPORTED
    with pytest.raises(capi.B200Error) as e:
        runtime.Model(st, max_batch=2, token_chunk_size=32, quant=2, quant_type="Int8", exact=True)
    assert e.value.code == capi.ERR_UNSUPPORTED
    # quant = 0 or quant_type = None is the plain f16 model
    m = runtime.Model(st, max_batch=2, token_chunk_size=32, quant=0, quant_type="NF4")
    m.close()


@pytest.mark.parametrize("qtype", [capi.QUANT_INT8, capi.QUANT_NF4])
def test_quantised_projections_at_the_7b_layer_shape(qtype):
    """One layer with the 7B dimensions (C = 4096, F = 14336, LoRA ranks 64 / 128): the tile counts and split-K slices of the
    BASELINE shape, batch 16, against the oracle on the dequantised weights.  Every quantised launch of this shape runs whole
    tiles per CTA (only the f16 head is cut); the quantised fix-up of cut tiles runs at the 3B width in
    tests/test_gpu_projections.py."""
    import dataclasses
    shp = dataclasses.replace(synth.PRESETS["v6-7b"], L=1, V=4096)
    st = synth.make_st(shp, 0)
    w = O.parse_st(st)
    orc = O.Oracle(Q.quantize_model(w, 1, qtype), "f16")
    m = runtime.Model(st, max_batch=16, token_chunk_size=64, quant=1, quant_type=qtype)
    try:
        rng = np.random.default_rng(5)
        toks = rng.integers(1, 4000, size=(16, 3))
        slots = list(range(16))
        for s in slots:
            m.state.load(m.state.init(), s)
        for j in range(3):
            rows = m.infer_raw(slots, [1] * 16, toks[:, j].tolist(), [capi.OPTION_LAST] * 16)
        for s in (0, 7, 15):
            want, want_state = orc.run(toks[s].tolist(), orc.state_init())
            assert rel_err(rows[s][0], want[0]) <= REL_TOL
            assert rows[s][0].argmax() == want[0].argmax()
            assert rel_err(m.state.back(s), want_state) <= REL_TOL
        # a 40-token prompt: four token tiles, whole output tiles per CTA
        ptoks = rng.integers(1, 4000, size=40).tolist()
        m.state.load(m.state.init(), 1)
        got = m.infer_raw([1], [40], ptoks, [capi.OPTION_LAST])[0][0]
        want, _ = orc.run(ptoks, orc.state_init())
        assert rel_err(got, want[0]) <= REL_TOL
        assert got.argmax() == want[0].argmax()
    finally:
        m.close()
