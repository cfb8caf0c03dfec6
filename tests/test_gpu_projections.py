"""Every projection launch plan against a float64 product.

Each case builds a small synthetic model and runs single-step `infer_raw` calls (one internal step each).  After a step the
engine's buffers still hold what the last layer's projections read and wrote (b200rwkv_debug_read): the WKV kernel only
reads its inputs, LN2 rewrites a_x0 / a_x1 (v5 / v6) and a_x0 (v7), so those serve as inputs of the channel mix only.  Each
output is compared with the float64 product of the f16 input the engine used and the weight from the `.st` file (Int8 / NF4
layers through oracle/quant_numpy's engine contract), with the fused epilogue restated in float64, under the bound of
oracle/projection_numpy.py.  The launch plans each case ran (b200rwkv_debug_plan) are recorded; the last test asserts that,
over all cases, every kind of cut the planner can make was taken (so a policy change cannot move coverage away silently)."""
import dataclasses

import numpy as np
import pytest

from ai00_server_b200 import capi, runtime, synth
from oracle import projection_numpy as P
from oracle import quant_numpy as Q
from oracle import rwkv_numpy as O

pytestmark = pytest.mark.gpu

# steps: name -> (slots, tokens per slot, option); every one is a single internal step of the engine
STEPS = {
    "decode16": (16, 1, capi.OPTION_LAST),     # batch-16 decode: MT 1
    "full20": (1, 20, capi.OPTION_FULL),       # MT 2, head at 2 row tiles
    "full40": (1, 40, capi.OPTION_FULL),       # MT 4: grid_wide
    "last40": (1, 40, capi.OPTION_LAST),       # MT 4 with a 1-row head (head operand rows != token rows)
    "full128": (1, 128, capi.OPTION_FULL),     # MT 8
}


def mt_of(rows):
    return 1 if rows <= 16 else (2 if rows <= 32 else (4 if rows <= 64 else 8))


W3B = dict(L=1, C=2560, F=8960, Dm=32, Dd=64, V=384)            # 3B width: R/K/V/G and ffn K+R cut across CTAs
CASES = {
    "A_v6_3b": (dataclasses.replace(synth.PRESETS["v6-3b"], **W3B), {}, ["decode16", "full20", "full40", "last40", "full128"]),
    "B_v6_3b_split": (dataclasses.replace(synth.PRESETS["v6-3b"], **W3B), dict(exact=True), ["decode16"]),
    "C_v6_3b_int8": (dataclasses.replace(synth.PRESETS["v6-3b"], **W3B), dict(quant=1, quant_type="Int8"), ["decode16", "full20", "full40"]),
    "C_v6_3b_nf4": (dataclasses.replace(synth.PRESETS["v6-3b"], **W3B), dict(quant=1, quant_type="NF4"), ["decode16", "full20", "full40"]),
    "D_v7_2b9": (dataclasses.replace(synth.PRESETS["v7-2b9"], L=2, V=256), {}, ["decode16", "full20", "full40", "full128"]),
    "E_v6_7b": (dataclasses.replace(synth.PRESETS["v6-7b"], L=1, V=256), {}, ["decode16"]),
    "F_small6_dd192": (dataclasses.replace(synth.PRESETS["small6"], L=1, Dd=192), {}, ["decode16", "full20"]),
    "F_small6_c320": (dataclasses.replace(synth.PRESETS["small6"], L=1, C=320, F=1152), {}, ["decode16", "full20"]),
    "G_v5_small5": (dataclasses.replace(synth.PRESETS["small5"], L=2), {}, ["decode16", "full40"]),
}
QTYPES = {"Int8": Q.QUANT_INT8, "NF4": Q.QUANT_NF4}

PLANS = {}          # case -> [(step, mt, layer, plan)] of the steps the case ran


class Weights:
    """The weights the engine multiplies with, as float64, converted once per tensor."""

    def __init__(self, st, quant=0, quant_type=None):
        w = O.parse_st(st)
        if quant:
            w = Q.quantize_model(w, quant, QTYPES[quant_type])
        self.raw, self.cache = w, {}

    def __call__(self, name):
        if name not in self.cache:
            self.cache[name] = np.asarray(self.raw[name], np.float64)
        return self.cache[name]

    def vec(self, name):
        return self(name).reshape(-1)


def plans_of(m, L, step):
    n, cnt, opt = STEPS[step]
    mt, mtr = mt_of(n * cnt), mt_of(n * cnt if opt == capi.OPTION_FULL else n)
    out = [(step, mt, l, p) for l in range(L) for p in m.debug_plan(l, mt)]
    return out + [(step, mtr, -1, p) for p in m.debug_plan(-1, mtr)]


def describe(plans):
    lines = []
    for step, mt, layer, p in plans:
        cs = [c for _, c, _ in P.contributors(p)]
        segs = ",".join(f"{P.ACT_NAMES[s['act']]}/{P.OUT_NAMES[s['out_mode']]}" for s in p["segs"])
        lines.append(f"  {step:8s} MT {mt} {'head' if layer < 0 else f'L{layer}'}: grid {p['grid_run']:3d} "
                     f"({'forced' if p['forced'] else 'wide' if mt >= 4 else 'sk'}) blocks {p['total_blocks']:4d} "
                     f"q{p['qtype']} contributors {min(cs)}..{max(cs)} [{segs}]")
    return "\n".join(lines)


def compare_step(m, wt, shape, split, logits, lerp_run, decay_run):
    """All checkable projections of the last layer of the step that just ran: [(name, Check)]."""
    rd = m.debug_read
    l = shape.L - 1
    a, f = f"blocks.{l}.att.", f"blocks.{l}.ffn."
    res = []

    def f32(name, x, wname, bias=None, act=P.ACT_NONE):
        res.append((name, P.check_f32(rd(name), x, wt(wname), bias, act)))

    def a16(name, x, w, bias=None, act=P.ACT_NONE, lerp=None, cols=None):
        got = rd(name)[:, :cols] if cols else rd(name)
        res.append((name, P.check_a16(got, x, w, bias, act, lerp, split)))

    if shape.version in (5, 6):
        f32("r", rd("a_x3"), a + "receptance.weight")
        f32("v", rd("a_x2"), a + "value.weight")
        f32("g", rd("a_x4"), a + "gate.weight", act=P.ACT_SILU)
        f32("rr", rd("a_x1"), f + "receptance.weight", act=P.ACT_SIGMOID)
        if shape.version == 6 and lerp_run:
            # ddlerp stage 1 (five tanh groups of Dm) and stage 2 into a_x2..4 (a_x0 / a_x1 are LN2's by now)
            Dm, x5 = shape.Dm, rd("a_x5")
            w1 = wt(a + "time_mix_w1")
            for i in range(5):
                a16(f"a_lora0_{i}", x5, w1[i * Dm:(i + 1) * Dm], act=P.ACT_TANH, cols=Dm)
            xx, sx = rd("xx1"), rd("sx1")
            for i, nm in ((2, "v"), (3, "r"), (4, "g")):
                a16(f"a_x{i}", rd(f"a_lora0_{i}")[:, :Dm], wt(a + "time_mix_w2")[i], lerp=(xx, sx, wt.vec(a + f"time_mix_{nm}")))
        if shape.version == 6 and decay_run:
            f32("w", rd("a_lora1_0")[:, :shape.Dd], a + "time_decay_w2", bias=wt.vec(a + "time_decay"), act=P.ACT_EXPNEGEXP)
    else:
        f32("k", rd("a_x2"), a + "key.weight")
        f32("v", rd("a_x3"), a + "value.weight")
        a16("a_lora0_0", rd("a_x1"), wt(a + "w1"), act=P.ACT_TANH, cols=shape.Dd)
        a16("a_lora1_0", rd("a_x4"), wt(a + "a1"), cols=shape.Da)
        if l > 0:
            a16("a_lora2_0", rd("a_x3"), wt(a + "v1"), cols=shape.Dv)
        a16("a_lora3_0", rd("a_x5"), wt(a + "g1"), act=P.ACT_SIGMOID, cols=shape.Dg)
        f32("w", rd("a_lora0_0")[:, :shape.Dd], a + "w2", bias=wt.vec(a + "w0"), act=P.ACT_V7DECAY)
        f32("a", rd("a_lora1_0")[:, :shape.Da], a + "a2", bias=wt.vec(a + "a0"), act=P.ACT_SIGMOID)
        if l > 0:
            f32("nu", rd("a_lora2_0")[:, :shape.Dv], a + "v2", bias=wt.vec(a + "v0"), act=P.ACT_SIGMOID)
        f32("g", rd("a_lora3_0")[:, :shape.Dg], a + "g2")
    f32("part_att", rd("a_out"), a + "output.weight")
    a16("a_kk", rd("a_x0"), wt(f + "key.weight"), act=P.ACT_RELU2)
    f32("part_ffn", rd("a_kk"), f + "value.weight")
    head_in = rd("a_head")
    assert head_in.shape[0] == logits.shape[0], (head_in.shape, logits.shape)
    res.append(("logits", P.check_f32(logits, head_in, wt("head.weight"))))
    return res


def run_case(name):
    shape, kw, steps = CASES[name]
    st = synth.make_st(shape, 0)
    wt = Weights(st, kw.get("quant", 0), kw.get("quant_type"))
    m = runtime.Model(st, max_batch=16, token_chunk_size=128, **kw)
    rng = np.random.default_rng(sum(map(ord, name)))
    failures, plans = [], []
    try:
        for step in steps:
            n, cnt, opt = STEPS[step]
            toks = rng.integers(0, shape.V, size=n * cnt).tolist()
            rows = m.infer_raw(list(range(n)), [cnt] * n, toks, [opt] * n)
            logits = np.concatenate(rows, 0)
            sp = plans_of(m, shape.L, step)
            plans += sp
            last = [p for _, _, layer, p in sp if layer == shape.L - 1]
            acts = {s["act"] for p in last for s in p["segs"]}
            lerp_run = any(s["out_mode"] == P.OUT_LERP_A16 for p in last for s in p["segs"])
            res = compare_step(m, wt, shape, kw.get("exact", False), logits, lerp_run, P.ACT_EXPNEGEXP in acts)
            f32w = max(c.worst for nm, c in res if not nm.startswith("a_"))
            a16w = max(c.worst for nm, c in res if nm.startswith("a_"))
            print(f"{name} {step}: worst f32 output {f32w:.3g} x sqrt(K) 2^-24 |x|.|w| (bound {P.TAU:g}); worst A16 output "
                  + (f"{a16w:.3g} x the same unit (hi + lo)" if kw.get("exact") else f"{a16w:.3g} f16 ulp"))
            failures += [f"{step} {nm}: {c}" for nm, c in res if not c.ok]
    finally:
        m.close()
    PLANS[name] = plans
    print(describe(plans))
    return failures


@pytest.mark.parametrize("case", list(CASES))
def test_projection_outputs_match_a_float64_product(case):
    failures = run_case(case)
    assert not failures, "\n".join(failures)


def coverage_gaps(plans_by_case):
    """Kinds of launch the planner makes that no case ran."""
    have = set()
    for plans in plans_by_case.values():
        for step, mt, layer, p in plans:
            tiles = P.contributors(p)
            cmax = max(c for _, c, _ in tiles)
            for s in p["segs"]:
                have.add(("act", s["act"]))
                have.add(("out", s["out_mode"]))
            if p["forced"]:
                have.add("forced split-K grid")
            if cmax > 1:
                if p["qtype"] == 0 and mt in (1, 2):
                    have.add(f"f16 cut tiles at MT {mt}")
                if mt >= 4:
                    have.add("cut tiles under grid_wide")
                if p["qtype"]:
                    have.add(f"quantised cut tiles q{p['qtype']}")
                if any(c > 1 and span for _, c, span in tiles):
                    have.add("cut tiles with a CTA across a segment boundary")
            if cmax > 4 and mt == 1:
                have.add("more than 4 contributors at MT 1")
    want = {("act", a) for a in range(7)} | {("out", o) for o in range(3)} | {
        "forced split-K grid", "f16 cut tiles at MT 1", "f16 cut tiles at MT 2", "cut tiles under grid_wide",
        "quantised cut tiles q1", "quantised cut tiles q2", "cut tiles with a CTA across a segment boundary",
        "more than 4 contributors at MT 1"}
    return sorted(map(str, want - have))


def all_plans():
    """Plans of every case: recorded by the case tests, or (cases deselected here) queried from a freshly built engine."""
    for name, (shape, kw, steps) in CASES.items():
        if name not in PLANS:
            m = runtime.Model(synth.make_st(shape, 0), max_batch=16, token_chunk_size=128, **kw)
            try:
                PLANS[name] = [x for step in steps for x in plans_of(m, shape.L, step)]
            finally:
                m.close()
    return PLANS


def test_the_cases_reach_every_launch_kind():
    plans = all_plans()
    assert not coverage_gaps(plans), coverage_gaps(plans)
    # and the check is not vacuous: without the quantised cases their cut tiles are missing
    gaps = coverage_gaps({k: v for k, v in plans.items() if not k.startswith("C_")})
    assert "quantised cut tiles q1" in gaps and "quantised cut tiles q2" in gaps, gaps
