"""GPU parity: the CUDA path (through the C ABI) against the oracle on identical instruction batches.

Criterion (north_star "1e-5 relative", read as SURVEY.md §8d prescribes): |gpu - ref| <= 1e-5 * max|ref| over
the block + 1e-7.  Integer/index/selection nodes (latch, counter, maxhold, rand, z, sdelay, compare ops) must
be bit-exact.  Every test renders from block 0, i.e. including the 20 ms root fade-in (960 samples @ 48 kHz).
"""
import math

import numpy as np
import pytest

from elementary_b200 import Runtime, el, graphs
from cases import plugin_nodes_batch, plugin_nodes_inputs
from helpers import block_peak_tolerance_check, oracle_render, reference_extra, sha16

pytestmark = pytest.mark.gpu

SR, BS = 48000.0, 512


def lcg_noise(n, seed, lo=-1.0, hi=1.0):
    s = (seed * 2654435761 + 1) & 0xFFFFFFFF
    out = np.empty(n, dtype=np.float32)
    for i in range(n):
        s = (s * 1664525 + 1013904223) & 0xFFFFFFFF
        out[i] = lo + (hi - lo) * ((s >> 8) / float(1 << 24))
    return out


def run_gpu(batch, n_voices, n_blocks, n_out=1, inputs=None, voice_batches=None, resources=None, **opts):
    rt = Runtime(SR, BS, n_voices, device=0, **opts)
    for name, data in (resources or {}).items():
        assert rt.add_shared_resource(name, data)
    assert rt.apply_instructions(batch) == 0, rt.last_error()
    if voice_batches is not None:
        for v, b in enumerate(voice_batches):
            if b:
                assert rt.apply_instructions(b, voices=(v, v + 1)) == 0, rt.last_error()
    got, mix = rt.render_voices(n_blocks, n_out, inputs)
    return got, mix, rt


def check(batch, n_voices=3, n_blocks=3, n_in=0, exact=False, resources=None, in_lo=-1.0, in_hi=1.0, n_out=1, **opts):
    inputs = None
    if n_in:
        inputs = np.stack([np.stack([lcg_noise(n_blocks * BS, 100 * v + c, in_lo, in_hi) for c in range(n_in)])
                           for v in range(n_voices)])
    got, mix, rt = run_gpu(batch, n_voices, n_blocks, n_out, inputs, resources=resources, **opts)
    ref = oracle_render(batch, n_blocks, n_out, SR, BS, inputs, voice_batches=[None] * n_voices, resources=resources)
    if exact:
        assert np.array_equal(got, ref), f"not bit exact: max diff {np.abs(got - ref).max()}"
    else:
        ok, worst, ex = block_peak_tolerance_check(got, ref, BS)
        assert ok, f"worst err/tol {worst:.3g}, bit-exact fraction {ex:.4f}"
    # mix bus == sum over voices (float64 reference sum, magnitude-scaled tolerance)
    want = ref.astype(np.float64).sum(axis=0)
    scale = np.abs(ref).astype(np.float64).sum(axis=0).max() + 1e-30
    assert np.abs(mix - want).max() <= 1e-6 * scale + 1e-7
    return got, ref


IN0, IN1, IN2 = el.in_(0), el.in_(1), el.in_(2)

UNARY = ["sin", "cos", "tan", "tanh", "asinh", "ceil", "floor", "round_", "exp", "abs_"]


@pytest.mark.parametrize("name", UNARY)
def test_unary(name):
    check(el.render(getattr(el, name)(el.mul(3.0, IN0))), n_in=1, exact=name in ("ceil", "floor", "round_", "abs_"))


@pytest.mark.parametrize("name", ["ln", "log", "log2", "sqrt"])
def test_unary_positive_domain(name):
    check(el.render(getattr(el, name)(IN0)), n_in=1, in_lo=0.01, in_hi=4.0, exact=name == "sqrt")


@pytest.mark.parametrize("name", ["le", "leq", "ge", "geq", "eq", "and_", "or_"])
def test_binary_compare(name):
    a = el.round_(el.mul(2.0, IN0))
    b = el.round_(el.mul(2.0, IN1))
    check(el.render(getattr(el, name)(a, b)), n_in=2, exact=True)


def test_pow():
    check(el.render(el.pow_(el.mul(2.0, IN0), el.round_(el.mul(3.0, IN1)))), n_in=2)
    check(el.render(el.pow_(el.abs_(IN0), IN1)), n_in=2)


@pytest.mark.parametrize("name", ["add", "sub", "mul", "div", "mod", "min_", "max_"])
def test_reduce(name):
    f = getattr(el, name)
    check(el.render(f(IN0, IN1, IN2, 0.37)), n_in=3, exact=name not in ("div", "mod") or True)


def test_add_100_children():
    # offline-renderer.test.js:78-95: a 100-child add of ones sums to 100
    g = el.add(*[el.const(1.0, key=f"c{i}") for i in range(100)])
    got, ref = check(el.render(g), n_voices=2, n_blocks=4, exact=True)
    assert np.all(got[:, 0, 3 * BS:] == 100.0)


def test_div_by_zero_is_zero():
    check(el.render(el.div(IN0, el.round_(IN1))), n_in=2, exact=True)


def test_phasor_cycle_saw_train():
    check(el.render(el.phasor(440.0)), exact=True, n_blocks=6)
    check(el.render(el.cycle(440.0)), n_blocks=8)
    check(el.render(el.saw(110.0)), exact=True)
    check(el.render(el.train(3000.0)), exact=True)
    check(el.render(el.phasor(el.mul(2000.0, IN0))), n_in=1, exact=True)   # negative and audio-rate frequencies


def test_cycle_440_anchor():
    # SURVEY.md Appendix E anchors, generated from the compiled reference
    got, _, _ = run_gpu(el.render(el.cycle(440.0)), 1, 8)
    b0, b2 = got[0, 0, :BS], got[0, 0, 2 * BS:3 * BS]
    assert b0[0] == 0.0 and abs(b0[1] - 5.99625273e-05) < 1e-9 and abs(b0[511] - (-0.487395674)) < 1e-5
    assert abs(b2[0] - 0.653447926) < 1e-5 and abs(float((b2.astype(np.float64) ** 2).sum()) - 248.14756698) < 1e-2


def test_sphasor_counter_accum_latch_maxhold():
    gate = el.le(el.phasor(900.0), 0.3)
    check(el.render(el.syncphasor(220.0, gate)), exact=True, n_blocks=4)
    check(el.render(el.counter(gate)), exact=True)
    check(el.render(el.accum(IN0, gate)), n_in=1, exact=True)
    check(el.render(el.latch(gate, IN0)), n_in=1, exact=True)
    check(el.render(el.maxhold({}, IN0, gate)), n_in=1, exact=True)
    check(el.render(el.maxhold({"hold": 1.0}, IN0, 0.0)), n_in=1, exact=True)


def test_rand_seeded():
    check(el.render(el.rand(seed=12345)), exact=True)
    check(el.render(el.noise(seed=7)), exact=True)


def test_pole_env_biquad_z():
    check(el.render(el.pole(0.95, IN0)), n_in=1)
    check(el.render(el.pole(el.mul(0.9, IN1), IN0)), n_in=2)
    check(el.render(el.env(0.9, 0.999, IN0)), n_in=1)
    check(el.render(el.biquad(0.2, 0.4, 0.2, -0.5, 0.3, IN0)), n_in=1)
    check(el.render(el.z(IN0)), n_in=1, exact=True)
    check(el.render(el.smooth(el.tau2pole(0.01), IN0)), n_in=1)


@pytest.mark.parametrize("mode", ["lowpass", "bandpass", "highpass", "notch", "allpass"])
def test_svf(mode):
    fc = el.add(1500.0, el.mul(1400.0, el.cycle(3.0)))
    check(el.render(el.svf({"mode": mode}, fc, 1.5, IN0)), n_in=1, n_blocks=4)


def test_svf_extreme_params_clamped():
    check(el.render(el.svf({}, el.mul(40000.0, IN0), el.mul(30.0, IN1), IN2)), n_in=3)


@pytest.mark.parametrize("mode", ["lowshelf", "highshelf", "bell"])
def test_svfshelf(mode):
    check(el.render(el.svfshelf({"mode": mode}, 900.0, 0.8, el.mul(12.0, IN1), IN0)), n_in=2)


@pytest.mark.parametrize("mode", ["lowpass", "highpass", "allpass"])
def test_mm1p_prewarp(mode):
    check(el.render(el.mm1p({"mode": mode}, el.prewarp(el.add(2000.0, el.mul(1500.0, IN1))), IN0)), n_in=2)


def test_delay_variants():
    check(el.render(el.delay({"size": 4800}, 3001.5, 0.35, IN0)), n_in=1, n_blocks=12)       # first wrap at block 9
    check(el.render(el.delay({"size": 100}, el.add(50.0, el.mul(49.0, IN1)), el.mul(1.5, IN2), IN0)), n_in=3, n_blocks=4)
    check(el.render(el.delay({"size": 64}, 0.0, 0.9, IN0)), n_in=1, exact=True)               # zero length: write-through
    check(el.render(el.delay({}, 17.25, 0.0, IN0)), n_in=1)                                  # default size = block size
    check(el.render(el.sdelay({"size": 10}, IN0)), n_in=1, exact=True)
    check(el.render(el.sdelay({"size": 3000}, IN0)), n_in=1, exact=True, n_blocks=8)
    check(el.render(el.sdelay({"size": 0}, IN0)), n_in=1, exact=True)


def test_table_lookup():
    tab = np.sin(np.linspace(0, 2 * np.pi, 1000, dtype=np.float64)).astype(np.float32)
    check(el.render(el.table({"path": "wt"}, el.phasor(441.0))), resources={"wt": tab}, n_blocks=4)
    check(el.render(el.table({"path": "wt"}, el.mul(1.3, IN0))), resources={"wt": tab}, n_in=1)   # clamped to [0,1]


@pytest.mark.parametrize("kind", ["blepsaw", "blepsquare", "bleptriangle"])
def test_blep(kind):
    check(el.render(getattr(el, kind)(el.add(1500.0, el.mul(1400.0, IN0)))), n_in=1, n_blocks=4)
    check(el.render(getattr(el, kind)(440.0)), n_blocks=4)


def test_taps_feedback_one_block_delay():
    # tap.test.js:5-50 — ones in, tapOut(add(tapIn, in)): blocks read 1, 2, 3 after the fade-in
    g = el.tap_out("test", el.add(el.tap_in("test"), IN0))
    n_blocks = 14
    inp = np.zeros((1, 1, n_blocks * BS), dtype=np.float32)
    inp[:, :, 10 * BS:] = 1.0
    got, _, _ = run_gpu(el.render(g), 1, n_blocks, inputs=inp)
    ref = oracle_render(el.render(g), n_blocks, 1, SR, BS, inp[0])
    assert np.array_equal(got, ref)
    for k in range(3):
        assert np.all(got[0, 0, (10 + k) * BS:(11 + k) * BS] == float(k + 1))


def test_two_roots_shared_subgraph():
    osc = el.cycle(330.0)
    batch = el.render(el.mul(0.5, osc), el.tanh(el.mul(3.0, osc)))
    check(batch, n_out=2, n_blocks=4)


def test_sr_node_and_leaf_host_inputs():
    check(el.render(el.div(el.sr(), 48000.0)), exact=True)
    # a leaf `sin` node reads host channel 0 (GraphRenderSequence.h:126-135)
    batch = [[0, 1, "root"], [0, 2, "sin"], [2, 1, 2, 0], [3, 1, "channel", 0], [4, [1]], [5]]
    check(batch, n_in=1)


def test_missing_inputs_give_zeros():
    batch = [[0, 1, "root"], [0, 2, "svf"], [0, 3, "const"], [2, 2, 3, 0], [2, 1, 2, 0], [3, 1, "channel", 0], [4, [1]], [5]]
    got, ref = check(batch, exact=True)
    assert not got.any()


SUBSYNTH_BLOCKS = 12


@pytest.mark.parametrize("tile_width", [0, 1, 2, 4, 8, 16, 32])     # every K1 instantiation: <1,0> <4,1> <4,2> <8,3> <8,4> <8,5>
def test_subsynth32_voices(tile_width):
    n_voices = 45   # ragged against every tile width; covers all 40 distinct f0 values
    vb = [graphs.subsynth32_voice_props(v) for v in range(n_voices)]
    opts = {"tile_width": tile_width} if tile_width else {}
    got, mix, rt = run_gpu(graphs.subsynth32(), n_voices, SUBSYNTH_BLOCKS, voice_batches=vb, **opts)
    ref = oracle_render(graphs.subsynth32(), SUBSYNTH_BLOCKS, 1, SR, BS, voice_batches=vb)
    ok, worst, ex = block_peak_tolerance_check(got, ref, BS)
    assert ok, f"worst err/tol {worst:.3g}, bit-exact {ex:.4f}"
    want = ref.astype(np.float64).sum(axis=0)
    assert np.abs(mix - want).max() <= 1e-5 * np.abs(want).max()


def test_subsynth32_anchor_f0_110():
    got, _, _ = run_gpu(graphs.subsynth32(110.0), 1, 12)
    b = got[0, 0].astype(np.float64)
    assert abs(b[1] - (-5.93334116e-05)) < 1e-9
    assert abs((b[2 * BS:3 * BS] ** 2).sum() - 226.292179392) < 5e-3
    assert abs((b[11 * BS:12 * BS] ** 2).sum() - 828.648815053) < 2e-2


def test_additive_voices():
    n_voices, partials = 5, 64
    vb = [graphs.additive64_voice_props(v, partials) for v in range(n_voices)]
    got, mix, rt = run_gpu(graphs.additive64(110.0, partials), n_voices, 4, voice_batches=vb)
    ref = oracle_render(graphs.additive64(110.0, partials), 4, 1, SR, BS, voice_batches=vb)
    ok, worst, ex = block_peak_tolerance_check(got, ref, BS)
    assert ok, f"worst err/tol {worst:.3g}, bit-exact {ex:.4f}"


def test_plumbing_graph_two_channels():
    check(graphs.plumbing(), n_out=2, n_blocks=4, n_voices=2)


def test_short_and_varying_num_samples():
    # numSamples may be smaller than blockSize and vary call to call (cli/Realtime.cpp:38-57)
    from oracle import oracle as orc
    from helpers import oracle_cls
    batch = graphs.subsynth32(220.0)
    rt = Runtime(SR, BS, 2, device=0)
    assert rt.apply_instructions(batch) == 0
    o = oracle_cls()(SR, BS)
    assert o.apply(batch) == 0
    for n in (512, 7, 100, 512, 1, 333, 512):
        got, _ = rt.process_voices(None, 1, n)
        ref = o.process(None, 1, n)
        tol = 1e-5 * np.abs(ref).max() + 1e-7
        assert np.abs(got[0] - ref).max() <= tol and np.array_equal(got[0], got[1])


def test_reference_goldens_delay_sdelay_table_maxhold():
    # jest snapshots of js/packages/offline-renderer/__tests__ (delays/vfs/maxhold .test.js.snap)
    def run(graph, inp, resources=None, sr=SR):
        rt = Runtime(sr, BS, 1, device=0)
        for k, v in (resources or {}).items():
            rt.add_shared_resource(k, v)
        assert rt.apply_instructions(el.render(graph)) == 0
        z = np.zeros((1, 1, BS), dtype=np.float32)
        for _ in range(10):
            rt.process_voices(z, 1, BS)
        x = np.zeros((1, 1, BS), dtype=np.float32)
        x[0, 0, :len(inp)] = inp
        got, _ = rt.process_voices(x, 1, BS)
        return got[0, 0, :len(inp)]

    assert np.array_equal(run(el.delay({"size": 10}, 0.5, 0, IN0), [1, 2, 3, 4]), [0, 0.5, 1, 1.5])
    assert np.array_equal(run(el.delay({"size": 10}, 0, 0, IN0), [1, 2, 3, 4]), [1, 2, 3, 4])
    sd_in = [1, 2, 3, 4, 4, 3, 2, 1] + [0] * 16
    assert np.array_equal(run(el.sdelay({"size": 10}, IN0), sd_in), [0] * 10 + [1, 2, 3, 4, 4, 3, 2, 1] + [0] * 6)
    assert np.array_equal(run(el.table({"path": "/v/increment"}, IN0), [0, 0.25, 0.5, 0.75, 1],
                              {"/v/increment": np.array([1, 2, 3, 4, 5], dtype=np.float32)}), [1, 2, 3, 4, 5])
    assert np.array_equal(run(el.maxhold({}, IN0, 0), [1, 2, 3, 4, 3, 2, 1]), [1, 2, 3, 4, 4, 4, 4])
    mh_in = [1, 2, 3, 4, 3, 2, 1] + [1] * 41
    # the jest suite runs at the OfflineRenderer default of 44.1 kHz: hold = 1 ms = 44 samples
    assert np.array_equal(run(el.maxhold({"hold": 1}, IN0, 0), mh_in, sr=44100.0), [1, 2, 3] + [4] * 44 + [1])


def test_const_math_goldens():
    # offline-renderer.test.js:5-23: el.mul(2,3) settles at 6 once the fade is over
    got, _, _ = run_gpu(el.render(el.mul(2, 3)), 1, 11)
    assert np.all(got[0, 0, 10 * BS:] == 6.0)


def test_root_fade_ramp():
    # SURVEY.md Appendix A: const 1 -> root: block 0 = i/960 ramp, block 1 reaches 1, then 1
    got, _, _ = run_gpu(el.render(el.const(1.0)), 1, 3)
    x = got[0, 0]
    assert x[0] == 0.0 and abs(x[1] - 0.00104166672) < 1e-10 and abs(x[511] - 0.53229171) < 1e-7
    assert abs(x[512] - 0.533333361) < 1e-7 and x[1023] == 1.0 and np.all(x[1024:] == 1.0)


def test_graph_update_crossfade_and_gc():
    # render A, run, render B (A's root fades out while B fades in), run; parity against the oracle throughout
    from helpers import oracle_cls
    r = el.Renderer()
    a = r.render(el.cycle(220.0))
    b = r.render(el.mul(0.5, el.saw(330.0)))
    rt = Runtime(SR, BS, 2, device=0)
    o = oracle_cls()(SR, BS)
    assert rt.apply_instructions(a) == 0 and o.apply(a) == 0
    outs_g, outs_r = [], []
    for _ in range(4):
        outs_g.append(rt.process_voices(None, 1, BS)[0][0]); outs_r.append(o.process(None, 1, BS))
    assert rt.apply_instructions(b) == 0 and o.apply(b) == 0
    for _ in range(6):
        outs_g.append(rt.process_voices(None, 1, BS)[0][0]); outs_r.append(o.process(None, 1, BS))
    g, rr = np.concatenate(outs_g, axis=1), np.concatenate(outs_r, axis=1)
    ok, worst, ex = block_peak_tolerance_check(g, rr, BS)
    assert ok, f"worst err/tol {worst:.3g}"
    if hasattr(o, "gc"):
        assert sorted(rt.gc()) == sorted(o.gc())


def test_heterogeneous_voice_groups():
    # different graphs on different voice ranges of one runtime (config 5 in miniature)
    rt = Runtime(SR, BS, 6, device=0)
    batches = [graphs.random_graph(seed, 24) for seed in range(3)]
    for i, b in enumerate(batches):
        assert rt.apply_instructions(b, voices=(2 * i, 2 * i + 2)) == 0, rt.last_error()
    got, mix = rt.render_voices(6, 1)
    for i, b in enumerate(batches):
        ref = oracle_render(b, 6, 1, SR, BS)
        for v in (2 * i, 2 * i + 1):
            ok, worst, ex = block_peak_tolerance_check(got[v], ref[0], BS)
            assert ok, f"graph {i}: worst err/tol {worst:.3g}"


def test_process_mix_api_shared_inputs():
    # Runtime::process shape: inputs broadcast to all voices, output = mix bus
    n_voices = 37
    batch = el.render(el.mul(IN0, el.cycle(el.const(200.0, key="f"))))
    rt = Runtime(SR, BS, n_voices, device=0)
    assert rt.apply_instructions(batch) == 0
    fid = el.const(0, key="f").id()
    freqs = 100.0 + 10.0 * np.arange(n_voices)
    assert rt.set_property_per_voice(fid, "value", freqs) == 0
    x = lcg_noise(3 * BS, 5)[None, :]
    outs = np.concatenate([rt.process(x[:, b * BS:(b + 1) * BS], 1, BS) for b in range(3)], axis=1)
    vb = [[[3, fid, "value", float(f)]] for f in freqs]
    ref = oracle_render(batch, 3, 1, SR, BS, x, voice_batches=vb)
    want = ref.astype(np.float64).sum(axis=0)
    assert np.abs(outs - want).max() <= 1e-5 * np.abs(want).max()


@pytest.mark.parametrize("tile_width", [0, 4])
def test_split_live_voice_group_keeps_every_voice_state(tile_width):
    """SURVEY.md §8f N1: a structural batch addressed to part of a running voice group cuts the group; the voices that
    move keep their phases, filter memories and delay lines (nodes shared by the old and the new graph continue
    seamlessly, exactly like they do inside one reference Runtime), the others are untouched."""
    from helpers import oracle_cls
    n_voices, bs = 8, BS
    core = el.svf({"mode": "lowpass"}, el.add(900.0, el.mul(500.0, el.cycle(0.7))), 2.0, el.saw(el.const(110.0, key="f")))
    g1 = el.add(core, el.mul(0.4, el.delay({"size": 3000}, 1234.5, 0.3, core)))
    g2 = el.tanh(el.add(g1, el.mul(0.25, el.cycle(el.const(330.0, key="f2")))))
    fid = el.const(0, key="f").id()
    freqs = 55.0 * (1 + np.arange(n_voices))

    opts = {"tile_width": tile_width} if tile_width else {}
    rt = Runtime(SR, bs, n_voices, device=0, **opts)
    rg = el.Renderer()
    a = rg.render(g1)
    b = rg.render(g2)                                  # incremental batch: only the new nodes + new root
    assert rt.apply_instructions(a) == 0
    assert rt.set_property_per_voice(fid, "value", freqs) == 0
    oracles = []
    for v in range(n_voices):
        o = oracle_cls()(SR, bs)
        assert o.apply(a) == 0 and o.apply([[3, fid, "value", float(freqs[v])]]) == 0
        oracles.append(o)

    got, ref = [], []
    for blk in range(10):
        if blk == 4:                                   # re-wire voices 4..7 only, while everything is running
            assert rt.apply_instructions(b, voices=(4, 8)) == 0, rt.last_error()
            for o in oracles[4:]:
                assert o.apply(b) == 0
            assert len(rt.describe()["groups"]) == 2
        got.append(rt.process_voices(None, 1, bs)[0])
        ref.append(np.stack([o.process(None, 1, bs) for o in oracles]))
    g, r = np.concatenate(got, axis=2), np.concatenate(ref, axis=2)
    ok, worst, ex = block_peak_tolerance_check(g, r, bs)
    assert ok, f"worst err/tol {worst:.3g}, bit-exact {ex:.4f}"
    # voices 0..3 never noticed anything
    assert np.abs(g[:4, :, 4 * bs:]).max() > 0


def test_split_must_respect_tile_boundaries():
    rt = Runtime(SR, BS, 16, device=0, tile_width=4)
    assert rt.apply_instructions(el.render(el.cycle(220.0))) == 0
    rt.process_voices(None, 1, BS)
    assert rt.apply_instructions([[0, 99, "sin"]], voices=(6, 16)) == 7        # 6 is not a multiple of the tile width
    assert rt.apply_instructions([[0, 99, "sin"]], voices=(8, 16)) == 0


@pytest.mark.parametrize("seed", list(range(100, 121)))
def test_random_graph_fuzz(seed):
    """Differential fuzz: random 48-node DAGs over the builtin set (the generator of BASELINE config 5), every tile geometry
    the host may pick, against the oracle from block 0."""
    batch = graphs.random_graph(seed, 48)
    tile_width = [0, 1, 4, 32, 2, 16, 8][seed % 7]
    opts = {"tile_width": tile_width} if tile_width else {}
    n_voices = 33 if tile_width >= 16 else 3
    got, _, _ = run_gpu(batch, n_voices, 5, **opts)
    ref = oracle_render(batch, 5, 1, SR, BS)
    for v in range(n_voices):
        ok, worst, ex = block_peak_tolerance_check(got[v], ref[0], BS)
        assert ok, f"seed {seed} voice {v}: worst err/tol {worst:.3g}, bit-exact {ex:.4f}"


# ---- the geometries and scales the benchmarks actually run (VERDICT r01, weak #1) ----------------------------------------

def _subsynth_class_refs(n_blocks):
    """SUBSYNTH32 has 40 distinct voices (f0 = 55 * (1 + v mod 40)): one oracle render per class."""
    vb = [graphs.subsynth32_voice_props(v) for v in range(40)]
    return oracle_render(graphs.subsynth32(), n_blocks, 1, SR, BS, voice_batches=vb)[:, 0]     # [40, n]


def test_subsynth32_4096_voices_is_the_benchmarked_kernel():
    """BASELINE config 2 at full size: 4096 voices, the tile width the host picks on its own (L = 2, the <4,1> instantiation with
    64-sample tiles that bench.py times).  EVERY voice x 12 blocks against its class reference, and the mix bus against the
    float64 sum of the references."""
    n_voices = 4096
    rt = Runtime(SR, BS, n_voices, device=0)
    assert rt.apply_instructions(graphs.subsynth32()) == 0, rt.last_error()
    ida, idb = graphs.subsynth32_param_ids()
    f0 = np.array([graphs.subsynth32_f0(v) for v in range(n_voices)])
    assert rt.set_property_per_voice(ida, "value", f0) == 0 and rt.set_property_per_voice(idb, "value", f0 * 1.007) == 0
    got, mix = rt.render_voices(SUBSYNTH_BLOCKS, 1)
    assert rt.describe()["groups"][0]["tile_width"] == 2
    ref = _subsynth_class_refs(SUBSYNTH_BLOCKS)
    full = ref[np.arange(n_voices) % 40]
    ok, worst, ex = block_peak_tolerance_check(got[:, 0], full, BS)
    assert ok, f"worst err/tol {worst:.3g}, bit-exact {ex:.4f}"
    want = full.astype(np.float64).sum(axis=0)
    blk = np.abs(want).reshape(-1, BS).max(axis=1).repeat(BS)
    assert (np.abs(mix[0] - want) <= 1e-5 * blk + 1e-7).all(), float((np.abs(mix[0] - want) / (1e-5 * blk + 1e-7)).max())


def test_subsynth32_wide_tiles_at_scale():
    """2048 voices in the L = 16 and L = 32 geometries with several warps per CTA (what 32k - 131k voice runs use)."""
    ref = _subsynth_class_refs(SUBSYNTH_BLOCKS)
    for L, n_voices in ((16, 2000), (32, 4100)):
        rt = Runtime(SR, BS, n_voices, device=0, tile_width=L, warps_per_cta=4)
        assert rt.apply_instructions(graphs.subsynth32()) == 0
        ida, idb = graphs.subsynth32_param_ids()
        f0 = np.array([graphs.subsynth32_f0(v) for v in range(n_voices)])
        assert rt.set_property_per_voice(ida, "value", f0) == 0 and rt.set_property_per_voice(idb, "value", f0 * 1.007) == 0
        got, mix = rt.render_voices(SUBSYNTH_BLOCKS, 1)
        ok, worst, ex = block_peak_tolerance_check(got[:, 0], ref[np.arange(n_voices) % 40], BS)
        assert ok, f"L={L}: worst err/tol {worst:.3g}, bit-exact {ex:.4f}"


@pytest.mark.parametrize("tile_width", [0, 2, 8])
def test_many_voice_groups_in_one_launch(tile_width):
    """BASELINE config 5 in small: 12 different random 64-node graphs on 12 voice groups, rendered by ONE render_groups_kernel
    launch per block; every voice against the oracle."""
    n_groups, per = 12, (2 if tile_width in (0, 2) else 8)
    opts = {"tile_width": tile_width} if tile_width else {}
    rt = Runtime(SR, BS, n_groups * per, device=0, **opts)
    batches = [graphs.random_graph(1000 + i, 64) for i in range(n_groups)]
    for i, b in enumerate(batches):
        assert rt.apply_instructions(b, voices=(per * i, per * (i + 1))) == 0, rt.last_error()
    l0 = rt.kernel_launches
    got, mix = rt.render_voices(6, 1)
    assert len(rt.describe()["groups"]) == n_groups
    assert rt.kernel_launches - l0 == 6 * 2, "one K1 launch for all groups + one mix reduce per block"
    for i, b in enumerate(batches):
        ref = oracle_render(b, 6, 1, SR, BS)
        for v in range(per * i, per * (i + 1)):
            ok, worst, ex = block_peak_tolerance_check(got[v], ref[0], BS)
            assert ok, f"graph {i} voice {v}: worst err/tol {worst:.3g}"


def test_soak_60_seconds_no_drift():
    """SURVEY.md §8(d): 60 s = 5625 blocks of SUBSYNTH32 in the benchmarked geometry (L = 2), 8 voices with distinct f0; per-block
    peak error against the reference must stay inside the tolerance for the WHOLE run (a phase that drifted by one float ulp per
    block would be far outside after a minute).  The summary is written to gpurun_out/ for profiles/."""
    import json, os
    n_voices, n_blocks = 8, 5625
    rt = Runtime(SR, BS, n_voices, device=0, tile_width=2)
    assert rt.apply_instructions(graphs.subsynth32()) == 0
    vb = [graphs.subsynth32_voice_props(5 * v) for v in range(n_voices)]
    for v, b in enumerate(vb):
        assert rt.apply_instructions(b, voices=(v, v + 1)) == 0
    ref = oracle_render(graphs.subsynth32(), n_blocks, 1, SR, BS, voice_batches=vb)[:, 0]
    worst_by_block = np.zeros(n_blocks)
    exact = 0
    for b in range(n_blocks):
        g = rt.process_voices(None, 1, BS, want_mix=False)[0][:, 0]
        r = ref[:, b * BS:(b + 1) * BS]
        tol = 1e-5 * np.abs(r).max(axis=1, keepdims=True) + 1e-7
        worst_by_block[b] = (np.abs(g.astype(np.float64) - r) / tol).max()
        exact += int((g == r).sum())
    summary = {"blocks": n_blocks, "voices": n_voices, "seconds_of_audio": n_blocks * BS / SR, "tile_width": 2,
               "worst_err_over_tol": float(worst_by_block.max()), "worst_first_100": float(worst_by_block[:100].max()),
               "worst_last_100": float(worst_by_block[-100:].max()), "bit_exact_rate": exact / (n_blocks * BS * n_voices),
               "specialised": bool(os.environ.get("ELEM_B200_SPECIALIZE") == "1")}
    try:
        os.makedirs("gpurun_out", exist_ok=True)
        with open("gpurun_out/soak_subsynth32%s.json" % ("_spec" if summary["specialised"] else ""), "w") as f:
            json.dump(summary, f)
    except OSError:
        pass
    assert worst_by_block.max() <= 1.0, summary
    assert worst_by_block[-100:].max() <= 4 * max(worst_by_block[:100].max(), 0.01), f"error grows: {summary}"


def test_control_thread_edits_while_render_thread_processes(tmp_path):
    """The two-thread contract on the real render path: tests/native/thread_stress.cpp (control thread: re-renders with cross-fades,
    a live voice-group cut, gc, events; render thread: elem_b200_process in a loop) against the GPU for two seconds."""
    import json, os, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run(["make", "stress"], cwd=os.path.join(root, "elementary_b200", "csrc"), capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    a, b = tmp_path / "a.json", tmp_path / "b.json"
    a.write_text(json.dumps(graphs.subsynth32()))
    b.write_text(json.dumps(el.render(el.tanh(el.add(graphs.subsynth32_graph(220.0), el.mul(0.2, el.cycle(330.0)))))))
    r = subprocess.run([os.path.join(root, "build", "thread_stress"), "0", "2.0", str(a), str(b)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout[-500:], r.stderr[-2000:])
    stats = json.loads(r.stdout.strip().splitlines()[-1])
    assert stats["blocks"] > 100 and stats["edits"] > 10 and stats["failures"] == 0, stats


@pytest.mark.parametrize("tile_width", [0, 2, 32])
def test_registered_device_node_types_match_the_reference_plugin_nodes(tile_width):
    """Runtime::registerNodeType (Runtime.h:105-106): two node types registered as CUDA text here and as GraphNode subclasses on the
    reference (oracle/ref_driver.cpp, through the reference's own registerNodeType) render the same samples: a stateless one
    (all lanes) and a stateful one (owner-lane recurrence whose state survives blocks).  The reference's samples are stored in
    tests/golden/reference_extra.npz: 64 fixed positions of every block of every voice, and the exact block peaks."""
    gold, meta = reference_extra()
    n_voices = 5 if tile_width != 32 else 37
    batch = plugin_nodes_batch()
    assert meta["sha256_16"]["plugin_nodes"] == sha16(batch), "graph changed: re-run tests/golden/make_ref_fixtures.py"
    opts = {"tile_width": tile_width} if tile_width else {}
    rt = Runtime(SR, BS, n_voices, device=0, **opts)
    assert rt.register_node_type("b200test.softclip", 1, 0, "const float x = in[0]; return x / (1.0f + fabsf(x));") == 0
    assert rt.register_node_type("b200test.leaky", 2, 1, "s[0] = in[0] + in[1] * s[0]; return s[0];") == 0
    assert rt.apply_instructions(batch) == 0, rt.last_error()
    got, mix = rt.render_voices(4, 1, plugin_nodes_inputs(n_voices))
    assert rt.describe()["groups"][0]["spec_state"] == 2
    idx = gold["plugin_nodes_idx"]
    want = gold["plugin_nodes"][:n_voices].astype(np.float64)
    tol = 1e-5 * gold["plugin_nodes_peak"][:n_voices][..., idx // BS].astype(np.float64) + 1e-7
    ratio = np.abs(got[..., idx] - want) / tol
    assert ratio.max() <= 1.0, f"worst err/tol {ratio.max():.3g}, bit-exact {(got[..., idx] == want).mean():.4f}"


def test_binary_batch_and_const_table_render_like_the_json_path():
    """SURVEY.md §8f N2: the binary instruction batch and the per-voice property table are the same stream in another encoding —
    the rendered samples must be identical bit for bit to the JSON + per-voice SET_PROPERTY path."""
    n_voices = 96
    ida, idb = graphs.subsynth32_param_ids()
    f0 = np.array([graphs.subsynth32_f0(v) for v in range(n_voices)])
    a = Runtime(SR, BS, n_voices, device=0)
    assert a.apply_instructions(graphs.subsynth32()) == 0
    assert a.set_property_per_voice(ida, "value", f0) == 0 and a.set_property_per_voice(idb, "value", f0 * 1.007) == 0
    b = Runtime(SR, BS, n_voices, device=0)
    assert b.apply_binary(el.encode_binary(graphs.subsynth32())) == 0, b.last_error()
    assert b.set_const_table([ida, idb], np.stack([f0, f0 * 1.007]).astype(np.float32)) == 0
    ga, _ = a.render_voices(4, 1)
    gb, _ = b.render_voices(4, 1)
    assert np.array_equal(ga, gb)


@pytest.mark.parametrize("tile_width", [0, 4])
def test_split_keeps_sequencer_and_analysis_state(tile_width):
    """SURVEY.md §8f N1 for the control / analysis nodes (VERDICT r01 missing #8): a live cut of a voice group carries the seq
    position, the sparseq tick state, the capture ring / scratch, the scope ring and the meter readout of the moving voices along;
    audio AND events of every voice match per-voice reference instances across the cut."""
    from helpers import oracle_cls
    from events_common import canon, same
    n_voices, bs = 8, BS
    clock = el.train(el.const(40.0, key="rate"))
    sq = el.seq({"seq": [0.1, 0.2, 0.3, 0.4, 0.5], "hold": True, "loop": True, "key": "sq"}, clock)
    sp = el.sparseq({"seq": [{"value": 1.0, "tickTime": 0}, {"value": 0.5, "tickTime": 3}, {"value": 0.25, "tickTime": 5}], "loop": [0, 7], "key": "sp"}, clock)
    # the carrier is a phasor-built saw, not el.cycle: events are compared EXACTLY (events_common.same) and only transcendental-free
    # signals are bit-exact between CUDA's libm and glibc's (DESIGN.md section 4, numerics)
    sig = el.mul(el.add(sq, sp), el.sub(el.mul(2.0, el.phasor(el.const(220.0, key="f"))), 1.0))
    g1 = el.add(el.meter({"name": "m"}, sig), el.mul(0.0, el.scope({"name": "s", "size": 512}, sig)),
                el.mul(0.0, el.capture({"name": "c"}, el.le(el.phasor(3.0), 0.5), sig)))
    g2 = el.tanh(el.add(g1, el.mul(0.1, el.cycle(el.const(330.0, key="f2")))))
    fid, rid = el.const(0, key="f").id(), el.const(0, key="rate").id()
    freqs, rates = 110.0 * (1 + np.arange(n_voices)), 30.0 + 7.0 * np.arange(n_voices)
    opts = {"tile_width": tile_width} if tile_width else {}
    rt = Runtime(SR, bs, n_voices, device=0, **opts)
    rg = el.Renderer()
    a, b = rg.render(g1), rg.render(g2)
    assert rt.apply_instructions(a) == 0, rt.last_error()
    assert rt.set_property_per_voice(fid, "value", freqs) == 0 and rt.set_property_per_voice(rid, "value", rates) == 0
    oracles = []
    for v in range(n_voices):
        o = oracle_cls()(SR, bs)
        assert o.apply(a) == 0 and o.apply([[3, fid, "value", float(freqs[v])], [3, rid, "value", float(rates[v])]]) == 0
        oracles.append(o)
    seen = 0
    for blk in range(14):
        if blk == 6:
            assert rt.apply_instructions(b, voices=(4, 8)) == 0, rt.last_error()
            for o in oracles[4:]:
                assert o.apply(b) == 0
            assert len(rt.describe()["groups"]) == 2
        got = rt.process_voices(None, 1, bs)[0]
        ref = np.stack([o.process(None, 1, bs) for o in oracles])
        ok, worst, ex = block_peak_tolerance_check(got, ref, bs)
        assert ok, f"block {blk}: worst err/tol {worst:.3g}"
        if blk % 3 == 2:
            events = rt.process_queued_events()
            for v, o in enumerate(oracles):
                want = canon(o.process_queued_events())
                have = canon([e for e in events if e["event"]["voice"] == v])
                assert same(have, want), f"block {blk} voice {v}: {str(have)[:300]} != {str(want)[:300]}"
                seen += len(want)
    assert seen > 0


def test_offline_render_equals_block_by_block_and_many_groups_stay_correct_in_steady_state():
    """elem_b200_render_offline (no host round trip per block, chunked device buffers, copy stream) gives the same samples as
    process_voices block by block — on a single voice group and on many batched groups, where after the root fade-in the steady-state
    fast path (cached descriptors, sample clock as a kernel argument) takes over; a live edit in between must be picked up."""
    n_blocks = 21                                     # not a multiple of the chunk size
    # one group
    a = Runtime(SR, BS, 37, device=0)
    b = Runtime(SR, BS, 37, device=0)
    for rt in (a, b):
        assert rt.apply_instructions(graphs.subsynth32()) == 0
    ref, _ = a.render_voices(n_blocks, 1)
    got = b.render_offline(n_blocks, 1, chunk_blocks=8)
    assert np.array_equal(got, ref)
    # many groups, with a `time` node in one of them (the sample clock is an argument of the many-groups kernel)
    batches = [graphs.random_graph(2000 + i, 32) for i in range(6)] + [el.render(el.mul(el.cycle(100.0), el.le(el.mod(el.time(), 4096.0), 2048.0)))]
    a = Runtime(SR, BS, 14, device=0)
    b = Runtime(SR, BS, 14, device=0)
    for rt in (a, b):
        for i, bt in enumerate(batches):
            assert rt.apply_instructions(bt, voices=(2 * i, 2 * i + 2)) == 0, rt.last_error()
    ref, _ = a.render_voices(n_blocks, 1)
    got = b.render_offline(n_blocks, 1, chunk_blocks=4)
    assert np.array_equal(got, ref)
    for i, bt in enumerate(batches):
        o = oracle_render(bt, n_blocks, 1, SR, BS)
        ok, worst, ex = block_peak_tolerance_check(got[2 * i], o[0], BS)
        assert ok, f"graph {i}: worst err/tol {worst:.3g}"
    # a live edit after the engine went steady: the next blocks must show it
    edit = [[3, el.const(0, key="zz").id(), "value", 1.0]]
    g = el.mul(el.const(0.0, key="zz"), el.cycle(50.0))
    c = Runtime(SR, BS, 4, device=0)
    assert c.apply_instructions(el.render(g), voices=(0, 2)) == 0 and c.apply_instructions(el.render(el.cycle(60.0)), voices=(2, 4)) == 0
    for _ in range(6):
        v, _ = c.process_voices(None, 1, BS)
    assert not v[0].any()
    assert c.apply_instructions(edit, voices=(0, 2)) == 0
    v, _ = c.process_voices(None, 1, BS)
    assert np.abs(v[0]).max() > 0.1


@pytest.mark.parametrize("n_voices,n_out", [(4096, 1), (33, 2), (1, 1)])
def test_process_host_delivery_equals_the_copy_path(n_voices, n_out):
    """Runtime::process hands the mix bus over through mapped host memory + a sequence word written by the kernel that finishes the
    mix (K2; kernels.h HostDeliver) instead of a D2H copy + stream synchronize.  Same samples, bit for bit, as with the option off —
    full blocks, short blocks, two output channels, the multi-group reduction (4096 voices: G > 1) and the single-pass one."""
    sig = graphs.subsynth32_graph(110.0)
    batch = el.render(sig) if n_out == 1 else el.render(sig, el.mul(-0.5, sig))
    a = Runtime(SR, BS, n_voices, device=0)
    b = Runtime(SR, BS, n_voices, device=0, host_deliver=0)
    for rt in (a, b):
        assert rt.apply_instructions(batch) == 0, rt.last_error()
    for n in (BS, BS, 100, 37, BS, 1, BS):
        oa, ob = a.process(None, n_out, n), b.process(None, n_out, n)
        assert oa.shape == (n_out, n) and np.array_equal(oa, ob)
        assert np.abs(oa).max() > 0 or n == 1


@pytest.mark.parametrize("tile_width,niter", [(1, 0), (1, 4), (2, 0), (4, 0), (8, 0), (16, 0)])
def test_delay_read_head_inside_the_tile_but_outside_its_slice(tile_width, niter):
    """Delays.h:108-159 with delay times around the slice length of every narrow geometry (the fast path only needs the read head to
    stay out of the 32/L-sample slice being processed; shorter delays take the serial path): fractional and integer times, feedback,
    audio-rate modulated time — against the oracle."""
    x = el.in_(0)
    taps = []
    for i, (size, length, fb) in enumerate([(64, 1.0, 0.3), (64, 2.5, 0.5), (128, 5.0, 0.2), (128, 17.3, 0.4), (256, 33.2, 0.3), (256, 40.0, 0.0),
                                           (512, 100.7, 0.45), (4096, 129.5, 0.25), (64, 62.9, 0.1), (64, 31.0, 0.2)]):
        taps.append(el.delay({"size": size}, el.const(length, key=f"len{i}"), el.const(fb, key=f"fb{i}"), x))
    mod = el.delay({"size": 300}, el.add(20.0, el.mul(15.0, el.phasor(7.0))), 0.3, x)
    batch = el.render(el.add(*taps, mod))
    check(batch, n_voices=5, n_blocks=4, n_in=1, tile_width=tile_width, **({"niter": niter} if niter else {}))


@pytest.mark.parametrize("stages,niter", [(2, 0), (3, 0), (4, 0), (3, 4), (0, 4)])
def test_pipelined_groups_equal_the_unpipelined_path(stages, niter):
    """BASELINE config 5 shape: one-voice groups of different random 64-node graphs.  The host cuts every program into `stages` pipeline
    stages (one warp each, render_groups_pipe_kernel); the samples must be the SAME BITS as with one warp running the whole program
    (pipeline_stages = 0) — same ops, same order per value — through the root fade-in, short blocks and into the steady state; and a
    sample of the graphs is checked against the reference."""
    n = 40
    batches = [graphs.random_graph(2000 + i, 64) for i in range(n)]
    extra = {"niter": niter} if niter else {}      # niter = 4: one-voice tiles of 128 samples instead of 32
    a = Runtime(SR, BS, n, device=0, pipeline_stages=stages, **extra)
    b = Runtime(SR, BS, n, device=0, pipeline_stages=0)
    for rt in (a, b):
        for i, bt in enumerate(batches):
            assert rt.apply_instructions(bt, voices=(i, i + 1)) == 0, rt.last_error()
    blocks = [BS, BS, 100, BS, 33, BS, BS, BS]
    outs_a, outs_b = [], []
    for nsmp in blocks:
        va, ma = a.process_voices(None, 1, nsmp)
        vb, mb = b.process_voices(None, 1, nsmp)
        assert np.array_equal(va, vb) and np.array_equal(ma, mb)
        outs_a.append(va)
    da, db = a.describe()["groups"], b.describe()["groups"]
    assert sum(1 for g in da if g.get("pipeline_stages") == max(1, stages)) >= n * 3 // 4, [g.get("pipeline_stages") for g in da]
    assert all(g.get("pipeline_stages") == 1 for g in db)
    # offline path (per-graph outputs, steady-state descriptors) on the pipelined engine == block by block
    c = Runtime(SR, BS, n, device=0, pipeline_stages=stages, **extra)
    d = Runtime(SR, BS, n, device=0, pipeline_stages=0)
    for rt in (c, d):
        for i, bt in enumerate(batches):
            assert rt.apply_instructions(bt, voices=(i, i + 1)) == 0
    oc, od = c.render_offline(11, 1), d.render_offline(11, 1)
    assert np.array_equal(oc, od)
    for i in (0, 7, 19, 39):
        ref = oracle_render(batches[i], 11, 1, SR, BS)
        ok, worst, ex = block_peak_tolerance_check(oc[i], ref[0], BS)
        assert ok, f"graph {i}: worst err/tol {worst:.3g}"
