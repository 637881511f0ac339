"""Graph cases shared by the CPU oracle tests (port vs compiled reference) — one entry per node family."""
import math

import numpy as np

from elementary_b200 import el, graphs

IN0, IN1, IN2 = el.in_(0), el.in_(1), el.in_(2)
_gate = el.le(el.phasor(900.0), 0.3)
_tab = np.sin(np.linspace(0, 2 * np.pi, 1000, dtype=np.float64)).astype(np.float32)


def _c(name, graph, n_in=0, n_blocks=3, resources=None, n_out=1, batch=None):
    return dict(name=name, batch=batch if batch is not None else el.render(*(graph if isinstance(graph, tuple) else (graph,))),
                n_in=n_in, n_blocks=n_blocks, resources=resources, n_out=n_out)


CASES = []
for _u in ["sin", "cos", "tan", "tanh", "asinh", "ceil", "floor", "round_", "exp", "abs_"]:
    CASES.append(_c(_u, getattr(el, _u)(el.mul(3.0, IN0)), 1))
for _u in ["ln", "log", "log2", "sqrt"]:
    CASES.append(_c(_u, getattr(el, _u)(el.abs_(IN0)), 1))
for _b in ["le", "leq", "ge", "geq", "eq", "and_", "or_"]:
    CASES.append(_c(_b, getattr(el, _b)(el.round_(el.mul(2.0, IN0)), el.round_(el.mul(2.0, IN1))), 2))
CASES.append(_c("pow", el.pow_(el.mul(2.0, IN0), el.round_(el.mul(3.0, IN1))), 2))
for _r in ["add", "sub", "mul", "div", "mod", "min_", "max_"]:
    CASES.append(_c(_r, getattr(el, _r)(IN0, IN1, IN2, 0.37), 3))
CASES += [
    _c("phasor", el.phasor(440.0), n_blocks=6),
    _c("cycle", el.cycle(440.0), n_blocks=8),
    _c("saw", el.saw(110.0)),
    _c("phasor_audio_rate", el.phasor(el.mul(2000.0, IN0)), 1),
    _c("sphasor", el.syncphasor(220.0, _gate), n_blocks=4),
    _c("counter", el.counter(_gate)),
    _c("accum", el.accum(IN0, _gate), 1),
    _c("latch", el.latch(_gate, IN0), 1),
    _c("maxhold", el.maxhold({}, IN0, _gate), 1),
    _c("maxhold_hold", el.maxhold({"hold": 1.0}, IN0, 0.0), 1),
    _c("rand", el.rand(seed=12345)),
    _c("pole", el.pole(el.mul(0.9, IN1), IN0), 2),
    _c("env", el.env(0.9, 0.999, IN0), 1),
    _c("biquad", el.biquad(0.2, 0.4, 0.2, -0.5, 0.3, IN0), 1),
    _c("z", el.z(IN0), 1),
    _c("smooth", el.smooth(el.tau2pole(0.01), IN0), 1),
    _c("svf_extreme", el.svf({}, el.mul(40000.0, IN0), el.mul(30.0, IN1), IN2), 3),
    _c("delay_4800", el.delay({"size": 4800}, 3001.5, 0.35, IN0), 1, 12),
    _c("delay_mod", el.delay({"size": 100}, el.add(50.0, el.mul(49.0, IN1)), el.mul(1.5, IN2), IN0), 3, 4),
    _c("delay_zero", el.delay({"size": 64}, 0.0, 0.9, IN0), 1),
    _c("delay_default", el.delay({}, 17.25, 0.0, IN0), 1),
    _c("sdelay_10", el.sdelay({"size": 10}, IN0), 1),
    _c("sdelay_3000", el.sdelay({"size": 3000}, IN0), 1, 8),
    _c("sdelay_0", el.sdelay({"size": 0}, IN0), 1),
    _c("table", el.table({"path": "wt"}, el.phasor(441.0)), 0, 4, {"wt": _tab}),
    _c("table_clamped", el.table({"path": "wt"}, el.mul(1.3, IN0)), 1, 3, {"wt": _tab}),
    _c("taps", el.tap_out("t", el.add(el.tap_in("t"), IN0)), 1, 5),
    _c("two_roots", (el.mul(0.5, el.cycle(330.0)), el.tanh(el.mul(3.0, el.cycle(330.0)))), 0, 4, None, 2),
    _c("sr", el.div(el.sr(), 48000.0)),
    _c("leaf_sin", None, 1, 3, None, 1, [[0, 1, "root"], [0, 2, "sin"], [2, 1, 2, 0], [3, 1, "channel", 0], [4, [1]], [5]]),
    _c("missing_inputs", None, 0, 2, None, 1,
       [[0, 1, "root"], [0, 2, "svf"], [0, 3, "const"], [2, 2, 3, 0], [2, 1, 2, 0], [3, 1, "channel", 0], [4, [1]], [5]]),
    _c("subsynth32", None, 0, 12, None, 1, graphs.subsynth32(110.0)),
    _c("additive16", None, 0, 4, None, 1, graphs.additive64(110.0, 16)),
    _c("plumbing", None, 0, 4, None, 2, graphs.plumbing()),
]
for _m in ["lowpass", "bandpass", "highpass", "notch", "allpass"]:
    CASES.append(_c("svf_" + _m, el.svf({"mode": _m}, el.add(1500.0, el.mul(1400.0, el.cycle(3.0))), 1.5, IN0), 1, 4))
for _m in ["lowshelf", "highshelf", "bell"]:
    CASES.append(_c("svfshelf_" + _m, el.svfshelf({"mode": _m}, 900.0, 0.8, el.mul(12.0, IN1), IN0), 2))
for _m in ["lowpass", "highpass", "allpass"]:
    CASES.append(_c("mm1p_" + _m, el.mm1p({"mode": _m}, el.prewarp(el.add(2000.0, el.mul(1500.0, IN1))), IN0), 2))
for _k in ["blepsaw", "blepsquare", "bleptriangle"]:
    CASES.append(_c(_k, getattr(el, _k)(el.add(1500.0, el.mul(1400.0, IN0))), 1, 4))
for _s in range(4):
    CASES.append(_c(f"random_graph_{_s}", None, 0, 6, None, 1, graphs.random_graph(_s, 32)))

# ---- sequencing / control nodes (SURVEY.md §8f N3): Core.h once/seq, Seq2.h, SparSeq.h, SparSeq2.h, wasm/Metro.h, SampleTime.h
_trig = el.train(2000.0)          # 24-sample period @ 48 kHz
_rst = el.train(170.0)
_sq = [1.0, -2.0, 3.5, 0.25, 7.0]
_sp = [{"value": 1.0, "tickTime": 0}, {"value": 4.0, "tickTime": 3}, {"value": -2.0, "tickTime": 4}, {"value": 9.0, "tickTime": 11}]
_sp2 = [{"value": 0.5, "time": 0.002}, {"value": 2.0, "time": 0.004}, {"value": -1.0, "time": 0.011}, {"value": 3.0, "time": 0.02}]
_secs = el.div(el.time(), el.sr())
CASES += [
    _c("time", el.time(), n_blocks=3),
    _c("time_scaled", el.mul(el.time(), 1.0e-3), n_blocks=3),
    _c("metro_default", el.metro({}), n_blocks=4),
    _c("metro_5ms", el.metro({"interval": 5.0}), n_blocks=4),
    _c("metro_tiny", el.metro({"interval": 0.001}), n_blocks=2),
    _c("once_armed", el.once({"arm": True}, el.train(150.0)), n_blocks=4),
    _c("once_unarmed", el.once({"arm": False}, el.train(150.0)), n_blocks=2),
    _c("once_scaled_pulse", el.once({"arm": True}, el.mul(el.train(700.0), IN0)), 1, 3),
    _c("seq_loop", el.seq({"seq": _sq}, _trig, _rst), n_blocks=4),
    _c("seq_hold", el.seq({"seq": _sq, "hold": True}, _trig, _rst), n_blocks=4),
    _c("seq_noloop", el.seq({"seq": _sq, "loop": False}, _trig, 0.0), n_blocks=2),
    _c("seq_noloop_hold", el.seq({"seq": _sq, "loop": False, "hold": True, "offset": 2}, _trig, _rst), n_blocks=4),
    _c("seq_offset", el.seq({"seq": _sq, "offset": 3}, _trig, _rst), n_blocks=4),
    _c("seq_single_child", None, 0, 2, None, 1,
       [[0, 1, "root"], [0, 2, "seq"], [0, 3, "le"], [0, 4, "phasor"], [0, 5, "const"], [0, 6, "const"],
        [2, 4, 5, 0], [2, 3, 4, 0], [2, 3, 6, 0], [2, 2, 3, 0], [2, 1, 2, 0],
        [3, 5, "value", 2000.0], [3, 6, "value", 0.5], [3, 2, "seq", [3.0, 1.0, 2.0]], [3, 1, "channel", 0], [4, [1]], [5]]),
    _c("seq_no_data", el.seq({}, _trig, _rst), n_blocks=1),
    _c("seq2_loop", el.seq2({"seq": _sq}, _trig, _rst), n_blocks=4),
    _c("seq2_hold", el.seq2({"seq": _sq, "hold": True, "offset": 1}, _trig, _rst), n_blocks=4),
    _c("seq2_noloop", el.seq2({"seq": _sq, "loop": False}, _trig, _rst), n_blocks=4),
    _c("seq2_noloop_hold", el.seq2({"seq": _sq, "loop": False, "hold": True}, _trig, 0.0), n_blocks=2),
    _c("sparseq_plain", el.sparseq({"seq": _sp}, _trig, _rst), n_blocks=4),
    _c("sparseq_loop", el.sparseq({"seq": _sp, "loop": [1, 7]}, _trig, 0.0), n_blocks=4),
    _c("sparseq_interp", el.sparseq({"seq": _sp, "interpolate": 1, "tickInterval": 0.0005}, _trig, _rst), n_blocks=4),
    _c("sparseq_interp_loop_offset", el.sparseq({"seq": _sp, "interpolate": 1, "loop": [0, 12], "offset": 2}, _trig, _rst), n_blocks=6),
    _c("sparseq2_hold", el.sparseq2({"seq": _sp2}, _secs), n_blocks=4),
    _c("sparseq2_interp", el.sparseq2({"seq": _sp2, "interpolate": 1}, _secs), n_blocks=4),
    _c("sparseq2_backwards", el.sparseq2({"seq": _sp2, "interpolate": 1}, el.mul(0.03, el.abs_(el.cycle(37.0)))), n_blocks=4),
    _c("meter_passthrough", el.meter({"name": "m"}, el.mul(0.5, IN0)), 1, 2),
    _c("snapshot_passthrough", el.snapshot({"name": "s"}, el.train(500.0), IN0), 1, 2),
    _c("scope_passthrough", el.scope({"name": "sc", "channels": 2}, IN0, IN1), 2, 2),
    _c("fft_passthrough", el.fft({"name": "f"}, IN0), 1, 2),
    _c("capture_passthrough", el.capture({"name": "c"}, el.train(40.0), IN0), 1, 2),
    _c("arp_voice", el.mul(el.seq({"seq": [0.2, 0.5, 1.0], "hold": True}, el.metro({"interval": 2.0})),
                        el.cycle(el.seq({"seq": [220.0, 330.0, 440.0, 660.0], "hold": True}, el.metro({"interval": 2.0})))), n_blocks=6),
]


def lcg_noise(n, seed, lo=-1.0, hi=1.0):
    s = (seed * 2654435761 + 1) & 0xFFFFFFFF
    out = np.empty(n, dtype=np.float32)
    for i in range(n):
        s = (s * 1664525 + 1013904223) & 0xFFFFFFFF
        out[i] = lo + (hi - lo) * ((s >> 8) / float(1 << 24))
    return out


def case_inputs(case, bs=512, seed=0):
    if not case["n_in"]:
        return None
    return np.stack([lcg_noise(case["n_blocks"] * bs, seed * 100 + c) for c in range(case["n_in"])])


def convolve_rounding_render(cls, taps, sr=48000.0, bs=512):
    """36 blocks of noise through the convolver on the first `taps` taps of the config-4 IR: [1, 36 * bs]."""
    ir = np.asarray(graphs.lcg_ir(16384)[:taps], dtype=np.float32)
    rng = np.random.RandomState(3)
    x = ((rng.rand(1, 36 * bs) - 0.5) * 0.5).astype(np.float32)
    r = cls(sr, bs)
    assert r.add_shared_resource("ir", ir) and r.apply(graphs.convolve_channel("ir")) == 0
    return r.render(36, 1, bs, x)


def plugin_nodes_batch():
    """The graph of the registered-node-type test: 3 * in0 -> softclip -> leaky (g = 0.9), plus 0.1 * cycle(330)."""
    soft = el.create_node("b200test.softclip", {}, [el.mul(3.0, IN0)])
    return el.render(el.add(el.create_node("b200test.leaky", {}, [soft, el.const(0.9, key="g")]), el.mul(0.1, el.cycle(330.0))))


def plugin_nodes_inputs(n_voices, bs=512):
    """[voice, 1, 4 * bs]: 4 blocks of LCG noise per voice."""
    return np.stack([np.stack([lcg_noise(4 * bs, 100 * v)]) for v in range(n_voices)])
