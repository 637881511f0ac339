"""CPU: pin the oracle.  (1) the restatement (oracle/elem_oracle.cpp) must agree BIT-EXACTLY with the reference engine's
outputs on every node family (stored under tests/golden/, rendered by the unmodified reference compiled into oracle/_ref);
(2) the restatement, and the compiled reference where oracle/_ref was built, must reproduce the reference's own golden
vectors (jest snapshots) and the Appendix-E anchors."""
import os

import numpy as np
import pytest

from elementary_b200 import el, graphs
from oracle import oracle as orc
from cases import CASES, case_inputs, convolve_rounding_render
from helpers import GOLDEN, reference_extra, sha16

SR, BS = 48000.0, 512
CASES_GOLD = np.load(os.path.join(GOLDEN, "reference_cases.npz"))
GOLD, META = reference_extra()


def render(cls, case, sr=SR):
    r = cls(sr, BS)
    for k, v in (case["resources"] or {}).items():
        assert r.add_shared_resource(k, v)
    assert r.apply(case["batch"]) == 0
    return r.render(case["n_blocks"], case["n_out"], BS, case_inputs(case))


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_port_matches_compiled_reference_bit_exactly(case):
    """Against the reference's render of the case, stored in tests/golden/reference_cases.npz (test_golden.py checks it is current)."""
    a = render(orc.PortRuntime, case)
    b = CASES_GOLD[case["name"]]
    assert np.array_equal(a, b), f"{case['name']}: max diff {np.abs(a - b).max()}"


def _checkers():
    out = [orc.PortRuntime]
    if orc.ref_available():
        out.append(orc.RefRuntime)
    return out


@pytest.mark.parametrize("cls", _checkers(), ids=lambda c: c.__name__)
def test_reference_jest_goldens(cls):
    """js/packages/offline-renderer/__tests__: delays.test.js.snap, vfs.test.js.snap, maxhold.test.js.snap,
    tap.test.js.snap, offline-renderer.test.js (const math) — 10 warm-up blocks pass the root fade first."""
    IN0 = el.in_(0)

    def run(graph, inp, resources=None, sr=SR, blocks=1):
        r = cls(sr, BS)
        for k, v in (resources or {}).items():
            r.add_shared_resource(k, v)
        assert r.apply(el.render(graph)) == 0
        z = np.zeros((1, BS), dtype=np.float32)
        for _ in range(10):
            r.process(z, 1, BS)
        x = np.zeros((1, BS), dtype=np.float32)
        x[0, :len(inp)] = inp
        outs = [r.process(x, 1, BS)[0] for _ in range(blocks)]
        return outs[0][:len(inp)] if blocks == 1 else outs

    assert np.array_equal(run(el.delay({"size": 10}, 0.5, 0, IN0), [1, 2, 3, 4]), [0, 0.5, 1, 1.5])
    assert np.array_equal(run(el.delay({"size": 10}, 0, 0, IN0), [1, 2, 3, 4]), [1, 2, 3, 4])
    sd_in = [1, 2, 3, 4, 4, 3, 2, 1] + [0] * 16
    assert np.array_equal(run(el.sdelay({"size": 10}, IN0), sd_in), [0] * 10 + [1, 2, 3, 4, 4, 3, 2, 1] + [0] * 6)
    assert np.array_equal(run(el.table({"path": "/v/increment"}, IN0), [0, 0.25, 0.5, 0.75, 1],
                              {"/v/increment": np.array([1, 2, 3, 4, 5], dtype=np.float32)}), [1, 2, 3, 4, 5])
    assert np.array_equal(run(el.maxhold({}, IN0, 0), [1, 2, 3, 4, 3, 2, 1]), [1, 2, 3, 4, 4, 4, 4])
    mh_in = [1, 2, 3, 4, 3, 2, 1] + [1] * 41
    assert np.array_equal(run(el.maxhold({"hold": 1}, IN0, 0), mh_in, sr=44100.0), [1, 2, 3] + [4] * 44 + [1])
    taps = run(el.tap_out("test", el.add(el.tap_in("test"), IN0)), [1.0] * BS, blocks=3)
    for k in range(3):
        assert np.all(taps[k] == float(k + 1))
    r = cls(SR, BS)
    assert r.apply(el.render(el.mul(2, 3))) == 0
    assert np.all(r.render(11)[0, 10 * BS:] == 6.0)
    r = cls(SR, BS)
    assert r.apply(el.render(el.add(*[el.const(1.0, key=f"c{i}") for i in range(100)]))) == 0
    assert np.all(r.render(11)[0, 10 * BS:] == 100.0)


@pytest.mark.parametrize("cls", _checkers(), ids=lambda c: c.__name__)
def test_appendix_e_anchors(cls):
    """Known-answer anchors generated from the compiled reference at survey time (SURVEY.md Appendix E)."""
    r = cls(SR, BS)
    assert r.apply(el.render(el.cycle(440.0))) == 0
    o = r.render(8)[0].astype(np.float64)
    assert o[0] == 0 and abs(o[1] - 5.99625273e-05) < 1e-12 and abs(o[511] - (-0.487395674)) < 1e-8
    assert abs((o[:BS] ** 2).sum() - 23.3739981235) < 1e-6
    assert abs(o[2 * BS] - 0.653447926) < 1e-8 and abs((o[2 * BS:3 * BS] ** 2).sum() - 248.14756698) < 1e-5
    assert abs(o[7 * BS] - (-0.796607792)) < 1e-8 and abs((o[7 * BS:8 * BS] ** 2).sum() - 249.701441144) < 1e-5
    r = cls(SR, BS)
    assert r.apply(graphs.subsynth32(110.0)) == 0
    o = r.render(12)[0].astype(np.float64)
    assert abs(o[1] - (-5.93334116e-05)) < 1e-12 and abs(o[511] - (-0.462336272)) < 1e-8
    assert abs((o[:BS] ** 2).sum() - 32.0823949536) < 1e-6
    assert abs((o[2 * BS:3 * BS] ** 2).sum() - 226.292179392) < 1e-5
    assert abs(o[11 * BS] - (-0.0105246305)) < 1e-8 and abs((o[11 * BS:12 * BS] ** 2).sum() - 828.648815053) < 1e-4
    # root fade ramp (Appendix A)
    r = cls(SR, BS)
    assert r.apply(el.render(el.const(1.0))) == 0
    x = r.render(3)[0]
    assert x[0] == 0.0 and abs(x[1] - 0.00104166672) < 1e-10 and abs(x[511] - 0.53229171) < 1e-7
    assert abs(x[512] - 0.533333361) < 1e-7 and x[1023] == 1.0 and np.all(x[1024:] == 1.0)


@pytest.mark.parametrize("cls", _checkers(), ids=lambda c: c.__name__)
def test_return_codes(cls):
    r = cls(SR, BS)
    assert r.apply([[0, 1, "nope"]]) == 1                       # UnknownNodeType
    assert r.apply([[0, 2, "sin"], [0, 2, "sin"]]) == 3         # NodeAlreadyExists
    assert r.apply([[2, 5, 6, 0]]) == 2                         # NodeNotFound
    assert r.apply([[0, 3, "const"], [3, 3, "value", "x"]]) == 5   # InvalidPropertyType
    assert r.apply([[0, 4, "table"], [3, 4, "path", "missing"]]) == 6   # InvalidPropertyValue


# ---- convolve (wasm/Convolve.h + wasm/FFTConvolver): the restatement uses its own double-precision FFT instead of
# Ooura's, so agreement with the compiled reference is to float rounding (1 ulp), not bit-for-bit; both are pinned
# against an exact double-precision convolution exactly like the reference's own self-test does
# (wasm/FFTConvolver/test/Test.cpp:82-140, 58 cases against a naive O(N*M) convolution).
@pytest.mark.parametrize("cls", _checkers(), ids=lambda c: c.__name__)
@pytest.mark.parametrize("taps,blocks", [(1, 4), (300, 6), (512, 6), (513, 6), (4096, 20), (4097, 22), (9000, 30), (16384, 40)])
def test_convolve_against_exact_convolution(cls, taps, blocks):
    ir = np.asarray(graphs.lcg_ir(16384)[:taps], dtype=np.float32) * 2.0
    rng = np.random.RandomState(taps)
    x = ((rng.rand(1, blocks * BS) - 0.5) * 0.5).astype(np.float32)
    r = cls(SR, BS)
    assert r.add_shared_resource("ir", ir) and r.apply(graphs.convolve_channel("ir")) == 0
    got = r.render(blocks, 1, BS, x)[0]
    want = np.convolve(x[0].astype(np.float64), ir.astype(np.float64))[: blocks * BS]
    peak = np.abs(want).max()
    assert np.abs(got[2 * BS:] - want[2 * BS:]).max() <= 1e-6 * peak      # after the 20 ms root fade-in


@pytest.mark.parametrize("taps", [300, 5000, 16384])
def test_convolve_port_matches_reference_to_float_rounding(taps):
    """Against the reference's output stored at 2048 fixed positions, with its exact peak (tests/golden/reference_extra.npz)."""
    got = convolve_rounding_render(orc.PortRuntime, taps)[0]
    idx = GOLD["convolve_rounding_idx"]
    assert np.abs(got[idx] - GOLD[f"convolve_rounding_{taps}"]).max() <= 5e-7 * GOLD[f"convolve_rounding_{taps}_peak"]


@pytest.mark.parametrize("cls", _checkers(), ids=lambda c: c.__name__)
def test_convolve_varying_call_lengths_is_still_a_plain_convolution(cls):
    ir = np.asarray(graphs.lcg_ir(2000), dtype=np.float32) * 2.0
    r = cls(SR, BS)
    assert r.add_shared_resource("ir", ir) and r.apply(graphs.convolve_channel("ir")) == 0
    rng = np.random.RandomState(9)
    xs, ys = [], []
    for n in [512, 512, 512, 7, 100, 512, 405, 1, 333, 512, 512]:
        x = ((rng.rand(1, n) - 0.5) * 0.5).astype(np.float32)
        xs.append(x[0]); ys.append(r.process(x, 1, n)[0])
    x, y = np.concatenate(xs), np.concatenate(ys)
    want = np.convolve(x.astype(np.float64), ir.astype(np.float64))[: len(x)]
    assert np.abs(y[1536:] - want[1536:]).max() <= 1e-6 * np.abs(want).max()


# ---- events (SURVEY.md §8f N4): the restatement's processQueuedEvents against the compiled reference ----------------
def test_port_events_match_compiled_reference():
    """Against the reference's event logs in their stored form (events_common.fingerprint, tests/golden/reference_extra.json)."""
    from events_common import event_log, scenarios, same_as_fingerprint
    for sc in scenarios():
        assert META["sha256_16"]["events_" + sc["name"]] == sha16(el.render(*sc["graph"])), \
            sc["name"] + ": graph changed: re-run tests/golden/make_ref_fixtures.py"
        got, want = event_log(orc.PortRuntime, sc), META["events"][sc["name"]]
        assert len(got) == len(want) and all(b0 == b1 and same_as_fingerprint(e0, e1) for (b0, e0), (b1, e1) in zip(got, want)), sc["name"]
        assert any(ev for _, ev in want) != bool(sc.get("silent")), sc["name"] + ": unexpected (lack of) events"
