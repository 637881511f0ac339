"""GPU: K1's latency-hiding paths (engine option k1_prefetch, default 1) compute the same bits as the plain paths they fall back to
(k1_prefetch = 0): prologue rows staged by cp.async, delay ring reads of a whole tile issued before its writes, tap promotion found
through the host's record offset.  Delay lengths sit on both sides of every tile and block boundary, voices of one tile disagree,
lengths run at audio rate, the ring is resized mid-stream and calls are ragged."""
import numpy as np
import pytest

from elementary_b200 import Runtime, el, graphs

pytestmark = pytest.mark.gpu

SR, BS = 48000.0, 512
SIZE = 1500
CALLS = [BS, 1, 37, BS, 100, BS, BS, 512, BS, 37, BS]

# (tile width, niter option) -> samples per tile
GEOMETRIES = {(1, 0): 32, (1, 4): 128, (2, 0): 64, (2, 8): 128, (4, 0): 32, (8, 0): 32, (16, 0): 16, (32, 0): 8, (32, 4): 4}


def delay_lengths(t):
    """Delay times around the tile (t samples) and the block (BS samples) limits of the whole-tile batch, integer and fractional."""
    out = []
    for edge in (t, t + 1, SIZE - t - 1, SIZE - t, BS, BS + 1, SIZE - BS - 1, SIZE - BS):
        out += [float(edge), edge - 0.5, edge + 0.5]
    return out + [3001.5 % SIZE, 0.0]


def delay_graph(lengths, n_voices):
    """One delay per length: even ones the same for every voice, odd ones rotated through the list voice by voice (so the voices of
    a tile disagree), plus one audio-rate delay time that must take the fallback."""
    x = el.in_(0)
    taps, per_voice = [], []
    for i, length in enumerate(lengths):
        k = el.const(length, key=f"len{i}")
        taps.append(el.delay({"size": SIZE, "key": f"d{i}"}, k, el.const(0.1 + 0.02 * (i % 9), key=f"fb{i}"), x))
        if i % 2:
            per_voice.append((k.id(), [lengths[(i + v) % len(lengths)] for v in range(n_voices)]))
    taps.append(el.delay({"size": SIZE, "key": "mod"}, el.add(700.0, el.mul(650.0, el.phasor(3.0))), 0.3, x))
    return el.render(el.add(*taps)), per_voice, taps[2].id()


def pair(batch, n_voices, per_voice=(), **opts):
    rts = []
    for pf in (1, 0):
        rt = Runtime(SR, BS, n_voices, device=0, k1_prefetch=pf, **opts)
        assert rt.apply_instructions(batch) == 0, rt.last_error()
        for nid, vals in per_voice:
            assert rt.set_property_per_voice(nid, "value", vals) == 0
        rts.append(rt)
    return rts


def inputs(n_voices, n, seed):
    return np.random.default_rng(seed).uniform(-1.0, 1.0, (n_voices, 1, n)).astype(np.float32)


def run_lockstep(a, b, n_voices, calls=CALLS, script=None, seed=0):
    peak = 0.0
    for i, n in enumerate(calls):
        for batch in (script or {}).get(i, ()):
            assert a.apply_instructions(batch) == 0 and b.apply_instructions(batch) == 0
        inp = inputs(n_voices, n, seed + i)
        va, ma = a.process_voices(inp, 1, n)
        vb, mb = b.process_voices(inp, 1, n)
        assert np.array_equal(va, vb), f"call {i} ({n} samples): per-voice outputs differ, max {np.abs(va - vb).max()}"
        assert np.array_equal(ma, mb), f"call {i} ({n} samples): mix differs"
        peak = max(peak, float(np.abs(va).max()))
    assert peak > 0


@pytest.mark.parametrize("tile_width,niter", list(GEOMETRIES))
def test_delay_boundaries_equal_the_plain_path(tile_width, niter):
    n_voices = 3 * tile_width + 1          # a ragged last tile as well
    batch, per_voice, resized = delay_graph(delay_lengths(GEOMETRIES[(tile_width, niter)]), n_voices)
    opts = {"niter": niter} if niter else {}
    a, b = pair(batch, n_voices, per_voice, tile_width=tile_width, **opts)
    run_lockstep(a, b, n_voices, script={6: [[[3, resized, "size", 900]]]})


@pytest.mark.parametrize("tile_width,niter", [(1, 0), (2, 0), (8, 0), (32, 0)])
def test_specialised_kernels_equal_the_plain_path(tile_width, niter):
    n_voices = 2 * tile_width
    batch, per_voice, _ = delay_graph(delay_lengths(GEOMETRIES[(tile_width, niter)]), n_voices)
    a, b = pair(batch, n_voices, per_voice, tile_width=tile_width, specialize=2, specialize_strict=1)
    run_lockstep(a, b, n_voices, seed=50)


@pytest.mark.parametrize("tile_width", [2, 32])
def test_subsynth32_equal_the_plain_path(tile_width):
    n_voices = 4 * tile_width
    f0 = np.array([graphs.subsynth32_f0(v) for v in range(n_voices)])
    ida, idb = graphs.subsynth32_param_ids()
    a, b = pair(graphs.subsynth32(), n_voices, [(ida, f0), (idb, f0 * 1.007)], tile_width=tile_width)
    run_lockstep(a, b, n_voices, calls=[BS] * 10 + [37, BS])


def test_taps_promote_on_both_paths():
    """tapOut(add(tapIn, delay(in))): the records behind the program must still promote the tap every block; a program without taps
    (the delay alone) must render the same with nothing to promote."""
    x = el.in_(0)
    dly = el.delay({"size": SIZE}, el.const(600.5, key="tl"), 0.2, x)
    with_taps = el.render(el.tap_out("fb", el.add(el.mul(0.5, el.tap_in("fb")), dly)))
    for batch in (with_taps, el.render(dly)):
        a, b = pair(batch, 4, tile_width=2)
        run_lockstep(a, b, 4, calls=[BS] * 6 + [100, BS], seed=7)


@pytest.mark.parametrize("stages", [0, 3])
def test_groups_equal_the_plain_path(stages):
    """BASELINE config 5 shape: one-voice groups of different random graphs, many-groups launch with and without pipeline stages."""
    n = 24
    batches = [graphs.random_graph(4000 + i, 64) for i in range(n)]
    rts = []
    for pf in (1, 0):
        rt = Runtime(SR, BS, n, device=0, k1_prefetch=pf, pipeline_stages=stages)
        for i, bt in enumerate(batches):
            assert rt.apply_instructions(bt, voices=(i, i + 1)) == 0, rt.last_error()
        rts.append(rt)
    for nsmp in [BS, BS, 100, BS, 33, BS, BS, BS]:
        va, ma = rts[0].process_voices(None, 1, nsmp)
        vb, mb = rts[1].process_voices(None, 1, nsmp)
        assert np.array_equal(va, vb) and np.array_equal(ma, mb)
