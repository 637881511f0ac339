"""Event scenarios shared by the CPU (port vs compiled reference) and GPU (CUDA path vs oracle) event tests.

A scenario = graph + per-block schedule: which blocks are followed by a processQueuedEvents() call (the reference's
hosts call it once per block — offline-renderer/index.ts:104-132 — but a control thread may poll less often, which is
what exercises the queue/ring arithmetic: a 32-slot readout queue that reads as empty when exactly full, an 8192-sample
scope ring that clobbers, capture's scratch/relay staging)."""
import numpy as np

from elementary_b200 import el

IN0, IN1 = el.in_(0), el.in_(1)


def scenarios():
    gate = el.le(el.phasor(31.0), 0.3)                       # ~1548-sample period, high for 30 %
    return [
        dict(name="meter_every_block", graph=(el.meter({"name": "lvl"}, el.mul(0.7, IN0)),), n_in=1, blocks=6, poll=lambda b: True),
        dict(name="meter_anonymous_polled_rarely", graph=(el.meter({}, IN0),), n_in=1, blocks=70, poll=lambda b: b in (30, 62, 63, 69)),
        dict(name="snapshot", graph=(el.snapshot({"name": "snap"}, el.train(130.0), el.mul(3.0, IN0)),), n_in=1, blocks=8, poll=lambda b: b % 3 == 2),
        # exactly 32 rising edges per block: the 32-slot queue wraps onto its read position and reads as EMPTY
        # (SingleWriterSingleReaderQueue.h:86-98) — the reference never reports anything here, and neither may we
        dict(name="snapshot_32_edges_per_poll", graph=(el.snapshot({"name": "s32"}, el.train(3000.0), IN0),), n_in=1, blocks=4, poll=lambda b: True, silent=True),
        dict(name="snapshot_33_edges_per_poll", graph=(el.snapshot({"name": "s33"}, el.train(3100.0), IN0),), n_in=1, blocks=4, poll=lambda b: True),
        dict(name="scope_two_channels", graph=(el.scope({"name": "sc", "channels": 2, "size": 512}, IN0, el.mul(-1.0, IN1)),), n_in=2, blocks=8, poll=lambda b: True),
        dict(name="scope_big_window_clobbered", graph=(el.scope({"name": "big", "size": 2048}, IN0),), n_in=1, blocks=40, poll=lambda b: b in (3, 4, 5, 6, 30, 31, 39)),
        dict(name="capture", graph=(el.capture({"name": "cap"}, gate, IN0),), n_in=1, blocks=14, poll=lambda b: b % 2 == 1),
        dict(name="capture_polled_once", graph=(el.capture({}, gate, el.mul(2.0, IN0)),), n_in=1, blocks=12, poll=lambda b: b == 11),
        dict(name="fft_default_1024", graph=(el.fft({"name": "spec"}, el.mul(0.5, IN0)),), n_in=1, blocks=7, poll=lambda b: True),
        dict(name="fft_4096_polled_late", graph=(el.fft({"name": "big", "size": 4096}, el.add(el.cycle(1000.0), IN0)),), n_in=1, blocks=30, poll=lambda b: b in (6, 7, 8, 20, 29)),
        dict(name="metro", graph=(el.metro({"name": "tick", "interval": 25.0}),), n_in=0, blocks=12, poll=lambda b: True),
        dict(name="several_nodes_two_roots",
             graph=(el.meter({"name": "a"}, el.snapshot({"name": "b"}, el.train(97.0), IN0)), el.meter({"name": "c"}, el.cycle(440.0))),
             n_in=1, blocks=5, poll=lambda b: True),
    ]


def event_log(cls, sc, sr=48000.0, bs=512):
    """[(block, canonical events)] of one scenario on an oracle class, polled on the scenario's schedule."""
    r = cls(sr, bs)
    assert r.apply(el.render(*sc["graph"])) == 0
    log = []
    for b in range(sc["blocks"]):
        x = np.stack([noise(bs, 1000 * b + c) for c in range(sc["n_in"])]) if sc["n_in"] else None
        r.process(x, len(sc["graph"]), bs)
        if sc["poll"](b):
            log.append((b, canon(r.process_queued_events())))
    return log


def noise(n, seed):
    rng = np.random.RandomState(seed)
    return (rng.rand(n).astype(np.float32) * 2.0 - 1.0)


def canon(events):
    """Order-preserving, float32-rounded canonical form for comparison across implementations."""
    def f32(x):
        if isinstance(x, dict):
            return {k: f32(v) for k, v in x.items()}
        if isinstance(x, list):
            return [f32(y) for y in x]
        if isinstance(x, (int, float)):
            return float(np.float32(x))
        return x
    out = []
    for e in events:
        evt = {k: f32(v) for k, v in e["event"].items() if k != "voice"}
        out.append((e["type"], evt))
    return out


def same(got, want):
    """Event lists (canonical form) equal: exactly, except `fft` spectra, whose double-precision transform may be evaluated by a
    different (equally exact) FFT algorithm than Ooura's and is compared to 2e-6 of the spectrum's peak."""
    if len(got) != len(want):
        return False
    for (tg, eg), (tw, ew) in zip(got, want):
        if tg != tw:
            return False
        if tg != "fft":
            if eg != ew:
                return False
            continue
        if eg.get("source") != ew.get("source"):
            return False
        for part in ("real", "imag"):
            a, b = np.asarray(eg["data"][part], dtype=np.float64), np.asarray(ew["data"][part], dtype=np.float64)
            scale = max(1e-30, np.abs(np.asarray(ew["data"]["real"])).max(), np.abs(np.asarray(ew["data"]["imag"])).max())
            if a.shape != b.shape or np.abs(a - b).max() > 2e-6 * scale:
                return False
    return True


FFT_BINS = 128


def fingerprint(events):
    """Compact stored form of a canonical event list (tests/golden/reference_extra.json): an event that `same` compares exactly
    is kept as a digest of its content; an `fft` event as its source, length, the peak `same` scales its tolerance by and
    FFT_BINS bins at fixed positions."""
    from helpers import sha16
    out = []
    for t, e in events:
        if t != "fft":
            out.append({"type": t, "sha256_16": sha16(e)})
            continue
        re_, im = np.asarray(e["data"]["real"], dtype=np.float64), np.asarray(e["data"]["imag"], dtype=np.float64)
        bins = np.sort(np.random.RandomState(len(re_)).choice(len(re_), min(FFT_BINS, len(re_)), replace=False))
        out.append({"type": t, "source": e.get("source"), "n": len(re_), "scale": max(1e-30, np.abs(re_).max(), np.abs(im).max()),
                    "bins": bins.tolist(), "real": re_[bins].tolist(), "imag": im[bins].tolist()})
    return out


def same_as_fingerprint(got, want):
    """`same`, with the expected event list in its stored form (`fingerprint`)."""
    from helpers import sha16
    if len(got) != len(want):
        return False
    for (tg, eg), w in zip(got, want):
        if tg != w["type"]:
            return False
        if tg != "fft":
            if sha16(eg) != w["sha256_16"]:
                return False
            continue
        if eg.get("source") != w["source"]:
            return False
        for part in ("real", "imag"):
            a = np.asarray(eg["data"][part], dtype=np.float64)
            if a.shape != (w["n"],) or np.abs(a[w["bins"]] - np.asarray(w[part])).max() > 2e-6 * w["scale"]:
                return False
    return True
