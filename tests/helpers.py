"""Shared helpers for the parity tests (tests only)."""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

from oracle import oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha16(obj) -> str:
    """First 16 hex digits of the SHA-256 of ``obj`` as JSON: ties a stored fixture to the definition it was rendered from."""
    return hashlib.sha256(json.dumps(obj, sort_keys=True).encode()).hexdigest()[:16]


def reference_extra():
    """(arrays, metadata) of tests/golden/reference_extra.{npz,json}: what the reference engine rendered for the tests that
    compare with it beyond reference_cases (tests/golden/make_ref_fixtures.py)."""
    with open(os.path.join(GOLDEN, "reference_extra.json")) as f:
        meta = json.load(f)
    return np.load(os.path.join(GOLDEN, "reference_extra.npz")), meta


def oracle_cls():
    """The strongest checker available: the compiled reference itself (oracle/_ref) if present, else the port."""
    return orc.RefRuntime if orc.ref_available() else orc.PortRuntime


def oracle_render(batch, n_blocks, n_out=1, sr=48000.0, bs=512, inputs=None, voice_batches=None, resources=None, cls=None):
    """Render `len(voice_batches)` independent oracle instances (or one). Returns [voice, n_out, n_blocks*bs]."""
    cls = cls or oracle_cls()
    vb = voice_batches if voice_batches is not None else [None]
    outs = []
    for v, extra in enumerate(vb):
        r = cls(sr, bs)
        for name, data in (resources or {}).items():
            assert r.add_shared_resource(name, data)
        assert r.apply(batch) == 0
        if extra:
            assert r.apply(extra) == 0
        inp = None
        if inputs is not None:
            inp = inputs[v] if np.asarray(inputs).ndim == 3 else inputs
        outs.append(r.render(n_blocks, n_out, bs, inp))
    return np.stack(outs)


def block_peak_tolerance_check(got, ref, bs=512, rtol=1e-5, floor=1e-7):
    """north_star tolerance, read as SURVEY.md §8(d) prescribes: |gpu - ref| <= 1e-5 * max|ref| over the block
    (plus a tiny absolute floor for all-zero blocks).  Returns (ok, worst_ratio, bit_exact_fraction)."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    n = got.shape[-1]
    nb = n // bs
    g = got[..., : nb * bs].reshape(got.shape[:-1] + (nb, bs))
    r = ref[..., : nb * bs].reshape(ref.shape[:-1] + (nb, bs))
    peak = np.abs(r).max(axis=-1, keepdims=True)
    err = np.abs(g - r)
    tol = rtol * peak + floor
    worst = float((err / tol).max()) if err.size else 0.0
    exact = float((got.astype(np.float32) == ref.astype(np.float32)).mean()) if got.size else 1.0
    return bool((err <= tol).all()), worst, exact
