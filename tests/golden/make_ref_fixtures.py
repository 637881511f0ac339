"""Generate tests/golden/reference_extra.{npz,json} from the UNMODIFIED reference compiled in place (oracle/_ref).

Run where the reference sources are present, after build() has compiled oracle/_ref/libelem_ref.so from them:
    python tests/golden/make_ref_fixtures.py
These are the reference's outputs for the comparisons that reference_cases.npz (make_golden.py) does not cover, so that the
tests which compare with the reference run without it:
  control_<scenario>          full output of each live-update scenario of tests/control_common.py
  convolve_rounding_<taps>    the convolver of cases.convolve_rounding_render at 2048 fixed positions (convolve_rounding_idx),
                              and its exact peak (convolve_rounding_<taps>_peak)
  plugin_nodes                the reference's plug-in node types (oracle/ref_driver.cpp) on cases.plugin_nodes_batch for 37 voices
                              at 64 fixed positions per block (plugin_nodes_idx), and the exact block peaks (plugin_nodes_peak)
  events (json)               each event scenario of tests/events_common.py in the stored form of events_common.fingerprint
The json also holds, per fixture, the digest of the definition it was rendered from (sha256_16), which the tests check.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as orc                                                   # noqa: E402
from elementary_b200 import el                                                      # noqa: E402
from cases import convolve_rounding_render, plugin_nodes_batch, plugin_nodes_inputs  # noqa: E402
from helpers import oracle_render, sha16                                            # noqa: E402
import control_common                                                               # noqa: E402
import events_common                                                                # noqa: E402

SR, BS = 48000.0, 512


def main():
    assert orc.ref_available(), "oracle/_ref/libelem_ref.so missing: build it where the reference sources are present"
    out, sha, events = {}, {}, {}
    for sc in control_common.scenarios():
        out["control_" + sc["name"]] = control_common.render_live(orc.RefRuntime, sc)
        sha["control_" + sc["name"]] = sha16(control_common.definition(sc))

    n = 36 * BS
    out["convolve_rounding_idx"] = np.sort(np.random.RandomState(36).choice(n, 2048, replace=False)).astype(np.int32)
    for taps in (300, 5000, 16384):
        y = convolve_rounding_render(orc.RefRuntime, taps)[0]
        out[f"convolve_rounding_{taps}"] = y[out["convolve_rounding_idx"]]
        out[f"convolve_rounding_{taps}_peak"] = np.float32(np.abs(y).max())

    batch, n_voices = plugin_nodes_batch(), 37
    y = oracle_render(batch, 4, 1, SR, BS, plugin_nodes_inputs(n_voices), voice_batches=[None] * n_voices, cls=orc.RefRuntime)
    rng = np.random.RandomState(37)
    idx = np.concatenate([b * BS + np.sort(rng.choice(BS, 64, replace=False)) for b in range(4)]).astype(np.int32)
    out["plugin_nodes_idx"] = idx
    out["plugin_nodes"] = y[..., idx]
    out["plugin_nodes_peak"] = np.abs(y.reshape(n_voices, 1, 4, BS)).max(axis=-1)
    sha["plugin_nodes"] = sha16(batch)

    for sc in events_common.scenarios():
        log = events_common.event_log(orc.RefRuntime, sc)
        events[sc["name"]] = [[b, events_common.fingerprint(ev)] for b, ev in log]
        sha["events_" + sc["name"]] = sha16(el.render(*sc["graph"]))

    np.savez_compressed(os.path.join(HERE, "reference_extra.npz"), **out)
    with open(os.path.join(HERE, "reference_extra.json"), "w") as f:
        json.dump({"sample_rate": SR, "block": BS, "generator": "tests/golden/make_ref_fixtures.py",
                   "engine": "elem::Runtime<float> of the unmodified reference, compiled by oracle/Makefile",
                   "sha256_16": sha, "events": events}, f, indent=1, sort_keys=True)
    print(len(out), "arrays,", os.path.getsize(os.path.join(HERE, "reference_extra.npz")), "bytes;",
          os.path.getsize(os.path.join(HERE, "reference_extra.json")), "bytes of json")


if __name__ == "__main__":
    main()
