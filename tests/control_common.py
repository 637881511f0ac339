"""Live-update scenarios for the sequencing / control nodes, shared by the GPU parity tests (CUDA path vs oracle) and the CPU
pinning test (restatement vs compiled reference): an initial batch plus batches applied before given blocks."""
import numpy as np

from elementary_b200 import el

TRIG = el.train(2000.0)
RST = el.train(170.0)


def scenarios():
    out = []
    node = el.seq({"seq": [1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0], "hold": True, "key": "s"}, TRIG, RST)
    nid = node.id()
    out.append(dict(name="seq_new_data_hold_offset", batch=el.render(node), n_blocks=9, n_out=1, exact=True, script={
        2: [[3, nid, "seq", [10.0, 20.0, 30.0]]],
        4: [[3, nid, "hold", False], [3, nid, "offset", 1]],
        6: [[3, nid, "loop", False], [3, nid, "seq", [-1.0, -2.0, -3.0, -4.0, -5.0]]]}))
    seq2 = el.seq2({"seq": [0.5, 1.5, -2.5], "key": "s2"}, TRIG, RST)
    once = el.once({"arm": False, "key": "o"}, el.train(300.0))
    sid, oid = seq2.id(), once.id()
    out.append(dict(name="seq2_and_once_rearm", batch=el.render(seq2, once), n_blocks=8, n_out=2, exact=True, script={
        1: [[3, oid, "arm", True]],
        3: [[3, sid, "seq", [9.0, 8.0, 7.0, 6.0]], [3, sid, "offset", 2]],
        4: [[3, oid, "arm", False], [3, oid, "arm", True]],
        6: [[3, sid, "hold", True], [3, sid, "loop", False]]}))
    sp = [{"value": 1.0, "tickTime": 0}, {"value": 4.0, "tickTime": 3}, {"value": -2.0, "tickTime": 4}, {"value": 9.0, "tickTime": 11}]
    sp_b = [{"value": 2.0, "tickTime": 0}, {"value": 6.0, "tickTime": 2}, {"value": 0.5, "tickTime": 9}, {"value": 3.0, "tickTime": 20}]
    for follow in (False, True):
        node = el.sparseq({"seq": sp, "follow": follow, "interpolate": 1, "tickInterval": 0.0005, "key": "sp"}, TRIG, RST)
        nid = node.id()
        out.append(dict(name=f"sparseq_loop_points_follow_{int(follow)}", batch=el.render(node), n_blocks=10, n_out=1, exact=False, script={
            1: [[3, nid, "loop", [0, 8]]],
            3: [[3, nid, "loop", [2, 6]]],
            4: [[3, nid, "seq", sp_b]],
            6: [[3, nid, "loop", False], [3, nid, "offset", 3]],
            7: [[3, nid, "loop", None], [3, nid, "interpolate", 0]]}))
    sp2 = [{"value": 0.5, "time": 0.002}, {"value": 2.0, "time": 0.004}, {"value": -1.0, "time": 0.011}, {"value": 3.0, "time": 0.02}]
    node = el.sparseq2({"seq": sp2, "key": "q"}, el.mul(0.03, el.abs_(el.cycle(37.0))))
    nid = node.id()
    out.append(dict(name="sparseq2_new_sequence_interpolation", batch=el.render(node), n_blocks=7, n_out=1, exact=False, script={
        2: [[3, nid, "interpolate", 1]],
        4: [[3, nid, "seq", [{"value": 5.0, "time": 0.001}, {"value": -5.0, "time": 0.025}]]]}))
    g = el.add(el.mul(1e-6, el.time()), el.metro({"interval": 3.0}))
    out.append(dict(name="time_metro_host_clock", batch=el.render(g), n_blocks=6, n_out=1, exact=True, script={},
                    sample_times=[0, 512, 10_000_000_000, 10_000_000_512, 77, 123456789]))
    x = el.saw(220.0)
    svf = el.svf({"mode": "lowpass", "key": "f"}, 800.0, 2.0, x)
    dly = el.delay({"size": 1000, "key": "d"}, 400.25, 0.4, x)
    out.append(dict(name="baked_props_next_block", batch=el.render(svf, dly), n_blocks=8, n_out=2, exact=False, script={
        2: [[3, svf.id(), "mode", "highpass"]],
        4: [[3, dly.id(), "size", 600]],
        5: [[3, svf.id(), "mode", "notch"]]}))
    return out


def definition(sc):
    """What a scenario renders, as JSON-able data (the stored reference outputs are tied to it by digest)."""
    return {k: sc.get(k) for k in ("batch", "n_blocks", "n_out", "sample_times")} | {"script": {str(b): v for b, v in sc["script"].items()}}


def render_live(cls, sc, sr=48000.0, bs=512):
    """A scenario on an oracle class: the script's batches applied before their blocks, [n_out, n_blocks * bs]."""
    r = cls(sr, bs)
    assert r.apply(sc["batch"]) == 0
    blocks = []
    for b in range(sc["n_blocks"]):
        if b in sc["script"]:
            assert r.apply(sc["script"][b]) == 0
        if sc.get("sample_times"):
            r.set_current_time(sc["sample_times"][b])
        blocks.append(r.process(None, sc["n_out"], bs))
    return np.concatenate(blocks, axis=1)
