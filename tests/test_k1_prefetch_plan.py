"""CPU (plan-only runtime): what the host hands K1 for its latency-hiding paths — the word offset of the tap promotion records (-1 when a
program has none, so the kernel neither walks nor reads the program after its sample loop) and the k1_prefetch engine option."""
from elementary_b200 import Runtime, el, graphs

SR, BS = 48000.0, 512
OP_END, OP_PROMOTE, HDR = 0, 30, 8


def group(batch, **opts):
    rt = Runtime(SR, BS, 4, device=-1, **opts)
    assert rt.apply_instructions(batch) == 0, rt.last_error()
    return rt, rt.describe()["groups"][0]


def test_program_without_taps_has_no_promotion_records():
    _, g = group(graphs.subsynth32())
    assert g["promote_at"] == -1


def test_promotion_offset_points_behind_the_first_end():
    x = el.in_(0)
    batch = el.render(el.tap_out("a", el.add(el.tap_in("a"), x)), el.tap_out("b", el.mul(0.5, el.tap_in("b"), x)))
    rt, g = group(batch)
    at = g["promote_at"]
    words = rt.program_words(0)
    assert at > 0 and words[at] & 0xFF == OP_PROMOTE and words[at + HDR] & 0xFF == OP_PROMOTE
    pc = 0                                  # the walk the kernel no longer needs: the first OP_END sits right in front
    while words[pc] & 0xFF != OP_END:
        pc += HDR + ((int(words[pc]) >> 8) & 0xFF)
    assert pc + HDR == at


def test_k1_prefetch_option_is_accepted():
    for v in (0, 1):
        rt, g = group(graphs.subsynth32(), k1_prefetch=v)
        assert g["promote_at"] == -1
