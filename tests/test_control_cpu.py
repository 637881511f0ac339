"""CPU: the restatement (oracle/elem_oracle.cpp) against the reference engine on the LIVE-UPDATE scenarios of the sequencing /
control nodes (tests/control_common.py) — new sequence data, loop points, re-arming, host clock jumps, baked properties changed
between blocks.  Everything except transcendental-free paths must be bit-exact; the others agree to float rounding of libm-free
double arithmetic, i.e. exactly as well.  The reference's outputs are stored in tests/golden/reference_extra.npz."""
import numpy as np
import pytest

from control_common import definition, render_live, scenarios
from helpers import reference_extra, sha16
from oracle import oracle as orc

SR, BS = 48000.0, 512
SCEN = scenarios()
GOLD, META = reference_extra()


@pytest.mark.parametrize("sc", SCEN, ids=[s["name"] for s in SCEN])
def test_port_matches_reference_through_live_updates(sc):
    assert META["sha256_16"]["control_" + sc["name"]] == sha16(definition(sc)), "scenario changed: re-run tests/golden/make_ref_fixtures.py"
    got, want = render_live(orc.PortRuntime, sc), GOLD["control_" + sc["name"]]
    assert np.array_equal(got, want), f"{sc['name']}: max diff {np.abs(got - want).max()}"
    assert np.abs(want).max() > 0
