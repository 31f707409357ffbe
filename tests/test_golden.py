"""The committed digests of the reference's output for every filter on the path (tests/golden/filters_golden.json, made
by tests/golden/make_filters_golden.py from the compiled reference) still describe what the reference produces here."""
import json
import sys
from pathlib import Path

import pytest

sys.path.insert(0, str(Path(__file__).parent / "golden"))
from filter_cases import FMT, cases, digest  # noqa: E402
from reference_runs import DIGEST_HEX, frame_digests  # noqa: E402

GOLDEN = json.loads((Path(__file__).parent / "golden" / "filters_golden.json").read_text())
CASES = cases()


def test_golden_file_covers_every_case():
    assert sorted(GOLDEN) == sorted(CASES)
    for name, g in GOLDEN.items():
        assert len(g["sha256"]) == len(g["start"]) == len(g["combed"]) > 0


@pytest.mark.parametrize("name", sorted(CASES))
def test_reference_matches_golden(ref, name):
    c, g = CASES[name], GOLDEN[name]
    r = ref.run(c["ref"], c["settings"], c["clip"], FMT[c["depth"]], c["w"], c["h"], flags=c["flags"], combed=c["combed"])
    assert r.start.tolist() == g["start"] and r.combed.tolist() == g["combed"]
    assert frame_digests(r.frames) == [d[:DIGEST_HEX] for d in g["sha256"]]


@pytest.mark.parametrize("name", sorted(CASES))
def test_host_filters_match_golden(name):
    """the product's host-side filter objects (same names as on the GPU) over the plain-C stand-ins for the device calls
    (oracle/_ref/libhostlogic.so, see tests/test_hostlogic.py): the committed digests again, chains included"""
    from handbrake_b200.hblib import FilterLib
    from test_hostlogic import HOSTLOGIC_SO
    if not HOSTLOGIC_SO.exists():
        pytest.skip("oracle/_ref/libhostlogic.so not built")
    c, g = CASES[name], GOLDEN[name]
    r = FilterLib(HOSTLOGIC_SO).run(c["cuda"], c["settings"], c["clip"], FMT[c["depth"]], c["w"], c["h"], flags=c["flags"], combed=c["combed"])
    assert not r.init_failed and r.saw_eof
    d = digest(r)
    assert d["start"] == g["start"] and d["combed"] == g["combed"] and d["sha256"] == g["sha256"]
