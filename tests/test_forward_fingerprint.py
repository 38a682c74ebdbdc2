"""The single-block forward driver takes the same decisions as when tests/golden/forward_fingerprint.json was
recorded: per case, every non-timing field of dark_bwt_stats (rounds, passes per round, active suffixes, kernel
launches, host round trips, ...) and the BWT's origin and CRC-32.  A change that alters the driver's control flow
on purpose regenerates the fixture with tests/golden/make_forward_fingerprint.py."""
import json
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_forward_fingerprint as F  # noqa: E402


def _fixture():
    with open(F.OUT) as f:
        return json.load(f)


def test_fixture_covers_every_case():
    assert sorted(_fixture()) == sorted(F.cases())


@pytest.mark.gpu
def test_forward_control_flow_matches_the_fixture():
    want = _fixture()
    got = F.collect()
    diffs = []
    for name in sorted(want):
        for k, (a, b) in enumerate(zip(want[name], got[name])):
            diffs += [f"{name}[{k}].{field}: {a[field]} -> {b.get(field)}" for field in a if a[field] != b.get(field)]
        if len(want[name]) != len(got[name]):
            diffs.append(f"{name}: {len(want[name])} records -> {len(got[name])}")
    assert not diffs, "\n".join(diffs[:60])
