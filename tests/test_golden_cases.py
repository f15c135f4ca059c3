"""CPU: the oracle must reproduce every committed golden case (tests/golden/), so the bundle the
GPU parity tests rely on cannot drift from the pinned oracle.  Runs everywhere (no GPU, no
reference sources)."""
import numpy as np
import pytest

import goldenutil as G

SHARE = {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}


@pytest.mark.parametrize("c", G.cases("filter"), ids=G.case_id)
def test_filter_case(oracle, c):
    s = G.fixture(c["fixture"])
    cfg = oracle.filter_cfg(**c["opts"])
    idx = oracle.filter_stream(s.raw, s.off, cfg)
    assert idx.tolist() == c["kept"]
    assert s.name_flags(idx) == c["name_flags"]
    assert bytes(oracle.emit_records(s.raw, s.off, idx, cfg)).hex() == c["records_hex"]
    st = oracle.record_stats(s.raw, s.off)
    for k, v in c["stats"].items():
        assert st[k].tolist() == v, k


@pytest.mark.parametrize("c", G.cases("profile"), ids=G.case_id)
def test_profile_case(oracle, c):
    s = G.fixture(c["fixture"])
    idx = None if c["pre"] is None else oracle.filter_stream(s.raw, s.off, oracle.filter_cfg(**c["pre"]))
    ab, st, ui, d = oracle.profile(s.raw, s.off, idx, len(s.ref_names), SHARE[c["mode"]])
    assert st == c["stats"]
    assert ui.tolist() == G.dense(c, "ui", np.uint32).tolist()
    assert np.array_equal(ab, G.dense(c, "abundance", np.float64))


@pytest.mark.parametrize("c", G.cases("coverage"), ids=G.case_id)
def test_coverage_case(oracle, c):
    s = G.fixture(c["fixture"])
    idx = None if c["pre"] is None else oracle.filter_stream(s.raw, s.off, oracle.filter_cfg(**c["pre"]))
    cov, touched, total, depth = oracle.coverage(s.raw, s.off, idx, s.target_len, want_depth=c["depth"] is not None)
    assert np.nonzero(cov)[0].tolist() == c["nz"]
    assert touched.tolist() == G.dense(c, "touched", np.int64).tolist()
    assert total.tolist() == G.dense(c, "sum", np.int64).tolist()
    if c["depth"] is not None:
        assert [x.tolist() for x in depth] == c["depth"]
