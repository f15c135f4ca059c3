"""Pins the CPU oracle against the expected values written in the reference's OWN test
scripts, on the reference's own fixtures (tests/fixtures/*.sam and tests/tiny_aln.bam of
msamtools v1.1.3, stored as record streams in tests/golden/fixtures.npz).

Every expected string below is restated from the cited reference test, not computed here.
"""
import numpy as np
import pytest

import goldenutil as G
import samutil

# tests/test_filter.sh:15
ALL_MAPPED = ("clip80:0,clip90:0,del99:0,id97:0,id98:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,pairX:129,"
              "perfect100:0,secondary98:256,supp98:2048")

# (options, expected QNAME:FLAG list) -- tests/test_filter.sh:34-132
FILTER_CASES = [
    (dict(l=79), ALL_MAPPED),
    (dict(l=80), ALL_MAPPED),
    (dict(l=81), "clip90:0,del99:0,id97:0,id98:0,ins99:0,md99:0,md_precedence:0,pairX:65,pairX:129,perfect100:0,secondary98:256,supp98:2048"),
    (dict(l=100), "del99:0,id97:0,id98:0,ins99:0,md99:0,md_precedence:0,pairX:65,pairX:129,perfect100:0,secondary98:256,supp98:2048"),
    (dict(p=97), ALL_MAPPED),
    (dict(p=98), "clip80:0,clip90:0,del99:0,id98:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,perfect100:0,secondary98:256,supp98:2048"),
    (dict(p=99), "clip80:0,clip90:0,del99:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,perfect100:0"),
    (dict(p=100), "clip80:0,clip90:0,len80:0,md_precedence:0,pairX:65,perfect100:0"),
    (dict(ppt=980), "clip80:0,clip90:0,del99:0,id98:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,perfect100:0,secondary98:256,supp98:2048"),
    (dict(ppt=-980), "id97:0,id98:0,pairX:129,secondary98:256,supp98:2048"),
    (dict(z=80), ALL_MAPPED),
    (dict(z=90), "clip90:0,del99:0,id97:0,id98:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,pairX:129,perfect100:0,secondary98:256,supp98:2048"),
    (dict(z=91), "del99:0,id97:0,id98:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,pairX:129,perfect100:0,secondary98:256,supp98:2048"),
    (dict(l=100, p=99), "del99:0,ins99:0,md99:0,md_precedence:0,pairX:65,perfect100:0"),
    (dict(l=90, z=91), "del99:0,id97:0,id98:0,ins99:0,md99:0,md_precedence:0,pairX:65,pairX:129,perfect100:0,secondary98:256,supp98:2048"),
    (dict(p=99, z=91), "del99:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,perfect100:0"),
    (dict(l=100, p=99, z=91), "del99:0,ins99:0,md99:0,md_precedence:0,pairX:65,perfect100:0"),
    (dict(p=99, invert=True), "id97:0,id98:0,pairX:129,secondary98:256,supp98:2048"),
    (dict(p=99, invert=True, keep_unmapped=True), "id97:0,id98:0,pairX:129,secondary98:256,supp98:2048,unmapped:4"),
    (dict(p=98, rescore=True), "clip80:0,clip90:0,del99:0,id98:0,ins99:0,len80:0,md99:0,md_precedence:0,pairX:65,perfect100:0,secondary98:256,supp98:2048"),
]

# tests/test_filter.sh:183-197 on cigar_eqx.sam
EQX_CASES = [
    (dict(p=98), "md_eqx100:0,md_eqx98:0,md_m100:0,md_m98:0"),
    (dict(l=100), "md_eqx100:0,md_eqx98:0,md_m100:0,md_m98:0"),
    (dict(z=90), "md_eqx0:0,md_eqx100:0,md_eqx98:0,md_m0:0,md_m100:0,md_m98:0,nm_eqx90:256,nm_m90:256"),
]

# tests/test_besthit.sh:32-83
BESTHIT_CASES = [
    ("besthit.sam", dict(besthit=True),
     "filterwin:0,interleaved:65,interleaved:385,interleaved_tie:65,interleaved_tie:321,interleaved_tie:129,paired:321,paired:129,"
     "same_ref:256,single:0,tie2:0,tie2:256,tie3:0,tie3:256,unique2:256,unique3:256"),
    ("besthit.sam", dict(uniqhit=True),
     "filterwin:0,interleaved:65,interleaved:385,interleaved_tie:129,paired:321,paired:129,same_ref:256,single:0,unique2:256,unique3:256"),
    ("besthit.sam", dict(p=95, besthit=True),
     "filterwin:256,interleaved:65,interleaved:385,interleaved_tie:65,interleaved_tie:321,interleaved_tie:129,paired:321,paired:129,"
     "same_ref:256,single:0,tie2:0,tie2:256,tie3:0,tie3:256,unique2:256,unique3:256"),
    ("besthit_rescore.sam", dict(besthit=True), "rescore:0"),
    ("besthit_rescore.sam", dict(l=1, rescore=True, besthit=True), "rescore:256"),
    ("besthit_rescore.sam", dict(rescore=True, besthit=True), "rescore:256"),
    ("besthit_rescore.sam", dict(rescore=True, uniqhit=True), "rescore:256"),
]


def _run_filter(oracle, sam, **opts):
    cfg = oracle.filter_cfg(**opts)
    return oracle.filter_stream(sam.raw, sam.off, cfg), cfg


@pytest.mark.parametrize("opts,expected", FILTER_CASES)
def test_filter_fixture(oracle, opts, expected):
    sam = G.fixture("filter")
    idx, _ = _run_filter(oracle, sam, **opts)
    assert sam.name_flags(idx) == expected


@pytest.mark.parametrize("opts,expected", EQX_CASES)
def test_cigar_eqx_fixture(oracle, opts, expected):
    sam = G.fixture("cigar_eqx")
    idx, _ = _run_filter(oracle, sam, **opts)
    assert sam.name_flags(idx) == expected


def _aux_text(rec, tag):
    """value of an integer aux field in an emitted BAM record (or None)"""
    import struct
    lq = rec[12]; nc, = struct.unpack_from("<H", rec, 16); ls, = struct.unpack_from("<i", rec, 20)
    p = 36 + lq + 4 * nc + (ls + 1) // 2 + ls
    while p + 3 <= len(rec):
        t, ty = rec[p:p + 2].decode(), chr(rec[p + 2]); p += 3
        sz = {"A": 1, "c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}.get(ty)
        if sz:
            if t == tag:
                fmt = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I"}[ty]
                return struct.unpack_from(fmt, rec, p)[0]
            p += sz
        elif ty in "ZH":
            e = rec.index(b"\0", p); p = e + 1
        else:
            return None
    return None


def test_filter_rescore_values(oracle):
    # tests/test_filter.sh:153-163: id98 -> AS:i:96, md_precedence -> AS:i:100
    sam = G.fixture("filter")
    idx, cfg = _run_filter(oracle, sam, p=98, rescore=True)
    recs = samutil.split_records(oracle.emit_records(sam.raw, sam.off, idx, cfg))
    by_name = {sam.record_fields(int(i))[0]: r for i, r in zip(idx, recs)}
    assert _aux_text(by_name["id98"], "AS") == 96
    assert _aux_text(by_name["md_precedence"], "AS") == 100
    # MD precedence: NM:i:10 is still in the record (tests/test_filter.sh:120-123)
    assert _aux_text(by_name["md_precedence"], "NM") == 10


@pytest.mark.parametrize("fixture,opts,expected", BESTHIT_CASES)
def test_besthit_fixture(oracle, fixture, opts, expected):
    sam = G.fixture(fixture.replace(".sam", ""))
    idx, cfg = _run_filter(oracle, sam, **opts)
    assert sam.name_flags(idx) == expected
    if opts.get("rescore"):
        # tests/test_besthit.sh:66-76: winning record carries AS:i:100
        rec = samutil.split_records(oracle.emit_records(sam.raw, sam.off, idx, cfg))[0]
        assert _aux_text(rec, "AS") == 100


@pytest.mark.parametrize("opts", [dict(besthit=True), dict(p=90, besthit=True)])
def test_long_qname_besthit(oracle, opts):
    # tests/test_besthit.sh:85-128: one winner per complete 127/128/254-char QNAME
    sam = G.fixture("long_qname")
    idx, _ = _run_filter(oracle, sam, **opts)
    got = [(len(sam.record_fields(int(i))[0]), sam.record_fields(int(i))[1], sam.ref_names[sam.record_fields(int(i))[2]]) for i in idx]
    assert got == [(127, 0, "A"), (128, 0, "A"), (254, 0, "A"), (254, 0, "B")]


# tests/test_profile.sh:49-67 : (mode, Unknown, A, B) with --total 7 --unit ab --nolen
PROFILE_CASES = [("all", 0, 6, 2), ("equal", 0, 5.5, 1.5), ("ignore", 1, 5, 1), ("proportional", 0, 5.833333333333, 1.166666666667)]


@pytest.mark.parametrize("mode,unknown,a,b", PROFILE_CASES)
def test_profile_fixture(oracle, mode, unknown, a, b):
    sam = G.fixture("profile")
    share = {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}[mode]
    ab, st, _, _ = oracle.profile(sam.raw, sam.off, None, len(sam.ref_names), share)
    assert (st["mapped_inserts"], st["multi"], st["uniq"]) == (7, 1, 6)             # test_profile.sh:38-46
    # Unknown = total - mapped + purged (+ multi when ignoring), msam_profile.c:912-917
    unk = 7 - st["mapped_inserts"] + st["purged"] + (st["multi"] if mode == "ignore" else 0)
    assert unk == unknown
    assert abs(ab[0] - a) <= 1e-6 and abs(ab[1] - b) <= 1e-6


def test_profile_long_qname(oracle):
    # tests/test_profile.sh:69-97
    sam = G.fixture("long_qname")
    ab, st, _, _ = oracle.profile(sam.raw, sam.off, None, len(sam.ref_names), 2)
    assert (st["mapped_inserts"], st["multi"], st["uniq"]) == (4, 4, 0)
    assert abs(ab[0] - 2) <= 1e-9 and abs(ab[1] - 2) <= 1e-9


@pytest.mark.parametrize("fixture", ["profile_empty.sam", "profile_unmapped.sam"])
def test_profile_zero(oracle, fixture):
    # tests/test_profile.sh:99-137
    sam = G.fixture(fixture.replace(".sam", ""))
    ab, st, _, _ = oracle.profile(sam.raw, sam.off, None, len(sam.ref_names), 2)
    assert (st["mapped_inserts"], st["multi"], st["uniq"]) == (0, 0, 0)
    assert not ab.any()


def test_profile_fractional(oracle):
    # tests/test_profile.sh:139-160: equal sharing -> A 1.3333 B 1.3333 C 0.3333
    sam = G.fixture("profile_fractional_mincount")
    ab, st, _, _ = oracle.profile(sam.raw, sam.off, None, len(sam.ref_names), 2)
    assert np.allclose(ab[:3], [4 / 3, 4 / 3, 1 / 3], atol=1e-6)


def test_coverage_fixture(oracle):
    # tests/test_coverage.sh:28-62
    sam = G.fixture("coverage")
    cov, touched, total, depth = oracle.coverage(sam.raw, sam.off, None, sam.target_len, want_depth=True)
    assert depth[0].tolist() == [1, 0, 1, 1, 2, 2, 1, 0, 0, 1]
    assert depth[1].tolist() == [0] * 5
    assert depth[2].tolist() == [0] * 9 + [1]
    assert depth[3].tolist() == [4, 4, 2, 4, 3, 0, 0, 0]
    assert cov.tolist() == [1, 0, 1, 1]
    lines = []
    for t, name in enumerate(sam.ref_names):
        tl = int(sam.target_len[t])
        lines.append("%s\t0\t0" % name if not cov[t] else "%s\t%.8f\t%.2f" % (name, touched[t] / tl, total[t] / tl))
    assert lines == ["A\t0.70000000\t0.90", "B\t0\t0", "C\t0.10000000\t0.10", "D\t0.62500000\t2.12"]


def test_integration(oracle):
    # tests/test_integration.sh:38-72: filter -p 95 | profile --multi equal
    sam = G.fixture("integration")
    ab, st, _, _ = oracle.profile(sam.raw, sam.off, None, 2, 2)
    assert (st["multi"], st["uniq"]) == (2, 2) and np.allclose(ab, [2, 2], atol=1e-9)
    idx, _ = _run_filter(oracle, sam, p=95)
    assert sam.name_flags(idx) == "filter_to_b:256,multi:0,multi:256,uA:0,uB:0"
    ab, st, _, _ = oracle.profile(sam.raw, sam.off, idx, 2, 2)
    assert (st["multi"], st["uniq"]) == (1, 3) and np.allclose(ab, [1.5, 2.5], atol=1e-9)


def test_tiny_aln_config1(oracle):
    # BASELINE.json configs[0]: filter -l 80 -p 95 -z 80 --besthit | profile --multi=proportional
    sam = G.fixture("tiny_aln")
    assert sam.n == 16 and len(sam.ref_names) == 2924
    idx, _ = _run_filter(oracle, sam, l=80, p=95, z=80, besthit=True)
    assert len(idx) == 14
    ab, st, _, _ = oracle.profile(sam.raw, sam.off, idx, len(sam.ref_names), 3)
    assert (st["mapped_inserts"], st["uniq"], st["multi"], st["purged"]) == (7, 4, 3, 3)
    assert st["iterations"] == 1 and st["converged"] == 1 and st["delta"][0] == 0
    assert sorted(sam.ref_names[i] for i in np.nonzero(ab)[0]) == sorted(
        ["MH0349_GL0038880", "MH0013_GL0018062", "479436.Vpar_1233", "MH0002_GL0008419"])
    assert set(ab[np.nonzero(ab)[0]].tolist()) == {1.0}
