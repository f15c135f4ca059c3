#!/usr/bin/env python
"""Generates tests/golden/fixtures.npz + cases.json from a checkout of the reference's sources (MSAMTOOLS_REFERENCE, else
BASELINE.json's reference_path):

    python tests/golden/make_golden.py

Inputs are the reference's own test fixtures (tests/fixtures/*.sam, tests/tiny_aln.bam of that
checkout), re-encoded as raw BAM record streams (the C-ABI input layout).  Expected
outputs are (a) the strings the reference's test scripts assert (restated with citations in
tests/test_oracle_golden.py, which asserts them again) and (b) the outputs of the pinned CPU
oracle, which (a) pins.  The reference's object code itself is not run here: its outputs on
seeded synthetic streams are what tests/golden/make_golden_streams.py stores.  The tests read
these files, so they need no reference checkout.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import samutil                                    # noqa: E402
from oracle import oracle as orc                  # noqa: E402
import test_oracle_golden as T                    # noqa: E402

REF = os.path.join(orc.reference_dir(), "tests")
FIXTURES = ["filter", "cigar_eqx", "besthit", "besthit_rescore", "long_qname", "profile", "profile_empty",
            "profile_unmapped", "profile_fractional_mincount", "coverage", "integration", "qname_coordinate", "qname_reopened"]


def main():
    orc.build()
    arrays, cases = {}, []
    sams = {}
    for name in FIXTURES:
        sams[name] = samutil.read_sam(os.path.join(REF, "fixtures", name + ".sam"))
    sams["tiny_aln"] = samutil.read_bam(os.path.join(REF, "tiny_aln.bam"))
    for name, s in sams.items():
        arrays[name + ".raw"] = s.raw
        arrays[name + ".off"] = s.off
        arrays[name + ".tlen"] = s.target_len
        arrays[name + ".names"] = np.array(s.ref_names, dtype="U")
        arrays[name + ".header"] = np.array([l for l in s.header_lines if not l.startswith("@SQ")], dtype="U")

    def filt(fixture, opts, expected=None, src=""):
        s = sams[fixture]
        cfg = orc.filter_cfg(**opts)
        idx = orc.filter_stream(s.raw, s.off, cfg)
        nf = s.name_flags(idx)
        if expected is not None:
            assert nf == expected, (fixture, opts, nf, expected)
        st = orc.record_stats(s.raw, s.off)
        rec = orc.emit_records(s.raw, s.off, idx, cfg)
        cases.append(dict(kind="filter", fixture=fixture, opts=opts, src=src, kept=idx.tolist(), name_flags=nf,
                          records_hex=bytes(rec).hex(),
                          stats={k: st[k].tolist() for k in ("alen", "qlen", "qclip", "edit", "score", "has_as", "has_tag")}))

    for opts, exp in T.FILTER_CASES:
        filt("filter", opts, exp, "tests/test_filter.sh:34-163")
    for opts, exp in T.EQX_CASES:
        filt("cigar_eqx", opts, exp, "tests/test_filter.sh:183-197")
    for fx, opts, exp in T.BESTHIT_CASES:
        filt(fx.replace(".sam", ""), opts, exp, "tests/test_besthit.sh:32-83")
    for opts in (dict(besthit=True), dict(p=90, besthit=True), dict(uniqhit=True)):
        filt("long_qname", opts, None, "tests/test_besthit.sh:85-128")
    filt("integration", dict(p=95), "filter_to_b:256,multi:0,multi:256,uA:0,uB:0", "tests/test_integration.sh:49-60")
    filt("tiny_aln", dict(l=80, p=95, z=80, besthit=True), None, "BASELINE.json configs[0]")
    filt("tiny_aln", dict(l=80, p=95, z=80), None, "BASELINE.json configs[0] (no besthit)")
    filt("tiny_aln", dict(uniqhit=True), None, "BASELINE.json configs[0] (uniqhit only)")

    def prof(fixture, mode, pre=None, src=""):
        s = sams[fixture]
        idx = None
        if pre is not None:
            idx = orc.filter_stream(s.raw, s.off, orc.filter_cfg(**pre))
        share = {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}[mode]
        ab, st, ui, d = orc.profile(s.raw, s.off, idx, len(s.ref_names), share)
        nz = np.nonzero((ab != 0) | (ui != 0) | (d != 0))[0]
        cases.append(dict(kind="profile", fixture=fixture, mode=mode, pre=pre, src=src, stats=st, n=len(ab), nz=nz.tolist(),
                          abundance=ab[nz].tolist(), ui=ui[nz].tolist(), d=d[nz].tolist()))

    for mode in ("all", "equal", "ignore", "proportional"):
        prof("profile", mode, None, "tests/test_profile.sh:49-67")
        prof("long_qname", mode, None, "tests/test_profile.sh:69-97")
        prof("profile_fractional_mincount", mode, None, "tests/test_profile.sh:139-173")
        prof("integration", mode, None, "tests/test_integration.sh:38-45")
        prof("integration", mode, dict(p=95), "tests/test_integration.sh:62-72")
        prof("tiny_aln", mode, dict(l=80, p=95, z=80, besthit=True), "BASELINE.json configs[0]")
        prof("tiny_aln", mode, None, "tiny_aln.bam plain profile")
        prof("besthit", mode, dict(besthit=True), "besthit.sam | profile")
    for fx in ("profile_empty", "profile_unmapped"):
        prof(fx, "equal", None, "tests/test_profile.sh:99-137")

    def cov(fixture, pre=None, src=""):
        s = sams[fixture]
        idx = None
        if pre is not None:
            idx = orc.filter_stream(s.raw, s.off, orc.filter_cfg(**pre))
        c, t, sm, depth = orc.coverage(s.raw, s.off, idx, s.target_len, want_depth=len(s.ref_names) < 50)
        nz = np.nonzero(c)[0]
        cases.append(dict(kind="coverage", fixture=fixture, pre=pre, src=src, n=len(c), nz=nz.tolist(), touched=t[nz].tolist(),
                          sum=sm[nz].tolist(), depth=None if depth is None else [d.tolist() for d in depth]))

    cov("coverage", None, "tests/test_coverage.sh:28-81")
    cov("filter", dict(p=98), "filter.sam | coverage")
    cov("besthit", dict(besthit=True), "besthit.sam --besthit | coverage")
    cov("tiny_aln", dict(l=80, p=95, z=80), "BASELINE.json configs[3] shape on tiny_aln")

    np.savez_compressed(os.path.join(HERE, "fixtures.npz"), **arrays)
    with open(os.path.join(HERE, "cases.json"), "w") as fh:
        json.dump(cases, fh)
    print(f"wrote {len(arrays)} arrays, {len(cases)} cases")


if __name__ == "__main__":
    main()
