#!/usr/bin/env python
"""Generates tests/golden/streams.json: what tests/test_ref_binary.py compares between the CPU oracle and the reference's
object code on its three seeded synthetic streams (every filter of FILTERS, every --multi mode plain and after
`filter ... --besthit`, coverage --summary), in the reduced form of test_ref_binary.stored_form.

    python tests/golden/make_golden_streams.py

The outputs are those of the reference's object code (oracle/_ref/msamtools) when it is built or can be built from the
reference's sources (MSAMTOOLS_REFERENCE, else BASELINE.json's reference_path), else those of the CPU oracle; "source"
in the file says which.  test_oracle_*_equals_stored check the oracle against the file on every machine; wherever the
reference's object code exists, test_oracle_*_equals_reference check the oracle against it on the same streams, so the
file is checked against the reference there too.  That binary links this project's host I/O (bamio.c, finflate.c,
crc32x.c, margs.c), so a BAM-decode or inflate bug in those files would show up on both sides of the comparison.
"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import samutil                                    # noqa: E402
from msamtools_b200 import synth                  # noqa: E402
from oracle import oracle as orc                  # noqa: E402
import test_ref_binary as T                       # noqa: E402


def main():
    orc.build()
    ref = orc.reference_dir()
    if ref:
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "-f", "Makefile.ref", "REF=" + ref])
    use_ref = os.access(T.REF_BIN, os.X_OK)
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for stream, (preset, nrec, seed, over) in T.STREAMS.items():
            p = synth.make_params(preset, n_records=nrec, seed=seed, **over)
            raw, off, _ = synth.generate(p)
            tlen = synth.target_lengths(p)
            names = [f"ref{i:04d}" for i in range(len(tlen))]
            path = os.path.join(d, "in.bam")
            samutil.write_bam(path, samutil.synth_header(names, tlen), names, tlen, raw)
            for argv, opts in T.FILTERS:
                res = T.reference_filter(T.REF_BIN, path, argv) if use_ref else T.oracle_filter(orc, raw, off, opts)
                out[T.filter_key(stream, argv)] = T.stored_form(res)
            for mode in T.MODES:
                for pre in (None, 1):
                    res = (T.reference_profile(T.REF_BIN, path, names, mode, pre, os.path.join(d, "p.gz")) if use_ref
                           else T.oracle_profile(orc, raw, off, len(tlen), mode, pre))
                    out[T.profile_key(stream, mode, pre)] = T.stored_form(res)
            res = T.reference_coverage(T.REF_BIN, path, os.path.join(d, "c.gz")) if use_ref else T.oracle_coverage(orc, raw, off, tlen, names)
            out[T.coverage_key(stream)] = T.stored_form(res)
    source = ("the reference's object code (oracle/_ref/msamtools: msamtools v1.1.3 sources, shim I/O)" if use_ref
              else "the CPU oracle (oracle/msam_oracle.c); the reference's object code was not available")
    with open(os.path.join(HERE, "streams.json"), "w") as fh:
        json.dump({"source": source, "outputs": out}, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(f"wrote {len(out)} outputs from {source}")


if __name__ == "__main__":
    main()
