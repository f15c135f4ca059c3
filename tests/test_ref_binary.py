"""oracle/_ref = the reference's OWN object code (its unmodified C sources compiled against the
shims in oracle/shim/ by oracle/Makefile.ref, where the reference's sources are present):

1. the reference's ten `make check` suites pass against it (needs the reference's sources) -> the shim is faithful;
2. the CPU oracle (our restatement) agrees with it on seeded synthetic streams (needs the binary) -> the oracle is
   pinned against the reference itself, not only against its test fixtures;
3. on every machine, the oracle reproduces what (2) compares, as stored in tests/golden/streams.json
   (tests/golden/make_golden_streams.py).  Where (2) runs too, the stored data is checked against the reference.
"""
import gzip
import hashlib
import json
import os
import re
import subprocess

import numpy as np
import pytest

import samutil
from conftest import GOLDEN, REF_TESTS, REFERENCE, ROOT, needs_reference

REF_BIN = os.path.join(ROOT, "oracle", "_ref", "msamtools")


@pytest.fixture(scope="module")
def ref_bin():
    if REFERENCE:
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "-f", "Makefile.ref", "REF=" + REFERENCE])
    if not os.access(REF_BIN, os.X_OK):
        pytest.skip("no reference object code: oracle/_ref/msamtools is not built and the reference's sources are absent")
    return REF_BIN


@needs_reference
@pytest.mark.parametrize("suite", ["smoke", "filter", "besthit", "profile", "coverage", "integration", "qname_order",
                                   "errors", "streaming", "summary"])
def test_reference_suite_passes_on_ref_binary(ref_bin, suite, tmp_path):
    env = dict(os.environ, MSAMTOOLS=ref_bin, TMPDIR=str(tmp_path))
    r = subprocess.run(["sh", os.path.join(REF_TESTS, f"test_{suite}.sh")], env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


STREAMS = {"mixed": ("mixed", 40_000, 424242, {}),
           # second stream: few references, heavy clipping / indels, unmapped pairs, up to 12 occurrences per insert
           "clippy": ("community", 30_000, 7, dict(n_refs=12, ref_len_min=3_000, ref_len_max=9_000, clip_fraction=0.35, indel_fraction=0.25,
                                                  unmapped_fraction=0.06, shared_fraction=0.45, single_fraction=0.15, max_occ=12)),
           # third stream: a gene catalogue (10 000 short references, log-normal abundances, 30 % multi-mappers): the PropSharing loop
           # of the restatement against the reference's own over thousands of features and lists
           "catalog": ("catalog10k", 60_000, 2026, {})}


@pytest.fixture(scope="module", params=list(STREAMS))
def synth_stream(request):
    from msamtools_b200 import synth
    preset, nrec, seed, over = STREAMS[request.param]
    p = synth.make_params(preset, n_records=nrec, seed=seed, **over)
    raw, off, _ = synth.generate(p)
    tlen = synth.target_lengths(p)
    names = [f"ref{i:04d}" for i in range(len(tlen))]
    return request.param, raw, off, tlen, names


@pytest.fixture(scope="module")
def synth_bam(synth_stream, tmp_path_factory):
    _, raw, off, tlen, names = synth_stream
    path = str(tmp_path_factory.mktemp("synth") / "in.bam")
    samutil.write_bam(path, samutil.synth_header(names, tlen), names, tlen, raw)
    return (path,) + synth_stream[1:]


FILTERS = [(["-l", "80", "-p", "95", "-z", "80"], dict(l=80, p=95, z=80)),
           (["-l", "80", "-p", "95", "-z", "80", "--besthit"], dict(l=80, p=95, z=80, besthit=True)),
           (["--uniqhit"], dict(uniqhit=True)),
           (["--ppt", "-990"], dict(ppt=-990)),
           (["-p", "99", "-v", "-k"], dict(p=99, invert=True, keep_unmapped=True)),
           (["-l", "100", "--rescore", "--besthit"], dict(l=100, rescore=True, besthit=True))]
MODES = ["all", "equal", "proportional", "ignore"]
PRE_ARGV, PRE_OPTS = ["-l", "80", "-p", "95", "-z", "80", "--besthit"], dict(l=80, p=95, z=80, besthit=True)   # filter | profile


def _payload(bam_bytes):
    """record stream of an (uncompressed-BGZF) BAM"""
    import struct
    data = gzip.decompress(bam_bytes)
    l_text, = struct.unpack_from("<i", data, 4)
    o = 8 + l_text
    n_ref, = struct.unpack_from("<i", data, o); o += 4
    for _ in range(n_ref):
        ln, = struct.unpack_from("<i", data, o); o += 4 + ln + 4
    return data[o:]


# ---- one output of each command, from the reference's object code and from the oracle, in the same form
def reference_filter(ref_bin, path, argv):
    return _payload(subprocess.run([ref_bin, "filter", "-b", "-u"] + argv + [path], capture_output=True, check=True).stdout)


def oracle_filter(oracle, raw, off, opts):
    cfg = oracle.filter_cfg(**opts)
    return bytes(oracle.emit_records(raw, off, oracle.filter_stream(raw, off, cfg), cfg))


def reference_profile(ref_bin, path, names, mode, pre, outp):
    """the three insert counts of the table's comments, every feature's value as printed, and for proportional sharing the
    PropSharing iterations and purged inserts reported on stderr"""
    prof = [ref_bin, "profile", "--label", "x", "--unit", "ab", "--nolen", "--multi", mode, "-o", outp]
    if pre:
        f = subprocess.Popen([ref_bin, "filter", "-b", "-u"] + PRE_ARGV + [path], stdout=subprocess.PIPE)
        r = subprocess.run(prof + ["-"], stdin=f.stdout, capture_output=True, text=True)
        f.wait()
    else:
        r = subprocess.run(prof + [path], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    comments, body = samutil.read_profile_gz(outp)
    res = {}
    for key, label in (("mapped_inserts", "Mapped inserts"), ("multi", "- Multiple mapped "), ("uniq", "- Uniquely mapped ")):
        res[key] = int(next(l for l in comments if label in l).split(":")[1].split("(")[0])
    got = {k: v for k, v in body[1:]}
    res["values"] = [got[n] for n in names]
    if mode == "proportional":
        res["iterations"] = sum("PropSharing Iteration" in l for l in r.stderr.splitlines())
        m = re.search(r"Purged (\d+) inserts", r.stderr)
        res["purged"] = int(m.group(1)) if m else None
    return res


def oracle_profile(oracle, raw, off, n_targets, mode, pre):
    idx = oracle.filter_stream(raw, off, oracle.filter_cfg(**PRE_OPTS)) if pre else None
    ab, st, _, _ = oracle.profile(raw, off, idx, n_targets, {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}[mode])
    res = {"mapped_inserts": st["mapped_inserts"], "multi": st["multi"], "uniq": st["uniq"], "values": ["%.8g" % x for x in ab]}
    if mode == "proportional":
        res.update(iterations=st["iterations"], purged=st["purged"])
    return res


def reference_coverage(ref_bin, path, outp):
    subprocess.run([ref_bin, "coverage", "--summary", "-o", outp, path], check=True)
    with gzip.open(outp, "rt") as fh:
        return fh.read().splitlines()


def oracle_coverage(oracle, raw, off, tlen, names):
    cov, touched, total, _ = oracle.coverage(raw, off, None, tlen)
    return ["%s\t0\t0" % n if not cov[t] else "%s\t%.8f\t%.2f" % (n, touched[t] / int(tlen[t]), total[t] / int(tlen[t]))
            for t, n in enumerate(names)]


def stored_form(result):
    """What tests/golden/streams.json keeps of one output: record bytes as count, size and SHA-256; a list of printed rows
    as count, SHA-256 of the rows and 32 rows at seeded positions; the counters of a profile as they are."""
    if isinstance(result, bytes):
        return {"records": len(samutil.split_records(result)), "bytes": len(result), "sha256": hashlib.sha256(result).hexdigest()}
    if isinstance(result, dict):
        return {k: stored_form(v) if k == "values" else v for k, v in result.items()}
    pick = np.sort(np.random.default_rng(97).choice(len(result), min(32, len(result)), replace=False))
    return {"rows": len(result), "sha256": hashlib.sha256("\n".join(result).encode()).hexdigest(),
            "sample": {str(i): result[i] for i in pick}}


def filter_key(stream, argv):
    return f"{stream} | filter {' '.join(argv)}"


def profile_key(stream, mode, pre):
    return f"{stream} | {'filter | ' if pre else ''}profile --multi {mode}"


def coverage_key(stream):
    return f"{stream} | coverage --summary"


# ---- (2) the oracle against the reference's object code
@pytest.mark.parametrize("argv,opts", FILTERS, ids=lambda x: " ".join(x) if isinstance(x, list) else "")
def test_oracle_filter_equals_reference(ref_bin, oracle, synth_bam, argv, opts):
    path, raw, off, tlen, names = synth_bam
    assert reference_filter(ref_bin, path, argv) == oracle_filter(oracle, raw, off, opts)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("pre", [None, 1], ids=["plain", "filter|profile"])
def test_oracle_profile_equals_reference(ref_bin, oracle, synth_bam, mode, pre, tmp_path):
    path, raw, off, tlen, names = synth_bam
    assert reference_profile(ref_bin, path, names, mode, pre, str(tmp_path / "p.gz")) == oracle_profile(oracle, raw, off, len(tlen), mode, pre)


def test_oracle_coverage_equals_reference(ref_bin, oracle, synth_bam, tmp_path):
    path, raw, off, tlen, names = synth_bam
    assert reference_coverage(ref_bin, path, str(tmp_path / "c.gz")) == oracle_coverage(oracle, raw, off, tlen, names)


# ---- (3) the oracle against the stored outputs, everywhere
@pytest.fixture(scope="module")
def stored():
    with open(os.path.join(GOLDEN, "streams.json")) as fh:
        return json.load(fh)["outputs"]


@pytest.mark.parametrize("argv,opts", FILTERS, ids=lambda x: " ".join(x) if isinstance(x, list) else "")
def test_oracle_filter_equals_stored(oracle, stored, synth_stream, argv, opts):
    stream, raw, off, tlen, names = synth_stream
    assert stored_form(oracle_filter(oracle, raw, off, opts)) == stored[filter_key(stream, argv)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("pre", [None, 1], ids=["plain", "filter|profile"])
def test_oracle_profile_equals_stored(oracle, stored, synth_stream, mode, pre):
    stream, raw, off, tlen, names = synth_stream
    assert stored_form(oracle_profile(oracle, raw, off, len(tlen), mode, pre)) == stored[profile_key(stream, mode, pre)]


def test_oracle_coverage_equals_stored(oracle, stored, synth_stream):
    stream, raw, off, tlen, names = synth_stream
    assert stored_form(oracle_coverage(oracle, raw, off, tlen, names)) == stored[coverage_key(stream)]
