"""Profiling input that is not grouped by QNAME: msg_config.collate / Context(collate=True) / `profile --collate`.

A collating context takes records in any order and groups them by QNAME on the device at the first finish.  Its results
must equal those of the same configuration without collate on the same records regrouped STABLY by QNAME (each read's
records contiguous, in their input order): integers exactly, f64 values within 1e-9 relative with the same PropSharing
iteration count.  The order of the groups does not matter (DESIGN.md §11), so the oracle here runs on `regroup(...)`,
which orders groups by first appearance.

CPU: the reorder / regroup helpers, the oracle's integers on a regrouped coordinate-ordered stream, and the CLI's
`profile --collate` against the null device (ASan/UBSan).  GPU (-m gpu): parity with the oracle on coordinate-ordered and
shuffled streams, identity with collate=0 on grouped input, and the edges (reads split over pushes, a read with 5 000
alignments, tid -1 reads, empty pushes, staged / pinned / device-resident chunks, forced hash collisions, error ordinals,
the CG placeholder, refused configurations), plus the CLI on a coordinate-sorted BGZF file.
"""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import edgeutil as E
import samutil
from conftest import ROOT
from edgeutil import M, N, S

REL = 1e-9
SHARE = {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}
gpu = pytest.mark.gpu


# ================================================================ stream helpers
def _core(raw, off):
    n = len(off) - 1
    tid = np.array([int.from_bytes(bytes(raw[int(off[i]) + 4:int(off[i]) + 8]), "little", signed=True) for i in range(n)])
    pos = np.array([int.from_bytes(bytes(raw[int(off[i]) + 8:int(off[i]) + 12]), "little", signed=True) for i in range(n)])
    flag = np.array([int(raw[int(off[i]) + 18]) | int(raw[int(off[i]) + 19]) << 8 for i in range(n)])
    return tid, pos, flag


def permute(raw, off, perm):
    """records in the order perm (perm[k] = input index of output record k)"""
    recs = E.split(raw, off)
    return E.stream([recs[int(i)] for i in perm])


def reorder(raw, off, how, seed=0):
    """(raw, off, perm): by (tid, pos) with unmapped / tid -1 records last ("coord"), a seeded shuffle ("shuffle"), or a
    given permutation (how = array)"""
    n = len(off) - 1
    if isinstance(how, str) and how == "coord":
        tid, pos, flag = _core(raw, off)
        unm = (tid < 0) | ((flag & 4) != 0)
        perm = np.lexsort((np.arange(n), pos, tid, unm))
    elif isinstance(how, str) and how == "shuffle":
        perm = np.random.default_rng(seed).permutation(n)
    else:
        perm = np.asarray(how, dtype=np.int64)
    r2, o2 = permute(raw, off, perm)
    return r2, o2, perm


def regroup(raw, off):
    """stable grouping by QNAME (bytes and length): groups in order of first appearance, records in input order"""
    recs = E.split(raw, off)
    first, order = {}, []
    for k, r in enumerate(recs):
        q = E.qname(r)
        if q not in first:
            first[q] = len(order); order.append([])
        order[first[q]].append(k)
    perm = [k for g in order for k in g]
    return permute(raw, off, perm)


def riffle(raw, off):
    """interleave the reads of a grouped stream, keeping each read's records in order and the reads' first records in
    read order: regroup() of the result is the input again"""
    recs = E.split(raw, off)
    g, key = -1, []
    for k, r in enumerate(recs):
        if k == 0 or E.qname(r) != E.qname(recs[k - 1]):
            g += 1; j = 0
        key.append((g + 3 * j, g, k)); j += 1
    return [k for _, _, k in sorted(key)]


def synth_stream(preset, n, seed):
    from msamtools_b200 import synth
    p = synth.make_params(preset, n_records=n, seed=seed)
    raw, off, _ = synth.generate(p)
    return np.ascontiguousarray(raw[:int(off[-1])]), off.copy(), synth.target_lengths(p)


# ================================================================ CPU
@pytest.mark.parametrize("preset,seed", [("mixed", 3), ("community", 5)])
def test_regroup_restores_grouped_stream(preset, seed):
    raw, off, _ = synth_stream(preset, 6000, seed)
    r2, o2, perm = reorder(raw, off, riffle(raw, off))
    assert not np.array_equal(perm, np.arange(len(perm)))
    g, go = regroup(r2, o2)
    assert bytes(g) == bytes(raw) and np.array_equal(go, off)
    # coordinate order and a shuffle: every read comes back whole, its records in their order in the reordered stream
    for how in ("coord", "shuffle"):
        r3, o3, perm3 = reorder(raw, off, how, seed=seed)
        g3, go3 = regroup(r3, o3)
        recs, out = E.split(raw, off), E.split(g3, go3)
        assert sorted(out) == sorted(recs)
        pos_in = {}
        for k, i in enumerate(perm3):
            pos_in.setdefault(E.qname(recs[i]), []).append(k)
        rank = 0
        for k in range(len(out)):
            if k == 0 or E.qname(out[k]) != E.qname(out[k - 1]):
                rank = 0
            assert out[k] == recs[perm3[pos_in[E.qname(out[k])][rank]]]
            rank += 1


def test_oracle_integers_same_on_regrouped_coordinate_order(oracle):
    raw, off, tl = synth_stream("mixed", 20000, 17)
    r2, o2, _ = reorder(raw, off, "coord")
    g, go = regroup(r2, o2)
    T = len(tl)
    cfg = oracle.filter_cfg(l=80, p=95, z=80, besthit=True)
    k1, k2 = oracle.filter_stream(raw, off, cfg), oracle.filter_stream(g, go, cfg)
    assert len(k1) == len(k2)
    a1, s1, u1, d1 = oracle.profile(raw, off, k1, T, SHARE["proportional"])
    a2, s2, u2, d2 = oracle.profile(g, go, k2, T, SHARE["proportional"])
    for key in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "n_lists", "n_entries"):
        assert s1[key] == s2[key], key
    assert np.array_equal(u1, u2)
    assert np.allclose(a1, a2, rtol=REL, atol=0)
    c1 = oracle.coverage(raw, off, k1, tl)
    c2 = oracle.coverage(g, go, k2, tl)
    for x, y in zip(c1[:3], c2[:3]):
        assert np.array_equal(x, y)


# ---------------------------------------------------------------- CLI on the null device
@pytest.fixture(scope="module")
def nullcli(tmp_path_factory):
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_cli_host_nulldev as H
    os.environ["ASAN_OPTIONS"] = "detect_leaks=0"
    return H.build(str(tmp_path_factory.mktemp("nulldev_collate")), "address,undefined")


def _coord_bam(path, n, seed, level=1):
    raw, off, tl = synth_stream("mixed", n, seed)
    r2, o2, _ = reorder(raw, off, "coord")
    names = [f"seq{i:03d}" for i in range(len(tl))]
    samutil.write_bam(path, samutil.synth_header(names, tl, so="coordinate"), names, tl, r2, level=level)
    return raw, off, r2, o2, tl, names


def test_cli_profile_collate_on_coordinate_sorted_bam_nulldev(nullcli, tmp_path):
    path = str(tmp_path / "coord.bam")
    _coord_bam(path, 30000, 23)
    out = str(tmp_path / "p.gz")
    r = subprocess.run([nullcli, "profile", "--collate", "--label", "x", "-o", out, path], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    comments, _ = samutil.read_profile_gz(out)
    assert any("QNAME grouping check: not required for this operation" in c for c in comments)
    r = subprocess.run([nullcli, "profile", "--label", "x", "-o", str(tmp_path / "q.gz"), path], capture_output=True)
    assert r.returncode != 0
    assert b"Please name-sort the input" in r.stdout + r.stderr


# ================================================================ GPU
@pytest.fixture(scope="module")
def m():
    import msamtools_b200 as mod
    assert mod._lib.load().msg_device_count() > 0, "no CUDA device: the GPU tests must not silently pass"
    return mod


def close(a, b, rel=REL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.all(np.abs(a - b) <= rel * np.maximum(np.abs(a), np.abs(b)))


def run_gpu(m, raw, off, cfg, chunks=None, how="staged", **kw):
    """push the stream (in `chunks` record ranges, default one push) and finish; returns profile / coverage results"""
    tl = kw.pop("target_len", None)
    if cfg.get("collate"):
        cfg = dict(cfg, kept=False)                      # a collating context has no per-chunk kept list
    ctx = m.Context(**cfg, **kw, target_len=tl)
    n = len(off) - 1
    bounds = chunks if chunks is not None else [(0, n)]
    held = []
    try:
        for lo, hi in bounds:
            o = (off[lo:hi + 1] - off[lo]).astype(np.uint64)
            r = np.ascontiguousarray(raw[int(off[lo]):int(off[hi])])
            if how == "staged":
                ctx.push(r, o)
            elif how == "pinned":
                pb = m.PinnedBuffer(max(len(r), 16))
                held.append(pb)
                a = pb.array[:len(r)]
                a[:] = r
                ctx.push(a, o)
            else:
                d_raw = ctx.device_alloc(max(len(r), 16)); d_off = ctx.device_alloc(len(o) * 8)
                held.append((d_raw, d_off))
                if len(r):
                    ctx.device_upload(d_raw, r)
                ctx.device_upload(d_off, o)
                ctx.push_device(d_raw, len(r), d_off, hi - lo)
        out = {}
        if cfg.get("profile"):
            ab, st = ctx.finish_profile()
            out["ab"], out["st"] = ab, st
            out["ui"] = ctx.pull_counts()[0]
        if cfg.get("coverage"):
            out["cov"] = ctx.finish_coverage()
            if not cfg.get("coverage_summary"):
                out["depth"] = [ctx.pull_coverage(t) for t in range(len(tl))]
        out["timing"] = ctx.timing()
        return out
    finally:
        for h in held:
            if isinstance(h, tuple):
                ctx.device_free(h[0]); ctx.device_free(h[1])
        ctx.close()
        for h in held:
            if not isinstance(h, tuple):
                h.close()


def expect_equal(a, b, what=""):
    if "st" in a:
        sa, sb = a["st"], b["st"]
        for k in ("mapped_inserts", "uniq_mapper_count", "multi_mapper_count", "purged_insert_count", "em_iterations", "multi_lists", "multi_entries"):
            assert sa[k] == sb[k], (what, k, sa[k], sb[k])
        assert np.array_equal(a["ui"], b["ui"]), what
        assert close(a["ab"], b["ab"]), what
    if "cov" in a:
        for x, y in zip(a["cov"], b["cov"]):
            assert np.array_equal(x, y), what
    if "depth" in a:
        for x, y in zip(a["depth"], b["depth"]):
            assert np.array_equal(x, y), what


def oracle_result(orc, raw, off, cfg, tl, fmap=None, n_features=None):
    fkw = {k: cfg[k] for k in ("l", "p", "z", "besthit", "uniqhit") if k in cfg}
    idx = orc.filter_stream(raw, off, orc.filter_cfg(**fkw)) if fkw else None
    out = {}
    if cfg.get("profile"):
        ab, st, ui, _ = orc.profile(raw, off, idx, len(tl), SHARE[cfg.get("multi", "proportional")], fmap=fmap, n_features=n_features)
        out["ab"], out["ui"] = ab, ui
        out["st"] = dict(mapped_inserts=st["mapped_inserts"], uniq_mapper_count=st["uniq"], multi_mapper_count=st["multi"],
                         purged_insert_count=st["purged"] if cfg.get("multi", "proportional") == "proportional" else 0,
                         em_iterations=st["iterations"] if cfg.get("multi", "proportional") == "proportional" else 0,
                         multi_lists=st["n_lists"], multi_entries=st["n_entries"])
    if cfg.get("coverage"):
        cov, touched, total, depth = orc.coverage(raw, off, idx, tl, want_depth=not cfg.get("coverage_summary"))
        out["cov"] = (cov, touched, total)
        if depth is not None:
            out["depth"] = depth
    return out


def gpu_stats(out):
    st = out["st"]
    return dict(mapped_inserts=st["mapped_inserts"], uniq_mapper_count=st["uniq"], multi_mapper_count=st["multi"],
                purged_insert_count=st["purged"], em_iterations=st["iterations"], multi_lists=st["n_lists"], multi_entries=st["n_entries"])


def run_cmp(m, raw, off, cfg, tl, **kw):
    out = run_gpu(m, raw, off, cfg, target_len=tl if cfg.get("coverage") else None, n_targets=len(tl), **kw)
    if "st" in out:
        out["st"] = gpu_stats(out)
    return out


FILT = dict(l=80, p=95, z=80)
CONFIGS = ([dict(profile=True, multi=mo) for mo in SHARE] +
           [dict(profile=True, besthit=True, kept=False, **FILT), dict(profile=True, uniqhit=True, kept=False, **FILT),
            dict(coverage=True, besthit=True, kept=False, **FILT), dict(coverage=True, coverage_summary=True, besthit=True, kept=False, **FILT)])
PRESETS = [("mixed", 30000, 41), ("community", 40000, 43), ("catalog10k", 40000, 47)]


def _oracle_cmp(oracle, g, go, cfg, tl, out, fmap=None, nf=None):
    exp = oracle_result(oracle, g, go, cfg, tl, fmap=fmap, n_features=nf)
    if "st" in out and cfg.get("multi", "proportional") != "proportional":
        exp["st"]["purged_insert_count"] = out["st"]["purged_insert_count"]
        exp["st"]["em_iterations"] = out["st"]["em_iterations"]
        exp["st"]["multi_lists"] = out["st"]["multi_lists"]                 # the lists are only built for PropSharing
        exp["st"]["multi_entries"] = out["st"]["multi_entries"]
    expect_equal(out, exp, str(cfg))


@gpu
@pytest.mark.parametrize("preset,n,seed", PRESETS)
@pytest.mark.parametrize("order", ["coord", "shuffle"])
def test_collate_parity_with_oracle(m, oracle, preset, n, seed, order):
    raw, off, tl = synth_stream(preset, n, seed)
    r2, o2, _ = reorder(raw, off, order, seed=seed)
    g, go = regroup(r2, o2)
    cuts = [(0, n // 3), (n // 3, n // 3 + 1), (n // 3 + 1, len(o2) - 1)]          # pushes cut anywhere
    for cfg in CONFIGS:
        out = run_cmp(m, r2, o2, dict(cfg, collate=True), tl, chunks=cuts)
        _oracle_cmp(oracle, g, go, cfg, tl, out)
    # a feature map: targets folded onto fewer features
    fmap = (np.arange(len(tl)) % max(len(tl) // 3, 1)).astype(np.int32)
    nf = int(fmap.max()) + 1
    cfg = dict(profile=True, besthit=True, kept=False, **FILT)
    out = run_cmp(m, r2, o2, dict(cfg, collate=True), tl, fmap=fmap, n_features=nf)
    _oracle_cmp(oracle, g, go, cfg, tl, out, fmap=fmap, nf=nf)


@gpu
@pytest.mark.parametrize("preset,n,seed", PRESETS[:2])
def test_collate_identity_on_grouped_input(m, preset, n, seed):
    raw, off, tl = synth_stream(preset, n, seed)
    split = int(m.split_point(raw, off, n // 2))
    cuts = [(0, split), (split, len(off) - 1)]
    for cfg in CONFIGS:
        a = run_cmp(m, raw, off, dict(cfg, collate=True), tl, chunks=cuts)
        b = run_cmp(m, raw, off, dict(cfg, kept=cfg.get("kept", True) and not cfg.get("coverage")), tl, chunks=cuts)
        expect_equal(a, b, str(cfg))


def _pe_read(name, hits, tid0=0, as0=60):
    """a paired read with `hits` alignment pairs, each with NM / MD / AS"""
    recs = []
    for h in range(hits):
        for mate, fl in ((0, 0x41), (1, 0x81)):
            aux = E.aux_int("NM", "C", 0) + E.aux_z("MD", "100") + E.aux_int("AS", "C", as0 - (h % 3))
            recs.append(E.record(name, flag=fl | 1, tid=(tid0 + h) % 40, pos=100 + 7 * h + mate * 50, cigar=((100, M),), aux=aux))
    return recs


def _edge_stream(n_reads=300, seed=5):
    rng = np.random.default_rng(seed)
    recs = []
    for r in range(n_reads):
        recs += _pe_read(f"r{r:05d}", int(rng.integers(1, 5)), tid0=int(rng.integers(40)))
    return recs


def _profile_cfgs():
    return [dict(profile=True, multi="proportional"), dict(profile=True, besthit=True, kept=False, **FILT)]


@gpu
@pytest.mark.parametrize("how", ["staged", "pinned", "device"])
def test_collate_edges_split_reads_empty_pushes_and_sources(m, oracle, how):
    recs = _edge_stream()
    # read r00000 (the stream's first records) and the last read, each spread over five pushes
    first, last = [r for r in recs if E.qname(r) == b"r00000"], [r for r in recs if E.qname(r) == b"r00299"]
    if len(first) < 5:
        first = _pe_read("r00000", 3)
    if len(last) < 5:
        last = _pe_read("r00299", 3, tid0=7)
    mid = [r for r in recs if E.qname(r) not in (b"r00000", b"r00299")]
    mid += [E.record("unplaced%d" % k, flag=4, tid=-1, pos=-1, cigar=()) for k in range(3)]       # reads with only tid -1 records
    mid += [E.record("minus%d" % (k // 2), flag=0x41 if k % 2 == 0 else 0x81, tid=-1, pos=-1, cigar=((100, M),),
                     aux=E.aux_int("NM", "C", 0) + E.aux_z("MD", "100") + E.aux_int("AS", "C", 50)) for k in range(4)]
    rng = np.random.default_rng(9)
    mid = [mid[int(i)] for i in rng.permutation(len(mid))]
    order = []
    step = len(mid) // 4
    for k in range(5):
        order.append(first[k * len(first) // 5:(k + 1) * len(first) // 5] + mid[k * step:(k + 1) * step if k < 4 else len(mid)] +
                     last[k * len(last) // 5:(k + 1) * len(last) // 5])
    pushes = []
    for k, grp in enumerate(order):
        pushes.append(grp)
        pushes.append([])                                                                        # empty pushes
    allrecs = [r for grp in pushes for r in grp]
    raw, off = E.stream(allrecs)
    bounds, lo = [], 0
    for grp in pushes:
        bounds.append((lo, lo + len(grp))); lo += len(grp)
    g, go = regroup(raw, off)
    tl = np.full(40, 5000, dtype=np.uint32)
    for cfg in _profile_cfgs() + [dict(coverage=True, besthit=True, kept=False, **FILT)]:
        out = run_cmp(m, raw, off, dict(cfg, collate=True), tl, chunks=bounds, how=how)
        _oracle_cmp(oracle, g, go, cfg, tl, out)


@gpu
def test_collate_read_with_5000_alignments(m, oracle):
    recs = _edge_stream(200, seed=8)
    big = []
    for h in range(2500):
        big += _pe_read("bigread", 1, tid0=h % 40, as0=60 - (h % 2))
    rng = np.random.default_rng(2)
    allr = recs + big
    allr = [allr[int(i)] for i in rng.permutation(len(allr))]
    raw, off = E.stream(allr)
    g, go = regroup(raw, off)
    tl = np.full(40, 5000, dtype=np.uint32)
    for cfg in _profile_cfgs():
        out = run_cmp(m, raw, off, dict(cfg, collate=True), tl)
        _oracle_cmp(oracle, g, go, cfg, tl, out)


_CHILD = r"""
import sys, numpy as np
sys.path[:0] = {paths!r}
import test_collate as T
import msamtools_b200 as m
from oracle import oracle as orc
orc.build(); orc.load()
raw, off, tl = T.synth_stream("mixed", 20000, 29)
r2, o2, _ = T.reorder(raw, off, "shuffle", seed=4)
g, go = T.regroup(r2, o2)
for cfg in T._profile_cfgs() + [dict(coverage=True, besthit=True, kept=False, **T.FILT)]:
    out = T.run_cmp(m, r2, o2, dict(cfg, collate=True), tl, chunks=[(0, 7000), (7000, len(o2) - 1)])
    T._oracle_cmp(orc, g, go, cfg, tl, out)
print("OK")
"""


@gpu
def test_collate_hash_collisions_in_child(m):
    env = dict(os.environ, MSG_COLLATE_HASH_BITS="8")
    code = _CHILD.format(paths=[ROOT, os.path.join(ROOT, "tests")])
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


@gpu
def test_collate_enoas_names_input_ordinal(m):
    recs = _edge_stream(120, seed=3)
    rng = np.random.default_rng(1)
    recs = [recs[int(i)] for i in rng.permutation(len(recs))]
    bad = 137
    q = recs[bad]
    recs[bad] = E.record(E.qname(q), flag=int.from_bytes(q[18:20], "little"), tid=int.from_bytes(q[4:8], "little", signed=True),
                         pos=int.from_bytes(q[8:12], "little", signed=True), cigar=((100, M),), aux=E.aux_int("NM", "C", 0) + E.aux_z("MD", "100"))
    raw, off = E.stream(recs)
    # the fused pass, and the general pipeline (coverage as a second consumer)
    for extra in (dict(), dict(coverage=True, target_len=np.full(40, 5000, dtype=np.uint32))):
        ctx = m.Context(profile=True, besthit=True, kept=False, collate=True, n_targets=40, **FILT, **extra)
        try:
            ctx.push(raw[:int(off[60])], off[:61].copy())
            ctx.push(np.ascontiguousarray(raw[int(off[60]):]), (off[60:] - off[60]).astype(np.uint64))
            with pytest.raises(m.MsgError) as ei:
                ctx.finish_profile()
            assert ei.value.code == -6 and f"(input record {bad})" in ei.value.text, ei.value.text
        finally:
            ctx.close()


@gpu
def test_collate_cg_placeholder(m):
    aux = E.aux_int("NM", "C", 0) + E.aux_z("MD", "100") + E.aux_int("AS", "C", 50)
    good = [E.record("a", tid=1, pos=5, cigar=((100, M),), aux=aux), E.record("b", tid=2, pos=9, cigar=((0, S), (100, N), (100, M)), aux=aux),
            E.record("a", tid=3, pos=1, cigar=((100, M),), aux=aux)]
    placeholder = E.record("c", tid=2, pos=9, cigar=((50, S), (100, N)), l_seq=50, aux=aux)
    for recs, ok in ((good, True), (good[:2] + [placeholder] + good[2:], False)):
        raw, off = E.stream(recs)
        ctx = m.Context(profile=True, besthit=True, kept=False, collate=True, n_targets=5, **FILT)
        try:
            if ok:
                ctx.push(raw, off)
                ab, st = ctx.finish_profile()
                assert st["mapped_inserts"] == 2
            else:
                with pytest.raises(m.MsgError) as ei:
                    ctx.push(raw, off)
                assert ei.value.code == -7 and "CG tag, near record 2" in ei.value.text, ei.value.text
        finally:
            ctx.close()


@gpu
def test_collate_refused_configurations_and_per_chunk_calls(m):
    for kw in (dict(records=True), dict(kept=True), dict(stats=True), dict(n_ranks=2, nccl_unique_id=b"\0" * 128)):
        with pytest.raises(m.MsgError) as ei:
            m.Context(collate=True, n_targets=3, **dict(dict(profile=True, kept=False), **kw))
        assert ei.value.code == -1 and "collate" in ei.value.text
    with pytest.raises(m.MsgError):
        m.Context(collate=True, n_targets=3, kept=False)
    raw, off = E.stream(_pe_read("x", 2))
    ctx = m.Context(profile=True, collate=True, kept=False, n_targets=40)
    try:
        ctx.push(raw, off)
        with pytest.raises(m.MsgError) as ei:
            ctx.kept_count()
        assert ei.value.code == -10
        ab, st = ctx.finish_profile()
        ab2, st2 = ctx.finish_profile()                                  # reuses the collation
        assert st["mapped_inserts"] == 1 and st2["mapped_inserts"] == 1 and np.array_equal(ab, ab2)
        ctx.push(raw, off)                                               # a new scope adds to the accumulators
        assert ctx.finish_profile()[1]["mapped_inserts"] == 2
        ctx.push(raw, off)
        ctx.reset()                                                      # drops the held records
        assert ctx.finish_profile()[1]["mapped_inserts"] == 0
    finally:
        ctx.close()


# ---------------------------------------------------------------- CLI on the GPU
CLI = os.path.join(ROOT, "msamtools_b200", "bin", "msamtools")


def _table(path):
    comments, body = samutil.read_profile_gz(path)
    keep = [c for c in comments if not c.startswith("# Command line") and "QNAME grouping check" not in c]
    return keep, body


@gpu
def test_cli_profile_collate_matches_grouped(m, tmp_path):
    raw, off, r2, o2, tl, names = _coord_bam(str(tmp_path / "coord.bam"), 60000, 31)
    samutil.write_bam(str(tmp_path / "grouped.bam"), samutil.synth_header(names, tl), names, tl, regroup(r2, o2)[0], level=1)
    a, b = str(tmp_path / "a.gz"), str(tmp_path / "b.gz")
    r = subprocess.run([CLI, "profile", "--collate", "--label", "x", "-o", a, str(tmp_path / "coord.bam")], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    assert "QNAME grouping check: not required for this operation" in "\n".join(samutil.read_profile_gz(a)[0])
    r = subprocess.run([CLI, "profile", "--label", "x", "-o", b, str(tmp_path / "grouped.bam")], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    ca, ba = _table(a)
    cb, bb = _table(b)
    assert ca == cb
    assert [x[0] for x in ba] == [x[0] for x in bb]
    assert close([float(x[1]) for x in ba[1:]], [float(x[1]) for x in bb[1:]], rel=1e-6)
    # filter (any order) | profile --collate  ==  grouped filter | profile
    outs = []
    for src, extra in ((str(tmp_path / "coord.bam"), ["--collate"]), (str(tmp_path / "grouped.bam"), [])):
        f = subprocess.Popen([CLI, "filter", "-b", "-l", "80", "-p", "95", "-z", "80", src], stdout=subprocess.PIPE)
        o = str(tmp_path / ("pipe%d.gz" % len(outs)))
        r = subprocess.run([CLI, "profile"] + extra + ["--label", "x", "-o", o, "-"], stdin=f.stdout, capture_output=True)
        f.stdout.close(); f.wait()
        assert f.returncode == 0 and r.returncode == 0, r.stderr.decode()[-2000:]
        outs.append(_table(o))
    assert outs[0][0] == outs[1][0]
    assert close([float(x[1]) for x in outs[0][1][1:]], [float(x[1]) for x in outs[1][1][1:]], rel=1e-6)
