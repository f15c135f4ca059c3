"""Collation past one grouped chunk: the chunk cuts, the global-memory sorts, long collision runs and error ordinals.

collate_run hands the grouped records to the pipeline in chunks of at most 2^24 records, cut where the key changes;
MSG_COLLATE_CHUNK_RECORDS=C lowers that limit so that every cut case is reachable with a few thousand records.
tests/collateutil.py restates the grouped order and the cut rule, so the tests know where each record lands: which
chunk holds it, whether a bucket holds exactly 2048 keys, which bad record an error must name.

CPU: the restated key against a scalar transcription of the kernel loop, the order's grouping, the cut rule's
invariants, and the constructors.  GPU (-m gpu): results against the oracle on the regrouped stream (integers, list
counts and PropSharing iterations exactly, f64 within 1e-9 relative, coverage exactly) and the predicted number of fused
chunks.  Tests that need an environment hook run in a child process.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import collateutil as CU
import edgeutil as E
import test_collate as T
from conftest import ROOT
from edgeutil import M

gpu = pytest.mark.gpu
FILT = T.FILT
TL40 = np.full(40, 5000, dtype=np.uint32)
AUX = E.aux_int("NM", "C", 0) + E.aux_z("MD", "100") + E.aux_int("AS", "C", 60)


# ================================================================ stream builders
def se_read(name, hits, tid0=0, as0=60, cigar=((100, M),), aux=None):
    """a single-end read with `hits` alignments"""
    out = []
    for h in range(hits):
        a = aux if aux is not None else E.aux_int("NM", "C", 0) + E.aux_z("MD", "100") + E.aux_int("AS", "C", as0 - (h % 3))
        out.append(E.record(name, flag=0, tid=(tid0 + h) % 40, pos=100 + 11 * h, cigar=cigar, aux=a))
    return out


def unplaced_read(name, k):
    """a read whose records are all unmapped (flag 4) or placed nowhere (tid -1)"""
    out = [E.record(name, flag=0x4D if j % 2 == 0 else 0x8D, tid=-1, pos=-1, cigar=()) for j in range(k)]
    if k > 2:
        out[-1] = E.record(name, flag=0x41, tid=-1, pos=-1, cigar=((100, M),), aux=AUX)
    return out


def background(n_reads, seed, prefix="r"):
    """{name: records}: paired reads of 1-4 alignment pairs, single-end reads of 1-5 alignments and, one read in four,
    reads with only unmapped or tid -1 records"""
    rng = np.random.default_rng(seed)
    reads = {}
    for r in range(n_reads):
        name = f"{prefix}{r:05d}"
        kind = r % 4
        if kind == 0:
            reads[name] = unplaced_read(name, int(rng.integers(1, 4)))
        elif kind == 1:
            reads[name] = se_read(name, int(rng.integers(1, 6)), tid0=int(rng.integers(40)))
        else:
            reads[name] = T._pe_read(name, int(rng.integers(1, 5)), tid0=int(rng.integers(40)))
    return reads


def shuffled(reads, seed):
    """a stream of all the reads' records in a seeded random order that keeps each read's records in order"""
    rng = np.random.default_rng(seed)
    tags = [name for name, recs in reads.items() for _ in recs]
    tags = [tags[int(i)] for i in rng.permutation(len(tags))]
    pos = {name: 0 for name in reads}
    out = []
    for name in tags:
        out.append(reads[name][pos[name]]); pos[name] += 1
    return E.stream(out)


def read_spans(raw, off, order):
    """grouped [start, end) of every read, in grouped order, and the read's QNAME"""
    lq, m = CU.names_all(raw, off)
    q = m[order]
    ql = lq[order]
    head = np.r_[True, (ql[1:] != ql[:-1]) | np.any(q[1:] != q[:-1], axis=1)]
    s = np.flatnonzero(head)
    e = np.r_[s[1:], len(order)]
    return [(int(a), int(b), bytes(q[a, :ql[a] - 1])) for a, b in zip(s, e)]


def is_fused(cfg):
    return bool(cfg.get("profile")) and (cfg.get("besthit") or cfg.get("uniqhit")) and not cfg.get("coverage")


def check(m, orc, raw, off, cfgs, tl, C=CU.CHUNK_RECORDS, bits=64, hows=("staged",), pushes=None):
    """every cfg on a collating context against the oracle on the regrouped stream; the fused ones must run the number
    of chunks the restated cut rule predicts"""
    _, ks = CU.grouped_order(raw, off, bits)
    nchunks = len(CU.cuts(ks, C)) - 1
    g, go = T.regroup(raw, off)
    for k, cfg in enumerate(cfgs):
        out = T.run_cmp(m, raw, off, dict(cfg, collate=True), tl, chunks=pushes, how=hows[k % len(hows)])
        T._oracle_cmp(orc, g, go, cfg, tl, out)
        if is_fused(cfg):
            assert out["timing"]["fused_chunks"] == nchunks, (cfg, out["timing"]["fused_chunks"], nchunks)
    return nchunks


def three_pushes(n):
    return [(0, n // 3), (n // 3, n // 3 + 1), (n // 3 + 1, n)]


# ================================================================ CPU
def test_vectorised_key_equals_kernel_loop():
    rng = np.random.default_rng(11)
    names = [bytes(rng.integers(33, 127, size=L, dtype=np.uint8)) for L in range(1, 255)]
    names += [b"A" * L for L in range(1, 255)] + [bytes([255]) * L for L in range(1, 255)]
    for bits in (64, 16, 4, 1):
        k = CU.names_keys(names, bits)
        assert [int(x) for x in k] == [CU.key_scalar(x, bits) for x in names], bits
    # from a stream, names of every length mod 4 at every byte alignment
    recs = [E.record(x, cigar=()) for x in names[:40]] + [E.record(names[k], cigar=((3, M),) * (k % 5)) for k in range(40, 254)]
    raw, off = E.stream(recs)
    assert [int(x) for x in CU.keys(raw, off)] == [CU.key_scalar(E.qname(r)) for r in recs]
    assert CU.key_scalar(b"a") != CU.key_scalar(b"a\0"[:1] + b"b") and CU.hash_mask(1) == 1 << 63


@pytest.mark.parametrize("bits", [64, 8, 1])
def test_restated_order_groups_reads_in_input_order(bits):
    reads = background(400, 3)
    reads.update({("L" * k): se_read("L" * k, 3) for k in range(1, 30)})       # names of many lengths
    raw, off = shuffled(reads, 4)
    order, ks = CU.grouped_order(raw, off, bits)
    assert sorted(order.tolist()) == list(range(len(order)))
    recs = E.split(raw, off)
    spans = read_spans(raw, off, order)
    assert len(spans) == len(reads) and len({q for _, _, q in spans}) == len(reads)     # every name in one run
    for a, b, q in spans:
        assert all(E.qname(recs[int(i)]) == q for i in order[a:b])
        assert np.all(np.diff(order[a:b]) > 0)                                       # input order kept
    assert np.all(ks[1:] >= ks[:-1])
    if bits == 1:
        assert len(np.unique(ks)) == 2                                               # two collision runs


@pytest.mark.parametrize("C", [1, 7, 64, 1000])
def test_cut_rule_invariants(C):
    reads = background(600, 5)
    for k, size in enumerate((C, C + 1, 2 * C - 1, 2 * C, 5 * C)):
        reads[f"big{k}"] = se_read(f"big{k}", size)
    raw, off = shuffled(reads, 6)
    order, ks = CU.grouped_order(raw, off)
    b = CU.cuts(ks, C)
    spans = read_spans(raw, off, order)
    starts = {a for a, _, _ in spans} | {len(order)}
    assert b[0] == 0 and b[-1] == len(order) and all(x < y for x, y in zip(b, b[1:]))
    assert set(b) <= starts                                                      # no cut inside a read
    for lo, hi in zip(b, b[1:]):
        inner = [a for a in starts if lo < a < hi]
        assert hi - lo <= C or not inner                                         # at most C records, or one read
        if hi < len(order):
            # the chunk is as long as it can be: no later read start within lo + C, unless the chunk is one read
            assert not any(hi < a <= lo + C for a in starts) or not inner


def test_constructors_give_claimed_sizes():
    bits = CU.bucket_bits(24000)
    assert bits == 6 and CU.bucket_bits(512) == 0 and CU.bucket_bits(513) == 1 and CU.bucket_bits(1 << 40) == 24
    names = CU.find_names(lambda k: CU.bucket_of(k, bits) == 17, 5, prefix="x")
    assert len(names) == 5 and all(int(CU.bucket_of(k, bits)) == 17 for k in CU.names_keys(names))
    raw, off, _ = _bucket_stream()
    order, ks = CU.grouped_order(raw, off)
    cnt = np.bincount(CU.bucket_of(ks, CU.bucket_bits(len(ks))), minlength=1 << CU.bucket_bits(len(ks)))
    assert CU.bucket_bits(len(ks)) == 6 and SMEM_EXACT in cnt.tolist() and SMEM_EXACT + 1 in cnt.tolist()
    run = _collision_run_names(16)
    k = CU.names_keys(run, 16)
    assert len(set(run)) == 3 and len({len(x) for x in run}) == 3 and np.all(k == k[0])
    # the vectorised riffle is test_collate.riffle, and stream_of is test_collate.permute
    raw, off, _ = T.synth_stream("mixed", 3000, 3)
    p = CU.riffle(raw, off)
    assert p.tolist() == T.riffle(raw, off)
    r2, o2 = CU.stream_of(raw, off, p)
    r3, o3 = T.permute(raw, off, p)
    assert bytes(r2) == bytes(r3) and np.array_equal(o2, o3)


# ================================================================ constructions shared with the GPU tests
SMEM_EXACT = CU.SMEM_KEYS


def _bucket_stream():
    """a stream of ~24 000 records (6 bucket bits) where one bucket holds exactly 2048 keys and another 2049"""
    reads = background(4500, 21, prefix="b")
    recs = [r for v in reads.values() for r in v]
    base = CU.names_keys(list(reads), 64)
    sizes = np.array([len(v) for v in reads.values()])
    n_plan = int(sizes.sum()) + 2 * CU.SMEM_KEYS           # close enough to fix the bucket bits
    bits = CU.bucket_bits(n_plan)
    cnt = np.bincount(CU.bucket_of(base, bits), weights=sizes, minlength=1 << bits).astype(int)
    big = {}
    for want, prefix in ((CU.SMEM_KEYS, "exact"), (CU.SMEM_KEYS + 1, "over")):
        name = CU.find_names(lambda k: ~np.isin(CU.bucket_of(k, bits), [CU.bucket_of(CU.names_keys([x]), bits)[0] for x in big]),
                             1, prefix=prefix)[0]
        b = int(CU.bucket_of(CU.names_keys([name]), bits)[0])
        big[name] = se_read(name, want - int(cnt[b]), tid0=3)
    reads.update({x.decode(): v for x, v in big.items()})
    raw, off = shuffled(reads, 22)
    assert CU.bucket_bits(len(off) - 1) == bits
    return raw, off, reads


def _collision_run_names(bits):
    """three names of different lengths whose keys agree in their top `bits` bits"""
    target = CU.names_keys([b"c0"], bits)[0]
    return [b"c0"] + [CU.find_names(lambda k: k == target, 1, prefix=p, bits=bits)[0] for p in ("cc", "ccccccccccc")]


# ================================================================ GPU: child processes with the environment hooks
@pytest.fixture(scope="module")
def m():
    import msamtools_b200 as mod
    assert mod._lib.load().msg_device_count() > 0, "no CUDA device: the GPU tests must not silently pass"
    return mod


_CHILD = r"""
import sys
sys.path[:0] = {paths!r}
import test_collate_chunks as T
T.{fn}(*{args!r})
print("OK")
"""


def in_child(env, fn, *args, timeout=1200):
    code = _CHILD.format(paths=[ROOT, os.path.join(ROOT, "tests")], fn=fn, args=args)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def _mods():
    import msamtools_b200 as m
    from oracle import oracle as orc
    orc.build(); orc.load()
    assert m._lib.load().msg_device_count() > 0
    return m, orc


def body_parity(preset, n, seed, order, C):
    m, orc = _mods()
    raw, off, tl = T.synth_stream(preset, n, seed)
    r2, o2, _ = T.reorder(raw, off, order, seed=seed)
    nchunks = check(m, orc, r2, o2, T.CONFIGS, tl, C=C, hows=("staged", "pinned", "device"), pushes=three_pushes(len(o2) - 1))
    assert nchunks > 1 if C < n else nchunks == 1


@gpu
@pytest.mark.parametrize("C,preset,n,seed,order", [(1, "mixed", 3000, 51, "shuffle"),
                                                   (64, "mixed", 30000, 41, "coord"), (64, "catalog10k", 40000, 47, "shuffle"),
                                                   (1000, "mixed", 30000, 41, "shuffle"), (1000, "catalog10k", 40000, 47, "coord")])
def test_multi_chunk_parity(m, C, preset, n, seed, order):
    in_child({"MSG_COLLATE_CHUNK_RECORDS": str(C)}, "body_parity", preset, n, seed, order, C)


def body_cut_placement(C):
    m, orc = _mods()
    cfgs = T._profile_cfgs() + [dict(coverage=True, besthit=True, kept=False, **FILT)]
    reads = background(240, 31)
    raw, off = shuffled(reads, 32)
    order, ks = CU.grouped_order(raw, off)
    b = CU.cuts(ks, C)
    spans = read_spans(raw, off, order)
    # a read straddles lo + C, and a cut follows a read of only unmapped / tid -1 records
    assert any(hi < lo + C for lo, hi in zip(b[:-2], b[1:-1]))
    unplaced = {q for _, _, q in spans if int(q[1:]) % 4 == 0}
    ends = {e: q for _, e, q in spans}
    assert any(ends[hi] in unplaced for hi in b[1:-1])
    check(m, orc, raw, off, cfgs, TL40, C=C)
    # a first chunk of exactly C records: the first read (first in key order) grows until a read starts at C
    s = [a for a, _, _ in spans]
    j = next(k for k, a in enumerate(s) if a >= C)
    first = spans[0][2].decode()
    grow = dict(reads, **{first: se_read(first, len(reads[first]) + (0 if s[j] == C else C - s[j - 1]))})
    raw1, off1 = shuffled(grow, 33)
    _, ks1 = CU.grouped_order(raw1, off1)
    b1 = CU.cuts(ks1, C)
    assert b1[1] == C, b1[:3]
    check(m, orc, raw1, off1, cfgs, TL40, C=C)
    # reads of C, C + 1, 2C - 1, 2C and 5C records, in the middle of the order and last in it
    top = int(ks.max())
    for size in (C, C + 1, 2 * C - 1, 2 * C, 5 * C):
        for where, pred in (("middle", lambda k: (k >> np.uint64(62)) == 1), ("last", lambda k: k > np.uint64(top))):
            name = CU.find_names(pred, 1, prefix=f"big{size}{where}")[0].decode()
            rr = dict(reads, **{name: se_read(name, size, tid0=size)})
            raw2, off2 = shuffled(rr, size)
            o2, ks2 = CU.grouped_order(raw2, off2)
            sp = {q: (a, e) for a, e, q in read_spans(raw2, off2, o2)}
            a, e = sp[name.encode()]
            assert (e == len(o2)) == (where == "last") and a > 0
            b2 = CU.cuts(ks2, C)
            assert a in b2 and e in b2                       # a chunk of its own
            check(m, orc, raw2, off2, cfgs, TL40, C=C)
    # later chunks of records the fixed window layout cannot hold: long names, 200-op CIGARs, long aux blocks
    rr = dict(reads)
    longname = CU.find_names(lambda k: k > np.uint64(1 << 63), 2, prefix="L" * 200)
    for x in longname:
        rr[x.decode()] = T._pe_read(x.decode(), 2, tid0=5)
    cig = tuple((1, M if k % 2 == 0 else E.I) for k in range(200))
    for x in CU.find_names(lambda k: k > np.uint64(1 << 63), 2, prefix="cig"):
        rr[x.decode()] = se_read(x.decode(), 3, cigar=cig, aux=E.aux_int("NM", "C", 100) + E.aux_z("MD", "100") + E.aux_int("AS", "C", 40))
    for x in CU.find_names(lambda k: k > np.uint64(1 << 63), 2, prefix="aux"):
        rr[x.decode()] = se_read(x.decode(), 3, aux=E.aux_b("XB", "i", list(range(120))) + AUX)
    raw3, off3 = shuffled(rr, 34)
    o3, ks3 = CU.grouped_order(raw3, off3)
    b3 = CU.cuts(ks3, C)
    slow = {q for q in rr if q.startswith(("L", "cig", "aux"))}
    for a, e, q in read_spans(raw3, off3, o3):
        if q.decode() in slow:
            assert a >= b3[1] + C, (q, a, b3[:3])            # past the chunk the layout comes from
    check(m, orc, raw3, off3, cfgs + [dict(profile=True, multi="proportional", kept=False)], TL40, C=C)


@gpu
@pytest.mark.parametrize("C", [16, 64])
def test_cut_placement(m, C):
    in_child({"MSG_COLLATE_CHUNK_RECORDS": str(C)}, "body_cut_placement", C)


def body_error_ordinals(C):
    m, _ = _mods()
    reads = {k: v for k, v in background(300, 41).items() if int(k[1:]) % 4 >= 2}        # paired reads
    raw, off = shuffled(reads, 42)
    order, ks = CU.grouped_order(raw, off)
    b = CU.cuts(ks, C)
    assert len(b) > 8
    spans = read_spans(raw, off, order)
    chunk_of = lambda g: int(np.searchsorted(b, g, side="right")) - 1
    # one read in each of chunks 5, 3 and 7 (in that order of choice), and the second read of chunk 3
    picked = []
    for c in (5, 3, 7):
        picked.append(next(q for a, e, q in spans if chunk_of(a) == c))
    picked.append([q for a, e, q in spans if chunk_of(a) == 3][1])
    for code, strip in ((-6, lambda r: E.aux_int("NM", "C", 0) + E.aux_z("MD", "100")),
                        (-5, lambda r: E.aux_int("AS", "C", 60))):
        recs = E.split(raw, off)
        bad = []
        for q in picked:
            mine = [i for i in range(len(recs)) if E.qname(recs[i]) == q]
            i = mine[-1]                                       # a mate record, not the read's first
            r = recs[i]
            recs[i] = E.record(q, flag=int.from_bytes(r[18:20], "little"), tid=int.from_bytes(r[4:8], "little", signed=True),
                               pos=int.from_bytes(r[8:12], "little", signed=True), cigar=((100, M),), aux=strip(r))
            bad.append(i)
        raw2, off2 = E.stream(recs)
        o2, _ = CU.grouped_order(raw2, off2)
        assert np.array_equal(o2, order)
        gpos = np.argsort(o2)
        want = min(bad, key=lambda i: gpos[i])
        assert chunk_of(gpos[want]) == 3
        cfgs = [dict(profile=True, besthit=True, kept=False, **FILT),
                dict(profile=True, besthit=True, kept=False, coverage=True, target_len=TL40, **FILT)]
        if code == -5:
            cfgs.append(dict(profile=True, kept=False, **FILT))
        for cfg in cfgs:
            ctx = m.Context(collate=True, n_targets=40, **cfg)
            try:
                h = len(off2) // 2
                ctx.push(raw2[:int(off2[h])], off2[:h + 1].copy())
                ctx.push(np.ascontiguousarray(raw2[int(off2[h]):]), (off2[h:] - off2[h]).astype(np.uint64))
                with pytest.raises(m.MsgError) as ei:
                    ctx.finish_profile()
                assert ei.value.code == code and f"(input record {want})" in ei.value.text, (cfg, want, ei.value.text)
            finally:
                ctx.close()


@gpu
def test_error_ordinals_in_later_chunks(m):
    in_child({"MSG_COLLATE_CHUNK_RECORDS": "16"}, "body_error_ordinals", 16)


def body_hash_bits(bits, C):
    m, orc = _mods()
    raw, off, tl = T.synth_stream("mixed", 8000, 61)
    recs = E.split(*T.reorder(raw, off, "shuffle", seed=62)[:2])
    rng = np.random.default_rng(63)
    extra = [r for k in range(1, 60) for r in se_read("M" * k, 1 + k % 4, tid0=k)]            # names of many lengths
    if bits == 16:
        for k, x in enumerate(_collision_run_names(16)):
            extra += se_read(x, 700 + 100 * k, tid0=k)                     # one run of 2 400 keys, three name lengths
    for r in extra:
        recs.insert(int(rng.integers(len(recs) + 1)), r)
    raw2, off2 = E.stream(recs)
    o, ks = CU.grouped_order(raw2, off2, bits)
    runs = np.diff(np.flatnonzero(np.r_[True, ks[1:] != ks[:-1], True]))
    if bits != 4:
        assert runs.max() > CU.SMEM_KEYS, runs.max()         # a by-name sort in global memory
    cfgs = T._profile_cfgs() + [dict(profile=True, multi="equal"), dict(coverage=True, coverage_summary=True, besthit=True, kept=False, **FILT)]
    check(m, orc, raw2, off2, cfgs, tl, C=C, bits=bits, pushes=three_pushes(len(off2) - 1))


@gpu
@pytest.mark.parametrize("bits", [1, 4, 16])
def test_hash_bits_collision_runs(m, bits):
    in_child({"MSG_COLLATE_HASH_BITS": str(bits), "MSG_COLLATE_CHUNK_RECORDS": "500"}, "body_hash_bits", bits, 500)


# ================================================================ GPU: sort paths with the default hooks
@gpu
def test_several_oversized_buckets(m, oracle):
    reads = background(1500, 71)
    for k, size in enumerate((2049, 2500, 4097, 9000)):
        reads[f"huge{k}"] = se_read(f"huge{k}", size, tid0=k, as0=60 - k)
    raw, off = shuffled(reads, 72)
    _, ks = CU.grouped_order(raw, off)
    bits = CU.bucket_bits(len(ks))
    cnt = np.bincount(CU.bucket_of(ks, bits), minlength=1 << bits)
    assert np.sum(cnt > CU.SMEM_KEYS) >= 3
    check(m, oracle, raw, off, T._profile_cfgs() + [dict(coverage=True, besthit=True, kept=False, **FILT)], TL40)


@gpu
def test_buckets_of_2048_and_2049_keys(m, oracle):
    raw, off, _ = _bucket_stream()
    check(m, oracle, raw, off, T._profile_cfgs() + [dict(profile=True, uniqhit=True, kept=False, **FILT)], TL40,
          hows=("staged", "device", "pinned"))


@gpu
def test_full_size_two_chunks(m, oracle):
    """2^24 + 2^21 riffled records with the default chunk limit: two chunks"""
    from msamtools_b200 import synth
    p = synth.make_params("community", n_records=(1 << 24) + (1 << 21), seed=81, read_len=20)
    raw, off, _ = synth.generate(p)
    raw = raw[:int(off[-1])]
    tl = synth.target_lengths(p)
    n = len(off) - 1
    perm = CU.riffle(raw, off)
    r2, o2 = CU.stream_of(raw, off, perm)
    _, ks = CU.grouped_order(r2, o2)
    assert len(CU.cuts(ks)) - 1 == 2
    cfg = dict(profile=True, besthit=True, kept=False, **FILT)
    out = T.run_cmp(m, r2, o2, dict(cfg, collate=True), tl, chunks=[(0, n // 2), (n // 2, n)])
    assert out["timing"]["fused_chunks"] == 2
    del r2, o2
    ref = T.run_cmp(m, raw, off, cfg, tl)                     # the input is the riffle's regrouped stream
    T.expect_equal(out, ref, "collate vs grouped")
    idx = oracle.filter_stream(raw, off, oracle.filter_cfg(besthit=True, **FILT))
    _, st, ui, _ = oracle.profile(raw, off, idx, len(tl), T.SHARE["proportional"])
    assert np.array_equal(out["ui"], ui)
    s = out["st"]
    assert (s["mapped_inserts"], s["uniq_mapper_count"], s["multi_mapper_count"], s["purged_insert_count"], s["em_iterations"]) == \
           (st["mapped_inserts"], st["uniq"], st["multi"], st["purged"], st["iterations"])
