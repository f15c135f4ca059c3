"""The CUDA path against the CPU oracle at the record shapes and size limits the synthetic streams never reach.

Synthetic streams (csrc/synth.c) have one record shape: 12-byte names, one to four M/I/D/S operations, an aux block of
exactly NM:C MD:Z AS, reads inside their targets.  The streams here come from tests/edgeutil.py, which writes record
bytes directly, and aim at the branches of the decoder's fast path (partial name words, the SWAR MD classifier, integer
aux types, the head / tail window layouts and the chunk's readable end), at the size limits of the fused, profile and
PropSharing kernels (pool and group sizes, distinct features per group, the feature count), at QNAME hash collisions and
at coverage runs that meet the end of a target or the edge of a bitmap word.

Integers, indices and bytes must match the oracle exactly; float64 values within 1e-9 relative, with the same
PropSharing iteration count, purged count and list totals.  The per-record flags of msg_pull_stats are checked too:
INPOOL against the filter predicates on the oracle's statistics, HAS_AS against the oracle, EQPREV against a byte
compare of adjacent QNAMEs, and SLOW (the record did not fit its staged windows) where a test builds records to fit or
to miss their windows on purpose.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import edgeutil as E
from edgeutil import M, I, D, N, S, H, P, EQ, X

SHARE = {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}
MODES = list(SHARE)
REL = 1e-9
F_INPOOL, F_HAS_AS, F_EQPREV, F_SLOW = 1, 2, 4, 8
HERE = os.path.dirname(os.path.abspath(__file__))
LETTERS = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789_.:", dtype=np.uint8)

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import msamtools_b200 as mod
    assert mod._lib.load().msg_device_count() > 0, "no CUDA device: the GPU tests must not silently pass"
    return mod


def close(a, b, rel=REL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.all(np.abs(a - b) <= rel * np.maximum(np.abs(a), np.abs(b)))


# ================================================================ stream generators
def _name(rng, n):
    return bytes(LETTERS[rng.integers(0, len(LETTERS), size=n)])


_INT_RANGE = {"c": (-128, 127), "C": (0, 255), "s": (-32768, 32767), "S": (0, 65535), "i": (-2**31, 2**31 - 1), "I": (0, 2**32 - 1)}


def _int_field(rng, tag, limits, small=20):
    """an integer tag of a random BAM type; at a range limit or sign boundary when `limits`, else a small value"""
    ty = "cCsSiI"[int(rng.integers(6))]
    lo, hi = _INT_RANGE[ty]
    if limits:
        cand = [lo, hi, 0, 1, min(hi, 127), min(hi, 128), max(lo, -1), max(lo, -129), int(rng.integers(lo, hi, endpoint=True))]
        v = cand[int(rng.integers(len(cand)))]
    else:
        v = int(rng.integers(0, min(small, hi) + 1))
    return E.aux_int(tag, ty, v)


def _md(rng, length, lead_letter=False):
    """an MD string of exactly `length` characters: numbers (0 tokens included), mismatches, deletions (^ after a number
    run or after a mismatch), optionally opening with a letter"""
    toks = [chr(int(rng.choice(LETTERS[:4])))] if lead_letter else []
    while sum(map(len, toks)) < length:
        k = int(rng.integers(7))
        if k < 2: toks.append(str(int(rng.integers(0, 80))))
        elif k < 4: toks.append("ACGTN"[int(rng.integers(5))])
        elif k == 4: toks.append("^" + "".join("ACGT"[int(x)] for x in rng.integers(0, 4, size=int(rng.integers(1, 4)))))
        else: toks.append("0")
    md = "".join(toks)[:length]
    return md[:-1] + "7" if md.endswith("^") else md


def _other(rng):
    k = int(rng.integers(8))
    if k == 0: return E.aux_a("XA", "q")
    if k == 1: return E.aux_f("XF", -2.5)
    if k == 2: return E.aux_b("XB", "sScCiIf"[int(rng.integers(7))], [int(x) for x in rng.integers(0, 100, size=int(rng.integers(0, 6)))])
    if k == 3: return E.aux_z("XZ", "z" * int(rng.integers(0, 60)))
    if k == 4: return E.aux_z("XH", "1AE3", "H")
    if k == 5: return E.aux_z("MC", "50M")                 # tags whose first letters match NM / MD / AS
    if k == 6: return E.aux_int("AM", "C", 7)
    return _int_field(rng, "XI", True)


def _aux(rng, *, need_tag, need_as, limits):
    """aux block of a mapped record in one of the orders / type mixes the decoder distinguishes"""
    nm = lambda: _int_field(rng, "NM", limits)
    as_ = lambda: _int_field(rng, "AS", True)
    mdlen = int(rng.integers(27, 35)) if rng.random() < 0.35 else int(rng.integers(1, 41))
    md = lambda: E.aux_z("MD", _md(rng, mdlen, lead_letter=rng.random() < 0.3))
    pats = [
        lambda: nm() + md() + as_(),                    # what the fast path takes
        lambda: nm() + md() + as_(),
        lambda: md() + nm() + as_(),                    # NM after MD
        lambda: md() + as_(),                           # MD without NM
        lambda: nm() + as_(),                           # NM without MD
        lambda: _other(rng) + nm() + md() + as_(),
        lambda: nm() + _other(rng) + md() + _other(rng) + as_() + _other(rng),
        lambda: nm() + md() + as_() + _other(rng),
        lambda: nm() + nm() + md() + md() + as_() + as_(),     # duplicate tags: the first one counts
        lambda: as_() + md() + nm(),
    ]
    if not need_as:
        pats += [lambda: nm() + md(), lambda: md() + _other(rng)]
    if not need_tag:
        pats += [lambda: as_(), lambda: _other(rng) + as_()]
        if not need_as:
            pats += [lambda: b"", lambda: _other(rng)]
    return pats[int(rng.integers(len(pats)))]()


_OPS = [M, M, M, I, D, N, S, H, P, EQ, X]


def _cigar(rng):
    r = rng.random()
    if r < 0.04:
        return []                                                # mapped record without a CIGAR
    nops = int(rng.integers(1, 5)) if r < 0.98 else int(rng.integers(5, 61))
    ops = []
    for _ in range(nops):
        op = _OPS[int(rng.integers(len(_OPS)))] if rng.random() > 0.03 else int(rng.integers(9, 16))   # 9-15: undefined
        ops.append((int(rng.integers(1, 60)), op))
    if len(ops) == 2 and ops[0][1] == S and ops[1][1] == N:      # that pair announces a CG-tag CIGAR
        ops[1] = (ops[1][0], M)
    return ops


def variety_records(seed, n, n_targets=24, need_tag=False, need_as=False, limits=True):
    """n records in QNAME groups: name lengths of every residue mod 4 (a few up to 254 bytes), neighbouring groups whose
    names differ in the last character only or in length only, every aux order / type, CIGARs of 0-60 operations,
    l_seq 0, unmapped records and tid -1 inside and between groups, READ1 / READ2 / unpaired groups."""
    rng = np.random.default_rng(seed)
    recs, prev, used = [], b"q", set()
    while len(recs) < n:
        k = rng.random()
        if k < 0.2 and len(prev) > 1:
            name = prev[:-1] + (b"x" if prev[-1:] != b"x" else b"y")            # differs in its last character only
        elif k < 0.3 and len(prev) < 250:
            name = prev + b"z"                                               # ab -> abz
        elif k < 0.35 and len(prev) > 1:
            name = prev[:-1]                                                 # abc -> ab
        else:
            ln = int(rng.integers(1, 41)) if rng.random() < 0.98 else int(rng.integers(100, 255))
            name = _name(rng, ln)
        while name in used:                                                  # groups stay QNAME-grouped (ab, abz, ab is not)
            name = _name(rng, int(rng.integers(4, 41)))
        used.add(name)
        prev = name
        gsize = int(rng.integers(1, 7)) if rng.random() < 0.97 else int(rng.integers(20, 45))
        paired = rng.random() < 0.5
        for j in range(gsize):
            flag = (0x40 if rng.random() < 0.5 else 0x80) | 1 if paired else 0
            if j:
                flag |= 0x100
            if rng.random() < 0.05:                                          # unmapped (placed with its mate, or not)
                tid = int(rng.integers(n_targets)) if rng.random() < 0.5 else -1
                recs.append(E.record(name, flag=flag | 4, tid=tid, pos=int(rng.integers(0, 500)) if tid >= 0 else -1, cigar=[],
                                     l_seq=int(rng.integers(0, 30)), aux=_aux(rng, need_tag=False, need_as=False, limits=limits) if rng.random() < 0.5 else b""))
                continue
            tid = int(rng.integers(n_targets)) if rng.random() > 0.03 else -1
            cig = _cigar(rng)
            ls = 0 if rng.random() < 0.1 else None
            recs.append(E.record(name, flag=flag, tid=tid, pos=int(rng.integers(0, 900)), cigar=cig, l_seq=ls,
                                 aux=_aux(rng, need_tag=need_tag, need_as=need_as, limits=limits), mapq=int(rng.integers(0, 61))))
    return recs[:n]


# ================================================================ GPU helpers
def push(m, ctx, raw, off, how, bufs):
    """push one chunk: 'staged' (pageable host buffer), 'device' (msg_push_device on a device copy), 'pinned' (pinned
    host buffer: the fused pass decodes it in place)"""
    n = len(off) - 1
    if how == "device":
        d_raw, d_off = ctx.device_alloc(max(raw.nbytes, 1)), ctx.device_alloc(off.nbytes)
        if raw.nbytes:
            ctx.device_upload(d_raw, raw)
        ctx.device_upload(d_off, off)
        bufs += [d_raw, d_off]
        ctx.push_device(d_raw, raw.nbytes, d_off, n)
    elif how == "pinned":
        pb = m.PinnedBuffer(max(raw.nbytes, 1))
        pb.array[:raw.nbytes] = raw
        bufs.append(pb)
        ctx.push(pb.array[:raw.nbytes], off)
    else:
        ctx.push(raw, off)


def release(ctx, bufs):
    for b in bufs:
        if hasattr(b, "close"):
            b.close()
        else:
            ctx.device_free(b)


def filter_has(opts):
    return bool(opts.get("l")) or opts.get("p") is not None or bool(opts.get("ppt")) or opts.get("z") is not None


def expected_inpool(opts, st, flag):
    """FB_INPOOL as msam_filter.c:132-136,181-183 defines it, from the oracle's per-record statistics"""
    do_filter = filter_has(opts) or opts.get("besthit") or opts.get("uniqhit") or opts.get("rescore")
    n = len(flag)
    if not do_filter:
        return np.ones(n, dtype=bool)
    unm = (flag & 4) != 0
    if not filter_has(opts):
        return ~unm
    ppt = 10 * opts["p"] if opts.get("p") is not None else opts.get("ppt", 0)
    max_clip = 100 - opts["z"] if opts.get("z") is not None else 100
    a, q, c, e = (st[k].astype(np.int64) for k in ("alen", "qlen", "qclip", "edit"))
    w = lambda v: ((v + 2**31) % 2**32) - 2**31                          # int32 arithmetic
    fail = np.zeros(n, dtype=bool)
    if opts.get("l"):
        fail |= a < opts["l"]
    if ppt < 0:
        fail |= w(1000 * w(e - a)) < w(a * ppt)
    elif ppt > 0:
        fail |= w(1000 * w(a - e)) < w(a * ppt)
    if max_clip < 100:
        fail |= w(100 * c) > w(max_clip * q)
    inv = bool(opts.get("invert"))
    unm_in = bool(opts.get("keep_unmapped")) and ppt >= 0 and inv
    return np.where(unm, unm_in, fail == inv)


def flags_of(recs):
    return np.array([int.from_bytes(r[18:20], "little") for r in recs], dtype=np.int64)


def check_decode(oracle, recs, raw, off, opts, st, kept=None, rec=None, lo=0):
    """per-record statistics and flags of records [lo, lo + n) of `recs` (the chunk raw / off) against the oracle"""
    exp = oracle.record_stats(raw, off)
    n = len(off) - 1
    for k in ("alen", "qlen", "qclip", "edit"):
        bad = np.nonzero(st[k] != exp[k])[0]
        assert len(bad) == 0, (k, [(int(i) + lo, int(st[k][i]), int(exp[k][i])) for i in bad[:5]])
    has_as = exp["has_as"] > 0
    assert np.array_equal(st["score"][has_as], exp["score"][has_as]) or opts.get("rescore")
    fl = st["flags"].astype(np.int64)
    if not opts.get("rescore"):
        bad = np.nonzero(((fl & F_HAS_AS) != 0) != has_as)[0]
        assert len(bad) == 0, ("HAS_AS", [int(i) + lo for i in bad[:5]])
    eqp = E.eqprev(recs)
    bad = np.nonzero(((fl & F_EQPREV) != 0) != eqp)[0]
    assert len(bad) == 0, ("EQPREV", [int(i) + lo for i in bad[:5]])
    inp = expected_inpool(opts, exp, flags_of(recs))
    bad = np.nonzero(((fl & F_INPOOL) != 0) != inp)[0]
    assert len(bad) == 0, ("INPOOL", [int(i) + lo for i in bad[:5]])
    assert n == len(recs)
    if kept is not None:
        cfg = oracle.filter_cfg(**opts)
        eidx = oracle.filter_stream(raw, off, cfg)
        assert np.array_equal(kept, eidx)
        if rec is not None:
            assert bytes(rec) == bytes(oracle.emit_records(raw, off, eidx, cfg))


def profile_check(st, est, ui, eui, d, ed, ab, eab):
    for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "converged", "n_lists", "n_entries"):
        assert st[k] == est[k], (k, st[k], est[k])
    assert np.array_equal(ui, eui)
    assert close(d, ed) and close(ab, eab)


# ================================================================ streams shared by the tests (built once per session)
_cache = {}


def cached(key, fn):
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


def variety(kind):
    """'any': every record shape (statistics only, no filter); 'tagged': every mapped record has NM or MD (filters);
    'scored': tagged and every mapped record has AS (best-hit)"""
    def make():
        seed = {"any": 11, "tagged": 12, "scored": 13}[kind]
        recs = variety_records(seed, 12_000, need_tag=kind != "any", need_as=kind == "scored", limits=kind == "any")
        return (recs,) + E.stream(recs)
    return cached(("variety", kind), make)


# ---- pinned window layouts: a 4096-record prefix fixes the layout, the body's records fit their windows exactly or miss by one byte
LAYOUTS = {                     # name: (QNAME bytes, CIGAR ops, aux bytes of the prefix records) -> (LPR, hc, tc)
    "synthetic": ((12, 1, 20), (8, 5, 3)),
    "lpr16": ((59, 4, 40), (16, 8, 4)),
    "clamped": ((149, 4, 60), (16, 12, 4)),
}


def _aux_exact(rng, length):
    """NM:C MD:Z AS:C [XZ:Z] block of exactly `length` bytes (>= 13)"""
    body = length - 12
    if body <= 30:
        return E.aux_int("NM", "C", int(rng.integers(0, 5))) + E.aux_z("MD", _md(rng, body)) + E.aux_int("AS", "C", int(rng.integers(0, 100)))
    return (E.aux_int("NM", "C", int(rng.integers(0, 5))) + E.aux_z("MD", _md(rng, 10)) + E.aux_int("AS", "C", int(rng.integers(0, 100)))
            + E.aux_z("XZ", "z" * (length - 26)))


def layout_stream(name, seed=5, n_body=1500):
    """(records, kinds) where kinds[i] is None for prefix / filler records, else (head fits, tail fits) by construction"""
    def make():
        (nl, nc, alen), (lpr, hc, tc) = LAYOUTS[name]
        rng = np.random.default_rng(seed)
        recs, kinds = [], []
        for k in range(4096):
            recs.append(E.record(b"p%0*d" % (nl - 1, k), tid=k % 7, pos=k % 300, cigar=[(10, M)] * (nc - 1) + [(30, M)],
                                 aux=_aux_exact(rng, alen)))
            kinds.append(None)
        o = sum(map(len, recs))
        for k in range(n_body):
            want_head, want_tail = [(True, True), (False, True), (True, False), (True, True), (False, False)][k % 5]
            if rng.random() < 0.5:
                want_head, want_tail = want_head or rng.random() < 0.5, want_tail
            ncig = int(rng.integers(1, 4))
            lq = 16 * hc - (o & 15) - 36 - 4 * ncig + (0 if want_head else 1)    # 36 + lq + 4 nc = room (+1)
            if not want_head and rng.random() < 0.5:
                lq += int(rng.integers(0, 3))                                     # a little further over
            lq = min(lq, 255)
            cig = [(int(rng.integers(1, 30)), M)] * (ncig - 1) + [(int(rng.integers(20, 60)), M)]
            ls = int(rng.integers(0, 80))
            ao = 36 + lq + 4 * ncig + (ls + 1) // 2 + ls
            room = E.tail_room(o + ao, tc)
            aux = _aux_exact(rng, room if want_tail else room + 1 + (int(rng.integers(0, 3)) if rng.random() < 0.3 else 0))
            r = E.record(_name(rng, lq - 1), flag=0, tid=int(rng.integers(7)), pos=int(rng.integers(0, 300)), cigar=cig, l_seq=ls, aux=aux)
            assert E.fits(r, o, hc, tc) == (want_head, want_tail) and (36 + lq + 4 * ncig) <= 16 * hc + 3
            recs.append(r); kinds.append((want_head, want_tail))
            o += len(r)
        for k in range(40):                                                       # the chunk's end: out of the body
            recs.append(E.record(b"t%011d" % k, tid=1, pos=5, cigar=[(20, M)], aux=_aux_exact(rng, 16)))
            kinds.append(None)
        return recs, kinds
    return cached(("layout", name, seed, n_body), make)


# ================================================================ CPU checks (no GPU needed)
def test_builder_reindexes_and_oracle_accepts(oracle):
    from msamtools_b200 import api
    for recs, raw, off in (variety("any"), variety("tagged"), variety("scored")):
        assert np.array_equal(api.index_records(raw), off)
        assert E.split(raw, off) == recs
        st = oracle.record_stats(raw, off)
        assert (st["has_tag"] > 0).sum() > 0.5 * len(recs)
    for name in LAYOUTS:
        recs, _ = layout_stream(name)
        raw, off = E.stream(recs)
        assert np.array_equal(api.index_records(raw), off)
        oracle.record_stats(raw, off)
    recs, raw, off = variety("scored")
    assert len(oracle.filter_stream(raw, off, oracle.filter_cfg(l=20, p=80, besthit=True))) > 0
    # the shapes the decoder branches on are all there
    lq = raw[off[:-1].astype(np.int64) + 12]
    assert set((lq % 4).tolist()) == {0, 1, 2, 3} and lq.max() >= 100
    assert E.eqprev(recs).sum() > 1000


def test_collision_pairs_collide(collisions):
    # a pair found by an independent search, and the session's pairs
    ha, hb = E.name_hash([b"ulE6tYRDkYKZ", b"6snSzweR6aqM"]).tolist()
    assert ha == hb
    for a, b in collisions:
        assert a != b and len(a) == len(b) == 12
        ha, hb = E.name_hash([a, b]).tolist()
        assert ha == hb


def test_probe_layout_restatement():
    for name, (_, want) in LAYOUTS.items():
        recs, kinds = layout_stream(name)
        raw, off = E.stream(recs)
        assert E.probe_layout(raw, off) == want, name
        assert E.probe_layout(*E.stream(recs[:4096])) == want, name
        k = np.array([x for x in kinds if x is not None])
        assert k[:, 0].sum() > 300 and (~k[:, 0]).sum() > 300 and k[:, 1].sum() > 300 and (~k[:, 1]).sum() > 300, name
    recs, _, _ = variety("any")
    assert E.probe_layout(*E.stream(recs))[0] in (8, 16)


@pytest.fixture(scope="session")
def collisions():
    return cached("collisions", lambda: E.find_collisions(4))


# ================================================================ 1. decoder record shapes
PUSHES = ["staged", "device", "slow"]


@gpu
@pytest.mark.parametrize("how", PUSHES)
def test_decode_field_variety(m, oracle, how):
    """statistics, AS and flags of every record shape, no filter (all of them in the pool)"""
    recs, raw, off = variety("any")
    bufs = []
    with m.Context(stats=True, n_targets=24, force_slow=how == "slow") as ctx:
        push(m, ctx, raw, off, "staged" if how == "slow" else how, bufs)
        st = ctx.pull_stats()
        release(ctx, bufs)
    check_decode(oracle, recs, raw, off, {}, st)
    slow = (st["flags"] & F_SLOW) != 0
    assert slow.all() if how == "slow" else (0 < slow.sum() < len(recs) // 4)


FILTERS = [
    dict(l=30), dict(p=90), dict(z=20), dict(l=25, p=85, z=30), dict(ppt=-900), dict(p=92, invert=True),
    dict(p=92, invert=True, keep_unmapped=True), dict(l=20, rescore=True), dict(rescore=True, uniqhit=True),
    dict(besthit=True), dict(uniqhit=True), dict(l=30, p=85, besthit=True), dict(z=30, uniqhit=True),
]
fid = lambda o: ",".join(f"{k}={v}" for k, v in o.items())


@gpu
@pytest.mark.parametrize("opts", FILTERS, ids=fid)
def test_decode_filters(m, oracle, opts):
    """kept indices, record bytes, statistics and flags for every filter kind; each through a staged push, push_device
    and the slow path, and once more without statistics (DM_NEED_STATS off unless the filter needs them)"""
    kind = "scored" if (opts.get("besthit") or opts.get("uniqhit")) else "tagged"
    recs, raw, off = variety(kind)
    for how in PUSHES:
        bufs = []
        with m.Context(stats=True, records=True, n_targets=24, force_slow=how == "slow", **opts) as ctx:
            push(m, ctx, raw, off, "staged" if how == "slow" else how, bufs)
            kept = ctx.pull_kept()
            st = ctx.pull_stats()
            rec, _ = ctx.pull_records()
            release(ctx, bufs)
        check_decode(oracle, recs, raw, off, opts, st, kept, rec)
    cfg = oracle.filter_cfg(**opts)
    eidx = oracle.filter_stream(raw, off, cfg)
    assert 0 < len(eidx) < len(recs)
    for records in (True, False):
        with m.Context(records=records, n_targets=24, **opts) as ctx:
            ctx.push(raw, off)
            assert np.array_equal(ctx.pull_kept(), eidx)
            if records:
                assert bytes(ctx.pull_records()[0]) == bytes(oracle.emit_records(raw, off, eidx, cfg))


@gpu
@pytest.mark.parametrize("name", list(LAYOUTS))
def test_decode_pinned_layouts(m, oracle, name):
    """records that fill their head or tail window exactly are staged (no SLOW flag); one byte more and they are read
    from global memory.  Same statistics and flags either way, through a staged push and push_device."""
    recs, kinds = layout_stream(name)
    raw, off = E.stream(recs)
    body = np.array([k is not None for k in kinds])
    fit = np.array([k is not None and k[0] and k[1] for k in kinds])
    opts = dict(l=20, p=80)
    for how in ("staged", "device"):
        bufs = []
        with m.Context(stats=True, records=True, n_targets=7, **opts) as ctx:
            push(m, ctx, raw, off, how, bufs)
            st = ctx.pull_stats()
            kept = ctx.pull_kept()
            rec, _ = ctx.pull_records()
            release(ctx, bufs)
        check_decode(oracle, recs, raw, off, opts, st, kept, rec)
        slow = (st["flags"] & F_SLOW) != 0
        assert not slow[fit].any(), (how, np.nonzero(fit & slow)[0][:5])
        assert slow[body & ~fit].all(), (how, np.nonzero(body & ~fit & ~slow)[0][:5])
        assert fit.sum() > 300 and (body & ~fit).sum() > 300


@gpu
def test_decode_tiles_and_windows(m, oracle):
    """pools of 1-40 records at every offset mod 32 and across 128-record decode tiles, names of every length mod 4"""
    rng = np.random.default_rng(21)
    recs = []
    for start in range(32):
        while len(recs) % 32 != start:
            recs.append(E.record(_name(rng, int(rng.integers(1, 9))), tid=1, pos=3, aux=_aux(rng, need_tag=True, need_as=True, limits=False)))
        for size in (1, 2, 3, 7, 8, 9, 31, 32, 33, 40):
            nm = _name(rng, 4 * int(rng.integers(1, 6)) + start % 4)
            for j in range(size):
                recs.append(E.record(nm, flag=0x100 if j else 0, tid=int(rng.integers(5)), pos=int(rng.integers(0, 200)),
                                     cigar=_cigar(rng), aux=_aux(rng, need_tag=True, need_as=True, limits=False)))
    raw, off = E.stream(recs)
    for opts in (dict(l=20, p=80), dict(besthit=True), dict(z=40, uniqhit=True)):
        for how in PUSHES:
            bufs = []
            with m.Context(stats=True, records=True, n_targets=5, force_slow=how == "slow", **opts) as ctx:
                push(m, ctx, raw, off, "staged" if how == "slow" else how, bufs)
                st = ctx.pull_stats(); kept = ctx.pull_kept(); rec, _ = ctx.pull_records()
                release(ctx, bufs)
            check_decode(oracle, recs, raw, off, opts, st, kept, rec)


@gpu
def test_decode_chunk_end_residues(m, oracle):
    """the chunk's last byte at every offset mod 16: device-resident and pinned chunks are read up to nbytes & ~15,
    staged ones up to nbytes + 64"""
    recs, raw, off = variety("scored")
    recs, raw, off = recs[:3000], raw[:int(off[3000])], off[:3001]
    opts = dict(l=20, p=80, besthit=True)
    seen = set()
    for r in range(16):
        k = E.cut_at_residue(off, r, lo=2500)
        assert k is not None
        sraw, soff, srecs = raw[:int(off[k])], off[:k + 1], recs[:k]
        seen.add(int(soff[-1]) % 16)
        for how in ("staged", "device"):
            bufs = []
            with m.Context(stats=True, records=True, n_targets=24, **opts) as ctx:
                push(m, ctx, sraw, soff, how, bufs)
                st = ctx.pull_stats(); kept = ctx.pull_kept(); rec, _ = ctx.pull_records()
                release(ctx, bufs)
            check_decode(oracle, srecs, sraw, soff, opts, st, kept, rec)
        # fused filter --besthit | profile, decoded in place from pinned host memory
        eidx = oracle.filter_stream(sraw, soff, oracle.filter_cfg(**opts))
        eab, est, eui, ed = oracle.profile(sraw, soff, eidx, 24, 3)
        bufs = []
        with m.Context(profile=True, multi="proportional", kept=False, n_targets=24, **opts) as ctx:
            push(m, ctx, sraw, soff, "pinned", bufs)
            ui, d = ctx.pull_counts(); ab, pst = ctx.finish_profile(); t = ctx.timing()
            release(ctx, bufs)
        assert (t["zero_copy_chunks"], t["fused_chunks"], t["fused_fallbacks"]) == (1, 1, 0)
        profile_check(pst, est, ui, eui, d, ed, ab, eab)
    assert seen == set(range(16))


@gpu
def test_decode_resident_layout_reuse(m, oracle):
    """push_device keeps the first chunk's window layout: a chunk of long records after a chunk of short ones runs with
    the short windows (most of its records then take the slow path) and must still match"""
    short, _ = layout_stream("synthetic")
    long_, _ = layout_stream("clamped")
    opts = dict(l=20, p=80)
    with m.Context(stats=True, records=True, n_targets=7, **opts) as ctx:
        bufs = []
        for recs in (short, long_):
            raw, off = E.stream(recs)
            push(m, ctx, raw, off, "device", bufs)
            st = ctx.pull_stats(); kept = ctx.pull_kept(); rec, _ = ctx.pull_records()
            check_decode(oracle, recs, raw, off, opts, st, kept, rec)
        assert ((st["flags"] & F_SLOW) != 0).mean() > 0.9
        release(ctx, bufs)


STAGING = {"async": {"MSG_STAGING": "async"}, "granule128": {"MSG_L2_GRANULE": "128"}}


@gpu
@pytest.mark.parametrize("variant", list(STAGING))
def test_decode_staging_variants(variant):
    """MSG_STAGING=async (LDGSTS) and MSG_L2_GRANULE=128 select four more decode_kernel instantiations; both switches are
    read once per process, so the decoder tests run again in a child process"""
    env = dict(os.environ, **STAGING[variant])
    sel = "field_variety or pinned_layouts or chunk_end or tiles or resident"
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", "-m", "gpu", "-k", sel, __file__],
                       cwd=os.path.dirname(HERE), env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and " failed" not in r.stdout


# ================================================================ 2. pools, groups and feature counts at the kernels' limits
def _pool_records(rng, name, size, n_features, *, tie=True, mates="mix", holes=False, score_hi=60):
    """one QNAME pool of `size` alignments over `n_features` distinct targets (0 .. n_features-1, in a shuffled first
    appearance order), equal best scores when `tie`"""
    feats = rng.permutation(n_features).tolist()
    seq = feats + [feats[int(rng.integers(n_features))] for _ in range(size - n_features)]
    out = []
    for j, t in enumerate(seq[:size]):
        if mates == "mix":
            flag = 1 | (0x40 if j % 3 else 0x80)
        elif mates == "r1":
            flag = 0x41
        else:
            flag = 0
        if j:
            flag |= 0x100
        sc = score_hi if tie else int(rng.integers(score_hi - 5, score_hi + 1))
        out.append(E.record(name, flag=flag, tid=int(t), pos=int(rng.integers(0, 400)), cigar=[(40, M)],
                            aux=E.aux_int("NM", "C", 0) + E.aux_z("MD", "40") + E.aux_int("AS", "C", sc)))
        if holes and j % 5 == 2:
            out.append(E.record(name, flag=flag | 0x104, tid=-1, pos=-1, cigar=[], aux=E.aux_int("AS", "C", 0)))
    return out


def pools_stream(case, seed=3):
    """pool / group shapes per case; 'small' stays inside every fused-walk limit"""
    def make():
        rng = np.random.default_rng(seed)
        recs, k = [], 0
        nm = lambda: b"g%07d_%s" % (k, _name(rng, int(rng.integers(0, 4))))
        filler = lambda: E.record(b"f%09d" % len(recs), tid=int(rng.integers(60)), pos=3, cigar=[(40, M)],
                                  aux=E.aux_int("NM", "C", 0) + E.aux_z("MD", "40") + E.aux_int("AS", "C", int(rng.integers(30, 60))))
        if case == "small":
            for start in range(32):
                for size in list(range(1, 41)) + [8, 9, 9]:
                    while len(recs) % 32 != start:
                        recs.append(filler())
                    nd = min(size, [1, 2, 4, 5, 8, 9, 12][int(rng.integers(7))])
                    recs += _pool_records(rng, nm(), size, nd, tie=rng.random() < 0.5, mates=["mix", "r1", "se"][int(rng.integers(3))],
                                          holes=rng.random() < 0.3)
                    k += 1
                    if rng.random() < 0.2:           # unmapped / tid -1 records between groups
                        recs.append(E.record(nm(), flag=4, tid=-1, pos=-1, cigar=[], aux=b""))
                        k += 1
            # a feature repeating right after the ninth distinct one: the PROF_CACHE rescan, in groups that leave a window
            for rep in range(6):
                while len(recs) % 32 != 20 + rep:
                    recs.append(filler())
                seq = list(range(10, 18)) + [30 + rep, 30 + rep, 40, 10, 41, 41, 30 + rep] + list(range(50, 58)) + [57, 56]
                name = nm(); k += 1
                for j, t in enumerate(seq):
                    recs.append(E.record(name, flag=0x100 if j else 0, tid=t, pos=5, cigar=[(40, M)],
                                         aux=E.aux_int("NM", "C", 0) + E.aux_z("MD", "40") + E.aux_int("AS", "C", 50)))
        else:
            size, nd = {"d48": (60, 48), "d49": (60, 49), "r1024": (1024, 12), "r1025": (1025, 12)}[case]
            for _ in range(3):
                recs += _pool_records(rng, nm(), 5, 3); k += 1
                for _ in range(int(rng.integers(3, 40))):
                    recs.append(filler())
            recs += _pool_records(rng, nm(), size, nd, tie=True, mates="se"); k += 1
            for _ in range(50):
                recs.append(filler())
        return (recs,) + E.stream(recs)
    return cached(("pools", case, seed), make)


@gpu
@pytest.mark.parametrize("case", ["small", "d48", "d49", "r1024", "r1025"])
def test_pools_and_groups(m, oracle, case):
    """all four --multi modes through the fused pass, the general pipeline and plain profile; the fused pass hands the
    chunk to the general pipeline exactly when a walked pool has more than 1024 records or 48 distinct features"""
    recs, raw, off = pools_stream(case)
    T = 60
    for hit in ("besthit", "uniqhit"):
        # a 1025-record pool is declined before its winners are known; 49 distinct winners need --besthit (all tied)
        fallback = case == "r1025" or (case == "d49" and hit == "besthit")
        opts = {hit: True}
        eidx = oracle.filter_stream(raw, off, oracle.filter_cfg(**opts))
        for mode in MODES:
            for path in ("fused", "general", "plain"):
                idx = None if path == "plain" else eidx
                eab, est, eui, ed = oracle.profile(raw, off, idx, T, SHARE[mode])
                with m.Context(profile=True, multi=mode, kept=path != "fused", n_targets=T, **({} if path == "plain" else opts)) as ctx:
                    ctx.push(raw, off)
                    if path != "plain":
                        assert ctx.kept_count() == len(eidx)
                    ui, d = ctx.pull_counts(); ab, st = ctx.finish_profile(); t = ctx.timing()
                profile_check(st, est, ui, eui, d, ed, ab, eab)
                if path == "fused":
                    assert (t["fused_chunks"], t["fused_fallbacks"]) == (1, int(fallback)), (hit, mode)
                else:
                    assert t["fused_chunks"] == 0
                if mode == "proportional" and hit == "besthit":
                    assert est["multi"] > 0 and est["n_entries"] > 0


def feature_stream(F, T, seed):
    """inserts over F features (T targets, fmap t -> t % F): skewed unique counts plus multi-mappers over 2-6 features,
    single-end and paired, so that proportional sharing needs several iterations"""
    rng = np.random.default_rng(seed)
    w = 1.0 / np.arange(1, T + 1) ** 0.8
    w /= w.sum()
    recs = []
    aux = lambda sc: E.aux_int("NM", "C", 1) + E.aux_z("MD", "20A19") + E.aux_int("AS", "C", sc)
    for q in range(5000):
        name = b"i%06d" % q
        nt = 1 if rng.random() < 0.55 else int(rng.integers(2, 7))
        ts = rng.choice(T, size=min(nt, T), replace=False, p=w)
        paired = rng.random() < 0.3
        for j, t in enumerate(ts):
            for mate in ((0x41, 0x81) if paired else (0,)):
                recs.append(E.record(name, flag=mate | (0x100 if j else 0), tid=int(t), pos=7, cigar=[(40, M)], aux=aux(50)))
        if rng.random() < 0.2:
            recs.append(E.record(name, flag=0x100, tid=int(rng.integers(T)), pos=9, cigar=[(40, M)], aux=aux(40)))
    return E.stream(recs)


FEATURES = [1, 2, 511, 512, 513, 2047, 2048, 2049, 4095, 4096, 4097]


@gpu
@pytest.mark.parametrize("F", FEATURES)
def test_feature_count_sweep(m, oracle, F):
    """n_features at the limits of em_copies (512), the shared-memory PropSharing loop (2048) and the shared-memory
    histograms (4096); with n_targets = F and with a map from 2F + 1 targets onto F features"""
    opts = dict(besthit=True)
    for T in (F, 2 * F + 1):
        raw, off = feature_stream(F, T, seed=F + T)
        fmap = None if T == F else (np.arange(T) % F).astype(np.int32)
        eidx = oracle.filter_stream(raw, off, oracle.filter_cfg(**opts))
        for mode in MODES:
            for path in ("fused", "general", "plain"):
                idx = None if path == "plain" else eidx
                eab, est, eui, ed = oracle.profile(raw, off, idx, T, SHARE[mode], fmap=fmap, n_features=F)
                with m.Context(profile=True, multi=mode, kept=path != "fused", n_targets=T, n_features=F, fmap=fmap,
                               **({} if path == "plain" else opts)) as ctx:
                    ctx.push(raw, off)
                    ui, d = ctx.pull_counts(); ab, st = ctx.finish_profile(); t = ctx.timing()
                profile_check(st, est, ui, eui, d, ed, ab, eab)
                assert t["fused_chunks"] == (path == "fused") and t["fused_fallbacks"] == 0
                if mode == "proportional" and F > 2:            # (with two features every list is the same pair: two iterations)
                    assert est["iterations"] >= 5, (F, T, est["iterations"])
                    assert close(st["delta"], est["delta"], 1e-6)


def collision_stream(pairs, where, seed=9):
    """each colliding pair (a, b) as two single-alignment inserts on different targets, placed per `where`"""
    rng = np.random.default_rng(seed)
    recs = []
    aux = lambda sc: E.aux_int("NM", "C", 0) + E.aux_z("MD", "40") + E.aux_int("AS", "C", sc)
    fill = lambda: recs.append(E.record(b"n%011d" % len(recs), tid=int(rng.integers(2, 8)), pos=3, cigar=[(40, M)], aux=aux(40)))
    at = {"window": lambda i: i * 64 + 5, "window_edge": lambda i: i * 64 + 31,
          "tile_edge": lambda i: i * 256 + 127, "separated": lambda i: i * 64 + 10}[where]
    for i, (a, b) in enumerate(pairs):
        while len(recs) < at(i):
            fill()
        recs.append(E.record(a, tid=0, pos=3, cigar=[(40, M)], aux=aux(50)))
        if where == "separated":
            recs.append(E.record(b"u%011d" % len(recs), flag=4, tid=-1, pos=-1, cigar=[], aux=b""))
            recs.append(E.record(b"v%011d" % len(recs), tid=-1, pos=-1, cigar=[(40, M)], aux=aux(45)))
        recs.append(E.record(b, tid=1, pos=3, cigar=[(40, M)], aux=aux(50)))
    for _ in range(40):
        fill()
    return recs


@gpu
@pytest.mark.parametrize("where", ["window", "window_edge", "tile_edge", "separated"])
def test_qname_hash_collisions(m, oracle, collisions, where):
    """different names with equal 32-bit hashes next to each other in the profile stream: the byte compare keeps them
    two inserts (plain profile, general pipeline); the fused pass's guard sees equal hashes and falls back"""
    recs = collision_stream(collisions, where)
    raw, off = E.stream(recs)
    T = 8
    hb = E.name_hash([E.qname(r) for r in recs if len(E.qname(r)) == 12])
    assert len(hb) - len(np.unique(hb)) >= len(collisions)
    opts = dict(besthit=True)
    eidx = oracle.filter_stream(raw, off, oracle.filter_cfg(**opts))
    for mode in MODES:
        for path in ("fused", "general", "plain"):
            idx = None if path == "plain" else eidx
            eab, est, eui, ed = oracle.profile(raw, off, idx, T, SHARE[mode])
            with m.Context(profile=True, multi=mode, kept=path != "fused", n_targets=T, **({} if path == "plain" else opts)) as ctx:
                ctx.push(raw, off)
                ui, d = ctx.pull_counts(); ab, st = ctx.finish_profile(); t = ctx.timing()
            profile_check(st, est, ui, eui, d, ed, ab, eab)
            assert eui[0] >= 2 * len(collisions) and eui[1] >= 2 * len(collisions)
            if path == "fused":
                assert (t["fused_chunks"], t["fused_fallbacks"]) == (1, 1)


# ================================================================ 3. coverage at target ends and bitmap words
COV_TLEN = [1, 2, 63, 64, 65, 127, 128, 129, 1000, 300, 4096]


def coverage_records(seed=17):
    rng = np.random.default_rng(seed)
    recs = []
    aux = lambda: E.aux_int("NM", "C", int(rng.integers(0, 3))) + E.aux_z("MD", "30A9") + E.aux_int("AS", "C", int(rng.integers(20, 60)))

    def add(tid, pos, cig):
        nm, a = b"c%07d" % len(recs), aux()
        recs.append(E.record(nm, tid=tid, pos=pos, cigar=cig, aux=a))
        if rng.random() < 0.2:                                        # a tied secondary: --besthit keeps both
            recs.append(E.record(nm, flag=0x100, tid=int(rng.integers(len(COV_TLEN))), pos=pos, cigar=cig, aux=a))
    for t, L in enumerate(COV_TLEN):
        add(t, 0, [(min(L, 40), M)])                                  # starts at 0
        add(t, 0, [(L, M)])                                           # covers the whole target
        add(t, max(L - 7, 0), [(min(L, 7), EQ)])                      # ends exactly at tlen
        for over in (1, 2, 63, 64, 65, 200):
            add(t, max(L - 5, 0), [(5 + over, M)])                    # runs past tlen
            add(t, max(L - 40, 0), [(3, S), (20, X), (2, I), (15 + over, EQ), (4, H)])
        add(t, L, [(10, M)])                                          # starts at tlen
        add(t, L + 37, [(10, M)])                                     # starts beyond it
        add(t, max(L - 3, 0), [(2, M), (6, D), (5, M)])               # a deletion across the end
        add(t, max(L - 3, 0), [(2, M), (60, N), (5, M)])              # a skip across the end
        add(t, -1, [(5, M)])                                          # no position: bases at -1 are dropped
        for a in (0, 1, 62, 63, 64, 65, 127, 128):
            for w in (1, 2, 63, 64, 65, 128, 129, 700):
                if a < L:
                    add(t, a, [(w, M)] if rng.random() < 0.7 else [(w // 2 + 1, EQ), (1, P), (w - w // 2 + 1, X)])
        add(t, 5, [(3, M), (9, 9), (2, 15), (3, M)])                 # undefined operations consume nothing
    rng.shuffle(recs)
    return recs


@gpu
@pytest.mark.parametrize("summary", [False, True], ids=["depth", "summary"])
@pytest.mark.parametrize("pre", [None, dict(l=5), dict(besthit=True)], ids=["plain", "fused", "besthit"])
def test_coverage_target_ends(m, oracle, pre, summary):
    """coverage of runs clamped at tlen, over targets of 1-4096 bases and runs starting / ending on bits 0 and 63 of a
    bitmap word; in the decode kernel (no filter, or a filter without best-hit) and after best-hit"""
    recs = cached("coverage", coverage_records)
    raw, off = E.stream(recs)
    tlen = np.array(COV_TLEN, dtype=np.uint32)
    idx = None if pre is None else oracle.filter_stream(raw, off, oracle.filter_cfg(**pre))
    ecov, et, es, edepth = oracle.coverage(raw, off, idx, tlen, want_depth=True)
    for how in ("staged", "device"):
        bufs = []
        with m.Context(coverage=True, coverage_summary=summary, n_targets=len(tlen), target_len=tlen, **(pre or {})) as ctx:
            push(m, ctx, raw, off, how, bufs)
            cov, touched, total = ctx.finish_coverage()
            assert np.array_equal(cov, ecov)
            assert np.array_equal(touched, et), (touched.tolist(), et.tolist())
            assert np.array_equal(total, es), (total.tolist(), es.tolist())
            if not summary:
                for t in range(len(tlen)):
                    assert np.array_equal(ctx.pull_coverage(t), edepth[t]), t
            release(ctx, bufs)
    assert (et > 0).all()
