"""Exact mode (msg_config.exact, Context(exact=True), MSAMTOOLS_EXACT=1): --multi=equal and --multi=proportional
abundances bit-identical to the CPU oracle, which restates the reference line for line.

"Equal to the oracle" below means: abundance and d[] equal as uint64 views, ui[] equal, and the same insert counters,
iterations, converged flag and purged count.  Runs with MSG_EXACT_DELTA=seq (read once per process, so in a child) take
the sequential DELTA^2 in every iteration and must also give the oracle's em_delta bits.

Covered: both modes on the seeded synthetic streams with and without a genome map, through plain `profile`, the general
pipeline and the fused pass; PropSharing problems from tests/emutil.py (slow blocks that stop at iteration 19 with and
without convergence, F from 1 to 10^6, the genes1m shape of tests/test_gpu_largeF.py); a feature in 120 000 lists and
buckets of 2047, 2048 and 2049 entries (shared-memory and global-memory bucket sorts); chunks the fused guard declines
and groups of more than 1024 records (profile_big_kernel); 1, 7 and ~2000 chunks by push, push_async,
push_device_async and pinned zero-copy; finish twice, push after finish, reset; a shuffled stream on a collating
context, also with MSG_COLLATE_CHUNK_RECORDS=1000; the host loop (MSG_EM_HOST_LOOP=1); the n_ranks refusal; and the
CLI's MSAMTOOLS_EXACT=1 (on the GPU against the oracle, and on the null device under ASan/UBSan).
"""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import collateutil as CU
import edgeutil as E
import emutil as X

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SHARE = {"equal": 2, "proportional": 3}
M = E.M
gpu = pytest.mark.gpu
IN_SEQ_CHILD = os.environ.get("MSG_EXACT_DELTA") == "seq"
IN_COLLATE_CHILD = os.environ.get("MSG_COLLATE_CHUNK_RECORDS") == "1000"


@pytest.fixture(scope="module")
def m():
    import msamtools_b200 as mod
    assert mod._lib.load().msg_device_count() > 0, "no CUDA device: the GPU tests must not silently pass"
    return mod


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def assert_exact(got, exp, delta=False):
    ab, st, ui, d = got
    eab, est, eui, ed = exp
    assert np.array_equal(ui, eui), "ui differs"
    assert np.array_equal(bits(d), bits(ed)), "d differs in %d features" % int(np.count_nonzero(bits(d) != bits(ed)))
    for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "converged"):
        assert st[k] == est[k], (k, st[k], est[k])
    nd = int(np.count_nonzero(bits(ab) != bits(eab)))
    assert nd == 0, "abundance differs in %d of %d features" % (nd, len(ab))
    if delta:
        assert np.array_equal(bits(st["delta"]), bits(est["delta"])), (st["delta"], est["delta"])


def expected(oracle, raw, off, mode, T, path="plain", fmap=None, F=None, opts=None):
    idx = None if path == "plain" else oracle.filter_stream(raw, off, oracle.filter_cfg(**(opts or dict(besthit=True))))
    return oracle.profile(raw, off, idx, T, SHARE[mode], fmap=fmap, n_features=F)


def cut_points(m, raw, off, chunks):
    n = len(off) - 1
    pts = sorted({0, n} | {m.split_point(raw, off, (n * k) // chunks) for k in range(1, chunks)})
    return list(zip(pts[:-1], pts[1:]))


def run(m, raw, off, mode, T, *, path="plain", fmap=None, F=None, chunks=1, push="push", opts=None, exact=True, timing=False):
    """push the stream in `chunks` pieces by one push kind; returns (ab, st, ui, d) [+ timing]"""
    opts = {} if path == "plain" else (opts or dict(besthit=True))
    with m.Context(profile=True, multi=mode, kept=path == "general", n_targets=T, n_features=F, fmap=fmap, exact=exact, **opts) as ctx:
        keep = []
        if push == "pinned":
            pb = m.PinnedBuffer(max(raw.nbytes, 1))
            pb.array[:raw.nbytes] = raw
            keep.append(pb)
        for a, b in cut_points(m, raw, off, chunks):
            lo, hi = int(off[a]), int(off[b])
            sub_off = np.ascontiguousarray(off[a:b + 1] - off[a], dtype=np.uint64)
            if push == "push":
                ctx.push(raw[lo:hi], sub_off)
            elif push == "async":
                sub = np.ascontiguousarray(raw[lo:hi])
                keep.append((sub, sub_off))
                ctx.push_async(sub, sub_off)
            elif push == "pinned":
                ctx.push(keep[0].array[lo:hi], sub_off)
            else:
                dr, do = ctx.device_alloc(max(hi - lo, 1)), ctx.device_alloc(sub_off.nbytes)
                ctx.device_upload(dr, raw[lo:hi]); ctx.device_upload(do, sub_off)
                keep.append((dr, do))
                ctx.push_device_async(dr, hi - lo, do, b - a)
        ctx.wait()
        ui, d = ctx.pull_counts()
        ab, st = ctx.finish_profile()
        t = ctx.timing()
        for k in keep:
            if isinstance(k, tuple) and not isinstance(k[0], np.ndarray):
                ctx.device_free(k[0]); ctx.device_free(k[1])
        if push == "pinned":
            keep[0].close()
    return ((ab, st, ui, d), t) if timing else (ab, st, ui, d)


# ================================================================ streams
_cache = {}


def cached(key, make):
    if key not in _cache:
        _cache[key] = make()
    return _cache[key]


def mixed():
    """the seeded `mixed` synthetic stream of tests/test_gpu_parity.py"""
    def make():
        from msamtools_b200 import synth
        p = synth.make_params("mixed", n_records=60_000, seed=24680)
        raw, off, _ = synth.generate(p)
        return raw, off, len(synth.target_lengths(p))
    return cached("mixed", make)


def em_problem(F, seed, n_lists=None):
    """U in 0..11 (10 % zero), random lists of 2-6 distinct features, and for 3 <= F <= 2049 a slow block on features
    0-2 (alone it runs all 19 iterations; the random lists can end the loop earlier, as at F = 97)"""
    rng = np.random.default_rng(seed)
    if F == 1:
        return np.array([7]), X.csr([])
    if F == 2:
        return np.array([1, 3]), X.csr([(0, 1), (1, 0)] * 50)
    U = rng.integers(0, 12, size=F)
    U[rng.random(F) < 0.1] = 0
    nl = n_lists if n_lists is not None else min(3 * F, 60_000)
    lens = np.minimum(rng.choice([2, 2, 3, 3, 4, 6], size=nl), F)
    lists = X.random_lists(rng, lens, 0, F)
    if F > 2049:
        return U, lists
    bu, m1, m2 = X.slow_block(F, 19, 0)
    U[:3] = bu
    return U, X.concat(X.block_lists(0, m1, m2), lists)


def problem_stream(F, seed, n_lists=None):
    def make():
        U, (off, fid) = em_problem(F, seed, n_lists)
        raw, rec_off, _ = X.lists_stream(U, off, fid)
        return raw, rec_off
    return cached(("em", F, seed, n_lists), make)


def heavy_stream():
    """feature 0 in 120 000 three-feature lists; features 1-3 in 2049, 4-6 in 2047, 7-9 in 2048 lists; lists shuffled"""
    def make():
        rng = np.random.default_rng(4242)
        F = 120
        lists = [(0, 10 + i % 50, 60 + (i * 7) % 50) for i in range(120_000)]
        lists += [(1, 2, 3)] * 2049 + [(4, 5, 6)] * 2047 + [(7, 8, 9)] * 2048
        perm = rng.permutation(len(lists))
        lists = [lists[i] for i in perm]
        U = rng.integers(1, 5, size=F)
        raw, off, _ = X.lists_stream(U, *X.csr(lists))
        return raw, off, F
    return cached("heavy", make)


def decline_stream():
    """grouped reads of 1-6 tied records, with reopened names (x, a read dropped by -l 8, x again: two pools, one
    insert, so the fused guard declines that chunk) at three places and one read of 5000 alignments (> 1024 records:
    the fused walk declines it and the general pipeline's profile_big_kernel counts it)"""
    def make():
        rng = np.random.default_rng(99)
        T = 40
        aux = E.aux_int("NM", "C", 0) + E.aux_z("MD", "40") + E.aux_int("AS", "C", 50)
        recs = []
        for q in range(3000):
            name = b"g%05d" % q
            if q in (400, 1500, 2600):
                recs.append(E.record(name, tid=int(rng.integers(T)), pos=5, cigar=[(40, M)], aux=aux))
                recs.append(E.record(b"y%05d" % q, tid=1, pos=5, cigar=[(5, M)], aux=aux))
                recs.append(E.record(name, tid=int(rng.integers(T)), pos=5, cigar=[(40, M)], aux=aux))
                recs.append(E.record(name, flag=0x100, tid=int(rng.integers(T)), pos=5, cigar=[(40, M)], aux=aux))
                continue
            if q == 2000:
                for k in range(5000):
                    recs.append(E.record(name, flag=0x100 if k else 0, tid=int(rng.integers(T)), pos=5, cigar=[(40, M)], aux=aux))
                continue
            ts = rng.choice(T, size=int(rng.integers(1, 7)), replace=False)
            for j, t in enumerate(ts):
                recs.append(E.record(name, flag=0x100 if j else 0, tid=int(t), pos=5, cigar=[(40, M)], aux=aux))
        raw, off = E.stream(recs)
        return raw, off, T
    return cached("decline", make)


# ================================================================ GPU
MODES = list(SHARE)


@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("path", ["plain", "general", "fused"])
@pytest.mark.parametrize("genome", [False, True], ids=["targets", "genomes"])
def test_synth_modes(m, oracle, mode, path, genome):
    raw, off, T = mixed()
    fmap, F = ((np.arange(T) % 7).astype(np.int32), 7) if genome else (None, None)
    opts = dict(l=80, p=95, z=80, besthit=True)
    exp = expected(oracle, raw, off, mode, T, path, fmap, F, opts)
    got, t = run(m, raw, off, mode, T, path=path, fmap=fmap, F=F, opts=opts, timing=True)
    assert_exact(got, exp)
    assert t["fused_chunks"] == (path == "fused") and t["fused_fallbacks"] == 0
    assert exp[1]["multi"] > 0


@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("push,chunks,path", [("push", 1, "fused"), ("push", 7, "fused"), ("push", 2000, "fused"), ("async", 7, "fused"),
                                              ("async", 2000, "fused"), ("device", 1, "fused"), ("device", 7, "fused"), ("pinned", 1, "fused"),
                                              ("pinned", 7, "fused"), ("push", 7, "general"), ("push", 2000, "plain"), ("device", 7, "plain")])
def test_chunking_and_push_kinds(m, oracle, mode, push, chunks, path):
    raw, off, T = mixed()
    exp = expected(oracle, raw, off, mode, T, path)
    assert_exact(run(m, raw, off, mode, T, path=path, chunks=chunks, push=push), exp)


EM_F = [1, 2, 3, 97, 2048, 2049, 10_007, 100_003, 1_000_000]


@gpu
@pytest.mark.parametrize("F", EM_F)
def test_em_problems(m, oracle, F):
    """PropSharing problems with a slow block; the cooperative loop and the host loop"""
    raw, off = problem_stream(F, 17 + F)
    exp = oracle.profile(raw, off, None, F, 3)
    if F in (3, 2048, 2049):                       # the slow block dominates: all 19 iterations
        assert exp[1]["iterations"] == 19
    assert_exact(run(m, raw, off, "proportional", F), exp)
    os.environ["MSG_EM_HOST_LOOP"] = "1"
    try:
        assert_exact(run(m, raw, off, "proportional", F, chunks=3), exp)
    finally:
        del os.environ["MSG_EM_HOST_LOOP"]


@gpu
@pytest.mark.parametrize("path", ["plain", "fused"])
def test_converges_at_19(m, oracle, path):
    bu, m1, m2 = X.slow_block(3, 19, 1)
    raw, roff, _ = X.lists_stream(bu, *X.block_lists(0, m1, m2))
    exp = expected(oracle, raw, roff, "proportional", 3, path)
    assert (exp[1]["iterations"], exp[1]["converged"]) == (19, 1)
    assert_exact(run(m, raw, roff, "proportional", 3, path=path), exp)


@gpu
@pytest.mark.parametrize("path", ["plain", "fused"])
def test_genes1m_shape(m, oracle, path):
    """the genes1m preset of tests/test_gpu_largeF.py (10^6 features), 2 M records, filtered for the fused pass"""
    from msamtools_b200 import synth
    p = synth.make_params("genes1m", n_records=2_000_000, seed=97531)
    raw, off, _ = synth.generate(p)
    T = len(synth.target_lengths(p))
    opts = dict(l=80, p=95, z=80, besthit=True)
    for mode in MODES:
        assert_exact(run(m, raw, off, mode, T, path=path, opts=opts, chunks=3), expected(oracle, raw, off, mode, T, path, opts=opts))


@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("path", ["plain", "fused"])
def test_heavy_features(m, oracle, mode, path):
    raw, off, F = heavy_stream()
    exp = expected(oracle, raw, off, mode, F, path)
    assert_exact(run(m, raw, off, mode, F, path=path, chunks=5), exp)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_declined_chunks_and_big_groups(m, oracle, mode):
    raw, off, T = decline_stream()
    opts = dict(l=8, besthit=True)
    for path, chunks in (("fused", 7), ("fused", 1), ("general", 7), ("plain", 7)):
        exp = expected(oracle, raw, off, mode, T, path, opts=opts)
        got, t = run(m, raw, off, mode, T, path=path, chunks=chunks, opts=opts, timing=True)
        assert_exact(got, exp)
        if path == "fused":
            assert t["fused_fallbacks"] >= (3 if chunks == 7 else 1), t
            assert t["fused_fallbacks"] < t["fused_chunks"] or chunks == 1


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_scopes(m, oracle, mode):
    """finish twice, push after a finish, pull_counts before and after, reset"""
    raw, off, T = mixed()
    n = len(off) - 1
    h = m.split_point(raw, off, n // 2)
    r1, o1 = raw[:int(off[h])], off[:h + 1]
    r2, o2 = raw[int(off[h]):], off[h:] - off[h]
    e1 = expected(oracle, r1, o1, mode, T)
    e2 = expected(oracle, r2, o2, mode, T)
    eall = expected(oracle, raw, off, mode, T)
    with m.Context(profile=True, multi=mode, n_targets=T, exact=True) as ctx:
        ctx.push(r1, o1)
        ui, d = ctx.pull_counts()
        a1, s1 = ctx.finish_profile()
        assert_exact((a1, s1, ui, d), e1)
        a1b, s1b = ctx.finish_profile()
        assert_exact((a1b, s1b, ui, d), e1)
        ctx.push(r2, o2)
        a, s = ctx.finish_profile()
        ui, d = ctx.pull_counts()
        assert_exact((a, s, ui, d), eall)
        ctx.reset()
        ctx.push(r2, o2)
        ui, d = ctx.pull_counts()
        a, s = ctx.finish_profile()
        assert_exact((a, s, ui, d), e2)


def _collate_case(m, oracle, mode):
    raw, off, T = mixed()
    n = len(off) - 1
    perm = np.random.default_rng(5).permutation(n)
    sraw, soff = CU.stream_of(raw, off, perm)
    order, _ = CU.grouped_order(sraw, soff)
    graw, goff = CU.stream_of(sraw, soff, order)
    exp = expected(oracle, graw, goff, mode, T)
    for chunks in (1, 7):
        with m.Context(profile=True, multi=mode, n_targets=T, collate=True, kept=False, exact=True) as ctx:
            for a, b in zip([n * k // chunks for k in range(chunks)], [n * (k + 1) // chunks for k in range(chunks)]):
                ctx.push(sraw[int(soff[a]):int(soff[b])], soff[a:b + 1] - soff[a])
            ui, d = ctx.pull_counts()
            ab, st = ctx.finish_profile()
        assert_exact((ab, st, ui, d), exp)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_collate(m, oracle, mode):
    _collate_case(m, oracle, mode)


@gpu
@pytest.mark.skipif(not IN_COLLATE_CHILD, reason="runs in a child process with MSG_COLLATE_CHUNK_RECORDS=1000 (test_collate_small_chunks)")
@pytest.mark.parametrize("mode", MODES)
def test_collate_child(m, oracle, mode):
    _collate_case(m, oracle, mode)


@gpu
@pytest.mark.skipif(not IN_SEQ_CHILD, reason="runs in a child process with MSG_EXACT_DELTA=seq (test_sequential_delta)")
@pytest.mark.parametrize("F", [2, 3, 97, 2049, 100_003])
def test_seq_delta_child(m, oracle, F):
    raw, off = problem_stream(F, 17 + F)
    exp = oracle.profile(raw, off, None, F, 3)
    assert_exact(run(m, raw, off, "proportional", F), exp, delta=True)
    assert_exact(run(m, raw, off, "proportional", F, path="fused", chunks=4, push="async"), expected(oracle, raw, off, "proportional", F, "fused"), delta=True)
    os.environ["MSG_EM_HOST_LOOP"] = "1"
    try:
        assert_exact(run(m, raw, off, "proportional", F), exp, delta=True)
    finally:
        del os.environ["MSG_EM_HOST_LOOP"]


@gpu
@pytest.mark.skipif(not IN_SEQ_CHILD, reason="runs in a child process with MSG_EXACT_DELTA=seq (test_sequential_delta)")
def test_seq_delta_child_heavy(m, oracle):
    raw, off, F = heavy_stream()
    assert_exact(run(m, raw, off, "proportional", F), expected(oracle, raw, off, "proportional", F), delta=True)


def _child(k, env, count):
    env = dict(os.environ, **env)
    env.pop("MSG_EM_HOST_LOOP", None)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", "-m", "gpu", "-k", k, __file__],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert f"{count} passed" in r.stdout, r.stdout[-2000:]


@gpu
def test_sequential_delta():
    """MSG_EXACT_DELTA=seq: every DELTA^2 is the sequential sum, bit-equal to the oracle's"""
    _child("seq_delta_child", dict(MSG_EXACT_DELTA="seq"), 6)


@gpu
def test_collate_small_chunks():
    """a collating context that hands the grouped stream to the pipeline in chunks of at most 1000 records"""
    _child("collate_child", dict(MSG_COLLATE_CHUNK_RECORDS="1000"), 2)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_cli_table_is_the_oracles(oracle, tmp_path, mode):
    """MSAMTOOLS_EXACT=1 msamtools profile: every value of the table is "%.8g" of the oracle's abundance, and the
    table does not depend on the chunking"""
    import samutil
    from msamtools_b200 import synth
    p = synth.make_params("mixed", n_records=200_000, seed=31337)
    raw, off, _ = synth.generate(p)
    tlen = synth.target_lengths(p)
    names = [f"ref{i:04d}" for i in range(len(tlen))]
    path = str(tmp_path / "in.bam")
    samutil.write_bam(path, samutil.synth_header(names, tlen), names, tlen, raw[:int(off[-1])])
    eab, est, _, _ = oracle.profile(raw, off, None, len(tlen), SHARE[mode])
    cli = os.path.join(ROOT, "msamtools_b200", "bin", "msamtools")
    tables = []
    for chunk in ("7001", "524288"):
        outp = str(tmp_path / f"p{chunk}.gz")
        r = subprocess.run([cli, "profile", "--label", "X", "--unit", "ab", "--nolen", "--multi", mode, "-o", outp, path],
                           env=dict(os.environ, MSAMTOOLS_EXACT="1", MSAMTOOLS_CHUNK_RECORDS=chunk), capture_output=True)
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        comments, body = samutil.read_profile_gz(outp)
        assert [k for k, _ in body[2:]] == names
        assert [v for _, v in body[2:]] == ["%.8g" % x for x in eab]
        tables.append(body)
    assert tables[0] == tables[1]


# ================================================================ CPU
def test_refuses_several_ranks():
    import msamtools_b200 as mod
    with pytest.raises(mod.MsgError) as ei:
        mod.Context(profile=True, multi="proportional", n_targets=4, n_ranks=2, rank=0, nccl_unique_id=b"\0" * 128, exact=True)
    assert ei.value.code == mod._lib.MSG_EINVAL and "n_ranks" in str(ei.value)


def test_cli_exact_knob_on_null_device(tmp_path):
    """MSAMTOOLS_EXACT=1 on the null device under ASan/UBSan: the knob only sets msg_config.exact, so the run is clean
    and its table equals the run without it"""
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    import test_cli_host_nulldev as N
    import samutil
    from msamtools_b200 import synth
    cli = N.build(str(tmp_path), "address,undefined")
    p = synth.make_params("mixed", n_records=20_000, seed=3)
    raw, off, _ = synth.generate(p)
    tlen = synth.target_lengths(p)
    names = [f"ref{i:04d}" for i in range(len(tlen))]
    path = str(tmp_path / "in.bam")
    samutil.write_bam(path, samutil.synth_header(names, tlen), names, tlen, raw[:int(off[-1])])
    out = []
    for exact in ("0", "1"):
        outp = str(tmp_path / f"p{exact}.gz")
        r = subprocess.run([cli, "profile", "--label", "S", "--multi", "prop", "-o", outp, path], capture_output=True,
                           env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0", MSAMTOOLS_EXACT=exact, MSAMTOOLS_CHUNK_RECORDS="3000"))
        assert r.returncode == 0, r.stderr.decode()[-3000:]
        out.append(samutil.read_profile_gz(outp)[1])
    assert out[0] == out[1] and len(out[0]) == len(names) + 2
