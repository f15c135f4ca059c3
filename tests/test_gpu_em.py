"""The PropSharing loop (--multi=proportional, msam_profile.c:331-404) of every single-GPU implementation against the
CPU oracle, on streams built to reach the loop's boundaries.

msg_finish_profile runs the loop in one of four ways: em_loop_smem_kernel with 8 private inc copies per CTA (F <= 512)
or 1 copy (F <= 2048), em_loop_kernel with a[] and inc[] in global memory (F > 2048), or the host loop of
em_gather_kernel, em_update_kernel, em_delta_kernel and em_purged_kernel (MSG_EM_HOST_LOOP=1, read at every finish).
All of them walk the lists in grid stride (em_share_lists), a thread taking lists l and l + gsz together and then at
most one lone list; gsz = grid x 256, and the cooperative kernels' grid is nsm x min(occupancy, MSG_EM_CTAS or 3 / 4).
The tests cover:
- every implementation at F = 2 ... ~10 000;
- the pair / lone boundaries with MSG_EM_CTAS=1 (gsz = nsm x 256 exactly), list counts 2 gsz q + r, every list at a
  boundary on features of its own, so that a lost or misweighted list moves abundances by O(1);
- the 19-iteration cap: loops that stop at k = 18, converge at k = 19 and do not converge;
- list lengths 2 to 1 500, zero-sum lists (alone, as either half of a pair, long) and lists with U = 0 features;
- F = 0, F = 1, finishing twice, finishing between pushes, and pushes in 1 and 7 chunks.

Each stream runs through plain `profile`, the general pipeline (--besthit, kept records) and the fused pass (--besthit);
every record carries tied AS, so all three see the same lists.  Integers must equal the oracle's, abundances agree within
1e-9 relative and the DELTA^2 sequence within 1e-6.  The CPU-only tests check that the streams hold the intended
problem and that rounding cannot flip a stop decision (tests/emutil.py restates the loop in float64 and long double).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

import edgeutil as E
import emutil as X

HERE = os.path.dirname(os.path.abspath(__file__))
PROP = 3
PATHS = ("plain", "general", "fused")
IMPL_F = [2, 511, 512, 513, 2047, 2048, 2049, 10007]
CLASS_F = {"smem8": 300, "smem1": 1500, "global": 3000}       # F <= 512, 513-2048, > 2048
B200_SMS = 148                                                 # gsz of the CPU-side checks

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def m():
    import msamtools_b200 as mod
    assert mod._lib.load().msg_device_count() > 0, "no CUDA device: the GPU tests must not silently pass"
    return mod


def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def close(a, b, rel):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.shape != b.shape:
        return False
    both_nan = np.isnan(a) & np.isnan(b)
    return bool(np.all(both_nan | (np.abs(a - b) <= rel * np.maximum(np.abs(a), np.abs(b)))))


# ================================================================ problems: (U, (off, fid)) over F features
def mixed_problem(F, n_lists, seed):
    """U in 1..11 except features [0, nz) with U = 0; lists of 2-9 features (some with U = 0 features) and ~1% zero-sum
    lists over [0, nz) only"""
    rng = np.random.default_rng(seed)
    if F == 2:
        return np.array([1, 3]), X.csr([(0, 1), (1, 0)] * (n_lists // 2))
    nz = max(2, F // 10)
    U = rng.integers(1, 12, size=F)
    U[:nz] = 0
    lens = rng.choice([2, 2, 2, 3, 3, 4, 5, 6, 9], size=n_lists)
    lens = np.minimum(lens, F)
    off, fid = X.random_lists(rng, lens, 0, F)
    zl = np.nonzero(rng.random(n_lists) < 0.01)[0]
    if len(zl):
        zlen = np.minimum(lens[zl], nz)
        zoff, zfid = X.random_lists(rng, zlen, 0, nz)
        lens = lens.copy()
        lens[zl] = zlen
        off2 = np.zeros(n_lists + 1, dtype=np.int64)
        np.cumsum(lens, out=off2[1:])
        fid2 = np.empty(int(off2[-1]), dtype=np.int32)
        keep = np.ones(n_lists, dtype=bool)
        keep[zl] = False
        src = np.repeat(keep, np.diff(off))
        dst = np.repeat(keep, lens)
        fid2[dst] = fid[src]
        fid2[~dst] = zfid
        off, fid = off2, fid2
    return U, (off, fid)


def boundary_positions(nl, gsz):
    """list indices at which the grid-stride walk changes between pair and lone lists, in the first and in the last
    group of 2 gsz lists, and the last two lists"""
    base = [0, 1, gsz - 2, gsz - 1, gsz, gsz + 1, 2 * gsz - 2, 2 * gsz - 1]
    last = (nl // (2 * gsz)) * 2 * gsz
    pos = set(base) | {last + p for p in base} | {nl - 2, nl - 1}
    return sorted(p for p in pos if 0 <= p < nl)


def boundary_problem(F, nl, gsz, seed):
    """nl lists; the list at every boundary position is a sentinel on two features of its own (U = 1 and 2, 3 or 4);
    zero-sum lists at index 5 (first half of a pair once nl > gsz + 5) and gsz + 6 (second half, 9 features); the other
    lists have 2-33 features from a shared pool in which 10% of the features have U = 0"""
    rng = np.random.default_rng(seed)
    pos = boundary_positions(nl, gsz)
    S, nz = len(pos), 12
    p0 = 2 * S + nz
    assert F - p0 >= 64
    U = np.zeros(F, dtype=np.int64)
    U[0:2 * S:2] = 1
    U[1:2 * S:2] = 2 + np.arange(S) % 3
    U[p0:] = rng.integers(1, 10, size=F - p0) * (rng.random(F - p0) > 0.1)
    lens = rng.choice([2, 2, 2, 3, 3, 4, 5, 6, 8, 9, 17, 33], size=nl)
    zpos = [z for z in (5, gsz + 6) if z < nl and z not in pos]
    lens[pos] = 2
    for z, ln in zip(zpos, (2, 9)):
        lens[z] = ln
    off, fid = X.random_lists(rng, lens, p0, F)
    for j, p in enumerate(pos):
        fid[off[p]:off[p] + 2] = (2 * j, 2 * j + 1) if j % 2 else (2 * j + 1, 2 * j)
    for z in zpos:
        fid[off[z]:off[z + 1]] = 2 * S + np.arange(lens[z])
    return U, (off, fid)


def shapes_problem(F, seed):
    """lists of 2, 3, 4, 5, 8, 9, 33, 64 and 1500 features (those that fit F), zero-sum lists of 2, 5, 9 and 33 features
    next to the long ones, lists that mix U = 0 features with others"""
    rng = np.random.default_rng(seed)
    nz = 40
    U = rng.integers(1, 30, size=F)
    U[:nz] = 0
    U[nz:][rng.random(F - nz) < 0.15] = 0
    parts = []
    for ln in [2, 3, 4, 5, 8, 9, 33, 64]:
        if ln <= F - nz:
            parts.append(X.random_lists(rng, np.full(60, ln), nz, F))
            zl = min(ln, nz)
            parts.append(X.random_lists(rng, np.full(3, zl), 0, nz))
            parts.append(X.random_lists(rng, np.full(20, min(ln + 3, F)), 0, F))
    if 1500 <= F - nz:                   # > 1024 records: profile_big_kernel, whose lists go after the chunk's others
        parts.append(X.random_lists(rng, np.full(3, 1500), nz, F))
        parts.append(X.random_lists(rng, np.full(2, 33), 0, nz))
    return U, X.concat(*parts)


def cap_problem(F, iterations, converged):
    """one slow block on features 0-2, F - 3 unused features"""
    Ub, m1, m2 = X.slow_block(F, iterations, converged)
    U = np.zeros(F, dtype=np.int64)
    U[:3] = Ub
    return U, X.block_lists(0, m1, m2)


def default_grid_lists(nsm):
    """more lists than two grid strides at any occupancy (<= 4 CTAs per SM): pairs are taken"""
    return 2 * nsm * 4 * 256 + 1


def boundary_counts(gsz):
    return [2 * gsz * q + r for q in (0, 1) for r in (0, 1, gsz - 1, gsz, gsz + 1, 2 * gsz - 1)]


CAPS = [(18, 1), (19, 1), (19, 0)]
# seeds whose DELTA^2 sequences stay a factor 1.5 away from 1e-10 (test_stream_holds_problem); otherwise
# the seed is F (impl) or F + 1 (shapes)
SEEDS = {("impl", 10007): 10012, ("shapes", 1500): 1503}


def streams(nsm):
    """name -> (F, builder of (U, (off, fid))) of every problem the GPU tests run, for a GPU of nsm SMs"""
    out = {}
    for F in IMPL_F:
        out["impl-%d" % F] = (F, lambda F=F: mixed_problem(F, 20000, seed=SEEDS.get(("impl", F), F)))
    gsz = nsm * 256
    for cls, F in CLASS_F.items():
        for nl in boundary_counts(gsz):
            out["bound-%s-%d" % (cls, nl)] = (F, lambda F=F, nl=nl: boundary_problem(F, nl, gsz, seed=nl + F))
        out["grid-%s" % cls] = (F, lambda F=F: mixed_problem(F, default_grid_lists(nsm), seed=7 * F))
        for k, c in CAPS:
            out["cap-%s-%d%s" % (cls, k, "c" if c else "n")] = (F, lambda F=F, k=k, c=c: cap_problem(F, k, c))
        out["shapes-%s" % cls] = (F, lambda F=F: shapes_problem(F, seed=SEEDS.get(("shapes", F), F + 1)))
    out["life"] = (700, lambda: mixed_problem(700, 30000, seed=11))
    out["life-more"] = (700, lambda: mixed_problem(700, 9000, seed=12))
    return out


_built = {}


def build(name, nsm=B200_SMS):
    """(F, U, off, fid, raw, rec_off, T, fmap) of a named problem; the implementation streams go through an fmap from
    2F + 1 targets"""
    key = (name, nsm)
    if key not in _built:
        F, make = streams(nsm)[name]
        U, (off, fid) = make()
        T = 2 * F + 1 if name.startswith("impl-") else None
        raw, rec_off, fmap = X.lists_stream(U, off, fid, T=T)
        _built[key] = (F, U, off, fid, raw, rec_off, F if T is None else T, fmap)
    return _built[key]


_expected = {}


def expected(oracle, name, nsm=B200_SMS):
    key = (name, nsm)
    if key not in _expected:
        F, U, off, fid, raw, rec_off, T, fmap = build(name, nsm)
        eab, est, eui, _ = oracle.profile(raw, rec_off, None, T, PROP, fmap=fmap, n_features=F)
        _expected[key] = (eab, est, eui)
    return _expected[key]


# ================================================================ CPU-only: the streams and the restatement
CPU_NAMES = sorted(streams(B200_SMS))


@pytest.mark.parametrize("name", CPU_NAMES)
def test_stream_holds_problem(oracle, name):
    """the oracle sees exactly the intended lists and unique counts; the float64 restatement matches it; the long
    double restatement takes the same stop decision, and no DELTA^2 lies within a factor of 1.5 of 1e-10"""
    F, U, off, fid, raw, rec_off, T, fmap = build(name)
    eab, est, eui = expected(oracle, name)
    nl = len(off) - 1
    assert (est["n_lists"], est["n_entries"], est["multi"], est["uniq"]) == (nl, len(fid), nl, int(U.sum()))
    assert est["mapped_inserts"] == nl + int(U.sum())
    assert np.array_equal(eui, 2 * U)
    r = X.em_reference(U, off, fid, F)
    assert (r["iterations"], r["converged"], r["purged"]) == (est["iterations"], est["converged"], est["purged"])
    assert close(r["ab"], eab, 1e-12)
    assert close(r["delta"], est["delta"], 1e-7)          # DELTA^2 cancels: a ~ 1e2, a_new - a_old down to ~1e-5
    q = X.em_reference(U, off, fid, F, np.longdouble)
    assert (q["iterations"], q["converged"], q["purged"]) == (r["iterations"], r["converged"], r["purged"])
    assert X.decision_margin(q["delta"]), q["delta"]
    if name.startswith("cap-"):
        k, c = int(name[-3:-1]), name.endswith("c")
        assert (est["iterations"], est["converged"]) == (k, int(c))
    if name.startswith("shapes-") or name.startswith("bound-"):
        assert np.all(eab[U == 0][np.isin(np.nonzero(U == 0)[0], fid)] == 0)
        assert est["purged"] > 0 or nl <= 5


def test_builder_records(oracle):
    """the builder's records equal edgeutil.record's, every record survives --besthit, and an fmap moves records to
    other targets of the same feature without changing the profile"""
    U = np.array([1, 3, 0, 2, 0, 5])
    off, fid = X.csr([(0, 1), (1, 2, 3), (4, 2), (5, 0, 1, 3, 2)])
    raw, rec_off, _ = X.lists_stream(U, off, fid)
    recs = E.split(raw, rec_off)
    aux = E.aux_int("NM", "C", 0) + E.aux_z("MD", "40") + E.aux_int("AS", "C", 50)
    assert recs[0] == E.record(b"r000000000", tid=0, pos=100, cigar=[(40, E.M)], l_seq=0, aux=aux)
    assert recs[12] == E.record(b"r000000011", tid=1, pos=100, flag=0x100, cigar=[(40, E.M)], l_seq=0, aux=aux)
    assert len(recs) == U.sum() + len(fid)
    assert np.array_equal(oracle.filter_stream(raw, rec_off, oracle.filter_cfg(besthit=True)), np.arange(len(recs)))
    eab, est, _, _ = oracle.profile(raw, rec_off, None, 6, PROP)
    raw2, rec_off2, fmap = X.lists_stream(U, off, fid, T=13)
    assert not np.array_equal(raw, raw2)
    eab2, est2, _, _ = oracle.profile(raw2, rec_off2, None, 13, PROP, fmap=fmap, n_features=6)
    assert est == est2 and np.array_equal(eab, eab2) and est["purged"] == 1


def test_boundary_positions_cover_the_walk():
    """with nl = 2 gsz q + r, the sentinels sit where a thread's last step changes between a pair and a lone list"""
    gsz = 4 * 256
    for nl in boundary_counts(gsz):
        pos = boundary_positions(nl, gsz)
        # the lone list of thread t is at the first l = t + 2 gsz j with l + gsz >= nl, if l < nl
        lone = [l for l in range(nl) if l + gsz >= nl and (l % (2 * gsz)) < gsz]
        if lone:
            assert lone[0] in pos and lone[-1] in pos
        if nl > gsz:
            assert 0 in pos and gsz in pos                     # the first pair
        if nl:
            assert nl - 1 in pos


# ================================================================ GPU
def push_chunks(m, ctx, raw, off, chunks):
    """the stream in `chunks` msg_push_async calls cut at QNAME boundaries with split_point"""
    if chunks == 1:
        ctx.push(raw, off)
        return
    n = len(off) - 1
    cuts = sorted({0, n} | {int(m.split_point(raw, off, n * c // chunks)) for c in range(1, chunks)})
    assert len(cuts) == chunks + 1
    keep = []
    for a, b in zip(cuts, cuts[1:]):
        r = np.ascontiguousarray(raw[int(off[a]):int(off[b])])
        o = np.ascontiguousarray(off[a:b + 1] - off[a])
        keep.append((r, o))
        ctx.push_async(r, o)
    ctx.wait()


def run(m, raw, off, F, T, fmap, path, chunks=1):
    """(abundance, stats, ui, timing) of one context over the stream"""
    opts = {} if path == "plain" else dict(besthit=True)
    with m.Context(profile=True, multi="proportional", kept=path != "fused", n_targets=T, n_features=F, fmap=fmap, **opts) as ctx:
        push_chunks(m, ctx, raw, off, chunks)
        ui, _ = ctx.pull_counts()
        ab, st = ctx.finish_profile()
        t = ctx.timing()
    assert t["fused_chunks"] == (chunks if path == "fused" else 0)
    return ab, st, ui, t


def check(got, exp, what):
    ab, st, ui = got[:3]
    eab, est, eui = exp
    for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "converged", "n_lists", "n_entries"):
        assert st[k] == est[k], (what, k, st[k], est[k])
    assert np.array_equal(ui, eui), what
    assert close(ab, eab, 1e-9), (what, np.max(np.abs(ab - eab)))
    assert close(st["delta"], est["delta"], 1e-6), (what, st["delta"], est["delta"])


def run_named(m, oracle, name, paths=PATHS, nsm=B200_SMS):
    F, U, off, fid, raw, rec_off, T, fmap = build(name, nsm)
    exp = expected(oracle, name, nsm)
    if nsm != B200_SMS:                  # a stream the CPU-only tests have not certified
        assert X.decision_margin(X.em_reference(U, off, fid, F, np.longdouble)["delta"]), name
    for path in paths:
        got = run(m, raw, rec_off, F, T, fmap, path)
        check(got, exp, (name, path))
        assert np.all(got[0][U == 0] == 0), (name, path)          # a feature without unique reads stays exactly 0
    return exp


LOOPS = ["cooperative", "host"]


@pytest.fixture(params=LOOPS)
def loop(request, monkeypatch):
    if request.param == "host":
        monkeypatch.setenv("MSG_EM_HOST_LOOP", "1")
    else:
        monkeypatch.delenv("MSG_EM_HOST_LOOP", raising=False)
    return request.param


@gpu
@pytest.mark.parametrize("F", IMPL_F)
def test_implementations(m, oracle, loop, F):
    """each F picks em_loop_smem_kernel (8 or 1 inc copies), em_loop_kernel or, with MSG_EM_HOST_LOOP=1, the
    host-loop gather from shared or global memory; 20 000 lists through an fmap of 2F + 1 targets"""
    exp = run_named(m, oracle, "impl-%d" % F)
    assert exp[1]["iterations"] >= (2 if F == 2 else 5)


@gpu
@pytest.mark.parametrize("cls", list(CLASS_F))
@pytest.mark.parametrize("cap", ["18c", "19c", "19n"])
def test_iteration_cap(m, oracle, loop, cls, cap):
    """loops that converge at k = 18, converge at k = 19 (the last iteration) and stop unconverged after 19"""
    exp = run_named(m, oracle, "cap-%s-%s" % (cls, cap))
    assert (exp[1]["iterations"], exp[1]["converged"]) == (int(cap[:2]), int(cap[2] == "c"))


@gpu
@pytest.mark.parametrize("cls", list(CLASS_F))
def test_list_shapes(m, oracle, loop, cls):
    """lists of 2 to 1 500 features, zero-sum lists next to long ones, U = 0 features inside lists"""
    exp = run_named(m, oracle, "shapes-%s" % cls)
    assert exp[1]["purged"] > 0


@gpu
@pytest.mark.parametrize("cls", list(CLASS_F))
def test_default_grid_pairs(m, oracle, cls):
    """more than 2 x nsm x 4 x 256 lists: the cooperative kernels take list pairs at the default grid"""
    name = "grid-%s" % cls
    nsm = sm_count()
    assert len(build(name, nsm)[2]) - 1 == default_grid_lists(nsm)
    run_named(m, oracle, name, nsm=nsm)


@gpu
@pytest.mark.skipif(os.environ.get("MSG_EM_CTAS") != "1", reason="runs in a child process with MSG_EM_CTAS=1 (test_pair_boundaries_one_cta_per_sm)")
@pytest.mark.parametrize("cls", list(CLASS_F))
@pytest.mark.parametrize("which", range(12))
def test_boundary_ctas1(m, oracle, cls, which):
    nsm = sm_count()
    nl = boundary_counts(nsm * 256)[which]
    name = "bound-%s-%d" % (cls, nl)
    # plain and general keep stream order in the CSR, so the sentinels sit at their positions; fused only at the largest count
    run_named(m, oracle, name, paths=PATHS if which == 11 else ("plain", "general"), nsm=nsm)


@gpu
def test_pair_boundaries_one_cta_per_sm():
    """MSG_EM_CTAS=1 (read once per process, so in a child): one CTA per SM, gsz = nsm x 256; list counts
    2 gsz q + r, q in {0, 1}, r in {0, 1, gsz - 1, gsz, gsz + 1, 2 gsz - 1}, in all three cooperative configurations"""
    env = dict(os.environ, MSG_EM_CTAS="1")
    env.pop("MSG_EM_HOST_LOOP", None)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", "-m", "gpu", "-k", "boundary_ctas1", __file__],
                       cwd=os.path.dirname(HERE), env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert "36 passed" in r.stdout, r.stdout[-2000:]


# ---------------------------------------------------------------- lifecycle
@gpu
@pytest.mark.parametrize("path", PATHS)
def test_no_features(m, oracle, loop, path):
    """F = 0 with n_targets = 0 and only unmapped records: 19 iterations, not converged, DELTA^2 NaN (0 / 0)"""
    aux = E.aux_int("AS", "C", 0)
    recs = [E.record(b"u%03d" % (k // 2), flag=4 | (0x41 if k % 2 == 0 else 0x81) | 1, tid=-1, pos=-1, cigar=[], aux=aux) for k in range(40)]
    raw, off = E.stream(recs)
    eab, est, eui, _ = oracle.profile(raw, off, None, 0, PROP)
    assert (est["iterations"], est["converged"]) == (19, 0) and np.all(np.isnan(est["delta"]))
    got = run(m, raw, off, 0, 0, None, path)
    check(got, (eab, est, eui), path)


@gpu
@pytest.mark.parametrize("path", PATHS)
def test_one_feature(m, oracle, loop, path):
    U = np.array([7])
    raw, off, _ = X.lists_stream(U, *X.csr([]))
    eab, est, eui, _ = oracle.profile(raw, off, None, 1, PROP)
    check(run(m, raw, off, 1, 1, None, path), (eab, est, eui), path)
    assert est["iterations"] == 1 and eab[0] == 7


@gpu
@pytest.mark.parametrize("path", PATHS)
def test_finish_twice_and_between_pushes(m, oracle, path):
    """finish twice on one state gives the same result; finish, push more, finish equals the oracle on the
    concatenated stream"""
    F, U, off, fid, raw, rec_off, T, fmap = build("life")
    exp = expected(oracle, "life")
    F2, U2, off2, fid2, raw2, rec_off2, _, _ = build("life-more")
    both_raw = np.concatenate([raw, raw2])
    both_off = np.concatenate([rec_off, rec_off2[1:] + rec_off[-1]])
    eab, est, eui, _ = oracle.profile(both_raw, both_off, None, T, PROP)
    opts = {} if path == "plain" else dict(besthit=True)
    with m.Context(profile=True, multi="proportional", kept=path != "fused", n_targets=T, **opts) as ctx:
        ctx.push(raw, rec_off)
        ui, _ = ctx.pull_counts()
        first = ctx.finish_profile()
        again = ctx.finish_profile()
        check((first[0], first[1], ui), exp, (path, "first"))
        check((again[0], again[1], ui), exp, (path, "again"))
        ctx.push(raw2, rec_off2)
        ui, _ = ctx.pull_counts()
        ab, st = ctx.finish_profile()
    check((ab, st, ui), (eab, est, eui), (path, "more"))


@gpu
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("chunks", [1, 7])
def test_chunked_pushes(m, oracle, path, chunks):
    F, U, off, fid, raw, rec_off, T, fmap = build("life")
    check(run(m, raw, rec_off, F, T, fmap, path, chunks=chunks), expected(oracle, "life"), (path, chunks))
