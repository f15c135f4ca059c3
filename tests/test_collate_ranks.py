"""Collation across ranks: msg_config.collate = MSG_COLLATE_RANKS (2) with n_ranks > 1.

Every rank pushes a piece of a stream in any order (cut at arbitrary record counts, not at QNAME boundaries); at the first
finish the ranks exchange record heads so that a record goes to rank floor(key * N / 2^64) of its 64-bit QNAME key
(collateutil.keys), and each rank collates what it received.  The input is rank 0's pushes, then rank 1's, and so on, so
the results must equal the oracle on the whole stream regrouped stably by QNAME: integers exactly, abundances within
1e-9 relative with the same PropSharing iteration count, and bit-identical vectors on every rank.

CPU: the destination rule restated in numpy -- one destination per read, the rank-order concatenation of the ranks'
grouped orders equals collateutil.grouped_order of the whole stream, and the oracle's integers summed over the ranks'
streams equal the whole stream's.  GPU (-m gpu, WORLD = MSG_TEST_WORLD devices, default 2): parity on coordinate-ordered
and shuffled streams, gene catalogues (reduce-scatter exchange) and the NCCL loop, exact routing (each rank's counts are
the oracle's over the reads the rule sends it), mixed push kinds, an empty rank, one read on all ranks, forced hash
collisions with many grouped chunks, scopes and reset, a record error on one rank, and the refused configurations.
"""
import multiprocessing
import os
import sys

import numpy as np
import pytest

import collateutil as CU
import edgeutil as E
from conftest import ROOT

WORLD = int(os.environ.get("MSG_TEST_WORLD", "2"))
REL = 1e-9
SHARE = {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}
FILT = dict(l=80, p=95, z=80)
JOIN_TIMEOUT_S = 600


# ================================================================ restatement
def dest(keys, n_ranks):
    """floor(key * N / 2^64), the 64x64 -> high-64 multiply of coll_dest, in two 32-bit halves"""
    k = np.asarray(keys, dtype=np.uint64)
    N = np.uint64(n_ranks)
    lo = (k & np.uint64(0xffffffff)) * N
    hi = (k >> np.uint64(32)) * N + (lo >> np.uint64(32))
    return (hi >> np.uint64(32)).astype(np.int64)


def log2_ceil(n):
    b = 0
    while (1 << b) < n:
        b += 1
    return b


def regroup_perm(raw, off):
    """the permutation that groups a stream stably by QNAME (groups by first appearance, records in input order)"""
    lq, m = CU.names_all(raw, off)
    full = np.zeros((len(lq), m.shape[1] + 1), dtype=np.uint8)
    full[:, 0] = lq
    full[:, 1:] = m
    _, first, inv = np.unique(np.ascontiguousarray(full).view(np.dtype((np.void, full.shape[1]))).ravel(),
                              return_index=True, return_inverse=True)
    return np.lexsort((np.arange(len(lq)), first[inv.ravel()]))


def regroup(raw, off):
    return CU.stream_of(raw, off, regroup_perm(raw, off))


def _i32(raw, off, at):
    o = np.asarray(off[:-1], dtype=np.int64) + at
    return np.ascontiguousarray(raw[o[:, None] + np.arange(4)]).view("<i4").ravel()


def coord_perm(raw, off):
    """by (tid, pos) with unmapped / tid -1 records last, as test_collate.reorder(..., "coord")"""
    tid, pos = _i32(raw, off, 4), _i32(raw, off, 8)
    o = np.asarray(off[:-1], dtype=np.int64)
    flag = raw[o + 18].astype(np.int64) | (raw[o + 19].astype(np.int64) << 8)
    unm = (tid < 0) | ((flag & 4) != 0)
    return np.lexsort((np.arange(len(tid)), pos, tid, unm))


def synth_stream(preset, n, seed, order):
    from msamtools_b200 import synth
    p = synth.make_params(preset, n_records=n, seed=seed)
    raw, off, _ = synth.generate(p)
    raw, off = np.ascontiguousarray(raw[:int(off[-1])]), off.astype(np.uint64)
    perm = coord_perm(raw, off) if order == "coord" else np.random.default_rng(seed).permutation(len(off) - 1)
    r2, o2 = CU.stream_of(raw, off, perm)
    return r2, o2, synth.target_lengths(p)


def per_rank_grouped(raw, off, n_ranks, bits=64):
    """global ordinals in the order the ranks' grouped streams hold them, concatenated in rank order: each rank sorts
    what it receives by (local bucket of bucket_bits(n) + ceil(log2 N) bits, key, global ordinal), collision runs by name"""
    k = CU.keys(raw, off, bits)
    d = dest(k, n_ranks)
    out = []
    for r in range(n_ranks):
        ords = np.flatnonzero(d == r)
        if not len(ords):
            continue
        sraw, soff = CU.stream_of(raw, off, ords)
        order, ks = CU.grouped_order(sraw, soff, bits)
        b = CU.bucket_of(ks, min(24, CU.bucket_bits(len(ords)) + log2_ceil(n_ranks)))
        assert np.all(np.diff(b) >= 0)                     # the buckets follow the key order
        out.append(ords[order])
    return np.concatenate(out) if out else np.zeros(0, dtype=np.int64)


# ================================================================ CPU
@pytest.mark.parametrize("bits", [64, 8])
@pytest.mark.parametrize("n_ranks", [2, 3, 4, 8])
def test_every_read_has_one_destination(n_ranks, bits):
    raw, off, _ = synth_stream("mixed", 20000, 11, "shuffle")
    k = CU.keys(raw, off, bits)
    d = dest(k, n_ranks)
    assert d.min() >= 0 and d.max() < n_ranks
    lq, m = CU.names_all(raw, off)
    names = np.ascontiguousarray(np.concatenate([lq[:, None].astype(np.uint8), m], axis=1))
    _, inv = np.unique(names.view(np.dtype((np.void, names.shape[1]))).ravel(), return_inverse=True)
    inv = inv.ravel()
    lo, hi = np.full(inv.max() + 1, n_ranks), np.full(inv.max() + 1, -1)
    np.minimum.at(lo, inv, d)
    np.maximum.at(hi, inv, d)
    assert np.array_equal(lo, hi)
    o = np.argsort(k, kind="stable")                       # ranks hold contiguous key ranges, in rank order
    assert np.all(np.diff(d[o]) >= 0)
    if bits == 64:
        assert len(np.unique(d)) == n_ranks


@pytest.mark.parametrize("bits", [64, 8])
@pytest.mark.parametrize("n_ranks", [2, 3, 4, 8])
@pytest.mark.parametrize("order", ["coord", "shuffle"])
def test_rank_order_concatenation_is_the_single_gpu_grouped_order(n_ranks, bits, order):
    raw, off, _ = synth_stream("community", 30000, 13, order)
    whole, _ = CU.grouped_order(raw, off, bits)
    assert np.array_equal(per_rank_grouped(raw, off, n_ranks, bits), whole)


@pytest.mark.parametrize("n_ranks", [2, 3, 8])
def test_oracle_integers_add_up_over_the_ranks(oracle, n_ranks):
    raw, off, tl = synth_stream("mixed", 20000, 17, "coord")
    T = len(tl)
    cfg = oracle.filter_cfg(besthit=True, **FILT)
    g, go = regroup(raw, off)
    idx = oracle.filter_stream(g, go, cfg)
    _, est, eui, _ = oracle.profile(g, go, idx, T, SHARE["proportional"])
    d = dest(CU.keys(raw, off), n_ranks)
    tot = dict(mapped_inserts=0, uniq=0, multi=0, n_lists=0, n_entries=0)
    ui = np.zeros_like(eui)
    for r in range(n_ranks):
        sraw, soff = CU.stream_of(raw, off, np.flatnonzero(d == r))
        sg, sgo = regroup(sraw, soff)
        sidx = oracle.filter_stream(sg, sgo, cfg)
        _, st, u, _ = oracle.profile(sg, sgo, sidx, T, SHARE["proportional"])
        for key in tot:
            tot[key] += st[key]
        ui += u
    assert np.array_equal(ui, eui)
    for key in tot:
        assert tot[key] == est[key], key


# ================================================================ GPU: ranks in spawned processes
def _ndev():
    try:
        import msamtools_b200 as m
        return m._lib.load().msg_device_count()
    except Exception:
        return 0


def _push(m, ctx, raw, off, lo, hi, how, held):
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
        held.append((ctx, d_raw, d_off))
        if len(r):
            ctx.device_upload(d_raw, r)
        ctx.device_upload(d_off, o)
        ctx.push_device(d_raw, len(r), d_off, hi - lo)


def _release(held):
    for h in held:
        if isinstance(h, tuple):
            h[0].device_free(h[1]); h[0].device_free(h[2])
        else:
            h.close()
    held.clear()


def _pieces(lo, hi, k, rng):
    """k pushes covering [lo, hi), cut at random record counts (empty pushes allowed)"""
    c = np.sort(rng.integers(lo, hi + 1, size=k - 1)) if hi > lo else np.full(k - 1, lo)
    b = [lo] + [int(x) for x in c] + [hi]
    return list(zip(b[:-1], b[1:]))


def _ctx(m, world, rank, uid, cfg, tl, **kw):
    return m.Context(**cfg, collate=m._lib.MSG_COLLATE_RANKS, n_targets=len(tl), target_len=tl if cfg.get("coverage") else None,
                     device=rank, n_ranks=world, rank=rank, nccl_unique_id=uid, **kw)


def _results(ctx, cfg):
    out = {}
    if cfg.get("coverage"):
        out["cov"], out["touched"], out["total"] = ctx.finish_coverage()
    if cfg.get("profile"):
        ab, st = ctx.finish_profile()
        out["ab"] = ab
        out["st"] = np.array([st[k] for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "n_lists")], dtype=np.int64)
        out["ui"] = ctx.pull_counts()[0]
    return out


def _rank_cuts(n, world, seed):
    c = np.sort(np.random.default_rng(seed).integers(0, n + 1, size=world - 1))
    return [0] + [int(x) for x in c] + [n]


def _worker(rank, world, uid, out_dir, scenario):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    data = np.load(os.path.join(out_dir, "stream.npz"), allow_pickle=True)
    spec = data["spec"].item()
    os.environ.update(spec.get("env", {}))
    import msamtools_b200 as m
    res = {}
    SCENARIOS[scenario](m, rank, world, uid, data, spec, res)
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), **{k: np.asarray(v) for k, v in res.items()})


def _sc_parity(m, rank, world, uid, data, spec, res):
    """every case of spec: this rank's piece [cuts[rank], cuts[rank + 1]) in three pushes of a kind that depends on rank"""
    kinds = ["staged", "pinned", "device"]
    for ci, case in enumerate(spec["cases"]):
        os.environ.update(case.get("env", {}))
        raw, off, tl = data[case["stream"] + "_raw"], data[case["stream"] + "_off"], data[case["stream"] + "_tl"]
        cuts = data[case["stream"] + "_cuts"]
        rng = np.random.default_rng(100 * ci + rank)
        held = []
        with _ctx(m, world, rank, uid, case["cfg"], tl) as ctx:
            for k, (lo, hi) in enumerate(_pieces(int(cuts[rank]), int(cuts[rank + 1]), 3, rng)):
                _push(m, ctx, raw, off, lo, hi, kinds[(rank + k) % 3], held)
            for key, v in _results(ctx, case["cfg"]).items():
                res[f"{ci}_{key}"] = v
            _release(held)
        for key in case.get("env", {}):
            del os.environ[key]


def _sc_scopes(m, rank, world, uid, data, spec, res):
    """scope 1: every rank pushes its piece; finish_coverage then finish_profile (one exchange), a second finish_profile
    (none).  Scope 2: only rank 0 pushes the whole stream again.  Then reset on every rank."""
    raw, off, tl, cuts = data["s_raw"], data["s_off"], data["s_tl"], data["s_cuts"]
    cfg = dict(profile=True, coverage=True, besthit=True, kept=False, **FILT)
    with _ctx(m, world, rank, uid, cfg, tl) as ctx:
        held = []
        _push(m, ctx, raw, off, int(cuts[rank]), int(cuts[rank + 1]), "staged", held)
        for key, v in _results(ctx, cfg).items():
            res[f"a_{key}"] = v
        ab2, st2 = ctx.finish_profile()
        res["a2_ab"] = ab2
        res["a2_st"] = np.array([st2[k] for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "n_lists")], dtype=np.int64)
        if rank == 0:
            _push(m, ctx, raw, off, 0, len(off) - 1, "device", held)
        for key, v in _results(ctx, cfg).items():
            res[f"b_{key}"] = v
        ctx.reset()
        for key, v in _results(ctx, cfg).items():
            res[f"c_{key}"] = v
        _release(held)


def _sc_error(m, rank, world, uid, data, spec, res):
    """a record without AS on rank 1 under --besthit: every rank's finish fails with the same code"""
    raw, off, cuts = data["e_raw"], data["e_off"], data["e_cuts"]
    for fused in (True, False):
        extra = dict(profile=True, besthit=True, kept=False, **FILT)
        if not fused:
            extra["coverage"] = True
        tl = np.full(40, 5000, dtype=np.uint32)
        with _ctx(m, world, rank, uid, extra, tl) as ctx:
            held = []
            lo, hi = int(cuts[rank]), int(cuts[rank + 1])
            mid = (lo + hi) // 2
            _push(m, ctx, raw, off, lo, mid, "staged", held)
            _push(m, ctx, raw, off, mid, hi, "pinned", held)
            try:
                ctx.finish_profile()
                res[f"{int(fused)}_code"], res[f"{int(fused)}_text"] = 0, ""
            except m.MsgError as e:
                res[f"{int(fused)}_code"], res[f"{int(fused)}_text"] = e.code, e.text
            _release(held)


SCENARIOS = {"parity": _sc_parity, "scopes": _sc_scopes, "error": _sc_error}


def _spawn(tmp_path, scenario, spec, streams):
    """run WORLD ranks of `scenario`; a rank that does not finish within JOIN_TIMEOUT_S fails the test, and every child is
    terminated, then killed, so that nothing is left behind"""
    import msamtools_b200 as m
    np.savez(tmp_path / "stream.npz", spec=np.array(spec, dtype=object), **streams)
    uid = m.nccl_unique_id()
    ctx = multiprocessing.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, WORLD, uid, str(tmp_path), scenario)) for r in range(WORLD)]
    for p in procs:
        p.start()
    import time
    t_end = time.monotonic() + JOIN_TIMEOUT_S
    try:
        for p in procs:
            p.join(max(0.0, t_end - time.monotonic()))
        hung = [r for r, p in enumerate(procs) if p.is_alive()]
        assert not hung, f"ranks {hung} did not finish within {JOIN_TIMEOUT_S} s"
        codes = [p.exitcode for p in procs]
        assert codes == [0] * WORLD, f"rank exit codes {codes}"
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
        for p in procs:
            p.join(10)
            if p.is_alive():
                p.kill()
                p.join()
    return [np.load(tmp_path / f"r{r}.npz", allow_pickle=True) for r in range(WORLD)]


def _oracle(orc, raw, off, cfg, tl):
    g, go = regroup(raw, off)
    fkw = {k: cfg[k] for k in ("l", "p", "z", "besthit", "uniqhit") if k in cfg}
    idx = orc.filter_stream(g, go, orc.filter_cfg(**fkw)) if fkw else None
    out = {}
    mode = cfg.get("multi", "proportional")
    if cfg.get("profile"):
        ab, st, ui, _ = orc.profile(g, go, idx, len(tl), SHARE[mode])
        out["ab"], out["ui"] = ab, ui
        out["st"] = [st["mapped_inserts"], st["uniq"], st["multi"], st["purged"], st["iterations"], st["n_lists"]]
    if cfg.get("coverage"):
        out["cov"], out["touched"], out["total"] = orc.coverage(g, go, idx, tl)[:3]
    return out


def _close(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.all(np.abs(a - b) <= REL * np.maximum(np.abs(a), np.abs(b)))


def _check(r, pre, exp, cfg, what):
    """every rank against the oracle's whole-stream result, vectors bit-identical across ranks"""
    prop = cfg.get("multi", "proportional") == "proportional"
    for k in range(WORLD):
        if "st" in exp:
            got = r[k][pre + "st"].tolist()
            n = 6 if prop else 3                          # purged / iterations / lists only exist for PropSharing
            assert got[:n] == exp["st"][:n], (what, k, got, exp["st"])
            assert _close(r[k][pre + "ab"], exp["ab"]), (what, k)
            assert np.array_equal(r[k][pre + "ab"], r[0][pre + "ab"]), (what, k)
        if "cov" in exp:
            for key in ("cov", "touched", "total"):
                assert np.array_equal(r[k][pre + key], exp[key]), (what, k, key)


def _routed_ui(orc, raw, off, cfg, tl):
    """the oracle's per-feature counts over exactly the reads the rule sends to each rank"""
    d = dest(CU.keys(raw, off), WORLD)
    out = []
    for r in range(WORLD):
        sraw, soff = CU.stream_of(raw, off, np.flatnonzero(d == r))
        out.append(_oracle(orc, sraw, soff, cfg, tl)["ui"])
    return out


PARITY_CFGS = [dict(profile=True, besthit=True, kept=False, **FILT),                     # fused best-hit -> proportional
               dict(profile=True, multi="all"), dict(profile=True, multi="equal"), dict(profile=True, multi="ignore"),
               dict(coverage=True, besthit=True, kept=False, **FILT)]                    # filter + coverage, depth mode


def _stream_set(name, preset, n, seed, order):
    raw, off, tl = synth_stream(preset, n, seed, order)
    return {f"{name}_raw": raw, f"{name}_off": off, f"{name}_tl": tl,
            f"{name}_cuts": np.array(_rank_cuts(len(off) - 1, WORLD, seed))}


@pytest.mark.gpu
@pytest.mark.skipif(_ndev() < WORLD, reason=f"needs {WORLD} GPUs")
@pytest.mark.parametrize("order", ["coord", "shuffle"])
def test_collate_ranks_parity_mixed(tmp_path, oracle, order):
    streams = _stream_set("x", "mixed", 200_000, 61, order)
    spec = dict(cases=[dict(stream="x", cfg=c) for c in PARITY_CFGS])
    r = _spawn(tmp_path, "parity", spec, streams)
    raw, off, tl = streams["x_raw"], streams["x_off"], streams["x_tl"]
    for ci, cfg in enumerate(PARITY_CFGS):
        _check(r, f"{ci}_", _oracle(oracle, raw, off, cfg, tl), cfg, (order, cfg))
    # routing is exact: rank k's own counts are the oracle's over the reads sent to rank k
    for k, ui in enumerate(_routed_ui(oracle, raw, off, PARITY_CFGS[0], tl)):
        assert np.array_equal(r[k]["0_ui"], ui), k



@pytest.mark.gpu
@pytest.mark.skipif(_ndev() < WORLD, reason=f"needs {WORLD} GPUs")
def test_collate_ranks_catalogues_and_nccl_loop(tmp_path, oracle):
    """catalog10k / genes1m: collation meets the reduce-scatter exchange (em_loop_rsag_kernel); MSG_NO_P2P=1: NCCL loop"""
    streams = {**_stream_set("c", "catalog10k", 200_000, 67, "coord"), **_stream_set("g", "genes1m", 200_000, 71, "shuffle"),
               **_stream_set("x", "mixed", 200_000, 73, "shuffle")}
    cfg = PARITY_CFGS[0]
    spec = dict(cases=[dict(stream="c", cfg=cfg), dict(stream="g", cfg=cfg), dict(stream="x", cfg=cfg, env={"MSG_NO_P2P": "1"})])
    r = _spawn(tmp_path, "parity", spec, streams)
    for ci, s in enumerate(("c", "g", "x")):
        _check(r, f"{ci}_", _oracle(oracle, streams[s + "_raw"], streams[s + "_off"], cfg, streams[s + "_tl"]), cfg, s)


def _big_read_stream():
    """200 paired reads plus one read of 5 000 alignments; WORLD - 1 cuts put rank 1's piece to nothing"""
    import test_collate as T
    recs = T._edge_stream(200, seed=8)
    big = []
    for h in range(2500):
        big += T._pe_read("bigread", 1, tid0=h % 40, as0=60 - (h % 2))
    rng = np.random.default_rng(2)
    allr = recs + big
    allr = [allr[int(i)] for i in rng.permutation(len(allr))]
    raw, off = E.stream(allr)
    return raw, off.astype(np.uint64)


@pytest.mark.gpu
@pytest.mark.skipif(_ndev() < WORLD, reason=f"needs {WORLD} GPUs")
def test_collate_ranks_edges(tmp_path, oracle):
    """one rank pushes nothing; one read of 5 000 alignments spread over every rank (its rank receives all of it)"""
    tl = np.full(40, 5000, dtype=np.uint32)
    raw, off = _big_read_stream()
    n = len(off) - 1
    empty = [0, n // 2] + [n // 2] * (WORLD - 2) + [n]                  # rank 1 pushes nothing
    only = np.array(sorted(np.random.default_rng(4).integers(0, n, WORLD - 1))) if WORLD > 1 else []
    streams = {"e_raw": raw, "e_off": off, "e_tl": tl, "e_cuts": np.array(empty),
               "b_raw": raw, "b_off": off, "b_tl": tl, "b_cuts": np.array([0] + [int(x) for x in only] + [n])}
    cfgs = [dict(profile=True, multi="proportional"), dict(profile=True, besthit=True, kept=False, **FILT)]
    spec = dict(cases=[dict(stream=s, cfg=c) for s in ("e", "b") for c in cfgs])
    r = _spawn(tmp_path, "parity", spec, streams)
    for ci, case in enumerate(spec["cases"]):
        _check(r, f"{ci}_", _oracle(oracle, raw, off, case["cfg"], tl), case["cfg"], case["stream"])


@pytest.mark.gpu
@pytest.mark.skipif(_ndev() < WORLD, reason=f"needs {WORLD} GPUs")
def test_collate_ranks_collisions_and_many_chunks(tmp_path, oracle):
    """MSG_COLLATE_HASH_BITS=8 (runs of one key holding many names, split over ranks only by key) with
    MSG_COLLATE_CHUNK_RECORDS=1000 (many grouped chunks per rank)"""
    streams = _stream_set("x", "mixed", 50_000, 79, "shuffle")
    cfgs = [PARITY_CFGS[0], dict(profile=True, multi="proportional"), PARITY_CFGS[4]]
    spec = dict(env={"MSG_COLLATE_HASH_BITS": "8", "MSG_COLLATE_CHUNK_RECORDS": "1000"}, cases=[dict(stream="x", cfg=c) for c in cfgs])
    r = _spawn(tmp_path, "parity", spec, streams)
    for ci, cfg in enumerate(cfgs):
        _check(r, f"{ci}_", _oracle(oracle, streams["x_raw"], streams["x_off"], cfg, streams["x_tl"]), cfg, cfg)


@pytest.mark.gpu
@pytest.mark.skipif(_ndev() < WORLD, reason=f"needs {WORLD} GPUs")
def test_collate_ranks_scopes_and_reset(tmp_path, oracle):
    streams = _stream_set("s", "mixed", 60_000, 83, "coord")
    r = _spawn(tmp_path, "scopes", {}, streams)
    raw, off, tl = streams["s_raw"], streams["s_off"], streams["s_tl"]
    cfg = dict(profile=True, coverage=True, besthit=True, kept=False, **FILT)
    exp = _oracle(oracle, raw, off, cfg, tl)
    _check(r, "a_", exp, cfg, "scope 1")
    for k in range(WORLD):                     # a second finish reuses the collation
        assert r[k]["a2_st"].tolist() == exp["st"] and _close(r[k]["a2_ab"], exp["ab"])
    # scope 2 adds the whole stream once more (rank 0 only): every integer doubles, not triples
    g, go = regroup(raw, off)
    dbl_raw = np.concatenate([g, g])
    dbl_off = np.concatenate([go, go[1:] + go[-1]]).astype(np.uint64)
    # the oracle on the stream twice: each read's two copies are separate groups, as in two scopes
    idx = oracle.filter_stream(dbl_raw, dbl_off, oracle.filter_cfg(besthit=True, **FILT))
    _, st2, ui2, _ = oracle.profile(dbl_raw, dbl_off, idx, len(tl), SHARE["proportional"])
    cov2 = oracle.coverage(dbl_raw, dbl_off, idx, tl)
    for k in range(WORLD):
        assert r[k]["b_st"].tolist()[:3] == [st2["mapped_inserts"], st2["uniq"], st2["multi"]], k
        assert r[k]["b_st"].tolist()[:3] == [2 * x for x in exp["st"][:3]], k
        assert np.array_equal(r[k]["b_total"], cov2[2]) and np.array_equal(r[k]["b_touched"], cov2[1]), k
        assert r[k]["c_st"].tolist()[:3] == [0, 0, 0] and not np.any(r[k]["c_total"]), k
    assert sum(r[k]["b_ui"] for k in range(WORLD)).tolist() == ui2.tolist()


@pytest.mark.gpu
@pytest.mark.skipif(_ndev() < WORLD, reason=f"needs {WORLD} GPUs")
def test_collate_ranks_enoas_names_global_ordinal_and_source(tmp_path):
    import test_collate as T
    recs = T._edge_stream(120, seed=3)
    rng = np.random.default_rng(1)
    recs = [recs[int(i)] for i in rng.permutation(len(recs))]
    n = len(recs)
    cuts = [0] + [n * (r + 1) // (WORLD + 1) for r in range(WORLD - 1)] + [n]
    bad = cuts[1] + 37                                   # record 37 of rank 1's pushes
    q = recs[bad]
    recs[bad] = E.record(E.qname(q), flag=int.from_bytes(q[18:20], "little"), tid=int.from_bytes(q[4:8], "little", signed=True),
                         pos=int.from_bytes(q[8:12], "little", signed=True), cigar=((100, E.M),), aux=E.aux_int("NM", "C", 0) + E.aux_z("MD", "100"))
    raw, off = E.stream(recs)
    off = off.astype(np.uint64)
    owner = int(dest(CU.keys(raw, off)[bad:bad + 1], WORLD)[0])
    r = _spawn(tmp_path, "error", {}, {"e_raw": raw, "e_off": off, "e_cuts": np.array(cuts)})
    for fused in (1, 0):
        for k in range(WORLD):
            assert int(r[k][f"{fused}_code"]) == -6, (fused, k, str(r[k][f"{fused}_text"]))
            text = str(r[k][f"{fused}_text"])
            if k == owner:
                assert f"(input record {bad}: rank 1, record 37 of its pushes)" in text, text
            else:
                assert f"record error on rank {owner}" in text, text


# ---------------------------------------------------------------- one process
@pytest.fixture(scope="module")
def m():
    import msamtools_b200 as mod
    assert mod._lib.load().msg_device_count() > 0, "no CUDA device: the GPU tests must not silently pass"
    return mod


@pytest.mark.gpu
def test_collate_ranks_refusals(m):
    R = m._lib.MSG_COLLATE_RANKS
    base = dict(profile=True, kept=False, n_targets=3)
    for kw in (dict(exact=True), dict(records=True), dict(kept=True), dict(stats=True)):
        with pytest.raises(m.MsgError) as ei:
            m.Context(**dict(base, **kw), collate=R, n_ranks=2, nccl_unique_id=b"\0" * 128)
        assert ei.value.code == -1
    for v in (3, 255):
        with pytest.raises(m.MsgError) as ei:
            m.Context(**base, collate=v)
        assert ei.value.code == -1 and "collate" in ei.value.text
    with pytest.raises(m.MsgError) as ei:
        m.Context(**base, collate=1, n_ranks=2, nccl_unique_id=b"\0" * 128)
    assert ei.value.code == -1 and "MSG_COLLATE_RANKS" in ei.value.text
    with pytest.raises(m.MsgError):
        m.Context(n_targets=3, kept=False, collate=R)                     # needs a profile or coverage consumer


@pytest.mark.gpu
def test_collate_ranks_on_one_rank_is_collate(m):
    import test_collate as T
    raw, off, tl = synth_stream("mixed", 30000, 89, "shuffle")
    cuts = [(0, 9000), (9000, 9001), (9001, len(off) - 1)]
    for cfg in T.CONFIGS[:5] + [T.CONFIGS[6]]:
        a = T.run_cmp(m, raw, off, dict(cfg, collate=m._lib.MSG_COLLATE_RANKS), tl, chunks=cuts)
        b = T.run_cmp(m, raw, off, dict(cfg, collate=1), tl, chunks=cuts)
        T.expect_equal(a, b, str(cfg))
        if "st" in a:
            assert a["st"] == b["st"]
