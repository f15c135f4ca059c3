"""GPU parity on the feature counts the metric is quoted on: BASELINE.json configs[2] (10 k references)
and configs[4] (1 M-gene catalogue).  These shapes leave the shared-memory fast paths (F <= 4096
histograms, F <= 2048 PropSharing loop) and run `em_loop_kernel`, `fused_warp_kernel<false>` and
`profile_warp_count_kernel<false>`; every case is compared with the CPU oracle on the same 2 M-record
seeded stream: integer counts bit-exact, abundances within 1e-9 relative, same PropSharing iteration
count / purged / list totals (msam_profile.c:331-404).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHARE = {"all": 1, "equal": 2, "proportional": 3, "ignore": 4}
REL = 1e-9
N_RECORDS = 2_000_000
FILTER = dict(l=80, p=95, z=80, besthit=True)


@pytest.fixture(scope="module")
def m():
    import msamtools_b200 as mod
    assert mod._lib.load().msg_device_count() > 0, "no CUDA device: the GPU tests must not silently pass"
    return mod


def close(a, b, rel=REL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.all(np.abs(a - b) <= rel * np.maximum(np.abs(a), np.abs(b)))


_streams = {}


def stream(preset):
    """2 M-record seeded stream of a preset + the oracle's filter output, generated once per session."""
    if preset not in _streams:
        from msamtools_b200 import synth
        from oracle import oracle as orc
        orc.load()
        p = synth.make_params(preset, n_records=N_RECORDS, seed=97531)
        raw, off, _ = synth.generate(p)
        tlen = synth.target_lengths(p)
        idx = orc.filter_stream(raw, off, orc.filter_cfg(**FILTER))
        _streams.clear()                      # one preset resident at a time (0.6 GB each)
        _streams[preset] = (raw, off, tlen, idx)
    return _streams[preset]


def check(st, est, ui, eui, d, ed, ab, eab):
    for k in ("mapped_inserts", "uniq", "multi", "purged", "iterations", "converged", "n_lists", "n_entries"):
        assert st[k] == est[k], (k, st[k], est[k])
    assert np.array_equal(ui, eui)
    assert close(d, ed) and close(ab, eab)
    assert est["multi"] > 1000 and est["uniq"] > 1000


@pytest.mark.parametrize("path", ["fused", "general", "plain"])
@pytest.mark.parametrize("mode", ["all", "equal", "proportional", "ignore"])
@pytest.mark.parametrize("preset", ["catalog10k", "genes1m"])
def test_large_feature_count_profile(m, oracle, preset, mode, path):
    """fused: filter --besthit | profile as the fused single pass (kept=False); general: the same through the kept stream
    (besthit_* + profile_warp_* kernels); plain: `msamtools profile` on the unfiltered stream."""
    raw, off, tlen, idx = stream(preset)
    F = len(tlen)
    assert F > 4096
    pre = None if path == "plain" else FILTER
    eab, est, eui, ed = oracle.profile(raw, off, None if pre is None else idx, F, SHARE[mode])
    with m.Context(profile=True, multi=mode, kept=(path != "fused"), n_targets=F, **(pre or {})) as ctx:
        ctx.push(raw, off)
        if pre is not None:
            assert ctx.kept_count() == len(idx)
        ui, d = ctx.pull_counts()
        ab, st = ctx.finish_profile()
        t = ctx.timing()
    if path == "fused":
        assert (t["fused_chunks"], t["fused_fallbacks"]) == (1, 0)
    else:
        assert t["fused_chunks"] == 0
    check(st, est, ui, eui, d, ed, ab, eab)
    if mode == "proportional":
        assert est["iterations"] >= 5, "the stream must need a real PropSharing loop, not a first-iteration exit"
        assert close(st["delta"], est["delta"], 1e-6)


@pytest.mark.parametrize("preset", ["catalog10k", "genes1m"])
def test_large_feature_count_chunked_resident(m, oracle, preset):
    """what bench.py does per step: several QNAME-boundary chunks pushed from device memory into one context,
    then one msg_finish_profile; and a second finish on the same state gives the same answer."""
    raw, off, tlen, idx = stream(preset)
    F, n = len(tlen), len(off) - 1
    eab, est, eui, ed = oracle.profile(raw, off, idx, F, 3)
    cuts = [0] + [m.split_point(raw, off, n * k // 4) for k in (1, 2, 3)] + [n]
    with m.Context(profile=True, multi="proportional", kept=False, n_targets=F, **FILTER) as ctx:
        bufs = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            lo, hi = int(off[a]), int(off[b])
            sub, soff = np.ascontiguousarray(raw[lo:hi]), np.ascontiguousarray(off[a:b + 1] - off[a])
            d_raw, d_off = ctx.device_alloc(sub.nbytes), ctx.device_alloc(soff.nbytes)
            ctx.device_upload(d_raw, sub); ctx.device_upload(d_off, soff)
            bufs.append((d_raw, sub.nbytes, d_off, b - a))
        for rep in range(2):
            ctx.reset()
            kept = 0
            for d_raw, nb, d_off, nr in bufs:
                ctx.push_device(d_raw, nb, d_off, nr)
                kept += ctx.kept_count()
            ui, d = ctx.pull_counts()
            ab, st = ctx.finish_profile()
            ab2, st2 = ctx.finish_profile()
            assert kept == len(idx)
            check(st, est, ui, eui, d, ed, ab, eab)
            assert close(ab2, eab) and st2["iterations"] == est["iterations"] and st2["purged"] == est["purged"]
        for d_raw, _, d_off, _ in bufs:
            ctx.device_free(d_raw); ctx.device_free(d_off)


def test_genes1m_genome_map(m, oracle):
    """--genome style map on the 1 M-gene catalogue: 1 M sequences -> 50 k features (fmap gather on the large-F path)."""
    raw, off, tlen, idx = stream("genes1m")
    T, F = len(tlen), 50_000
    fmap = ((np.arange(T, dtype=np.int64) * 7919) % F).astype(np.int32)
    eab, est, eui, ed = oracle.profile(raw, off, idx, T, 3, fmap=fmap, n_features=F)
    for kept in (False, True):
        with m.Context(profile=True, multi="proportional", kept=kept, n_targets=T, n_features=F, fmap=fmap, **FILTER) as ctx:
            ctx.push(raw, off)
            ui, d = ctx.pull_counts()
            ab, st = ctx.finish_profile()
        check(st, est, ui, eui, d, ed, ab, eab)
