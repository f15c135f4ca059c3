"""Streams with a chosen PropSharing problem, and a restatement of the loop, for tests/test_gpu_em.py.

`lists_stream` writes BAM record bytes whose --multi=proportional profile is exactly the one asked for: U[f]
single-record reads on feature f, then one read per multi-mapper list with one record per feature in list order.  All
records have the same size, so a stream of a few hundred thousand lists is one 2-D uint8 array filled column-wise.

`em_reference` restates msam_profile.c:284-404 (the oracle's orc_profile_finish) over a CSR of the lists, in float64
and in np.longdouble (a 64-bit mantissa on x86-64), so that a test can certify that rounding cannot change a stop
decision.  `slow_block` finds three-feature problems that stop at a chosen iteration.
"""
import functools

import numpy as np

NAME_DIGITS = 9                          # QNAME "r" + 9 digits: l_read_name 11
_NAME = 1 + NAME_DIGITS
_AUX = b"NMC\x00" + b"MDZ40\x00" + b"ASC\x32"          # NM:i:0 MD:Z:40 AS:i:50, the same for every record (tied AS)
_BLOCK = 32 + _NAME + 1 + 4 + len(_AUX)                # core, QNAME + NUL, one CIGAR op (40M), l_seq = 0, aux
REC = 4 + _BLOCK


def _template():
    import struct
    core = struct.pack("<iiBBHHHiiii", 0, 100, _NAME + 1, 60, 4681 + (100 >> 14), 1, 0, 0, -1, -1, 0)
    name = b"r" + b"0" * NAME_DIGITS + b"\0"
    body = core + name + struct.pack("<I", 40 << 4) + _AUX
    assert len(body) == _BLOCK
    return np.frombuffer(struct.pack("<i", _BLOCK) + body, dtype=np.uint8)


def csr(lists):
    """list of feature sequences -> (off int64 [n + 1], fid int32)"""
    lens = np.array([len(x) for x in lists], dtype=np.int64)
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    fid = np.fromiter((f for x in lists for f in x), dtype=np.int32, count=int(off[-1]))
    return off, fid


def concat(*parts):
    """concatenate CSRs in order"""
    offs, fids, base = [np.zeros(1, dtype=np.int64)], [], 0
    for off, fid in parts:
        offs.append(np.asarray(off[1:], dtype=np.int64) + base)
        fids.append(np.asarray(fid, dtype=np.int32))
        base += int(off[-1])
    return np.concatenate(offs), np.concatenate(fids) if fids else np.zeros(0, dtype=np.int32)


def random_lists(rng, lens, lo, hi):
    """CSR of lists with the given lengths, each of distinct features drawn from [lo, hi): a random first feature,
    then positive steps whose sum stays below hi - lo (vectorised; max(lens) <= hi - lo)"""
    lens = np.asarray(lens, dtype=np.int64)
    P = hi - lo
    L = int(lens.max()) if len(lens) else 1
    assert L <= P
    step_hi = max((P - 1) // max(L - 1, 1), 1)
    steps = rng.integers(1, step_hi + 1, size=(len(lens), L))
    steps[:, 0] = rng.integers(0, P, size=len(lens))
    feats = lo + np.cumsum(steps, axis=1) % P
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    return off, feats[np.arange(L)[None, :] < lens[:, None]].astype(np.int32)


def lists_stream(U, off, fid, *, T=None):
    """Record bytes of U[f] single-record reads on feature f followed by one read per list (off, fid), in list order.

    Features in a list must be distinct (the profile keeps each feature's first appearance once).  T: None = one target
    per feature; else T >= 2F targets with fmap t -> t % F, and the records of a feature alternate between its targets.
    Returns (raw uint8, rec_off uint64, fmap or None)."""
    U = np.asarray(U, dtype=np.int64)
    F = len(U)
    off = np.asarray(off, dtype=np.int64)
    fid = np.asarray(fid, dtype=np.int64)
    nl = len(off) - 1
    lens = np.diff(off)
    assert nl == 0 or lens.min() >= 2, "a list needs two features"
    assert len(fid) == 0 or (fid.min() >= 0 and fid.max() < F)
    ns = int(U.sum())
    n = ns + len(fid)
    read = np.concatenate([np.arange(ns, dtype=np.int64), ns + np.repeat(np.arange(nl, dtype=np.int64), lens)])
    feat = np.concatenate([np.repeat(np.arange(F, dtype=np.int64), U), fid])
    first = np.ones(n, dtype=bool)
    first[ns:][np.arange(len(fid)) != np.repeat(off[:-1], lens)] = False
    assert ns + nl < 10 ** NAME_DIGITS
    fmap = None
    if T is not None:
        assert T >= 2 * F
        fmap = (np.arange(T) % F).astype(np.int32)
        feat = feat + F * (np.arange(n) % (T // F))
    rec = np.tile(_template(), (n, 1))
    rec[:, 4:8] = feat.astype("<i4").view(np.uint8).reshape(n, 4)
    rec[:, 18:20] = np.where(first, 0, 0x100).astype("<u2").view(np.uint8).reshape(n, 2)
    digits = read.copy()
    for k in range(NAME_DIGITS - 1, -1, -1):
        rec[:, 37 + k] = (digits % 10 + 48).astype(np.uint8)
        digits //= 10
    rec_off = np.arange(n + 1, dtype=np.uint64) * np.uint64(REC)
    return rec.reshape(-1), rec_off, fmap


def em_reference(U, off, fid, F, dtype=np.float64):
    """msam_profile.c:284-404 over the CSR (off, fid): a = U; per iteration k = 1..19 each list with s = sum a[f] > 0
    adds a[f] / s to inc[f]; a = U + inc with values < 1e-20 flushed to 0; DELTA^2 = sum (a_new - a_old)^2 / F; stop when
    DELTA^2 < 1e-10.  purged = lists whose final sum is exactly 0.  With F == 0, DELTA^2 is NaN (0 / 0), as in the
    reference, and the loop runs 19 times.

    The flush never fires on these problems: a starts at U (0 or at least 1 here), a zero stays zero, and a positive
    value only grows."""
    off = np.asarray(off, dtype=np.int64)
    fid = np.asarray(fid, dtype=np.int64)
    nl = len(off) - 1
    lens = np.diff(off)
    owner = np.repeat(np.arange(nl), lens)
    starts = off[:-1]
    by_f = np.argsort(fid, kind="stable")               # entries grouped by feature, for the inc reduction
    fs = fid[by_f]
    f_start = np.searchsorted(fs, np.arange(F))
    has = np.zeros(F, dtype=bool)
    has[fs] = True
    Ud = np.asarray(U).astype(dtype)
    a = Ud.copy()
    deltas, conv, k = [], 0, 0

    def list_sums(a):
        return np.add.reduceat(a[fid], starts) if nl else np.zeros(0, dtype=dtype)

    for k in range(1, 20):
        s = list_sums(a)
        inc = np.zeros(F, dtype=dtype)
        if len(fid):
            se = s[owner]
            w = np.where(se > 0, a[fid] / np.where(se > 0, se, 1), 0).astype(dtype)
            inc[has] = np.add.reduceat(w[by_f], f_start[has])
        an = Ud + inc
        an[an < 1e-20] = 0
        with np.errstate(invalid="ignore"):
            delta = np.sum((an - a) ** 2) / dtype(F) if F else dtype(np.nan)
        a = an
        deltas.append(delta)
        if delta < 1e-10:
            conv = 1
            break
    purged = int(np.count_nonzero(list_sums(a) == 0))
    return dict(ab=a, iterations=k, converged=conv, delta=deltas, purged=purged)


def decision_margin(deltas, factor=1.5):
    """True when no DELTA^2 of the sequence lies within `factor` of the 1e-10 threshold (NaN is far from it)"""
    d = np.asarray(deltas, dtype=np.float64)
    d = d[~np.isnan(d)]
    return bool(np.all((d >= 1e-10 * factor) | (d <= 1e-10 / factor)))


# ---------------------------------------------------------------- slow-convergence blocks
def _block_deltas(U, M1, M2):
    """sum (a_new - a_old)^2 of iterations 1..19 of the block: features (x, y, z), M1 lists (x, y), M2 lists (y, z);
    vectorised over arrays M1, M2 (float64, closed form of the per-list sums)"""
    u = [np.full(M1.shape, float(v)) for v in U]
    x, y, z = (v.copy() for v in u)
    out = np.zeros((19,) + M1.shape)
    with np.errstate(invalid="ignore", divide="ignore"):
        for k in range(19):
            sxy, syz = x + y, y + z
            ix = np.where(sxy > 0, M1 * x / sxy, 0)
            iy = np.where(sxy > 0, M1 * y / sxy, 0) + np.where(syz > 0, M2 * y / syz, 0)
            iz = np.where(syz > 0, M2 * z / syz, 0)
            nx, ny, nz = u[0] + ix, u[1] + iy, u[2] + iz
            out[k] = (nx - x) ** 2 + (ny - y) ** 2 + (nz - z) ** 2
            x, y, z = nx, ny, nz
    return out


def _stop(d, F):
    """(iterations, converged) of a DELTA^2 sum sequence d over F features"""
    below = np.nonzero(d / F < 1e-10)[0]
    return (int(below[0]) + 1, 1) if len(below) else (19, 0)


_USETS = [(1, 3, 0), (2, 3, 4), (1, 2, 0), (1, 1, 1), (2, 1, 3), (1, 4, 2), (3, 1, 1), (1, 2, 5)]


@functools.lru_cache(maxsize=None)
def slow_block(F, iterations, converged, max_total=1500, margin=2.0):
    """(U (3,), M1, M2) of a block whose loop over F features (the other F - 3 unused) stops at `iterations` with the
    given converged flag and keeps every DELTA^2 at least `margin` away from 1e-10; the fewest lists first (searched in
    bands of M1 + M2)"""
    assert F >= 3
    band = 64
    for t0 in range(2, max_total + 1, band):
        tot = np.arange(t0, t0 + band)
        m1 = np.concatenate([np.arange(1, t) for t in tot]).astype(np.float64)
        m2 = np.concatenate([t - np.arange(1, t) for t in tot]).astype(np.float64)
        best = None
        for U in _USETS:
            d = _block_deltas(U, m1, m2) / F
            thr = d < 1e-10
            stop = np.where(thr.any(axis=0), thr.argmax(axis=0) + 1, 19)
            ok = (stop == iterations) & (thr.any(axis=0) == bool(converged))
            near = (d > 1e-10 / margin) & (d < 1e-10 * margin) & (np.arange(1, 20)[:, None] <= stop[None])
            ok &= ~near.any(axis=0)
            if ok.any():
                i = int(np.argmin(np.where(ok, m1 + m2, np.inf)))
                if best is None or m1[i] + m2[i] < best[1] + best[2]:
                    best = (U, int(m1[i]), int(m2[i]))
        if best is not None:
            return np.array(best[0], dtype=np.int64), best[1], best[2]
    raise AssertionError(("no block", F, iterations, converged))


def block_lists(f0, M1, M2, interleave=True):
    """CSR of the block's lists on features f0, f0 + 1, f0 + 2: M1 x (f0, f0 + 1) and M2 x (f0 + 1, f0 + 2)"""
    a = [(f0, f0 + 1)] * M1
    b = [(f0 + 1, f0 + 2)] * M2
    if interleave:
        out, i, j = [], 0, 0
        while i < M1 or j < M2:
            if i < M1:
                out.append(a[i]); i += 1
            if j < M2:
                out.append(b[j]); j += 1
        return csr(out)
    return csr(a + b)
