"""The collation's grouped order restated in numpy (csrc/collate.cuh, collate_run in csrc/api.cu), for the chunk tests
(tests/test_collate_chunks.py).

A collating context orders its records by a 64-bit key of each QNAME (collate_gather_kernel), then by the input ordinal;
runs of one key that hold different names are re-sorted by (l_read_name, name bytes, ordinal).  The pipeline then takes
the grouped records in chunks cut where the key changes.  Knowing that order exactly lets a test put a chunk cut, a
bucket size, a collision run or a bad record where it wants, and predict the error a finish reports.
"""
import numpy as np

MASK64 = (1 << 64) - 1
GOLDEN = 0x9E3779B97F4A7C15
LQ_MUL = 0xD6E8FEB86659FD93
SMEM_KEYS = 2048            # COLL_SMEM_KEYS: largest bucket sorted in shared memory
BUCKET_AVG = 512            # COLL_BUCKET_AVG
CHUNK_RECORDS = 1 << 24     # default grouped chunk limit (MSG_COLLATE_CHUNK_RECORDS)


# ---------------------------------------------------------------- the key
def hash_mask(bits=64):
    """the mask MSG_COLLATE_HASH_BITS=bits gives (coll_hash_mask): the top `bits` bits, all 64 outside [1, 63]"""
    return MASK64 if bits >= 64 or bits < 1 else (MASK64 << (64 - bits)) & MASK64


def mix64_scalar(x):
    x &= MASK64
    x ^= x >> 30; x = (x * 0xbf58476d1ce4e5b9) & MASK64
    x ^= x >> 27; x = (x * 0x94d049bb133111eb) & MASK64
    return x ^ (x >> 31)


def key_scalar(name, bits=64):
    """the kernel's loop, transcribed one word at a time: name is the QNAME without its NUL"""
    b = bytes(name) + b"\0"
    lq = len(b)
    h = 0
    w = 0
    while 4 * w < lq:
        x = 0
        for k in range(4):
            if 4 * w + k < lq:
                x |= b[4 * w + k] << (8 * k)
        h = (h + mix64_scalar(((w << 32) | x) + GOLDEN)) & MASK64
        w += 1
    return mix64_scalar(h ^ ((lq * LQ_MUL) & MASK64)) & hash_mask(bits)


def _mix64(x):
    x = x ^ (x >> np.uint64(30)); x = x * np.uint64(0xbf58476d1ce4e5b9)
    x = x ^ (x >> np.uint64(27)); x = x * np.uint64(0x94d049bb133111eb)
    return x ^ (x >> np.uint64(31))


def name_matrix(raw, off, lo=0, hi=None):
    """(l_read_name uint32[k], name bytes uint8[k, W]) of records lo..hi: W covers the longest l_read_name rounded up to
    4 bytes; bytes past a record's l_read_name are 0"""
    hi = len(off) - 1 if hi is None else hi
    o = np.asarray(off[lo:hi], dtype=np.int64)
    lq = raw[o + 12].astype(np.uint32)
    W = 4 * ((int(lq.max()) + 3) // 4) if len(lq) else 4
    col = np.arange(W, dtype=np.int64)
    idx = np.minimum(o[:, None] + 36 + col[None, :], len(raw) - 1)
    m = raw[idx]
    m[col[None, :] >= lq[:, None].astype(np.int64)] = 0
    return lq, m


def keys_of_names(lq, m, bits=64):
    """vectorised key of each row of name_matrix()"""
    words = np.ascontiguousarray(m).view("<u4")
    h = np.zeros(len(lq), dtype=np.uint64)
    with np.errstate(over="ignore"):
        for w in range(words.shape[1]):
            v = _mix64(((np.uint64(w) << np.uint64(32)) | words[:, w].astype(np.uint64)) + np.uint64(GOLDEN))
            h += np.where(4 * w < lq, v, np.uint64(0))
        return _mix64(h ^ (lq.astype(np.uint64) * np.uint64(LQ_MUL))) & np.uint64(hash_mask(bits))


def names_all(raw, off, block=1 << 20):
    """name_matrix() of the whole stream, built in blocks"""
    n = len(off) - 1
    parts = [name_matrix(raw, off, lo, min(n, lo + block)) for lo in range(0, n, block)]
    W = max(m.shape[1] for _, m in parts)
    return (np.concatenate([lq for lq, _ in parts]),
            np.concatenate([np.pad(m, ((0, 0), (0, W - m.shape[1]))) for _, m in parts]))


def keys(raw, off, bits=64, block=1 << 20):
    n = len(off) - 1
    out = np.empty(n, dtype=np.uint64)
    for lo in range(0, n, block):
        hi = min(n, lo + block)
        out[lo:hi] = keys_of_names(*name_matrix(raw, off, lo, hi), bits=bits)
    return out


def names_keys(names, bits=64):
    """keys of a list of QNAMEs (bytes or str, without the NUL)"""
    nb = [x.encode() if isinstance(x, str) else bytes(x) for x in names]
    lq = np.array([len(x) + 1 for x in nb], dtype=np.uint32)
    W = 4 * ((int(lq.max()) + 3) // 4)
    m = np.zeros((len(nb), W), dtype=np.uint8)
    for k, x in enumerate(nb):
        m[k, :len(x)] = np.frombuffer(x, dtype=np.uint8)
    return keys_of_names(lq, m, bits)


def bucket_bits(n):
    """bits of the partition: the smallest b <= 24 with 512 << b >= n"""
    b = 0
    while b < 24 and (BUCKET_AVG << b) < n:
        b += 1
    return b


def bucket_of(k, bits):
    k = np.asarray(k, dtype=np.uint64)
    return np.zeros(k.shape, dtype=np.int64) if bits == 0 else (k >> np.uint64(64 - bits)).astype(np.int64)


# ---------------------------------------------------------------- the grouped order and the chunk cuts
def grouped_order(raw, off, bits=64):
    """(order, sorted keys): order[g] = input ordinal of the record at grouped position g.  Records sort by (key,
    l_read_name, name bytes, ordinal), which is the bucket sort by (key, ordinal) followed by the collision re-sort."""
    k = keys(raw, off, bits)
    order = np.argsort(k, kind="stable")
    ks = k[order]
    same = np.flatnonzero(ks[1:] == ks[:-1])
    if len(same):
        lq, m = names_all(raw, off)
        a, b = order[same], order[same + 1]
        if np.any(lq[a] != lq[b]) or np.any(m[a] != m[b]):
            # a run of one key holds different names: rank the names (length first, then bytes) and sort again
            w = m.shape[1]
            full = np.zeros((len(lq), w + 1), dtype=np.uint8)
            full[:, 0] = lq
            full[:, 1:] = m
            _, rank = np.unique(np.ascontiguousarray(full).view(np.dtype((np.void, w + 1))).ravel(), return_inverse=True)
            order = np.lexsort((np.arange(len(k)), rank.ravel(), k))
            ks = k[order]
    return order, ks


def cuts(sorted_keys, C=CHUNK_RECORDS):
    """chunk bounds [0, h1, ..., n] of collate_run: while more than C records remain after lo, cut at the last key-run
    start in (lo, lo + C]; if there is none (one run longer than C), at the first run start after lo + C, or at n"""
    ks = np.asarray(sorted_keys)
    n = len(ks)
    starts = np.flatnonzero(ks[1:] != ks[:-1]) + 1
    b, lo = [0], 0
    while n - lo > C:
        i = int(np.searchsorted(starts, lo + C, side="right"))
        if i > 0 and starts[i - 1] > lo:
            hi = int(starts[i - 1])
        else:
            hi = int(starts[i]) if i < len(starts) else n
        b.append(hi)
        lo = hi
    if b[-1] != n:
        b.append(n)
    return b


# ---------------------------------------------------------------- constructors
def find_names(pred, count, prefix="q", start=0, batch=200_000, bits=64, width=None):
    """`count` names prefix + decimal number (zero-padded to `width` digits if given) whose key k satisfies pred(k)
    (a vectorised predicate over uint64 keys), in increasing number"""
    out, s = [], start
    while len(out) < count:
        nums = range(s, s + batch)
        names = [(prefix + (str(x).zfill(width) if width else str(x))).encode() for x in nums]
        k = names_keys(names, bits)
        out += [names[int(j)] for j in np.flatnonzero(pred(k))]
        s += batch
    return out[:count]


def stream_of(raw, off, perm, block=1 << 20):
    """records in the order perm (perm[k] = input ordinal of output record k), vectorised"""
    perm = np.asarray(perm, dtype=np.int64)
    o = np.asarray(off, dtype=np.int64)
    ln = (o[1:] - o[:-1])[perm]
    off2 = np.zeros(len(perm) + 1, dtype=np.uint64)
    off2[1:] = np.cumsum(ln, dtype=np.uint64)
    raw2 = np.empty(int(off2[-1]), dtype=np.uint8)
    for lo in range(0, len(perm), block):
        hi = min(len(perm), lo + block)
        src, d0, d1 = o[perm[lo:hi]], int(off2[lo]), int(off2[hi])
        idx = np.repeat(src - off2[lo:hi].astype(np.int64), ln[lo:hi]) + np.arange(d0, d1, dtype=np.int64)
        raw2[d0:d1] = raw[idx]
    return raw2, off2


def read_ids(raw, off):
    """read index of each record of a stream grouped by QNAME (0, 0, 1, 1, 1, 2, ...)"""
    lq, m = names_all(raw, off)
    head = np.r_[len(lq) > 0, (lq[1:] != lq[:-1]) | np.any(m[1:] != m[:-1], axis=1)]
    return np.cumsum(head) - 1


def riffle(raw, off):
    """the permutation test_collate.riffle gives, vectorised: read g's j-th record sorts by (g + 3 j, g)"""
    g = read_ids(raw, off)
    n = len(g)
    first = np.zeros(n, dtype=np.int64)
    if n:
        heads = np.flatnonzero(np.r_[True, g[1:] != g[:-1]])
        first[heads] = heads
        first = np.maximum.accumulate(first)
    j = np.arange(n) - first
    return np.lexsort((np.arange(n), g, g + 3 * j))
