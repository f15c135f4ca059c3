"""Byte-exact BAM record builder for the edge-case tests (tests/test_gpu_edges.py).

samutil goes through SAM text, which always picks the smallest integer type, derives l_seq from SEQ and cannot write
undefined CIGAR operations.  This module writes the record bytes directly (SAM spec 4.2), so every field the decoder
branches on is under the test's control: the QNAME length, each CIGAR operation (0-15), l_seq (0 included), and the aux
list with its tags, order, types and values.  Offsets are known while the stream is built, so a record can be placed
at any byte alignment.  It also restates two pieces of device logic the tests aim at: the decoder's window layout
(probe_layout in csrc/api.cu) and the QNAME hash (hash_step / hash_fin in csrc/decode.cuh).
"""
import struct

import numpy as np

M, I, D, N, S, H, P, EQ, X = range(9)
CORE = 36

_INT_FMT = {"c": "<b", "C": "<B", "s": "<h", "S": "<H", "i": "<i", "I": "<I"}
_B_FMT = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}


# ---------------------------------------------------------------- aux fields
def aux_int(tag, ty, v):
    return tag.encode() + ty.encode() + struct.pack(_INT_FMT[ty], v)


def aux_z(tag, s, ty="Z"):
    return tag.encode() + ty.encode() + (s.encode() if isinstance(s, str) else s) + b"\0"


def aux_a(tag, ch):
    return tag.encode() + b"A" + ch.encode()


def aux_f(tag, x):
    return tag.encode() + b"f" + struct.pack("<f", x)


def aux_b(tag, sub, vals):
    return tag.encode() + b"B" + sub.encode() + struct.pack("<i", len(vals)) + struct.pack("<%d%s" % (len(vals), _B_FMT[sub]), *vals)


def smallest_int(v):
    """the BAM type htslib gives an integer (samutil._aux_int)"""
    if v >= 0:
        return "C" if v <= 0xff else "S" if v <= 0xffff else "I"
    return "c" if v >= -128 else "s" if v >= -32768 else "i"


# ---------------------------------------------------------------- records
def reg2bin(beg, end):
    end -= 1
    for sh, base in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> sh == end >> sh:
            return base + (beg >> sh)
    return 0


def query_len(cigar):
    return sum(n for n, op in cigar if op in (M, I, S, EQ, X))


def ref_len(cigar):
    return sum(n for n, op in cigar if op in (M, D, N, EQ, X))


def record(name, *, flag=0, tid=0, pos=0, cigar=((50, M),), l_seq=None, aux=b"", mapq=60, mtid=-1, mpos=-1, isize=0):
    """One BAM record (block_size included).  name: str or bytes without the NUL (1 to 254 bytes, so l_read_name is
    2 to 255); cigar: (length, op) pairs, op 0-15; l_seq: None = the CIGAR's query length; aux: the aux block's bytes."""
    nb = (name.encode() if isinstance(name, str) else bytes(name)) + b"\0"
    assert 2 <= len(nb) <= 255
    ls = query_len(cigar) if l_seq is None else l_seq
    rl = max(ref_len(cigar), 1)
    b = reg2bin(pos, pos + rl) if pos >= 0 else 4680
    core = struct.pack("<iiBBHHHiiii", tid, pos, len(nb), mapq, b, len(cigar), flag, ls, mtid, mpos, isize)
    cig = b"".join(struct.pack("<I", n << 4 | op) for n, op in cigar)
    seq = bytes((0x12 + 0x21 * k) & 0xff for k in range((ls + 1) // 2))
    qual = bytes([30]) * ls
    body = core + nb + cig + seq + qual + bytes(aux)
    return struct.pack("<i", len(body)) + body


def aux_offset(rec):
    """offset of the aux block inside a record built by `record` (the decoder's aux_off)"""
    lq = rec[12]
    nc, = struct.unpack_from("<H", rec, 16)
    ls, = struct.unpack_from("<i", rec, 20)
    return CORE + lq + 4 * nc + (ls + 1) // 2 + ls


def qname(rec):
    return bytes(rec[CORE:CORE + rec[12] - 1])


def stream(recs):
    """list of record bytes -> (raw uint8, offsets uint64 [n + 1])"""
    off = np.zeros(len(recs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(r) for r in recs], dtype=np.uint64)
    raw = np.frombuffer(b"".join(recs), dtype=np.uint8).copy() if recs else np.zeros(0, dtype=np.uint8)
    return raw, off


def split(raw, off):
    return [bytes(raw[int(off[k]):int(off[k + 1])]) for k in range(len(off) - 1)]


def eqprev(recs):
    """EQPREV as the decoder defines it: the record's QNAME bytes equal the previous record's"""
    out = np.zeros(len(recs), dtype=bool)
    for k in range(1, len(recs)):
        out[k] = qname(recs[k]) == qname(recs[k - 1])
    return out


def cut_at_residue(off, r, lo=1):
    """largest k >= lo with off[k] % 16 == r (the chunk of records [0, k) then ends at that residue), or None"""
    o = np.asarray(off, dtype=np.uint64)
    ks = np.nonzero((o[lo:] % 16) == r)[0]
    return None if len(ks) == 0 else int(ks[-1]) + lo


# ---------------------------------------------------------------- decoder window layout (csrc/api.cu probe_layout)
def probe_layout(raw, off, need_cigar=True, need_aux=True):
    """(LPR, head chunks, tail chunks) the decoder picks for a chunk: the head window covers 36 + QNAME (+ CIGAR), the
    tail window the aux block, each sized for the 98th percentile of the chunk's first 4096 records."""
    n = len(off) - 1
    S = min(n, 4096)
    heads, auxs = [], []
    for k in range(S):
        o, ln = int(off[k]), int(off[k + 1]) - int(off[k])
        if ln < 36 or o + ln > len(raw):
            continue
        lq = int(raw[o + 12])
        nc = int(raw[o + 16]) | int(raw[o + 17]) << 8
        ls = int(np.frombuffer(bytes(raw[o + 20:o + 24]), dtype="<i4")[0])
        if ls < 0:
            continue
        ao = 36 + lq + 4 * nc + (ls + 1) // 2 + ls
        if ao > ln:
            continue
        heads.append(36 + lq + (4 * nc if need_cigar else 0))
        auxs.append(ln - ao)
    hc, tc = 4, (2 if need_aux else 0)
    if heads:
        heads.sort(); auxs.sort()
        q = min(len(heads) * 98 // 100, len(heads) - 1)
        hc = (15 + heads[q] + 15) // 16
        tc = (auxs[q] + 15 + 15) // 16 if need_aux else 0
    hc = max(hc, 4)
    lpr = 8 if hc + tc <= 8 else 16
    if hc + tc > 16:
        hc = min(hc, 12)
        tc = 16 - hc
    return lpr, hc, tc


def head_room(o, hc):
    """bytes of head window a record at chunk offset o has: 36 + lq (+ 4 nc) must not exceed it"""
    return 16 * hc - (o & 15)


def tail_room(aux_start, tc):
    """largest aux block that fits the tail window when the block starts at chunk offset aux_start (the window ends at
    the record's end rounded up to 16 bytes and spans tc chunks)"""
    return ((aux_start + 16 * tc) & ~15) - aux_start


def fits(rec, o, hc, tc):
    """(head fits, tail fits) of a record placed at chunk offset o, for need_cigar = need_aux = True"""
    lq = rec[12]
    nc, = struct.unpack_from("<H", rec, 16)
    ao = aux_offset(rec)
    aux_len = len(rec) - ao
    return (o & 15) + 36 + lq + 4 * nc <= 16 * hc, aux_len == 0 or aux_len <= tail_room(o + ao, tc)


# ---------------------------------------------------------------- QNAME hash (csrc/decode.cuh name_hash_eq)
def _mix(h, w):
    h = ((h ^ w) * np.uint32(0x9E3779B1)).astype(np.uint32)
    return h ^ (h >> np.uint32(15))


def name_hash(names):
    """32-bit QNAME hashes of equal-length names (bytes without the NUL), vectorised: the hash runs over the
    l_read_name bytes (NUL included) as little-endian 32-bit words, the last one zero-padded."""
    names = list(names)
    L = len(names[0]) + 1
    assert all(len(x) + 1 == L for x in names)
    W = (L + 3) // 4
    buf = np.zeros((len(names), 4 * W), dtype=np.uint8)
    buf[:, :L - 1] = np.frombuffer(b"".join(names), dtype=np.uint8).reshape(len(names), L - 1)
    words = buf.view("<u4")
    with np.errstate(over="ignore"):
        h = np.full(len(names), np.uint32(0x811c9dc5 ^ L), dtype=np.uint32)
        for k in range(W):
            h = _mix(h, words[:, k])
        h = (h * np.uint32(0x85ebca6b)).astype(np.uint32)
        return h ^ (h >> np.uint32(13))


def find_collisions(n_pairs, length=12, seed=2024, batch=400_000):
    """n_pairs pairs of distinct printable names of `length` characters with equal QNAME hashes"""
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789", dtype=np.uint8)
    pairs = []
    while len(pairs) < n_pairs:
        cand = alpha[rng.integers(0, len(alpha), size=(batch, length))]
        names = [bytes(r) for r in cand]
        h = name_hash(names)
        order = np.argsort(h, kind="stable")
        hs = h[order]
        for k in np.nonzero(hs[1:] == hs[:-1])[0]:
            a, b = names[order[k]], names[order[k + 1]]
            if a != b:
                pairs.append((a, b))
    return pairs[:n_pairs]
