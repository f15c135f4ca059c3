"""ctypes view of the CPU oracle (oracle/msam_oracle.c).  TEST INFRASTRUCTURE ONLY.

Imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs -- never by anything under msamtools_b200/.
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmsam_oracle.so")

ORC_ENOTAG, ORC_ENOAS, ORC_EFORMAT = -5, -6, -7


class OrcFilterCfg(C.Structure):
    _fields_ = [("min_length", C.c_int32), ("ppt", C.c_int32), ("max_clip", C.c_int32),
                ("do_filter", C.c_int32), ("hit_mode", C.c_int32), ("invert", C.c_int32),
                ("keep_unmapped", C.c_int32), ("rescore", C.c_int32)]


class OrcProfileOut(C.Structure):
    _fields_ = [("mapped_inserts", C.c_uint32), ("uniq", C.c_uint32), ("multi", C.c_uint32), ("purged", C.c_uint32),
                ("iterations", C.c_int32), ("converged", C.c_int32), ("delta", C.c_double * 20),
                ("n_lists", C.c_uint64), ("n_entries", C.c_uint64)]


class OracleError(RuntimeError):
    def __init__(self, code):
        super().__init__(f"oracle error {code}")
        self.code = code


_lib = None


def reference_dir():
    """The checkout of the reference msamtools sources that oracle/Makefile.ref compiles: MSAMTOOLS_REFERENCE if set, else
    BASELINE.json's reference_path; None when that directory does not exist."""
    d = os.environ.get("MSAMTOOLS_REFERENCE")
    if not d:
        with open(os.path.join(_HERE, "..", "BASELINE.json")) as fh:
            d = json.load(fh).get("reference_path", "")
    return d if d and os.path.isdir(d) else None


def build():
    subprocess.check_call(["make", "-s", "-C", _HERE])


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        lib = C.CDLL(LIB_PATH)
        vp, sz = C.c_void_p, C.c_size_t
        lib.orc_record_stats.argtypes = [vp, vp, sz, vp, vp, vp, vp, vp, vp, vp]
        lib.orc_filter.argtypes = [vp, vp, sz, C.POINTER(OrcFilterCfg), vp, C.POINTER(sz)]
        lib.orc_emit_records.argtypes = [vp, vp, vp, sz, C.POINTER(OrcFilterCfg), vp, sz, C.POINTER(sz)]
        lib.orc_profile_new.argtypes = [C.c_int32, C.c_int32, vp, C.c_int]; lib.orc_profile_new.restype = vp
        lib.orc_profile_free.argtypes = [vp]; lib.orc_profile_free.restype = None
        lib.orc_profile_push.argtypes = [vp, vp, vp, vp, sz]
        lib.orc_profile_counts.argtypes = [vp, vp, vp]
        lib.orc_profile_finish.argtypes = [vp, vp, C.POINTER(OrcProfileOut)]
        lib.orc_coverage_new.argtypes = [C.c_int32, vp]; lib.orc_coverage_new.restype = vp
        lib.orc_coverage_free.argtypes = [vp]; lib.orc_coverage_free.restype = None
        lib.orc_coverage_push.argtypes = [vp, vp, vp, vp, sz]
        lib.orc_coverage_finish.argtypes = [vp, vp, vp, vp]
        lib.orc_coverage_depth.argtypes = [vp, C.c_int32, vp]
        lib.orc_pipeline.argtypes = [vp, vp, sz, C.POINTER(OrcFilterCfg), C.c_int32, C.c_int32, vp, C.c_int, vp,
                                     C.POINTER(OrcProfileOut), C.POINTER(sz)]
        _lib = lib
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def filter_cfg(*, l=0, p=None, ppt=None, z=None, invert=False, keep_unmapped=False, rescore=False,
               besthit=False, uniqhit=False, do_filter=None):
    PPT = 10 * p if p is not None else (ppt if ppt is not None else 0)
    max_clip = 100 - z if z is not None else 100
    any_filter = bool(l) or PPT != 0 or max_clip < 100 or besthit or uniqhit or rescore
    return OrcFilterCfg(int(l), int(PPT), int(max_clip), int(any_filter if do_filter is None else do_filter),
                        2 if uniqhit else (1 if besthit else 0), int(invert), int(keep_unmapped), int(rescore))


def record_stats(raw, off):
    lib = load()
    n = len(off) - 1
    out = {k: np.zeros(n, dtype=np.int32) for k in ("alen", "qlen", "qclip", "edit", "score")}
    has_as = np.zeros(n, dtype=np.uint8)
    has_tag = np.zeros(n, dtype=np.uint8)
    rc = lib.orc_record_stats(_p(raw), _p(off), n, _p(out["alen"]), _p(out["qlen"]), _p(out["qclip"]), _p(out["edit"]),
                              _p(out["score"]), _p(has_as), _p(has_tag))
    if rc:
        raise OracleError(rc)
    out["has_as"], out["has_tag"] = has_as, has_tag
    return out


def filter_stream(raw, off, cfg):
    """mFilterFile + pool writers -> kept record indices in output order."""
    lib = load()
    n = len(off) - 1
    idx = np.zeros(max(n, 1), dtype=np.uint32)
    m = C.c_size_t()
    rc = lib.orc_filter(_p(raw), _p(off), n, C.byref(cfg), _p(idx), C.byref(m))
    if rc:
        raise OracleError(rc)
    return idx[:m.value].copy()


def emit_records(raw, off, idx, cfg):
    lib = load()
    cap = int(sum(int(off[i + 1] - off[i]) + 8 for i in idx)) + 16
    out = np.zeros(cap, dtype=np.uint8)
    nb = C.c_size_t()
    idx = np.ascontiguousarray(idx, dtype=np.uint32)
    rc = lib.orc_emit_records(_p(raw), _p(off), _p(idx), len(idx), C.byref(cfg), _p(out), cap, C.byref(nb))
    if rc:
        raise OracleError(rc)
    return out[:nb.value].copy()


def profile(raw, off, idx, n_targets, share_type, fmap=None, n_features=None, chunks=None):
    """Returns (abundance, stats dict, ui, d).  idx None = every record (plain `profile`)."""
    lib = load()
    nf = n_targets if n_features is None else n_features
    fm = None if fmap is None else np.ascontiguousarray(fmap, dtype=np.int32)
    h = lib.orc_profile_new(n_targets, nf, _p(fm), share_type)
    try:
        if idx is not None:
            idx = np.ascontiguousarray(idx, dtype=np.uint32)
        m = len(idx) if idx is not None else len(off) - 1
        rc = lib.orc_profile_push(h, _p(raw), _p(off), _p(idx), m)
        if rc:
            raise OracleError(rc)
        ui = np.zeros(max(nf, 1), dtype=np.uint32)
        d = np.zeros(max(nf, 1), dtype=np.float64)
        lib.orc_profile_counts(h, _p(ui), _p(d))
        ab = np.zeros(max(nf, 1), dtype=np.float64)
        po = OrcProfileOut()
        rc = lib.orc_profile_finish(h, _p(ab), C.byref(po))
        if rc:
            raise OracleError(rc)
    finally:
        lib.orc_profile_free(h)
    stats = dict(mapped_inserts=po.mapped_inserts, uniq=po.uniq, multi=po.multi, purged=po.purged,
                 iterations=po.iterations, converged=po.converged, delta=list(po.delta)[:max(po.iterations, 0)],
                 n_lists=po.n_lists, n_entries=po.n_entries)
    return ab[:nf], stats, ui[:nf], d[:nf]


def coverage(raw, off, idx, target_len, want_depth=False):
    lib = load()
    tl = np.ascontiguousarray(target_len, dtype=np.uint32)
    T = len(tl)
    h = lib.orc_coverage_new(T, _p(tl))
    try:
        if idx is not None:
            idx = np.ascontiguousarray(idx, dtype=np.uint32)
        m = len(idx) if idx is not None else len(off) - 1
        rc = lib.orc_coverage_push(h, _p(raw), _p(off), _p(idx), m)
        if rc:
            raise OracleError(rc)
        cov = np.zeros(max(T, 1), dtype=np.uint8)
        touched = np.zeros(max(T, 1), dtype=np.int64)
        total = np.zeros(max(T, 1), dtype=np.int64)
        lib.orc_coverage_finish(h, _p(cov), _p(touched), _p(total))
        depth = None
        if want_depth:
            depth = []
            for t in range(T):
                dd = np.zeros(max(int(tl[t]), 1), dtype=np.int32)
                lib.orc_coverage_depth(h, t, _p(dd))
                depth.append(dd[:int(tl[t])])
    finally:
        lib.orc_coverage_free(h)
    return cov[:T], touched[:T], total[:T], depth


def pipeline(raw, off, cfg, n_targets, share_type, fmap=None, n_features=None):
    """filter -> profile in one C call (what bench.py times as the CPU baseline)."""
    lib = load()
    nf = n_targets if n_features is None else n_features
    fm = None if fmap is None else np.ascontiguousarray(fmap, dtype=np.int32)
    ab = np.zeros(max(nf, 1), dtype=np.float64)
    po = OrcProfileOut()
    nk = C.c_size_t()
    rc = lib.orc_pipeline(_p(raw), _p(off), len(off) - 1, C.byref(cfg), n_targets, nf, _p(fm), share_type, _p(ab),
                          C.byref(po), C.byref(nk))
    if rc:
        raise OracleError(rc)
    stats = dict(mapped_inserts=po.mapped_inserts, uniq=po.uniq, multi=po.multi, purged=po.purged,
                 iterations=po.iterations, converged=po.converged, n_lists=po.n_lists, n_kept=nk.value)
    return ab[:nf], stats
