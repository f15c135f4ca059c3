"""Host-side handle over the C ABI, used by the tests and bench.py.

The product host is C (the drop-in `msamtools` CLI links the same library); this
module is the thin Python view of the same calls.  Option names follow the
reference's command line: filter -l/-p/--ppt/-z/-v/-k/--rescore/--besthit/--uniqhit
(msam_filter.c:304-347) and profile --multi (msam_profile.c:570,712-728).
"""
import ctypes as C

import numpy as np

from . import _lib as L


class MsgError(RuntimeError):
    def __init__(self, code, text):
        super().__init__(f"[{code}] {text}")
        self.code = code
        self.text = text


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def parse_multi(s):
    """--multi accepts any prefix, first match in order all, equal, proportional, ignore (msam_profile.c:715-722)."""
    for i, full in enumerate(("all", "equal", "proportional", "ignore"), start=1):
        if full.startswith(s):
            return i
    raise ValueError(f"Do not understand --multi={s}")


class Context:
    """One msg_ctx (one GPU).  Keyword arguments mirror msg_config."""

    def __init__(self, *, l=0, p=None, ppt=None, z=None, invert=False, keep_unmapped=False, rescore=False,
                 besthit=False, uniqhit=False, do_filter=None,
                 profile=False, multi="proportional", coverage=False, coverage_summary=False, records=False, stats=False, kept=True,
                 n_targets=0, n_features=None, fmap=None, target_len=None,
                 device=0, n_ranks=1, rank=0, nccl_unique_id=None, force_slow=False, collate=False, exact=False):
        self.lib = L.load()
        cfg = L.MsgConfig()
        cfg.abi_version = L.MSG_ABI_VERSION
        if p is not None and ppt is not None:
            raise ValueError("-p cannot be combined with --ppt")
        PPT = 10 * p if p is not None else (ppt if ppt is not None else 0)
        max_clip = 100 - z if z is not None else 100
        any_filter = bool(l) or PPT != 0 or max_clip < 100 or besthit or uniqhit or rescore
        cfg.do_filter = int(any_filter if do_filter is None else do_filter)
        cfg.hit_mode = L.HIT_UNIQUE if uniqhit else (L.HIT_BEST if besthit else L.HIT_NONE)
        cfg.invert, cfg.keep_unmapped, cfg.rescore = int(invert), int(keep_unmapped), int(rescore)
        # records in any order, grouped by QNAME on the device at finish: True / 1 on one GPU; L.MSG_COLLATE_RANKS (2)
        # also across ranks (the records are exchanged by QNAME hash; finish, finish_coverage and pull_counts are collective)
        cfg.collate = int(collate)
        cfg.exact = int(exact)                     # equal / proportional abundances bit-identical to the reference
        cfg.min_length, cfg.ppt, cfg.max_clip = int(l), int(PPT), int(max_clip)
        cfg.want_kept, cfg.want_records, cfg.want_profile = int(kept), int(records), int(profile)
        cfg.want_coverage, cfg.want_stats = int(coverage), int(stats)
        cfg.share_type = parse_multi(multi) if isinstance(multi, str) else int(multi)
        cfg.debug_force_slow = int(force_slow)
        cfg.coverage_summary = int(coverage_summary)
        cfg.n_targets = int(n_targets)
        self._fmap = None if fmap is None else np.ascontiguousarray(fmap, dtype=np.int32)
        self._tlen = None if target_len is None else np.ascontiguousarray(target_len, dtype=np.uint32)
        cfg.n_features = int(n_features if n_features is not None else n_targets)
        cfg.fmap = None if self._fmap is None else self._fmap.ctypes.data_as(C.POINTER(C.c_int32))
        cfg.target_len = None if self._tlen is None else self._tlen.ctypes.data_as(C.POINTER(C.c_uint32))
        cfg.device, cfg.n_ranks, cfg.rank = int(device), int(n_ranks), int(rank)
        self._uid = nccl_unique_id
        cfg.nccl_unique_id = None if nccl_unique_id is None else C.cast(C.c_char_p(nccl_unique_id), C.c_void_p)
        self.cfg = cfg
        self.n_targets, self.n_features = cfg.n_targets, cfg.n_features
        h = C.c_void_p()
        rc = self.lib.msg_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise MsgError(rc, self.lib.msg_last_error(None).decode())
        self.h = h
        self._last_n = 0

    # -- plumbing
    def _check(self, rc):
        if rc != 0:
            raise MsgError(rc, self.lib.msg_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.msg_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- data path
    def push(self, raw, rec_off):
        raw = np.ascontiguousarray(raw, dtype=np.uint8)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
        n = len(rec_off) - 1 if len(rec_off) else 0
        self._last_n = n
        self._check(self.lib.msg_push(self.h, _ptr(raw), raw.nbytes, _ptr(rec_off), n))

    def push_async(self, raw, rec_off):
        """msg_push_async: queue the chunk and return; raw / rec_off must stay alive and unmodified until wait() or two
        further push_async calls have returned (the caller keeps the references)."""
        assert raw.dtype == np.uint8 and raw.flags.c_contiguous and rec_off.dtype == np.uint64 and rec_off.flags.c_contiguous
        n = len(rec_off) - 1 if len(rec_off) else 0
        self._last_n = n
        self._check(self.lib.msg_push_async(self.h, _ptr(raw), raw.nbytes, _ptr(rec_off), n))

    def push_device_async(self, d_raw, nbytes, d_off, nrec):
        self._last_n = nrec
        self._check(self.lib.msg_push_device_async(self.h, d_raw, nbytes, d_off, nrec))

    def wait(self):
        self._check(self.lib.msg_wait(self.h))

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self.lib.msg_device_alloc(self.h, nbytes, C.byref(p)))
        return p

    def device_free(self, p):
        self._check(self.lib.msg_device_free(self.h, p))

    def device_upload(self, dptr, host):
        host = np.ascontiguousarray(host)
        self._check(self.lib.msg_device_upload(self.h, dptr, _ptr(host), host.nbytes))

    def push_device(self, d_raw, nbytes, d_off, nrec):
        self._last_n = nrec
        self._check(self.lib.msg_push_device(self.h, d_raw, nbytes, d_off, nrec))

    def sync(self):
        self._check(self.lib.msg_sync(self.h))

    def reset(self):
        self._check(self.lib.msg_reset(self.h))

    # -- results
    def kept_count(self):
        n = C.c_size_t()
        self._check(self.lib.msg_kept_count(self.h, C.byref(n)))
        return n.value

    def pull_kept(self):
        n = self.kept_count()
        idx = np.empty(n, dtype=np.uint32)
        got = C.c_size_t()
        self._check(self.lib.msg_pull_kept(self.h, _ptr(idx), n, C.byref(got)))
        return idx

    def pull_records(self, out=None):
        """filtered record bytes of the last completed chunk; `out` = caller's (ideally pinned) uint8 buffer to fill"""
        nb, nr = C.c_size_t(), C.c_size_t()
        self._check(self.lib.msg_pull_records(self.h, None, 0, C.byref(nb), C.byref(nr)))
        if out is None:
            out = np.empty(nb.value, dtype=np.uint8)
        self._check(self.lib.msg_pull_records(self.h, _ptr(out), out.nbytes, C.byref(nb), C.byref(nr)))
        return out[:nb.value], nr.value

    def pull_stats(self):
        n = self._last_n
        cols = {k: np.empty(n, dtype=np.int32) for k in ("alen", "qlen", "qclip", "edit", "score")}
        flags = np.empty(n, dtype=np.uint8)
        self._check(self.lib.msg_pull_stats(self.h, n, _ptr(cols["alen"]), _ptr(cols["qlen"]), _ptr(cols["qclip"]),
                                            _ptr(cols["edit"]), _ptr(cols["score"]), _ptr(flags)))
        cols["flags"] = flags
        return cols

    def pull_counts(self):
        ui = np.empty(self.n_features, dtype=np.uint32)
        d = np.empty(self.n_features, dtype=np.float64)
        self._check(self.lib.msg_pull_counts(self.h, _ptr(ui), _ptr(d)))
        return ui, d

    def finish_profile(self):
        ab = np.zeros(self.n_features, dtype=np.float64)
        st = L.MsgProfileStats()
        self._check(self.lib.msg_finish_profile(self.h, _ptr(ab), C.byref(st)))
        stats = dict(mapped_inserts=st.mapped_inserts, uniq=st.uniq_mapper_count, multi=st.multi_mapper_count,
                     purged=st.purged_insert_count, iterations=st.em_iterations, converged=st.em_converged,
                     delta=list(st.em_delta)[:max(st.em_iterations, 0)], n_lists=st.multi_lists, n_entries=st.multi_entries)
        return ab, stats

    def finish_coverage(self):
        cov = np.zeros(self.n_targets, dtype=np.uint8)
        touched = np.zeros(self.n_targets, dtype=np.int64)
        total = np.zeros(self.n_targets, dtype=np.int64)
        self._check(self.lib.msg_finish_coverage(self.h, _ptr(cov), _ptr(touched), _ptr(total)))
        return cov, touched, total

    def pull_coverage(self, tid):
        depth = np.zeros(int(self._tlen[tid]), dtype=np.int32)
        self._check(self.lib.msg_pull_coverage(self.h, tid, _ptr(depth)))
        return depth

    def mark(self, slot):
        self._check(self.lib.msg_mark(self.h, slot))

    def elapsed_ms(self, a, b):
        ms = C.c_double()
        self._check(self.lib.msg_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def timing(self, reset=False):
        t = L.MsgTiming()
        self._check(self.lib.msg_get_timing(self.h, C.byref(t), int(reset)))
        return {k: getattr(t, k) for k, _ in L.MsgTiming._fields_}


class PinnedBuffer:
    """Page-locked host memory from msg_host_alloc as a numpy uint8 array (`.array`).  msg_push decodes such buffers in
    place (zero-copy over PCIe) when the fused filter->profile pass applies; free with close() or a `with` block."""

    def __init__(self, nbytes, device=0):
        self.lib = L.load()
        self.ptr = C.c_void_p()
        rc = self.lib.msg_host_alloc(int(device), int(nbytes), C.byref(self.ptr))
        if rc != 0:
            raise RuntimeError(f"msg_host_alloc failed ({rc}): {self.lib.msg_last_error(None).decode()}")
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_uint8)), shape=(max(int(nbytes), 1),))[:int(nbytes)]

    def close(self):
        if self.ptr:
            self.array = None
            self.lib.msg_host_free(self.ptr)
            self.ptr = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


_host = None


def _hostlib():
    """libmsamhost.so: the CPU-only part of the ABI (csrc/host/recindex.c); never maps the CUDA library."""
    global _host
    if _host is None:
        import os
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libmsamhost.so")
        if not os.path.exists(path):
            raise ImportError(f"{path} not found: run `make`")
        lib = C.CDLL(path)
        sz = C.c_size_t
        lib.msg_index_records.argtypes = [C.c_void_p, sz, C.c_void_p, sz, C.POINTER(sz), C.POINTER(sz), C.c_int]
        lib.msg_index_records.restype = C.c_int
        lib.msg_split_point.argtypes = [C.c_void_p, C.c_void_p, sz, sz]
        lib.msg_split_point.restype = sz
        _host = lib
    return _host


def index_records(raw):
    """Host offset index over an uncompressed BAM record stream (msg_index_records)."""
    lib = _hostlib()
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    n, used = C.c_size_t(), C.c_size_t()
    rc = lib.msg_index_records(_ptr(raw), raw.nbytes, None, 0, C.byref(n), C.byref(used), 0)
    if rc != 0:
        raise MsgError(rc, "malformed record stream")
    off = np.empty(n.value + 1, dtype=np.uint64)
    rc = lib.msg_index_records(_ptr(raw), raw.nbytes, _ptr(off), len(off), C.byref(n), C.byref(used), 0)
    if rc != 0:
        raise MsgError(rc, "malformed record stream")
    return off


def split_point(raw, rec_off, want):
    lib = _hostlib()
    raw = np.ascontiguousarray(raw, dtype=np.uint8)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
    return lib.msg_split_point(_ptr(raw), _ptr(rec_off), len(rec_off) - 1, want)


def nccl_unique_id():
    lib = L.load()
    buf = C.create_string_buffer(128)
    rc = lib.msg_nccl_unique_id(buf)
    if rc != 0:
        raise MsgError(rc, lib.msg_last_error(None).decode())
    return buf.raw
