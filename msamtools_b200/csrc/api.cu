// api.cu -- context, chunk pipeline and the extern "C" surface of libmsamtools_b200.so
// (include/msamtools_b200.h).  Host orchestration only; all record work is in the kernels.
#include "../../include/msamtools_b200.h"
#include "common.cuh"
#include "scan.cuh"
#include "decode.cuh"
#include "besthit.cuh"
#include "profile.cuh"
#include "coverage.cuh"
#include "gather.cuh"
#include "fused.cuh"
#include "collate.cuh"

#include <nccl.h>        // types only; the library itself is dlopen'ed (no link-time dependency)
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>

#include "host/recindex.c"      // msg_index_records, msg_split_point

using namespace msg;

// ------------------------------------------------------------------------------------------------
namespace {

thread_local std::string g_create_error;

struct DevBuf {
    void *p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap && p) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    // grow but keep the first `keep` bytes (amortised doubling; used by the multi-mapper CSR)
    cudaError_t reserve_keep(size_t bytes, size_t keep, cudaStream_t st) {
        if (bytes <= cap && p) return cudaSuccess;
        size_t want = bytes + bytes / 2 + 256;
        void *np_ = nullptr;
        cudaError_t e = cudaMalloc(&np_, want);
        if (e != cudaSuccess) return e;
        if (p && keep) { e = cudaMemcpyAsync(np_, p, keep, cudaMemcpyDeviceToDevice, st); if (e == cudaSuccess) e = cudaStreamSynchronize(st); }
        if (p) cudaFree(p);
        p = np_; cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};


struct NcclApi {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    // point-to-point, for the record exchange of collation across ranks (MSG_COLLATE_RANKS)
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    bool load(std::string &err) {
        if (h) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so", nullptr};
        for (int i = 0; names[i] && !h; i++) h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
        if (!h) { err = std::string("cannot dlopen libnccl.so.2: ") + dlerror(); return false; }
        GetUniqueId = (decltype(GetUniqueId))dlsym(h, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(h, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(h, "ncclAllReduce");
        AllGather = (decltype(AllGather))dlsym(h, "ncclAllGather");
        CommDestroy = (decltype(CommDestroy))dlsym(h, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(h, "ncclGetErrorString");
        Send = (decltype(Send))dlsym(h, "ncclSend");
        Recv = (decltype(Recv))dlsym(h, "ncclRecv");
        GroupStart = (decltype(GroupStart))dlsym(h, "ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))dlsym(h, "ncclGroupEnd");
        if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) { err = "libnccl is missing required symbols"; return false; }
        return true;
    }
};
NcclApi g_nccl;

} // namespace

// One chunk in flight on the fused filter->profile pass (msg_push_async): where its bytes are, the pinned block its
// small results land in, and what is needed to rerun it on the general pipeline should the guard decline it.
struct Slot {
    DevBuf raw, off;                          // staged copies of host chunks
    uint32_t *h_res = nullptr;                // pinned: [0..4] inserts, uniq, multi, guard flag, kept; [5..6] list cursors; [8..9] error word
    cudaEvent_t copied = nullptr, done = nullptr;
    bool pending = false;
    const uint8_t *d_raw = nullptr, *h_raw = nullptr; const uint64_t *d_off = nullptr, *h_off = nullptr;
    uint64_t nbytes = 0, readable = 0, n = 0; bool zero_copy = false;
    uint64_t ub_lists = 0, ub_ent = 0;        // list space reserved for it (worst case) until its real counts are known
    uint64_t key_base = 0;                    // records pushed before it (exact mode: the input order of its lists)
};

struct msg_ctx {
    msg_config cfg;
    std::string err;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    Slot slot[2]; int next_slot = 0;          // slot[next_slot] is the older of the two
    bool cursor_dirty = true;                 // host csr_lists / csr_ent must be uploaded before the next fused pass
    uint64_t inflight_lists = 0, inflight_ent = 0;
    bool has_filter = false, need_stats = false, cov_fused = false;
    uint64_t zc_chunks = 0;                           // chunks decoded straight from pinned host memory
    uint32_t lay_lpr = 0, lay_hc = 0, lay_tc = 0;     // decode window layout (probe_layout)
    uint32_t decode_mode = 0;

    // static tables
    int32_t *d_fmap = nullptr; uint32_t *d_tlen = nullptr; uint64_t *d_covbase = nullptr;
    uint64_t cov_cells = 0;

    // chunk staging (msg_push) and per-chunk columns
    DevBuf tid, fb, score, hash, nid, st_alen, st_qlen, st_qclip, st_edit;
    DevBuf kbase, worklist, gmeta, out_idx, tile_sums, pcount, scanv, biglist;
    uint32_t *d_wl = nullptr;                  // [0] best-hit worklist length [1] profile worklist length
    // fused filter+besthit -> profile path (fused.cuh): chunk-local accumulators, list cursors, window summaries
    uint32_t *d_ui_tmp = nullptr; double *d_d_tmp = nullptr; uint32_t *d_fcnt = nullptr, *d_cursor = nullptr; DevBuf win;
    bool fused_enabled = false; uint64_t fused_chunks = 0, fused_fallbacks = 0;
    DevBuf out_len, out_off, plan, out_rec;
    const uint8_t *cur_raw = nullptr; const uint64_t *cur_off = nullptr;
    uint64_t cur_n = 0, cur_nbytes = 0;
    uint64_t n_kept = 0; bool have_stream = false;   // have_stream: out_idx valid (else identity)
    uint64_t out_bytes = 0;

    // device scalars: err[2], scan totals, accounting
    uint32_t *d_err = nullptr;                 // [0] flags [1] first bad record
    uint32_t *h_pin = nullptr;                 // 512 B of pinned host memory: small results land here with ONE stream sync
    double *h_ab = nullptr;                    // pinned staging for the abundance vector (F doubles)
    unsigned long long *d_acct = nullptr;      // [0] alg bytes [1] slow records
    void *d_total = nullptr;                   // 16 bytes scratch for scan totals

    // profile accumulators
    uint32_t *d_ui = nullptr; double *d_d = nullptr; uint32_t *d_counters = nullptr;   // counters[8]
    DevBuf csr_off, csr_len, csr_fid; uint64_t csr_lists = 0, csr_ent = 0;     // multi-mapper lists (CSR), appended per chunk
    // exact mode (cfg.exact): the input key of every list, and the per-feature incidence in key order (built at finish)
    DevBuf csr_key, ex_beg, ex_cur, ex_keys, ex_big, ex_list, ex_sums;
    uint64_t rec_base = 0, cur_key_base = 0;   // records pushed since the reset / before the chunk being profiled
    bool ex_ready = false;                     // the incidence (and, equal mode, d) match the lists
    DevBuf t_ui, t_d, t_cnt, t_cov;                                    // allreduce staging (n_ranks > 1)
    uint32_t *d_stamp = nullptr; uint32_t stamp_next = 0;
    double *d_U = nullptr, *d_a = nullptr, *d_inc = nullptr, *d_partial = nullptr, *d_delta = nullptr;
    uint32_t *d_purged = nullptr;
    uint32_t *d_bflag = nullptr;               // broadcast flag of em_loop_multi_kernel (monotonic epochs)

    // coverage accumulators
    int32_t *d_diff = nullptr, *d_depth = nullptr; uint8_t *d_covered = nullptr;
    bool cov_bits = false; unsigned long long *d_covbits = nullptr; uint64_t cov_words = 0;      // summary mode (coverage.cuh)
    bool l2_window = false;
    unsigned long long *d_touched = nullptr; long long *d_sum = nullptr;
    bool cov_finished = false;

    // multi-GPU
    ncclComm_t comm = nullptr;
    // peer-memory exchange for the fused EM loop (profile.cuh em_loop_multi_kernel): CUDA IPC mappings of every rank's region
    unsigned char *peer_region = nullptr; size_t peer_region_bytes = 0; PeerTable peer_tab; std::vector<void *> ipc_opened; bool p2p_ok = false; uint32_t em_epoch = 32;

    // timing
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_decode, ev_total;
    std::vector<cudaEvent_t> ev_free;
    cudaEvent_t marks[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    uint32_t err_rec = 0xffffffffu;            // record index of the last error reported (d_err[1]), 0xffffffff if none

    // collation (cfg.collate, collate.cuh): record heads held on the device until a finish groups them by QNAME
    DevBuf coll_arena, coll_aoff, coll_keys, coll_keys2, coll_len, coll_hist, coll_bstart, coll_list, coll_grouped, coll_goff;
    uint64_t coll_n = 0, coll_bytes = 0;       // records and head bytes held in this scope
    bool coll_dirty = false;                   // pushes since the last collation
    bool coll_done = false;                    // a finish collated this scope: the next push starts a new one
    // collation across ranks (MSG_COLLATE_RANKS, n_ranks > 1): the agreed size matrix and small flags, and the global
    // input ordinal where each rank's records start in the last exchange (n_ranks + 1 entries); coll_len then holds the
    // global ordinal of every received record
    DevBuf coll_xchg;
    std::vector<unsigned long long> coll_base;
    double decode_ms = 0, total_ms = 0; uint64_t decode_launches = 0, kernel_launches = 0;
    uint64_t h2d_bytes = 0, d2h_bytes = 0;
};

namespace {

int fail(msg_ctx *c, int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}

#define CU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) \
    return fail(c, e__ == cudaErrorMemoryAllocation ? MSG_ENOMEM : MSG_ECUDA, "%s failed: %s", #call, cudaGetErrorString(e__)); } while (0)
#define NC(call) do { ncclResult_t r__ = (call); if (r__ != ncclSuccess) \
    return fail(c, MSG_ENCCL, "%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "nccl error"); } while (0)
#define LAUNCHED(c) do { (c)->kernel_launches++; cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) \
    return fail(c, MSG_ECUDA, "kernel launch failed (%s:%d): %s", __FILE__, __LINE__, cudaGetErrorString(e__)); } while (0)

inline uint32_t nblocks(uint64_t n, uint32_t per) { return (uint32_t)((n + per - 1) / per); }

cudaEvent_t get_event(msg_ctx *c)
{
    if (!c->ev_free.empty()) { cudaEvent_t e = c->ev_free.back(); c->ev_free.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
}

void harvest_events(msg_ctx *c)
{   // stream must be idle
    for (auto &pr : c->ev_decode) { float ms = 0; cudaEventElapsedTime(&ms, pr.first, pr.second); c->decode_ms += ms; c->decode_launches++;
                                    c->ev_free.push_back(pr.first); c->ev_free.push_back(pr.second); }
    for (auto &pr : c->ev_total)  { float ms = 0; cudaEventElapsedTime(&ms, pr.first, pr.second); c->total_ms += ms;
                                    c->ev_free.push_back(pr.first); c->ev_free.push_back(pr.second); }
    c->ev_decode.clear(); c->ev_total.clear();
}

// exclusive scan driver: in -> out functor, total (T) left in c->d_total
template <class T, class In, class Out>
int run_scan(msg_ctx *c, In in, Out out, uint64_t n, T *h_total)
{
    uint32_t ntiles = nblocks(n, SCAN_TILE);
    if (ntiles == 0) { if (h_total) *h_total = T(0); return MSG_OK; }
    CU(c->tile_sums.reserve((size_t)ntiles * sizeof(T)));
    T *ts = c->tile_sums.as<T>();
    scan_reduce_kernel<T, In><<<ntiles, SCAN_BLOCK, 0, c->stream>>>(in, n, ts); LAUNCHED(c);
    scan_tiles_kernel<T><<<1, SCAN_BLOCK, 0, c->stream>>>(ts, ntiles, reinterpret_cast<T *>(c->d_total)); LAUNCHED(c);
    scan_apply_kernel<T, In, Out><<<ntiles, SCAN_BLOCK, 0, c->stream>>>(in, out, n, ts); LAUNCHED(c);
    if (h_total) {
        CU(cudaMemcpyAsync(h_total, c->d_total, sizeof(T), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->d2h_bytes += sizeof(T);
    }
    return MSG_OK;
}

int report_device_errors(msg_ctx *c, const uint32_t *h);
// CTAs per SM of the cooperative PropSharing kernels: 3 where a[] lives in shared memory (F <= 2048: measured best, round 1),
// 4 for the global-memory kernels of larger feature sets (latency-bound gathers; config-5 step at 100 M records: 2: 13.01,
// 3: 12.50, 4: 12.10, 6: 12.14 ms; at 20 M records: 2: 3.38, 4: 3.30, 6: 3.20, 8: 3.19 ms).  MSG_EM_CTAS overrides both.
static const int EM_CTAS_ENV = getenv("MSG_EM_CTAS") ? atoi(getenv("MSG_EM_CTAS")) : 0;

int check_device_errors(msg_ctx *c)
{
    uint32_t *h = c->h_pin + 8;
    CU(cudaMemcpyAsync(h, c->d_err, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->d2h_bytes += 8;
    return report_device_errors(c, h);
}

int report_device_errors(msg_ctx *c, const uint32_t *h)
{
    c->err_rec = h[1];
    if (h[0]) {                   // reported once: the next chunk starts with a clean error word
        cudaMemsetAsync(c->d_err, 0, 4, c->stream);
        cudaMemsetAsync(c->d_err + 1, 0xff, 4, c->stream);
    }
    if (h[0] & DERR_FORMAT) return fail(c, MSG_EFORMAT, "malformed BAM record or reference id out of range (first near record %u)", h[1]);
    if (h[0] & DERR_CGTAG)  return fail(c, MSG_EFORMAT, "CIGAR with more than 65535 operations (CG tag, near record %u) is not supported", h[1]);
    if (h[0] & DERR_NOTAG)  return fail(c, MSG_ENOTAG, "Either NM or MD must be present in SAM/BAM input for 'filter' command. Type 'msamtools filter -h' for details.");
    if (h[0] & DERR_NOAS)   return fail(c, MSG_ENOAS, "Required field AS not found in SAM/BAM input. Type 'msamtools -h' for details.");
    return MSG_OK;
}

int profile_stage(msg_ctx *c, const uint32_t *stream, uint64_t m)
{
    const msg_config &g = c->cfg;
    const uint64_t n = c->cur_n;
    if (m == 0) return MSG_OK;
    // QNAME run ids over ALL records of the chunk (inclusive count of run heads)
    CU(c->nid.reserve(n * 4));
    int rc = run_scan<uint32_t>(c, InFlagBit{c->fb.as<uint32_t>(), FB_EQPREV, 0u}, OutInclU32{c->nid.as<uint32_t>()}, n, (uint32_t *)nullptr);
    if (rc) return rc;

    // exact mode also writes lists for the inserts that add 1/n to d (MSG_MULTI_EQUAL); d is then summed at finish
    const bool ex = g.exact != 0;
    const bool lists = g.share_type == MSG_MULTI_PROPORTIONAL || (ex && g.share_type == MSG_MULTI_EQUAL);
    if (lists) CU(c->pcount.reserve(m * 4));
    const uint32_t big_cap = 65536;
    CU(c->biglist.reserve((size_t)big_cap * 4));
    ProfParams p;
    p.raw = c->cur_raw; p.off = c->cur_off; p.stream = stream; p.m = m;
    p.tid = c->tid.as<int32_t>(); p.nid = c->nid.as<uint32_t>(); p.hash = c->hash.as<uint32_t>();
    p.fmap = c->d_fmap; p.n_targets = g.n_targets; p.n_features = g.n_features; p.share_type = g.share_type;
    p.ui = c->d_ui; p.d = c->d_d; p.counters = c->d_counters;
    p.pcount = lists ? c->pcount.as<uint32_t>() : nullptr;
    p.big = c->biglist.as<uint32_t>(); p.big_cap = big_cap; p.big_threshold = 1024; p.err = c->d_err;
    p.key = nullptr; p.key_base = c->cur_key_base;
    CU(c->worklist.reserve((std::max<uint64_t>(n, m) / 32 + 2) * 4));
    if (lists) CU(c->gmeta.reserve(m));
    CU(cudaMemsetAsync(c->d_wl + 1, 0, 4, c->stream));
    uint8_t *gmeta = lists ? c->gmeta.as<uint8_t>() : nullptr;
    const uint32_t pgrid = std::min<uint32_t>(nblocks(m / 32 + 1, 256), 148u * 4u);
    const bool sh = (uint32_t)g.n_features <= 4096u;
    auto warp_count = sh ? (ex ? profile_warp_count_kernel<true, true> : profile_warp_count_kernel<true, false>)
                         : (ex ? profile_warp_count_kernel<false, true> : profile_warp_count_kernel<false, false>);
    warp_count<<<nblocks(m, 256), 256, sh ? (size_t)g.n_features * 4 : 0, c->stream>>>(p, gmeta, c->worklist.as<uint32_t>(), c->d_wl + 1); LAUNCHED(c);
    auto walk_count = ex ? profile_walk_count_kernel<true> : profile_walk_count_kernel<false>;
    walk_count<<<pgrid, 256, 0, c->stream>>>(p, c->worklist.as<uint32_t>(), c->d_wl + 1); LAUNCHED(c);
    auto big_kernel = ex ? profile_big_kernel<true> : profile_big_kernel<false>;

    uint32_t nbig = 0;
    if (lists) {
        CU(c->scanv.reserve(m * 8));
        unsigned long long tot = 0;
        rc = run_scan<unsigned long long>(c, InPcountPacked{p.pcount}, OutExclU64{c->scanv.as<unsigned long long>()}, m, &tot);
        if (rc) return rc;
        const uint32_t nl = (uint32_t)(tot >> 32), ne = (uint32_t)tot;
        if (nl) {
            if (c->csr_lists + nl >= 0xffffffffull || c->csr_ent + ne >= 0xffffffffull) return fail(c, MSG_ERANGE, "multi-mapper CSR exceeds 2^32 entries on one GPU");
            CU(c->csr_off.reserve_keep((c->csr_lists + nl + 1) * 4, c->csr_lists * 4, c->stream));
            CU(c->csr_len.reserve_keep((c->csr_lists + nl + 1) * 4, c->csr_lists * 4, c->stream));
            CU(c->csr_fid.reserve_keep((c->csr_ent + ne + 1) * 4, c->csr_ent * 4, c->stream));
            if (ex) { CU(c->csr_key.reserve_keep((c->csr_lists + nl + 1) * 8, c->csr_lists * 8, c->stream)); p.key = c->csr_key.as<unsigned long long>(); }
            (ex ? profile_warp_fill_kernel<true> : profile_warp_fill_kernel<false>)<<<nblocks(m, 256), 256, 0, c->stream>>>(p, gmeta, c->scanv.as<unsigned long long>(), c->csr_off.as<uint32_t>(),
                                                                             c->csr_len.as<uint32_t>(), c->csr_fid.as<int32_t>(), (uint32_t)c->csr_lists, (uint32_t)c->csr_ent); LAUNCHED(c);
            (ex ? profile_walk_fill_kernel<true> : profile_walk_fill_kernel<false>)<<<pgrid, 256, 0, c->stream>>>(p, c->scanv.as<unsigned long long>(), c->csr_off.as<uint32_t>(), c->csr_len.as<uint32_t>(),
                                                                   c->csr_fid.as<int32_t>(), (uint32_t)c->csr_lists, (uint32_t)c->csr_ent, c->worklist.as<uint32_t>(), c->d_wl + 1); LAUNCHED(c);
            c->csr_lists += nl; c->csr_ent += ne;
        }
    }
    CU(cudaMemcpyAsync(&nbig, c->d_counters + 3, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->d2h_bytes += 4;
    if (nbig) {
        if (nbig > big_cap) return fail(c, MSG_ERANGE, "more than %u oversized QNAME groups in one chunk", big_cap);
        if (!c->d_stamp) { CU(cudaMalloc(&c->d_stamp, (size_t)(g.n_features > 0 ? g.n_features : 1) * 4));
                           CU(cudaMemsetAsync(c->d_stamp, 0, (size_t)(g.n_features > 0 ? g.n_features : 1) * 4, c->stream)); }
        uint32_t *d_tot = reinterpret_cast<uint32_t *>(c->d_total);
        big_kernel<<<1, 1, 0, c->stream>>>(p, nbig, c->d_stamp, c->stamp_next, nullptr, nullptr, nullptr, d_tot, 0, 0, 0); LAUNCHED(c);
        c->stamp_next += nbig + 1;
        if (lists) {
            uint32_t tot[2];
            CU(cudaMemcpyAsync(tot, d_tot, 8, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            if (tot[0]) {
                if (c->csr_lists + tot[0] >= 0xffffffffull || c->csr_ent + tot[1] >= 0xffffffffull) return fail(c, MSG_ERANGE, "multi-mapper CSR exceeds 2^32 entries on one GPU");
                CU(c->csr_off.reserve_keep((c->csr_lists + tot[0] + 1) * 4, c->csr_lists * 4, c->stream));
                CU(c->csr_len.reserve_keep((c->csr_lists + tot[0] + 1) * 4, c->csr_lists * 4, c->stream));
                CU(c->csr_fid.reserve_keep((c->csr_ent + tot[1] + 2) * 4, c->csr_ent * 4, c->stream));
                if (ex) { CU(c->csr_key.reserve_keep((c->csr_lists + tot[0] + 1) * 8, c->csr_lists * 8, c->stream)); p.key = c->csr_key.as<unsigned long long>(); }
                big_kernel<<<1, 1, 0, c->stream>>>(p, nbig, c->d_stamp, c->stamp_next, c->csr_off.as<uint32_t>(), c->csr_len.as<uint32_t>(), c->csr_fid.as<int32_t>(),
                                                           d_tot, 1, (uint32_t)c->csr_lists, (uint32_t)c->csr_ent); LAUNCHED(c);
                c->stamp_next += nbig + 1;
                c->csr_lists += tot[0]; c->csr_ent += tot[1];
            }
        }
        CU(cudaMemsetAsync(c->d_counters + 3, 0, 4, c->stream));
    }
    return MSG_OK;
}

int records_stage(msg_ctx *c, const uint32_t *stream, uint64_t m)
{
    c->out_bytes = 0;
    if (m == 0) return MSG_OK;
    CU(c->out_len.reserve(m * 4)); CU(c->out_off.reserve(m * 8)); CU(c->plan.reserve(m * sizeof(GatherPlan)));
    const int rescore = c->cfg.do_filter && c->cfg.rescore;
    gather_plan_kernel<<<nblocks(m, 256), 256, 0, c->stream>>>(c->cur_raw, c->cur_off, stream, m, rescore,
                                                              c->out_len.as<uint32_t>(), c->plan.as<GatherPlan>()); LAUNCHED(c);
    unsigned long long tot = 0;
    int rc = run_scan<unsigned long long>(c, InLenU64{c->out_len.as<uint32_t>()}, OutExclU64{c->out_off.as<unsigned long long>()}, m, &tot);
    if (rc) return rc;
    CU(c->out_rec.reserve(tot + 16));
    gather_copy_kernel<<<nblocks(m * 32, 256), 256, 0, c->stream>>>(c->cur_raw, c->cur_off, stream, m, c->out_off.as<unsigned long long>(),
                                                                   c->out_len.as<uint32_t>(), c->plan.as<GatherPlan>(),
                                                                   c->score.as<int32_t>(), c->out_rec.as<uint8_t>()); LAUNCHED(c);
    c->out_bytes = tot;
    return MSG_OK;
}

int wait_all(msg_ctx *c);

// filter+besthit -> profile without materialising the kept stream (fused.cuh), enqueued WITHOUT a host round trip:
// the guard flag, counters, list cursors and the error word of the chunk are copied into the slot's pinned block and
// read when the slot is completed (complete_slot).  The list cursors live on the device between chunks; if the guard
// trips, fused_commit_kernel drops the chunk's partial sums and puts the cursors back, and the host later reruns the
// chunk on the general pipeline.  *queued = false: the chunk cannot take this path (list space would pass 2^32).
int fused_enqueue(msg_ctx *c, const DecodeParams &dp, uint64_t n, Slot &sl, bool *queued)
{
    const msg_config &g = c->cfg;
    *queued = false;
    const bool ex = g.exact != 0;
    const bool lists = g.share_type == MSG_MULTI_PROPORTIONAL || (ex && g.share_type == MSG_MULTI_EQUAL);
    const uint32_t nwin = nblocks(n, 32);
    CU(c->worklist.reserve(((size_t)nwin + 2) * 4));
    CU(c->win.reserve((size_t)nwin * sizeof(WinInfo)));
    sl.ub_lists = sl.ub_ent = 0;
    if (lists) {
        const uint64_t ul = n / 2 + 2, ue = n + 2;
        if (c->csr_lists + c->inflight_lists + ul >= 0xffffffffull || c->csr_ent + c->inflight_ent + ue >= 0xffffffffull) return MSG_OK;   // general path reports the overflow
        if ((c->csr_lists + c->inflight_lists + ul) * 4 > c->csr_off.cap || (c->csr_ent + c->inflight_ent + ue) * 4 > c->csr_fid.cap || !c->csr_off.p) {
            // growing the list storage copies the lists written so far: the counts of the chunks in flight must be known first
            int rc = wait_all(c); if (rc) return rc;
            CU(c->csr_off.reserve_keep((c->csr_lists + ul) * 4, c->csr_lists * 4, c->stream));
            CU(c->csr_len.reserve_keep((c->csr_lists + ul) * 4, c->csr_lists * 4, c->stream));
            CU(c->csr_fid.reserve_keep((c->csr_ent + ue) * 4, c->csr_ent * 4, c->stream));
        }
        if (ex && (c->csr_lists + c->inflight_lists + ul) * 8 > c->csr_key.cap) {
            int rc = wait_all(c); if (rc) return rc;
            CU(c->csr_key.reserve_keep((c->csr_lists + ul) * 8, c->csr_lists * 8, c->stream));
        }
        sl.ub_lists = ul; sl.ub_ent = ue;
    }
    if (c->cursor_dirty) {
        const uint32_t cur[2] = {(uint32_t)c->csr_lists, (uint32_t)c->csr_ent};
        memcpy(c->h_pin + 80, cur, 8);                                           // pinned: the async copy reads it later
        CU(cudaMemcpyAsync(c->d_cursor, c->h_pin + 80, 8, cudaMemcpyHostToDevice, c->stream));
        c->cursor_dirty = false;
    }
    CU(cudaMemcpyAsync(c->d_cursor + 2, c->d_cursor, 8, cudaMemcpyDeviceToDevice, c->stream));   // where the cursors go back to if the guard trips
    CU(cudaMemsetAsync(c->d_fcnt, 0, 32, c->stream));
    CU(cudaMemsetAsync(c->d_wl, 0, 4, c->stream));
    FusedParams p;
    p.fb = dp.fb; p.score = dp.score; p.tid = dp.tid; p.hash = dp.hash;
    p.fmap = c->d_fmap; p.n_targets = g.n_targets; p.n_features = g.n_features; p.n = n;
    p.uniq = g.hit_mode == MSG_HIT_UNIQUE; p.share_type = g.share_type;
    p.ui = c->d_ui_tmp; p.d = c->d_d_tmp; p.cnt = c->d_fcnt; p.cursor = c->d_cursor;
    p.l_start = c->csr_off.as<uint32_t>(); p.l_len = c->csr_len.as<uint32_t>(); p.l_fid = c->csr_fid.as<int32_t>();
    p.worklist = c->worklist.as<uint32_t>(); p.wl_count = c->d_wl; p.win = c->win.as<WinInfo>();
    p.big_threshold = 1024; p.err = c->d_err;
    p.l_key = c->csr_key.as<unsigned long long>(); p.key_base = sl.key_base;
    const bool sh = (uint32_t)g.n_features <= 4096u;
    auto warp = sh ? (ex ? fused_warp_kernel<true, true> : fused_warp_kernel<true, false>) : (ex ? fused_warp_kernel<false, true> : fused_warp_kernel<false, false>);
    warp<<<nblocks(n, 256), 256, sh ? (size_t)g.n_features * 4 : 0, c->stream>>>(p); LAUNCHED(c);
    (ex ? fused_walk_kernel<true> : fused_walk_kernel<false>)<<<std::min<uint32_t>(nblocks(nwin, 128), 148u * 8u), 128, 0, c->stream>>>(p); LAUNCHED(c);
    fused_guard_kernel<<<nblocks(nwin, 256), 256, 0, c->stream>>>(p.win, nwin, c->d_fcnt + 3); LAUNCHED(c);
    const size_t F = (size_t)(g.n_features > 0 ? g.n_features : 1);
    fused_commit_kernel<<<nblocks(F < 3 ? 3 : F, 256), 256, 0, c->stream>>>(c->d_ui, c->d_d, c->d_ui_tmp, c->d_d_tmp, (uint32_t)g.n_features,
                                                                           g.share_type == MSG_MULTI_EQUAL, c->d_counters, c->d_fcnt, c->d_cursor); LAUNCHED(c);
    uint32_t *h = sl.h_res;
    CU(cudaMemcpyAsync(h, c->d_fcnt, 20, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(h + 5, c->d_cursor, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(h + 8, c->d_err, 8, cudaMemcpyDeviceToHost, c->stream));
    c->inflight_lists += sl.ub_lists; c->inflight_ent += sl.ub_ent;
    *queued = true;
    return MSG_OK;
}

// Pick the decode kernel's window split from the sizes of the chunk's first records: head window
// covers 36 + qname (+ cigar) for ~98 % of them, tail window their aux block.  h_raw/h_off may be
// null (device-resident chunk): the sample is then copied back once per context.
int probe_layout(msg_ctx *c, const uint8_t *h_raw, const uint64_t *h_off, const uint8_t *d_raw, const uint64_t *d_off,
                 uint64_t nbytes, uint64_t n, bool need_cigar, bool need_aux)
{
    const uint64_t S = n < 4096 ? n : 4096;
    std::vector<uint64_t> offv; std::vector<uint8_t> rawv;
    if (!h_raw) {
        if (c->lay_lpr) return MSG_OK;                       // keep the first decision for resident chunks
        offv.resize(S + 1);
        CU(cudaMemcpyAsync(offv.data(), d_off, (S + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        uint64_t span = offv[S] <= nbytes ? offv[S] : nbytes;
        rawv.resize(span + 1);
        CU(cudaMemcpyAsync(rawv.data(), d_raw, span, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->d2h_bytes += span + (S + 1) * 8;
        h_raw = rawv.data(); h_off = offv.data();
    }
    std::vector<uint32_t> heads, auxs;
    heads.reserve(S); auxs.reserve(S);
    for (uint64_t k = 0; k < S; k++) {
        const uint64_t o = h_off[k], len = h_off[k + 1] - o;
        if (len < 36 || o + len > nbytes) continue;
        const uint8_t *r = h_raw + o;
        uint32_t lq = r[12], nc = (uint32_t)r[16] | (uint32_t)r[17] << 8;
        int32_t ls = (int32_t)((uint32_t)r[20] | (uint32_t)r[21] << 8 | (uint32_t)r[22] << 16 | (uint32_t)r[23] << 24);
        if (ls < 0) continue;
        uint64_t ao = 36ull + lq + 4ull * nc + (((uint64_t)ls + 1) >> 1) + (uint64_t)ls;
        if (ao > len) continue;
        heads.push_back(36 + lq + (need_cigar ? 4 * nc : 0));
        auxs.push_back((uint32_t)(len - ao));
    }
    uint32_t hc = 4, tc = need_aux ? 2 : 0;
    if (!heads.empty()) {
        std::sort(heads.begin(), heads.end()); std::sort(auxs.begin(), auxs.end());
        const size_t q = (heads.size() * 98) / 100 < heads.size() ? (heads.size() * 98) / 100 : heads.size() - 1;
        hc = (15 + heads[q] + 15) / 16;
        tc = need_aux ? (auxs[q] + 15 + 15) / 16 : 0;
    }
    if (hc < 4) hc = 4;
    uint32_t lpr = hc + tc <= 8 ? 8 : 16;
    if (hc + tc > 16) { if (hc > 12) hc = 12; tc = 16 - hc; }
    c->lay_lpr = lpr; c->lay_hc = hc; c->lay_tc = tc;
    return MSG_OK;
}

// Decode + filter statistics of one chunk: reserves the SoA columns, picks the window layout, launches decode_kernel.
int launch_decode(msg_ctx *c, const uint8_t *d_raw, uint64_t nbytes, uint64_t readable, const uint64_t *d_off, uint64_t n,
                  const uint8_t *h_raw, const uint64_t *h_off, DecodeParams *out, bool host_mapped = false)
{
    const msg_config &g = c->cfg;
    const bool hit = g.do_filter && g.hit_mode != MSG_HIT_NONE;
    const bool need_score = hit || g.want_stats || (g.do_filter && g.rescore && g.want_records);
    CU(c->tid.reserve(n * 4)); CU(c->fb.reserve(n * 4));
    if (need_score) CU(c->score.reserve(n * 4));
    if (g.want_profile) CU(c->hash.reserve(n * 4));
    if (g.want_stats) { CU(c->st_alen.reserve(n * 4)); CU(c->st_qlen.reserve(n * 4)); CU(c->st_qclip.reserve(n * 4)); CU(c->st_edit.reserve(n * 4)); }

    DecodeParams p;
    memset(&p, 0, sizeof p);
    p.raw = d_raw; p.off = d_off; p.n = n; p.nbytes = nbytes; p.nbytes_readable = readable;
    p.tid = c->tid.as<int32_t>(); p.fb = c->fb.as<uint32_t>();
    p.score = need_score ? c->score.as<int32_t>() : nullptr;
    p.hash = g.want_profile ? c->hash.as<uint32_t>() : nullptr;
    if (g.want_stats) { p.alen = c->st_alen.as<int32_t>(); p.qlen = c->st_qlen.as<int32_t>(); p.qclip = c->st_qclip.as<int32_t>(); p.edit = c->st_edit.as<int32_t>(); }
    p.min_length = g.min_length; p.ppt = g.ppt; p.max_clip = g.max_clip;
    uint32_t mode = c->decode_mode;
    const bool need_stats = c->need_stats || g.want_stats;
    if (need_stats) mode |= DM_NEED_STATS;
    if (c->need_stats) mode |= DM_REQ_STATS;
    if (need_stats || c->cov_fused) mode |= DM_NEED_CIGAR;
    if (need_stats || (need_score && !(g.do_filter && g.rescore))) mode |= DM_NEED_AUX;
    p.mode = mode;
    p.covbits = c->d_covbits; p.covsum = reinterpret_cast<unsigned long long *>(c->d_sum);
    p.diff = c->d_diff; p.covbase = c->d_covbase; p.tlen = c->d_tlen; p.covered = c->d_covered; p.n_targets = g.n_targets;
    p.err = c->d_err; p.acct = c->d_acct;

    { int prc = probe_layout(c, h_raw, h_off, d_raw, d_off, nbytes, n, (mode & DM_NEED_CIGAR) != 0, (mode & DM_NEED_AUX) != 0); if (prc) return prc; }
    p.head_chunks = c->lay_hc; p.tail_chunks = c->lay_tc;
    cudaEvent_t k0 = get_event(c), k1 = get_event(c);
    CU(cudaEventRecord(k0, c->stream));
    // L2 fill granularity of the window loads: 64-byte granules (.L2::64B) or whole 128-byte lines.  MSG_L2_GRANULE=64|128 overrides.
    static const int g_env = getenv("MSG_L2_GRANULE") ? atoi(getenv("MSG_L2_GRANULE")) : 0;
    const bool g64 = g_env ? g_env == 64 : true;
    // staging: register-staged 16-byte loads + STS.128 by default.  LDGSTS (cp.async) measured the same on device-resident
    // chunks of a single GPU (0.4172 vs 0.4190 ms), HALF the rate on chunks decoded in place from pinned host memory, and every
    // 8-rank run that used it had about half of the ranks -- a different set each time -- running each decode launch in 0.689 ms
    // instead of 0.420 ms while all their other kernels kept their times (profiles/r02/scale8/README.md); round 1's 8-rank runs,
    // which staged through registers, did not.  MSG_STAGING=async selects LDGSTS.
    static const char *st_env = getenv("MSG_STAGING");
    const bool async = st_env ? st_env[0] == 'a' : false;
    (void)host_mapped;
    const dim3 grid(nblocks(n, DEC_R)), block(DEC_R);
#define DEC_LAUNCH(L, G, A) decode_kernel<L, G, A><<<grid, block, 0, c->stream>>>(p)
    if (c->lay_lpr == 8) { if (g64) { if (async) DEC_LAUNCH(8, true, true); else DEC_LAUNCH(8, true, false); } else { if (async) DEC_LAUNCH(8, false, true); else DEC_LAUNCH(8, false, false); } }
    else                 { if (g64) { if (async) DEC_LAUNCH(16, true, true); else DEC_LAUNCH(16, true, false); } else { if (async) DEC_LAUNCH(16, false, true); else DEC_LAUNCH(16, false, false); } }
#undef DEC_LAUNCH
    LAUNCHED(c);
    CU(cudaEventRecord(k1, c->stream));
    c->ev_decode.push_back({k0, k1});
    *out = p;
    return MSG_OK;
}

int chunk_args_ok(msg_ctx *c, uint64_t nbytes, uint64_t n)
{
    if (n >= 0xffffffffull) return fail(c, MSG_EINVAL, "a chunk may hold at most 2^32-2 records");
    if (nbytes >= (1ull << 36)) return fail(c, MSG_EINVAL, "a chunk may hold at most 64 GiB of records");
    return MSG_OK;
}

// The general pipeline, synchronous: decode -> stream of kept records in reference output order -> profile / coverage /
// record output.  d_raw must be device memory (later kernels read whole records).  Every configuration can take it; the
// fused pass (fused_enqueue) is the fast path for filter --besthit|--uniqhit | profile.
int run_chunk_general(msg_ctx *c, const uint8_t *d_raw, uint64_t nbytes, uint64_t readable, const uint64_t *d_off, uint64_t n,
                      const uint8_t *h_raw = nullptr, const uint64_t *h_off = nullptr)
{
    const msg_config &g = c->cfg;
    { int rc0 = chunk_args_ok(c, nbytes, n); if (rc0) return rc0; }
    c->cur_raw = d_raw; c->cur_off = d_off; c->cur_n = n; c->cur_nbytes = nbytes;
    c->n_kept = 0; c->have_stream = false; c->out_bytes = 0;
    if (n == 0) return MSG_OK;

    cudaEvent_t t0 = get_event(c), t1 = get_event(c);
    CU(cudaEventRecord(t0, c->stream));
    DecodeParams p;
    int rc = launch_decode(c, d_raw, nbytes, readable, d_off, n, h_raw, h_off, &p);
    if (rc) return rc;
    // the kernels below follow rec_off[] into the record bytes: a malformed index must be reported before they run
    rc = check_device_errors(c);
    if (rc) return rc;

    const bool hit = g.do_filter && g.hit_mode != MSG_HIT_NONE;
    // ---- filter stage -> stream of kept records in reference output order
    const uint32_t *stream = nullptr; uint64_t m = n;
    if (g.do_filter) {
        CU(c->out_idx.reserve(n * 4));
        uint32_t tot = 0;
        if (!hit) {
            rc = run_scan<uint32_t>(c, InFlagBit{p.fb, FB_INPOOL, FB_INPOOL}, OutCompact{c->out_idx.as<uint32_t>()}, n, &tot);
            if (rc) return rc;
        } else {
            CU(c->kbase.reserve(n * 4)); CU(c->worklist.reserve((n / 32 + 2) * 4));
            CU(cudaMemsetAsync(c->d_wl, 0, 4, c->stream));
            BestHitParams bp{p.fb, p.score, n, g.hit_mode == MSG_HIT_UNIQUE, c->d_err, c->worklist.as<uint32_t>(), c->d_wl};
            const uint32_t wgrid = std::min<uint32_t>(nblocks(n / 32 + 1, 256), 148u * 4u);
            besthit_warp_select_kernel<<<nblocks(n, 256), 256, 0, c->stream>>>(bp); LAUNCHED(c);
            besthit_walk_select_kernel<<<wgrid, 256, 0, c->stream>>>(bp); LAUNCHED(c);
            rc = run_scan<uint32_t>(c, InFlagBit{p.fb, FB_KEEP, FB_KEEP}, OutExclU32{c->kbase.as<uint32_t>()}, n, &tot);
            if (rc) return rc;
            besthit_warp_emit_kernel<<<nblocks(n, 256), 256, 0, c->stream>>>(p.fb, c->kbase.as<uint32_t>(), c->out_idx.as<uint32_t>(), n); LAUNCHED(c);
            besthit_walk_emit_kernel<<<wgrid, 256, 0, c->stream>>>(p.fb, c->kbase.as<uint32_t>(), c->out_idx.as<uint32_t>(), n,
                                                                   c->worklist.as<uint32_t>(), c->d_wl); LAUNCHED(c);
        }
        stream = c->out_idx.as<uint32_t>(); m = tot; c->have_stream = true;
    }
    c->n_kept = m;

    if (g.want_profile) { rc = profile_stage(c, stream, m); if (rc) return rc; c->cursor_dirty = true; }
    if (g.want_coverage && !c->cov_fused && m) {
        coverage_stream_kernel<<<nblocks(m, 256), 256, 0, c->stream>>>(d_raw, d_off, stream, m, g.n_targets, c->d_diff, c->d_covbase,
                                                                      c->d_tlen, c->d_covered, c->d_err,
                                                                      c->cov_bits ? c->d_covbits : nullptr, reinterpret_cast<unsigned long long *>(c->d_sum)); LAUNCHED(c);
        c->cov_finished = false;
    }
    if (g.want_coverage) c->cov_finished = false;
    if (g.want_records) { rc = records_stage(c, stream, m); if (rc) return rc; }

    CU(cudaEventRecord(t1, c->stream));
    c->ev_total.push_back({t0, t1});
    return check_device_errors(c);
}

// Finish the chunk in flight in slot s: wait for its kernels, read its results out of the pinned block, report its
// errors; if the fused guard declined it, rerun it on the general pipeline (after the other chunk in flight, so that
// the host's list cursors are current).
int complete_slot(msg_ctx *c, int s)
{
    Slot &sl = c->slot[s];
    if (!sl.pending) return MSG_OK;
    CU(cudaEventSynchronize(sl.done));
    sl.pending = false;
    c->inflight_lists -= sl.ub_lists; c->inflight_ent -= sl.ub_ent;
    const uint32_t *h = sl.h_res;
    c->d2h_bytes += 36;
    c->fused_chunks++;
    c->cur_raw = sl.d_raw; c->cur_off = sl.d_off; c->cur_n = sl.n; c->cur_nbytes = sl.nbytes;
    c->out_bytes = 0;
    { int erc = report_device_errors(c, h + 8); if (erc) return erc; }
    if (!h[3]) {
        c->csr_lists = h[5]; c->csr_ent = h[6];
        c->n_kept = h[4]; c->have_stream = false;
        return MSG_OK;
    }
    // guard tripped: fused_commit_kernel dropped this chunk's partial sums and put the list cursors back
    c->fused_fallbacks++;
    int rc = complete_slot(c, s ^ 1);
    if (rc) return rc;
    const uint8_t *d_raw = sl.d_raw; uint64_t readable = sl.readable;
    if (sl.zero_copy) {                              // the kernels of the general pipeline re-read whole records: stage them
        CU(sl.raw.reserve(sl.nbytes + 64));
        CU(cudaMemcpyAsync(sl.raw.p, sl.h_raw, sl.nbytes, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemsetAsync((uint8_t *)sl.raw.p + sl.nbytes, 0, 64, c->stream));
        c->h2d_bytes += sl.nbytes;
        d_raw = sl.raw.as<uint8_t>(); readable = sl.nbytes + 64;
    }
    c->cur_key_base = sl.key_base;                   // the rerun's lists take the declined chunk's keys
    return run_chunk_general(c, d_raw, sl.nbytes, readable, sl.d_off, sl.n, sl.h_raw, sl.h_off);
}

int wait_all(msg_ctx *c)
{
    int rc = complete_slot(c, c->next_slot);         // older chunk first
    int rc2 = complete_slot(c, c->next_slot ^ 1);
    return rc ? rc : rc2;
}

// Queue one chunk.  Host chunks (h_raw != NULL) are staged into the slot's device buffers on the copy stream, or -- pinned,
// mapped, 16-byte aligned buffers -- decoded in place over PCIe (zero-copy windows); device chunks are used where they are.
// Configurations outside the fused pass complete the chunk before returning.
int push_chunk(msg_ctx *c, const uint8_t *h_raw, const uint8_t *dev_raw, size_t nbytes, const uint64_t *h_off, const uint64_t *dev_off, size_t nrec)
{
    const msg_config &g = c->cfg;
    { int rc0 = chunk_args_ok(c, nbytes, nrec); if (rc0) return rc0; }
    if (nrec == 0) { int rc = wait_all(c); c->cur_n = 0; c->n_kept = 0; c->out_bytes = 0; return rc; }
    const bool fused = c->fused_enabled && g.want_profile;
    const int s = c->next_slot;
    int rc = fused ? complete_slot(c, s) : wait_all(c);          // the chunk pushed two calls ago / everything
    if (rc) return rc;
    Slot &sl = c->slot[fused ? s : 0];
    sl.h_raw = h_raw; sl.h_off = h_off; sl.nbytes = nbytes; sl.n = nrec; sl.zero_copy = false;
    sl.key_base = c->rec_base; c->rec_base += nrec;     // chunks complete in push order, so this is their input position
    c->ex_ready = false;

    cudaEvent_t t0 = get_event(c), t1 = get_event(c);
    if (dev_raw) {
        sl.d_raw = dev_raw; sl.d_off = dev_off; sl.readable = nbytes & ~(size_t)15;          // never read past the caller's nbytes
        CU(cudaEventRecord(t0, c->stream));
    } else {
        CU(sl.off.reserve((nrec + 1) * 8));
        sl.d_off = sl.off.as<uint64_t>();
        // Pinned (mapped) host buffer + fused pass: do not copy the chunk at all.  The decode kernel reads its head / tail
        // windows straight from host memory, so only ~55 % of the BAM bytes cross PCIe (64-byte granules around the
        // windows; SEQ/QUAL stay on the host).  MSG_ZERO_COPY=0 forces the staged copy.
        static const bool zc_allowed = !(getenv("MSG_ZERO_COPY") && atoi(getenv("MSG_ZERO_COPY")) == 0);
        cudaPointerAttributes at;
        if (zc_allowed && fused && !((uintptr_t)h_raw & 15u) && cudaPointerGetAttributes(&at, h_raw) == cudaSuccess &&
            at.type == cudaMemoryTypeHost && at.devicePointer) {
            sl.zero_copy = true;
            sl.d_raw = static_cast<const uint8_t *>(at.devicePointer); sl.readable = nbytes & ~(size_t)15;
            CU(cudaEventRecord(t0, c->stream));
            CU(cudaMemcpyAsync(sl.off.p, h_off, (nrec + 1) * 8, cudaMemcpyHostToDevice, c->stream));
            c->h2d_bytes += (nrec + 1) * 8;
            c->zc_chunks++;
        } else {
            cudaGetLastError();
            CU(sl.raw.reserve(nbytes + 64));
            sl.d_raw = sl.raw.as<uint8_t>(); sl.readable = nbytes + 64;
            // the copy stream fills this slot while the previous chunk's kernels run on the main stream
            cudaStream_t cs = fused ? c->copy_stream : c->stream;
            CU(cudaEventRecord(t0, cs));
            CU(cudaMemcpyAsync(sl.raw.p, h_raw, nbytes, cudaMemcpyHostToDevice, cs));
            CU(cudaMemsetAsync((uint8_t *)sl.raw.p + nbytes, 0, 64, cs));
            CU(cudaMemcpyAsync(sl.off.p, h_off, (nrec + 1) * 8, cudaMemcpyHostToDevice, cs));
            if (fused) { CU(cudaEventRecord(sl.copied, cs)); CU(cudaStreamWaitEvent(c->stream, sl.copied, 0)); }
            c->h2d_bytes += nbytes + (nrec + 1) * 8;
        }
    }
    if (fused) {
        DecodeParams p;
        const uint64_t before = c->h2d_bytes;
        rc = launch_decode(c, sl.d_raw, nbytes, sl.readable, sl.d_off, nrec, h_raw, h_off, &p, sl.zero_copy);
        if (rc) return rc;
        // bytes the decode kernel asks for over PCIe (window chunks)
        if (sl.zero_copy && c->h2d_bytes == before) c->h2d_bytes += (uint64_t)nrec * (c->lay_hc + c->lay_tc) * 16;
        bool queued = false;
        rc = fused_enqueue(c, p, nrec, sl, &queued);
        if (rc) return rc;
        if (queued) {
            CU(cudaEventRecord(t1, c->stream));
            CU(cudaEventRecord(sl.done, c->stream));
            c->ev_total.push_back({t0, t1});
            sl.pending = true;
            c->next_slot = s ^ 1;
            return MSG_OK;
        }
        rc = wait_all(c);
        if (rc) return rc;
    }
    c->ev_free.push_back(t0); c->ev_free.push_back(t1);
    const uint8_t *d_raw = sl.d_raw; uint64_t readable = sl.readable;
    if (sl.zero_copy) {
        CU(sl.raw.reserve(nbytes + 64));
        CU(cudaMemcpyAsync(sl.raw.p, h_raw, nbytes, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemsetAsync((uint8_t *)sl.raw.p + nbytes, 0, 64, c->stream));
        c->h2d_bytes += nbytes;
        d_raw = sl.raw.as<uint8_t>(); readable = nbytes + 64;
    }
    c->cur_key_base = sl.key_base;
    return run_chunk_general(c, d_raw, nbytes, readable, sl.d_off, nrec, h_raw, h_off);
}

// ------------------------------------------------------------------------------------------------ collation (collate.cuh)
// MSG_COLLATE_HASH_BITS=k keeps the top k bits of the 64-bit QNAME hash, so that tests can reach the collision path.
unsigned long long coll_hash_mask()
{
    static const int bits = getenv("MSG_COLLATE_HASH_BITS") ? atoi(getenv("MSG_COLLATE_HASH_BITS")) : 64;
    return bits >= 64 || bits < 1 ? ~0ull : ~0ull << (64 - bits);
}

int coll_grow(msg_ctx *c, DevBuf &b, size_t bytes, size_t keep, uint64_t nrec, uint64_t head_bytes)
{
    if (bytes <= b.cap && b.p) return MSG_OK;
    size_t free_b = 0, total_b = 0;
    cudaError_t e = cudaMemGetInfo(&free_b, &total_b);
    if (e == cudaSuccess) e = bytes + bytes / 2 + 256 <= free_b ? b.reserve_keep(bytes, keep, c->stream) : cudaErrorMemoryAllocation;
    if (e == cudaSuccess) return MSG_OK;
    cudaGetLastError();
    return fail(c, e == cudaErrorMemoryAllocation ? MSG_ENOMEM : MSG_ECUDA,
                "cannot hold %llu records (%llu bytes of record heads) for collation in device memory (%zu bytes free): %s",
                (unsigned long long)nrec, (unsigned long long)head_bytes, free_b, cudaGetErrorString(e));
}

// A push on a collating context: append the chunk's record heads and keys to the scope (msg_config.collate).
int collate_push(msg_ctx *c, const uint8_t *h_raw, const uint8_t *dev_raw, size_t nbytes, const uint64_t *h_off, const uint64_t *dev_off, size_t nrec)
{
    { int rc0 = chunk_args_ok(c, nbytes, nrec); if (rc0) return rc0; }
    if (c->coll_done) { c->coll_n = 0; c->coll_bytes = 0; c->coll_done = false; }
    if (nrec == 0) return MSG_OK;
    if (c->coll_n + nrec > 0xfffffffeull)
        return fail(c, MSG_ERANGE, "collation holds at most 2^32-2 records per scope (%llu held, %zu pushed)", (unsigned long long)c->coll_n, nrec);
    Slot &sl = c->slot[0];
    const uint8_t *src = dev_raw; const uint64_t *offp = dev_off;
    if (!dev_raw) {
        CU(sl.off.reserve((nrec + 1) * 8));
        CU(cudaMemcpyAsync(sl.off.p, h_off, (nrec + 1) * 8, cudaMemcpyHostToDevice, c->stream));
        offp = sl.off.as<uint64_t>();
        c->h2d_bytes += (nrec + 1) * 8;
        // pinned, mapped host memory is read in place (only the heads and aux blocks cross PCIe); anything else is staged
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, h_raw) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
            src = static_cast<const uint8_t *>(at.devicePointer);
            c->zc_chunks++;
        } else {
            cudaGetLastError();
            CU(sl.raw.reserve(nbytes + 64));
            CU(cudaMemcpyAsync(sl.raw.p, h_raw, nbytes, cudaMemcpyHostToDevice, c->stream));
            src = sl.raw.as<uint8_t>();
            c->h2d_bytes += nbytes;
        }
    }
    const uint32_t base = (uint32_t)c->coll_n;
    CU(c->coll_len.reserve(nrec * 4));
    collate_size_kernel<<<nblocks(nrec, 256), 256, 0, c->stream>>>(src, offp, nrec, nbytes, base, c->need_stats || c->cov_fused,
                                                                   c->coll_len.as<uint32_t>(), c->d_err); LAUNCHED(c);
    { int rc = check_device_errors(c); if (rc) return rc; }
    const uint64_t n_all = c->coll_n + nrec;
    { int rc = coll_grow(c, c->coll_aoff, (n_all + 1) * 8, (c->coll_n + 1) * 8, n_all, c->coll_bytes); if (rc) return rc; }
    unsigned long long tot = 0;
    unsigned long long *aoff = c->coll_aoff.as<unsigned long long>();
    int rc = run_scan<unsigned long long>(c, InLenU64{c->coll_len.as<uint32_t>()}, OutExclU64Add{aoff + c->coll_n, c->coll_bytes}, nrec, &tot);
    if (rc) return rc;
    const uint64_t bytes_all = c->coll_bytes + tot;
    if (bytes_all >= (1ull << 36))      // the grouped stream is handed to the pipeline with offsets from its start
        return fail(c, MSG_ERANGE, "collation holds at most 64 GiB of record heads per scope (%llu records held)", (unsigned long long)c->coll_n);
    unsigned long long *h_end = reinterpret_cast<unsigned long long *>(c->h_pin + 84);
    *h_end = bytes_all;
    CU(cudaMemcpyAsync(aoff + n_all, h_end, 8, cudaMemcpyHostToDevice, c->stream));
    if ((rc = coll_grow(c, c->coll_arena, bytes_all + 64, c->coll_bytes, n_all, bytes_all))) return rc;
    if ((rc = coll_grow(c, c->coll_keys, n_all * sizeof(CollKey), c->coll_n * sizeof(CollKey), n_all, bytes_all))) return rc;
    collate_gather_kernel<<<std::min<uint32_t>(nblocks(nrec, 8), 148u * 64u), 256, 0, c->stream>>>(src, offp, nrec, aoff + c->coll_n, c->coll_len.as<uint32_t>(),
                                                                  c->coll_arena.as<uint8_t>(), c->coll_keys.as<CollKey>() + c->coll_n, base, coll_hash_mask()); LAUNCHED(c);
    CU(cudaStreamSynchronize(c->stream));             // the caller may reuse its buffers once the push returns
    c->coll_n = n_all; c->coll_bytes = bytes_all; c->coll_dirty = true;
    return MSG_OK;
}

// Largest grouped chunk handed to the pipeline: with at most 2^24 records per chunk no chunk can hold more than the
// profile stage's 65536 groups of > 1024 records.  A single read larger than that is a chunk of its own (one group).
// MSG_COLLATE_CHUNK_RECORDS=C (clamped to [1, 2^24]) lowers the limit, so that tests reach every cut with few records.
uint64_t coll_chunk_records()
{
    static const long long env = getenv("MSG_COLLATE_CHUNK_RECORDS") ? atoll(getenv("MSG_COLLATE_CHUNK_RECORDS")) : 1ll << 24;
    return (uint64_t)std::min<long long>(std::max<long long>(env, 1), 1ll << 24);
}

bool coll_across_ranks(const msg_ctx *c) { return c->cfg.collate == MSG_COLLATE_RANKS && c->cfg.n_ranks > 1; }

// Group everything held by QNAME and run the pipeline over it once.
int collate_local(msg_ctx *c)
{
    const uint64_t n = c->coll_n;
    if (n == 0) return MSG_OK;
    static const bool trace = getenv("MSG_TRACE_FINISH") != nullptr;
    cudaEvent_t tev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    auto tmark = [&](int k) { if (trace) { cudaEventCreate(&tev[k]); cudaEventRecord(tev[k], c->stream); } };
    tmark(0);
    const unsigned long long *aoff = c->coll_aoff.as<unsigned long long>();
    const uint8_t *arena = c->coll_arena.as<uint8_t>();
    int rc;
    // ---- partition by the top bits of the hash
    uint32_t bits = 0;
    while (bits < 24 && ((uint64_t)COLL_BUCKET_AVG << bits) < n) bits++;
    if (coll_across_ranks(c)) {
        // this rank holds 1/N of the hash space: ceil(log2 N) more bits keep its occupied buckets near COLL_BUCKET_AVG keys
        uint32_t lg = 0;
        while ((1u << lg) < (uint32_t)c->cfg.n_ranks) lg++;
        bits = std::min<uint32_t>(24, bits + lg);
    }
    const uint32_t nb = 1u << bits;
    if ((rc = coll_grow(c, c->coll_keys2, n * sizeof(CollKey), 0, n, c->coll_bytes))) return rc;
    CU(c->coll_hist.reserve((size_t)nb * 4)); CU(c->coll_bstart.reserve((size_t)nb * 4));
    CU(c->coll_list.reserve((size_t)nb * 4 + 8));
    uint32_t *hist = c->coll_hist.as<uint32_t>(), *bstart = c->coll_bstart.as<uint32_t>();
    CollKey *keys = c->coll_keys2.as<CollKey>();
    CU(cudaMemsetAsync(hist, 0, (size_t)nb * 4, c->stream));
    collate_hist_kernel<<<nblocks(n, 256), 256, 0, c->stream>>>(c->coll_keys.as<CollKey>(), n, bits, hist); LAUNCHED(c);
    if ((rc = run_scan<uint32_t>(c, InU32{hist}, OutExclU32{bstart}, nb, (uint32_t *)nullptr))) return rc;
    CU(cudaMemcpyAsync(hist, bstart, (size_t)nb * 4, cudaMemcpyDeviceToDevice, c->stream));
    collate_scatter_kernel<<<nblocks(n, 256), 256, 0, c->stream>>>(c->coll_keys.as<CollKey>(), n, bits, hist, keys); LAUNCHED(c);
    tmark(1);
    // ---- sort every bucket by (hash, ordinal)
    uint32_t *big = c->coll_list.as<uint32_t>(), *cnt = reinterpret_cast<uint32_t *>(c->d_total);
    CU(cudaMemsetAsync(cnt, 0, 4, c->stream));
    collate_bucket_sort_kernel<<<std::min<uint32_t>(nb, 148u * 8u), 256, 0, c->stream>>>(keys, bstart, nb, n, big, cnt); LAUNCHED(c);
    uint32_t *h_cnt = c->h_pin + 88;
    CU(cudaMemcpyAsync(h_cnt, cnt, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (*h_cnt) { collate_sort_global_kernel<<<*h_cnt, 1024, 0, c->stream>>>(keys, bstart, nb, n, big, false, arena, aoff); LAUNCHED(c); }
    // ---- runs of one hash that hold different names: sort them by (name bytes, ordinal).  Rare (64-bit hash).
    for (;;) {
        const uint32_t cap = (uint32_t)(c->coll_list.cap / 8);
        CU(cudaMemsetAsync(cnt, 0, 4, c->stream));
        collate_collide_kernel<<<nblocks(n, 256), 256, 0, c->stream>>>(keys, n, arena, aoff, c->coll_list.as<uint32_t>(), cap, cnt); LAUNCHED(c);
        CU(cudaMemcpyAsync(h_cnt, cnt, 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (*h_cnt <= cap) break;
        CU(c->coll_list.reserve((size_t)*h_cnt * 8));
    }
    if (*h_cnt) { collate_sort_global_kernel<<<*h_cnt, 1024, 0, c->stream>>>(keys, bstart, nb, n, c->coll_list.as<uint32_t>(), true, arena, aoff); LAUNCHED(c); }
    tmark(2);
    // ---- heads in grouped order; keys[g].ord maps a grouped position back to its input ordinal
    unsigned long long tot = 0;
    if ((rc = coll_grow(c, c->coll_goff, (n + 1) * 8, 0, n, c->coll_bytes))) return rc;
    unsigned long long *goff = c->coll_goff.as<unsigned long long>();
    if ((rc = run_scan<unsigned long long>(c, InGroupedLen{keys, aoff}, OutExclU64{goff}, n, &tot))) return rc;
    unsigned long long *h_end = reinterpret_cast<unsigned long long *>(c->h_pin + 84);
    *h_end = tot;
    CU(cudaMemcpyAsync(goff + n, h_end, 8, cudaMemcpyHostToDevice, c->stream));
    if ((rc = coll_grow(c, c->coll_grouped, tot + 64, 0, n, tot))) return rc;
    collate_grouped_gather_kernel<<<std::min<uint32_t>(nblocks(n, 8), 148u * 64u), 256, 0, c->stream>>>(keys, n, arena, aoff, goff, c->coll_grouped.as<uint8_t>()); LAUNCHED(c);
    tmark(3);
    // ---- the pipeline, one device chunk at a time.  Chunks are cut where the hash changes, which is a group start; any
    // group start is a safe cut here because every name occurs in exactly one run of the grouped stream, so no pool or
    // profile group can continue across it (the record before a cut can never share the next record's name, whatever
    // its flags or tid).  The chunk's index holds absolute offsets into the grouped arena.
    unsigned long long *dcut = reinterpret_cast<unsigned long long *>(c->d_total);
    unsigned long long *h_cut = reinterpret_cast<unsigned long long *>(c->h_pin + 92);
    std::vector<unsigned long long> hgo(1);
    const uint64_t C = coll_chunk_records();
    for (uint64_t lo = 0; lo < n;) {
        uint64_t hi = n;
        if (n - lo > C) {
            // the last run start in (lo, lo + C]; else (one read of more than C records) the first one after lo + C,
            // searched in windows that double until one is found or n is reached
            const uint64_t want = lo + C;
            uint64_t from = lo, end = std::min<uint64_t>(n, want + C + 1), step = C;
            for (;;) {
                const unsigned long long init[2] = {0ull, ~0ull};
                memcpy(h_cut, init, 16);
                CU(cudaMemcpyAsync(dcut, h_cut, 16, cudaMemcpyHostToDevice, c->stream));
                collate_cut_kernel<<<nblocks(end - from - 1, 256), 256, 0, c->stream>>>(keys, from, want, end, dcut, dcut + 1); LAUNCHED(c);
                CU(cudaMemcpyAsync(h_cut, dcut, 16, cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                if (h_cut[0] || h_cut[1] != ~0ull || end == n) break;
                from = end - 1; step *= 2; end = std::min<uint64_t>(n, end + step);
            }
            hi = h_cut[0] ? h_cut[0] : h_cut[1] != ~0ull ? h_cut[1] : n;
        }
        CU(cudaMemcpyAsync(hgo.data(), goff + hi, 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        // Groups come in hash order rather than input order.  Per read, the filter, best-hit and uniq-hit selection (a set
        // per mate class) and insert counting only see that read's records, which keep their input order; across reads,
        // the order changes only the order of the multi-mapper lists, i.e. the summation order of the f64 PropSharing
        // sums, which the f64 atomics already vary.  So every integer result equals that of the input regrouped stably
        // by QNAME, and every f64 result equals it up to rounding.
        rc = push_chunk(c, nullptr, c->coll_grouped.as<uint8_t>(), hgo[0], nullptr, reinterpret_cast<const uint64_t *>(goff + lo), hi - lo);
        if (!rc) rc = wait_all(c);
        if (rc) {
            // errors found after grouping name the record's input ordinal, not its grouped position
            if ((rc == MSG_ENOTAG || rc == MSG_ENOAS || rc == MSG_EFORMAT) && c->err_rec != 0xffffffffu && lo + c->err_rec < n) {
                CollKey k;
                uint32_t G = 0;
                if (cudaMemcpy(&k, keys + lo + c->err_rec, sizeof k, cudaMemcpyDeviceToHost) != cudaSuccess) {}
                else if (!coll_across_ranks(c)) c->err += " (input record " + std::to_string(k.ord) + ")";
                else if (cudaMemcpy(&G, c->coll_len.as<uint32_t>() + k.ord, 4, cudaMemcpyDeviceToHost) == cudaSuccess) {
                    const size_t r = std::upper_bound(c->coll_base.begin(), c->coll_base.end(), (unsigned long long)G) - c->coll_base.begin() - 1;
                    c->err += " (input record " + std::to_string(G) + ": rank " + std::to_string(r) + ", record " +
                              std::to_string(G - c->coll_base[r]) + " of its pushes)";
                }
            }
            return rc;
        }
        lo = hi;
    }
    if (trace) {
        tmark(4); cudaEventSynchronize(tev[4]);
        float ms[4] = {0, 0, 0, 0};
        for (int k = 0; k < 4; k++) cudaEventElapsedTime(&ms[k], tev[k], tev[k + 1]);
        fprintf(stderr, "[msg collate] %llu records, %llu head bytes: partition %.3f ms, sort %.3f ms, grouped gather %.3f ms, pipeline %.3f ms\n",
                (unsigned long long)n, (unsigned long long)tot, ms[0], ms[1], ms[2], ms[3]);
        for (auto e : tev) if (e) cudaEventDestroy(e);
    }
    return MSG_OK;
}

// The sender's half of the exchange: partition this rank's n held keys by destination rank, stably (collate.cuh), into
// coll_keys2 with each head length in the key's pad word, count records and head bytes per destination into row[], and
// gather the heads in that order into coll_grouped.  coll_keys2 and coll_grouped are otherwise only used after the
// exchange, so they are the send buffers.
int collate_send_prep(msg_ctx *c, uint64_t n, unsigned long long *row)
{
    const uint32_t N = (uint32_t)c->cfg.n_ranks, nblk = nblocks(n, COLL_DEST_TILE);
    const unsigned long long *aoff = c->coll_aoff.as<unsigned long long>();
    int rc;
    if ((rc = coll_grow(c, c->coll_keys2, n * sizeof(CollKey), 0, n, c->coll_bytes))) return rc;
    if ((rc = coll_grow(c, c->coll_goff, (n + 1) * 8, 0, n, c->coll_bytes))) return rc;
    CU(c->coll_hist.reserve((size_t)N * nblk * 4)); CU(c->coll_bstart.reserve((size_t)N * nblk * 4));
    uint32_t *cnt = c->coll_hist.as<uint32_t>(), *pos = c->coll_bstart.as<uint32_t>();
    CollKey *keys2 = c->coll_keys2.as<CollKey>();
    collate_dest_count_kernel<<<nblk, 256, 12 * (size_t)N, c->stream>>>(c->coll_keys.as<CollKey>(), n, N, aoff, cnt, nblk, row); LAUNCHED(c);
    if ((rc = run_scan<uint32_t>(c, InU32{cnt}, OutExclU32{pos}, (uint64_t)N * nblk, (uint32_t *)nullptr))) return rc;
    collate_dest_scatter_kernel<<<nblk, 256, 4 * (size_t)N * (256 / 32 + 1), c->stream>>>(c->coll_keys.as<CollKey>(), n, N, aoff, pos, nblk, keys2); LAUNCHED(c);
    unsigned long long *goff = c->coll_goff.as<unsigned long long>(), tot = 0;
    if ((rc = run_scan<unsigned long long>(c, InGroupedLen{keys2, aoff}, OutExclU64{goff}, n, &tot))) return rc;
    if ((rc = coll_grow(c, c->coll_grouped, tot + 64, 0, n, tot))) return rc;
    collate_grouped_gather_kernel<<<std::min<uint32_t>(nblocks(n, 8), 148u * 64u), 256, 0, c->stream>>>(keys2, n, c->coll_arena.as<uint8_t>(), aoff, goff,
                                                                                                         c->coll_grouped.as<uint8_t>()); LAUNCHED(c);
    return MSG_OK;
}

// Collation across ranks (MSG_COLLATE_RANKS, n_ranks > 1; DESIGN.md §11): every rank sends each held record head to rank
// floor(hash * N / 2^64), so that every QNAME ends up on exactly one rank, then collates what it received.  Every
// decision below is taken from data all ranks share (one allgather, one allreduce), so that no rank enters a collective
// its peers skip.  *run: some rank pushed since the last collation.  *sent: the send/recv group was issued; an error
// returned before that is the same on every rank, one after it is not (collate_run_ranks agrees on it).
int collate_exchange(msg_ctx *c, bool *run, bool *sent)
{
    *run = false; *sent = false;
    const uint32_t N = (uint32_t)c->cfg.n_ranks, me = (uint32_t)c->cfg.rank, R = 2 * N + 2;
    // a rank without pushes since the last collation sends nothing: its coll_n still counts what it received then
    const uint64_t n = c->coll_dirty ? c->coll_n : 0;
    static const bool trace = getenv("MSG_TRACE_FINISH") != nullptr;
    cudaEvent_t tev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    auto tmark = [&](int k) { if (trace) { cudaEventCreate(&tev[k]); cudaEventRecord(tev[k], c->stream); } };
    tmark(0);
    // the size matrix: rank s's row is [records, head bytes] for every destination, then {pushed, failed}
    CU(c->coll_xchg.reserve((size_t)N * R * 8 + 16));
    unsigned long long *dm = c->coll_xchg.as<unsigned long long>(), *row = dm + (size_t)me * R;
    int *d_agree = reinterpret_cast<int *>(dm + (size_t)N * R);
    CU(cudaMemsetAsync(row, 0, (size_t)R * 8, c->stream));
    const int prc = n ? collate_send_prep(c, n, row) : MSG_OK;
    cudaGetLastError();
    unsigned long long *h_flags = reinterpret_cast<unsigned long long *>(c->h_pin + 100);
    h_flags[0] = n > 0; h_flags[1] = prc != MSG_OK;
    CU(cudaMemcpyAsync(row + 2 * N, h_flags, 16, cudaMemcpyHostToDevice, c->stream));
    tmark(1);
    NC(g_nccl.AllGather(row, dm, R, ncclUint64, c->comm, c->stream));
    std::vector<unsigned long long> M((size_t)N * R);
    CU(cudaMemcpyAsync(M.data(), dm, M.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    auto rec = [&](uint32_t s, uint32_t d) { return M[(size_t)s * R + 2 * d]; };
    auto byt = [&](uint32_t s, uint32_t d) { return M[(size_t)s * R + 2 * d + 1]; };
    bool any = false; int failed = -1;
    for (uint32_t s = 0; s < N; s++) { any = any || M[(size_t)s * R + 2 * N]; if (failed < 0 && M[(size_t)s * R + 2 * N + 1]) failed = (int)s; }
    if (!any) { for (auto e : tev) if (e) cudaEventDestroy(e); return MSG_OK; }
    *run = true;
    c->coll_dirty = false; c->coll_done = true;
    if (failed >= 0) return prc ? prc : fail(c, MSG_ENOMEM, "collation across ranks: rank %d could not partition its records", failed);
    std::vector<unsigned long long> base(N + 1, 0);
    for (uint32_t s = 0; s < N; s++) { unsigned long long t = 0; for (uint32_t d = 0; d < N; d++) t += rec(s, d); base[s + 1] = base[s] + t; }
    if (base[N] > 0xfffffffeull)                       // input ordinals stay 32-bit
        return fail(c, MSG_ERANGE, "collation across ranks holds at most 2^32-2 records per scope (%llu pushed over %u ranks)", base[N], N);
    unsigned long long rn = 0, rb = 0;
    for (uint32_t d = 0; d < N; d++) {
        unsigned long long b = 0;
        for (uint32_t s = 0; s < N; s++) b += byt(s, d);
        if (b >= (1ull << 36)) return fail(c, MSG_ERANGE, "collation across ranks: rank %u would receive %llu bytes of record heads (at most 64 GiB per rank)", d, b);
        if (d == me) { rb = b; for (uint32_t s = 0; s < N; s++) rn += rec(s, d); }
    }
    // receive buffers: the arena's heads now sit in coll_grouped and the keys in coll_keys2, so the arena, the keys and
    // the head offsets are free (released first where they must grow, so the peak stays that of one-GPU collation)
    int arc = MSG_OK;
    if (rb + 64 > c->coll_arena.cap) c->coll_arena.release();
    if (rn * sizeof(CollKey) > c->coll_keys.cap) c->coll_keys.release();
    if ((rn + 1) * 8 > c->coll_aoff.cap) c->coll_aoff.release();
    arc = coll_grow(c, c->coll_arena, rb + 64, 0, rn, rb);
    if (!arc) arc = coll_grow(c, c->coll_keys, (rn ? rn : 1) * sizeof(CollKey), 0, rn, rb);
    if (!arc) arc = coll_grow(c, c->coll_aoff, (rn + 1) * 8, 0, rn, rb);
    if (!arc && c->coll_len.reserve((rn + 1) * 4) != cudaSuccess) { cudaGetLastError(); arc = fail(c, MSG_ENOMEM, "cannot hold the global ordinals of %llu received records", rn); }
    int *h_agree = reinterpret_cast<int *>(c->h_pin + 104);
    *h_agree = arc ? (int)me : (int)N;
    CU(cudaMemcpyAsync(d_agree, h_agree, 4, cudaMemcpyHostToDevice, c->stream));
    NC(g_nccl.AllReduce(d_agree, d_agree, 1, ncclInt32, ncclMin, c->comm, c->stream));
    CU(cudaMemcpyAsync(h_agree, d_agree, 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (*h_agree < (int)N) return arc ? arc : fail(c, MSG_ENOMEM, "collation across ranks: rank %d lacks device memory for the records it receives", *h_agree);
    if (n) { collate_rebase_kernel<<<nblocks(n, 256), 256, 0, c->stream>>>(c->coll_keys2.as<CollKey>(), n, (uint32_t)base[me]); LAUNCHED(c); }
    tmark(2);
    // ---- the exchange: one send / recv pair per peer for keys and for heads, in one group
    const uint8_t *sk = c->coll_keys2.as<uint8_t>(), *sh = c->coll_grouped.as<uint8_t>();
    uint8_t *rk = c->coll_keys.as<uint8_t>(), *rh = c->coll_arena.as<uint8_t>();
    std::vector<unsigned long long> so(N + 1, 0), sb(N + 1, 0), ro(N + 1, 0), rbo(N + 1, 0);
    for (uint32_t p = 0; p < N; p++) {
        so[p + 1] = so[p] + rec(me, p); sb[p + 1] = sb[p] + byt(me, p);         // send segments, in destination order
        ro[p + 1] = ro[p] + rec(p, me); rbo[p + 1] = rbo[p] + byt(p, me);       // receive segments, in source order
    }
    const size_t K = sizeof(CollKey);
    if (rec(me, me)) {
        CU(cudaMemcpyAsync(rk + ro[me] * K, sk + so[me] * K, rec(me, me) * K, cudaMemcpyDeviceToDevice, c->stream));
        CU(cudaMemcpyAsync(rh + rbo[me], sh + sb[me], byt(me, me), cudaMemcpyDeviceToDevice, c->stream));
    }
    NC(g_nccl.GroupStart());
    for (uint32_t p = 0; p < N; p++) {
        if (p == me) continue;
        if (rec(me, p)) {
            NC(g_nccl.Send(sk + so[p] * K, rec(me, p) * K, ncclUint8, (int)p, c->comm, c->stream));
            NC(g_nccl.Send(sh + sb[p], byt(me, p), ncclUint8, (int)p, c->comm, c->stream));
        }
        if (rec(p, me)) {
            NC(g_nccl.Recv(rk + ro[p] * K, rec(p, me) * K, ncclUint8, (int)p, c->comm, c->stream));
            NC(g_nccl.Recv(rh + rbo[p], byt(p, me), ncclUint8, (int)p, c->comm, c->stream));
        }
    }
    NC(g_nccl.GroupEnd());
    *sent = true;
    tmark(3);
    // ---- what this rank now holds: keys with their receive position as ordinal, head offsets from the carried lengths
    CollKey *keys = c->coll_keys.as<CollKey>();
    unsigned long long *aoff = c->coll_aoff.as<unsigned long long>(), tot = 0;
    if (rn) { collate_recv_kernel<<<nblocks(rn, 256), 256, 0, c->stream>>>(keys, rn, c->coll_len.as<uint32_t>()); LAUNCHED(c); }
    int rc = run_scan<unsigned long long>(c, InKeyPadLen{keys}, OutExclU64{aoff}, rn, &tot);
    if (rc) return rc;
    unsigned long long *h_end = reinterpret_cast<unsigned long long *>(c->h_pin + 84);
    *h_end = tot;
    CU(cudaMemcpyAsync(aoff + rn, h_end, 8, cudaMemcpyHostToDevice, c->stream));
    tmark(4);
    CU(cudaStreamSynchronize(c->stream));
    c->coll_n = rn; c->coll_bytes = tot;
    c->coll_base.assign(base.begin(), base.end());
    if (trace) {
        float ms[4] = {0, 0, 0, 0};
        for (int k = 0; k < 4; k++) cudaEventElapsedTime(&ms[k], tev[k], tev[k + 1]);
        fprintf(stderr, "[msg collate rank %u] exchange: partition + send gather %.3f ms, agree %.3f ms, send/recv %.3f ms, receive scan %.3f ms; "
                "sent %llu records, %llu head bytes (%llu to peers); received %llu records, %llu head bytes (%llu from peers)\n",
                me, ms[0], ms[1], ms[2], ms[3], so[N], sb[N], sb[N] - byt(me, me), rn, tot, tot - byt(me, me));
        for (auto e : tev) if (e) cudaEventDestroy(e);
    }
    return MSG_OK;
}

// Collation across ranks: the exchange, the local collation and pipeline, then one allreduce (min) of {return code,
// failing rank}, so that all ranks return the same code before any combine of the counts and no rank's error leaves its
// peers waiting in a later collective.  The failing rank keeps its own message.
int collate_run_ranks(msg_ctx *c)
{
    bool run = false, sent = false;
    int rc = collate_exchange(c, &run, &sent);
    if (!run || (rc && !sent)) return rc;
    if (!rc) rc = collate_local(c);
    cudaGetLastError();
    const int N = c->cfg.n_ranks;
    int *h = reinterpret_cast<int *>(c->h_pin + 104), *d = reinterpret_cast<int *>(c->coll_xchg.as<unsigned long long>() + (size_t)N * (2 * N + 2));
    h[0] = rc; h[1] = rc ? c->cfg.rank : N;
    CU(cudaMemcpyAsync(d, h, 8, cudaMemcpyHostToDevice, c->stream));
    NC(g_nccl.AllReduce(d, d, 2, ncclInt32, ncclMin, c->comm, c->stream));
    CU(cudaMemcpyAsync(h, d, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (h[0] == MSG_OK) return MSG_OK;
    if (rc) return h[0];
    const bool record = h[0] == MSG_ENOTAG || h[0] == MSG_ENOAS || h[0] == MSG_EFORMAT;
    return fail(c, h[0], "%s on rank %d while collating across ranks (see that rank's error)", record ? "record error" : "error", h[1]);
}

// The first msg_finish_profile / msg_finish_coverage / msg_pull_counts after pushes groups everything held by QNAME and
// runs the pipeline once; across ranks every such call is collective.
int collate_run(msg_ctx *c)
{
    if (coll_across_ranks(c)) return collate_run_ranks(c);
    if (!c->coll_dirty) return MSG_OK;
    c->coll_dirty = false; c->coll_done = true;
    return collate_local(c);
}

// Exact mode: the lists that hold each feature, sorted by their input key (profile.cuh, exact mode), built once per
// finish after pushes -- entries per feature, run_scan, scatter of {key, list}, collate.cuh's bucket sorts (shared memory
// up to COLL_SMEM_KEYS entries, global memory above) -- and, with MSG_MULTI_EQUAL, d[] summed from them in that order.
int exact_prepare(msg_ctx *c)
{
    const msg_config &g = c->cfg;
    if (!g.exact || c->ex_ready) return MSG_OK;
    const bool prop = g.share_type == MSG_MULTI_PROPORTIONAL, eq = g.share_type == MSG_MULTI_EQUAL;
    if (!prop && !eq) { c->ex_ready = true; return MSG_OK; }
    const uint32_t F = (uint32_t)g.n_features, nl = (uint32_t)c->csr_lists;
    const uint64_t ne = c->csr_ent;
    if (F == 0) { c->ex_ready = true; return MSG_OK; }
    CU(c->ex_beg.reserve((size_t)F * 4)); CU(c->ex_cur.reserve((size_t)F * 4)); CU(c->ex_big.reserve((size_t)F * 4 + 8));
    CU(c->ex_keys.reserve((ne + 1) * sizeof(CollKey))); CU(c->ex_list.reserve((ne + 1) * 4));
    if (prop) CU(c->ex_sums.reserve(((size_t)nl + 1) * 8));
    uint32_t *beg = c->ex_beg.as<uint32_t>(), *cur = c->ex_cur.as<uint32_t>();
    const uint32_t *off = c->csr_off.as<uint32_t>(), *len = c->csr_len.as<uint32_t>(); const int32_t *fid = c->csr_fid.as<int32_t>();
    CollKey *keys = c->ex_keys.as<CollKey>();
    static const bool trace = getenv("MSG_TRACE_FINISH") != nullptr;
    cudaEvent_t tev[2] = {nullptr, nullptr};
    if (trace) for (auto &e : tev) cudaEventCreate(&e);
    if (trace) cudaEventRecord(tev[0], c->stream);
    const uint32_t lgrid = std::max<uint32_t>(1u, std::min<uint32_t>(nblocks(nl, 256), 148u * 8u));
    CU(cudaMemsetAsync(cur, 0, (size_t)F * 4, c->stream));
    if (nl) { exact_hist_kernel<<<lgrid, 256, 0, c->stream>>>(off, len, fid, nl, cur); LAUNCHED(c); }
    int rc = run_scan<uint32_t>(c, InU32{cur}, OutExclU32{beg}, F, (uint32_t *)nullptr);
    if (rc) return rc;
    CU(cudaMemcpyAsync(cur, beg, (size_t)F * 4, cudaMemcpyDeviceToDevice, c->stream));
    if (nl) {
        exact_scatter_kernel<<<lgrid, 256, 0, c->stream>>>(off, len, fid, nl, c->csr_key.as<unsigned long long>(), cur, keys); LAUNCHED(c);
        uint32_t *big = c->ex_big.as<uint32_t>(), *cnt = reinterpret_cast<uint32_t *>(c->d_total);
        CU(cudaMemsetAsync(cnt, 0, 4, c->stream));
        collate_bucket_sort_kernel<<<std::min<uint32_t>(F, 148u * 8u), 256, 0, c->stream>>>(keys, beg, F, ne, big, cnt); LAUNCHED(c);
        uint32_t *h_cnt = c->h_pin + 88;
        CU(cudaMemcpyAsync(h_cnt, cnt, 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (*h_cnt) { collate_sort_global_kernel<<<*h_cnt, 1024, 0, c->stream>>>(keys, beg, F, ne, big, false, nullptr, nullptr); LAUNCHED(c); }
        exact_lists_kernel<<<std::max<uint32_t>(1u, std::min<uint32_t>(nblocks(ne, 256), 148u * 8u)), 256, 0, c->stream>>>(keys, ne, c->ex_list.as<uint32_t>()); LAUNCHED(c);
    }
    if (eq) { em_exact_equal_kernel<<<std::min<uint32_t>(nblocks(F, 256), 148u * 8u), 256, 0, c->stream>>>(beg, c->ex_list.as<uint32_t>(), ne, len, c->d_d, F); LAUNCHED(c); }
    if (trace) {                           // MSG_TRACE_FINISH: the one-off cost and the longest serial chain of the gather
        cudaEventRecord(tev[1], c->stream); cudaEventSynchronize(tev[1]);
        float ms = 0; cudaEventElapsedTime(&ms, tev[0], tev[1]);
        std::vector<uint32_t> hb(F);
        cudaMemcpy(hb.data(), beg, (size_t)F * 4, cudaMemcpyDeviceToHost);
        uint64_t longest = 0;
        for (uint32_t f = 0; f < F; f++) longest = std::max<uint64_t>(longest, (f + 1 < F ? hb[f + 1] : ne) - hb[f]);
        fprintf(stderr, "[msg exact] %u lists, %llu entries, longest incidence %llu: transposition%s %.3f ms\n", nl, (unsigned long long)ne,
                (unsigned long long)longest, eq ? " + equal shares" : "", ms);
        for (auto e : tev) cudaEventDestroy(e);
    }
    c->ex_ready = true;
    return MSG_OK;
}

// MSG_EXACT_DELTA=seq (tests): take the sequential delta of the exact loop in every iteration, not only near 1e-10
bool exact_force_seq()
{
    static const bool on = getenv("MSG_EXACT_DELTA") && strcmp(getenv("MSG_EXACT_DELTA"), "seq") == 0;
    return on;
}

int allreduce(msg_ctx *c, void *buf, size_t count, ncclDataType_t dt, ncclRedOp_t op)
{
    if (c->cfg.n_ranks <= 1) return MSG_OK;
    NC(g_nccl.AllReduce(buf, buf, count, dt, op, c->comm, c->stream));
    return MSG_OK;
}

} // namespace

// ================================================================================================
extern "C" {

int msg_abi_version(void) { return MSG_ABI_VERSION; }

int msg_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char *msg_last_error(const msg_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int msg_nccl_unique_id(void *id128)
{
    msg_ctx *c = nullptr;
    std::string e;
    if (!g_nccl.load(e)) return fail(c, MSG_ENCCL, "%s", e.c_str());
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    NC(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, 128);
    return MSG_OK;
}

int msg_create(const msg_config *cfg, msg_ctx **out)
{
    msg_ctx *c = nullptr;
    if (!cfg || !out) return fail(c, MSG_EINVAL, "null argument");
    if (cfg->abi_version != MSG_ABI_VERSION) return fail(c, MSG_EINVAL, "ABI version mismatch (got %u, library %u)", cfg->abi_version, MSG_ABI_VERSION);
    if (cfg->n_targets < 0 || cfg->n_features < 0) return fail(c, MSG_EINVAL, "negative n_targets/n_features");
    if (cfg->want_profile && (cfg->share_type < 1 || cfg->share_type > 4)) return fail(c, MSG_EINVAL, "Do not understand share_type=%d", cfg->share_type);
    if (cfg->want_coverage && !cfg->target_len) return fail(c, MSG_EINVAL, "want_coverage requires target_len");
    if (cfg->do_filter && cfg->invert && cfg->hit_mode) return fail(c, MSG_EINVAL, "--invert cannot be combined with --besthit or --uniqhit");
    if (cfg->hit_mode > MSG_HIT_UNIQUE) return fail(c, MSG_EINVAL, "bad hit_mode");
    if (cfg->exact && cfg->n_ranks > 1)
        return fail(c, MSG_EINVAL, "exact needs n_ranks == 1: bit-exact sums across GPUs would chain every rank's partial sums after the previous rank's");
    if (cfg->collate > MSG_COLLATE_RANKS) return fail(c, MSG_EINVAL, "bad collate value %u (0, 1 or MSG_COLLATE_RANKS = 2)", cfg->collate);
    if (cfg->collate) {
        if (!cfg->want_profile && !cfg->want_coverage) return fail(c, MSG_EINVAL, "collate needs want_profile and/or want_coverage");
        if (cfg->want_records || cfg->want_kept || cfg->want_stats)
            return fail(c, MSG_EINVAL, "collate cannot be combined with want_records, want_kept or want_stats: results come per grouped chunk, not per pushed one");
        if (cfg->n_ranks > 1 && cfg->collate != MSG_COLLATE_RANKS)
            return fail(c, MSG_EINVAL, "collate = 1 needs n_ranks == 1; with n_ranks > 1 use collate = MSG_COLLATE_RANKS (2), which exchanges records between the ranks");
    }
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(c, MSG_ENODEV, "no CUDA device available (%s); libmsamtools_b200 has no CPU fallback", ce != cudaSuccess ? cudaGetErrorString(ce) : "device count 0"); }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(c, MSG_EINVAL, "device %d out of range (0..%d)", cfg->device, ndev - 1);
    ce = cudaSetDevice(cfg->device);
    if (ce != cudaSuccess) return fail(c, MSG_ECUDA, "cudaSetDevice: %s", cudaGetErrorString(ce));
    {   // The decode kernel touches short, scattered spans: ask the L2 to fetch single 32-byte sectors
        // from HBM instead of 64/128-byte granules (a hint; MSG_L2_FETCH=64|128 overrides for A/B runs).
        size_t gran = 32;
        if (const char *e = getenv("MSG_L2_FETCH")) gran = (size_t)atoi(e);
        if (gran == 32 || gran == 64 || gran == 128) { cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran); cudaGetLastError(); }
    }

    msg_ctx *ctx = new msg_ctx();
    ctx->cfg = *cfg; ctx->cfg.fmap = nullptr; ctx->cfg.target_len = nullptr; ctx->cfg.nccl_unique_id = nullptr;
    c = ctx;
    const msg_config &g = ctx->cfg;
#define CUC(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { int rc__ = fail(nullptr, e__ == cudaErrorMemoryAllocation ? MSG_ENOMEM : MSG_ECUDA, "%s failed: %s", #call, cudaGetErrorString(e__)); msg_destroy(ctx); return rc__; } } while (0)
    CUC(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (Slot &sl : ctx->slot) {
        CUC(cudaHostAlloc((void **)&sl.h_res, 64, cudaHostAllocPortable)); memset(sl.h_res, 0, 64);
        CUC(cudaEventCreateWithFlags(&sl.copied, cudaEventDisableTiming));
        CUC(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    }
    ctx->has_filter = g.do_filter && (g.min_length > 0 || g.ppt != 0 || g.max_clip < 100);        // msam_filter.c:79-81
    ctx->need_stats = g.do_filter && (ctx->has_filter || g.rescore);                             // :104
    ctx->cov_fused = g.want_coverage && !(g.do_filter && g.hit_mode != MSG_HIT_NONE);
    uint32_t mode = 0;
    if (g.do_filter) mode |= DM_DO_FILTER;
    if (ctx->has_filter) mode |= DM_HAS_FILTER;
    if (g.invert) mode |= DM_INVERT;
    if (g.keep_unmapped) mode |= DM_KEEP_UNMAP;
    if (g.do_filter && g.rescore) mode |= DM_RESCORE;
    if (g.do_filter && g.hit_mode) mode |= DM_NEED_AS;
    if (g.want_profile) mode |= DM_WANT_HASH;
    if (ctx->cov_fused) mode |= DM_COV_FUSED;
    ctx->cov_bits = g.want_coverage && g.coverage_summary && g.n_ranks <= 1;      // (the cross-rank combine of the bitmap would need a bitwise-OR allreduce)
    if (ctx->cov_bits) mode |= DM_COV_BITS;
    if (g.debug_force_slow) mode |= DM_FORCE_SLOW;
    ctx->decode_mode = mode;

    CUC(cudaMalloc(&ctx->d_err, 8)); CUC(cudaMalloc(&ctx->d_acct, ACCT_SLOTS * 128)); CUC(cudaMalloc(&ctx->d_total, 16));
    CUC(cudaHostAlloc((void **)&ctx->h_pin, 512, cudaHostAllocPortable)); memset(ctx->h_pin, 0, 512);
    CUC(cudaMemset(ctx->d_acct, 0, ACCT_SLOTS * 128));
    CUC(cudaMalloc(&ctx->d_wl, 8));
    const size_t T = (size_t)(g.n_targets > 0 ? g.n_targets : 1), F = (size_t)(g.n_features > 0 ? g.n_features : 1);
    if (cfg->fmap) {
        CUC(cudaMalloc(&ctx->d_fmap, T * 4));
        CUC(cudaMemcpy(ctx->d_fmap, cfg->fmap, (size_t)g.n_targets * 4, cudaMemcpyHostToDevice));
        for (int32_t i = 0; i < g.n_targets; i++)
            if (cfg->fmap[i] < 0 || cfg->fmap[i] >= g.n_features) { int rc = fail(nullptr, MSG_EINVAL, "fmap[%d]=%d outside [0,%d)", i, cfg->fmap[i], g.n_features); msg_destroy(ctx); return rc; }
    } else if (g.want_profile && g.n_features != g.n_targets) { int rc = fail(nullptr, MSG_EINVAL, "identity fmap needs n_features == n_targets"); msg_destroy(ctx); return rc; }
    if (g.want_profile) {
        CUC(cudaMalloc(&ctx->d_ui, F * 4)); CUC(cudaMalloc(&ctx->d_d, F * 8)); CUC(cudaMalloc(&ctx->d_counters, 32));
        CUC(cudaMalloc(&ctx->d_U, F * 8)); CUC(cudaMalloc(&ctx->d_a, F * 8)); CUC(cudaMalloc(&ctx->d_inc, 3 * F * 8));
        CUC(cudaHostAlloc((void **)&ctx->h_ab, F * 8, cudaHostAllocPortable));
        CUC(cudaMalloc(&ctx->d_partial, ((F + 255) / 256) * 8)); CUC(cudaMalloc(&ctx->d_delta, 8 * 20)); CUC(cudaMalloc(&ctx->d_purged, 4)); CUC(cudaMalloc(&ctx->d_bflag, 8)); CUC(cudaMemset(ctx->d_bflag, 0, 8));
        CUC(cudaMalloc(&ctx->d_ui_tmp, F * 4)); CUC(cudaMalloc(&ctx->d_d_tmp, F * 8)); CUC(cudaMalloc(&ctx->d_fcnt, 32)); CUC(cudaMalloc(&ctx->d_cursor, 16));
        CUC(cudaMemset(ctx->d_ui_tmp, 0, F * 4)); CUC(cudaMemset(ctx->d_d_tmp, 0, F * 8));
        // the fused pass applies when the profile is the filter stage's only consumer (MSG_NO_FUSED=1 forces the general pipeline)
        ctx->fused_enabled = g.do_filter && g.hit_mode != MSG_HIT_NONE && !g.want_records && !g.want_kept && !g.want_coverage && !getenv("MSG_NO_FUSED");
    }
    if (g.want_coverage) {
        std::vector<uint64_t> base(T + 1, 0);
        if (ctx->cov_bits) for (int32_t t = 0; t < g.n_targets; t++) base[t + 1] = base[t] + ((uint64_t)cfg->target_len[t] + 63) / 64;     // 64-bit words
        else               for (int32_t t = 0; t < g.n_targets; t++) base[t + 1] = base[t] + (uint64_t)cfg->target_len[t] + 1;            // cells + spill cell
        CUC(cudaMalloc(&ctx->d_tlen, T * 4)); CUC(cudaMalloc(&ctx->d_covbase, (T + 1) * 8));
        CUC(cudaMemcpy(ctx->d_tlen, cfg->target_len, (size_t)g.n_targets * 4, cudaMemcpyHostToDevice));
        CUC(cudaMemcpy(ctx->d_covbase, base.data(), (T + 1) * 8, cudaMemcpyHostToDevice));
        if (ctx->cov_bits) {
            ctx->cov_words = base[g.n_targets];
            const size_t bytes = (size_t)(ctx->cov_words ? ctx->cov_words : 1) * 8;
            CUC(cudaMalloc(&ctx->d_covbits, bytes));
            // The bitmap is hit at random while gigabytes of records stream through the same L2: pin it there (persisting
            // access-policy window on the context's stream, as much of it as the device allows to set aside).
            cudaDeviceProp prop;
            if (!getenv("MSG_NO_L2_PERSIST") && cudaGetDeviceProperties(&prop, g.device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
                const size_t aside = std::min<size_t>(bytes, (size_t)prop.persistingL2CacheMaxSize);
                if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, aside) == cudaSuccess) {
                    cudaStreamAttrValue av; memset(&av, 0, sizeof av);
                    av.accessPolicyWindow.base_ptr = ctx->d_covbits;
                    av.accessPolicyWindow.num_bytes = std::min<size_t>(bytes, (size_t)prop.accessPolicyMaxWindowSize);
                    av.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)aside / (double)av.accessPolicyWindow.num_bytes);
                    av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
                    av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
                    if (cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &av) == cudaSuccess) ctx->l2_window = true;
                }
                cudaGetLastError();
            }
        } else {
            ctx->cov_cells = base[g.n_targets];
            const size_t cells = (size_t)(ctx->cov_cells ? ctx->cov_cells : 1);
            CUC(cudaMalloc(&ctx->d_diff, cells * 4)); CUC(cudaMalloc(&ctx->d_depth, cells * 4));
        }
        CUC(cudaMalloc(&ctx->d_covered, T)); CUC(cudaMalloc(&ctx->d_touched, T * 8)); CUC(cudaMalloc(&ctx->d_sum, T * 8));
    }
    if (g.n_ranks > 1) {
        std::string e;
        if (!cfg->nccl_unique_id) { int rc = fail(nullptr, MSG_EINVAL, "n_ranks > 1 requires nccl_unique_id"); msg_destroy(ctx); return rc; }
        if (!g_nccl.load(e)) { int rc = fail(nullptr, MSG_ENCCL, "%s", e.c_str()); msg_destroy(ctx); return rc; }
        if (g.collate == MSG_COLLATE_RANKS && (!g_nccl.Send || !g_nccl.Recv || !g_nccl.GroupStart || !g_nccl.GroupEnd || !g_nccl.AllGather)) {
            int rc = fail(nullptr, MSG_ENCCL, "libnccl lacks ncclSend / ncclRecv / ncclGroupStart / ncclGroupEnd / ncclAllGather, which collation across ranks needs");
            msg_destroy(ctx); return rc;
        }
        ncclUniqueId id; memcpy(&id, cfg->nccl_unique_id, 128);
        ncclResult_t r = g_nccl.CommInitRank(&ctx->comm, g.n_ranks, id, g.rank);
        if (r != ncclSuccess) { int rc = fail(nullptr, MSG_ENCCL, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"); msg_destroy(ctx); return rc; }
        if (g.want_profile && g.n_ranks <= 16 && g_nccl.AllGather) {
            // Map every rank's publish region into this process (CUDA IPC over NVLink).  If any rank cannot, all ranks
            // agree (allreduce-min) to keep the NCCL-per-iteration loop instead.
            // profile.cuh: small vectors travel as flagged words, all to all (purged[16] u64, slot[2][n_ranks][F + 8][2] u64);
            // gene catalogues use the reduce-scatter / all-gather layout (RsagLayout, ~4 * F * 8 bytes)
            const size_t region = F + 8 <= EM_XCHG_CTA0 ? 128 + 2 * (size_t)g.n_ranks * (F + 8) * 16 : rsag_layout((uint32_t)F, g.n_ranks).total();
            ctx->peer_region_bytes = region;
            int ok = 1;
            cudaIpcMemHandle_t mine; memset(&mine, 0, sizeof mine);
            unsigned char *d_hs = nullptr; int *d_ok = nullptr;
            std::vector<cudaIpcMemHandle_t> hs((size_t)g.n_ranks);
            CUC(cudaMalloc(&ctx->peer_region, region)); CUC(cudaMemset(ctx->peer_region, 0, region));
            CUC(cudaMalloc(&d_hs, sizeof(cudaIpcMemHandle_t) * (size_t)g.n_ranks)); CUC(cudaMalloc(&d_ok, 4));
            if ((getenv("MSG_NO_P2P") && atoi(getenv("MSG_NO_P2P"))) || cudaIpcGetMemHandle(&mine, ctx->peer_region) != cudaSuccess) { ok = 0; cudaGetLastError(); }
            CUC(cudaMemcpy(d_hs + sizeof mine * (size_t)g.rank, &mine, sizeof mine, cudaMemcpyHostToDevice));
            if (g_nccl.AllGather(d_hs + sizeof mine * (size_t)g.rank, d_hs, sizeof mine, ncclUint8, ctx->comm, ctx->stream) != ncclSuccess) ok = 0;
            CUC(cudaStreamSynchronize(ctx->stream));
            CUC(cudaMemcpy(hs.data(), d_hs, sizeof mine * (size_t)g.n_ranks, cudaMemcpyDeviceToHost));
            for (int pr = 0; pr < g.n_ranks && ok; pr++) {
                if (pr == g.rank) { ctx->peer_tab.base[pr] = ctx->peer_region; continue; }
                void *pp = nullptr;
                if (cudaIpcOpenMemHandle(&pp, hs[(size_t)pr], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); break; }
                ctx->ipc_opened.push_back(pp); ctx->peer_tab.base[pr] = (unsigned char *)pp;
            }
            CUC(cudaMemcpy(d_ok, &ok, 4, cudaMemcpyHostToDevice));
            if (g_nccl.AllReduce(d_ok, d_ok, 1, ncclInt32, ncclMin, ctx->comm, ctx->stream) != ncclSuccess) ok = 0;
            CUC(cudaStreamSynchronize(ctx->stream));
            int all_ok = 0; CUC(cudaMemcpy(&all_ok, d_ok, 4, cudaMemcpyDeviceToHost));
            ctx->p2p_ok = ok && all_ok;
            cudaFree(d_hs); cudaFree(d_ok);
        }
    }
#undef CUC
    int rc = msg_reset(ctx);
    if (rc) { g_create_error = ctx->err; msg_destroy(ctx); return rc; }
    *out = ctx;
    return MSG_OK;
}

void msg_destroy(msg_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->cfg.device);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->l2_window) { cudaCtxResetPersistingL2Cache(); cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0); cudaGetLastError(); }
    for (Slot &sl : c->slot) {
        sl.raw.release(); sl.off.release();
        if (sl.h_res) cudaFreeHost(sl.h_res);
        if (sl.copied) cudaEventDestroy(sl.copied);
        if (sl.done) cudaEventDestroy(sl.done);
    }
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    for (void *pp : c->ipc_opened) cudaIpcCloseMemHandle(pp);
    if (c->peer_region) cudaFree(c->peer_region);
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    DevBuf *bufs[] = {&c->tid, &c->fb, &c->score, &c->hash, &c->nid, &c->st_alen, &c->st_qlen, &c->st_qclip, &c->st_edit,
                      &c->kbase, &c->worklist, &c->gmeta, &c->out_idx, &c->tile_sums, &c->pcount, &c->scanv, &c->biglist, &c->out_len, &c->out_off, &c->plan, &c->out_rec,
                      &c->csr_off, &c->csr_len, &c->csr_fid, &c->csr_key, &c->ex_beg, &c->ex_cur, &c->ex_keys, &c->ex_big, &c->ex_list, &c->ex_sums, &c->win, &c->t_ui, &c->t_d, &c->t_cnt, &c->t_cov,
                      &c->coll_arena, &c->coll_aoff, &c->coll_keys, &c->coll_keys2, &c->coll_len, &c->coll_hist, &c->coll_bstart, &c->coll_list,
                      &c->coll_grouped, &c->coll_goff, &c->coll_xchg};
    for (DevBuf *b : bufs) b->release();
    void *ptrs[] = {c->d_fmap, c->d_tlen, c->d_covbase, c->d_err, c->d_acct, c->d_total, c->d_ui, c->d_d, c->d_counters, c->d_stamp, c->d_U, c->d_a,
                    c->d_inc, c->d_partial, c->d_delta, c->d_purged, c->d_bflag, c->d_wl, c->d_ui_tmp, c->d_d_tmp, c->d_fcnt, c->d_cursor, c->d_diff, c->d_depth, c->d_covered, c->d_touched, c->d_sum, c->d_covbits};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (c->h_pin) cudaFreeHost(c->h_pin);
    if (c->h_ab) cudaFreeHost(c->h_ab);
    for (auto &pr : c->ev_decode) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
    for (auto &pr : c->ev_total) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
    for (auto e : c->ev_free) cudaEventDestroy(e);
    for (auto e : c->marks) if (e) cudaEventDestroy(e);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int msg_reset(msg_ctx *c)
{
    if (!c) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    for (int k = 0; k < 2; k++)                       // results of chunks still in flight are dropped with the rest of the state
        if (c->slot[k].pending) { cudaEventSynchronize(c->slot[k].done); c->slot[k].pending = false; }
    c->inflight_lists = c->inflight_ent = 0; c->cursor_dirty = true; c->next_slot = 0;
    const msg_config &g = c->cfg;
    const size_t T = (size_t)(g.n_targets > 0 ? g.n_targets : 1), F = (size_t)(g.n_features > 0 ? g.n_features : 1);
    CU(cudaMemsetAsync(c->d_err, 0, 4, c->stream));
    CU(cudaMemsetAsync(c->d_err + 1, 0xff, 4, c->stream));
    if (g.want_profile) {
        CU(cudaMemsetAsync(c->d_ui, 0, F * 4, c->stream)); CU(cudaMemsetAsync(c->d_d, 0, F * 8, c->stream));
        CU(cudaMemsetAsync(c->d_counters, 0, 32, c->stream));
        c->csr_lists = c->csr_ent = 0;
    }
    c->rec_base = 0; c->ex_ready = false;
    if (g.want_coverage) {
        if (c->cov_bits) {
            CU(cudaMemsetAsync(c->d_covbits, 0, (size_t)(c->cov_words ? c->cov_words : 1) * 8, c->stream));
            CU(cudaMemsetAsync(c->d_sum, 0, T * 8, c->stream));
        } else CU(cudaMemsetAsync(c->d_diff, 0, (size_t)(c->cov_cells ? c->cov_cells : 1) * 4, c->stream));
        CU(cudaMemsetAsync(c->d_covered, 0, T, c->stream));
        c->cov_finished = false;
    }
    c->coll_n = c->coll_bytes = 0; c->coll_dirty = c->coll_done = false;
    c->n_kept = 0; c->have_stream = false; c->out_bytes = 0; c->cur_n = 0;
    CU(cudaStreamSynchronize(c->stream));
    return MSG_OK;
}

// ------------------------------------------------------------------ host index helpers: csrc/host/recindex.c (plain C, also built into libmsamhost.so)

// ------------------------------------------------------------------ data path
int msg_device_alloc(msg_ctx *c, size_t nbytes, void **d_ptr)
{
    if (!c || !d_ptr) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    CU(cudaMalloc(d_ptr, nbytes + 64));                 // 16-byte chunk loads may straddle the end
    CU(cudaMemset((uint8_t *)*d_ptr + nbytes, 0, 64));
    return MSG_OK;
}
int msg_device_free(msg_ctx *c, void *d_ptr) { if (!c) return MSG_EINVAL; CU(cudaSetDevice(c->cfg.device)); CU(cudaFree(d_ptr)); return MSG_OK; }
int msg_device_upload(msg_ctx *c, void *d_dst, const void *h_src, size_t nbytes)
{
    if (!c) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    CU(cudaMemcpyAsync(d_dst, h_src, nbytes, cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return MSG_OK;
}
int msg_host_alloc(int device, size_t nbytes, void **h_ptr)
{
    msg_ctx *c = nullptr;
    if (!h_ptr) return MSG_EINVAL;
    CU(cudaSetDevice(device));
    CU(cudaHostAlloc(h_ptr, nbytes ? nbytes : 1, cudaHostAllocPortable));
    return MSG_OK;
}
int msg_host_free(void *h_ptr)
{
    msg_ctx *c = nullptr;
    if (h_ptr) CU(cudaFreeHost(h_ptr));
    return MSG_OK;
}

int msg_sync(msg_ctx *c)
{
    if (!c) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    int wrc = wait_all(c);
    CU(cudaStreamSynchronize(c->stream));
    harvest_events(c);
    return wrc;
}

int msg_push_async(msg_ctx *c, const uint8_t *raw, size_t nbytes, const uint64_t *rec_off, size_t nrec)
{
    if (!c || (nrec && (!raw || !rec_off))) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    if (c->cfg.collate) return collate_push(c, raw, nullptr, nbytes, rec_off, nullptr, nrec);
    return push_chunk(c, raw, nullptr, nbytes, rec_off, nullptr, nrec);
}

int msg_push_device_async(msg_ctx *c, const uint8_t *d_raw, size_t nbytes, const uint64_t *d_rec_off, size_t nrec)
{
    if (!c || (nrec && (!d_raw || !d_rec_off))) return MSG_EINVAL;
    if ((uintptr_t)d_raw & 15u) return fail(c, MSG_EINVAL, "device chunk must be 16-byte aligned");
    CU(cudaSetDevice(c->cfg.device));
    if (c->cfg.collate) return collate_push(c, nullptr, d_raw, nbytes, nullptr, d_rec_off, nrec);
    return push_chunk(c, nullptr, d_raw, nbytes, nullptr, d_rec_off, nrec);
}

int msg_wait(msg_ctx *c)
{
    if (!c) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    return wait_all(c);
}

int msg_push(msg_ctx *c, const uint8_t *raw, size_t nbytes, const uint64_t *rec_off, size_t nrec)
{
    int rc = msg_push_async(c, raw, nbytes, rec_off, nrec);
    return rc ? rc : wait_all(c);
}

int msg_push_device(msg_ctx *c, const uint8_t *d_raw, size_t nbytes, const uint64_t *d_rec_off, size_t nrec)
{
    int rc = msg_push_device_async(c, d_raw, nbytes, d_rec_off, nrec);
    return rc ? rc : wait_all(c);
}

static const char *k_collate_chunk = "per-chunk results are not available on a collating context (records are grouped at finish)";

int msg_kept_count(msg_ctx *c, size_t *n_kept)
{
    if (!c || !n_kept) return MSG_EINVAL;
    if (c->cfg.collate) return fail(c, MSG_ESTATE, "%s", k_collate_chunk);
    CU(cudaSetDevice(c->cfg.device));
    { int wrc = wait_all(c); if (wrc) return wrc; }
    *n_kept = c->n_kept;
    return MSG_OK;
}

int msg_pull_kept(msg_ctx *c, uint32_t *idx, size_t cap, size_t *n_kept)
{
    if (!c) return MSG_EINVAL;
    if (c->cfg.collate) return fail(c, MSG_ESTATE, "%s", k_collate_chunk);
    CU(cudaSetDevice(c->cfg.device));
    { int wrc = wait_all(c); if (wrc) return wrc; }
    if (n_kept) *n_kept = c->n_kept;
    if (!idx) return MSG_OK;
    if (c->cfg.do_filter && !c->cfg.want_kept) return fail(c, MSG_ESTATE, "context was created without want_kept");
    if (cap < c->n_kept) return fail(c, MSG_ERANGE, "kept buffer too small (%zu < %llu)", cap, (unsigned long long)c->n_kept);
    if (c->have_stream) {
        CU(cudaMemcpyAsync(idx, c->out_idx.p, c->n_kept * 4, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->d2h_bytes += c->n_kept * 4;
    } else for (uint64_t i = 0; i < c->n_kept; i++) idx[i] = (uint32_t)i;
    return MSG_OK;
}

int msg_pull_records(msg_ctx *c, uint8_t *out, size_t cap, size_t *nbytes, size_t *nrec)
{
    if (!c) return MSG_EINVAL;
    if (c->cfg.collate) return fail(c, MSG_ESTATE, "%s", k_collate_chunk);
    if (!c->cfg.want_records) return fail(c, MSG_ESTATE, "context was created without want_records");
    CU(cudaSetDevice(c->cfg.device));
    { int wrc = wait_all(c); if (wrc) return wrc; }
    if (nbytes) *nbytes = c->out_bytes;
    if (nrec) *nrec = c->n_kept;
    if (!out) return MSG_OK;
    if (cap < c->out_bytes) return fail(c, MSG_ERANGE, "record buffer too small");
    if (c->out_bytes) {
        CU(cudaMemcpyAsync(out, c->out_rec.p, c->out_bytes, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->d2h_bytes += c->out_bytes;
    }
    return MSG_OK;
}

int msg_pull_stats(msg_ctx *c, size_t nrec, int32_t *alen, int32_t *qlen, int32_t *qclip, int32_t *edit, int32_t *score, uint8_t *flags)
{
    if (!c) return MSG_EINVAL;
    if (c->cfg.collate) return fail(c, MSG_ESTATE, "%s", k_collate_chunk);
    if (!c->cfg.want_stats) return fail(c, MSG_ESTATE, "context was created without want_stats");
    { int wrc = wait_all(c); if (wrc) return wrc; }
    if (nrec != c->cur_n) return fail(c, MSG_EINVAL, "nrec does not match the last chunk");
    CU(cudaSetDevice(c->cfg.device));
    if (nrec == 0) return MSG_OK;
    if (alen)  CU(cudaMemcpyAsync(alen, c->st_alen.p, nrec * 4, cudaMemcpyDeviceToHost, c->stream));
    if (qlen)  CU(cudaMemcpyAsync(qlen, c->st_qlen.p, nrec * 4, cudaMemcpyDeviceToHost, c->stream));
    if (qclip) CU(cudaMemcpyAsync(qclip, c->st_qclip.p, nrec * 4, cudaMemcpyDeviceToHost, c->stream));
    if (edit)  CU(cudaMemcpyAsync(edit, c->st_edit.p, nrec * 4, cudaMemcpyDeviceToHost, c->stream));
    if (score) CU(cudaMemcpyAsync(score, c->score.p, nrec * 4, cudaMemcpyDeviceToHost, c->stream));
    std::vector<uint32_t> fb;
    if (flags) { fb.resize(nrec); CU(cudaMemcpyAsync(fb.data(), c->fb.p, nrec * 4, cudaMemcpyDeviceToHost, c->stream)); }
    CU(cudaStreamSynchronize(c->stream));
    if (flags) for (size_t i = 0; i < nrec; i++)
        flags[i] = (uint8_t)(((fb[i] & FB_INPOOL) ? 1 : 0) | ((fb[i] & FB_HAS_AS) ? 2 : 0) | ((fb[i] & FB_EQPREV) ? 4 : 0) | ((fb[i] & FB_SLOW) ? 8 : 0));
    return MSG_OK;
}

int msg_pull_counts(msg_ctx *c, uint32_t *ui, double *d)
{
    if (!c) return MSG_EINVAL;
    if (!c->cfg.want_profile) return fail(c, MSG_ESTATE, "context was created without want_profile");
    CU(cudaSetDevice(c->cfg.device));
    { int wrc = wait_all(c); if (wrc) return wrc; }
    { int crc = collate_run(c); if (crc) return crc; }
    { int erc = exact_prepare(c); if (erc) return erc; }
    const size_t F = (size_t)c->cfg.n_features;
    if (ui && F) CU(cudaMemcpyAsync(ui, c->d_ui, F * 4, cudaMemcpyDeviceToHost, c->stream));
    if (d && F)  CU(cudaMemcpyAsync(d, c->d_d, F * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return MSG_OK;
}

// MSG_TRACE_FINISH=1: device-side time of each phase of msg_finish_profile, printed to stderr (diagnostics only).
// Events: 0 start, 1 counts combined over NCCL, 2 em_init done, 3 cooperative loop launched, 4 end.
struct FinishTrace {
    bool on;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    void mark(int k, cudaStream_t s) { if (on) { if (!ev[k]) cudaEventCreate(&ev[k]); cudaEventRecord(ev[k], s); } }
};

// With n_ranks > 1: ONE allreduce over NVLink for everything that is additive across ranks (per-reference counts, the
// insert counters and the number of multi-mapper lists, packed as u32[F + 8]) and one for the MSG_MULTI_EQUAL shares,
// on copies, so that finish can be called again after more chunks; ui and dd then point at the sums.  The insert
// counters (and, with n_ranks > 1, the list total) are copied to hc.
static int finish_combine_counts(msg_ctx *c, uint32_t *&ui, double *&dd, uint32_t *hc, FinishTrace &tr)
{
    const msg_config &g = c->cfg;
    const uint32_t F = (uint32_t)g.n_features;
    int rc;
    if (g.n_ranks <= 1) { CU(cudaMemcpyAsync(hc, c->d_counters, 16, cudaMemcpyDeviceToHost, c->stream)); return MSG_OK; }
    CU(c->t_ui.reserve(((size_t)F + 8) * 4));
    ui = c->t_ui.as<uint32_t>();
    uint32_t *cnt = ui + F;
    CU(cudaMemcpyAsync(ui, c->d_ui, (size_t)F * 4, cudaMemcpyDeviceToDevice, c->stream));
    CU(cudaMemcpyAsync(cnt, c->d_counters, 16, cudaMemcpyDeviceToDevice, c->stream));
    const uint32_t nl_lo[2] = {(uint32_t)(c->csr_lists & 0xffffu), (uint32_t)(c->csr_lists >> 16)};   // two 16-bit halves: sums stay exact in u32 for up to 65536 ranks
    CU(cudaMemcpyAsync(cnt + 4, nl_lo, 8, cudaMemcpyHostToDevice, c->stream));
    if ((rc = allreduce(c, ui, (size_t)F + 6, ncclUint32, ncclSum))) return rc;
    if (g.share_type == MSG_MULTI_EQUAL) {
        CU(c->t_d.reserve((size_t)(F ? F : 1) * 8));
        CU(cudaMemcpyAsync(c->t_d.p, c->d_d, (size_t)F * 8, cudaMemcpyDeviceToDevice, c->stream));
        dd = c->t_d.as<double>();
        if ((rc = allreduce(c, dd, F, ncclFloat64, ncclSum))) return rc;
    }
    tr.mark(1, c->stream);
    CU(cudaMemcpyAsync(hc, cnt, 24, cudaMemcpyDeviceToHost, c->stream));
    return MSG_OK;
}

// The whole PropSharing loop in one cooperative launch: grid-wide barriers, no host round trips.  With n_ranks > 1 the
// kernel also combines the counts (hc receives the insert counters and the list total) and runs every iteration's
// exchange through peer memory.  The loop's iterations, deltas and purged count go to res / h_delta.  *ran stays false
// when one GPU cannot co-schedule a CTA per SM: the caller then runs the host loop.
static int em_coop_loop(msg_ctx *c, uint32_t *hc, int32_t *res, double *h_delta, FinishTrace &tr, bool *ran)
{
    const msg_config &g = c->cfg;
    const uint32_t F = (uint32_t)g.n_features;
    const bool multi = g.n_ranks > 1, sm = F <= EM_SMEM_F;
    const bool rsag = multi && F + 8 > EM_XCHG_CTA0;               // gene catalogues: reduce-scatter / all-gather exchange
    const size_t shm = g.exact ? 0 : em_smem_bytes(F);
    int rc;
    // the argument arrays below hold the addresses of these; partial is set once the grid size is known
    const uint32_t *a0 = c->csr_off.as<uint32_t>(), *a1 = c->csr_len.as<uint32_t>(); const int32_t *a2 = c->csr_fid.as<int32_t>();
    uint32_t nl_arg = (uint32_t)c->csr_lists, F_arg = F;
    double *U = c->d_U, *av = c->d_a, *inc = c->d_inc, *dout = c->d_delta, *partial = nullptr;
    int32_t *d_res = reinterpret_cast<int32_t *>(c->d_total);
    const uint32_t *ui_arg = c->d_ui, *cnt_arg = c->d_counters;
    uint32_t nl_lo = (uint32_t)(c->csr_lists & 0xffffu), nl_hi = (uint32_t)(c->csr_lists >> 16);   // two 16-bit halves, as in the NCCL path
    uint32_t *hc_dev = nullptr, *bflag = c->d_bflag;
    double *totbuf = nullptr;
    unsigned long long *d_trace = nullptr;
    PeerTable pt = c->peer_tab; int nr = g.n_ranks, rk = g.rank; uint32_t epoch = c->em_epoch;
    static const double peer_timeout_s = getenv("MSG_PEER_TIMEOUT_S") ? atof(getenv("MSG_PEER_TIMEOUT_S")) : 120.0;
    unsigned long long timeout_ns = (unsigned long long)(peer_timeout_s * 1e9);
    if (multi) {
        CU(c->t_cnt.reserve(64)); hc_dev = c->t_cnt.as<uint32_t>();
        CU(c->t_d.reserve((size_t)F * 16)); totbuf = c->t_d.as<double>();
        if (tr.on) { CU(c->t_ui.reserve(20 * 8 * 8)); d_trace = c->t_ui.as<unsigned long long>(); CU(cudaMemsetAsync(d_trace, 0, 20 * 8 * 8, c->stream)); }
    }
    void *largs[] = {&a0, &a1, &a2, &nl_arg, &U, &av, &inc, &partial, &F_arg, &dout, &d_res};
    void *sargs[] = {&a0, &a1, &a2, &nl_arg, &U, &av, &inc, &F_arg, &dout, &d_res};
    void *margs[] = {&a0, &a1, &a2, &nl_arg, &ui_arg, &cnt_arg, &nl_lo, &nl_hi, &U, &av, &inc, &partial, &F_arg, &dout, &d_res, &hc_dev,
                     &totbuf, &bflag, &pt, &nr, &rk, &epoch, &timeout_ns};
    void *rargs[] = {&a0, &a1, &a2, &nl_arg, &ui_arg, &cnt_arg, &nl_lo, &nl_hi, &U, &av, &inc, &F_arg, &dout, &d_res, &hc_dev,
                     &pt, &nr, &rk, &epoch, &timeout_ns, &d_trace};
    // exact (one GPU): incidence from exact_prepare; list sums in ex_sums, the squared differences in the second third of inc
    const uint32_t *ibeg = c->ex_beg.as<uint32_t>(), *ilist = c->ex_list.as<uint32_t>();
    unsigned long long nent = c->csr_ent;
    double *sums = c->ex_sums.as<double>(), *sq = c->d_inc + F;
    int force_seq = exact_force_seq();
    void *xargs[] = {&a0, &a1, &a2, &nl_arg, &ibeg, &ilist, &nent, &U, &av, &sums, &sq, &partial, &F_arg, &dout, &d_res, &force_seq};
    const bool exact = g.exact != 0;
    const void *fn; void **args;
    if (exact)      { fn = (const void *)em_loop_exact_kernel; args = xargs; }
    else if (rsag)  { fn = (const void *)em_loop_rsag_kernel; args = rargs; }
    else if (multi) { fn = sm ? (const void *)em_loop_multi_kernel<true> : (const void *)em_loop_multi_kernel<false>; args = margs; }
    else if (sm)    { fn = (const void *)em_loop_smem_kernel; args = sargs; }
    else            { fn = (const void *)em_loop_kernel; args = largs; }
    int per_sm = 0, nsm = 0;
    CU(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, g.device));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 256, shm));
    if (per_sm < 1) {
        if (multi) return fail(c, MSG_ECUDA, "cannot launch the cooperative PropSharing kernel (F = %u needs too much shared memory?)", F);
        return MSG_OK;
    }
    const int want_ctas = EM_CTAS_ENV > 0 ? EM_CTAS_ENV : (sm && !exact ? 3 : 4);
    if (per_sm > want_ctas) per_sm = want_ctas;
    const uint32_t grid = (uint32_t)(nsm * per_sm);
    CU(c->tile_sums.reserve((size_t)grid * 8 + 16));                 // + the exact loop's sequential delta
    partial = c->tile_sums.as<double>();
    // one GPU: inc[3F], delta and d_res were cleared by em_init_kernel; the multi-GPU kernels clear their own state
    if (multi) {
        // The kernels of all ranks wait for one another inside the loop: line the ranks up first (a 4-byte NCCL
        // allreduce on the same stream; it waits, on the device, for however long the slowest rank's ingest takes),
        // so that the wall-clock limit inside the kernel (MSG_PEER_TIMEOUT_S, default 120 s) only ever measures a
        // peer that died, not one that is merely late.
        CU(cudaMemsetAsync(d_res, 0, 16, c->stream));
        if ((rc = allreduce(c, c->t_cnt.as<uint32_t>() + 8, 1, ncclUint32, ncclSum))) return rc;
        if (rsag) CU(cudaMemsetAsync(c->d_inc, 0, (size_t)F * 8, c->stream));
    }
    CU(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(256), args, shm, c->stream));
    LAUNCHED(c);
    if (multi) {
        c->em_epoch += 32;
        CU(cudaMemcpyAsync(hc, hc_dev, 24, cudaMemcpyDeviceToHost, c->stream));
    }
    tr.mark(3, c->stream);
    CU(cudaMemcpyAsync(res, d_res, 16, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(h_delta, c->d_delta, 8 * 20, cudaMemcpyDeviceToHost, c->stream));
    c->d2h_bytes += 176;
    *ran = true;
    return MSG_OK;
}

// The PropSharing loop with one launch per phase and a host read of delta per iteration: the NCCL fallback of the
// multi-GPU loop (MSG_EM_HOST_LOOP=1 selects it on one GPU too).  The purged count lands in *h_purged at the caller's
// stream sync.
static int em_host_loop(msg_ctx *c, msg_profile_stats &s, uint32_t *h_purged)
{
    const uint32_t F = (uint32_t)c->cfg.n_features, nb = nblocks(F, 256), nl32 = (uint32_t)c->csr_lists;
    const uint32_t em_grid = nl32 ? (nblocks(nl32, 256) < 148u * 8u ? nblocks(nl32, 256) : 148u * 8u) : 0;
    const uint32_t *off = c->csr_off.as<uint32_t>(), *len = c->csr_len.as<uint32_t>(); const int32_t *fid = c->csr_fid.as<int32_t>();
    int rc;
    const bool exact = c->cfg.exact != 0;
    for (int k = 1; k < 20; k++) {                                                                      // msam_profile.c:331
        if (exact) {
            if (!F) { s.em_delta[k - 1] = nan(""); s.em_iterations = k; continue; }
            if (nl32) { em_exact_sums_kernel<<<em_grid, 256, 0, c->stream>>>(off, len, fid, nl32, c->d_a, c->ex_sums.as<double>()); LAUNCHED(c); }
            em_exact_gather_kernel<<<nb, 256, 0, c->stream>>>(c->ex_beg.as<uint32_t>(), c->ex_list.as<uint32_t>(), c->csr_ent, c->ex_sums.as<double>(),
                                                              c->d_U, c->d_a, c->d_inc + F, c->d_partial, F); LAUNCHED(c);
            em_delta_kernel<<<1, 256, 0, c->stream>>>(c->d_partial, nb, F, c->d_delta + (k - 1)); LAUNCHED(c);
            double delta = 0;
            CU(cudaMemcpyAsync(&delta, c->d_delta + (k - 1), 8, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            if (exact_force_seq() || em_exact_near(delta, F)) {              // profile.cuh: the sum in order j = 0 .. F-1
                em_exact_seq_kernel<<<1, 32, 0, c->stream>>>(c->d_inc + F, F, c->d_delta + (k - 1)); LAUNCHED(c);
                CU(cudaMemcpyAsync(&delta, c->d_delta + (k - 1), 8, cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
            }
            c->d2h_bytes += 8;
            s.em_delta[k - 1] = delta; s.em_iterations = k;
            if (delta < 1e-10) { s.em_converged = 1; break; }
            continue;
        }
        CU(cudaMemsetAsync(c->d_inc, 0, (size_t)F * 8, c->stream));
        if (nl32) { em_gather_kernel<<<em_grid, 256, em_smem_bytes(F), c->stream>>>(off, len, fid, nl32, c->d_a, c->d_inc, F); LAUNCHED(c); }
        if ((rc = allreduce(c, c->d_inc, F, ncclFloat64, ncclSum))) return rc;
        double delta = 0;
        if (F) {
            em_update_kernel<<<nb, 256, 0, c->stream>>>(c->d_U, c->d_inc, c->d_a, c->d_partial, F); LAUNCHED(c);
            em_delta_kernel<<<1, 256, 0, c->stream>>>(c->d_partial, nb, F, c->d_delta + (k - 1)); LAUNCHED(c);
            CU(cudaMemcpyAsync(&delta, c->d_delta + (k - 1), 8, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            c->d2h_bytes += 8;
        } else delta = nan("");                                                                     // reference divides by n_features == 0
        s.em_delta[k - 1] = delta; s.em_iterations = k;
        if (delta < 1e-10) { s.em_converged = 1; break; }                                               // :383
    }
    CU(cudaMemsetAsync(c->d_purged, 0, 4, c->stream));
    if (nl32) { em_purged_kernel<<<em_grid, 256, 0, c->stream>>>(off, len, fid, nl32, c->d_a, c->d_purged); LAUNCHED(c); }
    if ((rc = allreduce(c, c->d_purged, 1, ncclUint32, ncclSum))) return rc;
    CU(cudaMemcpyAsync(h_purged, c->d_purged, 4, cudaMemcpyDeviceToHost, c->stream));
    return MSG_OK;
}

static void finish_trace_report(msg_ctx *c, FinishTrace &tr, bool rsag_trace)
{
    const msg_config &g = c->cfg;
    tr.mark(4, c->stream); cudaEventSynchronize(tr.ev[4]);
    float ms[4] = {0, 0, 0, 0};
    for (int k = 0; k < 4; k++) if (tr.ev[k] && tr.ev[k + 1]) cudaEventElapsedTime(&ms[k], tr.ev[k], tr.ev[k + 1]);
    if (tr.ev[0] && tr.ev[2] && !tr.ev[1]) cudaEventElapsedTime(&ms[1], tr.ev[0], tr.ev[2]);
    float chunk = 0, gap = 0, dec = 0;
    if (!c->ev_total.empty()) { cudaEventElapsedTime(&chunk, c->ev_total.back().first, c->ev_total.back().second); cudaEventElapsedTime(&gap, c->ev_total.back().second, tr.ev[0]); }
    if (!c->ev_decode.empty()) cudaEventElapsedTime(&dec, c->ev_decode.back().first, c->ev_decode.back().second);
    fprintf(stderr, "[msg finish rank %d] last chunk %.3f ms (decode %.3f), gap %.3f ms, allreduce %.3f ms, init %.3f ms, loop %.3f ms, tail %.3f ms\n",
            g.rank, chunk, dec, gap, ms[0], ms[1], ms[2], ms[3]);
    if (rsag_trace) {
        // CTA 0's view of the exchanges (ns): RS stores | fence+flags | owner blocks | announce | AG wait | grid barrier | delta ; gather = gap to the next exchange
        unsigned long long t[160]; cudaMemcpy(t, c->t_ui.p, sizeof t, cudaMemcpyDeviceToHost);
        double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}; int nx = 0;
        for (int k = 1; k < 20 && t[k * 8 + 7]; k++) {
            for (int j = 0; j < 7; j++) acc[j] += (double)(t[k * 8 + j + 1] - t[k * 8 + j]);
            if (k + 1 < 20 && t[(k + 1) * 8]) acc[7] += (double)(t[(k + 1) * 8] - t[k * 8 + 7]);
            nx++;
        }
        if (nx) fprintf(stderr, "[msg finish rank %d] rsag exchange, mean over %d (us): rs-store %.1f fence+flags %.1f owner %.1f announce %.1f ag-wait %.1f barrier %.1f delta %.1f | gather+barrier %.1f\n",
                        g.rank, nx, acc[0] / nx / 1e3, acc[1] / nx / 1e3, acc[2] / nx / 1e3, acc[3] / nx / 1e3, acc[4] / nx / 1e3, acc[5] / nx / 1e3, acc[6] / nx / 1e3, acc[7] / nx / 1e3);
    }
    for (auto e : tr.ev) if (e) cudaEventDestroy(e);
}

int msg_finish_profile(msg_ctx *c, double *abundance, msg_profile_stats *st)
{
    if (!c) return MSG_EINVAL;
    if (!c->cfg.want_profile) return fail(c, MSG_ESTATE, "context was created without want_profile");
    CU(cudaSetDevice(c->cfg.device));
    { int wrc = wait_all(c); if (wrc) return wrc; }
    { int crc = collate_run(c); if (crc) return crc; }
    { int erc = exact_prepare(c); if (erc) return erc; }
    const msg_config &g = c->cfg;
    const uint32_t F = (uint32_t)g.n_features;
    msg_profile_stats s; memset(&s, 0, sizeof s);
    int rc;
    static const bool trace = getenv("MSG_TRACE_FINISH") != nullptr;
    FinishTrace tr{trace};
    tr.mark(0, c->stream);
    // every small result is copied into pinned memory and read after ONE stream sync at the end
    uint32_t *hc = c->h_pin + 20; int32_t *res = reinterpret_cast<int32_t *>(c->h_pin + 16); uint32_t *h_purged = c->h_pin + 26;
    double *h_delta = reinterpret_cast<double *>(c->h_pin + 32);
    memset(c->h_pin + 16, 0, 4 * (72 - 16));
    const bool em = g.share_type == MSG_MULTI_PROPORTIONAL;
    const bool coop = em && F > 0 && (g.n_ranks <= 1 || c->p2p_ok) && !getenv("MSG_EM_HOST_LOOP");
    // with n_ranks > 1 the cooperative loop kernel also combines the counts, so no NCCL call and no em_init
    if (!coop || g.n_ranks <= 1) {
        uint32_t *ui = c->d_ui; double *dd = c->d_d;
        if ((rc = finish_combine_counts(c, ui, dd, hc, tr))) return rc;
        if (F) {
            em_init_kernel<<<nblocks(F, 256), 256, 0, c->stream>>>(ui, dd, g.share_type == MSG_MULTI_EQUAL, c->d_U, c->d_a, F, c->d_inc, c->d_delta,
                                                                  reinterpret_cast<int32_t *>(c->d_total));
            LAUNCHED(c);
        }
    }
    tr.mark(2, c->stream);
    bool looped = false;                              // the cooperative loop ran; it counts the purged lists itself
    if (coop && (rc = em_coop_loop(c, hc, res, h_delta, tr, &looped))) return rc;
    if (em && !looped && (rc = em_host_loop(c, s, h_purged))) return rc;
    if (abundance && F) CU(cudaMemcpyAsync(c->h_ab, c->d_a, (size_t)F * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(c->h_pin + 8, c->d_err, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (looped) {
        if (g.n_ranks > 1 && res[2]) return fail(c, MSG_ENCCL, "timed out waiting for a peer GPU inside the PropSharing loop");
        s.em_iterations = res[0]; s.em_converged = res[1]; s.purged_insert_count = (uint32_t)res[3];
        memcpy(s.em_delta, h_delta, sizeof s.em_delta);
    } else if (em) s.purged_insert_count = *h_purged;
    if (tr.on) finish_trace_report(c, tr, looped && g.n_ranks > 1 && F + 8 > EM_XCHG_CTA0);
    if (abundance && F) memcpy(abundance, c->h_ab, (size_t)F * 8);
    c->d2h_bytes += (size_t)F * 8 + 28;
    s.mapped_inserts = hc[0]; s.uniq_mapper_count = hc[1]; s.multi_mapper_count = hc[2];
    s.multi_lists = g.n_ranks > 1 ? (unsigned long long)hc[4] + ((unsigned long long)hc[5] << 16) : c->csr_lists;
    s.multi_entries = c->csr_ent;
    if (!em) s.multi_lists = s.multi_entries = 0;          // exact --multi=equal keeps lists of its own; they are not PropSharing's
    if (st) *st = s;
    return report_device_errors(c, c->h_pin + 8);
}

int msg_finish_coverage(msg_ctx *c, uint8_t *covered, int64_t *touched, int64_t *sum)
{
    if (!c) return MSG_EINVAL;
    if (!c->cfg.want_coverage) return fail(c, MSG_ESTATE, "context was created without want_coverage");
    CU(cudaSetDevice(c->cfg.device));
    { int wrc = wait_all(c); if (wrc) return wrc; }
    { int crc = collate_run(c); if (crc) return crc; }
    const msg_config &g = c->cfg;
    const size_t T = (size_t)g.n_targets;
    int rc;
    if (T == 0) return MSG_OK;
    if (c->cov_bits) {
        // summary mode: touched = popcount of every target's bitmap, sum = the run lengths added up during the pushes
        CU(cudaMemsetAsync(c->d_touched, 0, T * 8, c->stream));
        if (c->cov_words) {
            coverage_popcount_kernel<<<nblocks(nblocks(c->cov_words, 4), 256), 256, 0, c->stream>>>(c->d_covbits, c->cov_words, c->d_covbase, g.n_targets, c->d_touched);
            LAUNCHED(c);
        }
        if (covered) CU(cudaMemcpyAsync(covered, c->d_covered, T, cudaMemcpyDeviceToHost, c->stream));
        if (touched) CU(cudaMemcpyAsync(touched, c->d_touched, T * 8, cudaMemcpyDeviceToHost, c->stream));
        if (sum)     CU(cudaMemcpyAsync(sum, c->d_sum, T * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->d2h_bytes += T * 17;
        return check_device_errors(c);
    }
    CU(cudaMemcpyAsync(c->d_depth, c->d_diff, (size_t)c->cov_cells * 4, cudaMemcpyDeviceToDevice, c->stream));
    DevBuf &t_cov = c->t_cov;
    uint8_t *cov = c->d_covered;
    if (g.n_ranks > 1) {
        CU(t_cov.reserve(T));
        CU(cudaMemcpyAsync(t_cov.p, c->d_covered, T, cudaMemcpyDeviceToDevice, c->stream));
        cov = t_cov.as<uint8_t>();
        if ((rc = allreduce(c, c->d_depth, c->cov_cells, ncclInt32, ncclSum))) return rc;
        if ((rc = allreduce(c, cov, T, ncclUint8, ncclMax))) return rc;
    }
    rc = run_scan<int32_t>(c, InI32{c->d_depth}, OutInclI32{c->d_depth}, c->cov_cells, (int32_t *)nullptr);
    if (rc) return rc;
    CU(cudaMemsetAsync(c->d_touched, 0, T * 8, c->stream)); CU(cudaMemsetAsync(c->d_sum, 0, T * 8, c->stream));
    coverage_reduce_kernel<<<nblocks(nblocks(c->cov_cells, COV_SPAN), 256), 256, 0, c->stream>>>(c->d_depth, c->cov_cells, c->d_covbase, c->d_tlen,
                                                                                                 g.n_targets, c->d_touched, c->d_sum); LAUNCHED(c);
    if (covered) CU(cudaMemcpyAsync(covered, cov, T, cudaMemcpyDeviceToHost, c->stream));
    if (touched) CU(cudaMemcpyAsync(touched, c->d_touched, T * 8, cudaMemcpyDeviceToHost, c->stream));
    if (sum)     CU(cudaMemcpyAsync(sum, c->d_sum, T * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->d2h_bytes += T * 17;
    c->cov_finished = true;
    return check_device_errors(c);
}

int msg_pull_coverage(msg_ctx *c, int32_t tid, int32_t *depth)
{
    if (!c || !depth) return MSG_EINVAL;
    if (c->cov_bits) return fail(c, MSG_ESTATE, "context was created with coverage_summary: per-position depth is not kept");
    if (!c->cfg.want_coverage || !c->cov_finished) return fail(c, MSG_ESTATE, "call msg_finish_coverage first");
    if (tid < 0 || tid >= c->cfg.n_targets) return fail(c, MSG_EINVAL, "tid out of range");
    CU(cudaSetDevice(c->cfg.device));
    uint64_t base[2]; uint32_t tl;
    CU(cudaMemcpy(base, c->d_covbase + tid, 16, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&tl, c->d_tlen + tid, 4, cudaMemcpyDeviceToHost));
    if (tl) CU(cudaMemcpy(depth, c->d_depth + base[0], (size_t)tl * 4, cudaMemcpyDeviceToHost));
    return MSG_OK;
}

int msg_get_timing(msg_ctx *c, msg_timing *t, int reset)
{
    if (!c || !t) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    { int wrc = wait_all(c); if (wrc) return wrc; }
    CU(cudaStreamSynchronize(c->stream));
    harvest_events(c);
    unsigned long long acct[2] = {0, 0}, slots[ACCT_SLOTS * 16];
    CU(cudaMemcpy(slots, c->d_acct, sizeof slots, cudaMemcpyDeviceToHost));
    for (int k = 0; k < ACCT_SLOTS; k++) { acct[0] += slots[k * 16]; acct[1] += slots[k * 16 + 1]; }
    t->decode_ms = c->decode_ms; t->decode_launches = c->decode_launches; t->total_ms = c->total_ms;
    t->kernel_launches = c->kernel_launches; t->h2d_bytes = c->h2d_bytes; t->d2h_bytes = c->d2h_bytes;
    t->alg_bytes = acct[0]; t->slow_records = acct[1];
    t->fused_chunks = c->fused_chunks; t->fused_fallbacks = c->fused_fallbacks; t->zero_copy_chunks = c->zc_chunks;
    if (reset) {
        c->decode_ms = c->total_ms = 0; c->decode_launches = c->kernel_launches = 0; c->h2d_bytes = c->d2h_bytes = 0;
        c->fused_chunks = c->fused_fallbacks = 0; c->zc_chunks = 0;
        CU(cudaMemset(c->d_acct, 0, ACCT_SLOTS * 128));
    }
    return MSG_OK;
}

int msg_mark(msg_ctx *c, int slot)
{
    if (!c || slot < 0 || slot >= 8) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    if (!c->marks[slot]) CU(cudaEventCreate(&c->marks[slot]));
    CU(cudaEventRecord(c->marks[slot], c->stream));
    return MSG_OK;
}

int msg_elapsed_ms(msg_ctx *c, int a, int b, double *ms)
{
    if (!c || !ms || a < 0 || a >= 8 || b < 0 || b >= 8 || !c->marks[a] || !c->marks[b]) return MSG_EINVAL;
    CU(cudaSetDevice(c->cfg.device));
    CU(cudaEventSynchronize(c->marks[b]));
    float f = 0;
    CU(cudaEventElapsedTime(&f, c->marks[a], c->marks[b]));
    *ms = f;
    return MSG_OK;
}

} // extern "C"
