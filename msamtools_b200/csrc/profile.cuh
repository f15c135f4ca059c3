// profile.cuh -- K4/K5: insert counting over QNAME groups + multi-mapper sharing.
//
// Replaces mEstimateInsertCountOnFile (msam_profile.c:204-243), mEstimateInsertCountOnPool
// (:65-200) and the numeric part of mInsertCountToAbundanceMatrix (:248-425).
//
// The profile stage consumes a *stream* of records: either the chunk itself
// (plain `msamtools profile`) or the filter stage's kept list in reference output
// order (`filter | profile`), addressed through `stream[j]` (NULL = identity).
// A group is a maximal run of stream records with tid != -1 whose QNAME equals the
// previous such record's (:223-232).  Name equality is decided exactly without
// touching the record bytes again in the common case:
//   same QNAME run id (nid)            -> equal     (adjacent byte compares chained)
//   different run id, different hash   -> different
//   different run id, same 32-bit hash -> byte compare in global memory (rare)
// The group head walks its group, collects distinct features in first-appearance
// order (:136-142) and applies the share rule.  Proportional mode writes the feature
// lists into a CSR that the EM kernels iterate.
#pragma once
#include "common.cuh"
#include "collate.cuh"
#include <cooperative_groups.h>

namespace msg {

struct ProfParams {
    const uint8_t  *raw;
    const uint64_t *off;
    const uint32_t *stream;      // may be null (identity)
    uint64_t m;                  // stream length
    const int32_t  *tid;
    const uint32_t *nid;
    const uint32_t *hash;
    const int32_t  *fmap;        // may be null (identity)
    int32_t n_targets, n_features;
    int share_type;
    uint32_t *ui;                // [F]
    double   *d;                 // [F]
    uint32_t *counters;          // [0] inserts [1] uniq [2] multi [3] big groups
    uint32_t *pcount;            // [m] list length at group heads (proportional), else 0
    uint32_t *big;               // [big_cap] stream positions of oversized groups
    uint32_t big_cap;
    uint32_t big_threshold;
    uint32_t *err;
    unsigned long long *key;     // exact mode: [list] key_base + stream position of the list's group head (its input order)
    unsigned long long key_base; // records pushed before this chunk
};

__device__ __forceinline__ uint32_t stream_at(const ProfParams &p, uint64_t j) { return p.stream ? p.stream[j] : (uint32_t)j; }

__device__ bool qname_equal_global(const uint8_t *raw, const uint64_t *off, uint32_t a, uint32_t b)
{
    const uint8_t *pa = raw + off[a], *pb = raw + off[b];
    uint32_t la = pa[12], lb = pb[12];
    if (la != lb) return false;
    for (uint32_t k = 0; k < la; k++) if (pa[36 + k] != pb[36 + k]) return false;
    return true;
}

__device__ __forceinline__ bool same_name(const ProfParams &p, uint32_t a, uint32_t b)
{
    if (p.nid[a] == p.nid[b]) return true;
    if (p.hash[a] != p.hash[b]) return false;
    return qname_equal_global(p.raw, p.off, a, b);
}

__device__ __forceinline__ int32_t feature_of(const ProfParams &p, int32_t t) { return p.fmap ? p.fmap[t] : t; }

constexpr int PROF_CACHE = 8;

// Walk the group headed at stream position j.  act(f, k) is called for the k-th
// distinct feature in first-appearance order.  Returns #distinct; *size_out = group size;
// *end_out = stream position after the group's last record.
template <class Act>
__device__ __forceinline__ uint32_t walk_group(const ProfParams &p, uint64_t j, uint32_t r0, uint32_t *size_out, Act act, uint32_t max_size)
{
    int32_t cache[PROF_CACHE];
#pragma unroll
    for (int k = 0; k < PROF_CACHE; k++) cache[k] = -1;
    uint32_t nd = 0, size = 0;
    for (uint64_t jj = j; jj < p.m; jj++) {
        uint32_t rr = (jj == j) ? r0 : stream_at(p, jj);
        int32_t tt = p.tid[rr];
        if (tt == -1) continue;                                          // msam_profile.c:223-225
        if (jj != j && !same_name(p, r0, rr)) break;                     // :226
        if (tt < 0 || tt >= p.n_targets) { atomicOr(p.err, DERR_FORMAT); break; }
        size++;
        if (size > max_size) break;                                      // oversized: caller defers to the serial kernel
        int32_t f = feature_of(p, tt);
        bool seen = false;
#pragma unroll
        for (int k = 0; k < PROF_CACHE; k++) seen |= (cache[k] == f);
        if (!seen && nd >= PROF_CACHE) {
            // cache full: rescan the group's earlier records (exact, O(size) per probe)
            for (uint64_t q = j; q < jj && !seen; q++) {
                uint32_t rq = (q == j) ? r0 : stream_at(p, q);
                int32_t tq = p.tid[rq];
                if (tq == -1) continue;
                seen = feature_of(p, tq) == f;
            }
        }
        if (!seen) {
#pragma unroll
            for (int k = 0; k < PROF_CACHE; k++) if ((uint32_t)k == nd) cache[k] = f;
            act(f, nd);
            nd++;
        }
    }
    *size_out = size;
    return nd;
}

struct ActNone  { __device__ __forceinline__ void operator()(int32_t, uint32_t) const {} };
struct ActFirst { int32_t *f0, *f1; __device__ __forceinline__ void operator()(int32_t f, uint32_t k) const { if (k == 0) *f0 = f; if (k == 1) *f1 = f; } };
struct ActAddUi { uint32_t *ui; uint32_t v; __device__ __forceinline__ void operator()(int32_t f, uint32_t) const { atomicAdd(ui + f, v); } };
struct ActAddD  { double *d; double v; __device__ __forceinline__ void operator()(int32_t f, uint32_t) const { atomicAdd(d + f, v); } };
struct ActStore { int32_t *dst; __device__ __forceinline__ void operator()(int32_t f, uint32_t k) const { dst[k] = f; } };

// is stream position j a group head?  (prev valid record has a different QNAME, or none)
__device__ __forceinline__ bool group_head(const ProfParams &p, uint64_t j, uint32_t r)
{
    for (uint64_t k = j; k-- > 0;) {
        uint32_t rk = stream_at(p, k);
        if (p.tid[rk] == -1) continue;
        return !same_name(p, rk, r);
    }
    return true;
}

// ---- head-walks-its-group path (worklist fallback; exact for any group size) ----------------
// Applies the share rule of the group headed at stream position j; returns list length for
// proportional mode (0 otherwise).  ins/uq/mu are incremented for the caller's counters.
// EXACT (msg_config.exact): an insert that would add 1/n to d[] becomes a list instead (d is summed at finish, in order).
template <bool EXACT>
__device__ __forceinline__ uint32_t count_group_walk(const ProfParams &p, uint64_t j, uint32_t r, uint32_t &ins, uint32_t &uq, uint32_t &mu)
{
    int32_t f0 = -1, f1 = -1; uint32_t size = 0, pc = 0;
    const uint32_t nd = walk_group(p, j, r, &size, ActFirst{&f0, &f1}, p.big_threshold);
    if (size > p.big_threshold) {
        const uint32_t slot = atomicAdd(p.counters + 3, 1u);
        if (slot < p.big_cap) p.big[slot] = (uint32_t)j;
    } else if (size > 0) {
        ins++;
        if (nd == 1) { atomicAdd(p.ui + f0, 2u); uq++; }                                       // :75-78,87-91,152-159
        else {
            mu++;
            switch (p.share_type) {
            case 1: walk_group(p, j, r, &size, ActAddUi{p.ui, 2u}, p.big_threshold); break;               // :99-102,169-173
            case 2:
                if (size == 2) { atomicAdd(p.ui + f0, 1u); atomicAdd(p.ui + f1, 1u); }                    // :103-106
                else if (EXACT) pc = nd;
                else walk_group(p, j, r, &size, ActAddD{p.d, 1.0 / (int)nd}, p.big_threshold);            // :175-182
                break;
            case 3: pc = nd; break;                                                                        // :107-121,184-186
            default: break;                                                                                // ignore
            }
        }
    }
    return pc;
}

template <bool EXACT>
__global__ void __launch_bounds__(256) profile_walk_count_kernel(const ProfParams p, const uint32_t *worklist, const uint32_t *wl_count)
{
    const uint32_t nw = *wl_count;
    uint32_t ins = 0, uq = 0, mu = 0;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nw; q += gridDim.x * blockDim.x) {
        const uint64_t j = worklist[q];
        const uint32_t pc = count_group_walk<EXACT>(p, j, stream_at(p, j), ins, uq, mu);
        if (p.pcount) p.pcount[j] = pc;
    }
    ins = __reduce_add_sync(0xffffffffu, ins); uq = __reduce_add_sync(0xffffffffu, uq); mu = __reduce_add_sync(0xffffffffu, mu);
    if ((threadIdx.x & 31u) == 0) {      // one set of atomics per warp, not per thread
        if (ins) atomicAdd(p.counters + 0, ins);
        if (uq)  atomicAdd(p.counters + 1, uq);
        if (mu)  atomicAdd(p.counters + 2, mu);
    }
}

// proportional: worklist heads with pcount>0 write their list; scanv[j] = (lists before << 32) | entries before
template <bool EXACT>
__global__ void __launch_bounds__(256) profile_walk_fill_kernel(const ProfParams p, const unsigned long long *scanv, uint32_t *mm_off, uint32_t *mm_len, int32_t *mm_fid,
                                                                uint32_t list_base, uint32_t ent_base, const uint32_t *worklist, const uint32_t *wl_count)
{
    const uint32_t nw = *wl_count;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nw; q += gridDim.x * blockDim.x) {
        const uint64_t j = worklist[q];
        if (p.pcount[j] == 0) continue;
        const unsigned long long sv = scanv[j];
        const uint32_t li = list_base + (uint32_t)(sv >> 32), eo = ent_base + (uint32_t)sv;
        mm_off[li] = eo; mm_len[li] = p.pcount[j];
        if (EXACT) p.key[li] = p.key_base + j;
        uint32_t size;
        walk_group(p, j, stream_at(p, j), &size, ActStore{mm_fid + eo}, p.big_threshold);
    }
}

// ---- main path: one stream record per lane ---------------------------------------------------
// Group heads come from comparing every valid record (tid != -1) with the previous valid one
// (shuffle for neighbours in the window, a short look-back for the window's first); lanes of
// the same (group, feature) find each other with MATCH.ANY, the lowest lane of each match set is
// the feature's first appearance (msam_profile.c:136-142), and popc of those gives the number
// of distinct features.  Groups that leave the 32-record window go to the worklist.
constexpr uint8_t GM_MEMBER = 1, GM_HEAD = 2, GM_FIRST = 4;

struct GroupView {
    uint32_t gmask, gs;      // valid lanes of my group in this window, lane of its head
    bool member;             // valid record of a group that lies entirely inside the window
    bool head;               // ... and I am its head
    bool open_head;          // head of a group that leaves the window on the right
    int32_t feat;            // my feature id (members only)
    uint32_t r;
};

__device__ __forceinline__ GroupView group_view(const ProfParams &p, uint64_t j, uint64_t w0)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t NONE = 0xffffffffu;
    GroupView v;
    const bool inb = j < p.m;
    v.r = inb ? stream_at(p, j) : 0u;
    int32_t t = inb ? p.tid[v.r] : -1;
    bool valid = inb && t != -1;                                                     // msam_profile.c:223-225
    if (valid && (t < 0 || t >= p.n_targets)) { atomicOr(p.err, DERR_FORMAT); valid = false; }
    const uint32_t mynid = valid ? p.nid[v.r] : 0u, myhash = valid ? p.hash[v.r] : 0u;
    const uint32_t vmask = __ballot_sync(0xffffffffu, valid);

    // previous / next valid record outside the window (lane 0 looks back, lane 31 looks ahead)
    uint32_t out_r = NONE, out_nid = 0, out_hash = 0;
    if (lane == 0) {
        for (uint64_t k = w0; k-- > 0;) { const uint32_t rk = stream_at(p, k); if (p.tid[rk] != -1) { out_r = rk; break; } }
    } else if (lane == 31) {
        for (uint64_t k = w0 + 32; k < p.m; k++) { const uint32_t rk = stream_at(p, k); if (p.tid[rk] != -1) { out_r = rk; break; } }
    }
    if ((lane == 0 || lane == 31) && out_r != NONE) { out_nid = p.nid[out_r]; out_hash = p.hash[out_r]; }
    const uint32_t prev_r = __shfl_sync(0xffffffffu, out_r, 0), prev_nid = __shfl_sync(0xffffffffu, out_nid, 0), prev_hash = __shfl_sync(0xffffffffu, out_hash, 0);
    const uint32_t next_r = __shfl_sync(0xffffffffu, out_r, 31), next_nid = __shfl_sync(0xffffffffu, out_nid, 31), next_hash = __shfl_sync(0xffffffffu, out_hash, 31);

    // compare with the previous valid record (:226)
    const uint32_t lowv = vmask & ((1u << lane) - 1u);
    const int pl = lowv ? 31 - __clz((int)lowv) : 0;
    uint32_t pn = __shfl_sync(0xffffffffu, mynid, pl), ph = __shfl_sync(0xffffffffu, myhash, pl), pr = __shfl_sync(0xffffffffu, v.r, pl);
    bool have_prev = lowv != 0;
    if (!have_prev) { pn = prev_nid; ph = prev_hash; pr = prev_r; have_prev = prev_r != NONE; }
    bool same = false;
    if (valid && have_prev) same = (mynid == pn) || (myhash == ph && qname_equal_global(p.raw, p.off, v.r, pr));
    const bool ghead = valid && !same;
    const uint32_t hmask = __ballot_sync(0xffffffffu, ghead);

    const uint32_t le = hmask & (0xffffffffu >> (31u - lane));
    const uint32_t gt = lane == 31 ? 0u : (hmask & (0xffffffffu << (lane + 1)));
    const bool open_left = le == 0;
    v.gs = open_left ? 0u : 31u - (uint32_t)__clz((int)le);
    const uint32_t e = gt ? (uint32_t)__ffs((int)gt) - 1u : 32u;
    v.gmask = vmask & (e == 32 ? 0xffffffffu : ((1u << e) - 1u)) & (0xffffffffu << v.gs);
    // does the window's last group continue?  compare the next valid record with the last valid lane
    const int ll = vmask ? 31 - __clz((int)vmask) : 0;
    const uint32_t ln = __shfl_sync(0xffffffffu, mynid, ll), lh = __shfl_sync(0xffffffffu, myhash, ll), lr = __shfl_sync(0xffffffffu, v.r, ll);
    bool tail_same = false;                                                          // warp-uniform
    if (next_r != NONE && vmask) tail_same = (ln == next_nid) || (lh == next_hash && qname_equal_global(p.raw, p.off, lr, next_r));
    const bool open_right = gt == 0 && tail_same;
    v.member = valid && !open_left && !open_right;
    v.head = v.member && lane == v.gs;
    v.open_head = valid && !open_left && open_right && lane == v.gs;
    v.feat = valid ? feature_of(p, t) : -1;
    return v;
}

template <bool SMEM_HIST, bool EXACT>
__global__ void __launch_bounds__(256) profile_warp_count_kernel(const ProfParams p, uint8_t *gmeta, uint32_t *worklist, uint32_t *wl_count)
{
    extern __shared__ uint32_t s_hist[];                 // SMEM_HIST: CTA-private ui histogram (small feature sets)
    __shared__ uint32_t s_cnt[3];
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    if (SMEM_HIST) for (uint32_t k = threadIdx.x; k < (uint32_t)p.n_features; k += blockDim.x) s_hist[k] = 0;
    __syncthreads();
    uint32_t *ui = SMEM_HIST ? s_hist : p.ui;

    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t w0 = j & ~31ull;
    const uint32_t lane = threadIdx.x & 31u;
    if (w0 < p.m) {
        const GroupView v = group_view(p, j, w0);
        if (v.open_head) { const uint32_t slot = atomicAdd(wl_count, 1u); worklist[slot] = (uint32_t)j; }
        __syncwarp();
        const unsigned long long key = v.member ? (((unsigned long long)v.gs << 32) | (uint32_t)v.feat) : ((1ull << 40) | lane);
        const uint32_t mm = __match_any_sync(0xffffffffu, key);
        const bool first = v.member && lane == (uint32_t)__ffs((int)mm) - 1u;                       // first appearance of this feature
        const uint32_t fm = __ballot_sync(0xffffffffu, first) & v.gmask;
        const uint32_t nd = __popc(fm), size = __popc(v.gmask);
        const bool multi = nd > 1;
        uint32_t pc = 0;
        if (v.member) {
            if (!multi) { if (v.head) atomicAdd(ui + v.feat, 2u); }                                 // :75-78,87-91,152-159
            else if (first) {
                if (p.share_type == 1) atomicAdd(ui + v.feat, 2u);                                   // :99-102,169-173
                else if (p.share_type == 2) {
                    if (size == 2) atomicAdd(ui + v.feat, 1u);                                       // :103-106
                    else if (!EXACT) atomicAdd(p.d + v.feat, 1.0 / (int)nd);                         // :175-182
                }
            }
            if (v.head && multi && p.share_type == 3) pc = nd;                                       // :107-121,184-186
            if (EXACT && v.head && multi && p.share_type == 2 && size != 2) pc = nd;
        }
        if (j < p.m) {
            if (p.pcount) p.pcount[j] = pc;
            if (gmeta) gmeta[j] = (uint8_t)((v.member ? GM_MEMBER : 0) | (v.head ? GM_HEAD : 0) | (first ? GM_FIRST : 0));
        }
        const uint32_t heads = __ballot_sync(0xffffffffu, v.head);
        const uint32_t mheads = __ballot_sync(0xffffffffu, v.head && multi);
        if (lane == 0 && heads) {
            atomicAdd(&s_cnt[0], (uint32_t)__popc(heads));
            atomicAdd(&s_cnt[1], (uint32_t)__popc(heads & ~mheads));
            atomicAdd(&s_cnt[2], (uint32_t)__popc(mheads));
        }
    }
    __syncthreads();
    if (threadIdx.x < 3 && s_cnt[threadIdx.x]) atomicAdd(p.counters + threadIdx.x, s_cnt[threadIdx.x]);
    if (SMEM_HIST) for (uint32_t k = threadIdx.x; k < (uint32_t)p.n_features; k += blockDim.x) { const uint32_t c = s_hist[k]; if (c) atomicAdd(p.ui + k, c); }
}

// proportional: first-appearance lanes of in-window multi groups write their feature at
// (list offset of the head) + (rank among the group's first appearances)
template <bool EXACT>
__global__ void __launch_bounds__(256) profile_warp_fill_kernel(const ProfParams p, const uint8_t *gmeta, const unsigned long long *scanv,
                                                                uint32_t *mm_off, uint32_t *mm_len, int32_t *mm_fid, uint32_t list_base, uint32_t ent_base)
{
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t w0 = j & ~31ull;
    if (w0 >= p.m) return;
    const uint32_t lane = threadIdx.x & 31u;
    const uint8_t g = j < p.m ? gmeta[j] : 0;
    const uint32_t pc = j < p.m ? p.pcount[j] : 0u;
    const bool head = (g & GM_HEAD) != 0, first = (g & GM_FIRST) != 0, member = (g & GM_MEMBER) != 0;
    const uint32_t hmask = __ballot_sync(0xffffffffu, head);
    const uint32_t fmask = __ballot_sync(0xffffffffu, first);
    const uint32_t le = hmask & (0xffffffffu >> (31u - lane));
    const uint32_t gs = le ? 31u - (uint32_t)__clz((int)le) : 0u;
    const uint32_t gt = lane == 31 ? 0u : (hmask & (0xffffffffu << (lane + 1)));
    const uint32_t e = gt ? (uint32_t)__ffs((int)gt) - 1u : 32u;
    const uint32_t span = (e == 32 ? 0xffffffffu : ((1u << e) - 1u)) & (0xffffffffu << gs);
    unsigned long long sv = (head && pc) ? scanv[j] : 0ull;
    const uint32_t hpc = __shfl_sync(0xffffffffu, pc, (int)gs);
    sv = __shfl_sync(0xffffffffu, sv, (int)gs);
    if (member && le && hpc) {
        const uint32_t li = list_base + (uint32_t)(sv >> 32), eo = ent_base + (uint32_t)sv;
        if (head) { mm_off[li] = eo; mm_len[li] = hpc; if (EXACT) p.key[li] = p.key_base + j; }
        if (first) {
            const uint32_t rank = __popc(fmask & span & ((1u << lane) - 1u));
            mm_fid[eo + rank] = feature_of(p, p.tid[stream_at(p, j)]);
        }
    }
}

// Oversized groups (> big_threshold records): one thread, the reference's own
// ub_target_hit stamp algorithm (msam_profile.c:131-145) with a u32 stamp per feature.
// Lists for proportional mode (and, EXACT, the equal-share lists) are appended to big_fid / big_off.
template <bool EXACT>
__global__ void profile_big_kernel(const ProfParams p, uint32_t nbig, uint32_t *stamp, uint32_t stamp_base,
                                   uint32_t *big_off, uint32_t *big_len, int32_t *big_fid, uint32_t *big_tot /*[0]=lists,[1]=entries*/, int fill,
                                   uint32_t list_base, uint32_t ent_base)
{
    if (blockIdx.x || threadIdx.x) return;
    const bool lists = p.share_type == 3 || (EXACT && p.share_type == 2);
    uint32_t nl = fill ? list_base : 0, ne = fill ? ent_base : 0;
    for (uint32_t b = 0; b < nbig; b++) {
        const uint64_t j = p.big[b];
        const uint32_t r0 = stream_at(p, j);
        const uint32_t st = stamp_base + b + 1;
        uint32_t nd = 0, size = 0;
        uint32_t e0 = ne;
        for (uint64_t jj = j; jj < p.m; jj++) {
            uint32_t rr = stream_at(p, jj);
            int32_t tt = p.tid[rr];
            if (tt == -1) continue;
            if (jj != j && !same_name(p, r0, rr)) break;
            if (tt < 0 || tt >= p.n_targets) { atomicOr(p.err, DERR_FORMAT); break; }
            size++;
            int32_t f = feature_of(p, tt);
            if (stamp[f] != st) {
                stamp[f] = st;
                if (fill && lists) big_fid[ne] = f;
                ne++; nd++;
            }
        }
        if (!fill) {
            // counting pass applies the non-proportional share rules and the counters once
            atomicAdd(p.counters + 0, 1u);
            if (nd == 1) { atomicAdd(p.ui + feature_of(p, p.tid[r0]), 2u); atomicAdd(p.counters + 1, 1u); ne = e0; }
            else {
                atomicAdd(p.counters + 2, 1u);
                if (p.share_type == 1 || (!EXACT && p.share_type == 2)) {
                    // second walk with a fresh stamp to apply the adds
                    const uint32_t st2 = st | 0x80000000u;
                    for (uint64_t jj = j; jj < p.m; jj++) {
                        uint32_t rr = stream_at(p, jj);
                        int32_t tt = p.tid[rr];
                        if (tt == -1) continue;
                        if (jj != j && !same_name(p, r0, rr)) break;
                        if (tt < 0 || tt >= p.n_targets) break;
                        int32_t f = feature_of(p, tt);
                        if (stamp[f] != st2) {
                            stamp[f] = st2;
                            if (p.share_type == 1) atomicAdd(p.ui + f, 2u);
                            else atomicAdd(p.d + f, 1.0 / (int)nd);
                        }
                    }
                }
                if (!lists) ne = e0;
            }
            if (lists && nd > 1) nl++;
        } else {
            if (nd == 1 || !lists) ne = e0;
            else { big_off[nl] = e0; big_len[nl] = ne - e0; if (EXACT) p.key[nl] = p.key_base + j; nl++; }
        }
    }
    if (!fill) { big_tot[0] = nl; big_tot[1] = ne; }
}

// ---------------------------------------------------------------- abundance / EM (msam_profile.c:284-404)
// also clears what the single-GPU loop kernel expects to find zeroed (inc[F], delta[20], result[4]), so
// that PropSharing needs no separate memset launches
__global__ void em_init_kernel(const uint32_t *ui, const double *d, int use_d, double *U, double *a, uint32_t n,
                               double *inc, double *delta, int32_t *result)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 20 && delta) delta[i] = 0.0;
    if (i < 4 && result) result[i] = 0;
    if (i >= n) return;
    double u = 1.0 * ui[i] / 2;                                         // :286
    if (use_d) u += d[i];                                               // :305
    U[i] = u; a[i] = u;
    if (inc) { inc[i] = 0.0; inc[(size_t)n + i] = 0.0; inc[2 * (size_t)n + i] = 0.0; }      // three buffers (em_loop_smem_kernel)
}
// Small feature sets (genomes, F <= EM_SMEM_F): millions of lists hit a few hundred addresses.
// Each CTA keeps a private copy of a[] and inc[] in shared memory and flushes inc once.
// Large catalogs (F up to 1e6): the F-sized vectors live in L2, contention per address is low,
// so the adds go straight to global memory.
constexpr uint32_t EM_SMEM_F = 2048;
// private inc copies per CTA: one per warp while that stays under ~40 KB
__host__ __device__ __forceinline__ uint32_t em_copies(uint32_t F) { return F <= 512 ? 8u : 1u; }
// dynamic shared memory of a gather that works from shared memory: a[F] | inc copies [em_copies(F)][F]
__host__ __device__ __forceinline__ size_t em_smem_bytes(uint32_t F) { return F <= EM_SMEM_F ? (size_t)F * 8 * (1 + em_copies(F)) : 0; }

// One multi-mapper list in one PropSharing iteration: s = sum of a[f] in list order, inc[f] += a[f] / s (:341-365).
// The first four features (almost every list) stay in registers between the two passes; the share is a[f] * (1/s),
// one division per list instead of one per entry (<= 1 ulp from a[f]/s, far inside the 1e-9 tolerance).
__device__ __forceinline__ void em_share_list(const int32_t *mm_fid, uint32_t b, uint32_t n, const double *av, double *iv)
{
    int32_t fr[4]; double ar[4];
    double sum = 0;
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) if (j < n) { fr[j] = mm_fid[b + j]; ar[j] = av[fr[j]]; sum += ar[j]; }
    for (uint32_t q = 4; q < n; q++) sum += av[mm_fid[b + q]];
    if (!(sum > 0)) return;
    const double inv = 1.0 / sum;
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) if (j < n) atomicAdd(iv + fr[j], ar[j] * inv);
    for (uint32_t q = 4; q < n; q++) { const int32_t f = mm_fid[b + q]; atomicAdd(iv + f, av[f] * inv); }
}

// Two lists at once: the gather is latency bound (offsets -> features -> shared a[] -> divide -> atomics), so a
// thread keeps the loads of two independent lists in flight.  Same arithmetic per list as em_share_list.
__device__ __forceinline__ void em_share_list_pair(const int32_t *mm_fid, uint32_t b0, uint32_t n0, uint32_t b1, uint32_t n1,
                                                   const double *av, double *iv)
{
    int32_t f0[4], f1[4]; double a0[4], a1[4];
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) { f0[j] = j < n0 ? mm_fid[b0 + j] : 0; f1[j] = j < n1 ? mm_fid[b1 + j] : 0; }
    double s0 = 0, s1 = 0;
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) { if (j < n0) { a0[j] = av[f0[j]]; s0 += a0[j]; } if (j < n1) { a1[j] = av[f1[j]]; s1 += a1[j]; } }
    for (uint32_t q = 4; q < n0; q++) s0 += av[mm_fid[b0 + q]];
    for (uint32_t q = 4; q < n1; q++) s1 += av[mm_fid[b1 + q]];
    const double i0 = s0 > 0 ? 1.0 / s0 : 0.0, i1 = s1 > 0 ? 1.0 / s1 : 0.0;
    if (s0 > 0) {
#pragma unroll
        for (uint32_t j = 0; j < 4; j++) if (j < n0) atomicAdd(iv + f0[j], a0[j] * i0);
        for (uint32_t q = 4; q < n0; q++) { const int32_t f = mm_fid[b0 + q]; atomicAdd(iv + f, av[f] * i0); }
    }
    if (s1 > 0) {
#pragma unroll
        for (uint32_t j = 0; j < 4; j++) if (j < n1) atomicAdd(iv + f1[j], a1[j] * i1);
        for (uint32_t q = 4; q < n1; q++) { const int32_t f = mm_fid[b1 + q]; atomicAdd(iv + f, av[f] * i1); }
    }
}

// The gather of one iteration (:341-365) over this thread's lists of a grid-stride walk (first, first + stride, ...):
// lists l and l + stride as a pair, then at most one lone list.
__device__ __forceinline__ void em_share_lists(uint32_t first, uint32_t stride, const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid,
                                               uint32_t nlists, const double *av, double *iv)
{
    uint32_t l = first;
    for (; l + stride < nlists; l += 2 * stride) em_share_list_pair(mm_fid, mm_off[l], mm_len[l], mm_off[l + stride], mm_len[l + stride], av, iv);
    if (l < nlists) em_share_list(mm_fid, mm_off[l], mm_len[l], av, iv);
}

// The gather with F <= EM_SMEM_F: sa[F] holds a[] (written before the call by this CTA), si[] the em_copies(F) private
// inc copies.  With few features every warp gets a copy of its own, so the (CAS-loop) f64 shared atomics only collide
// inside a warp.  The summed copies are added to the global inc[] = inc_at() once per CTA.  inc_at is called after the
// walk: a triple-buffer pointer formed before it and held across it makes em_loop_smem_kernel spill.
template <class IncAt>
__device__ __forceinline__ void em_gather_smem(uint32_t first, uint32_t stride, const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid,
                                               uint32_t nlists, const double *sa, double *si, IncAt inc_at, uint32_t F)
{
    const uint32_t ncopy = em_copies(F);
    for (uint32_t i = threadIdx.x; i < F * ncopy; i += blockDim.x) si[i] = 0.0;
    __syncthreads();
    em_share_lists(first, stride, mm_off, mm_len, mm_fid, nlists, sa, si + (size_t)((threadIdx.x >> 5) % ncopy) * F);
    __syncthreads();
    double *inc = inc_at();
    for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) {
        double v = 0.0;
        for (uint32_t cp = 0; cp < ncopy; cp++) v += si[(size_t)cp * F + i];
        if (v != 0.0) atomicAdd(inc + i, v);
    }
}

// Sum of v over the 256 threads of the CTA, in one fixed tree order, so that every CTA that sums the same values gets
// the same bits (and takes the same stop decision).  The caller synchronises before it writes s_red again.
__device__ __forceinline__ double em_block_sum(double *s_red, double v)
{
    s_red[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) s_red[threadIdx.x] += s_red[threadIdx.x + o]; __syncthreads(); }
    return s_red[0];
}

// a_new = U + inc, flushed to 0 below 1e-20  (:369-376)
__device__ __forceinline__ double em_new_abundance(double u, double inc)
{
    const double an = u + inc;
    return an < 1e-20 ? 0.0 : an;
}

// purged = #lists whose final abundances sum to exactly 0  (:394-404): this thread's lists of a grid-stride walk,
// one atomic per warp into *purged
__device__ __forceinline__ void em_count_purged(uint32_t first, uint32_t stride, const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid,
                                                uint32_t nlists, const double *av, uint32_t *purged)
{
    uint32_t z = 0;
    for (uint32_t l = first; l < nlists; l += stride) {
        const uint32_t b = mm_off[l], e = b + mm_len[l];
        double sum = 0;
        for (uint32_t q = b; q < e; q++) sum += av[mm_fid[q]];
        z += (sum == 0);
    }
    z = __reduce_add_sync(0xffffffffu, z);
    if ((threadIdx.x & 31u) == 0 && z) atomicAdd(purged, z);
}

// The host loop (NCCL fallback): one launch per phase.  Gather, with a[] copied into shared memory for F <= EM_SMEM_F.
__global__ void __launch_bounds__(256) em_gather_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                        const double *a, double *inc, uint32_t F)
{
    extern __shared__ double s_em[];
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    if (F <= EM_SMEM_F) {
        for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) s_em[i] = a[i];
        em_gather_smem(gtid, gsz, mm_off, mm_len, mm_fid, nlists, s_em, s_em + F, [&] { return inc; }, F);
    } else em_share_lists(gtid, gsz, mm_off, mm_len, mm_fid, nlists, a, inc);
}
// a = U + inc; per-block partial of sum (a_new - a_old)^2 in a fixed order  (:369-379)
__global__ void __launch_bounds__(256) em_update_kernel(const double *U, const double *inc, double *a, double *partial, uint32_t n)
{
    __shared__ double s_red[256];
    uint32_t i = blockIdx.x * 256 + threadIdx.x;
    double dd = 0;
    if (i < n) {
        const double an = em_new_abundance(U[i], inc[i]);
        const double diff = an - a[i];
        dd = diff * diff;
        a[i] = an;
    }
    const double sum = em_block_sum(s_red, dd);
    if (threadIdx.x == 0) partial[blockIdx.x] = sum;
}
__global__ void __launch_bounds__(256) em_delta_kernel(const double *partial, uint32_t nblocks, uint32_t n, double *delta_out)
{
    __shared__ double s_red[256];
    double acc = 0;
    for (uint32_t b = threadIdx.x; b < nblocks; b += 256) acc += partial[b];
    const double sum = em_block_sum(s_red, acc);
    if (threadIdx.x == 0) *delta_out = sum / n;                         // :380
}
__global__ void __launch_bounds__(256) em_purged_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                        const double *a, uint32_t *purged)
{
    em_count_purged(blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x, mm_off, mm_len, mm_fid, nlists, a, purged);
}

// The whole PropSharing loop (msam_profile.c:331-389) in ONE cooperative launch (single-GPU case): grid-wide
// barriers replace the per-iteration launches and the host's read of delta.  Every CTA recomputes delta from the
// per-CTA partials in the same fixed order, so all of them take the same stop decision.  result[0] = last k,
// result[1] = converged flag; delta_out[k-1] = DELTA^2 of iteration k.
__global__ void __launch_bounds__(256) em_loop_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                      const double *U, double *a, double *inc, double *partial, uint32_t F,
                                                      double *delta_out, int32_t *result)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double s_red[256];
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    int k = 1, conv = 0;
    for (; k < 20; k++) {
        em_share_lists(gtid, gsz, mm_off, mm_len, mm_fid, nlists, a, inc);
        grid.sync();
        // update: a = U + inc, per-CTA partial of sum diff^2; inc is cleared for the next iteration   (:369-379)
        double dd = 0;
        for (uint32_t i = gtid; i < F; i += gsz) {
            const double an = em_new_abundance(U[i], inc[i]);
            const double diff = an - a[i];
            dd += diff * diff;
            a[i] = an; inc[i] = 0.0;
        }
        const double part = em_block_sum(s_red, dd);
        if (threadIdx.x == 0) partial[blockIdx.x] = part;
        grid.sync();
        // delta (every CTA, same order)                                   (:380-383)
        double acc = 0;
        for (uint32_t b = threadIdx.x; b < gridDim.x; b += 256) acc += partial[b];
        const double delta = em_block_sum(s_red, acc) / F;
        __syncthreads();
        if (gtid == 0) delta_out[k - 1] = delta;
        if (delta < 1e-10) { conv = 1; break; }
    }
    if (gtid == 0) { result[0] = k < 20 ? k : 19; result[1] = conv; }
    // a[] is final and visible (second grid.sync above)
    em_count_purged(gtid, gsz, mm_off, mm_len, mm_fid, nlists, a, reinterpret_cast<uint32_t *>(result + 3));
}

// Single GPU, F <= EM_SMEM_F: the loop with ONE grid barrier per iteration.  Every CTA keeps the whole abundance vector
// in shared memory and, after the barrier that completes inc[], redoes the (tiny) update a = U + inc and the delta
// reduction for ALL features itself -- same data, same order, so every CTA holds bit-identical a[] and takes the same
// stop decision without a second barrier or a partial-sum array.  inc[] is triple buffered: CTA 0 clears buffer
// (k+2) % 3 after barrier k; its last readers (update k-1) are before barrier k, its next writers (gather k+2) after
// barrier k+1.  inc3 must arrive zeroed (3 * F doubles).
__global__ void __launch_bounds__(256) em_loop_smem_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                           const double *U, double *a, double *inc3, uint32_t F,
                                                           double *delta_out, int32_t *result)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    extern __shared__ double s_em[];
    __shared__ double s_red[256];
    double *sa = s_em;
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) sa[i] = a[i];
    int k = 1, conv = 0;
    for (; k < 20; k++) {
        em_gather_smem(gtid, gsz, mm_off, mm_len, mm_fid, nlists, sa, s_em + F, [&] { return inc3 + (size_t)(k % 3) * F; }, F);
        grid.sync();
        const double *inc = inc3 + (size_t)(k % 3) * F;
        if (blockIdx.x == 0) { double *nxt = inc3 + (size_t)((k + 2) % 3) * F; for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) nxt[i] = 0.0; }
        // update (every CTA, all features): a = U + inc, delta = sum diff^2 / F   (:369-383)
        double dd = 0;
        for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) {
            const double an = em_new_abundance(U[i], __ldcg(inc + i));
            const double diff = an - sa[i];
            dd += diff * diff;
            sa[i] = an;
        }
        const double delta = em_block_sum(s_red, dd) / F;
        __syncthreads();
        if (gtid == 0) delta_out[k - 1] = delta;
        if (delta < 1e-10) { conv = 1; break; }
    }
    if (blockIdx.x == 0) for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) a[i] = sa[i];
    if (gtid == 0) { result[0] = k < 20 ? k : 19; result[1] = conv; }
    // from this CTA's own (identical) copy of a[]
    em_count_purged(gtid, gsz, mm_off, mm_len, mm_fid, nlists, sa, reinterpret_cast<uint32_t *>(result + 3));
}

// ---------------------------------------------------------------- exact mode (msg_config.exact)
// The reference adds every feature's shares in the input order of the lists (msam_profile.c:341-365, :175-182).  Exact
// mode does the same: the per-feature incidence ibeg[f] .. ibeg[f+1] of ilist[] holds the lists that contain f, sorted by
// their input key (built once per finish after pushes, from a histogram, run_scan, a scatter and collate.cuh's bucket
// sorts), and each feature's shares are added in that order, one after another.  Every f64 operation is uncontracted
// (__dadd_rn / __dmul_rn / __ddiv_rn): the reference's x86-64 build does not fuse a*b + c.  With the same IEEE
// operations in the same order, abundances, deltas and stop decisions are bit-identical to the reference's.

// the incidence of one feature: lists ilist[b .. e); e of the last feature is the entry total
__device__ __forceinline__ void exact_range(const uint32_t *ibeg, uint32_t F, unsigned long long nent, uint32_t f, uint32_t &b, uint32_t &e)
{
    b = ibeg[f]; e = f + 1 < F ? ibeg[f + 1] : (uint32_t)nent;
}

// transpose, step 1: entries per feature
__global__ void __launch_bounds__(256) exact_hist_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists, uint32_t *hist)
{
    for (uint32_t l = blockIdx.x * blockDim.x + threadIdx.x; l < nlists; l += gridDim.x * blockDim.x)
        for (uint32_t q = mm_off[l], e = q + mm_len[l]; q < e; q++) atomicAdd(hist + mm_fid[q], 1u);
}
// step 2 (after run_scan): {key, list} into the feature's bucket; cursor[] starts as the bucket starts.  The order inside a
// bucket does not matter: the bucket sort orders it by (key, list index).
__global__ void __launch_bounds__(256) exact_scatter_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                            const unsigned long long *key, uint32_t *cursor, CollKey *out)
{
    for (uint32_t l = blockIdx.x * blockDim.x + threadIdx.x; l < nlists; l += gridDim.x * blockDim.x) {
        CollKey k; k.hash = key[l]; k.ord = l; k.pad = 0;
        for (uint32_t q = mm_off[l], e = q + mm_len[l]; q < e; q++) out[atomicAdd(cursor + mm_fid[q], 1u)] = k;
    }
}
// step 3 (after the bucket sorts): the list indices alone
__global__ void __launch_bounds__(256) exact_lists_kernel(const CollKey *keys, unsigned long long n, uint32_t *ilist)
{
    for (unsigned long long q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (unsigned long long)gridDim.x * blockDim.x) ilist[q] = keys[q].ord;
}

// Phase 1: s_l = sum of a[f] in list order, from 0 (:341-350)
__device__ __forceinline__ void em_exact_list_sums(uint32_t first, uint32_t stride, const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid,
                                                   uint32_t nlists, const double *av, double *sums)
{
    for (uint32_t l = first; l < nlists; l += stride) {
        double s = 0.0;
        for (uint32_t q = mm_off[l], e = q + mm_len[l]; q < e; q++) s = __dadd_rn(s, __ldcg(av + mm_fid[q]));
        sums[l] = s;
    }
}

// The share list l gives feature f: PropSharing a[f] / s_l for s_l > 0 (:351-365), a true division; equal 1 / n (:175-182)
struct ExactShareProp { const double *sums, *av;
    __device__ __forceinline__ bool operator()(uint32_t l, uint32_t f, double &v) const {
        const double s = __ldcg(sums + l);
        if (!(s > 0)) return false;
        v = __ddiv_rn(__ldcg(av + f), s); return true;
    } };
struct ExactShareEqual { const uint32_t *mm_len;
    __device__ __forceinline__ bool operator()(uint32_t l, uint32_t, double &v) const { v = __ddiv_rn(1.0, (double)mm_len[l]); return true; } };

// Incidences longer than this are summed by the whole warp: the lanes compute 32 quotients at once and every lane then
// carries the same chain of adds over them, in order.  Shorter ones are summed by their own lane.
constexpr uint32_t EXACT_WARP_CHAIN = 32;

// Phase 2: inc[f] = the serial sum, in key order, of the shares of f's lists; put(f, inc) is called once per feature by
// the lane that owns f.  Features are taken 32 at a time by warps first_warp, first_warp + warp_stride, ...
template <class Share, class Put>
__device__ __forceinline__ void em_exact_gather(uint32_t first_warp, uint32_t warp_stride, const uint32_t *ibeg, const uint32_t *ilist,
                                                uint32_t F, unsigned long long nent, Share share, Put put)
{
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t f0 = first_warp * 32u; f0 < F; f0 += warp_stride * 32u) {
        const uint32_t f = f0 + lane;
        const bool own = f < F;
        uint32_t b = 0, e = 0;
        if (own) exact_range(ibeg, F, nent, f, b, e);
        const bool chain = e - b > EXACT_WARP_CHAIN;
        double acc = 0.0;
        if (!chain)
            for (uint32_t q = b; q < e; q++) { double v; if (share(ilist[q], f, v)) acc = __dadd_rn(acc, v); }
        for (uint32_t lm = __ballot_sync(0xffffffffu, chain); lm; lm &= lm - 1u) {
            const int src = __ffs((int)lm) - 1;
            const uint32_t fs = __shfl_sync(0xffffffffu, f, src), bs = __shfl_sync(0xffffffffu, b, src), es = __shfl_sync(0xffffffffu, e, src);
            double cs = 0.0;
            for (uint32_t q0 = bs; q0 < es; q0 += 32u) {
                double v = 0.0;
                const bool ok = q0 + lane < es && share(ilist[q0 + lane], fs, v);
                const uint32_t okm = __ballot_sync(0xffffffffu, ok);
                for (int k = 0; k < 32; k++) {
                    const double vk = __shfl_sync(0xffffffffu, v, k);
                    if ((okm >> k) & 1u) cs = __dadd_rn(cs, vk);
                }
            }
            if ((int)lane == src) acc = cs;
        }
        if (own) put(f, acc);
    }
}

// Phase 3 for feature f: a = U + inc, flushed below 1e-20 (em_new_abundance); sq[f] = (a_new - a_old)^2 (:369-379)
__device__ __forceinline__ double em_exact_update(const double *U, double *a, double *sq, uint32_t f, double inc)
{
    const double an = em_new_abundance(U[f], inc);
    const double diff = __dsub_rn(an, a[f]);
    const double d2 = __dmul_rn(diff, diff);
    a[f] = an; sq[f] = d2;
    return d2;
}

// Phase 4, the stop decision.  The grid sums the sq[] terms in a tree (em_block_sum) to D_tree = fl(S_tree / F); the
// reference sums them in order j = 0 .. F-1 to D_seq = fl(S_seq / F).  For F non-negative terms with true sum S, every
// summation order gives |S_hat - S| <= gamma_{F-1} S, gamma_k = k u / (1 - k u), u = 2^-53 (Higham, Accuracy and
// Stability, (4.4)).  So S_seq / S_tree lies in [(1-g)/(1+g), (1+g)/(1-g)], g = gamma_{F-1}, and the two correctly
// rounded divisions by F add a factor (1 +- u) each: D_seq / D_tree lies within 1 +- r, r = 2g + 2u + O(u^2).  For
// F < 2^31, g <= (F-1) u (1 + 2^-21), so r <= 3 (F + 2) u, with room left for the rounding of D_tree * (1 +- r) below.
// Outside [D_tree (1 - r), D_tree (1 + r)] the threshold cannot separate the two sums: D_tree decides as D_seq would.
// Inside it (rare), the sequential sum is taken and used for the decision and for delta.
__host__ __device__ __forceinline__ bool em_exact_near(double delta_tree, uint32_t F)
{
    const double r = 3.0 * ((double)F + 2.0) * 0x1p-53;
    return delta_tree * (1.0 - r) < 1e-10 && delta_tree * (1.0 + r) >= 1e-10;
}
// D_seq: one thread, j = 0 .. F-1 (:377-380)
__device__ __forceinline__ double em_exact_seq_delta(const double *sq, uint32_t F)
{
    double s = 0.0;
    for (uint32_t j = 0; j < F; j++) s = __dadd_rn(s, __ldcg(sq + j));
    return __ddiv_rn(s, (double)F);
}

// The exact loop in one cooperative launch: list sums | barrier | gather + update + per-CTA partial | barrier | every CTA
// sums the partials in the same order (D_tree) and takes the same decision; near the threshold (or with force_seq, the
// tests' MSG_EXACT_DELTA=seq) CTA 0 takes D_seq, which every CTA reads after one more barrier.  partial has gridDim.x + 1
// slots.  result / delta_out as em_loop_kernel.
__global__ void __launch_bounds__(256) em_loop_exact_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                            const uint32_t *ibeg, const uint32_t *ilist, unsigned long long nent,
                                                            const double *U, double *a, double *sums, double *sq, double *partial, uint32_t F,
                                                            double *delta_out, int32_t *result, int force_seq)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double s_red[256];
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    int k = 1, conv = 0;
    for (; k < 20; k++) {
        em_exact_list_sums(gtid, gsz, mm_off, mm_len, mm_fid, nlists, a, sums);
        grid.sync();
        double dd = 0;
        em_exact_gather(gtid >> 5, gsz >> 5, ibeg, ilist, F, nent, ExactShareProp{sums, a},
                        [&](uint32_t f, double inc) { dd = __dadd_rn(dd, em_exact_update(U, a, sq, f, inc)); });
        const double part = em_block_sum(s_red, dd);
        if (threadIdx.x == 0) partial[blockIdx.x] = part;
        grid.sync();
        double acc = 0;
        for (uint32_t b = threadIdx.x; b < gridDim.x; b += 256) acc = __dadd_rn(acc, __ldcg(partial + b));
        double delta = em_block_sum(s_red, acc) / F;
        __syncthreads();
        if (force_seq || em_exact_near(delta, F)) {                         // the same decision in every CTA
            if (gtid == 0) partial[gridDim.x] = em_exact_seq_delta(sq, F);
            grid.sync();
            delta = __ldcg(partial + gridDim.x);
        }
        if (gtid == 0) delta_out[k - 1] = delta;
        if (delta < 1e-10) { conv = 1; break; }
    }
    if (gtid == 0) { result[0] = k < 20 ? k : 19; result[1] = conv; }
    em_count_purged(gtid, gsz, mm_off, mm_len, mm_fid, nlists, a, reinterpret_cast<uint32_t *>(result + 3));
}

// The same phases one launch each, for the host loop
__global__ void __launch_bounds__(256) em_exact_sums_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                            const double *a, double *sums)
{
    em_exact_list_sums(blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x, mm_off, mm_len, mm_fid, nlists, a, sums);
}
__global__ void __launch_bounds__(256) em_exact_gather_kernel(const uint32_t *ibeg, const uint32_t *ilist, unsigned long long nent, const double *sums,
                                                              const double *U, double *a, double *sq, double *partial, uint32_t F)
{
    __shared__ double s_red[256];
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    double dd = 0;
    em_exact_gather(gtid >> 5, gsz >> 5, ibeg, ilist, F, nent, ExactShareProp{sums, a},
                    [&](uint32_t f, double inc) { dd = __dadd_rn(dd, em_exact_update(U, a, sq, f, inc)); });
    const double part = em_block_sum(s_red, dd);
    if (threadIdx.x == 0) partial[blockIdx.x] = part;
}
__global__ void em_exact_seq_kernel(const double *sq, uint32_t F, double *delta_out)
{
    if (blockIdx.x == 0 && threadIdx.x == 0) *delta_out = em_exact_seq_delta(sq, F);
}
// exact --multi=equal: d[f] = the serial sum, in key order, of 1 / n over f's lists
__global__ void __launch_bounds__(256) em_exact_equal_kernel(const uint32_t *ibeg, const uint32_t *ilist, unsigned long long nent, const uint32_t *mm_len,
                                                             double *d, uint32_t F)
{
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    em_exact_gather(gtid >> 5, gsz >> 5, ibeg, ilist, F, nent, ExactShareEqual{mm_len}, [&](uint32_t f, double v) { d[f] = v; });
}

// Multi-GPU PropSharing: counts exchange + the whole loop + the purged total in ONE cooperative kernel per GPU, with
// no NCCL call and no host round trip.  Collective = push over peer memory (CUDA IPC mappings, NVLink/NVSwitch) in a
// low-latency flagged format: every value travels as two 8-byte words {epoch tag : 32 | half of the f64 : 32}.  A rank
// STORES its vector into its slot of every peer's region and is done -- no fence, no separate flag; a receiver polls
// its OWN memory until both words of an element carry the expected tag (8-byte stores are single-copy atomic, so a
// matching tag proves the payload).  An exchange therefore costs one one-way NVLink latency.  Every rank then adds the
// N vectors in rank order -- the same order everywhere -- so abundances, delta and the stop decision are bit-identical
// on all ranks.
//
// Region of rank r (lives in r's memory, written by its peers):
//   [0,128)   purged[s]  u64   {tag : 32 | sender s's purged-list count : 32}
//   [128, )   slot[parity][s][V][2] u64, V = F + 8: vector of sender s for exchanges of that parity
// Exchange k (k = 0: doubled counts + insert counters, k >= 1: increments of iteration k) uses parity k & 1 and tag
// epoch + k.  A sender overwrites slot[k & 1] only after it received exchange k-1 from every peer, which a peer sends
// after all of its threads finished reading exchange k-2 (grid barriers in between).  The purged message (tag
// epoch + 24) closes a call the same way, so the next call may start writing at once.  Vectors of up to EM_XCHG_CTA0
// values are exchanged by CTA 0 alone (the other CTAs wait at the next grid barrier), longer ones by the whole grid.
struct PeerTable { unsigned char *base[16]; };
constexpr uint32_t EM_XCHG_CTA0 = 8192;

__device__ __forceinline__ void ll_store(unsigned long long *p, unsigned long long w0, unsigned long long w1)
{
    asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" :: "l"(p), "l"(w0), "l"(w1) : "memory");
}
__device__ __forceinline__ void ll_load(const unsigned long long *p, unsigned long long &w0, unsigned long long &w1)
{
    asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned long long *ll_slot(const PeerTable &pt, int dst, uint32_t parity, int src, int n_ranks, uint32_t V)
{
    return reinterpret_cast<unsigned long long *>(pt.base[dst] + 128) + (((size_t)parity * (size_t)n_ranks + (size_t)src) * V) * 2;
}

template <bool SMEM>
__global__ void __launch_bounds__(256) em_loop_multi_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                            const uint32_t *ui, const uint32_t *counters, uint32_t nl_lo, uint32_t nl_hi,
                                                            double *U, double *a, double *inc, double *partial, uint32_t F,
                                                            double *delta_out, int32_t *result, uint32_t *hc_out,
                                                            double *totbuf, uint32_t *bflag,
                                                            PeerTable peers, int n_ranks, int rank, uint32_t epoch, unsigned long long timeout_ns)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    extern __shared__ double s_em[];
    __shared__ double s_red[256];
    double *sa = s_em;
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    const uint32_t V = F + 8;
    // who takes part in the exchanges
    const bool cta0 = V <= EM_XCHG_CTA0;
    const bool part = !cta0 || blockIdx.x == 0;
    const uint32_t ptid = cta0 ? threadIdx.x : gtid, pn = cta0 ? blockDim.x : gsz, nparts = cta0 ? 1u : gridDim.x;
    int timeout = 0;
    unsigned long long t_start;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_start));
    auto expired = [&]() -> bool { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t - t_start > timeout_ns; };
    // push my vector (getv) to every rank, then wait for everyone's vector and hand the rank-ordered total of every
    // element to put().  Called by the participants only; needs no barrier of its own.
    auto exchange = [&](uint32_t tag, uint32_t parity, auto getv, auto put) {
        const unsigned long long want = (unsigned long long)(epoch + tag), t = want << 32;
        for (uint32_t i = ptid; i < V; i += pn) {
            const unsigned long long bits = (unsigned long long)__double_as_longlong(getv(i));
            const unsigned long long w0 = t | (bits & 0xffffffffull), w1 = t | (bits >> 32);
            for (int r = 0; r < n_ranks; r++) ll_store(ll_slot(peers, r, parity, rank, n_ranks, V) + 2 * (size_t)i, w0, w1);
        }
        for (uint32_t i = ptid; i < V; i += pn) {
            double tot = 0;
            for (int r = 0; r < n_ranks; r++) {
                const unsigned long long *src = ll_slot(peers, rank, parity, r, n_ranks, V) + 2 * (size_t)i;
                unsigned long long w0, w1; uint32_t spins = 0;
                for (;;) {
                    ll_load(src, w0, w1);
                    if ((w0 >> 32) == want && (w1 >> 32) == want) break;
                    // a peer that never shows up costs ONE time limit (wall clock, MSG_PEER_TIMEOUT_S), not one per exchange: the flag is sticky
                    if (timeout || ((++spins & 1023u) == 0 && expired())) { timeout = 1; break; }
                }
                tot += __longlong_as_double((long long)((w1 << 32) | (w0 & 0xffffffffull)));
            }
            put(i, tot);
        }
        if (timeout) result[2] = 1;
    };
    // ---- exchange 0: U = a = (sum over ranks of the doubled counts) / 2 (:286); insert counters and list totals for the host.
    //      Small integers are exact in f64, so the totals equal the integer sums.
    if (gtid < 20) delta_out[gtid] = 0.0;                   // result[0..3] is cleared by the host before the launch
    if (part)
        exchange(0u, 0u,
                 [&](uint32_t i) -> double { return i < F ? (double)ui[i] : i < F + 4 ? (double)counters[i - F] : i == F + 4 ? (double)nl_lo : i == F + 5 ? (double)nl_hi : 0.0; },
                 [&](uint32_t i, double tot) { if (i < F) { const double u = tot / 2; U[i] = u; a[i] = u; inc[i] = 0.0; } else hc_out[i - F] = (uint32_t)tot; });
    grid.sync();
    int k = 1, conv = 0;
    if constexpr (SMEM) {
        // F <= EM_SMEM_F: ONE grid barrier per iteration.  After the barrier that completes inc[], CTA 0 exchanges the
        // increments with the peers and broadcasts the rank-ordered totals through totbuf[k & 1] + a release flag; every
        // CTA then redoes the F-sized update and the delta reduction from its own shared-memory a[] (same data, same order:
        // bit-identical everywhere, no second barrier).  CTA 0 clears inc[] before it raises the flag, so the other CTAs'
        // next gather (which starts only after they have seen the flag) adds into zeros.
        for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) sa[i] = __ldcg(a + i);
        for (; k < 20; k++) {
            em_gather_smem(gtid, gsz, mm_off, mm_len, mm_fid, nlists, sa, s_em + F, [&] { return inc; }, F);
            grid.sync();
            double *tb = totbuf + (size_t)(k & 1) * F;
            if (blockIdx.x == 0) {
                exchange((uint32_t)k, (uint32_t)k & 1u,
                         [&](uint32_t i) -> double { if (i >= F) return 0.0; const double v = __ldcg(inc + i); inc[i] = 0.0; return v; },
                         [&](uint32_t i, double tot) { if (i < F) tb[i] = tot; });
                __threadfence();
                __syncthreads();
                if (threadIdx.x == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(bflag), "r"(epoch + (uint32_t)k) : "memory");
            }
            if (threadIdx.x == 0) {
                uint32_t seen;
                do { asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(bflag) : "memory"); } while ((int32_t)(seen - (epoch + (uint32_t)k)) < 0);
            }
            __syncthreads();
            double dd = 0;
            for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) {
                double an = U[i] + __ldcg(tb + i);
                if (an < 1e-20) an = 0;
                const double diff = an - sa[i];
                dd += diff * diff;
                sa[i] = an;
            }
            const double delta = em_block_sum(s_red, dd) / F;
            __syncthreads();
            if (gtid == 0) delta_out[k - 1] = delta;
            if (delta < 1e-10) { conv = 1; break; }
        }
        if (blockIdx.x == 0) for (uint32_t i = threadIdx.x; i < F; i += blockDim.x) a[i] = sa[i];
    } else {
        for (; k < 20; k++) {
            em_share_lists(gtid, gsz, mm_off, mm_len, mm_fid, nlists, a, inc);
            grid.sync();
            // exchange the increments; a = U + total, flush < 1e-20, per-CTA partial of sum diff^2   (:369-379)
            if (part) {
                double dd = 0;
                exchange((uint32_t)k, (uint32_t)k & 1u,
                         [&](uint32_t i) -> double { if (i >= F) return 0.0; const double v = inc[i]; inc[i] = 0.0; return v; },
                         [&](uint32_t i, double tot) {
                             if (i >= F) return;
                             double an = U[i] + tot;
                             if (an < 1e-20) an = 0;
                             const double diff = an - a[i];
                             dd += diff * diff;
                             a[i] = an;
                         });
                const double sum = em_block_sum(s_red, dd);
                if (threadIdx.x == 0) partial[blockIdx.x] = sum;
            }
            grid.sync();
            // delta (every CTA, same order)                                   (:380-383)
            double acc = 0;
            for (uint32_t b = threadIdx.x; b < nparts; b += 256) acc += __ldcg(partial + b);
            const double delta = em_block_sum(s_red, acc) / F;
            __syncthreads();
            if (gtid == 0) delta_out[k - 1] = delta;
            if (delta < 1e-10) { conv = 1; break; }
        }
    }
    // ---- purged = #lists whose final abundances sum to exactly 0 (:394-404), summed over ranks through the same regions
    {
        em_count_purged(gtid, gsz, mm_off, mm_len, mm_fid, nlists, SMEM ? sa : a, reinterpret_cast<uint32_t *>(result + 3));
        grid.sync();
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            const unsigned long long want = (unsigned long long)(epoch + 24u);
            const unsigned long long msg = (want << 32) | (unsigned long long)__ldcg(reinterpret_cast<const uint32_t *>(result + 3));
            for (int r = 0; r < n_ranks; r++)
                asm volatile("st.relaxed.sys.global.u64 [%0], %1;" :: "l"(reinterpret_cast<unsigned long long *>(peers.base[r]) + rank), "l"(msg) : "memory");
            uint32_t tot = 0;
            for (int r = 0; r < n_ranks; r++) {
                const unsigned long long *src = reinterpret_cast<const unsigned long long *>(peers.base[rank]) + r;
                unsigned long long w; uint32_t spins = 0;
                for (;;) {
                    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w) : "l"(src) : "memory");
                    if ((w >> 32) == want) break;
                    if (*reinterpret_cast<volatile int32_t *>(result + 2) || ((++spins & 1023u) == 0 && expired())) { result[2] = 1; break; }
                }
                tot += (uint32_t)w;
            }
            result[3] = (int32_t)tot;
            result[0] = k < 20 ? k : 19; result[1] = conv;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Multi-GPU PropSharing for gene catalogues (F + 8 > EM_XCHG_CTA0): the same single cooperative launch per GPU, but the
// per-iteration collective is a REDUCE-SCATTER + ALL-GATHER over peer memory instead of "every rank pushes its whole
// vector to every rank": rank r owns the slice [r*S, (r+1)*S) of the feature axis.
//   RS  every rank stores its partial increments of slice s into rank s's region (plain 16-byte stores over NVLink),
//       block by block (RSAG_BLK values), then fence.sys + one flag word per block.
//   upd the owner adds the N partials of a block IN RANK ORDER, applies a = U + inc, the 1e-20 flush and the block's
//       share of sum (a_new - a_old)^2 (msam_profile.c:369-380), and
//   AG  stores the new abundances of the block into every rank's copy of a[] (double buffered by exchange parity, so the
//       gather of the next iteration reads a[] where it landed -- no extra copy), followed by fence.sys and a flagged
//       16-byte word pair {tag|lo32, tag|hi32} carrying the block's delta share.  Every rank sums all N*nblk shares in
//       the same fixed order => DELTA^2, the stop decision (:383) and a[] are bit-identical on all ranks.
// Per rank and iteration 2*(N-1)/N * F * 8 bytes leave over NVLink (28 MB at F = 1e6, N = 8, against 128 MB + 128 MB of
// polling reads for the all-to-all push), the region is (2 + 2) * N*S * 8 bytes (32 MB), and there are two grid barriers
// per iteration.  Exchange 0 runs the doubled counts through the same path (U = a = total / 2, :286); the six host
// counters and the final purged count travel as flagged words through the 1 KB scalar area, as in the small-F kernel.
// Slot reuse is safe by parity exactly as above: a rank can only be one exchange ahead of any peer.
constexpr uint32_t RSAG_BLK = 512;                 // values per block: 256 threads x one 16-byte store
constexpr uint32_t RSAG_MAXB = 32;                 // owner blocks per CTA announced with one fence

struct RsagLayout {                                 // byte offsets inside a rank's region (after the 128-byte purged area)
    uint32_t S, nblk; int n_ranks;
    __host__ __device__ size_t scal() const { return 128; }                                              // [16 senders][8] u64 flagged scalars
    __host__ __device__ size_t rs_flag() const { return scal() + 16 * 8 * 8; }                            // [2][N][nblk] u32
    __host__ __device__ size_t dd() const { return rs_flag() + (((size_t)2 * n_ranks * nblk * 4 + 15) & ~(size_t)15); }   // [2][N][nblk][2] u64
    __host__ __device__ size_t rs_data() const { return dd() + (size_t)2 * n_ranks * nblk * 16; }        // [2][N][S] f64
    __host__ __device__ size_t ag_data() const { return rs_data() + (size_t)2 * n_ranks * S * 8; }       // [2][N*S] f64
    __host__ __device__ size_t total() const { return ag_data() + (size_t)2 * n_ranks * S * 8; }
};
__host__ __device__ inline RsagLayout rsag_layout(uint32_t F, int n_ranks)
{
    RsagLayout L; L.n_ranks = n_ranks;
    const uint32_t per = (F + (uint32_t)n_ranks - 1) / (uint32_t)n_ranks;
    L.nblk = (per + RSAG_BLK - 1) / RSAG_BLK; if (L.nblk == 0) L.nblk = 1;
    L.S = L.nblk * RSAG_BLK;
    return L;
}

// release / acquire fence at system scope (what a flag store after peer-memory data stores needs; cheaper than the
// sequentially consistent __threadfence_system)
__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
__device__ __forceinline__ unsigned long long globaltimer_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p) { uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void st_relaxed_sys_u32(uint32_t *p, uint32_t v) { asm volatile("st.relaxed.sys.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void st_weak_v2f64(double *p, double a, double b) { asm volatile("st.global.v2.f64 [%0], {%1, %2};" :: "l"(p), "d"(a), "d"(b) : "memory"); }
__device__ __forceinline__ void ld_cg_v2f64(const double *p, double &a, double &b) { asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "l"(p) : "memory"); }

__global__ void __launch_bounds__(256) em_loop_rsag_kernel(const uint32_t *mm_off, const uint32_t *mm_len, const int32_t *mm_fid, uint32_t nlists,
                                                           const uint32_t *ui, const uint32_t *counters, uint32_t nl_lo, uint32_t nl_hi,
                                                           double *U, double *a_out, double *inc, uint32_t F,
                                                           double *delta_out, int32_t *result, uint32_t *hc_out,
                                                           PeerTable peers, int n_ranks, int rank, uint32_t epoch, unsigned long long timeout_ns,
                                                           unsigned long long *trace /* diagnostics: [20][8] ns stamps of CTA 0, or null */)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ double s_red[256], s_dd[RSAG_MAXB];
    __shared__ int s_to;
    const RsagLayout L = rsag_layout(F, n_ranks);
    const uint32_t S = L.S, nblk = L.nblk, N = (uint32_t)n_ranks;
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    unsigned char *me = peers.base[rank];
    const unsigned long long t_start = globaltimer_ns();
    volatile int32_t *timed_out = result + 2;
    auto expired = [&]() -> bool {
        if (*timed_out) return true;
        if (globaltimer_ns() - t_start > timeout_ns) { *timed_out = 1; return true; }
        return false;
    };
    // a[] after exchange k lives in ag_data[k & 1] of MY region (every owner stored its slice there)
    auto a_buf = [&](uint32_t par) -> double * { return reinterpret_cast<double *>(me + L.ag_data()) + (size_t)par * N * S; };

    // One exchange.  first: the values are the doubled counts (U = a = total / 2, no delta); else the increments.
    bool dead = false;                               // a peer never showed up: same value in every thread (read after a grid barrier)
    auto stamp = [&](uint32_t k, uint32_t j) { if (trace && blockIdx.x == 0 && threadIdx.x == 0 && k < 20) trace[k * 8 + j] = globaltimer_ns(); };
    auto exchange = [&](uint32_t k, bool first) -> double {
        const uint32_t par = k & 1u, tag = epoch + k;
        stamp(k, 0);
        // ---- reduce-scatter, sender side: block (s, b) of my vector -> rank s.  All of this CTA's blocks first, then ONE
        //      fence.sys (it waits for the NVLink writes to be acknowledged: microseconds), then their flags.
        for (uint32_t blk = blockIdx.x; blk < N * nblk; blk += gridDim.x) {
            const uint32_t s = blk / nblk, b = blk - s * nblk;
            const uint32_t i0 = s * S + b * RSAG_BLK + 2 * threadIdx.x;
            double v0, v1;
            if (first) { v0 = i0 < F ? (double)ui[i0] : 0.0; v1 = i0 + 1 < F ? (double)ui[i0 + 1] : 0.0; }
            else {
                v0 = i0 < F ? __ldcg(inc + i0) : 0.0; v1 = i0 + 1 < F ? __ldcg(inc + i0 + 1) : 0.0;
                if (i0 < F) inc[i0] = 0.0;
                if (i0 + 1 < F) inc[i0 + 1] = 0.0;
            }
            double *dst = reinterpret_cast<double *>(peers.base[s] + L.rs_data()) + ((size_t)par * N + (size_t)rank) * S + b * RSAG_BLK + 2 * threadIdx.x;
            st_weak_v2f64(dst, v0, v1);
        }
        __syncthreads();
        stamp(k, 1);
        if (threadIdx.x == 0) {
            fence_acq_rel_sys();
            for (uint32_t blk = blockIdx.x; blk < N * nblk; blk += gridDim.x) {
                const uint32_t s = blk / nblk, b = blk - s * nblk;
                st_relaxed_sys_u32(reinterpret_cast<uint32_t *>(peers.base[s] + L.rs_flag()) + ((size_t)par * N + (size_t)rank) * nblk + b, tag);
            }
        }
        stamp(k, 2);
        // ---- owner side: blocks of my slice.  Wait for the N partials, reduce in rank order, update, all-gather; the
        //      blocks' delta shares are announced (flagged word pairs) after one fence.sys for all of them.
        const double *a_old = a_buf(par ^ 1u);
        uint32_t nmine = 0, b_first = blockIdx.x;
        auto announce = [&]() {                             // thread 0: one fence for the buffered blocks, then their flagged delta shares
            fence_acq_rel_sys();                         // cumulative over this CTA's stores (they happen-before through the barriers)
            uint32_t bb = b_first;
            for (uint32_t j = 0; j < nmine; j++, bb += gridDim.x) {
                const unsigned long long bits = (unsigned long long)__double_as_longlong(s_dd[j]), t = (unsigned long long)tag << 32;
                for (uint32_t r = 0; r < N; r++)
                    ll_store(reinterpret_cast<unsigned long long *>(peers.base[r] + L.dd()) + (((size_t)par * N + (size_t)rank) * nblk + bb) * 2,
                             t | (bits & 0xffffffffull), t | (bits >> 32));
            }
        };
        for (uint32_t b = blockIdx.x; b < nblk; b += gridDim.x) {
            if (threadIdx.x == 0) s_to = 0;
            __syncthreads();
            if (threadIdx.x < N) {
                const uint32_t *fl = reinterpret_cast<const uint32_t *>(me + L.rs_flag()) + ((size_t)par * N + threadIdx.x) * nblk + b;
                uint32_t v;
                for (;;) {
                    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(fl) : "memory");
                    if (v == tag) break;
                    if (expired()) { s_to = 1; break; }
                }
            }
            __syncthreads();
            const uint32_t li = b * RSAG_BLK + 2 * threadIdx.x, i0 = (uint32_t)rank * S + li;
            double t0 = 0, t1 = 0;
            if (!s_to)
                for (uint32_t r = 0; r < N; r++) {
                    double x0, x1;
                    ld_cg_v2f64(reinterpret_cast<const double *>(me + L.rs_data()) + ((size_t)par * N + r) * S + li, x0, x1);
                    t0 += x0; t1 += x1;
                }
            double n0, n1, dd = 0;
            if (first) {
                n0 = t0 / 2; n1 = t1 / 2;                                           // :286
                if (i0 < F) U[i0] = n0;
                if (i0 + 1 < F) U[i0 + 1] = n1;
            } else {
                n0 = i0 < F ? U[i0] + t0 : 0.0; n1 = i0 + 1 < F ? U[i0 + 1] + t1 : 0.0;   // :371
                if (n0 < 1e-20) n0 = 0;                                                 // :372-376
                if (n1 < 1e-20) n1 = 0;
                double o0, o1;
                ld_cg_v2f64(a_old + i0, o0, o1);
                const double d0 = i0 < F ? n0 - o0 : 0.0, d1 = i0 + 1 < F ? n1 - o1 : 0.0;
                dd = d0 * d0 + d1 * d1;                                                 // :377-379
            }
            for (uint32_t r = 0; r < N; r++)
                st_weak_v2f64(reinterpret_cast<double *>(peers.base[r] + L.ag_data()) + (size_t)par * N * S + i0, n0, n1);
            const double bsum = em_block_sum(s_red, dd);
            if (threadIdx.x == 0) s_dd[nmine] = bsum;
            nmine++;
            if (nmine == RSAG_MAXB) {                       // (huge catalogues only)
                __syncthreads();
                if (threadIdx.x == 0) announce();
                nmine = 0; b_first = b + gridDim.x;
            }
            __syncthreads();
        }
        stamp(k, 3);
        if (threadIdx.x == 0 && nmine) announce();
        stamp(k, 4);
        // ---- all-gather, receiver side: every block of every owner must have landed in my copy of a[]
        {
            const unsigned long long want = (unsigned long long)tag;
            for (uint32_t q = gtid; q < N * nblk; q += gsz) {
                const unsigned long long *src = reinterpret_cast<const unsigned long long *>(me + L.dd()) + ((size_t)par * N * nblk + q) * 2;
                unsigned long long w0, w1;
                for (;;) {
                    ll_load(src, w0, w1);
                    if ((w0 >> 32) == want && (w1 >> 32) == want) break;
                    if (expired()) break;
                }
            }
            fence_acq_rel_sys();
        }
        stamp(k, 5);
        grid.sync();
        stamp(k, 6);
        dead = *timed_out != 0;                      // nobody polls between this barrier and the next exchange: uniform
        // ---- DELTA^2: all N*nblk block shares, same order on every rank and in every CTA            (:380)
        double acc = 0;
        if (!first)
            for (uint32_t q = threadIdx.x; q < N * nblk; q += 256) {
                unsigned long long w0, w1;
                ll_load(reinterpret_cast<const unsigned long long *>(me + L.dd()) + ((size_t)par * N * nblk + q) * 2, w0, w1);
                acc += __longlong_as_double((long long)((w1 << 32) | (w0 & 0xffffffffull)));
            }
        const double delta = em_block_sum(s_red, acc) / F;
        __syncthreads();
        stamp(k, 7);
        return delta;
    };
    // flagged scalars: sender `rank` writes word j of its row in every peer's scalar area
    auto scal_send = [&](uint32_t j, uint32_t tag, uint32_t value) {
        const unsigned long long msg = ((unsigned long long)tag << 32) | value;
        for (uint32_t r = 0; r < N; r++)
            asm volatile("st.relaxed.sys.global.u64 [%0], %1;" :: "l"(reinterpret_cast<unsigned long long *>(peers.base[r] + L.scal()) + (size_t)rank * 8 + j), "l"(msg) : "memory");
    };
    auto scal_sum = [&](uint32_t j, uint32_t tag) -> uint32_t {
        uint32_t tot = 0;
        for (uint32_t r = 0; r < N; r++) {
            const unsigned long long *src = reinterpret_cast<const unsigned long long *>(me + L.scal()) + (size_t)r * 8 + j;
            unsigned long long w;
            for (;;) {
                asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w) : "l"(src) : "memory");
                if ((w >> 32) == tag || expired()) break;
            }
            tot += (uint32_t)w;
        }
        return tot;
    };

    if (gtid < 20) delta_out[gtid] = 0.0;                   // result[0..3] is cleared by the host before the launch
    // host counters (inserts, unique, multiple, big groups) and the two halves of the list total: six flagged scalars
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x < 6) {
        const uint32_t j = threadIdx.x;
        scal_send(j, epoch, j < 4 ? counters[j] : (j == 4 ? nl_lo : nl_hi));
        hc_out[j] = scal_sum(j, epoch);
    }
    exchange(0u, true);
    int k = 1, conv = 0;
    for (; k < 20; k++) {
        // gather: s = sum a[f] in list order; inc[f] += a[f]/s            (:341-365)
        em_share_lists(gtid, gsz, mm_off, mm_len, mm_fid, nlists, a_buf((uint32_t)(k - 1) & 1u), inc);
        grid.sync();
        const double delta = exchange((uint32_t)k, false);
        if (gtid == 0) delta_out[k - 1] = delta;
        if (dead) break;
        if (delta < 1e-10) { conv = 1; break; }                             // :383
    }
    // ---- final abundances to a_out, purged = #lists whose abundances sum to exactly 0 (:394-404), summed over ranks
    {
        const uint32_t kl = k < 20 ? (uint32_t)k : 19u;
        const double *av = a_buf(kl & 1u);
        for (uint32_t i = gtid; i < F; i += gsz) a_out[i] = av[i];
        em_count_purged(gtid, gsz, mm_off, mm_len, mm_fid, nlists, av, reinterpret_cast<uint32_t *>(result + 3));
        grid.sync();
        // the purged message also tells the peers that this rank is done reading its copy of a[]: only then may a peer's
        // next call overwrite it
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            scal_send(6, epoch + 24u, __ldcg(reinterpret_cast<const uint32_t *>(result + 3)));
            result[3] = (int32_t)scal_sum(6, epoch + 24u);
            result[0] = (int32_t)kl; result[1] = conv;
        }
    }
}

struct InPcountPacked {      // (is_list << 32) | entries, for one packed u64 scan
    const uint32_t *pc;
    __device__ __forceinline__ unsigned long long operator()(uint64_t i) const {
        uint32_t v = pc[i];
        return v ? ((1ull << 32) | v) : 0ull;
    }
};
struct OutExclU64 { unsigned long long *o; __device__ __forceinline__ void operator()(uint64_t i, unsigned long long ex, unsigned long long) const { o[i] = ex; } };

} // namespace msg
