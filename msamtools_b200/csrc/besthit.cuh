// besthit.cuh -- K3: per-pool best-hit selection + stable emission in reference order.
//
// Replaces mWriteBamPool (mBamVector.c:342-347), mWriteBestHitBamPoolByMate,
// mWriteBestHitBamPool, mWriteUniqueBestHitBamPool (msam_filter.c:192-263) and the
// pool segmentation of mFilterFile (msam_filter.c:120-125,170).
//
// Pool == maximal run of byte-identical adjacent QNAMEs: between two consecutive
// mapped records m < i the reference flushes iff some record in (m, i] differs from
// prev_read == QNAME(m), which is exactly "the FB_EQPREV chain from m to i is broken"
// (DESIGN.md gives the two-line proof).  No sort, no hash, no cross-CTA state.
//
// Main path: one record per lane.  Run heads come from a ballot of FB_EQPREV; lanes of
// the same (run, mate class) find each other with MATCH.ANY, take the class maximum with
// REDUX.MAX and count ties with a ballot -- a segmented warp reduction without loops or
// divergence.  Runs that straddle a 32-record window (a few per cent) are appended to a
// worklist and finished by a head-walks-its-run kernel, which is also the exact fallback
// for arbitrarily long runs.
#pragma once
#include "common.cuh"

namespace msg {

__device__ __forceinline__ int mate_class(uint32_t fb)
{   // class index by (flag & 0xC0): 0x00->0, 0x40->1 (READ1), 0x80->2 (READ2), 0xC0->3
    return (int)((fb >> 6) & 3u);
}

// Per-lane view of the QNAME runs inside one 32-record window.
struct RunView {
    uint32_t segmask;     // lanes of my run inside this window
    uint32_t s;           // lane of the run's first record in this window
    bool crossing;        // run continues beyond the window on either side
    bool is_open_head;    // I am the head of a run that leaves the window on the right
};

// f = fb word (0 for lanes past n), i = record index; next_f = fb of record w0+32 (fetched by the caller)
__device__ __forceinline__ RunView run_view(uint32_t f, uint64_t i, uint64_t n, bool next_is_head)
{
    const uint32_t lane = threadIdx.x & 31u;
    const bool head = i >= n || i == 0 || !(f & FB_EQPREV);
    const uint32_t hmask = __ballot_sync(0xffffffffu, head);
    const uint32_t le = hmask & (0xffffffffu >> (31u - lane));          // heads at or below my lane
    const uint32_t gt = lane == 31 ? 0u : (hmask & (0xffffffffu << (lane + 1)));
    RunView v;
    const bool open_left = le == 0;
    v.s = open_left ? 0u : 31u - (uint32_t)__clz((int)le);
    const uint32_t e = gt ? (uint32_t)__ffs((int)gt) - 1u : 32u;
    const bool open_right = gt == 0 && !next_is_head;
    v.segmask = (e == 32 ? 0xffffffffu : ((1u << e) - 1u)) & (0xffffffffu << v.s);
    v.crossing = open_left || open_right;
    v.is_open_head = open_right && !open_left && lane == v.s && i < n;
    return v;
}

struct BestHitParams {
    uint32_t *fb;             // in/out (FB_KEEP written)
    const int32_t *score;
    uint64_t n;
    int uniq;
    uint32_t *err;
    uint32_t *worklist;       // heads of runs that straddle a window
    uint32_t *wl_count;
};

// Winners of every complete pool inside one 32-record window.  Best score per (pool, mate class) is a shared-memory
// max per slot (pool's first lane * 4 + class; sb = 128 words owned by this warp).  A __reduce_max_sync over
// __match_any groups gives the same answer but executes once per distinct group (~16 serialized REDUX per window at
// 2-3 records per pool: 22 % of the fused kernel's stall samples).  Called by all 32 lanes.
__device__ __forceinline__ bool pool_winner(int32_t *sb, uint32_t lane, bool act, int32_t score, uint32_t slot, bool uniq)
{
    *reinterpret_cast<int4 *>(sb + lane * 4) = make_int4(INT32_MIN, INT32_MIN, INT32_MIN, INT32_MIN);
    __syncwarp();
    if (act) atomicMax(sb + slot, score);                                         // msam_filter.c:212-230
    __syncwarp();
    const bool tie = act && score == sb[slot];
    if (!uniq) return tie;
    __syncwarp();                                                                  // :232-244 winners must be alone in their class
    *reinterpret_cast<int4 *>(sb + lane * 4) = make_int4(0, 0, 0, 0);
    __syncwarp();
    if (tie) atomicAdd(sb + slot, 1);
    __syncwarp();
    return tie && sb[slot] == 1;
}

// the first record of pool [i, end) that the best-hit writers read without an AS tag (for the error message)
__device__ __forceinline__ uint32_t noas_record(const uint32_t *fb, uint64_t i, uint64_t end, bool paired)
{
    for (uint64_t j = i; j < end; j++) {
        const uint32_t f = fb[j];
        const int c = mate_class(f);
        if ((f & FB_INPOOL) && !(f & FB_HAS_AS) && (paired ? (c == 1 || c == 2) : c == 0)) return (uint32_t)j;
    }
    return 0xffffffffu;
}

__global__ void __launch_bounds__(256) besthit_warp_select_kernel(const BestHitParams p)
{
    __shared__ __align__(16) int32_t s_best[8][128];
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t w0 = i & ~31ull;
    if (w0 >= p.n) return;                                                        // whole warp out of range
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t f = i < p.n ? p.fb[i] : 0u;
    uint32_t nf = 0;
    if (lane == 31 && w0 + 32 < p.n) nf = p.fb[w0 + 32];
    nf = __shfl_sync(0xffffffffu, nf, 31);
    const bool next_is_head = w0 + 32 >= p.n || !(nf & FB_EQPREV);
    const RunView v = run_view(f, i, p.n, next_is_head);
    if (v.is_open_head) { uint32_t slot = atomicAdd(p.wl_count, 1u); p.worklist[slot] = (uint32_t)i; }

    const bool mine = i < p.n && !v.crossing;
    const bool pooled = mine && (f & FB_INPOOL);
    const int cls = mate_class(f);
    // pool pairedness (msam_filter.c:196-204) and the classes the reference visits (:247-254)
    const bool paired = (__ballot_sync(0xffffffffu, pooled && cls != 0) & v.segmask) != 0;
    const bool act = pooled && (paired ? (cls == 1 || cls == 2) : true);
    if (act && !(f & FB_HAS_AS)) { atomicOr(p.err, DERR_NOAS); atomicMin(p.err + 1, (uint32_t)i); }       // :219-221
    const int32_t sc = act ? p.score[i] : INT32_MIN;
    const bool keep = pool_winner(s_best[threadIdx.x >> 5], lane, act, sc, v.s * 4u + (uint32_t)cls, p.uniq);
    if (mine) {
        const uint32_t out = keep ? (f | FB_KEEP) : (f & ~FB_KEEP);
        if (out != f) p.fb[i] = out;
    }
}

// worklist: the head walks its run (exact for any run length)
__global__ void __launch_bounds__(256) besthit_walk_select_kernel(const BestHitParams p)
{
    const uint32_t nw = *p.wl_count;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nw; q += gridDim.x * blockDim.x) {
        const uint64_t i = p.worklist[q];
        int32_t best[4] = {INT32_MIN, INT32_MIN, INT32_MIN, INT32_MIN};
        int32_t cnt[4] = {0, 0, 0, 0};
        uint32_t noas = 0;
        bool paired = false;
        uint64_t j = i;
        uint32_t f = p.fb[i];
        for (;;) {
            if (f & FB_INPOOL) {
                const int c = mate_class(f);
                paired |= (c != 0);
                if (!(f & FB_HAS_AS)) noas |= 1u << c;
                const int32_t s = p.score[j];
#pragma unroll
                for (int k = 0; k < 4; k++) if (k == c) {
                    if (s > best[k]) { best[k] = s; cnt[k] = 1; } else if (s == best[k]) cnt[k]++;
                }
            }
            if (++j >= p.n) break;
            f = p.fb[j];
            if (!(f & FB_EQPREV)) break;
        }
        const uint64_t end = j;
        if (paired ? (noas & 6u) : (noas & 1u)) { atomicOr(p.err, DERR_NOAS); atomicMin(p.err + 1, noas_record(p.fb, i, end, paired)); }
        for (j = i; j < end; j++) {
            f = p.fb[j];
            bool keep = false;
            if (f & FB_INPOOL) {
                const int c = mate_class(f);
                const bool act = paired ? (c == 1 || c == 2) : (c == 0);
                const int32_t s = p.score[j];
                int32_t b = INT32_MIN, n = 0;
#pragma unroll
                for (int k = 0; k < 4; k++) if (k == c) { b = best[k]; n = cnt[k]; }
                keep = act && s == b && (!p.uniq || n == 1);
            }
            const uint32_t nf = keep ? (f | FB_KEEP) : (f & ~FB_KEEP);
            if (nf != f) p.fb[j] = nf;
        }
    }
}

// Emission.  kbase[i] = number of kept records before record i (exclusive scan of FB_KEEP).
// A pool's winners go out as: all READ1-class (or unpaired) winners in input order, then
// all READ2-class winners (msam_filter.c:247-254), starting at kbase[first record of the run].
__global__ void __launch_bounds__(256) besthit_warp_emit_kernel(const uint32_t *fb, const uint32_t *kbase, uint32_t *out_idx, uint64_t n)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t w0 = i & ~31ull;
    if (w0 >= n) return;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t f = i < n ? fb[i] : 0u;
    uint32_t nf = 0;
    if (lane == 31 && w0 + 32 < n) nf = fb[w0 + 32];
    nf = __shfl_sync(0xffffffffu, nf, 31);
    const RunView v = run_view(f, i, n, w0 + 32 >= n || !(nf & FB_EQPREV));
    const bool keep = i < n && !v.crossing && (f & FB_KEEP);
    const bool r2 = mate_class(f) == 2;
    const uint32_t k1 = __ballot_sync(0xffffffffu, keep && !r2) & v.segmask;
    const uint32_t k2 = __ballot_sync(0xffffffffu, keep && r2) & v.segmask;
    const uint32_t base = __shfl_sync(0xffffffffu, i < n ? kbase[i] : 0u, (int)v.s);
    if (keep) {
        const uint32_t below = (1u << lane) - 1u;
        const uint32_t rank = r2 ? __popc(k1) + __popc(k2 & below) : __popc(k1 & below);
        out_idx[base + rank] = (uint32_t)i;
    }
}

__global__ void __launch_bounds__(256) besthit_walk_emit_kernel(const uint32_t *fb, const uint32_t *kbase, uint32_t *out_idx, uint64_t n,
                                                                const uint32_t *worklist, const uint32_t *wl_count)
{
    const uint32_t nw = *wl_count;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nw; q += gridDim.x * blockDim.x) {
        const uint64_t i = worklist[q];
        uint32_t c1 = 0;
        uint64_t j = i;
        for (;;) {
            const uint32_t f = fb[j];
            if (j > i && !(f & FB_EQPREV)) break;
            if ((f & FB_KEEP) && mate_class(f) != 2) c1++;
            if (++j >= n) break;
        }
        const uint64_t end = j;
        uint32_t w1 = kbase[i], w2 = w1 + c1;
        for (j = i; j < end; j++) {
            const uint32_t f = fb[j];
            if (f & FB_KEEP) { if (mate_class(f) == 2) out_idx[w2++] = (uint32_t)j; else out_idx[w1++] = (uint32_t)j; }
        }
    }
}

// ---- scan functors -----------------------------------------------------------------------
struct InFlagBit {           // 1 where (fb & mask) == want
    const uint32_t *fb; uint32_t mask, want;
    __device__ __forceinline__ uint32_t operator()(uint64_t i) const { return (fb[i] & mask) == want ? 1u : 0u; }
};
struct InU32 { const uint32_t *v; __device__ __forceinline__ uint32_t operator()(uint64_t i) const { return v[i]; } };
struct OutExclU32 { uint32_t *o; __device__ __forceinline__ void operator()(uint64_t i, uint32_t ex, uint32_t) const { o[i] = ex; } };
struct OutInclU32 { uint32_t *o; __device__ __forceinline__ void operator()(uint64_t i, uint32_t ex, uint32_t v) const { o[i] = ex + v; } };
struct OutCompact {          // stable compaction: out[ex] = i where the flag was set
    uint32_t *o; __device__ __forceinline__ void operator()(uint64_t i, uint32_t ex, uint32_t v) const { if (v) o[ex] = (uint32_t)i; }
};

} // namespace msg
