// fused.cuh -- `filter --besthit|--uniqhit ... | profile` in one pass over the SoA columns.
//
// When the only consumer of the filter stage is the profile stage (no record output, no kept
// list, no coverage) the kept-record stream never has to exist: a QNAME pool (run of equal
// names, besthit.cuh) is also a profile group, PROVIDED no two consecutive non-empty pools
// carry the same QNAME (then the reference's profile would merge them, msam_profile.c:226).
// This kernel therefore does, per 32-record window and without leaving registers:
//   pool heads by ballot -> per (pool, mate class) best score / ties (MATCH.ANY + REDUX.MAX)
//   -> winners in reference order (READ1-class first, msam_filter.c:247-254)
//   -> distinct features in first-appearance order of THAT order (msam_profile.c:136-142)
//   -> share rule (msam_profile.c:65-200) into chunk-local accumulators and list storage.
// Pools that straddle a window go to a worklist (fused_walk_kernel, one thread per pool).
// fused_guard_kernel then checks the proviso exactly (32-bit QNAME hashes of consecutive
// non-empty pools must differ); if it fails -- possible only on input that is not QNAME-grouped,
// or on a hash collision -- the chunk's accumulators are discarded and the general
// stream-based pipeline (besthit.cuh + profile.cuh) runs instead.  Results are identical
// either way; tests/test_gpu_parity.py::test_reopened_* exercises the fallback.
#pragma once
#include "common.cuh"
#include "besthit.cuh"

namespace msg {

struct WinInfo { uint32_t first_hash, last_hash, n_nonempty, cross_hash; };   // cross_hash valid iff bit 31 of n_nonempty

struct FusedParams {
    uint32_t *fb; const int32_t *score; const int32_t *tid; const uint32_t *hash;
    const int32_t *fmap; int32_t n_targets, n_features;
    uint64_t n;
    int uniq, share_type;
    uint32_t *ui; double *d;          // chunk-local accumulators [F]
    uint32_t *cnt;                    // [0] inserts [1] uniq [2] multi [3] guard/fallback flag [4] kept records
    uint32_t *cursor;                 // [0] lists [1] entries (global, persistent across chunks)
    uint32_t *l_start, *l_len; int32_t *l_fid;
    uint32_t *worklist, *wl_count;
    WinInfo *win;                     // [ceil(n/32)]
    uint32_t big_threshold;
    uint32_t *err;
    unsigned long long *l_key;        // exact mode: [list] key_base + position of the list's group in the chunk (input order)
    unsigned long long key_base;      // records pushed before this chunk
};

// Whether the chunk writes multi-mapper lists: PropSharing always; with EXACT (msg_config.exact) also --multi=equal, whose
// 1/n shares are then summed at finish in input order instead of by atomics.
template <bool EXACT> __device__ __forceinline__ bool fused_lists(const FusedParams &p) { return p.share_type == 3 || (EXACT && p.share_type == 2); }

__device__ __forceinline__ int32_t fused_feature(const FusedParams &p, int32_t t) { return p.fmap ? p.fmap[t] : t; }

template <bool SMEM_HIST, bool EXACT>
__global__ void __launch_bounds__(256) fused_warp_kernel(const FusedParams p)
{
    extern __shared__ uint32_t s_hist[];
    __shared__ uint32_t s_cnt[4];
    __shared__ __align__(16) int32_t s_best[8][128];
    if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
    if (SMEM_HIST) for (uint32_t k = threadIdx.x; k < (uint32_t)p.n_features; k += blockDim.x) s_hist[k] = 0;
    __syncthreads();
    uint32_t *ui = SMEM_HIST ? s_hist : p.ui;

    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t w0 = i & ~31ull;
    const uint32_t lane = threadIdx.x & 31u;
    // proportional-mode list allocation state (filled per lane below, consumed after the CTA-wide allocation)
    uint32_t w_lists = 0, w_ents = 0, l_rank = 0, e_off = 0, e_off_group = 0, f_rank = 0, my_nd = 0; int32_t my_feat = -1;
    bool is_lhead = false, writes_fid = false;
    if (w0 < p.n) {
        const uint32_t f = i < p.n ? p.fb[i] : 0u;
        uint32_t nf = 0;
        if (lane == 31 && w0 + 32 < p.n) nf = p.fb[w0 + 32];
        nf = __shfl_sync(0xffffffffu, nf, 31);
        const RunView v = run_view(f, i, p.n, w0 + 32 >= p.n || !(nf & FB_EQPREV));
        if (v.is_open_head) { const uint32_t slot = atomicAdd(p.wl_count, 1u); p.worklist[slot] = (uint32_t)i; }
        __syncwarp();

        // ---- best-hit selection (same as besthit_warp_select_kernel)
        const bool mine = i < p.n && !v.crossing;
        const bool pooled = mine && (f & FB_INPOOL);
        const int cls = mate_class(f);
        const bool paired = (__ballot_sync(0xffffffffu, pooled && cls != 0) & v.segmask) != 0;
        const bool act = pooled && (paired ? (cls == 1 || cls == 2) : true);
        if (act && !(f & FB_HAS_AS)) { atomicOr(p.err, DERR_NOAS); atomicMin(p.err + 1, (uint32_t)i); }
        const int32_t sc = act ? p.score[i] : INT32_MIN;
        const bool keep = pool_winner(s_best[threadIdx.x >> 5], lane, act, sc, v.s * 4u + (uint32_t)cls, p.uniq);

        // ---- profile group = the pool's winners with tid != -1, READ1-class first
        int32_t t = keep ? p.tid[i] : -1;
        bool member = keep && t != -1;
        if (member && (t < 0 || t >= p.n_targets)) { atomicOr(p.err, DERR_FORMAT); member = false; }
        const int32_t feat = member ? fused_feature(p, t) : -1;
        const bool r2 = cls == 2;
        const uint32_t memmask = __ballot_sync(0xffffffffu, member);
        const uint32_t r1mask = __ballot_sync(0xffffffffu, member && !r2);
        const uint32_t gmask = memmask & v.segmask;
        const unsigned long long fkey = member ? (((unsigned long long)v.s << 32) | (uint32_t)feat) : ((1ull << 40) | lane);
        const uint32_t fm_all = __match_any_sync(0xffffffffu, fkey);
        const uint32_t fm_r1 = fm_all & r1mask;
        const bool first = member && lane == (uint32_t)__ffs((int)(fm_r1 ? fm_r1 : fm_all)) - 1u;
        const uint32_t firsts = __ballot_sync(0xffffffffu, first) & v.segmask;
        const uint32_t nd = __popc(firsts), size = __popc(gmask);
        const bool ghead = member && lane == (uint32_t)__ffs((int)gmask) - 1u;
        const bool multi = nd > 1;
        if (member) {
            if (!multi) { if (ghead) atomicAdd(ui + feat, 2u); }
            else if (first && p.share_type != 3) {
                if (p.share_type == 1) atomicAdd(ui + feat, 2u);
                else if (p.share_type == 2) { if (size == 2) atomicAdd(ui + feat, 1u); else if (!EXACT) atomicAdd(p.d + feat, 1.0 / (int)nd); }
            }
        }
        // proportional: list space for this warp's multi-feature groups = (lists, entries); offsets inside the warp by ballot / scan
        if (fused_lists<EXACT>(p)) {
            const bool glist = multi && (p.share_type == 3 || size != 2);          // equal: the two-record case adds to ui
            const bool lhead = ghead && glist;
            const uint32_t lmask = __ballot_sync(0xffffffffu, lhead);
            uint32_t x = lhead ? nd : 0u, incl = x;                                   // inclusive scan of list lengths over lanes
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += u; }
            w_lists = (uint32_t)__popc(lmask); w_ents = __shfl_sync(0xffffffffu, incl, 31);
            l_rank = (uint32_t)__popc(lmask & ((1u << lane) - 1u)); e_off = incl - x;
            is_lhead = lhead; my_nd = nd; my_feat = feat;
            const uint32_t gl = gmask ? (uint32_t)__ffs((int)gmask) - 1u : 0u;
            e_off_group = __shfl_sync(0xffffffffu, e_off, (int)gl);                    // entry offset of my group's list (within the warp)
            if (first && glist) {
                const uint32_t below = (1u << lane) - 1u;
                const uint32_t f1 = firsts & r1mask, f2 = firsts & ~r1mask;
                f_rank = r2 ? __popc(f1) + __popc(f2 & below) : __popc(f1 & below);
                writes_fid = true;
            }
        }
        // ---- window summary for the guard: hashes of the first / last non-empty complete pools,
        //      and adjacent non-empty pools inside the window must already differ
        const uint32_t h = ghead ? p.hash[i] : 0u;
        const uint32_t gheads = __ballot_sync(0xffffffffu, ghead);
        const uint32_t mheads = __ballot_sync(0xffffffffu, ghead && multi);
        const uint32_t lowg = gheads & ((1u << lane) - 1u);
        const int pg = lowg ? 31 - __clz((int)lowg) : 0;
        const uint32_t ph = __shfl_sync(0xffffffffu, h, pg);
        if (ghead && lowg && ph == h) atomicOr(p.cnt + 3, 1u);
        const uint32_t fh = __shfl_sync(0xffffffffu, h, gheads ? __ffs((int)gheads) - 1 : 0);
        const uint32_t lh = __shfl_sync(0xffffffffu, h, gheads ? 31 - __clz((int)gheads) : 0);
        const uint32_t keptmask = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) {
            WinInfo wi; wi.first_hash = fh; wi.last_hash = lh; wi.n_nonempty = (uint32_t)__popc(gheads); wi.cross_hash = 0;
            p.win[w0 >> 5] = wi;
            if (gheads) {
                atomicAdd(&s_cnt[0], (uint32_t)__popc(gheads));
                atomicAdd(&s_cnt[1], (uint32_t)__popc(gheads & ~mheads));
                atomicAdd(&s_cnt[2], (uint32_t)__popc(mheads));
            }
            if (keptmask) atomicAdd(&s_cnt[3], (uint32_t)__popc(keptmask));
        }
    }
    // ---- proportional: ONE pair of global atomics per CTA reserves list slots and entries for all of its warps
    __shared__ uint32_t s_wl[8], s_we[8], s_base[2];
    if (fused_lists<EXACT>(p)) {
        const uint32_t wid = threadIdx.x >> 5;
        if (lane == 0) { s_wl[wid] = w_lists; s_we[wid] = w_ents; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tl = 0, te = 0;
            for (int k = 0; k < 8; k++) { const uint32_t a = s_wl[k], b = s_we[k]; s_wl[k] = tl; s_we[k] = te; tl += a; te += b; }
            s_base[0] = tl ? atomicAdd(p.cursor + 0, tl) : 0u;
            s_base[1] = te ? atomicAdd(p.cursor + 1, te) : 0u;
        }
        __syncthreads();
        const uint32_t lbase = s_base[0] + s_wl[wid], ebase = s_base[1] + s_we[wid];
        if (is_lhead) { p.l_start[lbase + l_rank] = ebase + e_off; p.l_len[lbase + l_rank] = my_nd; if (EXACT) p.l_key[lbase + l_rank] = p.key_base + i; }
        if (writes_fid) p.l_fid[ebase + e_off_group + f_rank] = my_feat;
    }
    __syncthreads();
    if (threadIdx.x < 3 && s_cnt[threadIdx.x]) atomicAdd(p.cnt + threadIdx.x, s_cnt[threadIdx.x]);
    if (threadIdx.x == 3 && s_cnt[3]) atomicAdd(p.cnt + 4, s_cnt[3]);
    if (SMEM_HIST) for (uint32_t k = threadIdx.x; k < (uint32_t)p.n_features; k += blockDim.x) { const uint32_t c = s_hist[k]; if (c) atomicAdd(p.ui + k, c); }
}

// One thread per pool that straddles a window: the head walks its run twice (best score per mate
// class, then the winners) and finishes the group from a small local list.  Pools longer than
// big_threshold records or with more than FUSED_MAXM winners send the chunk to the general pipeline.
constexpr int FUSED_MAXM = 48;    // distinct features per walked pool (more: the chunk goes to the general pipeline)
constexpr int FUSED_PF = 8;       // records whose columns are prefetched per walked pool
constexpr int FUSED_DR = 8;       // distinct features kept in registers

template <bool EXACT>
__global__ void __launch_bounds__(128) fused_walk_kernel(const FusedParams p)
{
    const uint32_t nw = *p.wl_count;
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t ins = 0, uq = 0, mu = 0, keptn = 0;
    // warp-uniform trip count, so that the list-space allocation below can be aggregated per warp
    for (uint32_t qb = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; qb < nw; qb += gridDim.x * blockDim.x) {
      const uint32_t q = qb + lane;
      int32_t df[FUSED_MAXM]; uint32_t dr[FUSED_DR]; uint32_t nd = 0, nm = 0; bool emit = false;
      uint64_t i = 0;
#pragma unroll
      for (int k = 0; k < FUSED_DR; k++) dr[k] = 0xffffffffu;
      // k-th distinct feature: registers first, local-memory list beyond FUSED_DR
#pragma nv_diag_suppress 549      // df[k] is only read for k >= FUSED_DR, which add_feature has written by then
      auto feat_at = [&](uint32_t k) -> int32_t {
          int32_t v = k >= FUSED_DR ? df[k] : 0;
#pragma unroll
          for (int j = 0; j < FUSED_DR; j++) if ((uint32_t)j == k) v = (int32_t)dr[j];
          return v;
      };
#pragma nv_diag_default 549
      if (q < nw) do {
        i = p.worklist[q];
        // The walk is latency bound (one thread per pool, dependent loads), so the first FUSED_PF records' columns are
        // fetched up front with independent loads; both passes then run out of registers for the usual short pool
        // and only touch memory again for the rare records beyond the prefetch.
        uint32_t fr[FUSED_PF]; int32_t sr[FUSED_PF], tr[FUSED_PF];
#pragma unroll
        for (int k = 0; k < FUSED_PF; k++) {
            const uint64_t j = i + k; const bool ok = j < p.n;
            fr[k] = ok ? p.fb[j] : 0u; sr[k] = ok ? p.score[j] : 0; tr[k] = ok ? p.tid[j] : -1;
        }
        uint32_t len = 1; bool open = true;                                  // run = i plus the following FB_EQPREV records
#pragma unroll
        for (int k = 1; k < FUSED_PF; k++) { open = open && (fr[k] & FB_EQPREV); len += open; }
        uint64_t end = i + len;
        if (open) { while (end < p.n && (p.fb[end] & FB_EQPREV)) end++; }
        if (end - i > p.big_threshold) { atomicOr(p.cnt + 3, 1u); break; }
        // pass 1: per mate class best / ties, pairedness (msam_filter.c:196-230)
        int32_t b0 = INT32_MIN, b1 = INT32_MIN, b2 = INT32_MIN; uint32_t c0 = 0, c1 = 0, c2 = 0;
        uint32_t noas = 0; bool paired = false;
        auto pass1 = [&](uint32_t f, int32_t sc) {
            if (!(f & FB_INPOOL)) return;
            const int c = mate_class(f);
            paired |= (c != 0);
            if (!(f & FB_HAS_AS)) noas |= 1u << c;
            if (c == 0) { if (sc > b0) { b0 = sc; c0 = 1; } else if (sc == b0) c0++; }
            else if (c == 1) { if (sc > b1) { b1 = sc; c1 = 1; } else if (sc == b1) c1++; }
            else if (c == 2) { if (sc > b2) { b2 = sc; c2 = 1; } else if (sc == b2) c2++; }
        };
#pragma unroll
        for (int k = 0; k < FUSED_PF; k++) if ((uint32_t)k < len) pass1(fr[k], sr[k]);
        for (uint64_t j = i + FUSED_PF; j < end; j++) pass1(p.fb[j], p.score[j]);
        if (paired ? (noas & 6u) : (noas & 1u)) { atomicOr(p.err, DERR_NOAS); atomicMin(p.err + 1, noas_record(p.fb, i, end, paired)); }
        // pass 2: the winners' features, distinct, in the order READ1-class winners then READ2-class winners, each in input
        // order (msam_filter.c:247-254 -> msam_profile.c:136-142).  Two sweeps over the run (the usual short pool sits in the
        // prefetched registers); the first FUSED_DR distinct features live in registers (compare / insert fully unrolled),
        // only larger sets touch the local-memory list.
        bool overflow = false;
        auto add_feature = [&](int32_t fe) {
            bool seen = false;
#pragma unroll
            for (int k = 0; k < FUSED_DR; k++) seen |= (dr[k] == (uint32_t)fe);
            for (uint32_t d2 = FUSED_DR; d2 < nd && !seen; d2++) seen = (df[d2] == fe);
            if (seen) return;
            if (nd >= FUSED_MAXM) { overflow = true; return; }
#pragma unroll
            for (int k = 0; k < FUSED_DR; k++) if ((uint32_t)k == nd) dr[k] = (uint32_t)fe;
            if (nd >= FUSED_DR) df[nd] = fe;
            nd++;
        };
        auto pass2 = [&](uint32_t f, int32_t sc, int32_t tt, int want_r2) {
            if (overflow || !(f & FB_INPOOL)) return;
            const int c = mate_class(f);
            if (paired ? !(c == 1 || c == 2) : c != 0) return;
            if ((c == 2) != (want_r2 != 0)) return;
            const int32_t bb = c == 0 ? b0 : (c == 1 ? b1 : b2); const uint32_t cc = c == 0 ? c0 : (c == 1 ? c1 : c2);
            if (sc != bb || (p.uniq && cc != 1)) return;
            keptn++;
            if (tt == -1) return;
            if (tt < 0 || tt >= p.n_targets) { atomicOr(p.err, DERR_FORMAT); return; }
            nm++;
            add_feature(fused_feature(p, tt));
        };
        for (int ph = 0; ph < 2; ph++) {
#pragma unroll
            for (int k = 0; k < FUSED_PF; k++) if ((uint32_t)k < len) pass2(fr[k], sr[k], tr[k], ph);
            for (uint64_t j = i + FUSED_PF; j < end; j++) pass2(p.fb[j], p.score[j], p.tid[j], ph);
        }
        if (overflow) { atomicOr(p.cnt + 3, 1u); nm = 0; nd = 0; break; }
        if (nm == 0) break;
        emit = true;
      } while (0);
      if (emit) {
        WinInfo *wi = p.win + (i >> 5);
        wi->cross_hash = p.hash[i];
        atomicOr(&wi->n_nonempty, 0x80000000u);
        ins++;
        if (nd == 1) { atomicAdd(p.ui + dr[0], 2u); uq++; }
        else {
            mu++;
            if (p.share_type == 1) { for (uint32_t k = 0; k < nd; k++) atomicAdd(p.ui + feat_at(k), 2u); }
            else if (p.share_type == 2) {
                if (nm == 2) { atomicAdd(p.ui + dr[0], 1u); atomicAdd(p.ui + dr[1], 1u); }
                else if (!EXACT) { const double share = 1.0 / (int)nd; for (uint32_t k = 0; k < nd; k++) atomicAdd(p.d + feat_at(k), share); }
            }
        }
      }
      if (fused_lists<EXACT>(p)) {        // one pair of atomics per warp reserves the list slots / entries of its multi-feature groups
        const bool lhead = emit && nd > 1 && (p.share_type == 3 || nm != 2);
        const uint32_t lmask = __ballot_sync(0xffffffffu, lhead);
        uint32_t x = lhead ? nd : 0u, incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (uint32_t)o) incl += u; }
        const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
        uint32_t lb = 0, eb = 0;
        if (lane == 0 && lmask) { lb = atomicAdd(p.cursor + 0, (uint32_t)__popc(lmask)); eb = atomicAdd(p.cursor + 1, tot); }
        lb = __shfl_sync(0xffffffffu, lb, 0); eb = __shfl_sync(0xffffffffu, eb, 0);
        if (lhead) {
            const uint32_t li = lb + (uint32_t)__popc(lmask & ((1u << lane) - 1u)), base = eb + incl - x;
            p.l_start[li] = base; p.l_len[li] = nd;
            if (EXACT) p.l_key[li] = p.key_base + i;          // the pool's first record: any position inside the group orders alike
#pragma unroll
            for (int k = 0; k < FUSED_DR; k++) if ((uint32_t)k < nd) p.l_fid[base + k] = (int32_t)dr[k];
            for (uint32_t k = FUSED_DR; k < nd; k++) p.l_fid[base + k] = df[k];
        }
      }
    }
    ins = __reduce_add_sync(0xffffffffu, ins); uq = __reduce_add_sync(0xffffffffu, uq);
    mu = __reduce_add_sync(0xffffffffu, mu); keptn = __reduce_add_sync(0xffffffffu, keptn);
    if (lane == 0) {
        if (ins) atomicAdd(p.cnt + 0, ins);
        if (uq) atomicAdd(p.cnt + 1, uq);
        if (mu) atomicAdd(p.cnt + 2, mu);
        if (keptn) atomicAdd(p.cnt + 4, keptn);
    }
}

// Order of pools: for w = 0,1,...: the complete pools of window w, then the pool that starts in w
// and leaves it.  Consecutive NON-EMPTY pools must have different QNAME hashes (then their names
// differ and the reference's profile keeps them apart too).  One thread per window.
__global__ void __launch_bounds__(256) fused_guard_kernel(const WinInfo *win, uint32_t nwin, uint32_t *flag)
{
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nwin) return;
    const WinInfo me = win[w];
    const uint32_t ncomp = me.n_nonempty & 0x7fffffffu; const bool cross = me.n_nonempty >> 31;
    if (!ncomp && !cross) return;
    if (ncomp && cross && me.last_hash == me.cross_hash) { atomicOr(flag, 1u); return; }
    const uint32_t my_first = ncomp ? me.first_hash : me.cross_hash;
    for (uint32_t k = w; k-- > 0;) {                       // last non-empty pool before this window
        const WinInfo o = win[k];
        const uint32_t oc = o.n_nonempty & 0x7fffffffu; const bool ox = o.n_nonempty >> 31;
        if (!oc && !ox) continue;
        if ((ox ? o.cross_hash : o.last_hash) == my_first) atomicOr(flag, 1u);
        return;
    }
}

// commit the chunk-local accumulators: ui += ui_tmp, d += d_tmp (then clear them for the next chunk).  Launched before
// the host has seen the guard flag, so the decision is repeated here on the device; a declined chunk also gives its
// list space back (cursor[2..3] = the cursors before the chunk), so that the next chunk may already be queued behind it.
__global__ void __launch_bounds__(256) fused_commit_kernel(uint32_t *ui, double *d, uint32_t *ui_tmp, double *d_tmp, uint32_t F, int use_d,
                                                           uint32_t *counters, uint32_t *cnt_tmp, uint32_t *cursor)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    const bool tripped = cnt_tmp[3] != 0;          // guard flag: drop the chunk's partial sums (the host reruns it on the general path)
    if (k == 0 && tripped) { cursor[0] = cursor[2]; cursor[1] = cursor[3]; }
    if (k < F) {
        const uint32_t a = ui_tmp[k]; if (a) { if (!tripped) ui[k] += a; ui_tmp[k] = 0; }
        if (use_d) { const double b = d_tmp[k]; if (b != 0.0) { if (!tripped) d[k] += b; d_tmp[k] = 0.0; } }
    }
    if (k < 3 && !tripped) { counters[k] += cnt_tmp[k]; }
}

} // namespace msg
