// collate.cuh -- grouping records by QNAME on the device, for input in any order (msg_config.collate).
//
// Push: collate_size_kernel validates every record with decode's rules and sizes its HEAD (the record without SEQ/QUAL);
// collate_gather_kernel appends the head to the context's arena as a pseudo-record (l_seq = 0, block_size adjusted) and
// writes a key {64-bit QNAME hash, input ordinal}.  Finish: one counting-sort pass partitions the keys by the top bits of
// the hash (histogram, run_scan, scatter), every bucket is sorted by (hash, ordinal) -- in shared memory, or in global
// memory for buckets too large for it -- and runs of equal hash whose names differ are re-sorted by (name bytes, ordinal).
// collate_grouped_gather_kernel then writes the heads in that order, which the decode pipeline takes as a device chunk.
// DESIGN.md §11 has the layout and the exactness argument.
#pragma once
#include "common.cuh"

namespace msg {

struct CollKey { unsigned long long hash; uint32_t ord, pad; };     // 16 bytes

constexpr uint32_t COLL_SMEM_KEYS = 2048;         // largest bucket sorted in shared memory (32 KB)
constexpr uint32_t COLL_BUCKET_AVG = 512;         // target mean bucket size: buckets past COLL_SMEM_KEYS are rare for distinct names

__device__ __forceinline__ uint32_t coll_ld32(const uint8_t *p)
{
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

__device__ __forceinline__ unsigned long long coll_mix64(unsigned long long x)
{   // splitmix64 finaliser
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull; x ^= x >> 27; x *= 0x94d049bb133111ebull; return x ^ (x >> 31);
}

// Validation (same rules and MSG_EFORMAT as decode_kernel) and the head length of each record: len[i] = record length
// minus SEQ and QUAL, 0 for a malformed record.  err[1] gets the INPUT ordinal (base_ord + i) of the first bad record.
// check_cg: the pipeline reads CIGARs (decode's DM_NEED_CIGAR), where decode refuses the CG-tag placeholder "<l_seq>S<n>N".
// The test must use the original l_seq: the pseudo-record has l_seq = 0 and would never trip it.
__global__ void __launch_bounds__(256) collate_size_kernel(const uint8_t *raw, const uint64_t *off, uint64_t n, uint64_t nbytes,
                                                           uint32_t base_ord, bool check_cg, uint32_t *len, uint32_t *err)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t o = off[i], o1 = off[i + 1];
    bool bad = !(o1 <= nbytes && o <= o1);
    const uint64_t len64 = bad ? 0 : o1 - o;
    bad = bad || len64 < 36 || len64 > 0x7fffffffull;
    uint32_t L = 0;
    if (!bad) {
        const uint8_t *r = raw + o;
        const uint32_t lq = r[12], nc = (uint32_t)r[16] | ((uint32_t)r[17] << 8);
        const int32_t lseq = (int32_t)coll_ld32(r + 20);
        const uint64_t sq = lseq < 0 ? 0 : (((uint64_t)lseq + 1) >> 1) + (uint64_t)lseq;
        if (lseq < 0 || 36ull + lq + 4ull * nc + sq > len64) bad = true;
        else {
            L = (uint32_t)(len64 - sq);
            if (check_cg && nc == 2 && lseq > 0 && coll_ld32(r + 36 + lq) == (((uint32_t)lseq << 4) | 4u) && (coll_ld32(r + 40 + lq) & 0xfu) == 3u) {
                atomicOr(err, DERR_CGTAG); atomicMin(err + 1, base_ord + (uint32_t)i);
            }
        }
    }
    if (bad) { atomicOr(err, DERR_FORMAT); atomicMin(err + 1, base_ord + (uint32_t)i); L = 0; }
    len[i] = L;
}

// One warp per record: copy the head (block_size, core, name, CIGAR) and the aux block to arena + aoff[i], with block_size
// = head length - 4 and l_seq = 0, and write the key.  The 64-bit QNAME hash covers l_read_name and the name bytes
// (equal names hash equal); hash_mask keeps its top bits only (MSG_COLLATE_HASH_BITS, tests).
__global__ void __launch_bounds__(256) collate_gather_kernel(const uint8_t *raw, const uint64_t *off, uint64_t n, const unsigned long long *aoff,
                                                             const uint32_t *len, uint8_t *arena, CollKey *keys, uint32_t base_ord,
                                                             unsigned long long hash_mask)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t nw = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += nw) {
        const uint8_t *src = raw + off[i];
        uint8_t *dst = arena + aoff[i];
        const uint32_t L = len[i];
        const uint32_t lq = src[12], nc = (uint32_t)src[16] | ((uint32_t)src[17] << 8);
        const uint32_t lseq = coll_ld32(src + 20);
        const uint32_t head = 36u + lq + 4u * nc, skip = ((lseq + 1u) >> 1) + lseq;
        const uint32_t bs = L - 4u;
        for (uint32_t k = lane; k < head; k += 32) {
            uint8_t b = src[k];
            if (k < 4) b = (uint8_t)(bs >> (8 * k));
            else if (k >= 20 && k < 24) b = 0;
            dst[k] = b;
        }
        for (uint32_t k = head + lane; k < L; k += 32) dst[k] = src[k + skip];
        // hash: every lane mixes its 32-bit words of the name with their position; the sum over the warp is order-free
        unsigned long long h = 0;
        for (uint32_t w = lane; 4 * w < lq; w += 32) {
            const uint32_t rem = lq - 4 * w;
            uint32_t x = 0;
            for (uint32_t b = 0; b < 4 && b < rem; b++) x |= (uint32_t)src[36 + 4 * w + b] << (8 * b);
            h += coll_mix64(((unsigned long long)w << 32 | x) + 0x9E3779B97F4A7C15ull);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
        if (lane == 0) {
            CollKey key; key.hash = coll_mix64(h ^ ((unsigned long long)lq * 0xD6E8FEB86659FD93ull)) & hash_mask;
            key.ord = base_ord + (uint32_t)i; key.pad = 0;
            keys[i] = key;
        }
    }
}

// ---------------------------------------------------------------- partition by the top `bits` bits of the hash
__device__ __forceinline__ uint32_t coll_bucket(unsigned long long h, uint32_t bits) { return bits ? (uint32_t)(h >> (64 - bits)) : 0u; }

__global__ void __launch_bounds__(256) collate_hist_kernel(const CollKey *keys, uint64_t n, uint32_t bits, uint32_t *hist)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(hist + coll_bucket(keys[i].hash, bits), 1u);
}

// cursor[] starts as the exclusive scan of the histogram.  The order inside a bucket that the atomics produce does not
// matter: the bucket sort orders by (hash, ordinal), so the result equals that of a stable scatter.
__global__ void __launch_bounds__(256) collate_scatter_kernel(const CollKey *keys, uint64_t n, uint32_t bits, uint32_t *cursor, CollKey *out)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const CollKey k = keys[i];
    out[atomicAdd(cursor + coll_bucket(k.hash, bits), 1u)] = k;
}

// ---------------------------------------------------------------- sorting one range, by one CTA
struct CollLess {
    __device__ __forceinline__ bool operator()(const CollKey &a, const CollKey &b) const { return a.hash < b.hash || (a.hash == b.hash && a.ord < b.ord); }
};

// names of two keys: (l_read_name, bytes), then the ordinal
struct CollNameLess {
    const uint8_t *arena; const unsigned long long *aoff;
    __device__ bool operator()(const CollKey &a, const CollKey &b) const {
        const uint8_t *x = arena + aoff[a.ord], *y = arena + aoff[b.ord];
        if (x[12] != y[12]) return x[12] < y[12];
        for (uint32_t k = 0; k < x[12]; k++) if (x[36 + k] != y[36 + k]) return x[36 + k] < y[36 + k];
        return a.ord < b.ord;
    }
};

__device__ __forceinline__ bool coll_name_eq(const uint8_t *arena, const unsigned long long *aoff, uint32_t a, uint32_t b)
{
    const uint8_t *x = arena + aoff[a], *y = arena + aoff[b];
    if (x[12] != y[12]) return false;
    for (uint32_t k = 0; k < x[12]; k++) if (x[36 + k] != y[36 + k]) return false;
    return true;
}

// Bitonic network over a[0..m) (shared or global memory) with every comparator ascending: the first step of each merge
// compares mirrored positions.  Positions >= m act as +infinity, so a comparator whose upper position is >= m is skipped.
template <class Less>
__device__ void coll_bitonic(CollKey *a, uint32_t m, Less less)
{
    uint32_t P = 1; while (P < m) P <<= 1;
    for (uint32_t k = 2; k <= P; k <<= 1) {
        for (uint32_t d = k >> 1; d > 0; d >>= 1) {
            for (uint32_t t = threadIdx.x; t < P / 2; t += blockDim.x) {
                const uint32_t i = (t / d) * 2 * d + (t % d);
                const uint32_t j = d == (k >> 1) ? (i / k) * k + k - 1 - (i % k) : i + d;
                if (j < m) {
                    const CollKey x = a[i], y = a[j];
                    if (less(y, x)) { a[i] = y; a[j] = x; }
                }
            }
            __syncthreads();
        }
    }
}

// one CTA per bucket (grid-stride): buckets up to COLL_SMEM_KEYS keys are sorted in shared memory, larger ones are listed
// for collate_sort_global_kernel
__global__ void __launch_bounds__(256) collate_bucket_sort_kernel(CollKey *keys, const uint32_t *bstart, uint32_t nb, uint64_t n,
                                                                  uint32_t *big, uint32_t *nbig)
{
    __shared__ CollKey s[COLL_SMEM_KEYS];
    for (uint32_t b = blockIdx.x; b < nb; b += gridDim.x) {
        const uint32_t lo = bstart[b], hi = b + 1 < nb ? bstart[b + 1] : (uint32_t)n, m = hi - lo;
        if (m <= 1) continue;
        if (m > COLL_SMEM_KEYS) { if (threadIdx.x == 0) big[atomicAdd(nbig, 1u)] = b; continue; }
        for (uint32_t t = threadIdx.x; t < m; t += blockDim.x) s[t] = keys[lo + t];
        __syncthreads();
        coll_bitonic(s, m, CollLess{});
        for (uint32_t t = threadIdx.x; t < m; t += blockDim.x) keys[lo + t] = s[t];
        __syncthreads();
    }
}

// one CTA per listed range, sorted in place in global memory: oversized buckets (by hash, ordinal; one read with
// thousands of alignments is one) or, with by_name, runs of equal hash that hold different names
__global__ void __launch_bounds__(1024) collate_sort_global_kernel(CollKey *keys, const uint32_t *bstart, uint32_t nb, uint64_t n, const uint32_t *list,
                                                                   bool by_name, const uint8_t *arena, const unsigned long long *aoff)
{
    uint32_t lo, hi;
    if (by_name) { lo = list[2 * blockIdx.x]; hi = list[2 * blockIdx.x + 1]; }
    else { const uint32_t b = list[blockIdx.x]; lo = bstart[b]; hi = b + 1 < nb ? bstart[b + 1] : (uint32_t)n; }
    if (by_name) coll_bitonic(keys + lo, hi - lo, CollNameLess{arena, aoff});
    else         coll_bitonic(keys + lo, hi - lo, CollLess{});
}

// After the sort the keys are ordered by (hash, ordinal).  The head of every run of equal hash walks its run; if two
// neighbours' names differ (different names with one hash, which may interleave), the run [lo, hi) is listed for the
// by-name sort.  *nruns counts all such runs, even past cap.
__global__ void __launch_bounds__(256) collate_collide_kernel(const CollKey *keys, uint64_t n, const uint8_t *arena, const unsigned long long *aoff,
                                                              uint32_t *runs, uint32_t cap, uint32_t *nruns)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (i > 0 && keys[i - 1].hash == keys[i].hash)) return;
    const unsigned long long h = keys[i].hash;
    bool collide = false;
    uint64_t j = i + 1;
    for (; j < n && keys[j].hash == h; j++)
        if (!collide && !coll_name_eq(arena, aoff, keys[j - 1].ord, keys[j].ord)) collide = true;
    if (collide) {
        const uint32_t s = atomicAdd(nruns, 1u);
        if (s < cap) { runs[2 * s] = (uint32_t)i; runs[2 * s + 1] = (uint32_t)j; }
    }
}

struct InGroupedLen {          // head length of the record at grouped position i
    const CollKey *keys; const unsigned long long *aoff;
    __device__ __forceinline__ unsigned long long operator()(uint64_t i) const { const uint32_t o = keys[i].ord; return aoff[o + 1] - aoff[o]; }
};
struct OutExclU64Add { unsigned long long *o; unsigned long long base;
    __device__ __forceinline__ void operator()(uint64_t i, unsigned long long ex, unsigned long long) const { o[i] = base + ex; } };

// one warp per record: arena[aoff[ord]] -> grouped[goff[g]]
__global__ void __launch_bounds__(256) collate_grouped_gather_kernel(const CollKey *keys, uint64_t n, const uint8_t *arena, const unsigned long long *aoff,
                                                                     const unsigned long long *goff, uint8_t *grouped)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t nw = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t g = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < n; g += nw) {
        const uint32_t o = keys[g].ord;
        const uint8_t *src = arena + aoff[o];
        uint8_t *dst = grouped + goff[g];
        const uint32_t L = (uint32_t)(aoff[o + 1] - aoff[o]);
        for (uint32_t k = lane; k < L; k += 32) dst[k] = src[k];
    }
}

// ---------------------------------------------------------------- across ranks (MSG_COLLATE_RANKS, DESIGN.md §11)
// A record goes to rank floor(hash * N / 2^64): every rank holds one contiguous range of the hash space, so every QNAME
// (and every run of one hash) lands whole on one rank, and the ranks' ranges follow hash order.
__device__ __forceinline__ uint32_t coll_dest(unsigned long long h, uint32_t nr) { return (uint32_t)__umul64hi(h, (unsigned long long)nr); }

constexpr uint32_t COLL_DEST_TILE = 2048;         // keys per CTA of the destination partition (8 rounds of 256)

// Records and head bytes per destination: cnt[d * nblk + b] = records of tile b for rank d (for the stable scatter), and
// row[2d], row[2d + 1] += records, head bytes for rank d.  Dynamic shared memory: 12 * nr bytes.
__global__ void __launch_bounds__(256) collate_dest_count_kernel(const CollKey *keys, uint64_t n, uint32_t nr, const unsigned long long *aoff,
                                                                 uint32_t *cnt, uint32_t nblk, unsigned long long *row)
{
    extern __shared__ unsigned long long s_dyn[];
    unsigned long long *s_bytes = s_dyn;
    uint32_t *s_cnt = reinterpret_cast<uint32_t *>(s_dyn + nr);
    for (uint32_t t = threadIdx.x; t < nr; t += blockDim.x) { s_cnt[t] = 0; s_bytes[t] = 0; }
    __syncthreads();
    const uint64_t lo = (uint64_t)blockIdx.x * COLL_DEST_TILE;
    for (uint32_t r = 0; r < COLL_DEST_TILE; r += blockDim.x) {
        const uint64_t i = lo + r + threadIdx.x;
        if (i >= n) break;
        const uint32_t d = coll_dest(keys[i].hash, nr);
        atomicAdd(s_cnt + d, 1u);
        atomicAdd(s_bytes + d, aoff[i + 1] - aoff[i]);
    }
    __syncthreads();
    for (uint32_t t = threadIdx.x; t < nr; t += blockDim.x) {
        cnt[(uint64_t)t * nblk + blockIdx.x] = s_cnt[t];
        if (s_cnt[t]) { atomicAdd(row + 2 * t, (unsigned long long)s_cnt[t]); atomicAdd(row + 2 * t + 1, s_bytes[t]); }
    }
}

// Stable partition by destination: pos[] is the exclusive scan of collate_dest_count_kernel's cnt[], so the keys of one
// destination keep their input order (the receiver relies on it, see collate_recv_kernel).  out[] gets {hash, ord, head
// length in pad}.  Dynamic shared memory: 4 * nr * (blockDim / 32 + 1) bytes.
__global__ void __launch_bounds__(256) collate_dest_scatter_kernel(const CollKey *keys, uint64_t n, uint32_t nr, const unsigned long long *aoff,
                                                                   const uint32_t *pos, uint32_t nblk, CollKey *out)
{
    extern __shared__ uint32_t s_u32[];
    const uint32_t nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    uint32_t *s_off = s_u32, *s_w = s_u32 + nr;                     // s_w[w * nr + d]: keys of warp w for d in this round
    for (uint32_t t = threadIdx.x; t < nr; t += blockDim.x) {
        s_off[t] = pos[(uint64_t)t * nblk + blockIdx.x];
        for (uint32_t w = 0; w < nwarp; w++) s_w[w * nr + t] = 0;
    }
    __syncthreads();
    const uint64_t lo = (uint64_t)blockIdx.x * COLL_DEST_TILE;
    for (uint32_t r = 0; r < COLL_DEST_TILE && lo + r < n; r += blockDim.x) {
        const uint64_t i = lo + r + threadIdx.x;
        CollKey k; uint32_t d = 0xffffffffu;
        if (i < n) { k = keys[i]; d = coll_dest(k.hash, nr); }
        const uint32_t same = __match_any_sync(0xffffffffu, d);
        const uint32_t rank = __popc(same & ((1u << lane) - 1u));
        if (i < n && rank == 0) s_w[warp * nr + d] = __popc(same);
        __syncthreads();
        if (i < n) {
            uint32_t p = s_off[d] + rank;
            for (uint32_t w = 0; w < warp; w++) p += s_w[w * nr + d];
            k.pad = (uint32_t)(aoff[i + 1] - aoff[i]);
            out[p] = k;
        }
        __syncthreads();
        for (uint32_t t = threadIdx.x; t < nr; t += blockDim.x) {
            uint32_t s = 0;
            for (uint32_t w = 0; w < nwarp; w++) { s += s_w[w * nr + t]; s_w[w * nr + t] = 0; }
            s_off[t] += s;
        }
        __syncthreads();
    }
}

// After the send gather: input ordinals of this rank's records become global ones (records pushed by lower ranks + k).
__global__ void __launch_bounds__(256) collate_rebase_kernel(CollKey *keys, uint64_t n, uint32_t base)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i].ord += base;
}

// Received keys sit in source-rank order, and in input order within each source (stable scatter), so the receive
// position orders them exactly as their global ordinals do: the position becomes the key's ordinal (the arena index the
// sorts and gathers use), and gord[] keeps the global ordinal for error messages.
__global__ void __launch_bounds__(256) collate_recv_kernel(CollKey *keys, uint64_t n, uint32_t *gord)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    gord[i] = keys[i].ord;
    keys[i].ord = (uint32_t)i;
}

struct InKeyPadLen {           // head length carried in a received key's pad word
    const CollKey *keys;
    __device__ __forceinline__ unsigned long long operator()(uint64_t i) const { return keys[i].pad; }
};

// Chunk cuts: the largest grouped position s in (lo, hi] that starts a run of equal hash (*best, atomicMax), and the
// smallest such start in (hi, end) (*next, atomicMin).
__global__ void __launch_bounds__(256) collate_cut_kernel(const CollKey *keys, uint64_t lo, uint64_t hi, uint64_t end,
                                                          unsigned long long *best, unsigned long long *next)
{
    const uint64_t s = lo + 1 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= end || keys[s].hash == keys[s - 1].hash) return;
    if (s <= hi) atomicMax(best, (unsigned long long)s);
    else atomicMin(next, (unsigned long long)s);
}

} // namespace msg
