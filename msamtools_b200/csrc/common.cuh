// common.cuh -- shared definitions for the sm_100a kernels of libmsamtools_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

// ---- per-record packed column `fb` (u32): low 16 bits = BAM FLAG -----------------------
#define FB_FLAG_MASK 0x0000ffffu
#define FB_INPOOL    (1u << 16)   // record entered the QNAME pool (msam_filter.c:181-183 / :132-136)
#define FB_HAS_AS    (1u << 17)   // AS present (or rescored)      (msam_filter.c:219-221)
#define FB_EQPREV    (1u << 18)   // QNAME byte-identical to the previous record's
#define FB_SLOW      (1u << 19)   // parsed through the global-memory slow path
#define FB_KEEP      (1u << 20)   // survived best-hit selection   (msam_filter.c:235-244)

// ---- device error word (ctx->d_err[0]) ---------------------------------------------------
#define DERR_NOTAG   1u           // mapped record without NM and MD while stats are needed
#define DERR_NOAS    2u           // best-hit candidate without AS
#define DERR_FORMAT  4u           // malformed record / tid out of range
#define DERR_CGTAG   8u           // CIGAR of more than 65535 operations stored in the CG tag (SAM spec 4.2.2): not expanded here

#define BAM_FUNMAP 4u
#define BAM_FREAD1 0x40u
#define BAM_FREAD2 0x80u

// decode kernel mode bits
#define DM_DO_FILTER   (1u << 0)
#define DM_HAS_FILTER  (1u << 1)   // any of -l/-p/-z active (filter != NULL, msam_filter.c:79-85)
#define DM_NEED_STATS  (1u << 2)   // filter != NULL || rescore (msam_filter.c:104)
#define DM_INVERT      (1u << 3)
#define DM_KEEP_UNMAP  (1u << 4)
#define DM_RESCORE     (1u << 5)
#define DM_NEED_AS     (1u << 6)   // best-hit writers read AS
#define DM_WANT_HASH   (1u << 7)
#define DM_COV_FUSED   (1u << 8)
#define DM_FORCE_SLOW  (1u << 9)
#define DM_NEED_CIGAR  (1u << 10)
#define DM_NEED_AUX    (1u << 11)
#define DM_REQ_STATS   (1u << 12)  // reference's need_alignment_stats: a mapped record without NM/MD is fatal
#define DM_COV_BITS    (1u << 13)  // coverage in summary mode: one bit per position + per-target sums

__device__ __forceinline__ uint4 ldg_stream128(const uint4 *p)
{
    // streaming 16-byte load: record bytes are touched once, keep them out of L1.  The L2::64B qualifier matters: a
    // plain load makes B200's L2 fill whole 128-byte lines from HBM (measured: 2.34 GB of DRAM reads per 10 M records,
    // 1.70 GB with the qualifier) although the decode windows only need ~129 B of 32-byte sectors per 295-byte record.
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
// same without the qualifier (L2 fills whole 128-byte lines)
__device__ __forceinline__ uint4 ldg_stream128_line(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
