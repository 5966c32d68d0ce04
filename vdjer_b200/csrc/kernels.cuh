/*
 * kernels.cuh -- sm_100a device code of the V'DJer de Bruijn graph build.
 *
 * Implements the order-free form of the reference's hot path (SURVEY.md Appendix A); each kernel
 * cites the reference lines (/root/reference/src/main/c/assembler2_vdj.c) whose result it must
 * reproduce bit for bit.  Nothing here is a dense contraction: the work is integer/byte traffic
 * bounded by HBM and by L2 atomics, so tensor cores are not used.
 *
 * Design (see DESIGN.md): a hash table probed at random from 3e8 windows misses L2 on almost
 * every probe, and this B200 sustains only ~20 G random read-modify-writes/s out of HBM
 * (profiles/microbench_r1.json) against ~190 G/s inside its 126 MB L2.  So the windows are first
 * SCATTERED into hash partitions and both table passes then walk them partition by partition: the
 * slice of the table a partition addresses is a few MB and stays L2-resident, every probe and
 * atomic is an L2 hit, and HBM only sees streaming traffic.
 *
 * What is scattered is not one tuple per window but one RUN per stretch of consecutive windows
 * ("super-k-mer", KMC2 / Gerbil style): the partition of a k-mer is chosen by its MINIMIZER (the
 * smallest hashed m-mer inside it, m = 10), which consecutive windows of a read share, so a
 * stretch of up to 24 windows travels as one 32-byte record (its bases once, two flag bits per
 * window, the stamp of its first window, the read's fingerprint): 3-5 bytes per window instead of
 * 16.  The table passes expand a run back into its windows on the fly, in registers.
 *
 * Packed read layout in HBM (written by k_pack from the caller's text records, which the host
 * staging code in vdjgraph.cu streams to the device):
 *   bases [R][nb] u64 : 2 bits/base, A=0 C=1 G=2 T=3 (N stored as 0), base j at bits 2j of the record
 *   good  [R][nm] u64 : bit j = base j is ACGT and phred >= 20      (pass-1 gate, :240-259)
 *   hiq   [R][nm] u64 : bit j = base j is ACGT and phred >= 30      (prune's quality-sum bound)
 *   valid [R][nm] u64 : bit j = base j is ACGT                      (pass 2 has no quality gate, :272-274)
 *   qual  [R][L]  u8  : (unsigned char)(ch - '!')                   (phred33 :150-152)
 *   strand[R]     u8  : strand char - '0'                           (contributing_strand :336, :350)
 * with nb = ceil(L/32), nm = ceil(L/64); R is padded to a multiple of the tile size with zeros.
 */
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace vdjg {

typedef unsigned long long u64;
typedef unsigned int u32;
typedef unsigned short u16;
typedef unsigned char u8;

constexpr u64 EMPTY64 = ~0ull;
constexpr u64 INF64 = ~0ull;
constexpr u32 NIL32 = 0xFFFFFFFFu;
constexpr u32 CNT_CAP = 32765;   /* MAX_FREQUENCY-1, :66, :262, :345 */
constexpr int GATE_Q = 20;       /* MIN_BASE_QUALITY, :76 */
constexpr int HIQ = 30;          /* "high quality": windows whose phreds are all >= HIQ let prune bound the quality
                                    sums without reading quality rows (k_prune) */
constexpr int FLB = 6;           /* window flag bits: has-next, next base (2), then pass 1: window all >= HIQ, record start
                                    all >= HIQ; pass 2: has-previous, previous base (2) */
constexpr u32 CNT2_MASK = 0x00FFFFFFu; /* Slot2::count: N-free occurrences; bits 24..27: in-mask (base c preceded the k-mer
                                          in some read): the export probes only the predecessors that can exist */
constexpr int CNT2_IN = 24;
constexpr u32 CNT2_DISP = 1u << 28;    /* Slot2::count bit 28: some k-mer whose home is this slot was inserted further on
                                          (set by t2_insert).  Clear: a k-mer that is not here is not in the table */
constexpr u64 LOG_A = 1ull << 62, LOG_B = 1ull << 63;   /* those two flags in a log entry, above the stamp */
constexpr int QSUM_SAT = 214;    /* MAX_QUAL_SUM-41, :356 */
constexpr int MAX_LOG_RANKS = 11;/* ceil(214/20) */
constexpr u32 CNT_MULTI = 0x80000000u; /* bit 31 of Slot1::count = hasMultipleUniqueReads */
constexpr u32 CNT_SURV = 0x40000000u;  /* bit 30: survived prune_pre_graph (set by k_prune) */
constexpr u32 CNT_MASK = 0x3FFFFFFFu;
constexpr int THREADS = 256;
constexpr int WARPS = THREADS / 32;
constexpr u32 LOG_CHUNK = 64;    /* log blocks a warp reserves per global atomic */
constexpr u32 MAX_PROBE = 1u << 14;
constexpr int HIST_BITS = 8;     /* minimizer buckets: the finest hash partitioning (<= 256 partitions) */
constexpr int NBUCKET = 1 << HIST_BITS;
constexpr int BHLL_BITS = 7;     /* HyperLogLog registers (bytes) per bucket: sigma ~ 9 % per bucket, < 1 % over all */
constexpr int BHLL = 1 << BHLL_BITS;
constexpr int BATCH = 4;         /* independent table probes a thread keeps in flight */
#ifndef PASS1_MIN_BLOCKS
#define PASS1_MIN_BLOCKS 4
#endif
#ifndef PASS2_MIN_BLOCKS
#define PASS2_MIN_BLOCKS 3
#endif
constexpr int MINI_M = 10;       /* minimizer length in bases (m = min(k, MINI_M)) */
constexpr int RUN_MAX = 24;      /* windows per run: two 24-bit flag fields share one word of the run record */
constexpr int SEG_MAX = 32;      /* windows per thread segment of the streaming kernels (a run never crosses a segment) */
constexpr int STAMP_BITS = 40;   /* records < 2^32, windows per record <= 255 */

/* pass-1 table slot: exactly one 32-byte sector */
struct __align__(32) Slot1 {
    u64 klo, khi;     /* packed k-mer; all ones = empty */
    u32 count;        /* bits 0..29: gated occurrences AFTER the one that claimed the slot (the k-mer's count is
                         this + 1; stops counting a little above CNT_CAP); bit 30 CNT_SURV; bit 31 CNT_MULTI:
                         hasMultipleUniqueReads :349-352 */
    u32 head;         /* this k-mer's block of NB log entries (stamps of its first NB arrivals);
                         NIL32 until the thread that claimed the slot has published it */
    u32 first_rec;    /* record of the occurrence that claimed the slot: contributingRead :335.  Written (with
                         first_fp, one 64-bit store) by the claiming thread AFTER head: a slot is usable by
                         others once they see it */
    u32 first_fp;     /* fingerprint of that record's sequence (as carried by the runs) */
};
static_assert(sizeof(Slot1) == 32, "Slot1 must be one sector");

/* pass-2 table slot (survivors only): two sectors, the hot one first */
struct __align__(64) Slot2 {
    u64 klo, khi;
    u32 count;        /* N-free occurrences -> node->frequency */
    u32 rank;         /* creation rank (node id - 1), filled by k_assign_rank.  During pass 2: four bytes, byte c =
                         an upper bound of out_first[c] >> cshift (255 = nothing yet), lowered AFTER out_first[c]: a
                         window whose coarse stamp is above it cannot lower out_first[c] and skips that sector */
    u64 first_any;    /* min stamp over occurrences -> node->kmer, node id order */
    u64 out_first[4]; /* min stamp of an occurrence followed by base c -> toNodes order */
};
static_assert(sizeof(Slot2) == 64, "Slot2 must be two sectors");


struct Geom {
    int L, k, w, nb, nm;
    int seg;            /* windows per thread segment: ceil(w / segs) <= SEG_MAX */
    int segs;           /* thread segments per record: ceil(w / SEG_MAX) */
    u32 tile_rec;       /* records per block tile (even): THREADS / segs */
    u64 R;              /* real records */
    u64 n_tiles;
    u64 kmask_lo, kmask_hi; /* 2k ones */
    u64 kones;          /* k ones */
    int m, span;        /* minimizer length min(k, MINI_M); m-mers per window: k - m + 1 */
    u32 mmask;          /* 2m ones */
    int run_max;        /* windows per run: min(RUN_MAX, 64 - k), so that a run's bases fit 128 bits */
    u64 w_magic;        /* ceil(2^64 / w): stamp / w = umul64hi(stamp, w_magic) for stamps < 2^STAMP_BITS (w = 1: see make_geom) */
    u32 stage_runs;     /* runs a k_scatter block stages per tile (expected count + margin; the rest go out one by one) */
};

/* The tables of one device as seen by the kernels: hash unit u (= minimizer bucket >> ushift; a unit
 * is what is assigned to a device and a round) owns slots [off, off+len) of each table.  A k-mer's
 * home slot is inside its unit's slice; linear probing may run past the slice's end. */
struct __align__(16) UnitTab { u32 off1, len1, off2, len2; };

/* hash partitioning + the per-window tuple format of the slow-path queues */
struct Part {
    int ushift;         /* unit = bucket >> ushift; NBUCKET >> ushift units */
    int hb;             /* bits of the k-mer above 64: max(0, 2k-64) */
    int wide;           /* 1: 24-byte queue tuples (stamp in a third word) */
    int fb;             /* read-fingerprint bits carried by a tuple (<= RUN_FP_BITS; fewer only via the test hook) */
    u32 hot_t, hot_flush; /* pass 1: fast-path increments of k-mers whose count is already >= hot_t are summed in a
                             small per-warp shared-memory cache and added to the table every hot_flush batches */
    u32 qflush1, qdense1, qflush2, qdense2; /* slow-path queue policy of pass 1 / pass 2 (<= QFLUSH, see WarpQueue) */
    u32 flat;           /* 1: one slice [0, flat_len) for every k-mer (the merged table of a sharded / multi-round
                           finish): no minimizer is computed */
    u32 flat_len;
    u32 cshift;         /* coarse stamp = min(254, stamp >> cshift) */
    u64 n_runs;         /* runs in this device's buffer (this round) */
    const UnitTab *ut;  /* [NBUCKET >> ushift], device memory */
};

/* The packed reads of all devices of a sharded build (one entry when there is one device).
 * Record numbers are global: device d holds records [rec_base[d], rec_base[d+1]).  Peer arrays
 * are read through NVLink (peer-mapped memory); only the rare exact read comparison and the
 * quality rows of border k-mers ever touch them. */
constexpr int MAX_DEV = 8;
struct Reads {
    const u64 *bases[MAX_DEV], *valid[MAX_DEV];
    const u8 *qual[MAX_DEV], *strand[MAX_DEV];
    u64 rec_base[MAX_DEV + 1];
    int n_dev, any_strand;
    __device__ __forceinline__ int dev_of(u64 r) const {
        int d = 0;
        while (d + 1 < n_dev && r >= rec_base[d + 1]) d++;
        return d;
    }
};

struct Counters {
    u64 n_gated;
    u64 n_distinct;
    u64 n_surv_hot, n_surv_cold; /* survivors k_prune listed at the front / back of the survivor list */
    u64 n_hits;
    u64 n_nodes;
    u64 n_slow1, n_slow2; /* windows that took the slow path of pass 1 / pass 2 */
    u64 n_hits_ungated;   /* pass-2 hits of windows that did not pass the quality gate (the ones that add to the count) */
    u32 log_used;
    u32 overflow;     /* table full / probe bound hit / region overrun */
    u32 internal;     /* invariant violated */
    u32 pad;
};

/* ------------------------------------------------------------------------------------------ */
/* PTX helpers                                                                                  */
/* ------------------------------------------------------------------------------------------ */
__device__ __forceinline__ void ld_sector(const void *p, u64 &a, u64 &b, u64 &c, u64 &d) {
    /* one 256-bit load = one 32-B sector, cached in L2 only (table probes have no L1 reuse) */
    asm volatile("ld.global.cg.v4.b64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_sector(void *p, u64 a, u64 b, u64 c, u64 d) {
    asm volatile("st.global.v4.b64 [%0], {%1,%2,%3,%4};" :: "l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}
__device__ __forceinline__ void ld_cg_v2(const void *p, u64 &a, u64 &b) {
    asm volatile("ld.global.cg.v2.b64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ u64 ld_cg_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.global.cg.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
/* L1-cached variants for the fast paths of the table passes.  Ig reads are extremely skewed
 * (every read that touches the constant region repeats the same few hundred k-mers), so a dozen
 * slots per partition take half of all probes; L1 absorbs them.  L1 is not coherent across SMs:
 * the fast paths only test MONOTONIC facts on the loaded words (key present, MULTI set, count
 * past a threshold, a min-stamp already <= ours), so a stale line can only send a tuple to the
 * slow path or cost a redundant RED, never change a result. */
__device__ __forceinline__ void ld_sector_ca(const void *p, u64 &a, u64 &b, u64 &c, u64 &d) {
    asm volatile("ld.global.ca.v4.b64 {%0,%1,%2,%3}, [%4];"
                 : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ u64 ld_ca_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.global.ca.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
/* streaming (touched-once) tuple traffic: evict-first so it does not push the L2-resident
 * table slice out */
__device__ __forceinline__ void ld_stream_v2(const void *p, u64 &a, u64 &b) {
    asm volatile("ld.global.cs.v2.b64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ u64 ld_stream_u64(const void *p) {
    u64 v;
    asm volatile("ld.global.cs.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_stream_v2(void *p, u64 a, u64 b) {
    asm volatile("st.global.cs.v2.b64 [%0], {%1,%2};" :: "l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void st_stream_u64(void *p, u64 a) {
    asm volatile("st.global.cs.b64 [%0], %1;" :: "l"(p), "l"(a) : "memory");
}
__device__ __forceinline__ void st_cg_u64(u64 *p, u64 v) {
    asm volatile("st.global.cg.b64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}
/* 128-bit compare-and-swap on a 16-byte aligned key (ATOMG.E.CAS.128 on sm_100a) */
__device__ __forceinline__ void cas128(void *addr, u64 cmp_lo, u64 cmp_hi, u64 val_lo, u64 val_hi,
                                       u64 &old_lo, u64 &old_hi) {
    asm volatile("{\n\t.reg .b128 c, v, o;\n\t"
                 "mov.b128 c, {%2, %3};\n\t"
                 "mov.b128 v, {%4, %5};\n\t"
                 "atom.global.relaxed.gpu.cas.b128 o, [%6], c, v;\n\t"
                 "mov.b128 {%0, %1}, o;\n\t}"
                 : "=l"(old_lo), "=l"(old_hi)
                 : "l"(cmp_lo), "l"(cmp_hi), "l"(val_lo), "l"(val_hi), "l"(addr) : "memory");
}

__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "WAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE_%=;\n\t"
                 "bra WAIT_%=;\n\t"
                 "DONE_%=:\n\t}" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
/* TMA 1-D bulk copy global -> shared, completion counted on an mbarrier (UBLKCP in SASS) */
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src, u32 bytes, u64 *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
/* TMA 1-D bulk copy shared -> global (to this or a peer device), tracked by the bulk async-group */
__device__ __forceinline__ void tma_store_1d(void *dst_global, const void *src_smem, u32 bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(dst_global), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
/* the shared-memory source of every committed bulk store has been read */
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

/* ------------------------------------------------------------------------------------------ */
/* k-mer arithmetic                                                                             */
/* ------------------------------------------------------------------------------------------ */
__device__ __forceinline__ u64 hash_key(u64 lo, u64 hi) {
    u64 h = lo ^ (hi * 0x9E3779B97F4A7C15ull);
    h ^= h >> 32; h *= 0xD6E8FEB86659FD93ull;
    h ^= h >> 32; h *= 0xD6E8FEB86659FD93ull;
    h ^= h >> 32;
    return h;
}
/* 32-bit hash of a packed k-mer for the table slots (hash_key's three 64-bit multiplies are the
 * most expensive thing the fast paths of the table passes would do per window) */
__device__ __forceinline__ u32 hash_slot(u64 lo, u64 hi) {
    u32 x = (u32)lo * 0x9E3779B1u ^ (u32)(lo >> 32) * 0x85EBCA77u ^ (u32)hi * 0xC2B2AE3Du ^ (u32)(hi >> 32) * 0x27D4EB2Fu;
    x ^= x >> 15; x *= 0x2C1B3C6Du;
    x ^= x >> 12; x *= 0x297A2D39u;
    x ^= x >> 15;
    return x;
}
/* home slot of a k-mer with slot hash h in the table slice [off, off+len): len < 2^32 (the host
 * checks the table capacities), one 32-bit multiply-high */
__device__ __forceinline__ u32 slot_in(u32 h, u32 off, u32 len) { return off + __umulhi(h, len); }

/* Minimizers.  An m-mer (m <= 10 bases, 2 bits each) is hashed to 32 bits; the minimizer value of a
 * k-mer is the SMALLEST hash among its k-m+1 m-mers, a function of the k-mer alone, and the k-mer's
 * bucket (the finest partitioning) is a second hash of that value: the minimum of ~26 hashes is far
 * from uniform, its re-hash is. */
__device__ __forceinline__ u32 mini_hash(u32 x) {
    u32 h = x * 0x9E3779B1u;
    h ^= h >> 15;
    return h * 0x2C1B3C6Du;
}
__device__ __forceinline__ u32 mini_bucket(u32 minh) {
    u32 h = (minh ^ 0x5BD1E995u) * 0x85EBCA77u;
    h ^= h >> 13;
    h *= 0xC2B2AE3Du;
    return h >> (32 - HIST_BITS);
}

/* bits [2i, 2i+2k) of a record's base words */
__device__ __forceinline__ void extract_kmer(const u64 *b, int nb, int i, u64 mlo, u64 mhi, u64 &lo, u64 &hi) {
    int bit = 2 * i, wi = bit >> 6, sh = bit & 63;
    u64 w0 = b[wi];
    u64 w1 = wi + 1 < nb ? b[wi + 1] : 0ull;
    u64 w2 = wi + 2 < nb ? b[wi + 2] : 0ull;
    if (sh) { lo = (w0 >> sh) | (w1 << (64 - sh)); hi = (w1 >> sh) | (w2 << (64 - sh)); }
    else { lo = w0; hi = w1; }
    lo &= mlo; hi &= mhi;
}
/* k mask bits starting at bit i (k <= 50 < 64) */
__device__ __forceinline__ u64 extract_mask(const u64 *m, int nm, int i) {
    int wi = i >> 6, sh = i & 63;
    u64 m0 = m[wi];
    u64 m1 = wi + 1 < nm ? m[wi + 1] : 0ull;
    return sh ? (m0 >> sh) | (m1 << (64 - sh)) : m0;
}
__device__ __forceinline__ u32 base_at(const u64 *b, int j) { return (u32)(b[j >> 5] >> ((j & 31) * 2)) & 3u; }
__device__ __forceinline__ bool bit_at(const u64 *m, int j) { return (m[j >> 6] >> (j & 63)) & 1ull; }

/* successor K[1:]+c and predecessor c+K[:-1] of a packed k-mer */
__device__ __forceinline__ void kmer_succ(u64 lo, u64 hi, u32 c, int k, u64 &slo, u64 &shi) {
    slo = (lo >> 2) | (hi << 62);
    shi = hi >> 2;
    int bit = 2 * (k - 1);
    if (bit < 64) slo |= (u64)c << bit; else shi |= (u64)c << (bit - 64);
}
__device__ __forceinline__ void kmer_pred(u64 lo, u64 hi, u32 c, u64 mlo, u64 mhi, u64 &plo, u64 &phi) {
    phi = ((hi << 2) | (lo >> 62)) & mhi;
    plo = ((lo << 2) | (u64)c) & mlo;
}
__device__ __forceinline__ u32 kmer_last(u64 lo, u64 hi, int k) {
    int bit = 2 * (k - 1);
    return (u32)(bit < 64 ? lo >> bit : hi >> (bit - 64)) & 3u;
}

/* bucket of an arbitrary packed k-mer (table builds and edge lookups; the streaming kernels slide the
 * minimum along the read instead, see Mini) */
__device__ __forceinline__ u32 kmer_bucket_of(u64 lo, u64 hi, int span, u32 mmask) {
    u32 minh = ~0u;
    for (int j = 0; j < span; j++) {
        minh = min(minh, mini_hash((u32)lo & mmask));
        lo = (lo >> 2) | (hi << 62);
        hi >>= 2;
    }
    return mini_bucket(minh);
}

/* ------------------------------------------------------------------------------------------ */
/* Per-window tuples.  The table passes expand the runs into one tuple per window, in registers; */
/* windows that need the slow path are parked in shared-memory queues in this form:             */
/* word0 = k-mer bits 0..63; word1 = k-mer bits 64.. (hb bits) | flags << hb (FLB bits) |       */
/* fp << (hb+FLB) | stamp << (hb+FLB+fb) (narrow, 16 B); when fewer than 4 fingerprint bits      */
/* would fit the stamp moves to a third word (wide, 24 B).  fp = fingerprint of the record's    */
/* whole sequence: two records with different fingerprints hold different reads, which settles  */
/* hasMultipleUniqueReads without touching the reads again (equal fingerprints fall back to the */
/* exact comparison).                                                                            */
/* ------------------------------------------------------------------------------------------ */
template <bool WIDE>
__device__ __forceinline__ void tuple_decode(const Part &pt, u64 w1, u64 w2, u64 &hi, u32 &fl, u32 &fp, u64 &stamp) {
    hi = pt.hb ? (w1 & ((1ull << pt.hb) - 1)) : 0ull;
    fl = (u32)(w1 >> pt.hb) & ((1u << FLB) - 1);
    fp = (u32)(w1 >> (pt.hb + FLB)) & (u32)((1ull << pt.fb) - 1);
    stamp = WIDE ? w2 : (w1 >> (pt.hb + FLB + pt.fb));
}
/* all operands must be computed before anything after this point is issued: keeps independent
 * loads of a batch back to back instead of interleaved with the address arithmetic of the next */
__device__ __forceinline__ void issue_fence(u32 &a, u32 &b, u32 &c, u32 &d) {
    asm volatile("" : "+r"(a), "+r"(b), "+r"(c), "+r"(d));
}

/* ------------------------------------------------------------------------------------------ */
/* K-1 k_pack: the reference's text records (bam_read.c:206-244: strand char, L bases, L         */
/* phred+33 qualities) -> the packed layout described at the top of this file.  One warp per     */
/* record; lane j looks at bases j, j+32, ...: the masks are warp ballots, the 2-bit codes two   */
/* ballots interleaved.  Also validates what the reference only trips over later: the strand     */
/* byte (exit(-1) at :383-391) and the alphabet (seq_to_int exit(-1), seq_to_kmer.c:23-25).      */
/* ------------------------------------------------------------------------------------------ */
struct PackArgs {
    const unsigned char *text;   /* n text records; packed record numbers start at r0 */
    u64 r0, n;
    u32 fwd_only;                /* the text holds forward reads only (vdjgraph_stage_forward): every text record
                                    yields two packed records, the read and its reverse complement */
    u64 *bases, *good, *valid, *hiq;
    u8 *qual, *strand;
    u64 *bad;                    /* [0] first record with a bad strand byte, [1] with a bad base (atomicMin), [2] any strand '1' */
};
/* bits of a (bit i -> bit 2i) */
__device__ __forceinline__ u64 spread_bits(u32 a) {
    u64 x = a;
    x = (x | (x << 16)) & 0x0000FFFF0000FFFFull;
    x = (x | (x << 8)) & 0x00FF00FF00FF00FFull;
    x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0Full;
    x = (x | (x << 2)) & 0x3333333333333333ull;
    x = (x | (x << 1)) & 0x5555555555555555ull;
    return x;
}
/* one record by one warp.  rev: emit the record's reverse complement instead (bases complemented
 * and reversed, qualities reversed, same strand byte: what add_to_buffer writes as the second record
 * of every read, bam_read.c:230-243 with rc :130-137 / reverse :139-145) */
__device__ __forceinline__ void pack_record(const PackArgs &a, const Geom &g, const unsigned char *rec, u64 r, bool rev, u32 lane) {
    if (lane == 0) {
        const unsigned sc = rec[0];
        if (sc != '0' && sc != '1') atomicMin(&a.bad[0], r);
        if (sc == '1') a.bad[2] = 1;
        a.strand[r] = (u8)(sc - '0');
    }
    u64 vword = 0, gword = 0, hword = 0;
    for (int j0 = 0; j0 < g.L; j0 += 32) {
        const int j = j0 + (int)lane;
        unsigned code = 4;   /* beyond the read: neither valid nor an error */
        bool okq = false, hiq = false;
        if (j < g.L) {
            const int sj = rev ? g.L - 1 - j : j;
            const unsigned ch = rec[1 + sj];
            code = ch == 'A' ? 0u : ch == 'C' ? 1u : ch == 'G' ? 2u : ch == 'T' ? 3u : ch == 'N' ? 4u : 5u;
            if (rev && code < 4) code = 3u - code;   /* complement :116-128; N stays N */
            const u8 q = (u8)(rec[1 + g.L + sj] - '!');
            a.qual[r * (u64)g.L + j] = q;
            okq = q >= GATE_Q;
            hiq = q >= HIQ;
        }
        const u32 b0 = __ballot_sync(0xFFFFFFFFu, code < 4 && (code & 1u));
        const u32 b1 = __ballot_sync(0xFFFFFFFFu, code < 4 && (code & 2u));
        const u32 bv = __ballot_sync(0xFFFFFFFFu, code < 4);
        const u32 bg = __ballot_sync(0xFFFFFFFFu, code < 4 && okq);
        const u32 bh = __ballot_sync(0xFFFFFFFFu, code < 4 && hiq);
        const u32 be = __ballot_sync(0xFFFFFFFFu, code == 5);
        if (lane == 0) {
            if (be) atomicMin(&a.bad[1], r);
            a.bases[r * (u64)g.nb + (j0 >> 5)] = spread_bits(b0) | (spread_bits(b1) << 1);
            if (j0 & 32) {
                a.valid[r * (u64)g.nm + (j0 >> 6)] = vword | ((u64)bv << 32);
                a.good[r * (u64)g.nm + (j0 >> 6)] = gword | ((u64)bg << 32);
                a.hiq[r * (u64)g.nm + (j0 >> 6)] = hword | ((u64)bh << 32);
            } else {
                vword = bv; gword = bg; hword = bh;
                if (j0 + 32 >= g.L) {   /* last, half-filled mask word */
                    a.valid[r * (u64)g.nm + (j0 >> 6)] = vword;
                    a.good[r * (u64)g.nm + (j0 >> 6)] = gword;
                    a.hiq[r * (u64)g.nm + (j0 >> 6)] = hword;
                }
            }
        }
    }
}
__global__ void __launch_bounds__(THREADS)
k_pack(PackArgs a, Geom g) {
    const u32 lane = threadIdx.x & 31;
    const u64 warp = ((u64)blockIdx.x * THREADS + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * THREADS) >> 5;
    const u64 rec_len = 2ull * g.L + 1;
    for (u64 i = warp; i < a.n; i += n_warps) {
        const unsigned char *rec = a.text + i * rec_len;
        if (!a.fwd_only) {
            pack_record(a, g, rec, a.r0 + i, false, lane);
        } else {   /* text record i is a forward read: packed records r0+2i (the read) and r0+2i+1 (derived here) */
            pack_record(a, g, rec, a.r0 + 2 * i, false, lane);
            pack_record(a, g, rec, a.r0 + 2 * i + 1, true, lane);
        }
    }
}

/* ------------------------------------------------------------------------------------------ */
/* Streaming the packed reads (k_count, k_scatter).  A block walks tiles of g.tile_rec records   */
/* block-stride; the arrays of a tile are brought into shared memory by TMA bulk copies (double  */
/* buffered, one elected thread issues, everybody waits on the mbarrier).  Thread t owns one     */
/* SEGMENT of a record: up to SEG_MAX consecutive windows, whose k-mer, gate/N masks and          */
/* minimizer it ROLLS (one new base and one new mask bit per window) instead of re-extracting.   */
/* ------------------------------------------------------------------------------------------ */
struct BlockTiles {
    u64 *buf;   /* [2][a | b | c | d] */
    u64 *bar;   /* [2] */
    u32 words, off_b, off_c, off_d;
    __device__ __forceinline__ const u64 *a(int i) const { return buf + i * words; }
    __device__ __forceinline__ const u64 *b(int i) const { return buf + i * words + off_b; }
    __device__ __forceinline__ const u64 *c(int i) const { return buf + i * words + off_c; }
    __device__ __forceinline__ const u64 *d(int i) const { return buf + i * words + off_d; }
};
/* n_masks = 2 (good, valid) or 3 (+ hiq) */
__host__ __device__ inline size_t block_tile_bytes(const Geom &g, int n_masks) {
    return (size_t)2 * g.tile_rec * (size_t)(g.nb + n_masks * g.nm) * 8 + 16;
}
__device__ __forceinline__ BlockTiles tiles_setup(unsigned char *smem, const Geom &g, int n_masks) {
    BlockTiles t;
    t.words = g.tile_rec * (u32)(g.nb + n_masks * g.nm);
    t.off_b = g.tile_rec * (u32)g.nb;
    t.off_c = t.off_b + g.tile_rec * (u32)g.nm;
    t.off_d = t.off_c + g.tile_rec * (u32)g.nm;
    t.buf = reinterpret_cast<u64 *>(smem);
    t.bar = t.buf + 2 * t.words;
    if (threadIdx.x == 0) {
        mbar_init(&t.bar[0], 1);
        mbar_init(&t.bar[1], 1);
        fence_mbar_init();
        fence_proxy_async();
    }
    __syncthreads();
    return t;
}
/* one thread: start the bulk copies of `tile` into buffer i */
__device__ __forceinline__ void tiles_issue(const BlockTiles &t, int i, const Geom &g, u64 tile,
                                            const u64 *ga, const u64 *gb, const u64 *gc, const u64 *gd = nullptr) {
    const u32 bytes_a = g.tile_rec * (u32)g.nb * 8u, bytes_m = g.tile_rec * (u32)g.nm * 8u;
    u64 *dst = t.buf + i * t.words;
    mbar_expect_tx(&t.bar[i], bytes_a + (gd ? 3 : 2) * bytes_m);
    tma_load_1d(dst, ga + tile * g.tile_rec * (u64)g.nb, bytes_a, &t.bar[i]);
    tma_load_1d(dst + t.off_b, gb + tile * g.tile_rec * (u64)g.nm, bytes_m, &t.bar[i]);
    tma_load_1d(dst + t.off_c, gc + tile * g.tile_rec * (u64)g.nm, bytes_m, &t.bar[i]);
    if (gd) tma_load_1d(dst + t.off_d, gd + tile * g.tile_rec * (u64)g.nm, bytes_m, &t.bar[i]);
}

/* 128 bits of a bit array (nw words) starting at bit `bit0`; bits beyond the array read as zero */
__device__ __forceinline__ void extract_bits128(const u64 *m, int nw, int bit0, u64 &lo, u64 &hi) {
    const int wi = bit0 >> 6, sh = bit0 & 63;
    const u64 w0 = wi < nw ? m[wi] : 0ull;
    const u64 w1 = wi + 1 < nw ? m[wi + 1] : 0ull;
    const u64 w2 = wi + 2 < nw ? m[wi + 2] : 0ull;
    if (sh) { lo = (w0 >> sh) | (w1 << (64 - sh)); hi = (w1 >> sh) | (w2 << (64 - sh)); }
    else { lo = w0; hi = w1; }
}
__device__ __forceinline__ void shr128(u64 &lo, u64 &hi, int s) {   /* 0 <= s < 128 */
    if (s >= 64) { lo = hi >> (s - 64); hi = 0ull; }
    else if (s) { lo = (lo >> s) | (hi << (64 - s)); hi >>= s; }
}
/* Erosion by k: bit i of the result = bits i .. i+k-1 of (lo,hi) are all ones, i.e. "the window that
 * starts at i passes" for a per-base mask.  Built from erosions by powers of two (E_{a+b}[i] =
 * E_a[i] & E_b[i+a]): ~2 log2 k shift-and steps for ALL windows of a segment at once, instead of one
 * rolling mask per window.  Only the low word of the result is used (<= SEG_MAX + 1 windows). */
__device__ __forceinline__ u64 erode128(u64 lo, u64 hi, int k) {
    u64 pl = lo, ph = hi, al = ~0ull, ah = ~0ull;
    int alen = 0;
    for (int plen = 1; plen <= k; plen <<= 1) {
        if (k & plen) {
            u64 tl = pl, th = ph;
            shr128(tl, th, alen);
            al &= tl; ah &= th;
            alen += plen;
        }
        u64 tl = pl, th = ph;
        shr128(tl, th, plen);
        pl &= tl; ph &= th;
    }
    return al;
}
/* the same when windows + k - 1 <= 64 bits are looked at (shifts below 64 only: k <= 50) */
__device__ __forceinline__ u64 erode64(u64 m, int k) {
    u64 p = m, a = ~0ull;
    int alen = 0;
    for (int plen = 1; plen <= k; plen <<= 1) {
        if (k & plen) { a &= p >> alen; alen += plen; }
        p &= p >> plen;
    }
    return a;
}
/* bit j of the result: the window that starts at bit i0+j of the per-base mask m (nw words) passes */
__device__ __forceinline__ u64 window_mask(const u64 *m, int nw, int i0, const Geom &g) {
    u64 lo, hi;
    extract_bits128(m, nw, i0, lo, hi);
    return g.seg + g.k <= 64 ? erode64(lo, g.k) : erode128(lo, hi, g.k);
}

/* Sliding minimum of the m-mer hashes along a segment (the minimizer value of every window),
 * branch-uniform: the m-mer positions are cut into blocks of `span`; a window that starts at offset
 * r of block t covers the suffix [r, span) of block t and the prefix [0, r) of block t+1, so its
 * minimum is min(suffix-min of t at r, running prefix-min of t+1).  The thread's scratch (span words
 * of shared memory, stride THREADS) holds block t's suffix minima; slot r-1 is dead once window r is
 * reached and takes block t+1's hash as it arrives; when block t+1 is complete one backward sweep
 * turns it into suffix minima.  Every thread of a warp is at the same r, so nothing diverges. */
struct Mini {
    u32 *buf;
    u32 x, pre;
    int r;
    __device__ __forceinline__ void sweep(int span) {
        u32 run = ~0u;
        for (int j = span - 1; j >= 0; j--) { run = min(run, buf[j * THREADS]); buf[j * THREADS] = run; }
    }
    /* first window of the segment: its k-mer holds all m-mers of block 0 */
    __device__ __forceinline__ u32 start(u64 lo, u64 hi, const Geom &g) {
        for (int j = 0; j < g.span; j++) {
            x = (u32)lo & g.mmask;
            buf[j * THREADS] = mini_hash(x);
            lo = (lo >> 2) | (hi << 62);
            hi >>= 2;
        }
        sweep(g.span);
        r = 0; pre = ~0u;
        return buf[0];
    }
    /* next window: base c enters */
    __device__ __forceinline__ u32 step(u32 c, const Geom &g) {
        x = (x >> 2) | (c << (2 * (g.m - 1)));
        const u32 h = mini_hash(x);
        buf[r * THREADS] = h;          /* offset r of the next block; this slot's suffix minimum is no longer needed */
        r++;
        if (r == g.span) { sweep(g.span); r = 0; pre = ~0u; return buf[0]; }
        pre = min(pre, h);
        return min(buf[r * THREADS], pre);
    }
};

/* Walks one thread segment (windows i0 .. i0+n-1 of record `rec`) and finds its RUNS: maximal
 * stretches of consecutive N-free windows whose k-mers fall into the same minimizer bucket, cut
 * at run_max windows and at the segment's end.
 * Which windows are N-free / gated / all >= HIQ comes from one erosion of the per-base masks per
 * segment; the window loop rolls only the m-mer and its sliding minimum and notes where a run
 * starts (bit j of `starts`) and with which bucket (sbk[ordinal * THREADS], a byte array in shared
 * memory).  It runs g.seg times in every thread, so the warp stays converged for Mini's sweeps.
 * KMERS: also roll the k-mer itself and call on_gated(k-mer, bucket) for every window that passes
 * the quality gate (k_count's cardinality registers; the scatter needs m-mers only). */
struct SegRuns {
    u64 V, G, H;     /* bit j: window i0+j is N-free / passes the quality gate / has all phreds >= HIQ; V also has bit n */
    u32 starts;      /* bit j: a run starts at window i0+j */
    u32 left;        /* starts not yet taken by next() */
    u32 ord;         /* ordinal of the next run */
    /* the next run: first window (relative to i0), length; false when there is none */
    __device__ __forceinline__ bool next(int n, int &s, int &len) {
        if (!left) return false;
        s = __ffs((int)left) - 1;
        left &= left - 1;
        /* it ends before the next start, the next window that is not N-free, or the segment's end */
        const u64 stop = ((((u64)starts | ~V) >> s) >> 1) | (1ull << (n - s - 1));
        len = __ffsll((long long)stop);
        ord++;
        return true;
    }
    /* does the window after run (s, len) exist, and is it N-free? */
    __device__ __forceinline__ u32 has_next(int s, int len) const { return (u32)(V >> (s + len)) & 1u; }
};
template <bool KMERS, class OnGated>
__device__ __forceinline__ SegRuns scan_runs(const u64 *sb, const u64 *sg, const u64 *sv, const u64 *sh, u32 rec, int i0, int n,
                                             const Geom &g, u32 *scratch, u8 *sbk, OnGated on_gated) {
    Mini mn;
    mn.buf = scratch;
    SegRuns sr;
    sr.V = sr.G = sr.H = 0; sr.starts = 0; sr.ord = 0;
    u64 lo = 0, hi = 0, nbase = 0;
    if (n > 0) {
        sr.V = window_mask(sv + (size_t)rec * g.nm, g.nm, i0, g);
        sr.G = window_mask(sg + (size_t)rec * g.nm, g.nm, i0, g);
        if (sh) sr.H = window_mask(sh + (size_t)rec * g.nm, g.nm, i0, g);
        const u64 *b = sb + (size_t)rec * g.nb;
        extract_kmer(b, g.nb, i0, g.kmask_lo, g.kmask_hi, lo, hi);
        /* the bases that enter the window: positions i0+k .. i0+k+31 */
        const int j = i0 + g.k;
        u64 nl = 0, nh;
        if (j < 32 * g.nb) extract_kmer(b, g.nb, j, ~0ull, 0ull, nl, nh);
        nbase = nl;
    }
    u32 run_len = 0, run_b = 0, minh = 0, n_starts = 0;
    for (int j = 0; j < g.seg; j++) {
        if (j < n) {
            if (j == 0) minh = mn.start(lo, hi, g);
            else {
                const u32 c = (u32)nbase & 3u;
                nbase >>= 2;
                minh = mn.step(c, g);
                if (KMERS) kmer_succ(lo, hi, c, g.k, lo, hi);
            }
            const bool v = (sr.V >> j) & 1ull;
            const u32 b = mini_bucket(minh);
            const bool fresh = v && (run_len == 0 || b != run_b || run_len == (u32)g.run_max);
            if (fresh) {
                sbk[n_starts * THREADS] = (u8)b;
                n_starts++;
                sr.starts |= 1u << j;
                run_b = b;
                run_len = 0;
            }
            run_len = v ? run_len + 1 : 0;
            if (KMERS && ((sr.G >> j) & 1ull)) on_gated(lo, hi, b);
        }
    }
    sr.left = sr.starts;
    return sr;
}

/* ------------------------------------------------------------------------------------------ */
/* K0 k_count: one streaming pass over the packed reads that sizes everything else, per        */
/* minimizer bucket:                                                                             */
/*   - runs, gated windows and N-free windows (exact: the scatter's region sizes),              */
/*   - a small HyperLogLog of the gated k-mers -> table-1 slice sizes, so that the table is     */
/*     neither rehashed (the reference's dense_hash_map doubles, internal/densehashtable.h      */
/*     :631-653) nor grossly over-allocated.                                                     */
/* hist [3][NBUCKET] u64 (runs | gated | N-free), hll [NBUCKET][BHLL] bytes (4 per u32 word).    */
/* Runs once per staged read set (its results do not depend on mf / mq).                         */
/* ------------------------------------------------------------------------------------------ */
__host__ __device__ inline size_t align128(size_t x) { return (x + 127) & ~(size_t)127; }
__host__ __device__ inline size_t count_head_bytes() {
    return ((size_t)NBUCKET * BHLL / 4 + (size_t)3 * NBUCKET) * sizeof(u32);
}
__host__ __device__ inline size_t scratch_bytes(const Geom &g) { return (size_t)g.span * THREADS * sizeof(u32); }
__host__ __device__ inline size_t sbk_bytes(const Geom &g) { return align128((size_t)g.seg * THREADS); }
/* max of the byte at position idx of a packed byte array */
__device__ __forceinline__ void byte_max(u32 *words, u32 idx, u32 v, bool global) {
    u32 *wp = words + (idx >> 2);
    const u32 sh = (idx & 3u) * 8u;
    u32 cur = *reinterpret_cast<volatile u32 *>(wp);
    while (((cur >> sh) & 0xFFu) < v) {
        const u32 nv = (cur & ~(0xFFu << sh)) | (v << sh);
        const u32 old = atomicCAS(wp, cur, nv);
        if (old == cur) break;
        cur = old;
    }
}
__global__ void __launch_bounds__(THREADS)
k_count(const u64 *__restrict__ bases, const u64 *__restrict__ good, const u64 *__restrict__ valid,
        Geom g, u64 tile0, u64 tile1 /* tiles [tile0, tile1): one staging chunk, or everything */, u32 *hll, u64 *hist /* [3][NBUCKET] */) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int HW = NBUCKET * BHLL / 4;
    u32 *reg = reinterpret_cast<u32 *>(smem);
    u32 *sh = reg + HW;  /* [3][NBUCKET] */
    for (int i = threadIdx.x; i < HW + 3 * NBUCKET; i += THREADS) reg[i] = 0;
    u32 *scratch = reinterpret_cast<u32 *>(smem + count_head_bytes()) + threadIdx.x;
    u8 *sbk = smem + count_head_bytes() + scratch_bytes(g) + threadIdx.x;   /* [g.seg][THREADS] run buckets */
    BlockTiles t = tiles_setup(smem + count_head_bytes() + scratch_bytes(g) + sbk_bytes(g), g, 2);
    const u32 rec = threadIdx.x / (u32)g.segs, i0 = (threadIdx.x % (u32)g.segs) * (u32)g.seg;
    const int n = rec < g.tile_rec ? max(0, min(g.seg, g.w - (int)i0)) : 0;
    const u64 n_iter = (tile1 - tile0 + gridDim.x - 1) / gridDim.x;
    if (threadIdx.x == 0 && tile0 + blockIdx.x < tile1) tiles_issue(t, 0, g, tile0 + blockIdx.x, bases, good, valid);
    u64 tile = tile0 + blockIdx.x;
    for (u64 it = 0; it < n_iter; it++, tile += gridDim.x) {
        const int buf = (int)(it & 1);
        if (tile < tile1) {
            if (threadIdx.x == 0 && tile + gridDim.x < tile1) tiles_issue(t, buf ^ 1, g, tile + gridDim.x, bases, good, valid);
            mbar_wait(&t.bar[buf], (u32)(it >> 1) & 1);
            SegRuns sr = scan_runs<true>(t.a(buf), t.b(buf), t.c(buf), nullptr, rec, (int)i0, n, g, scratch, sbk,
                [&](u64 lo, u64 hi, u32 b) {
                    const u64 h = hash_key(lo, hi);
                    /* register = low hash bits, rank = leading zeros of the rest (1..58) */
                    byte_max(reg, b * BHLL + ((u32)h & (BHLL - 1)), (u32)__clzll((long long)(h >> BHLL_BITS)) - (BHLL_BITS - 1), false);
                });
            int rs, len;
            while (sr.next(n, rs, len)) {
                const u32 b = sbk[(sr.ord - 1) * THREADS], gm = (u32)(sr.G >> rs) & ((1u << len) - 1u);
                atomicAdd(&sh[b], 1u);
                if (gm) atomicAdd(&sh[NBUCKET + b], (u32)__popc(gm));
                atomicAdd(&sh[2 * NBUCKET + b], (u32)len);
            }
        }
        __syncthreads();   /* everybody is done with buffer `buf` before it is refilled */
        /* u32 counters: flush long before they can overflow (uniform trip count) */
        if ((it & 0xFFFF) == 0xFFFF) {
            for (int i = threadIdx.x; i < 3 * NBUCKET; i += THREADS) { u32 v = sh[i]; if (v) { atomicAdd(&hist[i], (u64)v); sh[i] = 0; } }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < HW; i += THREADS) {
        const u32 v = reg[i];
        for (int b = 0; v && b < 4; b++) if ((v >> (8 * b)) & 0xFFu) byte_max(hll, 4u * i + b, (v >> (8 * b)) & 0xFFu, true);
    }
    for (int i = threadIdx.x; i < 3 * NBUCKET; i += THREADS)
        if (sh[i]) atomicAdd(&hist[i], (u64)sh[i]);
}

/* ------------------------------------------------------------------------------------------ */
/* Run records: 32 bytes = one sector.                                                           */
/*   w0, w1 : the bases first window .. last window + k - 1 (+ the base after them when the      */
/*            window after the run exists), 2 bits each from bit 0: at most 64 bases            */
/*   w2     : gate bit of window j at bit j (24) | window-all->=HIQ bit at 24+j (24) |           */
/*            length-1 at 48 (5) | next-window-exists at 53 | record-start-all->=HIQ at 54 |     */
/*            previous-window-exists at 55 | the base before the run at 56 (2) |                 */
/*            fingerprint bits 16..21 at 58 (6)                                                  */
/*   w3     : stamp of the first window (STAMP_BITS) | bucket at 40 (8) | fingerprint bits 0..15 at 48 */
/* ------------------------------------------------------------------------------------------ */
constexpr int RUN_WORDS = 4;
constexpr int RUN_FP_BITS = 22;
__device__ __forceinline__ u32 run_len(u64 w2) { return ((u32)(w2 >> 48) & 31u) + 1u; }
__device__ __forceinline__ u32 run_bucket(u64 w3) { return (u32)(w3 >> STAMP_BITS) & (NBUCKET - 1); }
__device__ __forceinline__ void ld_run(const u64 *p, u64 &a, u64 &b, u64 &c, u64 &d) {
    /* streaming (touched once per pass): evict-first so that it does not push the L2-resident table slice out */
    asm volatile("ld.global.cs.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
}

/* ------------------------------------------------------------------------------------------ */
/* K1 k_scatter: every run goes to the region of its hash unit in the run buffer of the         */
/* device that owns the unit (cursor[] starts at this device's share of each region, from the   */
/* all-gathered k_count histograms).  Per tile a block                                           */
/*   1. rolls its windows once: run descriptors go to a list in shared memory, units are counted,*/
/*   2. scans the counters into stage offsets and reserves one range per non-empty unit with a  */
/*      single global atomic,                                                                    */
/*   3. builds the run records from the list (balanced over the threads) into a stage ordered   */
/*      by unit,                                                                                 */
/*   4. copies the stage out: one TMA bulk store per non-empty unit, straight to the unit's     */
/*      region on this device or, through peer-mapped memory, on the owner's: the scatter IS    */
/*      the all-to-all of a sharded build.                                                       */
/* Runs beyond the list's capacity (a tile with pathologically short runs) are written one by   */
/* one.  Units of other rounds have no destination and are skipped.                              */
/* ------------------------------------------------------------------------------------------ */
struct ScatterArgs {
    const u64 *bases, *good, *valid, *hiq;
    u64 *const *tbase; /* [units] run buffer of the device that owns the unit (peer-mapped when that is another
                          device); null: not in this round */
    u64 *cursor;       /* [units] next free run of this device's share of the unit's region */
    const u64 *limit;  /* [units] end of that share (overrun check) */
    u64 rec_base;      /* global number of this device's first record */
    Counters *ctr;
};
struct ScatterSmem {
    u32 *cnt;    /* [NBUCKET] runs of the tile per unit */
    u32 *fill;   /* [NBUCKET] fill cursor of phase 3 */
    u32 *boff;   /* [NBUCKET + 1] start of each unit's range in the stage */
    u64 *gbase;  /* [NBUCKET] global run index of the range */
    u64 **dst;   /* [NBUCKET] copy of tbase */
    u32 *fp;     /* [tile_rec] read fingerprint | record-start-all->=HIQ << 31 */
    u32 *n_list; /* runs in the list */
    u8 *sbk;     /* [g.seg][THREADS] buckets of a thread's runs, in order */
    u64 *list;   /* [g.stage_runs][2] run descriptors */
    u64 *stage;  /* [g.stage_runs][4]; the same memory serves as Mini's scratch while the windows are rolled */
    unsigned char *tiles;
};
__host__ __device__ inline size_t scatter_carve(ScatterSmem *o, unsigned char *base, const Geom &g) {
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t at = off; off = align128(off + bytes); return at; };
    const size_t a_cnt = take((size_t)NBUCKET * 4), a_fill = take((size_t)NBUCKET * 4), a_boff = take((size_t)(NBUCKET + 1) * 4), a_gbase = take((size_t)NBUCKET * 8);
    const size_t a_dst = take((size_t)NBUCKET * 8), a_fp = take((size_t)g.tile_rec * 4), a_n = take(16);
    const size_t a_list = take((size_t)g.stage_runs * 16), a_sbk = take(sbk_bytes(g));
    const size_t stage_b = (size_t)g.stage_runs * RUN_WORDS * 8, scr_b = scratch_bytes(g);
    const size_t a_stage = take(stage_b > scr_b ? stage_b : scr_b), a_tiles = take(block_tile_bytes(g, 3));
    if (o) {
        o->cnt = reinterpret_cast<u32 *>(base + a_cnt); o->fill = reinterpret_cast<u32 *>(base + a_fill); o->boff = reinterpret_cast<u32 *>(base + a_boff);
        o->gbase = reinterpret_cast<u64 *>(base + a_gbase); o->dst = reinterpret_cast<u64 **>(base + a_dst);
        o->fp = reinterpret_cast<u32 *>(base + a_fp); o->n_list = reinterpret_cast<u32 *>(base + a_n);
        o->sbk = base + a_sbk;
        o->list = reinterpret_cast<u64 *>(base + a_list); o->stage = reinterpret_cast<u64 *>(base + a_stage);
        o->tiles = base + a_tiles;
    }
    return off;
}
/* run descriptor (phase 1 -> phase 3): d0 = gate bits | HIQ bits << 24 | (len-1) << 48 | next << 53;
 * d1 = record in tile | first window << 16 | bucket << 24 */
__device__ __forceinline__ void build_run(u64 d0, u64 d1, const u64 *sb, const u64 *sv, const u32 *sfp, const Geom &g, u64 rec0,
                                          u64 &w0, u64 &w1, u64 &w2, u64 &w3) {
    const u32 rec = (u32)d1 & 0xFFFFu, a = (u32)(d1 >> 16) & 0xFFu, b = (u32)(d1 >> 24) & 0xFFu;
    extract_kmer(sb + (size_t)rec * g.nb, g.nb, (int)a, ~0ull, ~0ull, w0, w1);
    const u32 f = sfp[rec], fp = f & ((1u << RUN_FP_BITS) - 1);
    /* the window before the run's first one exists and is N-free iff the base before it is ACGT */
    u64 prev = 0;
    if (a > 0 && bit_at(sv + (size_t)rec * g.nm, (int)a - 1)) prev = 1ull | ((u64)base_at(sb + (size_t)rec * g.nb, (int)a - 1) << 1);
    w2 = d0 | ((u64)(f >> 31) << 54) | (prev << 55) | ((u64)(fp >> 16) << 58);
    w3 = ((rec0 + rec) * (u64)g.w + a) | ((u64)b << STAMP_BITS) | ((u64)(fp & 0xFFFFu) << 48);
}

__global__ void __launch_bounds__(THREADS)
k_scatter(ScatterArgs a, Geom g, Part pt) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int NU = NBUCKET >> pt.ushift;
    ScatterSmem sm;
    scatter_carve(&sm, smem, g);
    BlockTiles t = tiles_setup(sm.tiles, g, 3);
    const u32 lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    u32 *scratch = reinterpret_cast<u32 *>(sm.stage) + threadIdx.x;
    const u32 rec = threadIdx.x / (u32)g.segs, i0 = (threadIdx.x % (u32)g.segs) * (u32)g.seg;
    const int n = rec < g.tile_rec ? max(0, min(g.seg, g.w - (int)i0)) : 0;
    const u64 n_iter = (g.n_tiles + gridDim.x - 1) / gridDim.x;
    for (int u = threadIdx.x; u < NU; u += THREADS) sm.dst[u] = a.tbase[u];
    if (threadIdx.x == 0 && blockIdx.x < g.n_tiles) tiles_issue(t, 0, g, blockIdx.x, a.bases, a.good, a.valid, a.hiq);
    u64 tile = blockIdx.x;
    for (u64 it = 0; it < n_iter; it++, tile += gridDim.x) {
        const int buf = (int)(it & 1);
        if (tile >= g.n_tiles) break;   /* block-uniform */
        for (int i = threadIdx.x; i < NU; i += THREADS) { sm.cnt[i] = 0; sm.fill[i] = 0; }
        if (threadIdx.x == 0) {
            *sm.n_list = 0;
            if (tile + gridDim.x < g.n_tiles) tiles_issue(t, buf ^ 1, g, tile + gridDim.x, a.bases, a.good, a.valid, a.hiq);
        }
        mbar_wait(&t.bar[buf], (u32)(it >> 1) & 1);
        __syncthreads();
        const u64 *sb = t.a(buf), *sg = t.b(buf), *sv = t.c(buf), *sh = t.d(buf);
        const u64 rec0 = a.rec_base + tile * g.tile_rec;
        /* read fingerprints of the tile's records; are the record's first k phreds all >= HIQ?  (the first
         * occurrence of a k-mer contributes the RECORD's first k qualities to the sums, :337-339) */
        for (u32 r = threadIdx.x; r < g.tile_rec; r += THREADS) {
            u64 h = 0x9E3779B97F4A7C15ull;
            for (int i = 0; i < g.nb; i++) h = hash_key(sb[(size_t)r * g.nb + i], h);
            for (int i = 0; i < g.nm; i++) h = hash_key(sv[(size_t)r * g.nm + i], h);
            const u32 rec_hi = (extract_mask(sh + (size_t)r * g.nm, g.nm, 0) & g.kones) == g.kones ? 1u : 0u;
            sm.fp[r] = ((u32)(h >> 32) & ((1u << RUN_FP_BITS) - 1)) | (rec_hi << 31);
        }
        __syncthreads();   /* fingerprints are read by the overflow path of phase 1 */
        /* 1. roll the windows, then (warp-converged) run descriptors -> list, per-unit counts */
        {
            SegRuns sr = scan_runs<false>(sb, sg, sv, sh, rec, (int)i0, n, g, scratch, sm.sbk + threadIdx.x, [](u64, u64, u32) {});
            for (;;) {
                int rs = 0, len = 1;
                const bool has = sr.next(n, rs, len);
                if (!__ballot_sync(0xFFFFFFFFu, has)) break;
                const u32 b = has ? sm.sbk[(sr.ord - 1) * THREADS + threadIdx.x] : 0u, u = b >> pt.ushift;
                const bool ship = has && sm.dst[u];   /* no destination: another round's share of the hash space */
                const u32 ball = __ballot_sync(0xFFFFFFFFu, ship);
                if (!ball) continue;
                u32 e0 = 0;
                if (lane == 0) e0 = atomicAdd(sm.n_list, (u32)__popc(ball));
                e0 = __shfl_sync(0xFFFFFFFFu, e0, 0);
                if (ship) {
                    const u32 lm = (1u << len) - 1u;
                    const u64 d0 = (u64)((u32)(sr.G >> rs) & lm) | ((u64)((u32)(sr.H >> rs) & lm) << 24) | ((u64)(len - 1) << 48) |
                                   ((u64)sr.has_next(rs, len) << 53);
                    const u64 d1 = (u64)rec | ((u64)(i0 + rs) << 16) | ((u64)b << 24);
                    const u32 e = e0 + (u32)__popc(ball & ((1u << lane) - 1u));
                    if (e < g.stage_runs) {
                        sm.list[2 * e] = d0; sm.list[2 * e + 1] = d1;
                        atomicAdd(&sm.cnt[u], 1u);
                    } else {   /* list full: this run goes out on its own */
                        u64 w0, w1, w2, w3;
                        build_run(d0, d1, sb, sv, sm.fp, g, rec0, w0, w1, w2, w3);
                        const u64 at = atomicAdd(&a.cursor[u], 1ull);
                        if (at < a.limit[u]) st_sector(sm.dst[u] + at * RUN_WORDS, w0, w1, w2, w3);
                        else atomicExch(&a.ctr->overflow, 4u);
                    }
                }
            }
        }
        __syncthreads();
        /* 2. reserve the global ranges; stage offsets = exclusive scan of the counts */
        for (int u = threadIdx.x; u < NU; u += THREADS) {
            const u32 c = sm.cnt[u];
            u64 gbs = INF64;
            if (c) {
                gbs = atomicAdd(&a.cursor[u], (u64)c);
                if (gbs + c > a.limit[u]) { atomicExch(&a.ctr->overflow, 4u); gbs = INF64; }
            }
            sm.gbase[u] = gbs;
        }
        if (wid == 0) {   /* one warp: lane owns NU/32 consecutive units */
            const int per = (NU + 31) / 32;
            u32 sum = 0;
            for (int j = 0; j < per; j++) { int u = lane * per + j; if (u < NU) sum += sm.cnt[u]; }
            u32 incl = sum;
            for (int o = 1; o < 32; o <<= 1) { u32 v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((int)lane >= o) incl += v; }
            u32 run = incl - sum;
            for (int j = 0; j < per; j++) {
                int u = lane * per + j;
                if (u < NU) { sm.boff[u] = run; run += sm.cnt[u]; }
            }
            if (lane == 31) sm.boff[NU] = run;
        }
        __syncthreads();
        /* 3. build the runs into the stage, unit by unit */
        const u32 n_list = min(*sm.n_list, g.stage_runs);
        for (u32 e = threadIdx.x; e < n_list; e += THREADS) {
            const u64 d0 = sm.list[2 * e], d1 = sm.list[2 * e + 1];
            const u32 u = ((u32)(d1 >> 24) & 0xFFu) >> pt.ushift;
            u64 w0, w1, w2, w3;
            build_run(d0, d1, sb, sv, sm.fp, g, rec0, w0, w1, w2, w3);
            u64 *dst = sm.stage + (size_t)(sm.boff[u] + atomicAdd(&sm.fill[u], 1u)) * RUN_WORDS;
            dst[0] = w0; dst[1] = w1; dst[2] = w2; dst[3] = w3;
        }
        fence_proxy_async();     /* the stage was written with ordinary stores */
        __syncthreads();
        /* 4. copy out: a range is contiguous on both sides */
        for (int u = threadIdx.x; u < NU; u += THREADS) {
            const u32 c = sm.boff[u + 1] - sm.boff[u];
            const u64 gbs = sm.gbase[u];
            if (c && gbs != INF64) tma_store_1d(sm.dst[u] + gbs * RUN_WORDS, sm.stage + (size_t)sm.boff[u] * RUN_WORDS, c * (u32)(RUN_WORDS * 8));
        }
        tma_store_commit();
        tma_store_wait_read();   /* the stage becomes Mini's scratch again */
        __syncthreads();
    }
}

/* ------------------------------------------------------------------------------------------ */
/* table initialisation                                                                         */
/* ------------------------------------------------------------------------------------------ */
__global__ void k_init_table1(Slot1 *t, u64 cap) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    for (; i < cap; i += stride)
        st_sector(&t[i], EMPTY64, EMPTY64, (u64)0 | ((u64)NIL32 << 32), (u64)NIL32);
}
__global__ void k_init_table2(Slot2 *t, u64 cap) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    for (; i < cap; i += stride) {
        st_sector(&t[i], EMPTY64, EMPTY64, (u64)0 | ((u64)NIL32 << 32), INF64);
        st_sector(reinterpret_cast<char *>(&t[i]) + 32, INF64, INF64, INF64, INF64);
    }
}

/* do records r1 and r2 hold the same L-character sequence and strand?
 * compare_read :142-144 (strncmp over read_length) and the strand test :350.
 * The words of both records are fetched together (one round trip, possibly to a peer device). */
__device__ __noinline__ bool same_words(const u64 *b1, const u64 *b2, int nb, const u64 *v1, const u64 *v2, int nm) {
    u64 diff = 0;
    for (int i = 0; i < nb; i++) diff |= b1[i] ^ b2[i];
    for (int i = 0; i < nm; i++) diff |= v1[i] ^ v2[i];
    return diff == 0;
}
__device__ __forceinline__ bool same_read(const Reads &rd, u64 r1, u64 r2, int nb, int nm) {
    const int d1 = rd.dev_of(r1), d2 = rd.dev_of(r2);
    const u64 l1 = r1 - rd.rec_base[d1], l2 = r2 - rd.rec_base[d2];
    if (rd.any_strand && rd.strand[d1][l1] != rd.strand[d2][l2]) return false;
    return same_words(rd.bases[d1] + l1 * nb, rd.bases[d2] + l2 * nb, nb, rd.valid[d1] + l1 * nm, rd.valid[d2] + l2 * nm, nm);
}

/* ------------------------------------------------------------------------------------------ */
/* K2 k_pass1: pass 1 = build_pre_graph / add_to_table (:322-409) as commutative reductions    */
/* over the GATED windows of the runs, walked unit by unit so that the table slice being updated is */
/* L2-resident:                                                                                  */
/*   count        -> pre_node.frequency (:334, :345-347)                                        */
/*   CNT_MULTI    -> hasMultipleUniqueReads (:349-352): some occurrence's record differs from   */
/*                   the first ARRIVING one's; equivalent to ">= 2 distinct record sequences"   */
/*   occurrence log: the first NB arrivals of every k-mer append their stamp, so that k-mers    */
/*                   whose final count is <= NB have ALL their occurrences listed; only those   */
/*                   can fail the quality-sum test (every gated quality is >= 20), see k_prune. */
/* ------------------------------------------------------------------------------------------ */
struct Pass1Args {
    const u64 *runs;  /* [pt.n_runs][RUN_WORDS], grouped by hash unit */
    Reads rd;
    Slot1 *table;
    u64 cap;
    u64 *log;         /* [log_blocks][NB] stamps */
    u32 log_blocks;
    u32 nb_ranks;     /* NB: arrivals with rank < NB are logged */
    Counters *ctr;
};

/* Per-warp queue of deferred tuples in shared memory.  Both table passes split their work in
 * two: a branch-free FAST path for tuples whose home slot resolves them with plain loads and at
 * most a fire-and-forget RED, and a SLOW path (insertion, probing past the home slot, arrival
 * ranks, read comparison, logging) for the rest.  Slow tuples are queued and drained by a lane
 * state machine in which every lane always holds a tuple: a lane that finishes takes the next
 * queue entry, so probe chains of different length do not idle the warp. */
constexpr u32 QFLUSH = 96;                       /* drain when at least this many are queued */
constexpr u32 QCAP = 32 * BATCH + QFLUSH;        /* a batch can add 32*BATCH entries */
constexpr u32 QDENSE = 20;                       /* a non-final drain stops when fewer lanes than this are busy
                                                    and puts their tuples (with the probe position reached)
                                                    back in the queue: long probe chains do not idle the warp */
/* QC = capacity: a batch can add 32*BATCH entries on top of the flush threshold.  Pass 1 drains
 * almost every batch and keeps its queue small: shared memory it does not take stays L1, which is
 * what absorbs the probes of the hot k-mers. */
constexpr int HOTC_BITS = 6;
constexpr u32 HOTC = 1u << HOTC_BITS;            /* entries of a warp's hot-k-mer increment cache */
constexpr u32 QFLUSH1 = 32;
constexpr u32 QCAP1 = 32 * BATCH + QFLUSH1;
template <bool WIDE, u32 QC = QCAP>
struct WarpQueue {
    u64 *lo, *w1, *w2;
    u32 *idx;
    __device__ __forceinline__ void setup(unsigned char *smem) {
        unsigned char *p = smem + (threadIdx.x >> 5) * bytes();
        lo = reinterpret_cast<u64 *>(p);
        w1 = lo + QC;
        w2 = w1 + QC;
        idx = reinterpret_cast<u32 *>(w1 + (WIDE ? 2 : 1) * QC);
    }
    __host__ __device__ static constexpr size_t bytes() { return (size_t)QC * (WIDE ? 28 : 20); }
    /* the same, the tuple words being built (by the deferred lanes only) by make(t1, t2) */
    template <class Make>
    __device__ __forceinline__ u32 push_lazy(u32 qn, bool defer, u64 l, u32 i, Make make) {
        const u32 lane = threadIdx.x & 31;
        const u32 ballot = __ballot_sync(0xFFFFFFFFu, defer);
        if (defer) {
            const u32 pos = qn + __popc(ballot & ((1u << lane) - 1));
            u64 a, b;
            make(a, b);
            lo[pos] = l; w1[pos] = a; idx[pos] = i;
            if (WIDE) w2[pos] = b;
        }
        return qn + __popc(ballot);
    }
    /* warp-converged push of the lanes with `defer` set; returns the new count */
    __device__ __forceinline__ u32 push(u32 qn, bool defer, u64 l, u64 a, u64 b, u32 i) {
        const u32 lane = threadIdx.x & 31;
        const u32 ballot = __ballot_sync(0xFFFFFFFFu, defer);
        if (defer) {
            const u32 pos = qn + __popc(ballot & ((1u << lane) - 1));
            lo[pos] = l; w1[pos] = a; idx[pos] = i;
            if (WIDE) w2[pos] = b;
        }
        return qn + __popc(ballot);
    }
};

/* Expansion of runs into per-window tuples.  A warp takes 32 runs at a time (one per lane, parked
 * in shared memory), counts the windows this pass looks at (pass 1: the gated ones, pass 2: all) and
 * deals them out evenly: every lane takes BATCH CONSECUTIVE windows of the chunk's window sequence.
 * The first one is located by a search over the runs' prefix counts (five shuffles); from there a
 * cursor walks the selected windows of the run and steps into the next run when it is used up, so
 * that everything that is per run (stamp, fingerprint, table slice) is decoded once per run, not
 * per window.  Every lane holds BATCH independent windows whatever the run lengths are. */
struct RunCursor {
    u64 w0, w1, w2;     /* the run's bases and flag word */
    u64 stamp0;         /* stamp of its window 0 */
    u32 off, len;       /* table slice of its hash unit */
    u32 l;              /* run index in the chunk */
    u32 j;              /* current window */
    u32 rem;            /* selected windows above j, shifted down by j+1 */
};
struct RunFeed {
    u64 *rw;        /* [32][RUN_WORDS] this warp's chunk */
    u32 cnt, incl, total;
    u32 live;       /* bit l: run l of the chunk has windows this pass looks at */
    template <bool GATED_ONLY>
    __device__ __forceinline__ static u32 selected(u64 w2) {
        return GATED_ONLY ? (u32)w2 & 0xFFFFFFu : (1u << run_len(w2)) - 1u;   /* run_len <= 24 */
    }
    template <bool GATED_ONLY>
    __device__ __forceinline__ void load(const u64 *runs, u64 ri, u64 n_runs) {
        const u32 lane = threadIdx.x & 31;
        u64 w0 = 0, w1 = 0, w2 = 0, w3 = 0;
        cnt = 0;
        if (ri < n_runs) {
            ld_run(runs + ri * RUN_WORDS, w0, w1, w2, w3);
            cnt = (u32)__popc(selected<GATED_ONLY>(w2));
        }
        incl = cnt;
        for (int o = 1; o < 32; o <<= 1) { const u32 v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if ((int)lane >= o) incl += v; }
        total = __shfl_sync(0xFFFFFFFFu, incl, 31);
        live = __ballot_sync(0xFFFFFFFFu, cnt != 0);
        __syncwarp();
        u64 *p = rw + lane * RUN_WORDS;
        p[0] = w0; p[1] = w1; p[2] = ri < n_runs ? w2 : 0ull; p[3] = w3;
        __syncwarp();
    }
    /* decode run c.l; TAB2: the slice of table 2, else of table 1 */
    template <bool TAB2>
    __device__ __forceinline__ void open(RunCursor &c, const Part &pt) const {
        const u64 *p = rw + c.l * RUN_WORDS;
        c.w0 = p[0]; c.w1 = p[1]; c.w2 = p[2];
        const u64 w3 = p[3];
        c.stamp0 = w3 & ((1ull << STAMP_BITS) - 1);
        const uint4 ut = __ldg(reinterpret_cast<const uint4 *>(pt.ut + (run_bucket(w3) >> pt.ushift)));   /* off1, len1, off2, len2 */
        c.off = TAB2 ? ut.z : ut.x;
        c.len = TAB2 ? ut.w : ut.y;
    }
    /* position the cursor on window t (< total) of the chunk.  Warp-converged (shuffles). */
    template <bool GATED_ONLY, bool TAB2>
    __device__ __forceinline__ void seek(u32 t, RunCursor &c, const Part &pt) const {
        u32 l = 0;
#pragma unroll
        for (int s = 16; s; s >>= 1) { const u32 v = __shfl_sync(0xFFFFFFFFu, incl, l + s - 1); if (v <= t) l += s; }
        u32 nth = t - __shfl_sync(0xFFFFFFFFu, incl - cnt, l);
        c.l = l;
        open<TAB2>(c, pt);
        u32 m = selected<GATED_ONLY>(c.w2), j = 0;
        if (GATED_ONLY) {   /* position of the nth set bit */
#pragma unroll
            for (int s = 16; s; s >>= 1) {
                const u32 k = (u32)__popc(m & ((1u << s) - 1u));
                if (nth >= k) { nth -= k; m >>= s; j += s; }
            }
            m >>= 1;
        } else {
            j = nth;
            m >>= j + 1;
        }
        c.j = j; c.rem = m;
    }
    /* the fingerprint carried by run l (fb bits) */
    __device__ __forceinline__ u32 fingerprint(u32 l, const Part &pt) const {
        const u64 *p = rw + l * RUN_WORDS;
        return (((u32)(p[3] >> 48) & 0xFFFFu) | (((u32)(p[2] >> 58) & 0x3Fu) << 16)) & (u32)((1ull << pt.fb) - 1);
    }
    /* the next selected window of the chunk (the caller knows there is one) */
    template <bool GATED_ONLY, bool TAB2>
    __device__ __forceinline__ void next(RunCursor &c, const Part &pt) const {
        if (c.rem) {
            const u32 s = (u32)__ffs((int)c.rem);
            c.j += s; c.rem >>= s;
            return;
        }
        /* the next run that has any (the caller knows there is one) */
        const u32 ahead = c.l < 31 ? live >> (c.l + 1) : 0u;
        c.l += ahead ? (u32)__ffs((int)ahead) : 0u;
        open<TAB2>(c, pt);
        const u32 m = selected<GATED_ONLY>(c.w2);
        const u32 s = m ? (u32)__ffs((int)m) : 1u;
        c.j = s - 1; c.rem = m >> s;
    }
};
/* the cursor's window -> its k-mer and home slot: all the fast path of pass 1 needs */
__device__ __forceinline__ void run_kmer(const Geom &g, const RunCursor &c, u64 &lo, u64 &hi, u32 &idx) {
    const u32 sh = 2u * c.j;   /* <= 46 */
    lo = sh ? (c.w0 >> sh) | (c.w1 << (64 - sh)) : c.w0;
    hi = c.w1 >> sh;
    lo &= g.kmask_lo; hi &= g.kmask_hi;
    idx = slot_in(hash_slot(lo, hi), c.off, c.len);
}
/* flag bits of window j of a run (FLB bits: has-next, next base, window all >= HIQ, record start all >= HIQ) */
__device__ __forceinline__ u32 run_flags(const Geom &g, u64 w0, u64 w1, u64 w2, u32 j) {
    const u32 p = j + (u32)g.k;   /* the base after the window: position <= 63 of the run's bases */
    const u32 nb = (u32)((p < 32 ? w0 >> (2 * p) : w1 >> (2 * (p - 32)))) & 3u;
    const bool has_next = j + 1 < run_len(w2) || ((w2 >> 53) & 1ull);
    return (has_next ? 1u | (nb << 1) : 0u) | ((u32)(w2 >> (24 + j)) & 1u) << 3 | ((u32)(w2 >> 54) & 1u) << 4;
}
/* the same for pass 2: has-next, next base, has-previous, previous base */
__device__ __forceinline__ u32 run_flags2(const Geom &g, u64 w0, u64 w1, u64 w2, u32 j) {
    const u32 p = j + (u32)g.k;
    const u32 nb = (u32)((p < 32 ? w0 >> (2 * p) : w1 >> (2 * (p - 32)))) & 3u;
    const bool has_next = j + 1 < run_len(w2) || ((w2 >> 53) & 1ull);
    /* window j > 0 follows window j-1 of the same run; window 0 follows the base noted in the run, if any */
    const u32 prev = j ? 1u | (((u32)(w0 >> (2 * (j - 1))) & 3u) << 1) : (u32)(w2 >> 55) & 7u;
    return (has_next ? 1u | (nb << 1) : 0u) | prev << 3;
}
/* tuple words (the form the slow-path queues hold) of a window with these flags, fingerprint and stamp */
template <bool WIDE>
__device__ __forceinline__ void pack_tuple(const Part &pt, u64 hi, u32 fl, u32 fp, u64 stamp, u64 &t1, u64 &t2) {
    t1 = hi | ((u64)fl << pt.hb) | ((u64)fp << (pt.hb + FLB));
    if (WIDE) t2 = stamp;
    else { t1 |= stamp << (pt.hb + FLB + pt.fb); t2 = 0; }
}

struct LogCursor { u32 base, used; };   /* warp-uniform: the warp's current chunk of log blocks */

/* slow path of pass 1 for `qn` queued tuples.  One loop iteration = at most two dependent
 * round trips to L2 per lane: (1) the probe (sector load, plus the 128-bit CAS when the slot is
 * empty), (2) the arrival-rank atomicAdd and the first-record CAS, issued together. */
template <bool WIDE>
__device__ __forceinline__ u32 pass1_drain(const Pass1Args &a, const Geom &g, const Part &pt, WarpQueue<WIDE, QCAP1> &q,
                                           u32 qn, LogCursor &lc, bool final) {
    const u32 lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    u32 next = 0;
    bool have = false;
    u64 lo = 0, hi = 0, stamp = 0, rw1 = 0, rw2 = 0;
    u32 idx = 0, probe = 0, fp = 0, fl = 0;
    __syncwarp();
    for (;;) {
        /* refill idle lanes */
        const u32 need = __ballot_sync(0xFFFFFFFFu, !have);
        const u32 avail = qn - next;
        if (avail == 0 && (need == 0xFFFFFFFFu || (!final && 32 - __popc(need) < (int)pt.qdense1))) break;
        if (need && avail) {
            const u32 my = __popc(need & lt);
            if (!have && my < avail) {
                const u32 e = next + my;
                lo = q.lo[e]; rw1 = q.w1[e]; rw2 = WIDE ? q.w2[e] : 0ull;
                tuple_decode<WIDE>(pt, rw1, rw2, hi, fl, fp, stamp);
                idx = q.idx[e];
                probe = 0;
                have = true;
            }
            next += min((u32)__popc(need), avail);
        }
        /* probe step: find or claim the slot of (lo,hi) */
        bool found = false, claimed = false;
        u64 q2 = 0, q3 = 0;
        Slot1 *slot = a.table + idx;
        if (have) {
            u64 q0, q1;
            ld_sector(slot, q0, q1, q2, q3);
            if (q0 == EMPTY64 && q1 == EMPTY64) {
                cas128(slot, EMPTY64, EMPTY64, lo, hi, q0, q1);
                if (q0 == EMPTY64 && q1 == EMPTY64) { found = claimed = true; q2 = (u64)NIL32 << 32; q3 = (u64)NIL32; }
                else if (q0 == lo && q1 == hi) q2 = (u64)NIL32 << 32;   /* lost the race to the same k-mer: look again */
            } else if (q0 == lo && q1 == hi) {
                /* a slot whose claimer has not published its first record (and log block) yet is looked
                 * at again next iteration */
                found = (u32)q3 != NIL32 && (a.nb_ranks == 0 || (u32)(q2 >> 32) != NIL32);
            }
            if (!found && !(q0 == lo && q1 == hi)) {
                if (++idx == (u32)a.cap) idx = 0;
                if (++probe >= MAX_PROBE) { atomicExch(&a.ctr->overflow, 1u); have = false; }
            }
        }
        /* the claiming lane reserves the k-mer's log block (warp-aggregated) and publishes it */
        u32 blk = (u32)(q2 >> 32);
        if (a.nb_ranks) {
            const u32 ballot = __ballot_sync(0xFFFFFFFFu, claimed);
            if (ballot) {
                /* blocks come from the warp's current chunk of LOG_CHUNK; when it runs out the remaining
                 * claims of this step continue in a new chunk (nothing of a chunk is ever left unused) */
                const u32 n = __popc(ballot), room = LOG_CHUNK - lc.used, my = __popc(ballot & lt);
                u32 fresh = 0;
                if (n > room) {
                    if (lane == 0) fresh = atomicAdd(&a.ctr->log_used, LOG_CHUNK);
                    fresh = __shfl_sync(0xFFFFFFFFu, fresh, 0);
                }
                if (claimed) {
                    blk = my < room ? lc.base + lc.used + my : fresh + (my - room);
                    if (blk < a.log_blocks) slot->head = blk;
                    else { atomicExch(&a.ctr->overflow, 2u); blk = NIL32; slot->head = 0; }
                }
                if (n > room) { lc.base = fresh; lc.used = n - room; }
                else lc.used += n;
            }
        }
        /* update the slot (:334-352) */
        if (found) {
            const u32 r = g.w_magic ? (u32)__umul64hi(stamp, g.w_magic) : (u32)stamp;   /* stamp / w, exact for stamps below 2^40 */
            const u64 entry = stamp | ((fl & 8u) ? LOG_A : 0ull) | ((fl & 16u) ? LOG_B : 0ull);
            if (claimed) {
                /* first arrival: arrival rank 0, nothing to compare with, and nobody else touches the slot
                 * until the first-record word is published: plain stores, no atomics */
                if (a.nb_ranks && blk != NIL32) a.log[(u64)blk * a.nb_ranks] = entry;
                st_cg_u64(reinterpret_cast<u64 *>(&slot->first_rec), (u64)r | ((u64)fp << 32));
            } else {
                const u32 cw = (u32)q2, cnt = cw & CNT_MASK;       /* arrivals after the claimer seen so far */
                const u32 first_rec = (u32)q3, first_fp = (u32)(q3 >> 32);
                u32 rank = NIL32;
                if (cnt + 1 < a.nb_ranks) rank = (atomicAdd(&slot->count, 1u) & CNT_MASK) + 1;   /* arrival rank decides logging */
                else if (cnt + 1 < CNT_CAP) atomicAdd(&slot->count, 1u);                          /* result unused: RED */
                /* different fingerprints: different reads.  Equal ones: compare the reads (:142-144) */
                if (!(cw & CNT_MULTI) && first_rec != r &&
                    (first_fp != fp || !same_read(a.rd, first_rec, r, g.nb, g.nm)))
                    atomicOr(&slot->count, CNT_MULTI);
                if (rank < a.nb_ranks && blk != NIL32) a.log[(u64)blk * a.nb_ranks + rank] = entry;
            }
            have = false;
        }
    }
    /* unfinished tuples go back to the (now empty) queue with the slot they have reached */
    __syncwarp();
    const u32 left = q.push(0, have, lo, rw1, rw2, idx);
    __syncwarp();
    return left;
}

/* adds a warp's cached increments of hot k-mers to the table.  The count shares its word with the
 * SURV / MULTI flags (bits 30, 31): a k-mer that is already far past the cap (the cached adds are
 * not bounded by the fast path's stale view of the count) gets nothing more, so the count can never
 * carry into the flags however often a k-mer occurs. */
__device__ __forceinline__ void hot_flush(Slot1 *table, u32 *hidx, u32 *hcnt) {
    for (u32 i = threadIdx.x & 31; i < HOTC; i += 32) {
        const u32 c = hcnt[i];
        if (c) {
            u32 *cp = &table[hidx[i]].count;
            if ((*reinterpret_cast<volatile u32 *>(cp) & CNT_MASK) < (1u << 24)) atomicAdd(cp, c);
        }
        hidx[i] = NIL32; hcnt[i] = 0;
    }
}

template <bool WIDE>
__global__ void __launch_bounds__(THREADS, PASS1_MIN_BLOCKS)
k_pass1(Pass1Args a, Geom g, Part pt) {
    extern __shared__ __align__(128) unsigned char smem[];
    WarpQueue<WIDE, QCAP1> q;
    q.setup(smem);
    /* per-warp cache of pending increments for hot k-mers: [HOTC] slot index, [HOTC] count */
    u32 *hidx = reinterpret_cast<u32 *>(smem + WARPS * WarpQueue<WIDE, QCAP1>::bytes()) + (threadIdx.x >> 5) * 2 * HOTC;
    u32 *hcnt = hidx + HOTC;
    for (u32 i = threadIdx.x & 31; i < HOTC; i += 32) { hidx[i] = NIL32; hcnt[i] = 0; }
    RunFeed feed;
    feed.rw = reinterpret_cast<u64 *>(smem + WARPS * (WarpQueue<WIDE, QCAP1>::bytes() + 2 * HOTC * sizeof(u32))) + (threadIdx.x >> 5) * 32 * RUN_WORDS;
    __syncwarp();
    const u32 lane = threadIdx.x & 31;
    u32 since_flush = 0;
    LogCursor lc; lc.base = 0; lc.used = LOG_CHUNK;
    u32 qn = 0, n_slow = 0;   /* warp-uniform */
    const u64 n_chunk = (pt.n_runs + THREADS - 1) / THREADS;
    static_assert(BATCH == 4, "issue_fence takes four operands");
    for (u64 chunk = blockIdx.x; chunk < n_chunk; chunk += gridDim.x) {
        feed.load<true>(a.runs, chunk * THREADS + threadIdx.x, pt.n_runs);
        for (u32 base = 0; base < feed.total; base += 32 * BATCH) {
            u64 lo[BATCH], k0[BATCH], k1[BATCH], m2[BATCH], hi[BATCH];
            u32 idx[BATCH];   /* table capacities stay below 2^32 slots (checked on the host) */
            u32 ref[BATCH];   /* run in the chunk | window in the run << 8 */
            /* A1: this lane's BATCH consecutive windows of the chunk -> k-mer, home slot */
            {
                const u32 t0 = base + lane * BATCH;
                RunCursor cur;
                feed.seek<true, false>(min(t0, feed.total - 1), cur, pt);
#pragma unroll
                for (int u = 0; u < BATCH; u++) {
                    lo[u] = hi[u] = 0; idx[u] = NIL32; ref[u] = 0;
                    if (t0 + u < feed.total) {
                        if (u) feed.next<true, false>(cur, pt);
                        run_kmer(g, cur, lo[u], hi[u], idx[u]);
                        ref[u] = cur.l | (cur.j << 8);
                    }
                }
            }
            issue_fence(idx[0], idx[1], idx[2], idx[3]);
            /* A2: the home slots, all loads in flight together */
#pragma unroll
            for (int u = 0; u < BATCH; u++) {
                k0[u] = k1[u] = m2[u] = 0;
                if (idx[u] != NIL32) {
                    u64 unused;
                    ld_sector_ca(a.table + idx[u], k0[u], k1[u], m2[u], unused);
                }
            }
            /* B: fast path = the k-mer sits in its home slot, is already known to come from several
             * reads and has passed the logging ranks: one RED.  Everything else is queued, with its
             * flags, fingerprint and stamp (only now read from the run). */
#pragma unroll
            for (int u = 0; u < BATCH; u++) {
                const bool valid = idx[u] != NIL32;
                const u32 cw = (u32)m2[u], cnt = cw & CNT_MASK;
                const bool fast = valid && k0[u] == lo[u] && k1[u] == hi[u] && (cw & CNT_MULTI) && cnt + 1 >= a.nb_ranks;
                if (fast && cnt + 1 < CNT_CAP) {
                    bool cached = false;
                    if (cnt >= pt.hot_t) {
                        const u32 e = (idx[u] * 0x9E3779B1u) >> (32 - HOTC_BITS);
                        const u32 old = atomicCAS(&hidx[e], NIL32, idx[u]);
                        if (old == NIL32 || old == idx[u]) { atomicAdd(&hcnt[e], 1u); cached = true; }
                    }
                    if (!cached) atomicAdd(&a.table[idx[u]].count, 1u);
                }
                qn = q.push_lazy(qn, valid && !fast, lo[u], idx[u], [&](u64 &t1, u64 &t2) {
                    const u32 l = ref[u] & 0xFFu, j = ref[u] >> 8;
                    const u64 *p = feed.rw + l * RUN_WORDS;
                    pack_tuple<WIDE>(pt, hi[u], run_flags(g, p[0], p[1], p[2], j), feed.fingerprint(l, pt),
                                     (p[3] & ((1ull << STAMP_BITS) - 1)) + j, t1, t2);
                });
            }
            if (++since_flush >= pt.hot_flush) {
                since_flush = 0;
                __syncwarp();
                hot_flush(a.table, hidx, hcnt);
                __syncwarp();
            }
            if (qn >= pt.qflush1) {
                n_slow += qn; qn = pass1_drain<WIDE>(a, g, pt, q, qn, lc, false); n_slow -= qn;
            }
        }
    }
    __syncwarp();
    hot_flush(a.table, hidx, hcnt);
    n_slow += qn;
    pass1_drain<WIDE>(a, g, pt, q, qn, lc, true);
    if (lane == 0 && n_slow) atomicAdd(&a.ctr->n_slow1, (u64)n_slow);
}

/* Position of this thread's element in a global append-only array: warps sum their counts in
 * shared memory and ONE global atomic per block reserves the block's range (a per-warp atomic on
 * the single counter serialises: 400 k same-address atomics cost more than the scan itself).
 * Must be called by all threads of the block; `take` = this thread appends one element to the array
 * of `counter`, `take_b` (exclusive with take) one to the array of `counter_b`: two arrays cost one
 * round of barriers, and their two atomics are in flight together. */
__device__ __forceinline__ u64 block_append(bool take, u64 *counter, bool take_b = false, u64 *counter_b = nullptr) {
    __shared__ u32 s_cnt[2];
    __shared__ u64 s_base[2];
    const u32 lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const u32 ballot = __ballot_sync(0xFFFFFFFFu, take), ballot_b = __ballot_sync(0xFFFFFFFFu, take_b);
    u32 wbase = 0, wbase_b = 0;
    if (lane == 0 && ballot) wbase = atomicAdd(&s_cnt[0], (u32)__popc(ballot));
    if (lane == 0 && ballot_b) wbase_b = atomicAdd(&s_cnt[1], (u32)__popc(ballot_b));
    wbase = __shfl_sync(0xFFFFFFFFu, wbase, 0);
    wbase_b = __shfl_sync(0xFFFFFFFFu, wbase_b, 0);
    __syncthreads();
    if (threadIdx.x == 0) s_base[0] = s_cnt[0] ? atomicAdd(counter, (u64)s_cnt[0]) : 0ull;
    if (threadIdx.x == 32) s_base[1] = s_cnt[1] ? atomicAdd(counter_b, (u64)s_cnt[1]) : 0ull;
    __syncthreads();
    return take_b ? s_base[1] + wbase_b + __popc(ballot_b & lt) : s_base[0] + wbase + __popc(ballot & lt);
}

/* ------------------------------------------------------------------------------------------ */
/* K3 k_prune = prune_pre_graph (:467-484) + is_base_quality_good (:454-465).                   */
/* keep K iff frequency >= mf && hasMultipleUniqueReads && for all j qual_sums[j] >= mq.        */
/* qual_sums[j] = S_j < 214 ? S_j : 255 with S_j = q_r0[j] + sum over the other gated           */
/* occurrences of q_r[i+j] ((r0,i0) = first gated occurrence; seeding from the RECORD's first   */
/* k qualities is the reference's behaviour, :337-339).  With mq <= 254 the test is             */
/* S_j >= T, T = min(mq, 214).  Every gated quality is >= 20, so S_j >= 20*(count-1): k-mers    */
/* with 20*(count-1) >= T pass without looking at qualities; the others have count <= NB and    */
/* their complete occurrence list is in the log.                                                */
/* The survivors' slots go to a list that table 2 is built from: k-mers with a gated count >= hot */
/* from the front, the others from the back, so that the hot ones can be inserted first.          */
/* ------------------------------------------------------------------------------------------ */
struct PruneArgs {
    Slot1 *table;
    u64 cap;
    const u64 *log;
    u32 nb_ranks;
    Reads rd;
    int mf, T;
    u32 hot;
    u32 *surv;         /* [cap]: hot survivors' slots at [0, n_surv_hot), the others at [cap - n_surv_cold, cap) */
    Counters *ctr;
};

/* 8 blocks per SM: the host's grid of 8 blocks per SM is resident at once.  Every iteration ends in a
 * block-wide append; with fewer resident warps its barriers and atomic round trip are not hidden
 * (configs[1] on a B200 at 1000 W: 0.83 ms at 6 blocks per SM and 40 registers, 0.52 ms at 8 and 32). */
__global__ void __launch_bounds__(THREADS, 8)
k_prune(PruneArgs a, Geom g) {
    /* lane = one slot; slots whose quality sums must be evaluated are then handled by the whole
     * warp: lane j owns k-mer positions j and j+32, so each occurrence's k quality bytes are one
     * coalesced read */
    const u32 lane = threadIdx.x & 31;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    const u64 n_iter = (a.cap + stride - 1) / stride;
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u32 n_distinct = 0;
    for (u64 itn = 0; itn < n_iter; itn++, i += stride) {
        u32 cnt = 0, cw = 0, head = NIL32;
        int lb_first = 0;
        bool pass = false, border = false;
        if (i < a.cap) {
            u64 q0, q1, q2, q3;
            ld_sector(&a.table[i], q0, q1, q2, q3);
            if (!(q0 == EMPTY64 && q1 == EMPTY64)) {
                n_distinct++;
                cw = (u32)q2;
                cnt = (cw & CNT_MASK) + 1;          /* the claiming occurrence + the others */
                head = (u32)(q2 >> 32);
                if (cnt > CNT_CAP) cnt = CNT_CAP;
                if ((int)cnt >= a.mf && (cw & CNT_MULTI)) {
                    pass = true;
                    if (GATE_Q * ((int)cnt - 1) < a.T) {
                        border = true;
                        if (cnt > a.nb_ranks || head == NIL32) { atomicExch(&a.ctr->internal, 1u); border = false; pass = false; }
                    }
                    if (border) {
                        /* lower bound of every quality sum from the flags logged with the stamps: a later
                         * occurrence adds >= HIQ at every position when its window is all-HIQ, else >= 20
                         * (it passed the gate); the first one adds its RECORD's first k qualities: >= HIQ
                         * when those are all-HIQ, else nothing is known.  Bound >= T: no rows needed. */
                        const u64 *lg = a.log + (u64)head * a.nb_ranks;
                        u64 first = INF64;
                        int lb = 0;
                        bool first_b = false;
                        for (u32 e = 0; e < cnt; e++) {
                            const u64 en = lg[e], st = en & ~(LOG_A | LOG_B);
                            lb += (en & LOG_A) ? HIQ : GATE_Q;
                            if (st < first) { first = st; first_b = en & LOG_B; lb_first = (en & LOG_A) ? HIQ : GATE_Q; }
                        }
                        lb += (first_b ? HIQ : 0) - lb_first;
                        if (lb >= a.T) border = false;
                    }
                }
            }
        }
        u32 todo = __ballot_sync(0xFFFFFFFFu, border);
        while (todo) {
            const int b = __ffs(todo) - 1;
            todo &= todo - 1;
            const int n = (int)__shfl_sync(0xFFFFFFFFu, cnt, b);
            const u32 hd = __shfl_sync(0xFFFFFFFFu, head, b);
            /* lane e < n holds occurrence e */
            u64 st = (int)lane < n ? (a.log[(u64)hd * a.nb_ranks + lane] & ~(LOG_A | LOG_B)) : INF64;
            u64 first = st;
            for (int o = 16; o; o >>= 1) first = min(first, __shfl_xor_sync(0xFFFFFFFFu, first, o));
            int s0 = 0, s1 = 0;
            for (int e = 0; e < n; e++) {
                const u64 se = __shfl_sync(0xFFFFFFFFu, st, e);
                const u64 r = se / (u64)g.w;
                const u64 o = se == first ? 0 : se - r * (u64)g.w;   /* first occurrence reads q_r0[j], :337-339 */
                const int d = a.rd.dev_of(r);
                const u8 *qp = a.rd.qual[d] + (r - a.rd.rec_base[d]) * (u64)g.L + o;
                if ((int)lane < g.k) s0 += qp[lane];
                if ((int)lane + 32 < g.k) s1 += qp[lane + 32];
            }
            const bool bad = ((int)lane < g.k && s0 < a.T) || ((int)lane + 32 < g.k && s1 < a.T);
            const u32 any_bad = __ballot_sync(0xFFFFFFFFu, bad);
            if ((int)lane == b && any_bad) pass = false;
        }
        if (pass) a.table[i].count = cw | CNT_SURV;
        const bool hot = cnt >= a.hot;
        const u64 at = block_append(pass && hot, &a.ctr->n_surv_hot, pass && !hot, &a.ctr->n_surv_cold);
        if (pass) a.surv[hot ? at : a.cap - 1 - at] = (u32)i;
    }
    for (int o = 16; o; o >>= 1) n_distinct += __shfl_xor_sync(0xFFFFFFFFu, n_distinct, o);
    if (lane == 0 && n_distinct) atomicAdd(&a.ctr->n_distinct, (u64)n_distinct);
}

/* ------------------------------------------------------------------------------------------ */
/* survivor table (pass-2 membership + per-node reductions), partitioned like table 1           */
/* ------------------------------------------------------------------------------------------ */
/* inserts from the home slot idx and marks the home CNT2_DISP when another k-mer holds it.  The count
 * word of a slot is only ever OR-ed or added to (k_init_table2 zeroes it), so the mark survives the
 * seeding of the k-mer that holds the home. */
__device__ __forceinline__ u64 t2_insert(Slot2 *t, u64 cap, u64 idx, u64 lo, u64 hi) {
    for (u32 probe = 0; probe < MAX_PROBE; probe++) {
        u64 o0, o1;
        cas128(&t[idx], EMPTY64, EMPTY64, lo, hi, o0, o1);
        if ((o0 == EMPTY64 && o1 == EMPTY64) || (o0 == lo && o1 == hi)) return idx;
        if (probe == 0) atomicOr(&t[idx].count, CNT2_DISP);
        if (++idx == cap) idx = 0;
    }
    return INF64;
}
/* q2 = word 2 of a k-mer's home slot that holds another k-mer: can the k-mer be further on? */
__device__ __forceinline__ bool home_displaced(u64 q2) { return (u32)q2 & CNT2_DISP; }
/* linear probe from idx; returns slot index or INF64; fills word 2 of the hot sector.  home: idx is
 * the k-mer's home slot, so another k-mer there ends the search unless home_displaced */
__device__ __forceinline__ u64 t2_probe_from(const Slot2 *t, u64 cap, u64 idx, u64 lo, u64 hi, u64 &q2, bool home) {
    for (u32 probe = 0; probe < MAX_PROBE; probe++) {
        u64 q0, q1, q3;
        ld_sector(&t[idx], q0, q1, q2, q3);
        if (q0 == lo && q1 == hi) return idx;
        if (q0 == EMPTY64 && q1 == EMPTY64) return INF64;
        if (home && probe == 0 && !home_displaced(q2)) return INF64;
        if (++idx == cap) idx = 0;
    }
    return INF64;
}
/* home slot in table 2 of a k-mer: in the slice of its hash unit (bucket() = its minimizer bucket), or anywhere in a
 * flat (merged) table, where bucket() is not called */
template <class Bucket>
__device__ __forceinline__ u32 t2_home_in(const Part &pt, Bucket bucket, u64 lo, u64 hi) {
    const u32 h = hash_slot(lo, hi);
    if (pt.flat) return slot_in(h, 0u, pt.flat_len);
    const uint4 ut = __ldg(reinterpret_cast<const uint4 *>(pt.ut + (bucket() >> pt.ushift)));
    return slot_in(h, ut.z, ut.w);
}
__device__ __forceinline__ u32 t2_home(const Part &pt, const Geom &g, u64 lo, u64 hi) {
    return t2_home_in(pt, [&] { return kmer_bucket_of(lo, hi, g.span, g.mmask); }, lo, hi);
}

/* inserts the survivors whose table-1 slots are surv[0, n).  The host launches it on the hot part of
 * k_prune's list first: a k-mer inserted early is more likely to sit at its home slot, where pass 2
 * finds it with one probe, and most windows are windows of hot k-mers. */
__global__ void __launch_bounds__(THREADS)
k_build_table2(const Slot1 *t1, const u32 *surv, u64 n, Slot2 *t2, u64 cap2, Geom g, Part pt, Counters *ctr) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        u64 q0, q1, q2, q3;
        ld_sector(&t1[surv[i]], q0, q1, q2, q3);
        /* (the slice a table-1 slot lies in says nothing: probing runs past slice ends) */
        const u64 at = t2_insert(t2, cap2, t2_home(pt, g, q0, q1), q0, q1);
        if (at == INF64) { atomicExch(&ctr->overflow, 3u); continue; }
        /* the gated occurrences are N-free occurrences: seed node->frequency with them */
        const u32 cnt = ((u32)q2 & CNT_MASK) + 1;
        atomicOr(&t2[at].count, cnt > CNT_CAP ? CNT_CAP : cnt);
    }
}

/* Sharded or multi-round build: a device's survivors as dense Slot2 records, appended round after round,
 * and the finish's flat table over the records of all rounds of this device. */
__global__ void __launch_bounds__(THREADS)
k_compact_table2(const Slot2 *t, u64 cap, Slot2 *out, u64 *n_out) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    const u64 n_iter = (cap + stride - 1) / stride;
    for (u64 itn = 0; itn < n_iter; itn++, i += stride) {
        bool occ = false;
        u64 q0 = 0, q1 = 0, q2 = 0, q3 = 0;
        if (i < cap) { ld_sector(&t[i], q0, q1, q2, q3); occ = !(q0 == EMPTY64 && q1 == EMPTY64); }
        const u64 at = block_append(occ, n_out);
        if (occ) {
            Slot2 *o = out + at;
            u64 r0, r1, r2, r3;
            ld_sector(reinterpret_cast<const char *>(&t[i]) + 32, r0, r1, r2, r3);
            st_sector(o, q0, q1, q2, q3);
            st_sector(reinterpret_cast<char *>(o) + 32, r0, r1, r2, r3);
        }
    }
}
__global__ void __launch_bounds__(THREADS)
k_table2_from_records(const Slot2 *rec, u64 n, Slot2 *t2, u64 cap2, Geom g, Part pt, Counters *ctr) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        u64 q0, q1, q2, q3, r0, r1, r2, r3;
        ld_sector(&rec[i], q0, q1, q2, q3);
        ld_sector(reinterpret_cast<const char *>(&rec[i]) + 32, r0, r1, r2, r3);
        const u64 at = t2_insert(t2, cap2, t2_home(pt, g, q0, q1), q0, q1);
        if (at == INF64) { atomicExch(&ctr->overflow, 3u); continue; }
        Slot2 *o = t2 + at;
        atomicOr(&o->count, (u32)q2 & ~CNT2_DISP);   /* the record's mark is about the table it was compacted from */
        o->rank = 0; o->first_any = q3;
        st_sector(reinterpret_cast<char *>(o) + 32, r0, r1, r2, r3);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* K4 k_pass2: pass 2 = build_graph2 / add_to_graph (:267-320, :412-452) as commutative         */
/* reductions over every N-free window whose k-mer survived (no quality gate, :272-274):        */
/*   count        -> node->frequency (:199, :261-265, :308)                                     */
/*   first_any    -> node->kmer and creation order / node id (:197-201)                         */
/*   out_first[c] -> first time the edge K -> K[1:]+c can have been linked (:311-313); ordering */
/*                   these reproduces the head-insertion order of toNodes (:223-229) and, read  */
/*                   from the predecessor's side, of fromNodes (:231-236).                      */
/* All windows of all runs, unit by unit; atomics are skipped when                                */
/* the loaded value already dominates, so hot k-mers cost reads only.                           */
/* ------------------------------------------------------------------------------------------ */
struct Pass2Args {
    const u64 *runs;
    Slot2 *table;
    u64 cap;
    Counters *ctr;
};

__device__ __forceinline__ u32 coarse_stamp(u64 stamp, u32 cshift) { return (u32)min((u64)254, stamp >> cshift); }
/* can a window with this stamp, followed by base c, still lower out_first[c]?  c2 = the slot's count | coarse word */
__device__ __forceinline__ bool edge_open(u64 c2, u32 c, u32 coarse) { return coarse <= ((u32)(c2 >> (32 + 8 * c)) & 0xFFu); }
/* reductions of one pass-2 hit; c2/c3/o are the loaded count word, first_any and out_first[c]
 * (o is only looked at when edge_open) */
__device__ __forceinline__ void pass2_update(Slot2 *slot, bool count_it, u64 c2, u64 c3, u64 o, bool edge, u32 c, u64 stamp, u32 coarse, u32 fl) {
    if (count_it && ((u32)c2 & CNT2_MASK) < CNT_CAP) atomicAdd(&slot->count, 1u);
    /* in-mask: this k-mer was seen preceded by base (fl >> 4) & 3 */
    const u32 in_bit = ((fl >> 3) & 1u) << (CNT2_IN + ((fl >> 4) & 3u));
    if (in_bit & ~(u32)c2) atomicOr(&slot->count, in_bit);
    if (stamp < c3) atomicMin(&slot->first_any, stamp);
    if (edge && stamp < o) {
        atomicMin(&slot->out_first[c], stamp);
        /* then (never before) lower the coarse bound in the hot sector */
        const u32 sh = 8 * c;
        u32 cur = *reinterpret_cast<volatile u32 *>(&slot->rank);
        while (((cur >> sh) & 0xFFu) > coarse) {
            const u32 old = atomicCAS(&slot->rank, cur, (cur & ~(0xFFu << sh)) | (coarse << sh));
            if (old == cur) break;
            cur = old;
        }
    }
}

/* slow path of pass 2: tuples whose home slot holds a different k-mer; queue entries carry the
 * tuple, its home slot and (top bit of idx) whether the window failed the quality gate */
template <bool WIDE>
__device__ __forceinline__ u32 pass2_drain(const Pass2Args &a, const Part &pt, WarpQueue<WIDE> &q, u32 &qn, bool final, u32 &n_hits_u) {
    const u32 lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    u32 next = 0, n_hits = 0;
    bool have = false, count_it = false;
    u64 lo = 0, hi = 0, stamp = 0, rw1 = 0, rw2 = 0;
    u32 idx = 0, probe = 0, fl = 0;
    __syncwarp();
    for (;;) {
        const u32 need = __ballot_sync(0xFFFFFFFFu, !have);
        const u32 avail = qn - next;
        if (avail == 0 && (need == 0xFFFFFFFFu || (!final && 32 - __popc(need) < (int)pt.qdense2))) break;
        if (need && avail) {
            const u32 my = __popc(need & lt);
            if (!have && my < avail) {
                const u32 e = next + my;
                lo = q.lo[e]; rw1 = q.w1[e]; rw2 = WIDE ? q.w2[e] : 0ull;
                u32 fp;
                tuple_decode<WIDE>(pt, rw1, rw2, hi, fl, fp, stamp);
                idx = q.idx[e];
                count_it = idx >> 31;
                idx &= 0x7FFFFFFFu;
                probe = 0;
                have = true;
            }
            next += min((u32)__popc(need), avail);
        }
        if (have) {
            if (++idx == (u32)a.cap) idx = 0;
            Slot2 *slot = a.table + idx;
            u64 q0, q1, q2, q3;
            ld_sector(slot, q0, q1, q2, q3);
            if (q0 == lo && q1 == hi) {
                const u32 c = (fl >> 1) & 3u, coarse = coarse_stamp(stamp, pt.cshift);
                const bool edge = (fl & 1u) && edge_open(q2, c, coarse);
                u64 o = 0;
                if (edge) o = ld_cg_u64(&slot->out_first[c]);
                pass2_update(slot, count_it, q2, q3, o, edge, c, stamp, coarse, fl);
                n_hits++;
                n_hits_u += count_it;
                have = false;
            } else if ((q0 == EMPTY64 && q1 == EMPTY64) || ++probe >= MAX_PROBE) {
                have = false;
            }
        }
    }
    /* unfinished tuples go back to the (now empty) queue with the slot they have reached */
    __syncwarp();
    qn = q.push(0, have, lo, rw1, rw2, idx | (count_it ? 0x80000000u : 0u));
    __syncwarp();
    return n_hits;
}

template <bool WIDE>
__global__ void __launch_bounds__(THREADS, PASS2_MIN_BLOCKS)
k_pass2(Pass2Args a, Geom g, Part pt) {
    extern __shared__ __align__(128) unsigned char smem[];
    WarpQueue<WIDE> q;
    q.setup(smem);
    RunFeed feed;
    feed.rw = reinterpret_cast<u64 *>(smem + WARPS * WarpQueue<WIDE>::bytes()) + (threadIdx.x >> 5) * 32 * RUN_WORDS;
    const u32 lane = threadIdx.x & 31;
    const u64 n_chunk = (pt.n_runs + THREADS - 1) / THREADS;
    u32 n_hits = 0, qn = 0, n_slow = 0, n_hits_u = 0;
    for (u64 chunk = blockIdx.x; chunk < n_chunk; chunk += gridDim.x) {
        feed.load<false>(a.runs, chunk * THREADS + threadIdx.x, pt.n_runs);
        for (u32 base = 0; base < feed.total; base += 32 * BATCH) {
            u64 lo[BATCH], hi[BATCH], stamp[BATCH], q0[BATCH], q1[BATCH], q2[BATCH], q3[BATCH], of[BATCH];
            u32 idx[BATCH], fl[BATCH];   /* fl: the window's FLB flag bits | gated << FLB | coarse stamp << 8 */
            /* A1: this lane's BATCH consecutive windows of the chunk */
            {
                const u32 t0 = base + lane * BATCH;
                RunCursor cur;
                feed.seek<false, true>(min(t0, feed.total - 1), cur, pt);
#pragma unroll
                for (int u = 0; u < BATCH; u++) {
                    lo[u] = hi[u] = stamp[u] = 0; idx[u] = NIL32; fl[u] = 0;
                    if (t0 + u < feed.total) {
                        if (u) feed.next<false, true>(cur, pt);
                        run_kmer(g, cur, lo[u], hi[u], idx[u]);
                        fl[u] = run_flags2(g, cur.w0, cur.w1, cur.w2, cur.j) | ((u32)(cur.w2 >> cur.j) & 1u) << FLB;
                        stamp[u] = cur.stamp0 + cur.j;
                        fl[u] |= coarse_stamp(stamp[u], pt.cshift) << 8;
                    }
                }
            }
            issue_fence(idx[0], idx[1], idx[2], idx[3]);
            /* A2: the hot sector of the home slot, all loads of the batch in flight together */
#pragma unroll
            for (int u = 0; u < BATCH; u++) {
                q0[u] = q1[u] = q2[u] = q3[u] = 0;
                if (idx[u] != NIL32) ld_sector_ca(a.table + idx[u], q0[u], q1[u], q2[u], q3[u]);
            }
            /* A3: the out_first word a hit would update -- only when the coarse bound in the hot sector says
             * this window can still lower it (the first occurrences of an edge; later ones cost one sector) */
            u32 edges = 0;
#pragma unroll
            for (int u = 0; u < BATCH; u++) {
                of[u] = 0;
                if (idx[u] != NIL32 && q0[u] == lo[u] && q1[u] == hi[u] && (fl[u] & 1u) &&
                    edge_open(q2[u], (fl[u] >> 1) & 3u, (fl[u] >> 8) & 0xFFu)) {
                    edges |= 1u << u;
                    of[u] = ld_ca_u64(&a.table[idx[u]].out_first[(fl[u] >> 1) & 3u]);
                }
            }
            /* B: hit at home -> reductions; home without CNT2_DISP (empty, or nothing was displaced from it;
             * q2 is zero for a window with an N) -> the k-mer did not survive; otherwise queue.
             * node->frequency counts every N-free occurrence; the gated ones were already counted by
             * pass 1 (k_build_table2 seeds count with them), so only ungated windows add to it. */
#pragma unroll
            for (int u = 0; u < BATCH; u++) {
                const bool valid = idx[u] != NIL32;
                const bool ungated = !((fl[u] >> FLB) & 1u);
                const bool hit = valid && q0[u] == lo[u] && q1[u] == hi[u];
                if (hit) {
                    pass2_update(a.table + idx[u], ungated, q2[u], q3[u], of[u], (edges >> u) & 1u, (fl[u] >> 1) & 3u, stamp[u],
                                 (fl[u] >> 8) & 0xFFu, fl[u]);
                    n_hits++;
                    n_hits_u += ungated;
                }
                qn = q.push_lazy(qn, !hit && home_displaced(q2[u]), lo[u], idx[u] | (ungated ? 0x80000000u : 0u), [&](u64 &t1, u64 &t2) {
                    pack_tuple<WIDE>(pt, hi[u], fl[u] & ((1u << FLB) - 1), 0u, stamp[u], t1, t2);
                });
            }
            if (qn >= pt.qflush2) {
                n_slow += qn; n_hits += pass2_drain<WIDE>(a, pt, q, qn, false, n_hits_u); n_slow -= qn;
            }
        }
    }
    n_slow += qn;
    n_hits += pass2_drain<WIDE>(a, pt, q, qn, true, n_hits_u);
    if (lane == 0 && n_slow) atomicAdd(&a.ctr->n_slow2, (u64)n_slow);
    for (int o = 16; o; o >>= 1) { n_hits += __shfl_xor_sync(0xFFFFFFFFu, n_hits, o); n_hits_u += __shfl_xor_sync(0xFFFFFFFFu, n_hits_u, o); }
    if (lane == 0 && n_hits) atomicAdd(&a.ctr->n_hits, (u64)n_hits);
    if (lane == 0 && n_hits_u) atomicAdd(&a.ctr->n_hits_ungated, (u64)n_hits_u);
}

/* ------------------------------------------------------------------------------------------ */
/* K5 export.  collect (first_any, slot) -> radix sort by first_any (host calls CUB) ->        */
/* assign ranks -> emit nodes in creation order with ordered edge lists.                        */
/* ------------------------------------------------------------------------------------------ */
__global__ void __launch_bounds__(THREADS)
k_collect(const Slot2 *t, u64 cap, u64 *keys, u32 *vals, Counters *ctr) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    u64 n_iter = (cap + stride - 1) / stride;
    for (u64 itn = 0; itn < n_iter; itn++, i += stride) {
        bool occ = false;
        u64 q0 = 0, q1 = 0, q2 = 0, q3 = 0;
        if (i < cap) {
            ld_sector(&t[i], q0, q1, q2, q3);
            occ = !(q0 == EMPTY64 && q1 == EMPTY64);
        }
        const u64 o = block_append(occ, &ctr->n_nodes);
        if (occ) {
            keys[o] = q3;            /* first_any */
            vals[o] = (u32)i;
            if (q3 == INF64) atomicExch(&ctr->internal, 2u);
        }
    }
}

__global__ void k_assign_rank(Slot2 *t, const u32 *vals, u64 n) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) t[vals[i]].rank = (u32)i;
}

/* The minimizer values of a k-mer's four successors and four predecessors from ONE scan of its
 * m-mers: a successor K[1:]+c keeps K's m-mers but the first and gains one at the end, a
 * predecessor c+K[:-1] keeps all but the last and gains one at the front. */
struct NeighbourMini {
    u32 tail, head;      /* min hash over K's m-mer positions >= 1 / <= span-2 (~0 when there is none) */
    u32 x_first, x_last; /* K's first and last m-mer */
    __device__ __forceinline__ void scan(u64 lo, u64 hi, const Geom &g) {
        tail = head = ~0u;
        x_first = (u32)lo & g.mmask;
        for (int j = 0; j < g.span; j++) {
            x_last = (u32)lo & g.mmask;
            const u32 h = mini_hash(x_last);
            if (j > 0) tail = min(tail, h);
            if (j < g.span - 1) head = min(head, h);
            lo = (lo >> 2) | (hi << 62);
            hi >>= 2;
        }
    }
    __device__ __forceinline__ u32 succ_bucket(u32 c, const Geom &g) const {
        return mini_bucket(min(tail, mini_hash((x_last >> 2) | (c << (2 * (g.m - 1))))));
    }
    __device__ __forceinline__ u32 pred_bucket(u32 c, const Geom &g) const {
        return mini_bucket(min(head, mini_hash(((x_first << 2) | c) & g.mmask)));
    }
};

/* out = v[0, n) in descending order of t, NIL32 beyond n */
__device__ __forceinline__ void sort_desc4(u64 (&t)[4], u32 (&v)[4], int n, u32 (&out)[4]) {
    for (int a = 1; a < n; a++)
        for (int b = a; b > 0 && t[b] > t[b - 1]; b--) {
            u64 x = t[b]; t[b] = t[b - 1]; t[b - 1] = x;
            u32 y = v[b]; v[b] = v[b - 1]; v[b - 1] = y;
        }
    for (int e = 0; e < 4; e++) out[e] = e < n ? v[e] : NIL32;
}
struct Edges { int n_out, n_in; u32 succ[4], pred[4]; };   /* NIL32 beyond the degrees */

/* The edge lists of the node with key (lo, hi), count word cw and out_first words of[4], in the reference's order.
 * Lookup: buckets() (may find ask for a bucket?), find(bucket, lo, hi, q2) = a neighbour's slot or null (bucket() =
 * its minimizer bucket, q2 = word 2: its rank above bit 32), out_first(slot, c). */
template <class Lookup>
__device__ __forceinline__ Edges node_edges(const Lookup &lk, const Geom &g, u64 lo, u64 hi, u32 cw, const u64 *of) {
    Edges e;
    u64 tt[4]; u32 vv[4];
    NeighbourMini nm;
    if (lk.buckets()) nm.scan(lo, hi, g);     /* the buckets of all eight neighbours from one scan of the k-mer */
    /* toNodes: successors K[1:]+c that survived, newest first-seen at the head (:223-229) */
    int n = 0;
#pragma unroll 1   /* the probes are serial anyway (ld_sector is volatile); unrolled, k_export spills */
    for (u32 c = 0; c < 4; c++) {
        const u64 tf = of[c];
        if (tf == INF64) continue;
        u64 slo, shi, q2;
        kmer_succ(lo, hi, c, g.k, slo, shi);
        if (!lk.find([&] { return nm.succ_bucket(c, g); }, slo, shi, q2)) continue;
        tt[n] = tf; vv[n] = (u32)(q2 >> 32); n++;
    }
    sort_desc4(tt, vv, n, e.succ); e.n_out = n;
    /* fromNodes: predecessors c+K[:-1] that survived and were seen followed by K's last base;
     * the edge P->K was first linked at P.out_first[last(K)] + 1 (:231-236) */
    n = 0;
    const u32 last = kmer_last(lo, hi, g.k), in_mask = (cw >> CNT2_IN) & 15u;
    for (u32 c = 0; c < 4; c++) {
        if (!((in_mask >> c) & 1u)) continue;   /* never seen after base c: c+K[:-1] -> K was never linked */
        u64 plo, phi, q2;
        kmer_pred(lo, hi, c, g.kmask_lo, g.kmask_hi, plo, phi);
        const Slot2 *p = lk.find([&] { return nm.pred_bucket(c, g); }, plo, phi, q2);
        if (!p) continue;
        const u64 tf = lk.out_first(p, last);
        if (tf == INF64) continue;
        tt[n] = tf; vv[n] = (u32)(q2 >> 32); n++;
    }
    sort_desc4(tt, vv, n, e.pred); e.n_in = n;
    return e;
}

/* neighbours in this device's table: sliced by hash unit, or flat (merged), where no bucket is needed */
struct LocalTable {
    const Slot2 *table; u64 cap; Part pt;
    __device__ __forceinline__ bool buckets() const { return !pt.flat; }
    template <class Bucket> __device__ __forceinline__ const Slot2 *find(Bucket bucket, u64 lo, u64 hi, u64 &q2) const {
        const u64 idx = t2_probe_from(table, cap, t2_home_in(pt, bucket, lo, hi), lo, hi, q2, true);
        return idx == INF64 ? nullptr : table + idx;
    }
    __device__ __forceinline__ u64 out_first(const Slot2 *s, u32 c) const { return s->out_first[c]; }
};

struct ExportArgs {
    const Slot2 *table;
    u64 cap;
    const u64 *keys;   /* sorted first_any */
    const u32 *vals;   /* slot of rank i */
    u64 n;
    u64 *first_pos;
    u16 *frequency;
    u8 *out_deg, *in_deg;
    u32 *out_succ, *in_pred;
    u64 *kmer_lo, *kmer_hi; /* may be null */
};

/* one thread per node, in creation order (coalesced result rows).  Measured and rejected: walking
 * the table in slot order with a bucket-sliced merged table, to keep the <= 8 neighbour lookups of
 * a node inside one L2-resident slice (its neighbours mostly share its minimizer): the scattered
 * 64-byte result records and the denser slices cost more than the locality gave (finish at 8 GPUs
 * 7.7 -> 13.8 ms, configs[4] at full size 140 -> 245 ms). */
__global__ void __launch_bounds__(THREADS)
k_export(ExportArgs a, Geom g, Part pt) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const Slot2 *s = a.table + a.vals[i];
    const u64 lo = s->klo, hi = s->khi;
    const u32 cw = s->count, cnt = cw & CNT2_MASK;
    a.first_pos[i] = a.keys[i];
    a.frequency[i] = (u16)(cnt > CNT_CAP ? CNT_CAP : cnt);
    if (a.kmer_lo) { a.kmer_lo[i] = lo; a.kmer_hi[i] = hi; }
    const Edges ed = node_edges(LocalTable{a.table, a.cap, pt}, g, lo, hi, cw, s->out_first);
    a.out_deg[i] = (u8)ed.n_out;
    a.in_deg[i] = (u8)ed.n_in;
    for (int e = 0; e < 4; e++) { a.out_succ[i * 4 + e] = ed.succ[e]; a.in_pred[i * 4 + e] = ed.pred[e]; }
}

/* ------------------------------------------------------------------------------------------ */
/* K5 on several devices: every device finishes ITS survivors (the k-mers of the hash units it   */
/* owns) and only the finished node rows travel.  Per device r, with n_r survivors of n in all:   */
/*   F1  flat table over its own survivor records, (first_any, slot) sorted by first_any          */
/*   F2  creation rank of a node = its position in the merge of all devices' sorted stamps:       */
/*       own position + sum over the peers of lower_bound(peer's stamps, stamp)  (stamps are      */
/*       window numbers: no two nodes share one); written into the table slot for the peers       */
/*   F3  edge lists: a neighbour is looked up in the table of the device that owns its minimizer  */
/*       bucket (a peer load over NVLink for about one neighbour in eight: consecutive k-mers     */
/*       mostly share their minimizer), the finished 32-byte row is stored at its creation rank   */
/*       in the finishing device's row buffer (one peer store per node), which unpacks the rows   */
/*       into the result arrays.                                                                  */
/* Between the steps the devices meet at k_peer_barrier (flags in peer memory), not on the host.  */
/* ------------------------------------------------------------------------------------------ */
/* A finished node as it travels to the finishing device: one 32-byte sector.
 * w0 = first_pos (STAMP_BITS) | frequency << 40 | out_deg << 56 | in_deg << 59 ; w1..w3 = the first three
 * successors and the first three predecessors (NIL32 beyond the degree).  A node with four successors or four
 * predecessors (rare) also appends {rank | 4th successor << 32, 4th predecessor} to an overflow list; the
 * k-mer, when the caller wants it, goes to a second array of 16-byte entries. */
constexpr int ROW_WORDS = 4;
static_assert(STAMP_BITS <= 40, "first_pos shares a word with the frequency and the degrees");
struct RowSink {
    u64 *rows;         /* [n][ROW_WORDS], indexed by creation rank */
    ulonglong2 *over;  /* overflow entries */
    u32 *n_over;
    ulonglong2 *kmers; /* [n] or null */
};

/* neighbours in the flat table of the device that owns their bucket (node_edges' Lookup) */
struct PeerTables {
    const Slot2 *table[MAX_DEV];   /* every device's flat survivor table (own: local pointer) */
    u32 len[MAX_DEV];
    const u8 *owner;               /* [hash units] owning device */
    u32 ushift;
    __device__ __forceinline__ bool buckets() const { return true; }
    template <class Bucket> __device__ __forceinline__ const Slot2 *find(Bucket bucket, u64 lo, u64 hi, u64 &q2) const {
        const u32 d = __ldg(owner + (bucket() >> ushift));
        const u64 idx = t2_probe_from(table[d], len[d], slot_in(hash_slot(lo, hi), 0u, len[d]), lo, hi, q2, true);
        return idx == INF64 ? nullptr : table[d] + idx;
    }
    __device__ __forceinline__ u64 out_first(const Slot2 *s, u32 c) const { return ld_cg_u64(&s->out_first[c]); }
};
struct KeySegs {
    u64 off[MAX_DEV + 1];          /* device d's sorted stamps are all_keys[off[d] .. off[d+1]) */
};

__device__ __forceinline__ u64 lower_bound_u64(const u64 *a, u64 n, u64 key) {
    u64 lo = 0;
    while (n) {
        const u64 half = n >> 1;
        const bool right = ld_ca_u64(a + lo + half) < key;
        lo = right ? lo + half + 1 : lo;
        n = right ? n - half - 1 : half;
    }
    return lo;
}

/* One thread per own node, in stamp order.  The block's first and last stamp bracket every other one of the block:
 * 2 G threads first find those two positions in each peer's array, the per-node searches then run over the
 * short stretch between them (about THREADS elements, not the whole array). */
__global__ void __launch_bounds__(THREADS)
k_global_rank(const u64 *all_keys, const __grid_constant__ KeySegs ks, int G, int self, Slot2 *table, const u32 *vals, u32 *gid, const Counters *ctr) {
    __shared__ u64 s_lo[MAX_DEV], s_hi[MAX_DEV];
    if (ctr->internal) return;   /* block-uniform */
    const u64 n = ks.off[self + 1] - ks.off[self];
    const u64 b0 = (u64)blockIdx.x * blockDim.x, i = b0 + threadIdx.x;
    const u64 *mine = all_keys + ks.off[self];
    if (threadIdx.x < 2 * G && b0 < n) {
        const int d = threadIdx.x % G;
        const u64 key = threadIdx.x < G ? mine[b0] : mine[min(b0 + blockDim.x, n) - 1];
        const u64 at = d == self ? 0 : lower_bound_u64(all_keys + ks.off[d], ks.off[d + 1] - ks.off[d], key);
        if (threadIdx.x < G) s_lo[d] = at; else s_hi[d] = at;
    }
    __syncthreads();
    if (i >= n) return;
    const u64 key = mine[i];
    u64 r = i;
    for (int d = 0; d < G; d++)
        if (d != self) r += s_lo[d] + lower_bound_u64(all_keys + ks.off[d] + s_lo[d], s_hi[d] - s_lo[d], key);
    gid[i] = (u32)r;
    table[vals[i]].rank = (u32)r;
}

struct ExportDistArgs {
    const u64 *keys;   /* this device's sorted first_any */
    const u32 *vals;   /* slot (own table) of its i-th node */
    const u32 *gid;    /* creation rank of its i-th node */
    u64 n;
    RowSink sink;      /* the finishing device's row buffer (peer memory) */
    int self;
};

__global__ void __launch_bounds__(THREADS)
k_export_dist(ExportDistArgs a, const __grid_constant__ PeerTables pt, Geom g, const Counters *ctr) {
    if (ctr->internal) return;
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const Slot2 *s = pt.table[a.self] + a.vals[i];
    const u64 lo = s->klo, hi = s->khi;
    const u32 cw = s->count, cnt = cw & CNT2_MASK;
    const Edges e = node_edges(pt, g, lo, hi, cw, s->out_first);
    const u32 id = a.gid[i];
    const u64 w0 = a.keys[i] | ((u64)(cnt > CNT_CAP ? CNT_CAP : cnt) << 40) | ((u64)e.n_out << 56) | ((u64)e.n_in << 59);
    st_sector(a.sink.rows + (u64)id * ROW_WORDS, w0, (u64)e.succ[0] | ((u64)e.succ[1] << 32), (u64)e.succ[2] | ((u64)e.pred[0] << 32),
              (u64)e.pred[1] | ((u64)e.pred[2] << 32));
    if (e.n_out == 4 || e.n_in == 4) {
        const u32 at = atomicAdd_system(a.sink.n_over, 1u);
        a.sink.over[at] = make_ulonglong2((u64)id | ((u64)e.succ[3] << 32), (u64)e.pred[3]);
    }
    if (a.sink.kmers) a.sink.kmers[id] = make_ulonglong2(lo, hi);
}

/* the finishing device: rows (creation order) -> the result arrays */
__global__ void __launch_bounds__(THREADS)
k_unpack_rows(RowSink r, u64 n, ExportArgs a) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 w0, w1, w2, w3;
    ld_sector(r.rows + i * ROW_WORDS, w0, w1, w2, w3);
    a.first_pos[i] = w0 & ((1ull << 40) - 1);
    a.frequency[i] = (u16)(w0 >> 40);
    a.out_deg[i] = (u8)((w0 >> 56) & 7u);
    a.in_deg[i] = (u8)((w0 >> 59) & 7u);
    reinterpret_cast<uint4 *>(a.out_succ)[i] = make_uint4((u32)w1, (u32)(w1 >> 32), (u32)w2, NIL32);
    reinterpret_cast<uint4 *>(a.in_pred)[i] = make_uint4((u32)(w2 >> 32), (u32)w3, (u32)(w3 >> 32), NIL32);
    if (a.kmer_lo) { const ulonglong2 km = r.kmers[i]; a.kmer_lo[i] = km.x; a.kmer_hi[i] = km.y; }
}
/* ... and the fourth edges of the few nodes that have them (after k_unpack_rows) */
__global__ void __launch_bounds__(THREADS)
k_unpack_overflow(RowSink r, ExportArgs a) {
    const u32 n = *r.n_over;
    for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const ulonglong2 e = r.over[j];
        const u32 id = (u32)e.x;
        a.out_succ[(u64)id * 4 + 3] = (u32)(e.x >> 32);
        a.in_pred[(u64)id * 4 + 3] = (u32)e.y;
    }
}

/* Barrier between the devices of a sharded finish, on the device: every device owns a block of
 * MAX_DEV flag words that its peers can store to (peer-mapped); arriving = storing this barrier's
 * sequence number into my word of everybody's block (after a system-wide fence: the preceding
 * kernels' peer stores are ordered before it), leaving = all words of my own block have reached it.
 * One warp; the rest of the stream waits behind this kernel.  A peer that never arrives (its process
 * died) is given up on after `patience_ns`: the build fails with an error instead of hanging. */
struct PeerFlags { u64 *flags[MAX_DEV]; };
__global__ void k_peer_barrier(const __grid_constant__ PeerFlags pf, int G, int self, u64 seq, u64 patience_ns, Counters *ctr) {
    const int t = threadIdx.x;
    if (t >= G) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(pf.flags[t] + self), "l"(seq) : "memory");
    const u64 *mine = pf.flags[self] + t;
    u64 t0, now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        u64 v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(mine) : "memory");
        if (v >= seq) break;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (now - t0 > patience_ns) { atomicExch(&ctr->internal, 9u); break; }
        __nanosleep(100);
    }
    __threadfence_system();
}

/* ------------------------------------------------------------------------------------------ */
/* Layout of the reference's `nodes` map (SURVEY 8f-2, first half).  Everything downstream of   */
/* the block iterates dense_hash_map<const char*, node*, my_hash, eqstr> (:599, :659, :1139), so */
/* vdjer.dot, the ROOT_INIT lines and the root list depend on the BUCKET every node lands in:   */
/* MurmurHash64A of the k ASCII characters (hash_utils.c:5-46, seed 97), divided by 8 because    */
/* the key is a pointer (sparsehash hashtable-common.h:352-361), first-come-first-served         */
/* triangular probing (densehashtable.h:119), the table doubling whenever an insert would fill   */
/* more than half of it, each time by re-inserting the old table in BUCKET order (:631-653).     */
/* The glue used to replay those inserts on one host thread (0.25 us per node, 80 % of its      */
/* cost).  Here every doubling stage is laid out in parallel: first-come-first-served open       */
/* addressing is the unique stable assignment in which every bucket prefers the element that is  */
/* earlier in the insertion sequence, so elements simply keep proposing (atomicMin of their      */
/* sequence key) to the next bucket of their probe sequence until nobody is displaced any more.  */
/* ------------------------------------------------------------------------------------------ */
__device__ __forceinline__ u64 murmur64a_kmer(u64 lo, u64 hi, int k) {
    const u64 m = 0xc6a4a7935bd1e995ull;
    const int r = 47;
    u64 h = 97ull ^ ((u64)k * m);
    int done = 0;
    for (; done + 8 <= k; done += 8) {   /* eight characters = one little-endian word */
        u64 w = 0;
        for (int j = 0; j < 8; j++) {
            const u32 c = (u32)lo & 3u;
            w |= (u64)(c == 0 ? 'A' : c == 1 ? 'C' : c == 2 ? 'G' : 'T') << (8 * j);
            lo = (lo >> 2) | (hi << 62);
            hi >>= 2;
        }
        w *= m; w ^= w >> r; w *= m;
        h ^= w; h *= m;
    }
    if (done < k) {
        u64 w = 0;
        for (int j = 0; done + j < k; j++) {
            const u32 c = (u32)lo & 3u;
            w |= (u64)(c == 0 ? 'A' : c == 1 ? 'C' : c == 2 ? 'G' : 'T') << (8 * j);
            lo = (lo >> 2) | (hi << 62);
            hi >>= 2;
        }
        h ^= w; h *= m;
    }
    h ^= h >> r; h *= m; h ^= h >> r;
    return h;
}
/* the hash as the container uses it, per node in creation order */
__global__ void __launch_bounds__(THREADS)
k_hm_hash(const u64 *klo, const u64 *khi, u64 n, int k, u64 *hash) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) hash[i] = murmur64a_kmer(klo[i], khi[i], k) >> 3;
}
struct HmStage {
    const u64 *hash;     /* [n] */
    u64 *owner;          /* [buckets] sequence key << 32 | element; all ones = empty */
    u32 *probe;          /* [n] collisions so far in this stage */
    u32 *prev_bucket;    /* [n] bucket in the previous stage's table */
    u32 *changed;
    u32 n_old, n_all;    /* elements re-inserted from the previous table / elements of this stage */
    u32 prev_buckets;    /* size of the previous table: keys of the newly inserted elements start there */
    u32 mask;
};
__device__ __forceinline__ u32 hm_bucket(const HmStage &a, u32 e) {
    const u64 p = a.probe[e];
    return (u32)(a.hash[e] + p * (p + 1) / 2) & a.mask;
}
__device__ __forceinline__ u64 hm_key(const HmStage &a, u32 e) {
    /* the old table's elements come first, in its bucket order; then the new ones in creation order */
    const u32 key = e < a.n_old ? a.prev_bucket[e] : a.prev_buckets + (e - a.n_old);
    return ((u64)key << 32) | e;
}
/* one round: an element that does not (or no longer) own its bucket moves on; everybody (re)proposes */
__global__ void __launch_bounds__(THREADS)
k_hm_round(HmStage a, int first) {
    const u32 e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.n_all) return;
    if (first) a.probe[e] = 0;
    else if ((u32)ld_cg_u64(&a.owner[hm_bucket(a, e)]) != e) {
        a.probe[e]++;
        *a.changed = 1u;
    }
    atomicMin(&a.owner[hm_bucket(a, e)], hm_key(a, e));
}
/* after the last round: remember the buckets for the next stage */
__global__ void __launch_bounds__(THREADS)
k_hm_settle(HmStage a) {
    const u32 e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < a.n_all) a.prev_bucket[e] = hm_bucket(a, e);
}
/* the final table as the glue reads it: node per bucket, NIL32 = empty */
__global__ void __launch_bounds__(THREADS)
k_hm_slots(const u64 *owner, u64 buckets, u32 *slots) {
    const u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (b < buckets) slots[b] = owner[b] == ~0ull ? NIL32 : (u32)owner[b];
}

/* pruned pass-1 table for parity checks */
__global__ void __launch_bounds__(THREADS)
k_export_pre(const Slot1 *t, u64 cap, u64 *klo, u64 *khi, u16 *freq, u64 *n_out) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x, stride = (u64)gridDim.x * blockDim.x;
    for (; i < cap; i += stride) {
        u64 q0, q1, q2, q3;
        ld_sector(&t[i], q0, q1, q2, q3);
        if (q0 == EMPTY64 && q1 == EMPTY64) continue;
        if (!((u32)q2 & CNT_SURV)) continue;
        u64 o = atomicAdd(n_out, 1ull);
        u32 cnt = ((u32)q2 & CNT_MASK) + 1;
        klo[o] = q0; khi[o] = q1; freq[o] = (u16)(cnt > CNT_CAP ? CNT_CAP : cnt);
    }
}

/* ------------------------------------------------------------------------------------------ */
/* Queries (vdjgraph_query): the node of every k-mer window of caller sequences, looked up in the */
/* finished survivor table (rank in the upper half of word 2, as k_export reads it).  The host     */
/* streams the batch in chunks of whole queries; per chunk k_query_pack packs the text and        */
/* k_query answers its windows.                                                                    */
/* ------------------------------------------------------------------------------------------ */
/* One thread per 64 bytes of the chunk's text: 2-bit bases (A0 C1 G2 T3, N stored as 0, base j at bits
 * 2j of the chunk's words: the key layout) and a mask, bit j = byte j is not ACGT.  A byte outside ACGTN
 * lowers bad[0] to its position in the batch (base + j), as staging flags a bad base.  The text buffer is
 * readable up to the next multiple of 64 bytes; bytes past n are ignored. */
__global__ void __launch_bounds__(THREADS)
k_query_pack(const unsigned char *text, u64 n, u64 base, u64 *bases, u64 *nmask, u64 *bad) {
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 j0 = t * 64;
    if (j0 >= n) return;
    const uint4 *src = reinterpret_cast<const uint4 *>(text + j0);
    u64 b[2] = { 0, 0 }, nm = 0, first_bad = ~0ull;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint4 v = src[q];
        const u32 words[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int j = 16 * q; j < 16 * q + 16; j++) {
            const u32 ch = (words[(j >> 2) & 3] >> (8 * (j & 3))) & 0xFFu;
            const u32 code = ch == 'C' ? 1u : ch == 'G' ? 2u : ch == 'T' ? 3u : 0u;
            const bool acgt = code != 0u || ch == 'A';
            b[j >> 5] |= (u64)code << (2 * (j & 31));
            if (!acgt && j0 + j < n) {
                nm |= 1ull << j;
                if (ch != 'N') first_bad = min(first_bad, j0 + j);
            }
        }
    }
    bases[2 * t] = b[0];
    bases[2 * t + 1] = b[1];
    nmask[t] = nm;
    if (first_bad != ~0ull) atomicMin(bad, base + first_bad);
}

struct QueryArgs {
    const u64 *bases, *nmask;   /* k_query_pack's output for the chunk */
    u64 n_words, n_mwords;      /* their lengths in words */
    const u64 *qoff;            /* [nq] first byte of query i in the chunk */
    const u64 *woff;            /* [nq + 1] first window of query i in the chunk; woff[nq] = nw */
    u64 nq, nw;
    const Slot2 *table;         /* the finished survivor table; null when the graph has no nodes */
    u64 cap;
    u32 *out;                   /* [nw] creation rank, NIL32 = N in the window or not a node */
    u64 *found;                 /* += windows whose k-mer is a node (one atomic per warp) */
};

/* BATCH consecutive windows per thread: their first probes are issued back to back (the table is far
 * larger than L2 on real inputs, every probe is a random HBM sector); the rare longer probe sequences
 * continue one by one.  The query of the first window is found by binary search over woff, the others
 * by stepping forward. */
__global__ void __launch_bounds__(THREADS)
k_query(QueryArgs a, Geom g, Part pt) {
    const u64 w0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * BATCH;
    u32 n_found = 0;
    if (w0 < a.nw) {
        u64 l = 0, r = a.nq;   /* woff[l] <= w0 < woff[r] */
        while (r - l > 1) {
            const u64 m = (l + r) >> 1;
            if (a.woff[m] <= w0) l = m; else r = m;
        }
        u64 q = l, cur = a.woff[q], next = a.woff[q + 1];
        u64 lo[BATCH], hi[BATCH], idx[BATCH], q2[BATCH], q3[BATCH];
        bool live[BATCH];
        u32 rank[BATCH];
#pragma unroll
        for (int b = 0; b < BATCH; b++) {
            const u64 w = w0 + b;
            live[b] = false; rank[b] = NIL32; lo[b] = hi[b] = 0; idx[b] = 0;
            if (w >= a.nw) continue;
            while (w >= next) { q++; cur = next; next = a.woff[q + 1]; }
            const u64 p = a.qoff[q] + (w - cur);   /* first byte of the window in the chunk */
            const u64 mw = p >> 6, bw = p >> 5;
            if (extract_mask(a.nmask + mw, (int)min((u64)2, a.n_mwords - mw), (int)(p & 63)) & g.kones) continue;
            extract_kmer(a.bases + bw, (int)min((u64)3, a.n_words - bw), (int)(p & 31), g.kmask_lo, g.kmask_hi, lo[b], hi[b]);
            if (!a.table) continue;
            idx[b] = t2_home(pt, g, lo[b], hi[b]);
            live[b] = true;
        }
        u64 k0[BATCH], k1[BATCH];
#pragma unroll
        for (int b = 0; b < BATCH; b++)
            if (live[b]) ld_sector(&a.table[idx[b]], k0[b], k1[b], q2[b], q3[b]);
#pragma unroll
        for (int b = 0; b < BATCH; b++) {
            if (!live[b]) continue;
            bool hit = k0[b] == lo[b] && k1[b] == hi[b];
            if (!hit && home_displaced(q2[b])) {
                const u64 from = idx[b] + 1 == a.cap ? 0 : idx[b] + 1;
                hit = t2_probe_from(a.table, a.cap, from, lo[b], hi[b], q2[b], false) != INF64;
            }
            if (hit) { rank[b] = (u32)(q2[b] >> 32); n_found++; }
        }
#pragma unroll
        for (int b = 0; b < BATCH; b++)
            if (w0 + b < a.nw) a.out[w0 + b] = rank[b];
    }
    n_found = __reduce_add_sync(0xFFFFFFFFu, n_found);
    if ((threadIdx.x & 31) == 0 && n_found) atomicAdd(a.found, (u64)n_found);
}

} // namespace vdjg
