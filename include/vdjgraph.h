/*
 * vdjgraph.h -- C ABI of libvdjgraph.so: B200-native de Bruijn graph build for V'DJer.
 *
 * This is the drop-in boundary for ONE stage of the reference: the scoped block in assemble(),
 * /root/reference/src/main/c/assembler2_vdj.c:1381-1415, i.e. the calls
 *
 *     build_pre_graph(input, pre_nodes)            :1388   (definition :369-409)
 *     build_pre_graph(unaligned_input, pre_nodes)  :1390
 *     prune_pre_graph(pre_nodes)                   :1393   (definition :467-484)
 *     build_graph2(input, nodes, pool, 1, pre_nodes)           :1402 (definition :412-452)
 *     build_graph2(unaligned_input, nodes, pool, 0, pre_nodes) :1407
 *
 * The reference has no plugin/FFI interface for this stage; the functions above take C++
 * sparsehash maps and read globals (read_length :97, kmer_size :98, p.min_node_freq,
 * p.min_base_quality params.h:6-7).  The entry points below are what a cgo/ctypes/C++ caller
 * binds instead: plain pointers and sizes in, plain arrays out.  INTEGRATION.md shows the
 * reference-side call site and the host glue that rebuilds `nodes`/`pool` from the result.
 *
 * Conventions: every function returns VDJGRAPH_OK (0) or a negative vdjgraph_status; the library
 * never calls exit(), never writes to stdout (the reference reserves stdout for SAM,
 * quick_map3.c:168-180) and never throws across the ABI.  One build at a time per context.
 * There is no CPU fallback: without a usable CUDA device every call fails with
 * VDJGRAPH_ERR_CUDA.
 */
#ifndef VDJGRAPH_H
#define VDJGRAPH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VDJGRAPH_ABI_VERSION 5

typedef enum vdjgraph_status {
    VDJGRAPH_OK = 0,
    VDJGRAPH_ERR_PARAM = -1,          /* k > 50 (MAX_KMER_LEN :70), k > read_length, read_length > 255 (bam_read.c:208), NULL pointers */
    VDJGRAPH_ERR_STRAND = -2,         /* record does not start with '0' or '1'; the reference exit(-1)s, :383-391 */
    VDJGRAPH_ERR_BASE = -3,           /* base outside ACGTN; the reference would hash it literally and exit(-1) in seq_to_int, seq_to_kmer.c:23-25 */
    VDJGRAPH_ERR_TOO_MANY_NODES = -4, /* more than MAX_NODES = 900 M distinct gated k-mers (:73, :379) or > 2^32-2 records */
    VDJGRAPH_ERR_CUDA = -5,           /* no device / CUDA runtime error; see vdjgraph_last_error() */
    VDJGRAPH_ERR_NOMEM = -6,
    VDJGRAPH_ERR_STATE = -7,          /* call sequence violated (e.g. run before stage); see "Call order" */
    VDJGRAPH_ERR_INTERNAL = -8
} vdjgraph_status;

/*
 * Call order.  A context is in one of the states EMPTY, STAGED, COUNTED, PLANNED, PEERS_SET, SCATTERED,
 * PASSES_DONE, FINISH_PLANNED, FINISH_STEP0, FINISH_STEP1, FINISH_STEP2, FINISHED ("staged": any but EMPTY).
 * A call made in a state it does not accept fails with VDJGRAPH_ERR_STATE and changes nothing; the message
 * names the call, the state and the states that accept it.
 *
 *   call                              accepted in                              success leaves
 *   vdjgraph_stage*, _shard_stage*    any                                      STAGED
 *   vdjgraph_set_params               any                                      EMPTY if read_length or kmer_size
 *                                                                              changed, else STAGED if staged
 *   vdjgraph_run                      staged, one rank                         FINISHED
 *   vdjgraph_shard_count              STAGED, FINISHED                         COUNTED
 *   vdjgraph_shard_plan               COUNTED                                  PLANNED
 *   vdjgraph_shard_set_peers          PLANNED .. FINISHED                      PEERS_SET from PLANNED, else unchanged
 *   vdjgraph_shard_rounds             PLANNED .. FINISHED                      unchanged
 *   vdjgraph_shard_scatter            PEERS_SET; PASSES_DONE with rounds left  SCATTERED
 *   vdjgraph_shard_passes             SCATTERED                                PASSES_DONE
 *   vdjgraph_shard_gather_plan        PASSES_DONE of the last round            FINISH_PLANNED
 *   vdjgraph_shard_finish_step(s)     FINISH_PLANNED (s = 0), FINISH_STEP<s-1> FINISH_STEP<s>
 *   vdjgraph_shard_finish             FINISH_STEP2                             FINISHED
 *   vdjgraph_fetch, _fetch_pre_table  FINISHED, one rank or rank 0             unchanged
 *   vdjgraph_stats                    FINISHED                                 unchanged
 *   vdjgraph_query                    FINISHED, one rank                       unchanged
 *
 * Calls not listed accept any state.  vdjgraph_fetch_pre_table also needs a one-device, one-round build
 * (VDJGRAPH_ERR_STATE otherwise).  Any other failure of a staging call leaves EMPTY; of another call on
 * staged records, STAGED: the records stay staged, and vdjgraph_run or vdjgraph_shard_count builds again.
 * Failed argument checks (NULL pointers, parameters) and the read-only calls (fetch, stats, pre_table,
 * query) leave the state as it was.
 */

/* What the stage reads from the reference's globals, as one POD. */
typedef struct vdjgraph_params {
    int32_t read_length;      /* global read_length (:97); all records have exactly this many bases */
    int32_t kmer_size;        /* global kmer_size (:98) = --k; 1..50 */
    int32_t min_node_freq;    /* p.min_node_freq = --mf */
    int32_t min_base_quality; /* p.min_base_quality = --mq; values > 254 are clamped like main() :1514-1516 */
    int32_t device;           /* CUDA device ordinal; -1 = the calling thread's current device */
    int32_t host_threads;     /* staging threads (pageable text -> pinned chunks -> H2D; packing runs on the device); 0 = auto */
    uint64_t table_capacity;  /* pass-1 table slots; 0 = auto (cardinality estimate on device) */
    uint32_t flags;           /* VDJGRAPH_FLAG_* */
    uint32_t partitions;      /* hash units (power of two <= 256: groups of the 256 minimizer buckets, each with its own
                                 slice of the tables); 0 = auto (table slice ~12 MB, L2-resident) */
    uint32_t rounds;          /* groups of hash units processed one after the other (power of two, rounds * devices
                                 <= 256): the run buffer and both tables hold one group at a time and the packed
                                 reads are streamed once per round -- for inputs whose working set does not fit HBM
                                 (BASELINE configs[4] on the finishing rank).  0 = auto: the smallest count whose
                                 working set fits the device (1 for everything up to configs[3] and for configs[4]'s
                                 per-GPU share).  Results do not depend on it */
    uint32_t reserved;        /* 0 */
} vdjgraph_params;

#define VDJGRAPH_FLAG_EXPORT_KEYS 1u /* also export the packed k-mer of every node (kmer_lo/kmer_hi) */
#define VDJGRAPH_FLAG_WIDE_TUPLES 2u /* force the 24-byte form of the per-window tuples the slow-path queues hold (normally chosen when k
                                        and the input size need it) */
#define VDJGRAPH_FLAG_HASHMAP_LAYOUT 4u /* also export the layout of the reference's `nodes` map (hm_buckets, hm_slots): which
                                           bucket of dense_hash_map<const char*, node*, my_hash, eqstr> every node occupies after
                                           build_graph2's inserts (:305), so that the glue can load the map in one pass instead of
                                           replaying the inserts.  Computed on the device (MurmurHash64A, sparsehash's probing and
                                           doubling); see glue/vdjgraph_glue.inc */

/*
 * The graph the reference holds after build_graph2 (:1408), as structure-of-arrays indexed by
 * node creation rank: node i is the node whose reference `id` is i+1 (new_node :190-204).
 *
 * Positions ("stamps"): records are numbered in processing order, primary buffer first, then
 * secondary; w = read_length - kmer_size + 1; window o of record r has stamp r*w + o.
 * node->kmer of the reference points at base o of record r (first_pos = r*w + o).
 *
 * Arrays are owned by the context and stay valid until the next vdjgraph_stage/build or
 * vdjgraph_destroy on it.  They live in page-locked host memory.
 */
typedef struct vdjgraph_result {
    uint64_t n_nodes;
    const uint64_t *first_pos; /* [n] stamp of the first pass-2 occurrence -> node->kmer, node->kmer_seq[0] */
    const uint16_t *frequency; /* [n] node->frequency: min(#N-free occurrences, 32765) (:199, :261-265) */
    const uint8_t *out_deg;    /* [n] length of node->toNodes (0..4) */
    const uint8_t *in_deg;     /* [n] length of node->fromNodes (0..4) */
    const uint32_t *out_succ;  /* [n*4] toNodes in the reference's list order (head first = last first-seen, :223-229); node index, 0xFFFFFFFF = none */
    const uint32_t *in_pred;   /* [n*4] fromNodes in the reference's list order (:231-236) */
    const uint64_t *kmer_lo;   /* [n] packed k-mer, 2 bits/base, A=0 C=1 G=2 T=3, base j at bits 2j..2j+1; NULL unless VDJGRAPH_FLAG_EXPORT_KEYS */
    const uint64_t *kmer_hi;   /* [n] bits 64.. of the same (bases 32..) */

    /* counters the reference prints (:406-407, :449-450, :1394) and the roofline's h (SURVEY 8d) */
    uint64_t n_records;        /* primary + secondary */
    uint64_t n_windows;        /* n_records * w : the unit of "k-mers/s" */
    uint64_t n_gated;          /* windows passing include_kmer (:240-259) */
    uint64_t n_pre_total;      /* "Pre Num nodes": distinct gated k-mers */
    uint64_t n_pre;            /* "pre nodes after pruning" (= n_nodes) */
    uint64_t n_hits;           /* pass-2 windows whose k-mer survived (uncapped) */
    uint64_t n_slow1, n_slow2; /* diagnostics: windows that took the slow (queued) path of pass 1 / pass 2 */
    uint64_t n_hits_ungated;   /* pass-2 hits among the windows that failed the quality gate (only those add to node->frequency in pass 2) */

    /* timings of the last build, milliseconds */
    float ms_stage;            /* H2D of the text + device packing (wall clock) */
    float ms_device;           /* whole vdjgraph_run, CUDA events on the build stream (includes the
                                  two small counter read-backs that size the tables) */
    /* per-kernel CUDA-event times: k_count (window histogram + cardinality estimate), k_scatter,
     * pass-1 table init, k_pass1, k_prune, survivor-table init+insert, k_pass2,
     * export (collect + sort + rank + edges) */
    float ms_estimate, ms_scatter, ms_init1, ms_pass1, ms_prune, ms_table2, ms_pass2, ms_export;
    float ms_fetch;            /* D2H of the result (wall clock) */
    uint64_t table1_slots, table2_slots; /* capacities used */
    uint32_t partitions, tuple_bytes;    /* hash units used; bytes of a queued per-window tuple (16 or 24) */
    uint32_t rounds, reserved;           /* super-partition rounds used */
    uint64_t h2d_bytes, d2h_bytes;       /* bytes moved by stage / fetch */
    uint64_t kernel_launches;            /* our kernels launched by the last run (CUB's sort passes not counted) */
    uint64_t n_runs;                     /* run records ("super-k-mers") this device shipped: stretches of consecutive
                                            N-free windows that share a minimizer bucket, one 32-byte record each */
    uint32_t run_bytes, reserved2;       /* bytes per run record */
    /* VDJGRAPH_FLAG_HASHMAP_LAYOUT: the reference's `nodes` map after the block, bucket by bucket */
    uint64_t hm_buckets;                 /* its bucket count (0 without the flag) */
    const uint32_t *hm_slots;            /* [hm_buckets] node in the bucket (creation rank), 0xFFFFFFFF = empty bucket */
    float ms_hashmap, reserved3;         /* device time of the layout, inside ms_device */
} vdjgraph_result;

/* Pruned pass-1 table (debug/parity export; unordered): what pre_nodes holds after :1393. */
typedef struct vdjgraph_pre_table {
    uint64_t n;
    const uint64_t *kmer_lo, *kmer_hi; /* packed k-mer as above */
    const uint16_t *frequency;         /* pre_node.frequency: min(#gated occurrences, 32765) */
} vdjgraph_pre_table;

typedef struct vdjgraph_ctx vdjgraph_ctx;

int vdjgraph_version(void);
/* Message of the last failure on the calling thread ("" if none). */
const char *vdjgraph_last_error(void);

/* Create a context (CUDA context, streams, staging threads' pinned buffers are created lazily
 * and reused across builds).  Replaces nothing in the reference; it has no equivalent. */
int vdjgraph_create(const vdjgraph_params *params, vdjgraph_ctx **out);
void vdjgraph_destroy(vdjgraph_ctx *ctx);
/* Change --k/--mf/--mq/read_length between builds without recreating the context. */
int vdjgraph_set_params(vdjgraph_ctx *ctx, const vdjgraph_params *params);

/*
 * One call = the whole block :1381-1415 on HOST buffers in the reference's record format
 * (bam_read.c:206-244): record = strand char + read_length bases + read_length phred+33
 * qualities, 2*read_length+1 bytes, no separators.  `primary` = assemble()'s `input`,
 * `secondary` = `unaligned_input`; record counts replace the reference's strlen()/record_len
 * (:370-374).  Buffers are borrowed for the call.  Equivalent to stage + run + fetch.
 */
int vdjgraph_build(vdjgraph_ctx *ctx, const char *primary, size_t n_primary_records,
                   const char *secondary, size_t n_secondary_records, vdjgraph_result *out);

/*
 * Page-locked memory for the two record buffers.  The reference allocates them with calloc
 * (bam_read.c:386-388); a caller that takes them from vdjgraph_host_alloc instead (or registers
 * its own allocation once) lets vdjgraph_stage/vdjgraph_build DMA straight out of them: no host
 * copy into bounce buffers, no host threads, and N ranks on one host do not compete for cores and
 * memory bandwidth.  Pageable buffers keep working (bounced through page-locked chunks by
 * `host_threads` workers).  Unlike calloc's, the memory is not zero-filled: a caller that relies
 * on the terminating NUL writes it itself.
 */
int vdjgraph_host_alloc(size_t bytes, void **out);
int vdjgraph_host_free(void *ptr);
int vdjgraph_host_register(void *ptr, size_t bytes);
int vdjgraph_host_unregister(void *ptr);

/* The same in three steps, so that callers (and bench.py) can keep a read set resident in HBM. */
/* 1. staging: the text goes to the device in pinned chunks and is packed there (2-bit bases, gate/N
 *    masks, quality bytes); validates strand bytes and the alphabet */
int vdjgraph_stage(vdjgraph_ctx *ctx, const char *primary, size_t n_primary_records,
                   const char *secondary, size_t n_secondary_records);
/*
 * SURVEY 8f-3 (reads handed over where they are extracted): the same staging from FORWARD reads
 * only.  The reference's buffers hold every read twice, the read and its reverse complement
 * (add_to_buffer, bam_read.c:206-244; rc/reverse :130-145), so half of the text is redundant.  A
 * producer that also appends each read once, in the same record format ('0' + bases + qualities),
 * to a compact buffer passes that one here: text record i becomes packed records 2i (the read) and
 * 2i+1 (its reverse complement, derived on the device), i.e. exactly the read set of the doubled
 * buffers, at half the host-to-device bytes.  Stamps and node positions keep referring to the
 * doubled numbering, so the glue's text buffers stay the ones node->kmer points into.
 * n_*_reads count forward reads (= half the records of the corresponding doubled buffer).
 */
int vdjgraph_stage_forward(vdjgraph_ctx *ctx, const char *primary_reads, size_t n_primary_reads,
                           const char *secondary_reads, size_t n_secondary_reads);
int vdjgraph_build_forward(vdjgraph_ctx *ctx, const char *primary_reads, size_t n_primary_reads,
                           const char *secondary_reads, size_t n_secondary_reads, vdjgraph_result *out);
/* 2. device only: estimate -> pass 1 -> prune -> pass 2 -> rank/edges/compaction; blocks until done */
int vdjgraph_run(vdjgraph_ctx *ctx);
/* 3. copy the compacted graph to host memory */
int vdjgraph_fetch(vdjgraph_ctx *ctx, vdjgraph_result *out);

/*
 * Sharded build over G = 1, 2, 4 or 8 devices (SURVEY 8e): records are split into contiguous
 * ranges, k-mers are owner-computed (every hash unit belongs to one device; units are dealt to devices
 * largest-first from the all-gathered window counts, identically on every rank).  The caller
 * runs one context per device (one process per GPU, or several contexts in one process) and
 * drives the phases below on all of them, exchanging three small host messages in between.  The
 * bulk exchange is done by the scatter kernel itself, which writes every run into the owner's
 * buffer through peer-mapped memory (NVLink).  The finish is distributed as well: every device
 * ranks and links ITS survivors (three steps; a neighbour k-mer is looked up in the table of the
 * device that owns it, a peer load) and stores the finished node rows into rank 0's result buffer
 * (peer stores); between the steps the devices meet at a barrier kept in peer memory
 * (device_barrier = 1: the three steps are queued back to back, no host round trip) or on the
 * host (device_barrier = 0: every step returns with its stream synchronised and the caller holds
 * a barrier of its own before the next; needed when several ranks share one process and thread).
 * Results are identical to the one-device build.
 *
 *   all ranks : vdjgraph_shard_stage -> vdjgraph_shard_count                      -> hist, hll
 *   exchange  : all-gather hist and record counts, element-wise max of hll
 *   all ranks : vdjgraph_shard_plan  -> vdjgraph_shard_buffers                    -> device pointers
 *   exchange  : all-gather the pointers (vdjgraph_ipc_export/open across processes)
 *   all ranks : vdjgraph_shard_set_peers ; BARRIER ; vdjgraph_shard_release_retired ; vdjgraph_shard_scatter ; BARRIER
 *   all ranks : vdjgraph_shard_passes                                             -> survivor count
 *   (more than one round, vdjgraph_shard_rounds() > 1: BARRIER ; vdjgraph_shard_scatter ; BARRIER ;
 *    vdjgraph_shard_passes again, once per further round: the scatter of round r+1 overwrites the run
 *    buffers that the owners' passes of round r read)
 *   exchange  : all-gather the survivor counts
 *   all ranks : vdjgraph_shard_gather_plan ; everybody's GATHER pointer to everybody (only when one
 *               had to grow: vdjgraph_shard_finish_bytes tells) ; set_peers ; BARRIER
 *   all ranks : vdjgraph_shard_finish_step 0, 1, 2  (device_barrier = 0: BARRIER after each)
 *   all ranks : vdjgraph_shard_finish ; BARRIER ; rank 0: vdjgraph_fetch
 */
#define VDJGRAPH_SHARD_NBUF 6       /* bases, valid, qual, strand, runs, gather (= the finish's exchange buffer) */
#define VDJGRAPH_SHARD_HIST 768     /* uint64 per rank: [runs | gated windows | N-free windows][256 minimizer buckets] */
#define VDJGRAPH_SHARD_HLL 32768    /* bytes: 128 HyperLogLog registers per minimizer bucket */

typedef struct vdjgraph_shard_info {
    uint32_t n_ranks, rank;
    uint64_t record_base;      /* global number of this rank's first record (primary ++ secondary of all ranks, in rank order) */
    uint64_t total_records;    /* over all ranks */
} vdjgraph_shard_info;

int vdjgraph_shard_stage(vdjgraph_ctx *ctx, const char *primary, size_t n_primary_records,
                         const char *secondary, size_t n_secondary_records, const vdjgraph_shard_info *info);
/* the same from forward reads only (vdjgraph_stage_forward): n_*_reads count reads; record_base,
 * total_records and the record counts of vdjgraph_shard_plan stay in the doubled numbering */
int vdjgraph_shard_stage_forward(vdjgraph_ctx *ctx, const char *primary_reads, size_t n_primary_reads,
                                 const char *secondary_reads, size_t n_secondary_reads, const vdjgraph_shard_info *info);
int vdjgraph_shard_count(vdjgraph_ctx *ctx, uint64_t *hist /*[VDJGRAPH_SHARD_HIST]*/, uint8_t *hll /*[VDJGRAPH_SHARD_HLL]*/);
int vdjgraph_shard_plan(vdjgraph_ctx *ctx, const uint64_t *hist_all /*[n_ranks][VDJGRAPH_SHARD_HIST]*/,
                        const uint8_t *hll_merged /*[VDJGRAPH_SHARD_HLL], element-wise max over the ranks*/,
                        const uint64_t *record_counts /*[n_ranks]*/);
/* rounds the plan settled on (every rank computes the same number from the all-gathered inputs);
 * negative status before vdjgraph_shard_plan */
int vdjgraph_shard_rounds(vdjgraph_ctx *ctx);
int vdjgraph_shard_buffers(vdjgraph_ctx *ctx, void **ptrs /*[NBUF]*/, size_t *bytes /*[NBUF] or NULL*/);
int vdjgraph_shard_set_peers(vdjgraph_ctx *ctx, void *const *ptrs /*[n_ranks][NBUF]; this rank's row is ignored*/);
int vdjgraph_shard_scatter(vdjgraph_ctx *ctx);
int vdjgraph_shard_passes(vdjgraph_ctx *ctx, uint64_t *n_survivors /* of this rank, all rounds so far */);
int vdjgraph_shard_gather_plan(vdjgraph_ctx *ctx, const uint64_t *survivors_all /*[n_ranks]*/);
/* bytes of rank `rank`'s GATHER buffer that vdjgraph_shard_gather_plan will ask for (a function of the
 * survivor counts and of the build flags, which are the same on every rank: every rank can tell which
 * buffers have to grow, i.e. which handles travel again) */
int vdjgraph_shard_finish_bytes(vdjgraph_ctx *ctx, const uint64_t *survivors_all /*[n_ranks]*/, uint32_t rank, size_t *bytes);
/* step 0: own survivor table + sorted stamps; 1: creation ranks; 2: edge lists, node rows to rank 0 */
int vdjgraph_shard_finish_step(vdjgraph_ctx *ctx, int step, int device_barrier);
/* every rank: waits for its stream, checks its counters; rank 0 also unpacks the rows into the result */
int vdjgraph_shard_finish(vdjgraph_ctx *ctx);
/* Peers may keep their mappings across builds.  A buffer that had to grow is replaced, not freed;
 * call this after a barrier that follows vdjgraph_shard_set_peers to free the replaced ones. */
int vdjgraph_shard_release_retired(vdjgraph_ctx *ctx);
/* peer mapping helpers: CUDA IPC handles (64 opaque bytes) between processes, peer access within one */
int vdjgraph_ipc_export(const void *device_ptr, unsigned char *handle64);
int vdjgraph_ipc_open(const unsigned char *handle64, void **device_ptr);
int vdjgraph_ipc_close(void *device_ptr);
int vdjgraph_enable_peer_access(int device, int peer_device);

/*
 * The same sharded build as ONE call, for a caller that is a single process (V'DJer is): one context
 * per entry of `devices` (1, 2, 4 or 8 CUDA device ordinals; peer access between them is enabled),
 * and inside vdjgraph_multi_build one host thread per device walks the phases above, meeting the
 * others at thread barriers (and, between the steps of the finish, at the barriers the devices keep
 * in peer memory).  Records are split into contiguous, even-sized ranges in rank order; stamps and
 * node positions are those of the one-device build on the same buffers, and so is the result, which
 * lands on devices[0] and is fetched from there.  `params->device` is ignored.  The same device may be
 * named more than once (tests on one GPU).  _forward: the buffers hold forward reads only
 * (vdjgraph_build_forward).  vdjgraph_multi_stats: counters of one rank's share.
 */
typedef struct vdjgraph_multi vdjgraph_multi;
int vdjgraph_multi_create(const vdjgraph_params *params, const int *devices, uint32_t n_devices, vdjgraph_multi **out);
void vdjgraph_multi_destroy(vdjgraph_multi *m);
int vdjgraph_multi_build(vdjgraph_multi *m, const char *primary, size_t n_primary_records,
                         const char *secondary, size_t n_secondary_records, vdjgraph_result *out);
int vdjgraph_multi_build_forward(vdjgraph_multi *m, const char *primary_reads, size_t n_primary_reads,
                                 const char *secondary_reads, size_t n_secondary_reads, vdjgraph_result *out);
int vdjgraph_multi_stats(vdjgraph_multi *m, uint32_t rank, vdjgraph_result *out);

/* Counters and timings of the last run without copying the graph (array pointers are NULL). */
int vdjgraph_stats(vdjgraph_ctx *ctx, vdjgraph_result *out);

/* Parity/debug: the pruned pass-1 table of the last run. */
int vdjgraph_fetch_pre_table(vdjgraph_ctx *ctx, vdjgraph_pre_table *out);

/*
 * Look sequences up in the graph of the last finished vdjgraph_run / vdjgraph_build / _forward on this
 * context: which node is the k-mer of every window, and where along a sequence does the graph break.
 * The lookups run on the device against the graph's own survivor table.
 *
 * Query i is seqs[offsets[i] .. offsets[i+1]); offsets must not decrease (offsets may be NULL when
 * n_queries is 0).  Its windows are the k-mers starting at bytes 0 .. len-k; a query shorter than k has
 * none.  The alphabet is the staging alphabet: an N ends the windows over it, as in a read, and any
 * other byte outside ACGT (lower case included) fails the call with VDJGRAPH_ERR_BASE.  n_windows must
 * be the exact window count, sum over queries of max(0, len - k + 1), or the call fails with
 * VDJGRAPH_ERR_PARAM.  On any failure node_of_window is not written.
 *
 * VDJGRAPH_ERR_STATE: no run has finished since the context was created or since the last
 * vdjgraph_stage* / vdjgraph_set_params / vdjgraph_shard_stage* or a failed call, or the last build ran
 * the sharded phases over more than one rank (each rank's table holds its own share only).
 * Synchronous, on the context's stream; the graph and what vdjgraph_fetch returns are unchanged.
 */
typedef struct vdjgraph_query_stats {
    uint64_t n_queries, n_windows;   /* windows = sum over queries of max(0, len - k + 1) */
    uint64_t n_found;                /* windows whose k-mer is a node */
    uint64_t h2d_bytes, d2h_bytes;
    float ms_kernels;                /* CUDA events around the query kernels */
    float ms_total;                  /* wall clock of the call */
} vdjgraph_query_stats;

/* node (creation rank, = reference id - 1) of every k-mer window of every query, in query order;
 * 0xFFFFFFFF where the window holds an N or its k-mer is not a node */
int vdjgraph_query(vdjgraph_ctx *ctx, const char *seqs, const uint64_t *offsets /*[n_queries+1]*/,
                   size_t n_queries, uint32_t *node_of_window, size_t n_windows,
                   vdjgraph_query_stats *stats /* may be NULL */);

#ifdef __cplusplus
}
#endif
#endif
