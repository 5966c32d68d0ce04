/*
 * vdjgraph.cu -- host side of libvdjgraph.so: C ABI (include/vdjgraph.h), read staging,
 * kernel orchestration and result export.  Device code is in kernels.cuh.
 *
 * Replaces the scoped block assembler2_vdj.c:1381-1415 of the reference
 * (build_pre_graph x2 -> prune_pre_graph -> build_graph2 x2).  There is no CPU fallback: every
 * entry point fails with VDJGRAPH_ERR_CUDA when no sm_100a device is usable.
 */
#include "kernels.cuh"
#include "../../include/vdjgraph.h"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace vdjg;

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CK(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(VDJGRAPH_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                      \
    } while (0)

/* performance knobs, overridable from the environment for tuning runs (results never depend on them) */
double env_double(const char *name, double dflt) {
    const char *v = getenv(name);
    return v && *v ? atof(v) : dflt;
}

double wall_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

/* DevBuf and PinBuf own their allocation: it is freed when they are destroyed.  They move (a growing
 * std::vector<StageWorker> moves its workers' buffers) but do not copy, which would free twice. */
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    /* buffers that other devices map (sharded build) are not freed when they grow: peers may still
     * have the old allocation mapped.  It is parked here until vdjgraph_shard_release_retired(). */
    bool exported = false;
    std::vector<void *> retired;
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap), exported(o.exported), retired(std::move(o.retired)) { o.p = nullptr; o.cap = 0; }
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) { if (exported) retired.push_back(p); else cudaFree(p); }
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 16 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(VDJGRAPH_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        }
        cap = want;
        return 0;
    }
    /* grow to `bytes`, keeping the first `keep` bytes (survivor records accumulate over the rounds) */
    int ensure_keep(size_t bytes, size_t keep, cudaStream_t s) {
        if (bytes <= cap) return 0;
        void *old = p;
        const size_t old_cap = cap;
        const bool was_exported = exported;
        p = nullptr; cap = 0; exported = false;
        int rc = ensure(bytes + bytes / 4);
        exported = was_exported;
        if (rc) { p = old; cap = old_cap; return rc; }   /* the old buffer and its contents stay */
        if (old && keep) {
            cudaError_t e = cudaMemcpyAsync(p, old, keep, cudaMemcpyDeviceToDevice, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
            if (e != cudaSuccess) { cudaFree(old); return fail(VDJGRAPH_ERR_CUDA, "copy into the grown buffer failed: %s", cudaGetErrorString(e)); }
        }
        if (old) { if (exported) retired.push_back(old); else cudaFree(old); }
        return 0;
    }
    void release_retired() { for (void *q : retired) cudaFree(q); retired.clear(); }
    void release() { release_retired(); if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    PinBuf() = default;
    PinBuf(PinBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    PinBuf(const PinBuf &) = delete;
    PinBuf &operator=(const PinBuf &) = delete;
    ~PinBuf() { release(); }
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 16 + 256;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(VDJGRAPH_ERR_NOMEM, "cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(e));
        }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

/* one staging worker: a stream, two page-locked chunk buffers (double buffering) and the two
 * device chunk buffers their text lands in (the text is never held on the device as a whole:
 * k_pack turns a chunk into packed reads right behind its copy, on the same stream) */
struct StageWorker {
    cudaStream_t stream = nullptr;
    PinBuf buf[2];
    DevBuf dbuf[2];
    cudaEvent_t done[2] = { nullptr, nullptr };   /* recorded behind the chunk that buffer b holds */
    bool busy[2] = { false, false };
};

/* the nodes' k-mers are exported: asked for, or hashed by the hash-map layout */
bool want_keys(uint32_t flags) { return flags & (VDJGRAPH_FLAG_EXPORT_KEYS | VDJGRAPH_FLAG_HASHMAP_LAYOUT); }

/* The graph's node arrays on the device (k_export / k_unpack_* write them) and their page-locked host
 * mirrors (vdjgraph_fetch).  kmer_lo and kmer_hi are last: they exist only when keys are wanted. */
struct NodeArrays {
    enum { FIRST_POS, FREQUENCY, OUT_DEG, IN_DEG, OUT_SUCC, IN_PRED, KMER_LO, KMER_HI, N };
    static constexpr size_t elem_bytes[N] = { 8, 2, 1, 1, 16, 16, 8, 8 };
    DevBuf d[N];
    PinBuf h[N];
    static int count(bool keys) { return keys ? N : KMER_LO; }
    int ensure(uint64_t n, bool keys) {
        for (int i = 0; i < count(keys); i++)
            if (int rc = d[i].ensure(std::max<uint64_t>(n, 1) * elem_bytes[i])) return rc;
        return 0;
    }
    /* k_export / k_unpack_* arguments that write into these arrays (the other fields zero) */
    ExportArgs export_args(bool keys) const {
        ExportArgs a{};
        a.first_pos = d[FIRST_POS].as<u64>(); a.frequency = d[FREQUENCY].as<u16>();
        a.out_deg = d[OUT_DEG].as<u8>(); a.in_deg = d[IN_DEG].as<u8>();
        a.out_succ = d[OUT_SUCC].as<u32>(); a.in_pred = d[IN_PRED].as<u32>();
        a.kmer_lo = keys ? d[KMER_LO].as<u64>() : nullptr; a.kmer_hi = keys ? d[KMER_HI].as<u64>() : nullptr;
        return a;
    }
    /* the first n nodes to the host mirrors (s is synchronised) and r's arrays pointed at them; adds the bytes copied to `bytes` */
    int fetch(uint64_t n, bool keys, cudaStream_t s, vdjgraph_result &r, uint64_t &bytes) {
        for (int i = 0; i < count(keys); i++)
            if (int rc = h[i].ensure(std::max<uint64_t>(n, 1) * elem_bytes[i])) return rc;
        if (n) {
            for (int i = 0; i < count(keys); i++) {
                CK(cudaMemcpyAsync(h[i].p, d[i].p, n * elem_bytes[i], cudaMemcpyDeviceToHost, s));
                bytes += n * elem_bytes[i];
            }
            CK(cudaStreamSynchronize(s));
        }
        r.first_pos = h[FIRST_POS].as<uint64_t>(); r.frequency = h[FREQUENCY].as<uint16_t>();
        r.out_deg = h[OUT_DEG].as<uint8_t>(); r.in_deg = h[IN_DEG].as<uint8_t>();
        r.out_succ = h[OUT_SUCC].as<uint32_t>(); r.in_pred = h[IN_PRED].as<uint32_t>();
        r.kmer_lo = keys ? h[KMER_LO].as<uint64_t>() : nullptr; r.kmer_hi = keys ? h[KMER_HI].as<uint64_t>() : nullptr;
        return 0;
    }
};

/* Events recorded on the context's stream, named after the point of the build they mark */
enum Ev {
    EV_BUILD,                                /* start of the build's device time (run_plan) */
    EV_SCATTER, EV_SCATTER_END,              /* around k_scatter */
    EV_INIT1, EV_PASS1, EV_PRUNE, EV_PRUNE_END,   /* before k_init_table1, k_pass1, k_prune; after k_prune */
    EV_TABLE2, EV_PASS2, EV_PASS2_END,       /* before the survivor table, before k_pass2, after k_pass2 */
    /* the finish, from its start to its end; a distributed finish records after each of its three steps and
     * after the barrier behind it (the order is the order on the stream) */
    EV_FINISH, EV_STEP0, EV_STEP0_MET, EV_STEP1, EV_STEP1_MET, EV_STEP2, EV_STEP2_MET, EV_FINISH_END,
    EV_HASHMAP, EV_HASHMAP_END,              /* around the hash-map layout */
    EV_COUNT
};
static_assert(EV_FINISH_END == EV_FINISH + 7, "the finish's events are consecutive");

/* The finished graph's survivor table as vdjgraph_query looks k-mers up in it: the table k_export read
 * (one round: d_t2 with the per-unit slices of the plan; several rounds: the merged flat table d_t2m)
 * and the slicing and geometry it was read with.  Recorded by a one-device finish, current while the context
 * is queryable(); table is null when the graph has no nodes. */
struct GraphView {
    const Slot2 *table = nullptr;
    uint64_t cap = 0, n_nodes = 0;
    Part pt{};
    Geom g{};
};

/* vdjgraph_query's buffers: chunks of the batch go through page-locked text and offset buffers, are
 * copied on their own stream (h2d) and answered on the context's stream, double buffered: the next
 * chunk's copy overlaps the current chunk's kernels.  The answers of the whole batch stay on the device
 * until every chunk has passed the alphabet check. */
struct QueryBufs {
    cudaStream_t h2d = nullptr;
    cudaEvent_t copied[2] = {}, k_begin[2] = {}, k_end[2] = {};
    bool pending[2] = { false, false };  /* chunk kernels queued behind k_end[b] whose time is not yet added */
    PinBuf text[2], meta[2], ctr;
    DevBuf d_text[2], d_meta[2], d_bases, d_nmask, d_out, d_ctr;
    int init() {
        if (h2d) return 0;
        CK(cudaStreamCreateWithFlags(&h2d, cudaStreamNonBlocking));
        for (int b = 0; b < 2; b++) {
            CK(cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming));
            CK(cudaEventCreate(&k_begin[b]));
            CK(cudaEventCreate(&k_end[b]));
        }
        return 0;
    }
    void destroy() {
        for (int b = 0; b < 2; b++)
            for (cudaEvent_t e : { copied[b], k_begin[b], k_end[b] }) if (e) cudaEventDestroy(e);
        if (h2d) cudaStreamDestroy(h2d);
        h2d = nullptr;
    }
};

constexpr uint32_t STAGE_CHUNK = 32768; /* records per staging chunk (3.3 MB of text at L=50) */
constexpr size_t QUERY_CHUNK = 32ull << 20;   /* bytes of query text per chunk (VDJGRAPH_QUERY_CHUNK_KB overrides) */
constexpr double MERGED_SLOTS_PER_NODE = 2.0;   /* slots of the merged survivor table per node (load 0.5) */
constexpr uint64_t REF_MAX_NODES = 900000000ull; /* MAX_NODES, assembler2_vdj.c:73 */
constexpr uint64_t SLICE_BYTES = 12ull << 20;   /* table-1 bytes one hash unit addresses: L2-resident (12 MB measured better than 24 and 6) */

} // namespace

/* buffers other devices of a sharded build read or write (vdjgraph_shard_buffers order) */
enum { BUF_BASES = 0, BUF_VALID, BUF_QUAL, BUF_STRAND, BUF_TUPLES, BUF_GATHER, NBUF };
static_assert(NBUF == VDJGRAPH_SHARD_NBUF, "header and library disagree");

/* What a context may do next (include/vdjgraph.h, "Call order"): the last step of staging or of a build it has completed.
 * FINISH_STEPn: step n of the finish has been queued or done; FINISH_PLANNED and the three steps are consecutive. */
enum class State { EMPTY, STAGED, COUNTED, PLANNED, PEERS_SET, SCATTERED, PASSES_DONE, FINISH_PLANNED, FINISH_STEP0, FINISH_STEP1,
                   FINISH_STEP2, FINISHED };

struct Shard {
    int G = 1, rank = 0;
    uint64_t rec_base[MAX_DEV + 1] = {};
    uint64_t total_records = 0;
    /* the plan (identical on every rank: a function of the all-gathered histograms only) */
    int NU = 1, ushift = HIST_BITS;               /* hash units = minimizer buckets >> ushift */
    std::vector<uint64_t> runs, gated, valid;     /* [G][NU] per source device and unit */
    std::vector<double> est;                      /* [NU] distinct gated k-mers (HyperLogLog) */
    std::vector<int> owner, round_of;             /* [NU] device and round that process the unit */
    std::vector<UnitTab> utab;                    /* [NU] this device's table slices of the current round */
    double load1 = 0;                             /* target load of table 1 (VDJGRAPH_LOAD1) */
    double slot_scale = 1.0;                      /* table-1 slots per estimated k-mer, relative to the default */
    bool ignore_hint = false;                     /* the caller's table_capacity turned out too small */
    void *peer[MAX_DEV][NBUF] = {};
    uint64_t n_runs_own = 0, n_gated_own = 0;     /* what this device receives in the current round */
    uint64_t n_gated_src = 0, n_valid_src = 0;    /* windows this device produces */
    double est_distinct = 0;
    uint64_t surv_all[MAX_DEV] = {}, surv_off[MAX_DEV + 1] = {};
    /* rounds: groups of hash units processed one after the other (runs and tables of one round in HBM at a time) */
    int S = 1, rnd = 0;
    uint64_t surv_done = 0;                       /* survivor records of the finished rounds (in d_rec) */
    float acc[6] = {};                            /* scatter, init1, pass1, prune, table2, pass2 ms summed over the rounds */
    bool merged() const { return G > 1 || S > 1; } /* the finish builds a table over survivor RECORDS */
    uint64_t bar_seq = 0;                         /* device barriers of this build so far (k_peer_barrier) */
};

struct vdjgraph_ctx {
    vdjgraph_params prm;
    int device = 0;
    int sm_count = 0;
    size_t mem_total = 0;
    Geom g;
    uint64_t R_pad = 0;
    bool any_strand1 = false;
    State state = State::EMPTY;   /* here, not in Shard: staging resets Shard */
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[EV_COUNT] = {};
    std::vector<StageWorker> workers;

    DevBuf d_bad, d_bases, d_good, d_valid, d_hiq, d_qual, d_strand;
    PinBuf h_bad;
    DevBuf d_t1, d_log, d_t2, d_hll, d_ctr, d_hist, d_cursor, d_tuples, d_utab;
    DevBuf d_keys[2], d_vals[2], d_cub;
    NodeArrays nodes;
    DevBuf d_pre_klo, d_pre_khi, d_pre_freq, d_pre_n;
    PinBuf h_ctr, h_hll, h_hist, h_cursor, h_utab;
    float ms_count = 0;
    size_t count_smem = 0;
    int count_bps = 1;
    Part part;
    PinBuf h_pre_klo, h_pre_khi, h_pre_freq, h_pre_n;

    DevBuf d_tbase, d_rec, d_gather, d_t2m, d_gid, d_owner;
    DevBuf d_hm_hash, d_hm_probe, d_hm_prev, d_hm_owner, d_hm_slots, d_hm_flag;
    PinBuf h_hm_slots, h_hm_flag;
    PinBuf h_tbase;
    Shard sh;

    /* the buffers that peers of a sharded build map, in BUF_* order */
    std::array<DevBuf *, NBUF> peer_bufs() { return { &d_bases, &d_valid, &d_qual, &d_strand, &d_tuples, &d_gather }; }

    uint64_t cap1 = 0, cap2 = 0;
    uint32_t log_cap = 0;
    Counters ctr;
    vdjgraph_result res;

    GraphView view;   /* what vdjgraph_query looks k-mers up in */
    QueryBufs q;

    /* what a finished build leaves: the graph (on rank 0 of a sharded build) and a table that holds all of it (one rank) */
    bool has_graph() const { return state == State::FINISHED && (sh.G == 1 || sh.rank == 0); }
    bool queryable() const { return state == State::FINISHED && sh.G == 1; }
    bool rounds_left() const { return sh.rnd + 1 < sh.S; }
};

namespace {

int check_params(const vdjgraph_params *p) {
    if (!p) return fail(VDJGRAPH_ERR_PARAM, "params is NULL");
    if (p->read_length < 1 || p->read_length > 255)
        return fail(VDJGRAPH_ERR_PARAM, "read_length %d outside 1..255 (bam_read.c:208 stores reads in char[256])", p->read_length);
    if (p->kmer_size < 1 || p->kmer_size > 50)
        return fail(VDJGRAPH_ERR_PARAM, "kmer_size %d outside 1..50 (MAX_KMER_LEN, assembler2_vdj.c:70)", p->kmer_size);
    if (p->kmer_size > p->read_length)
        return fail(VDJGRAPH_ERR_PARAM, "kmer_size %d > read_length %d", p->kmer_size, p->read_length);
    if (p->rounds & (p->rounds - 1) || p->rounds > (1u << HIST_BITS))
        return fail(VDJGRAPH_ERR_PARAM, "rounds %u is not a power of two <= %u", p->rounds, 1u << HIST_BITS);
    return 0;
}

/* Geometry of the packed reads and of the streaming kernels' tiles: a record's w windows are cut
 * into `segs` thread segments of at most SEG_MAX windows, a block tile holds THREADS / segs records. */
void make_geom(vdjgraph_ctx *c, uint64_t R) {
    Geom &g = c->g;
    g.L = c->prm.read_length;
    g.k = c->prm.kmer_size;
    g.w = g.L - g.k + 1;
    g.nb = (g.L + 31) / 32;
    g.nm = (g.L + 63) / 64;
    g.R = R;
    int bits = 2 * g.k;
    g.kmask_lo = bits >= 64 ? ~0ull : ((1ull << bits) - 1);
    g.kmask_hi = bits > 64 ? ((1ull << (bits - 64)) - 1) : 0ull;
    g.kones = (1ull << g.k) - 1;
    g.m = std::min(g.k, MINI_M);
    g.span = g.k - g.m + 1;
    g.mmask = (1u << (2 * g.m)) - 1u;
    g.run_max = std::min(RUN_MAX, 64 - g.k);
    /* ceil(2^64 / w); for w = 1 the quotient 2^64 does not fit: 2^64 - 1 gives stamp - 1 for stamp > 0, so w = 1 keeps the plain division (see k_pass1) */
    g.w_magic = g.w > 1 ? (~0ull / (uint64_t)g.w) + 1 : 0;
    g.segs = (g.w + SEG_MAX - 1) / SEG_MAX;
    g.seg = (g.w + g.segs - 1) / g.segs;
    uint32_t tr = (uint32_t)THREADS / (uint32_t)g.segs;
    tr &= ~1u;   /* even: TMA bulk copies need 16-byte sizes and addresses */
    g.tile_rec = tr;
    g.n_tiles = (R + tr - 1) / tr;
    /* runs a tile is expected to hold: one per segment plus one per minimizer change (every (span+1)/2
     * windows on random sequence), with a third on top; tiles with more spill to single stores */
    const double expect = (double)tr * g.segs + (double)tr * g.w * 2.0 / (g.span + 1);
    g.stage_runs = (uint32_t)std::min<double>(2048.0, std::max(256.0, std::ceil(expect * 1.35 / 128.0) * 128.0));
    c->R_pad = g.n_tiles * g.tile_rec;
}

int ensure_workers(vdjgraph_ctx *c, int n) {
    if ((int)c->workers.size() >= n) return 0;
    size_t old = c->workers.size();
    c->workers.resize(n);
    for (size_t i = old; i < c->workers.size(); i++) {
        CK(cudaStreamCreateWithFlags(&c->workers[i].stream, cudaStreamNonBlocking));
        for (cudaEvent_t &e : c->workers[i].done) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    return 0;
}

/* Staging = raw text to the device + k_pack there.  The host only moves bytes: worker threads
 * copy chunks of the caller's (pageable) buffers into their page-locked buffers and queue the
 * H2D copy and the chunk's k_pack launch on their own stream, double buffered. */
/* text records per staging chunk: a multiple of the streaming kernels' tile, so that a chunk's packed
 * records are whole tiles and k_count can run on them right behind k_pack */
uint64_t chunk_records(const vdjgraph_ctx *c, uint32_t base) {
    const uint64_t tr = c->g.tile_rec;
    return std::max<uint64_t>(tr, (base / tr) * tr);
}
int count_chunk(vdjgraph_ctx *c, cudaStream_t s, uint64_t rec_lo, uint64_t rec_hi, bool last);

/* queues k_pack of text records [r_lo, r_hi) of R, whose text is at `text` on the device, and k_count of
 * the packed records behind it on stream s */
int pack_chunk(vdjgraph_ctx *c, cudaStream_t s, const unsigned char *text, uint64_t r_lo, uint64_t r_hi, uint64_t R, uint32_t fwd) {
    const uint64_t n = r_hi - r_lo;
    PackArgs pa;
    pa.text = text; pa.r0 = r_lo << fwd; pa.n = n; pa.fwd_only = fwd;
    pa.bases = c->d_bases.as<u64>(); pa.good = c->d_good.as<u64>(); pa.valid = c->d_valid.as<u64>();
    pa.hiq = c->d_hiq.as<u64>();
    pa.qual = c->d_qual.as<u8>(); pa.strand = c->d_strand.as<u8>();
    pa.bad = c->d_bad.as<u64>();
    const int grid = (int)std::min<uint64_t>((n + WARPS - 1) / WARPS, (uint64_t)c->sm_count * 8);
    k_pack<<<grid, THREADS, 0, s>>>(pa, c->g);
    CK(cudaGetLastError());
    return count_chunk(c, s, r_lo << fwd, r_hi << fwd, r_hi == R);
}

struct StageShared {
    vdjgraph_ctx *c;
    const char *primary, *secondary;
    uint64_t np, R;      /* TEXT records: primary, primary + secondary */
    uint32_t fwd;        /* 1: forward reads only, every text record packs into two records */
    std::atomic<uint64_t> next_chunk{0};
    std::atomic<int> status{0};
};

void stage_worker(StageShared *s, int wi) {
    vdjgraph_ctx *c = s->c;
    StageWorker &w = c->workers[wi];
    const Geom &g = c->g;
    if (cudaSetDevice(c->device) != cudaSuccess) { s->status = VDJGRAPH_ERR_CUDA; return; }
    const size_t rec_len = (size_t)2 * g.L + 1;
    const uint64_t CH = chunk_records(c, STAGE_CHUNK);
    const uint64_t n_chunks = (s->R + CH - 1) / CH;
    int b = 0;
    for (;;) {
        uint64_t ch = s->next_chunk.fetch_add(1);
        if (ch >= n_chunks || s->status.load() != 0) break;
        const uint64_t r_lo = ch * CH, r_hi = std::min<uint64_t>(s->R, r_lo + CH);
        const uint64_t n = r_hi - r_lo;
        if (w.busy[b]) { cudaEventSynchronize(w.done[b]); w.busy[b] = false; }
        char *pin = w.buf[b].as<char>();
        /* records [r_lo, r_hi) of primary ++ secondary */
        const uint64_t np_part = r_lo < s->np ? std::min<uint64_t>(r_hi, s->np) - r_lo : 0;
        if (np_part) memcpy(pin, s->primary + r_lo * rec_len, np_part * rec_len);
        if (np_part < n) memcpy(pin + np_part * rec_len, s->secondary + (r_lo + np_part - s->np) * rec_len, (n - np_part) * rec_len);
        /* stream order keeps the chunk's previous k_pack ahead of this copy */
        unsigned char *dst = w.dbuf[b].as<unsigned char>();
        cudaError_t e = cudaMemcpyAsync(dst, pin, n * rec_len, cudaMemcpyHostToDevice, w.stream);
        if (e == cudaSuccess && pack_chunk(c, w.stream, dst, r_lo, r_hi, s->R, s->fwd)) e = cudaErrorUnknown;
        if (e == cudaSuccess) e = cudaEventRecord(w.done[b], w.stream);
        if (e != cudaSuccess) { s->status = VDJGRAPH_ERR_CUDA; break; }
        w.busy[b] = true;
        b ^= 1;
    }
    if (cudaStreamSynchronize(w.stream) != cudaSuccess) s->status = VDJGRAPH_ERR_CUDA;
    w.busy[0] = w.busy[1] = false;
}

/* is [p, p+bytes) page-locked memory this process registered or allocated through CUDA? */
bool is_page_locked(const void *p, size_t bytes) {
    if (!p || !bytes) return true;
    cudaPointerAttributes a0, a1;
    if (cudaPointerGetAttributes(&a0, p) != cudaSuccess ||
        cudaPointerGetAttributes(&a1, (const char *)p + bytes - 1) != cudaSuccess) { cudaGetLastError(); return false; }
    return a0.type == cudaMemoryTypeHost && a1.type == cudaMemoryTypeHost;
}

constexpr uint32_t DIRECT_CHUNK = 8 * STAGE_CHUNK;   /* records per DMA when the caller's buffers are page-locked */
constexpr int DIRECT_STREAMS = 4;

/* Staging from page-locked caller buffers (vdjgraph_host_alloc / vdjgraph_host_register): no host
 * copy at all.  One thread queues, chunk by chunk on a few streams, the DMA from the caller's
 * memory into that stream's device chunk buffer and the chunk's k_pack behind it: copies of one
 * stream overlap the packing of the others, the host cores stay idle (which is what lets N ranks of
 * one host stage at the same time). */
int stage_direct(vdjgraph_ctx *c, const char *primary, uint64_t np, const char *secondary, uint64_t R, uint32_t fwd) {
    const Geom &g = c->g;
    const size_t rec_len = (size_t)2 * g.L + 1;
    int rc;
    if ((rc = ensure_workers(c, DIRECT_STREAMS))) return rc;
    for (int i = 0; i < DIRECT_STREAMS; i++)
        if ((rc = c->workers[i].dbuf[0].ensure((size_t)chunk_records(c, DIRECT_CHUNK) * rec_len))) return rc;
    const uint64_t CH = chunk_records(c, DIRECT_CHUNK);
    const uint64_t n_chunks = (R + CH - 1) / CH;
    for (uint64_t ch = 0; ch < n_chunks; ch++) {
        StageWorker &w = c->workers[ch % DIRECT_STREAMS];
        const uint64_t r_lo = ch * CH, r_hi = std::min<uint64_t>(R, r_lo + CH), n = r_hi - r_lo;
        unsigned char *dst = w.dbuf[0].as<unsigned char>();   /* stream order: its previous k_pack has read it */
        const uint64_t np_part = r_lo < np ? std::min<uint64_t>(r_hi, np) - r_lo : 0;
        if (np_part) CK(cudaMemcpyAsync(dst, primary + r_lo * rec_len, np_part * rec_len, cudaMemcpyHostToDevice, w.stream));
        if (np_part < n)
            CK(cudaMemcpyAsync(dst + np_part * rec_len, secondary + (r_lo + np_part - np) * rec_len, (n - np_part) * rec_len,
                               cudaMemcpyHostToDevice, w.stream));
        if ((rc = pack_chunk(c, w.stream, dst, r_lo, r_hi, R, fwd))) return rc;
    }
    for (int i = 0; i < DIRECT_STREAMS; i++) CK(cudaStreamSynchronize(c->workers[i].stream));
    return 0;
}

/* Staging from pageable caller buffers: up to host_threads workers (stage_worker) */
int stage_pageable(vdjgraph_ctx *c, const char *primary, uint64_t np, const char *secondary, uint64_t R, uint32_t fwd) {
    const size_t rec_len = (size_t)2 * c->g.L + 1;
    const uint64_t CH = chunk_records(c, STAGE_CHUNK);
    const uint64_t n_chunks = (R + CH - 1) / CH;
    int nt = c->prm.host_threads > 0 ? c->prm.host_threads : (int)std::min(16u, std::thread::hardware_concurrency());
    nt = std::max(1, std::min<int>(nt, 64));
    nt = (int)std::min<uint64_t>((uint64_t)nt, n_chunks);
    int rc;
    if ((rc = ensure_workers(c, nt))) return rc;
    for (int i = 0; i < nt; i++)
        for (int b = 0; b < 2; b++)
            if ((rc = c->workers[i].buf[b].ensure((size_t)CH * rec_len)) ||
                (rc = c->workers[i].dbuf[b].ensure((size_t)CH * rec_len))) return rc;
    StageShared sh;
    sh.c = c; sh.primary = primary; sh.secondary = secondary; sh.np = np; sh.R = R; sh.fwd = fwd;
    std::vector<std::thread> th;
    for (int i = 1; i < nt; i++) th.emplace_back(stage_worker, &sh, i);
    stage_worker(&sh, 0);
    for (auto &t : th) t.join();
    if (int st = sh.status.load()) {
        cudaError_t e = cudaGetLastError();
        return fail(st, "staging failed: %s", cudaGetErrorString(e));
    }
    return 0;
}

/* resident blocks per SM of a persistent kernel; `cap` > 0 limits them and shrinks the shared-memory
 * carve-out to what that many blocks need, so that the rest of the SM's 256 KB stays L1 (the table
 * passes live on L1 hits of the hot k-mers' slots) */
int blocks_per_sm(const void *kernel, size_t smem, int cap = 0) {
    int n = 0;
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, THREADS, smem);
    n = std::max(1, n);
    if (cap > 0) {
        n = std::min(n, cap);
        const double need = (double)n * (double)(smem + 1024) / (228.0 * 1024.0) * 100.0;
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)std::min(100.0, std::ceil(need)));
    }
    return n;
}

/* HyperLogLog estimate from one bucket's BHLL byte registers */
double hll_estimate(const uint8_t *reg) {
    const int M = BHLL;
    double sum = 0;
    int zeros = 0;
    /* 2^-r from a table: the plan adds up 32768 registers per build */
    static const std::array<double, 256> pow2neg = [] { std::array<double, 256> t{}; for (int r = 0; r < 256; r++) t[r] = std::ldexp(1.0, -r); return t; }();
    for (int i = 0; i < M; i++) { sum += pow2neg[reg[i]]; zeros += reg[i] == 0; }
    double alpha = 0.7213 / (1.0 + 1.079 / M);
    double e = alpha * M * (double)M / sum;
    if (e <= 2.5 * M && zeros) e = M * std::log((double)M / zeros);
    return e;
}

int bits_for(uint64_t v) { int b = 1; while (b < 64 && (v >> b)) b++; return b; }

} // namespace

/* ========================================================================================== */
/* C ABI                                                                                       */
/* ========================================================================================== */
extern "C" int vdjgraph_version(void) { return VDJGRAPH_ABI_VERSION; }
extern "C" const char *vdjgraph_last_error(void) { return g_err.c_str(); }

extern "C" int vdjgraph_create(const vdjgraph_params *params, vdjgraph_ctx **out) {
    if (!out) return fail(VDJGRAPH_ERR_PARAM, "out is NULL");
    *out = nullptr;
    int rc = check_params(params);
    if (rc) return rc;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(VDJGRAPH_ERR_CUDA, "no CUDA device (%s); libvdjgraph has no CPU path", cudaGetErrorString(e));
    }
    int dev = params->device;
    if (dev < 0) CK(cudaGetDevice(&dev));
    if (dev >= ndev) return fail(VDJGRAPH_ERR_PARAM, "device %d out of range (have %d)", dev, ndev);
    CK(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10)
        return fail(VDJGRAPH_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", dev, prop.major, prop.minor);
    vdjgraph_ctx *c = new (std::nothrow) vdjgraph_ctx();
    if (!c) return fail(VDJGRAPH_ERR_NOMEM, "out of host memory");
    c->prm = *params;
    c->device = dev;
    c->sm_count = prop.multiProcessorCount;
    c->mem_total = prop.totalGlobalMem;
    memset(&c->res, 0, sizeof(c->res));
    memset(&c->ctr, 0, sizeof(c->ctr));
    e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    for (cudaEvent_t &ev : c->ev) if (e == cudaSuccess) e = cudaEventCreate(&ev);
    if (e != cudaSuccess) { vdjgraph_destroy(c); return fail(VDJGRAPH_ERR_CUDA, "stream/event creation failed: %s", cudaGetErrorString(e)); }
    *out = c;
    return 0;
}

extern "C" void vdjgraph_destroy(vdjgraph_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto &w : c->workers) {
        for (cudaEvent_t ev : w.done) if (ev) cudaEventDestroy(ev);
        if (w.stream) cudaStreamDestroy(w.stream);
    }
    for (cudaEvent_t ev : c->ev) if (ev) cudaEventDestroy(ev);
    c->q.destroy();
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;   /* the buffers free themselves */
}

extern "C" int vdjgraph_set_params(vdjgraph_ctx *c, const vdjgraph_params *params) {
    if (!c) return fail(VDJGRAPH_ERR_PARAM, "ctx is NULL");
    int rc = check_params(params);
    if (rc) return rc;
    bool regeom = params->read_length != c->prm.read_length || params->kmer_size != c->prm.kmer_size;
    int dev = c->prm.device;
    c->prm = *params;
    c->prm.device = dev;
    /* the build is dropped; the staged records stay unless their geometry changed */
    c->state = regeom ? State::EMPTY : std::min(c->state, State::STAGED);
    return 0;
}

namespace { int count_begin(vdjgraph_ctx *c); int count_end(vdjgraph_ctx *c); }

/* np / ns count TEXT records.  fwd = 0: the reference's buffers (every read followed by its reverse
 * complement).  fwd = 1: forward reads only; the packed read set is the same as if the reverse
 * complements had been in the text (packed record 2i = read i, 2i+1 = derived by k_pack).
 * info: this rank's share of a sharded build (vdjgraph_shard_stage*), NULL for one device. */
static int stage_impl(vdjgraph_ctx *c, const char *primary, size_t np, const char *secondary, size_t ns, uint32_t fwd,
                      const vdjgraph_shard_info *info) {
    if (!c) return fail(VDJGRAPH_ERR_PARAM, "ctx is NULL");
    if ((np && !primary) || (ns && !secondary)) return fail(VDJGRAPH_ERR_PARAM, "NULL record buffer");
    c->state = State::EMPTY;   /* until the records are staged */
    const uint64_t Rt = (uint64_t)np + (uint64_t)ns;   /* text records */
    const uint64_t R = Rt << fwd;                      /* packed records */
    if (info) {
        const uint32_t G = info->n_ranks;
        if (G < 1 || G > (uint32_t)MAX_DEV || (G & (G - 1)) || info->rank >= G)
            return fail(VDJGRAPH_ERR_PARAM, "n_ranks %u must be 1, 2, 4 or 8 and rank %u below it", G, info->rank);
        if (info->record_base + R > info->total_records)
            return fail(VDJGRAPH_ERR_PARAM, "record range exceeds total_records");
        if (info->total_records > 0xFFFFFFFEull)
            return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "%llu records exceed the 2^32-2 record limit", (unsigned long long)info->total_records);
        for (DevBuf *b : c->peer_bufs()) b->exported = G > 1;
    }
    CK(cudaSetDevice(c->device));
    if (R > 0xFFFFFFFEull) return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "%llu records exceed the 2^32-2 record limit", (unsigned long long)R);
    double t0 = wall_ms();
    make_geom(c, R);
    const Geom &g = c->g;
    int rc;
    if ((rc = c->d_bases.ensure(std::max<size_t>(16, c->R_pad * g.nb * 8)))) return rc;
    if ((rc = c->d_good.ensure(std::max<size_t>(16, c->R_pad * g.nm * 8)))) return rc;
    if ((rc = c->d_valid.ensure(std::max<size_t>(16, c->R_pad * g.nm * 8)))) return rc;
    if ((rc = c->d_hiq.ensure(std::max<size_t>(16, c->R_pad * g.nm * 8)))) return rc;
    if ((rc = c->d_qual.ensure(std::max<size_t>(16, c->R_pad * (size_t)g.L)))) return rc;
    if ((rc = c->d_strand.ensure(std::max<size_t>(16, c->R_pad)))) return rc;
    /* zero the padding records of the last tile: no window of theirs is gated or N-free */
    if (c->R_pad > R) {
        CK(cudaMemsetAsync(c->d_bases.as<uint64_t>() + R * g.nb, 0, (c->R_pad - R) * g.nb * 8, c->stream));
        CK(cudaMemsetAsync(c->d_good.as<uint64_t>() + R * g.nm, 0, (c->R_pad - R) * g.nm * 8, c->stream));
        CK(cudaMemsetAsync(c->d_valid.as<uint64_t>() + R * g.nm, 0, (c->R_pad - R) * g.nm * 8, c->stream));
        CK(cudaMemsetAsync(c->d_hiq.as<uint64_t>() + R * g.nm, 0, (c->R_pad - R) * g.nm * 8, c->stream));
    }
    uint64_t h2d = 0;
    c->any_strand1 = false;
    if ((rc = count_begin(c))) return rc;
    if (R) {
        const size_t rec_len = (size_t)2 * g.L + 1;
        if ((rc = c->d_bad.ensure(3 * sizeof(uint64_t))) || (rc = c->h_bad.ensure(3 * sizeof(uint64_t)))) return rc;
        uint64_t *hb = c->h_bad.as<uint64_t>();
        hb[0] = hb[1] = ~0ull; hb[2] = 0;
        CK(cudaMemcpyAsync(c->d_bad.p, hb, 3 * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));   /* padding memsets, flags and zeroed counters are in place before the workers start */
        const bool direct = is_page_locked(primary, np * rec_len) && is_page_locked(secondary, ns * rec_len);
        if ((rc = direct ? stage_direct(c, primary, np, secondary, Rt, fwd) : stage_pageable(c, primary, np, secondary, Rt, fwd))) return rc;
        CK(cudaMemcpyAsync(hb, c->d_bad.p, 3 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        if (hb[0] != ~0ull)
            return fail(VDJGRAPH_ERR_STRAND, "record %llu does not start with '0' or '1' (assembler2_vdj.c:383-391)", (unsigned long long)hb[0]);
        if (hb[1] != ~0ull)
            return fail(VDJGRAPH_ERR_BASE, "record %llu holds a base outside ACGTN", (unsigned long long)hb[1]);
        c->any_strand1 = hb[2] != 0;
        h2d = Rt * rec_len;
    }
    CK(cudaStreamSynchronize(c->stream));
    /* per-bucket window / run counts and cardinality registers of the packed reads (k_count ran chunk
     * by chunk behind the packing): the build's plan needs nothing else */
    if ((rc = count_end(c))) return rc;
    memset(&c->res, 0, sizeof(c->res));
    c->res.ms_stage = (float)(wall_ms() - t0);
    c->res.h2d_bytes = h2d;
    c->res.n_records = R;
    c->res.n_windows = R * (uint64_t)g.w;
    c->sh = Shard();
    Shard &sh = c->sh;
    if (info) { sh.G = (int)info->n_ranks; sh.rank = (int)info->rank; }
    sh.total_records = info ? info->total_records : R;
    sh.rec_base[sh.rank] = info ? info->record_base : 0;   /* the other ranks' arrive with vdjgraph_shard_plan */
    sh.rec_base[sh.rank + 1] = sh.rec_base[sh.rank] + R;
    c->state = State::STAGED;
    return 0;
}

extern "C" int vdjgraph_stage(vdjgraph_ctx *c, const char *primary, size_t np, const char *secondary, size_t ns) {
    return stage_impl(c, primary, np, secondary, ns, 0, nullptr);
}
extern "C" int vdjgraph_stage_forward(vdjgraph_ctx *c, const char *primary_reads, size_t np, const char *secondary_reads, size_t ns) {
    return stage_impl(c, primary_reads, np, secondary_reads, ns, 1, nullptr);
}

/* ========================================================================================== */
/* The build, in phases.  One device: vdjgraph_run() runs them back to back.  Sharded over G     */
/* devices (one process per GPU, or G contexts in one process): the caller interleaves them with */
/* three tiny host exchanges (window histograms, peer pointers, survivor counts); the only bulk  */
/* data movement between devices is done by the kernels themselves through peer-mapped memory:  */
/* k_scatter writes each run straight into the buffer of the device that owns its hash unit.     */
/* ========================================================================================== */
namespace {

const char *const STATE_NAMES[] = { "EMPTY", "STAGED", "COUNTED", "PLANNED", "PEERS_SET", "SCATTERED", "PASSES_DONE",
                                    "FINISH_PLANNED", "FINISH_STEP0", "FINISH_STEP1", "FINISH_STEP2", "FINISHED" };
static_assert(sizeof(STATE_NAMES) / sizeof(*STATE_NAMES) == (size_t)State::FINISHED + 1, "a name per state");

/* sets of states: bit(s), and from(s) = s .. FINISHED */
constexpr unsigned bit(State s) { return 1u << (int)s; }
constexpr unsigned from(State s) { return 2 * bit(State::FINISHED) - bit(s); }

/* The check of call order: `call` is accepted when the context is in a state of `accepted` and the caller gives no `refusal`
 * (a reason the sequence rules it out in that state).  A refused call fails with VDJGRAPH_ERR_STATE and changes nothing. */
int check_state(const vdjgraph_ctx *c, const char *call, unsigned accepted, const char *refusal = nullptr) {
    if (!c) return fail(VDJGRAPH_ERR_PARAM, "ctx is NULL");
    if (accepted & bit(c->state)) return refusal ? fail(VDJGRAPH_ERR_STATE, "%s", refusal) : 0;
    std::string names;
    for (int s = 0; s <= (int)State::FINISHED; s++)
        if (accepted & bit(State(s))) { names += names.empty() ? "" : ", "; names += STATE_NAMES[s]; }
    return fail(VDJGRAPH_ERR_STATE, "%s in state %s; it is accepted in %s", call, STATE_NAMES[(int)c->state], names.c_str());
}

/* the device counters to the host (c->h_ctr), the stream synchronised */
int read_counters(vdjgraph_ctx *c) {
    CK(cudaMemcpyAsync(c->h_ctr.p, c->d_ctr.p, sizeof(Counters), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

/* adds this round's kernel times (scatter, init1, pass1, prune, table2, pass2) into sh.acc; every event
 * of the round has completed */
void add_kernel_times(vdjgraph_ctx *c) {
    static const Ev span[6][2] = { { EV_SCATTER, EV_SCATTER_END }, { EV_INIT1, EV_PASS1 }, { EV_PASS1, EV_PRUNE },
                                   { EV_PRUNE, EV_PRUNE_END }, { EV_TABLE2, EV_PASS2 }, { EV_PASS2, EV_PASS2_END } };
    for (int i = 0; i < 6; i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev[span[i][0]], c->ev[span[i][1]]);
        c->sh.acc[i] += ms;
    }
}

/* this device's times once the finish has completed: per kernel, summed over the rounds (k_count ran with
 * the staging: ms_estimate), the hash-map layout and the finish */
void take_times(vdjgraph_ctx *c) {
    vdjgraph_result &res = c->res;
    const float *acc = c->sh.acc;
    res.ms_scatter = acc[0]; res.ms_init1 = acc[1]; res.ms_pass1 = acc[2]; res.ms_prune = acc[3]; res.ms_table2 = acc[4]; res.ms_pass2 = acc[5];
    if (res.hm_buckets) cudaEventElapsedTime(&res.ms_hashmap, c->ev[EV_HASHMAP], c->ev[EV_HASHMAP_END]);
    cudaEventElapsedTime(&res.ms_export, c->ev[EV_FINISH], c->ev[EV_FINISH_END]);
}

constexpr size_t HIST_WORDS = 3 * NBUCKET;          /* runs | gated windows | N-free windows, per bucket */
constexpr size_t HLL_BYTES = (size_t)NBUCKET * BHLL;
static_assert(HIST_WORDS == VDJGRAPH_SHARD_HIST && HLL_BYTES == VDJGRAPH_SHARD_HLL, "header and library disagree");

/* K0, part of staging (its results depend on the reads and on k only): runs / gated / N-free windows
 * per minimizer bucket + per-bucket HyperLogLog of the gated k-mers.  count_begin zeroes the device
 * accumulators, count_chunk queues k_count on the whole tiles of one staging chunk behind the chunk's
 * k_pack (same stream; a fraction of the SMs: it hides behind the next chunk's copy), count_end
 * brings the totals to the host: h_hist, h_hll. */
int count_begin(vdjgraph_ctx *c) {
    cudaStream_t s = c->stream;
    int rc;
    if ((rc = c->d_ctr.ensure(sizeof(Counters)))) return rc;
    if ((rc = c->d_hll.ensure(HLL_BYTES))) return rc;
    if ((rc = c->d_hist.ensure(HIST_WORDS * sizeof(uint64_t)))) return rc;
    if ((rc = c->d_cursor.ensure(2 * NBUCKET * sizeof(uint64_t)))) return rc;
    if ((rc = c->d_tbase.ensure(NBUCKET * sizeof(void *)))) return rc;
    if ((rc = c->d_utab.ensure(NBUCKET * sizeof(UnitTab)))) return rc;
    if ((rc = c->h_ctr.ensure(sizeof(Counters)))) return rc;
    if ((rc = c->h_hll.ensure(HLL_BYTES))) return rc;
    if ((rc = c->h_hist.ensure(HIST_WORDS * sizeof(uint64_t)))) return rc;
    if ((rc = c->h_cursor.ensure(2 * NBUCKET * sizeof(uint64_t)))) return rc;
    if ((rc = c->h_tbase.ensure(NBUCKET * sizeof(void *)))) return rc;
    if ((rc = c->h_utab.ensure(NBUCKET * sizeof(UnitTab)))) return rc;
    CK(cudaMemsetAsync(c->d_hll.p, 0, HLL_BYTES, s));
    CK(cudaMemsetAsync(c->d_hist.p, 0, HIST_WORDS * sizeof(uint64_t), s));
    c->count_smem = count_head_bytes() + scratch_bytes(c->g) + sbk_bytes(c->g) + block_tile_bytes(c->g, 2);
    c->count_bps = blocks_per_sm((const void *)k_count, c->count_smem);
    return 0;
}
/* packed records [rec_lo, rec_hi) have just been packed on stream s; rec_lo is a tile boundary, and so
 * is rec_hi unless this is the last chunk (then the zeroed padding records complete the last tile) */
int count_chunk(vdjgraph_ctx *c, cudaStream_t s, uint64_t rec_lo, uint64_t rec_hi, bool last) {
    const Geom &g = c->g;
    const uint64_t tile0 = rec_lo / g.tile_rec, tile1 = last ? g.n_tiles : rec_hi / g.tile_rec;
    if (tile1 <= tile0) return 0;
    /* a quarter of the machine per chunk: several chunks are in flight on their streams */
    const int grid = (int)std::min<uint64_t>(tile1 - tile0, std::max(1, c->sm_count * c->count_bps / 4));
    k_count<<<grid, THREADS, c->count_smem, s>>>(c->d_bases.as<u64>(), c->d_good.as<u64>(), c->d_valid.as<u64>(), g, tile0, tile1,
                                                  c->d_hll.as<u32>(), c->d_hist.as<u64>());
    CK(cudaGetLastError());
    return 0;
}
int count_end(vdjgraph_ctx *c) {
    cudaStream_t s = c->stream;
    CK(cudaMemcpyAsync(c->h_hist.p, c->d_hist.p, HIST_WORDS * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(c->h_hll.p, c->d_hll.p, HLL_BYTES, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}

void reset_run_stats(vdjgraph_ctx *c) {
    memset(&c->ctr, 0, sizeof(c->ctr));
    vdjgraph_result &res = c->res;
    res.n_nodes = 0; res.n_gated = res.n_pre_total = res.n_pre = res.n_hits = res.n_slow1 = res.n_slow2 = res.n_hits_ungated = 0;
    res.ms_device = res.ms_scatter = res.ms_init1 = res.ms_pass1 = res.ms_prune = 0;
    res.ms_table2 = res.ms_pass2 = res.ms_export = 0;
    res.ms_estimate = c->ms_count;
    res.table1_slots = res.table2_slots = 0;
    res.partitions = 0; res.tuple_bytes = 0;
    res.kernel_launches = 0;
}

/* table-1 slots of hash unit u (all of it, whichever device / round holds it) */
uint64_t unit_slots1(const Shard &sh, const vdjgraph_params &prm, int u) {
    /* 1.15: the per-unit HyperLogLog has a relative error of ~9 % / sqrt(buckets per unit); a slice that
     * comes out too small only runs at a higher load (probing continues into the next slice) */
    double slots = sh.est[u] * 1.15 / sh.load1 * sh.slot_scale;
    if (prm.table_capacity && !sh.ignore_hint) slots = (double)prm.table_capacity * (sh.est[u] + 1.0) / (sh.est_distinct + sh.NU) * sh.slot_scale;
    return (uint64_t)slots + 64;
}

/* Partitioning, devices, rounds, table sizes, this device's run buffer.
 * hist_all: [G][3][NBUCKET] per-bucket counts of every device; hll: registers merged (max) over the devices.
 * Everything here is a function of the all-gathered inputs only, so every rank of a sharded build
 * arrives at the same plan. */
int run_plan(vdjgraph_ctx *c, const uint64_t *hist_all, const uint8_t *hll) {
    Shard &sh = c->sh;
    const Geom &g = c->g;
    const int G = sh.G;
    reset_run_stats(c);
    CK(cudaEventRecord(c->ev[EV_BUILD], c->stream));
    /* per-bucket estimates of the distinct gated k-mers */
    double est_b[NBUCKET];
    sh.est_distinct = 0;
    for (int b = 0; b < NBUCKET; b++) {
        uint64_t gb = 0;
        for (int d = 0; d < G; d++) gb += hist_all[((size_t)d * 3 + 1) * NBUCKET + b];
        est_b[b] = gb ? std::min<double>(hll_estimate(hll + (size_t)b * BHLL), (double)gb) : 0.0;
        sh.est_distinct += est_b[b];
    }
    const double load1 = sh.load1 = std::min(0.9, std::max(0.05, env_double("VDJGRAPH_LOAD1", 0.5)));
    const uint64_t cap1_all = c->prm.table_capacity ? c->prm.table_capacity : (uint64_t)(sh.est_distinct * 1.15 / load1) + 1024;

    Part pt;
    memset(&pt, 0, sizeof(pt));
    int pbits0 = 0;
    if (c->prm.partitions) {
        while ((1u << pbits0) < c->prm.partitions && pbits0 < HIST_BITS) pbits0++;
    } else {
        /* table-1 slices of about SLICE_BYTES so that the slice being updated is L2-resident */
        const uint64_t slice_bytes = (uint64_t)(env_double("VDJGRAPH_SLICE_MB", (double)(SLICE_BYTES >> 20)) * 1048576.0);
        while (pbits0 < HIST_BITS && ((cap1_all * sizeof(Slot1)) >> pbits0) > slice_bytes) pbits0++;
    }
    pt.hb = std::max(0, 2 * g.k - 64);
    const int sbits = bits_for(sh.total_records * (uint64_t)g.w);
    /* narrow queue tuples need room for at least 4 read-fingerprint bits beside the stamp */
    pt.wide = (pt.hb + FLB + 4 + sbits > 64) || (c->prm.flags & VDJGRAPH_FLAG_WIDE_TUPLES) ? 1 : 0;
    pt.fb = std::min(RUN_FP_BITS, pt.wide ? 64 - pt.hb - FLB : 64 - pt.hb - FLB - sbits);
    /* test hook: fewer fingerprint bits force the exact read comparison on (almost) every k-mer */
    pt.fb = std::max(0, std::min(pt.fb, (int)env_double("VDJGRAPH_FP_BITS", 32.0)));
    pt.cshift = (u32)std::max(0, sbits - 8);
    pt.hot_t = (u32)env_double("VDJGRAPH_HOT_T", 1024);
    pt.hot_flush = (u32)std::max(1.0, env_double("VDJGRAPH_HOT_FLUSH", 3));
    pt.qflush1 = (u32)std::min<double>(QFLUSH1, std::max(1.0, env_double("VDJGRAPH_QFLUSH1", 32)));
    pt.qdense1 = (u32)std::min<double>(32, env_double("VDJGRAPH_QDENSE1", 0));
    pt.qflush2 = (u32)std::min<double>(QFLUSH, std::max(1.0, env_double("VDJGRAPH_QFLUSH2", 96)));
    pt.qdense2 = (u32)std::min<double>(32, env_double("VDJGRAPH_QDENSE2", QDENSE));

    /* Working set of one device with S rounds, against its memory: packed reads stay resident; runs,
     * both tables and the log hold one round; survivor records and the finishing device's merged
     * table, sort and export buffers hold the whole graph (~0.6 of the distinct k-mers survive on
     * repertoire data; an underestimate only costs an allocation error, and `rounds` can be set by
     * the caller). */
    int mqc = std::min(std::min(c->prm.min_base_quality, 254), QSUM_SAT);
    const int NBq = mqc > 0 ? (mqc + GATE_Q - 1) / GATE_Q : 0;
    uint64_t rec_max = 0;
    for (int d = 0; d < G; d++) rec_max = std::max(rec_max, sh.rec_base[d + 1] - sh.rec_base[d]);
    const double reads_bytes = (double)rec_max * ((double)g.nb * 8 + 3.0 * g.nm * 8 + g.L + 1);
    const double budget = env_double("VDJGRAPH_MEM_BUDGET_MB", 0.9 * (double)c->mem_total / 1048576.0) * 1048576.0;
    sh.slot_scale = 1.0; sh.ignore_hint = false;

    /* Layout for S rounds over NU units: units go to devices, largest first, each to the device with
     * the fewest N-free windows so far (minimizer buckets are far from equal: a few hold the constant
     * region's k-mers); a device's units go to its rounds the same way, by runs. */
    std::vector<uint64_t> tot_runs, tot_gated, tot_valid, load_dev, load_rnd, gated_rnd;
    std::vector<double> est_rnd;
    auto layout = [&](int S, int pbits) {
        const int NU = 1 << pbits, fold = NBUCKET / NU;
        sh.NU = NU; sh.ushift = HIST_BITS - pbits; sh.S = S;
        sh.runs.assign((size_t)G * NU, 0); sh.gated.assign((size_t)G * NU, 0); sh.valid.assign((size_t)G * NU, 0);
        sh.est.assign(NU, 0.0);
        tot_runs.assign(NU, 0); tot_gated.assign(NU, 0); tot_valid.assign(NU, 0);
        for (int b = 0; b < NBUCKET; b++) {
            const int u = b / fold;
            sh.est[u] += est_b[b];
            for (int d = 0; d < G; d++) {
                const uint64_t *h = hist_all + (size_t)d * HIST_WORDS;
                sh.runs[(size_t)d * NU + u] += h[b]; sh.gated[(size_t)d * NU + u] += h[NBUCKET + b]; sh.valid[(size_t)d * NU + u] += h[2 * NBUCKET + b];
                tot_runs[u] += h[b]; tot_gated[u] += h[NBUCKET + b]; tot_valid[u] += h[2 * NBUCKET + b];
            }
        }
        std::vector<int> order(NU);
        for (int u = 0; u < NU; u++) order[u] = u;
        sh.owner.assign(NU, 0); sh.round_of.assign(NU, 0);
        if (G > 1) {
            std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return tot_valid[x] > tot_valid[y]; });
            load_dev.assign(G, 0);
            for (int u : order) {
                int best = 0;
                for (int d = 1; d < G; d++) if (load_dev[d] < load_dev[best]) best = d;
                sh.owner[u] = best;
                load_dev[best] += tot_valid[u] + 1;   /* + 1: empty units spread out too */
            }
        }
        load_rnd.assign((size_t)G * S, 0); gated_rnd.assign((size_t)G * S, 0); est_rnd.assign((size_t)G * S, 0.0);
        for (int u = 0; u < NU; u++) order[u] = u;
        std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return tot_runs[x] > tot_runs[y]; });
        for (int u : order) {
            const int d = sh.owner[u];
            int best = 0;
            for (int r = 1; r < S; r++) if (load_rnd[(size_t)d * S + r] < load_rnd[(size_t)d * S + best]) best = r;
            sh.round_of[u] = best;
            load_rnd[(size_t)d * S + best] += tot_runs[u] + 1;
            gated_rnd[(size_t)d * S + best] += tot_gated[u];
            est_rnd[(size_t)d * S + best] += (double)unit_slots1(sh, c->prm, u);
        }
    };
    const bool free_tables = env_double("VDJGRAPH_FREE_TABLES_MB", -1.0) >= 0;
    auto working_set = [&]() {
        double worst = 0;
        /* survivors / distinct gated k-mers: 0.19 .. 0.42 on the BASELINE workloads */
        const double nodes = 0.45 * sh.est_distinct;
        const bool merged = G * sh.S > 1;
        for (size_t i = 0; i < load_rnd.size(); i++) {
            const double cap1_dev = est_rnd[i];
            const double tables = cap1_dev * sizeof(Slot1)
                                + std::min((double)gated_rnd[i], cap1_dev * load1 / 1.15 * 1.3) * NBq * 8.0
                                + nodes / ((double)G * sh.S) * 4.0 * sizeof(Slot2);
            /* the finish.  One device, several rounds: merged table over all survivor records, sort buffers,
             * result (with VDJGRAPH_FREE_TABLES_MB set, run_finish first frees the last round's tables, see
             * there).  Several devices (finish_layout): everybody's sorted stamps, a table and sort buffers for
             * the device's own share, and on the finishing device the node rows, their overflow list and the
             * result arrays of the whole graph. */
            const double finish = !merged ? nodes * 70.0
                                : G == 1 ? nodes * (sizeof(Slot2) + MERGED_SLOTS_PER_NODE * sizeof(Slot2) + 70.0)
                                         : nodes * (8.0 + ROW_WORDS * 8.0 + 16.0 + 60.0) + nodes / (double)G * (MERGED_SLOTS_PER_NODE * sizeof(Slot2) + 20.0);
            const double records = merged ? nodes * sizeof(Slot2) / (double)G : 0.0;
            const double ws = reads_bytes + (double)load_rnd[i] * RUN_WORDS * 8 + records + (merged && free_tables ? std::max(tables, finish) : tables + finish);
            worst = std::max(worst, ws);
        }
        return worst;
    };
    int gb = 0;
    while ((1 << gb) < G) gb++;
    int rb = 0;
    const int rb_max = HIST_BITS - gb;
    if (c->prm.rounds) {
        while ((1u << rb) < c->prm.rounds) rb++;
        if (rb > rb_max) return fail(VDJGRAPH_ERR_PARAM, "rounds %u x %d devices exceed %d hash units", c->prm.rounds, G, NBUCKET);
        layout(1 << rb, std::max(pbits0, gb + rb));   /* every (device, round) can own at least one unit */
    } else {
        for (;; rb++) {
            layout(1 << rb, std::max(pbits0, gb + rb));
            if (working_set() <= budget || rb == rb_max) break;
        }
    }
    sh.rnd = 0; sh.surv_done = 0;
    memset(sh.acc, 0, sizeof(sh.acc));
    pt.ushift = sh.ushift;
    pt.ut = c->d_utab.as<UnitTab>();
    c->part = pt;

    /* what this device produces, and the largest round it receives */
    sh.n_gated_src = sh.n_valid_src = 0;
    for (int u = 0; u < sh.NU; u++) { sh.n_gated_src += sh.gated[(size_t)sh.rank * sh.NU + u]; sh.n_valid_src += sh.valid[(size_t)sh.rank * sh.NU + u]; }
    uint64_t runs_max = 0;
    for (int r = 0; r < sh.S; r++) {
        uint64_t n = 0;
        for (int u = 0; u < sh.NU; u++) if (sh.owner[u] == sh.rank && sh.round_of[u] == r) n += tot_runs[u];
        runs_max = std::max(runs_max, n);
    }
    int rc;
    if ((rc = c->d_tuples.ensure(std::max<size_t>(32, runs_max * RUN_WORDS * 8)))) return rc;
    c->res.partitions = (uint32_t)sh.NU;
    c->res.tuple_bytes = (uint32_t)(pt.wide ? 24 : 16);
    c->res.rounds = (uint32_t)sh.S;
    c->res.n_gated = sh.n_gated_src;
    c->res.n_runs = 0;
    for (int u = 0; u < sh.NU; u++) c->res.n_runs += sh.runs[(size_t)sh.rank * sh.NU + u];
    c->res.run_bytes = (uint32_t)(RUN_WORDS * 8);
    return 0;
}

void own_buffers(vdjgraph_ctx *c, void **ptrs, size_t *bytes) {
    const auto b = c->peer_bufs();
    for (int i = 0; i < NBUF; i++) { ptrs[i] = b[i]->p; if (bytes) bytes[i] = b[i]->cap; }
}

/* K1: scatter this device's runs into the buffers of the units' owners */
int run_scatter(vdjgraph_ctx *c) {
    Shard &sh = c->sh;
    const Geom g = c->g;
    cudaStream_t s = c->stream;
    const int G = sh.G, NU = sh.NU;
    /* Region of unit u of THIS ROUND in its owner's buffer (units in unit order, each holding the runs
     * of device 0, 1, ... in that order), then this device's share of it; the units of other rounds
     * get no destination (the kernel skips their runs). */
    uint64_t *cur = c->h_cursor.as<uint64_t>(), *lim = cur + NBUCKET;
    void **tb = c->h_tbase.as<void *>();
    uint64_t off[MAX_DEV] = {};
    sh.n_runs_own = sh.n_gated_own = 0;
    for (int u = 0; u < NBUCKET; u++) { cur[u] = 0; lim[u] = 0; tb[u] = nullptr; }
    for (int u = 0; u < NU; u++) {
        if (sh.round_of[u] != sh.rnd) continue;
        const int o = sh.owner[u];
        uint64_t before = 0, total = 0, gated = 0;
        for (int d = 0; d < G; d++) {
            const uint64_t n = sh.runs[(size_t)d * NU + u];
            if (d < sh.rank) before += n;
            total += n;
            gated += sh.gated[(size_t)d * NU + u];
        }
        cur[u] = off[o] + before;
        lim[u] = cur[u] + sh.runs[(size_t)sh.rank * NU + u];
        tb[u] = sh.peer[o][BUF_TUPLES];
        if (!tb[u]) {
            if (lim[u] > cur[u]) return fail(VDJGRAPH_ERR_STATE, "no run buffer for device %d", o);
            tb[u] = sh.peer[sh.rank][BUF_TUPLES];   /* nothing goes there; the kernel only needs "this round" */
        }
        off[o] += total;
        if (o == sh.rank) { sh.n_runs_own += total; sh.n_gated_own += gated; }
    }
    c->part.n_runs = sh.n_runs_own;
    const Part pt = c->part;
    CK(cudaMemcpyAsync(c->d_cursor.p, cur, 2 * NBUCKET * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(c->d_tbase.p, tb, NBUCKET * sizeof(void *), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(c->d_ctr.p, 0, sizeof(Counters), s));
    CK(cudaEventRecord(c->ev[EV_SCATTER], s));
    if (g.R) {
        ScatterArgs as;
        as.bases = c->d_bases.as<u64>(); as.good = c->d_good.as<u64>(); as.valid = c->d_valid.as<u64>();
        as.hiq = c->d_hiq.as<u64>();
        as.tbase = c->d_tbase.as<u64 *>();
        as.cursor = c->d_cursor.as<u64>(); as.limit = c->d_cursor.as<u64>() + NBUCKET;
        as.rec_base = sh.rec_base[sh.rank];
        as.ctr = c->d_ctr.as<Counters>();
        const size_t smem_scatter = scatter_carve(nullptr, nullptr, g);
        const int grid_scatter = (int)std::min<uint64_t>(g.n_tiles, (uint64_t)c->sm_count * blocks_per_sm((const void *)k_scatter, smem_scatter));
        k_scatter<<<grid_scatter, THREADS, smem_scatter, s>>>(as, g, pt);
        c->res.kernel_launches++;
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(c->ev[EV_SCATTER_END], s));
    if (G > 1) CK(cudaStreamSynchronize(s));   /* the peers' runs are complete once every device got here */
    return 0;
}

Reads make_reads(vdjgraph_ctx *c) {
    Reads rd;
    memset(&rd, 0, sizeof(rd));
    const Shard &sh = c->sh;
    rd.n_dev = sh.G;
    rd.any_strand = c->any_strand1 || sh.G > 1;   /* peers may hold strand-'1' records */
    for (int d = 0; d < sh.G; d++) {
        rd.bases[d] = (const u64 *)sh.peer[d][BUF_BASES];
        rd.valid[d] = (const u64 *)sh.peer[d][BUF_VALID];
        rd.qual[d] = (const u8 *)sh.peer[d][BUF_QUAL];
        rd.strand[d] = (const u8 *)sh.peer[d][BUF_STRAND];
    }
    for (int d = 0; d <= sh.G; d++) rd.rec_base[d] = sh.rec_base[d];
    return rd;
}

/* K2..K4 on this device's hash units of the current round: pass 1, prune, survivor table, pass 2 */
int run_passes(vdjgraph_ctx *c) {
    Shard &sh = c->sh;
    const Geom g = c->g;
    Part pt = c->part;
    cudaStream_t s = c->stream;
    int rc;
    vdjgraph_result &res = c->res;
    Counters *d_ctr = c->d_ctr.as<Counters>();
    Counters *h_ctr = c->h_ctr.as<Counters>();
    const uint64_t n_runs = pt.n_runs, n_gated = sh.n_gated_own;
    const Reads rd = make_reads(c);
    const int grid_flat = c->sm_count * 8;

    /* pruning constants: T = min(mq, 214) after the <=254 clamp (:1514-1516, :356-360);
     * NB = ceil(T/20) = largest count whose quality sums can still fail */
    int mq = std::min(c->prm.min_base_quality, 254);
    int T = std::min(mq, QSUM_SAT);
    int NB = T > 0 ? (T + GATE_Q - 1) / GATE_Q : 0;

    const size_t feed_bytes = (size_t)WARPS * 32 * RUN_WORDS * 8;
    const size_t smem_q1 = WARPS * ((pt.wide ? WarpQueue<true, QCAP1>::bytes() : WarpQueue<false, QCAP1>::bytes()) + 2 * HOTC * sizeof(u32)) + feed_bytes;
    const size_t smem_q = WARPS * (pt.wide ? WarpQueue<true>::bytes() : WarpQueue<false>::bytes()) + feed_bytes;
    const uint64_t n_chunk = (n_runs + THREADS - 1) / THREADS;
    const int grid_p1 = (int)std::max<uint64_t>(1, std::min<uint64_t>(n_chunk,
                                                (uint64_t)c->sm_count * blocks_per_sm(pt.wide ? (const void *)k_pass1<true> : (const void *)k_pass1<false>, smem_q1, (int)env_double("VDJGRAPH_P1_BLOCKS", 0))));
    const int grid_p2 = (int)std::max<uint64_t>(1, std::min<uint64_t>(n_chunk,
                                                (uint64_t)c->sm_count * blocks_per_sm(pt.wide ? (const void *)k_pass2<true> : (const void *)k_pass2<false>, smem_q, (int)env_double("VDJGRAPH_P2_BLOCKS", PASS2_MIN_BLOCKS))));
    UnitTab *ut = c->h_utab.as<UnitTab>();
    sh.utab.assign(sh.NU, UnitTab{0, 0, 0, 0});

    /* ---- K2 + K3: pass 1 and prune (retried with a larger table / log if they overflow) ---- */
    uint64_t cap1 = 0;
    double log_scale = 1.0;
    for (int attempt = 0;; attempt++) {
        if (attempt > 6) return fail(VDJGRAPH_ERR_INTERNAL, "pass-1 table kept overflowing (capacity %llu)", (unsigned long long)cap1);
        /* table-1 slices of this device's units of this round, in unit order */
        cap1 = 0;
        for (int u = 0; u < sh.NU; u++) {
            if (sh.owner[u] != sh.rank || sh.round_of[u] != sh.rnd) continue;
            const uint64_t len = unit_slots1(sh, c->prm, u);
            if (cap1 + len > 0xFFFFFFF0ull) return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "pass-1 table would need more than 2^32 slots");
            sh.utab[u].off1 = (u32)cap1; sh.utab[u].len1 = (u32)len;
            cap1 += len;
        }
        cap1 = std::max<uint64_t>(cap1, 64);
        /* log: one block of NB stamps per distinct k-mer (<= table slots, <= gated windows), plus
         * one partially used chunk of blocks per warp */
        uint64_t warps = (uint64_t)grid_p1 * WARPS;
        /* (distinct k-mers, estimated: 1.3x the HyperLogLog figure of this device's units; an overrun doubles it) */
        double est_own = 0;
        for (int u = 0; u < sh.NU; u++) if (sh.owner[u] == sh.rank && sh.round_of[u] == sh.rnd) est_own += sh.est[u];
        const uint64_t distinct_cap = std::min<uint64_t>(std::min<uint64_t>(n_gated, cap1), (uint64_t)(est_own * 1.3) + 4096);
        uint64_t log_cap = (uint64_t)((double)distinct_cap * log_scale) + warps * LOG_CHUNK + LOG_CHUNK;
        if (NB == 0) log_cap = 1;
        if (log_cap > 0xFFFFFFF0ull) return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "occurrence log would need %llu blocks", (unsigned long long)log_cap);
        if ((rc = c->d_t1.ensure(cap1 * sizeof(Slot1)))) return rc;
        if ((rc = c->d_log.ensure(log_cap * (uint64_t)std::max(NB, 1) * sizeof(uint64_t)))) return rc;
        c->cap1 = cap1; c->log_cap = (uint32_t)log_cap;
        memcpy(ut, sh.utab.data(), sh.NU * sizeof(UnitTab));
        CK(cudaMemcpyAsync(c->d_utab.p, ut, sh.NU * sizeof(UnitTab), cudaMemcpyHostToDevice, s));

        if (attempt) CK(cudaMemsetAsync(d_ctr, 0, sizeof(Counters), s));   /* first attempt: zeroed before the scatter */
        CK(cudaEventRecord(c->ev[EV_INIT1], s));
        k_init_table1<<<grid_flat, THREADS, 0, s>>>(c->d_t1.as<Slot1>(), cap1);
        CK(cudaEventRecord(c->ev[EV_PASS1], s));
        Pass1Args a1;
        a1.runs = c->d_tuples.as<u64>();
        a1.rd = rd;
        a1.table = c->d_t1.as<Slot1>(); a1.cap = cap1;
        a1.log = c->d_log.as<u64>(); a1.log_blocks = (uint32_t)log_cap; a1.nb_ranks = (uint32_t)NB;
        a1.ctr = d_ctr;
        if (pt.wide) k_pass1<true><<<grid_p1, THREADS, smem_q1, s>>>(a1, g, pt);
        else k_pass1<false><<<grid_p1, THREADS, smem_q1, s>>>(a1, g, pt);
        CK(cudaEventRecord(c->ev[EV_PRUNE], s));
        PruneArgs ap;
        ap.table = c->d_t1.as<Slot1>(); ap.cap = cap1; ap.log = c->d_log.as<u64>(); ap.nb_ranks = (uint32_t)NB;
        ap.rd = rd; ap.mf = c->prm.min_node_freq; ap.T = T; ap.ctr = d_ctr;
        k_prune<<<grid_flat, THREADS, 0, s>>>(ap, g);
        CK(cudaEventRecord(c->ev[EV_PRUNE_END], s));
        res.kernel_launches += 3;
        CK(cudaGetLastError());
        if ((rc = read_counters(c))) return rc;
        if (h_ctr->overflow == 4) return fail(VDJGRAPH_ERR_INTERNAL, "run region overrun in k_scatter");
        if (h_ctr->overflow == 2) { log_scale *= 2.0; continue; }   /* the occurrence log ran out of blocks */
        if (h_ctr->overflow) {   /* table full or a probe chain past MAX_PROBE: a too small hint is dropped, else more room */
            if (c->prm.table_capacity && !sh.ignore_hint) sh.ignore_hint = true;
            else sh.slot_scale *= 2.0;
            continue;
        }
        if (h_ctr->internal) return fail(VDJGRAPH_ERR_INTERNAL, "occurrence log inconsistent (code %u)", h_ctr->internal);
        break;
    }
    const uint64_t n_surv = h_ctr->n_surv;
    res.n_slow1 += h_ctr->n_slow1;          /* sums over the rounds (zeroed by run_plan) */
    res.n_pre_total += h_ctr->n_distinct;
    res.n_pre += n_surv;
    if (res.n_pre_total > REF_MAX_NODES)
        return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "%llu distinct gated k-mers exceed MAX_NODES (assembler2_vdj.c:73)", (unsigned long long)res.n_pre_total);

    /* ---- survivor table + pass 2 ---- */
    /* table-2 slices: the survivors are spread over the units like the distinct k-mers (no per-unit
     * survivor count exists; at the default load of 0.25 a unit with twice the average survival
     * rate runs at 0.5) */
    const double load2 = std::min(0.9, std::max(0.05, env_double("VDJGRAPH_LOAD2", 0.25)));
    uint64_t cap2 = 0;
    {
        double est_own = 0;
        for (int u = 0; u < sh.NU; u++) if (sh.owner[u] == sh.rank && sh.round_of[u] == sh.rnd) est_own += sh.est[u] + 1.0;
        for (int u = 0; u < sh.NU; u++) {
            if (sh.owner[u] != sh.rank || sh.round_of[u] != sh.rnd) continue;
            const uint64_t len = (uint64_t)((double)n_surv / load2 * (sh.est[u] + 1.0) / est_own) + 64;
            if (cap2 + len > 0x7FFFFFF0ull) return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "survivor table too large");
            sh.utab[u].off2 = (u32)cap2; sh.utab[u].len2 = (u32)len;
            cap2 += len;
        }
        cap2 = std::max<uint64_t>(cap2, 64);
    }
    if ((rc = c->d_t2.ensure(cap2 * sizeof(Slot2)))) return rc;
    c->cap2 = cap2;
    memcpy(ut, sh.utab.data(), sh.NU * sizeof(UnitTab));
    CK(cudaMemcpyAsync(c->d_utab.p, ut, sh.NU * sizeof(UnitTab), cudaMemcpyHostToDevice, s));
    CK(cudaEventRecord(c->ev[EV_TABLE2], s));
    k_init_table2<<<grid_flat, THREADS, 0, s>>>(c->d_t2.as<Slot2>(), cap2);
    k_build_table2<<<grid_flat, THREADS, 0, s>>>(c->d_t1.as<Slot1>(), cap1, c->d_t2.as<Slot2>(), cap2, g, pt, d_ctr);
    CK(cudaEventRecord(c->ev[EV_PASS2], s));
    Pass2Args a2;
    a2.runs = c->d_tuples.as<u64>();
    a2.table = c->d_t2.as<Slot2>(); a2.cap = cap2; a2.ctr = d_ctr;
    if (pt.wide) k_pass2<true><<<grid_p2, THREADS, smem_q, s>>>(a2, g, pt);
    else k_pass2<false><<<grid_p2, THREADS, smem_q, s>>>(a2, g, pt);
    CK(cudaEventRecord(c->ev[EV_PASS2_END], s));
    res.kernel_launches += 3;
    CK(cudaGetLastError());
    res.table1_slots = cap1; res.table2_slots = cap2;
    if (sh.merged()) {
        /* the survivors as dense records: appended to those of the earlier rounds, ready to be sent
         * to the finishing device */
        const uint64_t done = sh.surv_done;
        const uint64_t expect = sh.rnd == 0 && sh.S > 1 ? n_surv * (uint64_t)sh.S + n_surv / 8 : done + n_surv;
        if ((rc = c->d_rec.ensure_keep(std::max<uint64_t>(done + n_surv, 1) * sizeof(Slot2), done * sizeof(Slot2), s))) return rc;
        if (expect > done + n_surv) c->d_rec.ensure_keep(expect * sizeof(Slot2), done * sizeof(Slot2), s);   /* best effort */
        CK(cudaMemsetAsync(&d_ctr->n_nodes, 0, sizeof(u64), s));
        k_compact_table2<<<grid_flat, THREADS, 0, s>>>(c->d_t2.as<Slot2>(), cap2, c->d_rec.as<Slot2>() + done, &d_ctr->n_nodes);
        res.kernel_launches++;
        if ((rc = read_counters(c))) return rc;
        if (h_ctr->overflow) return fail(VDJGRAPH_ERR_INTERNAL, "survivor table overflow (code %u)", h_ctr->overflow);
        if (h_ctr->n_nodes != n_surv) return fail(VDJGRAPH_ERR_INTERNAL, "compacted %llu survivors, expected %llu", (unsigned long long)h_ctr->n_nodes, (unsigned long long)n_surv);
        res.n_hits += h_ctr->n_hits;
        res.n_slow2 += h_ctr->n_slow2;
        res.n_hits_ungated += h_ctr->n_hits_ungated;
        sh.surv_done = done + n_surv;
        add_kernel_times(c);
    } else {
        sh.surv_done = n_surv;
    }
    sh.surv_all[sh.rank] = sh.surv_done;
    return 0;
}

/* VDJGRAPH_FLAG_HASHMAP_LAYOUT: the bucket of every node in the reference's `nodes` map (kernels.cuh,
 * k_hm_*).  One stage per table size 32, 64, ...: the stage's elements are the old table's, in its
 * bucket order, then the nodes created while the table had this size; rounds of propose / move-on
 * until a batch of rounds changes nothing. */
int run_hashmap_layout(vdjgraph_ctx *c, uint64_t n) {
    cudaStream_t s = c->stream;
    int rc;
    vdjgraph_result &res = c->res;
    CK(cudaEventRecord(c->ev[EV_HASHMAP], s));
    uint64_t final_buckets = 32;
    while (n > final_buckets / 2) final_buckets *= 2;
    if (final_buckets > (1ull << 32)) return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "hash-map layout for %llu nodes", (unsigned long long)n);
    const size_t na = std::max<uint64_t>(n, 1);
    if ((rc = c->d_hm_hash.ensure(na * 8)) || (rc = c->d_hm_probe.ensure(na * 4)) || (rc = c->d_hm_prev.ensure(na * 4)) ||
        (rc = c->d_hm_owner.ensure(final_buckets * 8)) || (rc = c->d_hm_slots.ensure(final_buckets * 4)) ||
        (rc = c->d_hm_flag.ensure(16)) || (rc = c->h_hm_flag.ensure(16)))
        return rc;
    const int gb = (int)((na + THREADS - 1) / THREADS);
    if (n) k_hm_hash<<<gb, THREADS, 0, s>>>(c->nodes.d[NodeArrays::KMER_LO].as<u64>(), c->nodes.d[NodeArrays::KMER_HI].as<u64>(), n, c->g.k,
                                            c->d_hm_hash.as<u64>());
    HmStage st;
    st.hash = c->d_hm_hash.as<u64>(); st.owner = c->d_hm_owner.as<u64>(); st.probe = c->d_hm_probe.as<u32>();
    st.prev_bucket = c->d_hm_prev.as<u32>(); st.changed = c->d_hm_flag.as<u32>();
    uint64_t T = 32, n_prev = 0, prev_T = 0;
    u32 *h_flag = c->h_hm_flag.as<u32>();
    for (;;) {
        const uint64_t n_t = std::min<uint64_t>(n, T / 2);
        st.n_old = (u32)n_prev; st.n_all = (u32)n_t; st.prev_buckets = (u32)prev_T; st.mask = (u32)(T - 1);
        CK(cudaMemsetAsync(st.owner, 0xFF, T * 8, s));
        const int g_t = (int)std::max<uint64_t>(1, (n_t + THREADS - 1) / THREADS);
        if (n_t) {
            k_hm_round<<<g_t, THREADS, 0, s>>>(st, 1);
            for (int batch = 0;; batch++) {
                if (batch > 4096) return fail(VDJGRAPH_ERR_INTERNAL, "hash-map layout did not settle");
                CK(cudaMemsetAsync(st.changed, 0, 4, s));
                for (int r = 0; r < 4; r++) k_hm_round<<<g_t, THREADS, 0, s>>>(st, 0);
                res.kernel_launches += 4;
                CK(cudaMemcpyAsync(h_flag, st.changed, 4, cudaMemcpyDeviceToHost, s));
                CK(cudaStreamSynchronize(s));
                if (!*h_flag) break;
            }
            k_hm_settle<<<g_t, THREADS, 0, s>>>(st);
        }
        if (n_t == n) break;
        prev_T = T; n_prev = n_t; T *= 2;
    }
    k_hm_slots<<<(int)((T + THREADS - 1) / THREADS), THREADS, 0, s>>>(st.owner, T, c->d_hm_slots.as<u32>());
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->ev[EV_HASHMAP_END], s));
    res.hm_buckets = T;
    return 0;
}

/* K5: creation ranks and edge lists on ONE device: straight from its survivor table, or (several rounds) from
 * one table over the survivor records of all rounds.  Several devices: finish_step / finish_end below. */
int run_finish(vdjgraph_ctx *c) {
    Shard &sh = c->sh;
    const Geom g = c->g;
    cudaStream_t s = c->stream;
    int rc;
    vdjgraph_result &res = c->res;
    Counters *d_ctr = c->d_ctr.as<Counters>();
    Counters *h_ctr = c->h_ctr.as<Counters>();
    const int grid_flat = c->sm_count * 8;
    Part pt = c->part;
    uint64_t n_surv = sh.surv_all[sh.rank];
    uint64_t cap2 = c->cap2;
    Slot2 *table = c->d_t2.as<Slot2>();
    CK(cudaEventRecord(c->ev[EV_FINISH], s));
    if (sh.merged()) {
        /* several rounds on one device: the survivor records of all rounds */
        const Slot2 *records = c->d_rec.as<Slot2>();
        n_surv = sh.surv_done;
        /* merged table: one flat slice (the finish looks k-mers up by slot hash alone) */
        cap2 = std::max<uint64_t>(1024, (uint64_t)((double)n_surv * MERGED_SLOTS_PER_NODE) + 64);
        /* VDJGRAPH_FREE_TABLES_MB = m: when the merged table exceeds m MB, the tables and the log of the last
         * round (dead: the survivors are records now) are freed before the finish takes its own memory, and
         * the plan counts on that.  Off by default: re-allocating them for the next build costs as much as the
         * saved round; it pays for a single build that would otherwise not fit. */
        const double free_mb = env_double("VDJGRAPH_FREE_TABLES_MB", -1.0);
        if (free_mb >= 0 && (double)(cap2 * sizeof(Slot2)) > free_mb * 1048576.0) {
            CK(cudaStreamSynchronize(s));
            c->d_t1.release(); c->d_log.release(); c->d_t2.release();
        }
        pt.flat = 1; pt.flat_len = (u32)cap2;
        if ((rc = c->d_t2m.ensure(cap2 * sizeof(Slot2)))) return rc;
        table = c->d_t2m.as<Slot2>();
        CK(cudaMemsetAsync(&d_ctr->n_nodes, 0, sizeof(u64), s));
        k_init_table2<<<grid_flat, THREADS, 0, s>>>(table, cap2);
        k_table2_from_records<<<grid_flat, THREADS, 0, s>>>(records, n_surv, table, cap2, g, pt, d_ctr);
        res.kernel_launches += 2;
    }
    const size_t na = std::max<uint64_t>(n_surv, 1);
    const bool keys = want_keys(c->prm.flags);
    if ((rc = c->d_keys[0].ensure(na * 8)) || (rc = c->d_keys[1].ensure(na * 8)) ||
        (rc = c->d_vals[0].ensure(na * 4)) || (rc = c->d_vals[1].ensure(na * 4)) ||
        (rc = c->nodes.ensure(n_surv, keys)))
        return rc;
    const int end_bit = bits_for(sh.total_records * (uint64_t)g.w);
    size_t cub_bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, c->d_keys[0].as<u64>(), c->d_keys[1].as<u64>(),
                                       c->d_vals[0].as<u32>(), c->d_vals[1].as<u32>(), (int64_t)n_surv, 0, end_bit, s));
    if ((rc = c->d_cub.ensure(std::max<size_t>(cub_bytes, 16)))) return rc;
    if (n_surv) {
        k_collect<<<grid_flat, THREADS, 0, s>>>(table, cap2, c->d_keys[0].as<u64>(), c->d_vals[0].as<u32>(), d_ctr);
        CK(cub::DeviceRadixSort::SortPairs(c->d_cub.p, cub_bytes, c->d_keys[0].as<u64>(), c->d_keys[1].as<u64>(),
                                           c->d_vals[0].as<u32>(), c->d_vals[1].as<u32>(), (int64_t)n_surv, 0, end_bit, s));
        const int gb = (int)((n_surv + THREADS - 1) / THREADS);
        k_assign_rank<<<gb, THREADS, 0, s>>>(table, c->d_vals[1].as<u32>(), n_surv);
        ExportArgs ae = c->nodes.export_args(keys);
        ae.table = table; ae.cap = cap2; ae.keys = c->d_keys[1].as<u64>(); ae.vals = c->d_vals[1].as<u32>(); ae.n = n_surv;
        k_export<<<gb, THREADS, 0, s>>>(ae, g, pt);
        res.kernel_launches += 3;
    }
    res.hm_buckets = 0; res.ms_hashmap = 0;
    if ((c->prm.flags & VDJGRAPH_FLAG_HASHMAP_LAYOUT) && (rc = run_hashmap_layout(c, n_surv))) return rc;
    CK(cudaEventRecord(c->ev[EV_FINISH_END], s));
    CK(cudaGetLastError());
    if ((rc = read_counters(c))) return rc;
    if (h_ctr->overflow) return fail(VDJGRAPH_ERR_INTERNAL, "survivor table overflow (code %u)", h_ctr->overflow);
    if (h_ctr->internal) return fail(VDJGRAPH_ERR_INTERNAL, "export invariant violated (code %u)", h_ctr->internal);
    if (n_surv && h_ctr->n_nodes != n_surv)
        return fail(VDJGRAPH_ERR_INTERNAL, "collected %llu nodes, expected %llu", (unsigned long long)h_ctr->n_nodes, (unsigned long long)n_surv);
    c->ctr = *h_ctr;
    res.n_nodes = n_surv;
    if (!sh.merged()) {
        res.n_hits = h_ctr->n_hits;
        res.n_slow2 = h_ctr->n_slow2;
        res.n_hits_ungated = h_ctr->n_hits_ungated;
        add_kernel_times(c);   /* the only round (a merged build adds each round's in run_passes) */
    } else {
        res.n_pre = n_surv;
    }
    take_times(c);
    cudaEventElapsedTime(&res.ms_device, c->ev[EV_BUILD], c->ev[EV_FINISH_END]);
    c->view.table = n_surv ? table : nullptr;
    c->view.cap = cap2; c->view.n_nodes = n_surv; c->view.pt = pt; c->view.g = g;
    return 0;
}

/* The finish of a build over several devices (kernels.cuh, "K5 on several devices").  Every device's exchange
 * buffer (BUF_GATHER, mapped by its peers) holds: 256 bytes of barrier flags and counters | the sorted stamps of ALL
 * devices (its own segment is sorted into place, the peers' are copied in) | its flat survivor table | on the
 * finishing device, the node rows of the whole graph, their overflow list and (when wanted) their k-mers.  Every
 * offset follows from the all-gathered survivor counts and the build flags (the same on every rank). */
constexpr size_t FLAGS_BYTES = 256;      /* [0, 64): barrier flags; [128, 132): overflow entries of the node rows */
constexpr size_t OVER_COUNT_OFF = 128;
struct FinishLayout { size_t keys_off, table_off, rows_off, over_off, kmers_off, bytes; uint64_t n_total, cap; };
FinishLayout finish_layout(const uint64_t *surv, int G, int rank, uint32_t flags) {
    FinishLayout f;
    f.n_total = 0;
    for (int d = 0; d < G; d++) f.n_total += surv[d];
    const uint64_t na = std::max<uint64_t>(f.n_total, 1);
    f.keys_off = FLAGS_BYTES;
    f.table_off = (f.keys_off + na * 8 + 255) & ~(size_t)255;
    f.cap = std::max<uint64_t>(1024, (uint64_t)((double)surv[rank] * MERGED_SLOTS_PER_NODE) + 64);
    f.rows_off = f.table_off + f.cap * sizeof(Slot2);
    f.over_off = f.rows_off + (rank == 0 ? na * ROW_WORDS * 8 : 0);
    f.kmers_off = f.over_off + (rank == 0 ? na * 16 : 0);
    f.bytes = f.kmers_off + (rank == 0 && want_keys(flags) ? na * 16 : 0);
    return f;
}
RowSink row_sink(char *arena0, const FinishLayout &f0, uint32_t flags) {
    RowSink r;
    r.rows = reinterpret_cast<u64 *>(arena0 + f0.rows_off);
    r.over = reinterpret_cast<ulonglong2 *>(arena0 + f0.over_off);
    r.n_over = reinterpret_cast<u32 *>(arena0 + OVER_COUNT_OFF);
    r.kmers = want_keys(flags) ? reinterpret_cast<ulonglong2 *>(arena0 + f0.kmers_off) : nullptr;
    return r;
}

int finish_plan(vdjgraph_ctx *c) {
    Shard &sh = c->sh;
    int rc;
    const FinishLayout f = finish_layout(sh.surv_all, sh.G, sh.rank, c->prm.flags);
    if (f.n_total >= NIL32) return fail(VDJGRAPH_ERR_TOO_MANY_NODES, "%llu nodes", (unsigned long long)f.n_total);
    /* everything the finish needs is allocated here: its steps are queued without a host synchronisation in
     * between (an allocation would be one) */
    void *before = c->d_gather.p;
    if ((rc = c->d_gather.ensure(f.bytes))) return rc;
    if (c->d_gather.p != before) CK(cudaMemset(c->d_gather.p, 0, FLAGS_BYTES));   /* fresh barrier flags */
    const size_t nr = std::max<uint64_t>(sh.surv_all[sh.rank], 1);
    if ((rc = c->d_keys[0].ensure(nr * 8)) || (rc = c->d_vals[0].ensure(nr * 4)) || (rc = c->d_vals[1].ensure(nr * 4)) ||
        (rc = c->d_gid.ensure(nr * 4)) || (rc = c->d_owner.ensure(NBUCKET)))
        return rc;
    size_t cub_bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, c->d_keys[0].as<u64>(), c->d_keys[0].as<u64>(), c->d_vals[0].as<u32>(),
                                       c->d_vals[1].as<u32>(), (int64_t)nr, 0, 64, c->stream));
    if ((rc = c->d_cub.ensure(std::max<size_t>(cub_bytes, 16)))) return rc;
    std::vector<u8> owner(NBUCKET, 0);
    for (int u = 0; u < sh.NU; u++) owner[u] = (u8)sh.owner[u];
    CK(cudaMemcpy(c->d_owner.p, owner.data(), NBUCKET, cudaMemcpyHostToDevice));
    if (sh.rank == 0 && (rc = c->nodes.ensure(f.n_total, want_keys(c->prm.flags)))) return rc;
    return 0;
}

/* one of the three steps (see kernels.cuh); then the devices meet: on the device (device_barrier: the next step
 * can be queued at once) or on the host (the stream is synchronised; the caller holds a barrier of its own) */
int finish_step(vdjgraph_ctx *c, int step, bool device_barrier) {
    Shard &sh = c->sh;
    const Geom g = c->g;
    cudaStream_t s = c->stream;
    vdjgraph_result &res = c->res;
    Counters *d_ctr = c->d_ctr.as<Counters>();
    const FinishLayout f = finish_layout(sh.surv_all, sh.G, sh.rank, c->prm.flags);
    char *arena = c->d_gather.as<char>();
    const uint64_t n_r = sh.surv_all[sh.rank];
    Slot2 *table = reinterpret_cast<Slot2 *>(arena + f.table_off);
    u64 *all_keys = reinterpret_cast<u64 *>(arena + f.keys_off);
    const int grid_flat = c->sm_count * 8;
    const int gb = (int)std::max<uint64_t>(1, (n_r + THREADS - 1) / THREADS);
    for (int d = 0; d < sh.G; d++)
        if (!sh.peer[d][BUF_GATHER]) return fail(VDJGRAPH_ERR_STATE, "device %d's exchange buffer is not set", d);
    if (step == 0) {
        CK(cudaEventRecord(c->ev[EV_FINISH], s));
        Part pt = c->part;
        pt.flat = 1; pt.flat_len = (u32)f.cap;
        CK(cudaMemsetAsync(&d_ctr->n_nodes, 0, sizeof(u64), s));
        k_init_table2<<<grid_flat, THREADS, 0, s>>>(table, f.cap);
        res.kernel_launches++;
        if (n_r) {
            k_table2_from_records<<<grid_flat, THREADS, 0, s>>>(c->d_rec.as<Slot2>(), n_r, table, f.cap, g, pt, d_ctr);
            k_collect<<<grid_flat, THREADS, 0, s>>>(table, f.cap, c->d_keys[0].as<u64>(), c->d_vals[0].as<u32>(), d_ctr);
            size_t cub_bytes = c->d_cub.cap;
            CK(cub::DeviceRadixSort::SortPairs(c->d_cub.p, cub_bytes, c->d_keys[0].as<u64>(), all_keys + sh.surv_off[sh.rank],
                                               c->d_vals[0].as<u32>(), c->d_vals[1].as<u32>(), (int64_t)n_r, 0,
                                               bits_for(sh.total_records * (uint64_t)g.w), s));
            res.kernel_launches += 2;
        }
    } else if (step == 1) {
        KeySegs ks;
        for (int d = 0; d <= sh.G; d++) ks.off[d] = sh.surv_off[d];
        for (int d = 0; d < sh.G; d++)
            if (d != sh.rank && sh.surv_all[d])
                CK(cudaMemcpyAsync(all_keys + sh.surv_off[d], (const char *)sh.peer[d][BUF_GATHER] + f.keys_off + sh.surv_off[d] * 8,
                                   sh.surv_all[d] * 8, cudaMemcpyDefault, s));
        if (n_r) {
            k_global_rank<<<gb, THREADS, 0, s>>>(all_keys, ks, sh.G, sh.rank, table, c->d_vals[1].as<u32>(), c->d_gid.as<u32>(), d_ctr);
            res.kernel_launches++;
        }
    } else {
        if (n_r) {
            PeerTables pt;
            for (int d = 0; d < MAX_DEV; d++) { pt.table[d] = nullptr; pt.len[d] = 1; }
            for (int d = 0; d < sh.G; d++) {
                const FinishLayout fd = finish_layout(sh.surv_all, sh.G, d, c->prm.flags);
                pt.table[d] = reinterpret_cast<const Slot2 *>((const char *)sh.peer[d][BUF_GATHER] + fd.table_off);
                pt.len[d] = (u32)fd.cap;
            }
            pt.owner = c->d_owner.as<u8>();
            pt.ushift = (u32)sh.ushift;
            const FinishLayout f0 = finish_layout(sh.surv_all, sh.G, 0, c->prm.flags);
            ExportDistArgs a;
            a.keys = all_keys + sh.surv_off[sh.rank]; a.vals = c->d_vals[1].as<u32>(); a.gid = c->d_gid.as<u32>();
            a.n = n_r; a.self = sh.rank;
            a.sink = row_sink((char *)sh.peer[0][BUF_GATHER], f0, c->prm.flags);
            k_export_dist<<<gb, THREADS, 0, s>>>(a, pt, g, d_ctr);
            res.kernel_launches++;
        }
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(c->ev[EV_STEP0 + 2 * step], s));
    if (device_barrier) {
        PeerFlags pf;
        for (int d = 0; d < MAX_DEV; d++) pf.flags[d] = reinterpret_cast<u64 *>(sh.peer[d < sh.G ? d : sh.rank][BUF_GATHER]);
        const double patience_s = env_double("VDJGRAPH_BARRIER_PATIENCE_S", 20.0);
        k_peer_barrier<<<1, 32, 0, s>>>(pf, sh.G, sh.rank, ++sh.bar_seq, (u64)(patience_s * 1e9), d_ctr);
        res.kernel_launches++;
        CK(cudaGetLastError());
    } else {
        CK(cudaStreamSynchronize(s));
    }
    CK(cudaEventRecord(c->ev[EV_STEP0_MET + 2 * step], s));
    return 0;
}

/* after the third step (and the barrier behind it): the finishing device unpacks the rows; every device checks
 * its counters */
int finish_end(vdjgraph_ctx *c) {
    Shard &sh = c->sh;
    cudaStream_t s = c->stream;
    vdjgraph_result &res = c->res;
    Counters *h_ctr = c->h_ctr.as<Counters>();
    const FinishLayout f = finish_layout(sh.surv_all, sh.G, sh.rank, c->prm.flags);
    int rc;
    res.hm_buckets = 0; res.ms_hashmap = 0;
    if (sh.rank == 0) {
        if (f.n_total) {
            ExportArgs ae = c->nodes.export_args(want_keys(c->prm.flags));
            ae.n = f.n_total;
            const RowSink sink = row_sink(c->d_gather.as<char>(), f, c->prm.flags);
            k_unpack_rows<<<(int)((f.n_total + THREADS - 1) / THREADS), THREADS, 0, s>>>(sink, f.n_total, ae);
            k_unpack_overflow<<<c->sm_count, THREADS, 0, s>>>(sink, ae);
            res.kernel_launches++;
            res.kernel_launches++;
            CK(cudaGetLastError());
        }
        if (c->prm.flags & VDJGRAPH_FLAG_HASHMAP_LAYOUT) {
            /* a peer that never arrived must not send the layout into a loop over garbage keys */
            if ((rc = read_counters(c))) return rc;
            if (h_ctr->internal) return fail(VDJGRAPH_ERR_INTERNAL, "sharded finish failed (code %u)", h_ctr->internal);
            if ((rc = run_hashmap_layout(c, f.n_total))) return rc;
        }
    }
    CK(cudaEventRecord(c->ev[EV_FINISH_END], s));
    if ((rc = read_counters(c))) return rc;
    if (h_ctr->overflow) return fail(VDJGRAPH_ERR_INTERNAL, "survivor table overflow (code %u)", h_ctr->overflow);
    if (h_ctr->internal == 9) return fail(VDJGRAPH_ERR_INTERNAL, "a peer device did not reach the barrier of the sharded finish");
    if (h_ctr->internal) return fail(VDJGRAPH_ERR_INTERNAL, "export invariant violated (code %u)", h_ctr->internal);
    if (sh.surv_all[sh.rank] && h_ctr->n_nodes != sh.surv_all[sh.rank])
        return fail(VDJGRAPH_ERR_INTERNAL, "collected %llu nodes, expected %llu", (unsigned long long)h_ctr->n_nodes,
                    (unsigned long long)sh.surv_all[sh.rank]);
    c->ctr = *h_ctr;
    take_times(c);
    if (env_double("VDJGRAPH_FINISH_TIMES", 0) > 0) {
        /* where a distributed finish spends its time on this device: the three steps, the wait at the barrier
         * behind each, and (finishing device) unpacking the rows */
        float t[7];
        for (int i = 0; i < 7; i++) cudaEventElapsedTime(&t[i], c->ev[EV_FINISH + i], c->ev[EV_FINISH + i + 1]);
        fprintf(stderr, "vdjgraph finish rank %d: table+sort %.3f wait %.3f | rank %.3f wait %.3f | edges+rows %.3f wait %.3f | unpack %.3f ms\n",
                sh.rank, t[0], t[1], t[2], t[3], t[4], t[5], t[6]);
    }
    res.ms_device = res.ms_scatter + res.ms_init1 + res.ms_pass1 + res.ms_prune + res.ms_table2 + res.ms_pass2 + res.ms_export;
    res.n_nodes = sh.rank == 0 ? f.n_total : 0;
    if (sh.rank == 0) res.n_pre = f.n_total;   /* (the other ranks keep their own survivor count) */
    return 0;
}

} // namespace

extern "C" int vdjgraph_run(vdjgraph_ctx *c) {
    if (!c) return fail(VDJGRAPH_ERR_PARAM, "ctx is NULL");
    int rc = check_state(c, "vdjgraph_run", from(State::STAGED),
                         c->sh.G == 1 ? nullptr : "vdjgraph_run on a sharded context; use the vdjgraph_shard_* phases");
    if (rc) return rc;
    c->state = State::STAGED;   /* until the build has finished */
    CK(cudaSetDevice(c->device));
    if (c->g.R == 0) {
        reset_run_stats(c);
        c->view = GraphView();   /* no nodes: every window answers NIL */
        c->view.g = c->g;
    } else {
        if ((rc = run_plan(c, c->h_hist.as<uint64_t>(), c->h_hll.as<uint8_t>()))) return rc;
        own_buffers(c, c->sh.peer[c->sh.rank], nullptr);   /* the only peer */
        for (int r = 0; r < c->sh.S; r++) {
            c->sh.rnd = r;
            if ((rc = run_scatter(c))) return rc;
            if ((rc = run_passes(c))) return rc;
        }
        if ((rc = run_finish(c))) return rc;
    }
    c->state = State::FINISHED;
    return 0;
}

/* ---------------------------------------------------------------------------------------- */
/* sharded build: the same phases, driven by the caller                                       */
/* ---------------------------------------------------------------------------------------- */
extern "C" int vdjgraph_shard_stage(vdjgraph_ctx *c, const char *primary, size_t np, const char *secondary, size_t ns,
                                    const vdjgraph_shard_info *info) {
    return info ? stage_impl(c, primary, np, secondary, ns, 0, info) : fail(VDJGRAPH_ERR_PARAM, "NULL argument");
}
/* forward reads only (vdjgraph_stage_forward); record_base / total_records / the record counts handed
 * to vdjgraph_shard_plan stay in the doubled numbering (two records per read) */
extern "C" int vdjgraph_shard_stage_forward(vdjgraph_ctx *c, const char *primary_reads, size_t np, const char *secondary_reads,
                                            size_t ns, const vdjgraph_shard_info *info) {
    return info ? stage_impl(c, primary_reads, np, secondary_reads, ns, 1, info) : fail(VDJGRAPH_ERR_PARAM, "NULL argument");
}

/* the per-bucket counts and HyperLogLog registers of this rank's staged records (k_count ran with the staging);
 * after a finished build, the next build of the same records */
extern "C" int vdjgraph_shard_count(vdjgraph_ctx *c, uint64_t *hist, uint8_t *hll) {
    int rc = check_state(c, "vdjgraph_shard_count", bit(State::STAGED) | bit(State::FINISHED));
    if (rc) return rc;
    if (!hist || !hll) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    memcpy(hist, c->h_hist.p, HIST_WORDS * sizeof(uint64_t));
    memcpy(hll, c->h_hll.p, HLL_BYTES);
    c->state = State::COUNTED;
    return 0;
}

extern "C" int vdjgraph_shard_plan(vdjgraph_ctx *c, const uint64_t *hist_all, const uint8_t *hll_merged,
                                   const uint64_t *record_counts) {
    int rc = check_state(c, "vdjgraph_shard_plan", bit(State::COUNTED));
    if (rc) return rc;
    if (!hist_all || !hll_merged || !record_counts) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    c->state = State::STAGED;   /* until the plan is made */
    CK(cudaSetDevice(c->device));
    Shard &sh = c->sh;
    uint64_t base = 0;
    for (int d = 0; d < sh.G; d++) { sh.rec_base[d] = base; base += record_counts[d]; }
    sh.rec_base[sh.G] = base;
    if (base != sh.total_records || record_counts[sh.rank] != c->g.R)
        return fail(VDJGRAPH_ERR_PARAM, "record counts do not add up to total_records / this rank's staged records");
    if ((rc = run_plan(c, hist_all, hll_merged))) return rc;
    /* the barrier flags of the finish start every build at zero (the peers' stores of this build come after
     * several host exchanges; those of the last build arrived before its final one) */
    sh.bar_seq = 0;
    if (sh.G > 1 && c->d_gather.p) CK(cudaMemset(c->d_gather.p, 0, FLAGS_BYTES));
    c->state = State::PLANNED;
    return 0;
}

extern "C" int vdjgraph_shard_buffers(vdjgraph_ctx *c, void **ptrs, size_t *bytes) {
    if (!c || !ptrs) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    own_buffers(c, ptrs, bytes);
    return 0;
}

extern "C" int vdjgraph_shard_set_peers(vdjgraph_ctx *c, void *const *ptrs) {
    if (!c || !ptrs) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    int rc = check_state(c, "vdjgraph_shard_set_peers", from(State::PLANNED));
    if (rc) return rc;
    Shard &sh = c->sh;
    for (int d = 0; d < sh.G; d++)
        for (int i = 0; i < NBUF; i++) sh.peer[d][i] = ptrs[d * NBUF + i];
    own_buffers(c, sh.peer[sh.rank], nullptr);
    if (c->state == State::PLANNED) c->state = State::PEERS_SET;   /* called again for the finish: the state stays */
    return 0;
}

extern "C" int vdjgraph_shard_rounds(vdjgraph_ctx *c) {
    int rc = check_state(c, "vdjgraph_shard_rounds", from(State::PLANNED));
    return rc ? rc : c->sh.S;
}

extern "C" int vdjgraph_shard_scatter(vdjgraph_ctx *c) {
    if (!c) return fail(VDJGRAPH_ERR_PARAM, "ctx is NULL");
    /* the first round once the peers are set, each further one after the passes of the round before */
    int rc = check_state(c, "vdjgraph_shard_scatter", bit(State::PEERS_SET) | (c->rounds_left() ? bit(State::PASSES_DONE) : 0));
    if (rc) return rc;
    if (c->state == State::PASSES_DONE) c->sh.rnd++;
    c->state = State::STAGED;   /* until the runs are scattered */
    CK(cudaSetDevice(c->device));
    if ((rc = run_scatter(c))) return rc;
    c->state = State::SCATTERED;
    return 0;
}

extern "C" int vdjgraph_shard_passes(vdjgraph_ctx *c, uint64_t *n_survivors) {
    int rc = check_state(c, "vdjgraph_shard_passes", bit(State::SCATTERED));
    if (rc) return rc;
    c->state = State::STAGED;   /* until the passes are done */
    CK(cudaSetDevice(c->device));
    if ((rc = run_passes(c))) return rc;
    if (c->sh.G == 1) { CK(cudaStreamSynchronize(c->stream)); }
    if (n_survivors) *n_survivors = c->sh.surv_all[c->sh.rank];
    c->state = State::PASSES_DONE;
    return 0;
}

extern "C" int vdjgraph_shard_gather_plan(vdjgraph_ctx *c, const uint64_t *survivors_all) {
    if (!c || !survivors_all) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    int rc = check_state(c, "vdjgraph_shard_gather_plan", bit(State::PASSES_DONE),
                         c->rounds_left() ? "vdjgraph_shard_gather_plan before the last round: vdjgraph_shard_scatter comes next" : nullptr);
    if (rc) return rc;
    c->state = State::STAGED;   /* until the finish is planned */
    CK(cudaSetDevice(c->device));
    Shard &sh = c->sh;
    if (survivors_all[sh.rank] != sh.surv_done)
        return fail(VDJGRAPH_ERR_PARAM, "survivors_all[%d] is not this rank's survivor count", sh.rank);
    uint64_t off = 0;
    for (int d = 0; d < sh.G; d++) { sh.surv_all[d] = survivors_all[d]; sh.surv_off[d] = off; off += survivors_all[d]; }
    sh.surv_off[sh.G] = off;
    if (sh.G > 1 && (rc = finish_plan(c))) return rc;
    c->state = State::FINISH_PLANNED;
    return 0;
}

extern "C" int vdjgraph_shard_finish_bytes(vdjgraph_ctx *c, const uint64_t *survivors_all, uint32_t rank, size_t *bytes) {
    if (!c || !survivors_all || !bytes || rank >= (uint32_t)c->sh.G) return fail(VDJGRAPH_ERR_PARAM, "bad argument");
    *bytes = c->sh.G > 1 ? finish_layout(survivors_all, c->sh.G, (int)rank, c->prm.flags).bytes : 0;
    return 0;
}

extern "C" int vdjgraph_shard_finish_step(vdjgraph_ctx *c, int step, int device_barrier) {
    if (step < 0 || step > 2) return fail(VDJGRAPH_ERR_PARAM, "finish step %d", step);
    const State before = State((int)State::FINISH_PLANNED + step);   /* FINISH_PLANNED or the step before */
    int rc = check_state(c, "vdjgraph_shard_finish_step", bit(before));
    if (rc) return rc;
    c->state = State::STAGED;   /* until the step is queued */
    CK(cudaSetDevice(c->device));
    /* one device: everything happens in vdjgraph_shard_finish */
    if (c->sh.G > 1 && (rc = finish_step(c, step, device_barrier != 0))) return rc;
    c->state = State((int)before + 1);
    return 0;
}

extern "C" int vdjgraph_shard_finish(vdjgraph_ctx *c) {
    int rc = check_state(c, "vdjgraph_shard_finish", bit(State::FINISH_STEP2));
    if (rc) return rc;
    c->state = State::STAGED;   /* until the graph is finished */
    CK(cudaSetDevice(c->device));
    if ((rc = c->sh.G == 1 ? run_finish(c) : finish_end(c))) return rc;
    c->state = State::FINISHED;
    return 0;
}

/* Frees allocations that were replaced by larger ones while peers could still have them mapped.
 * Call it once every rank has installed (and mapped) the current buffers. */
extern "C" int vdjgraph_shard_release_retired(vdjgraph_ctx *c) {
    if (!c) return fail(VDJGRAPH_ERR_PARAM, "ctx is NULL");
    CK(cudaSetDevice(c->device));
    for (DevBuf *b : c->peer_bufs()) b->release_retired();
    return 0;
}

/* opaque CUDA IPC handles for callers that run one process per GPU (64 bytes each) */
extern "C" int vdjgraph_ipc_export(const void *dptr, unsigned char *out64) {
    if (!dptr || !out64) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, const_cast<void *>(dptr)));
    memcpy(out64, &h, 64);
    return 0;
}
extern "C" int vdjgraph_ipc_open(const unsigned char *in64, void **dptr) {
    if (!in64 || !dptr) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, in64, 64);
    CK(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
extern "C" int vdjgraph_ipc_close(void *dptr) {
    if (!dptr) return 0;
    CK(cudaIpcCloseMemHandle(dptr));
    return 0;
}
/* same-process peers (G contexts on several devices of one process) */
extern "C" int vdjgraph_enable_peer_access(int device, int peer_device) {
    if (device == peer_device) return 0;
    CK(cudaSetDevice(device));
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return 0; }
    CK(e);
    return 0;
}

/* Page-locked host memory for the caller's record buffers: staging then DMAs straight out of them. */
extern "C" int vdjgraph_host_alloc(size_t bytes, void **out) {
    if (!out) return fail(VDJGRAPH_ERR_PARAM, "out is NULL");
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, std::max<size_t>(bytes, 1), cudaHostAllocPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *out = nullptr;
        return fail(e == cudaErrorMemoryAllocation ? VDJGRAPH_ERR_NOMEM : VDJGRAPH_ERR_CUDA,
                    "cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    return 0;
}
extern "C" int vdjgraph_host_free(void *p) {
    if (!p) return 0;
    CK(cudaFreeHost(p));
    return 0;
}
extern "C" int vdjgraph_host_register(void *p, size_t bytes) {
    if (!p || !bytes) return fail(VDJGRAPH_ERR_PARAM, "NULL or empty buffer");
    CK(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return 0;
}
extern "C" int vdjgraph_host_unregister(void *p) {
    if (!p) return 0;
    CK(cudaHostUnregister(p));
    return 0;
}

extern "C" int vdjgraph_fetch(vdjgraph_ctx *c, vdjgraph_result *out) {
    if (!c || !out) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    int rc = check_state(c, "vdjgraph_fetch", bit(State::FINISHED), c->has_graph() ? nullptr : "vdjgraph_fetch on a rank other than 0");
    if (rc) return rc;
    CK(cudaSetDevice(c->device));
    double t0 = wall_ms();
    vdjgraph_result &r = c->res;
    uint64_t bytes = 0;
    if ((rc = c->nodes.fetch(r.n_nodes, c->prm.flags & VDJGRAPH_FLAG_EXPORT_KEYS, c->stream, r, bytes))) return rc;
    if (c->res.hm_buckets) {   /* the layout exists even for an empty graph: 32 empty buckets */
        cudaStream_t s = c->stream;
        if ((rc = c->h_hm_slots.ensure(c->res.hm_buckets * 4))) return rc;
        CK(cudaMemcpyAsync(c->h_hm_slots.p, c->d_hm_slots.p, c->res.hm_buckets * 4, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        bytes += c->res.hm_buckets * 4;
    }
    r.hm_slots = c->res.hm_buckets ? c->h_hm_slots.as<uint32_t>() : nullptr;
    r.d2h_bytes = bytes;
    r.ms_fetch = (float)(wall_ms() - t0);
    *out = r;
    return 0;
}

extern "C" int vdjgraph_stats(vdjgraph_ctx *c, vdjgraph_result *out) {
    if (!c || !out) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    if (int rc = check_state(c, "vdjgraph_stats", bit(State::FINISHED))) return rc;
    *out = c->res;
    out->first_pos = nullptr; out->frequency = nullptr; out->out_deg = out->in_deg = nullptr;
    out->out_succ = out->in_pred = nullptr; out->kmer_lo = out->kmer_hi = nullptr; out->hm_slots = nullptr;
    return 0;
}

extern "C" int vdjgraph_build(vdjgraph_ctx *c, const char *primary, size_t np, const char *secondary, size_t ns,
                              vdjgraph_result *out) {
    int rc = vdjgraph_stage(c, primary, np, secondary, ns);
    if (rc) return rc;
    if ((rc = vdjgraph_run(c))) return rc;
    return vdjgraph_fetch(c, out);
}

extern "C" int vdjgraph_build_forward(vdjgraph_ctx *c, const char *primary_reads, size_t np, const char *secondary_reads, size_t ns,
                                      vdjgraph_result *out) {
    int rc = vdjgraph_stage_forward(c, primary_reads, np, secondary_reads, ns);
    if (rc) return rc;
    if ((rc = vdjgraph_run(c))) return rc;
    return vdjgraph_fetch(c, out);
}

extern "C" int vdjgraph_fetch_pre_table(vdjgraph_ctx *c, vdjgraph_pre_table *out) {
    if (!c || !out) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    int rc = check_state(c, "vdjgraph_fetch_pre_table", bit(State::FINISHED),
                         c->has_graph() ? nullptr : "vdjgraph_fetch_pre_table on a rank other than 0");
    if (rc) return rc;
    if (c->sh.merged()) return fail(VDJGRAPH_ERR_STATE, "the pruned pass-1 table is only kept by a one-device, one-round build");
    CK(cudaSetDevice(c->device));
    const uint64_t n = c->res.n_pre;
    const size_t na = std::max<uint64_t>(n, 1);
    if ((rc = c->d_pre_klo.ensure(na * 8)) || (rc = c->d_pre_khi.ensure(na * 8)) || (rc = c->d_pre_freq.ensure(na * 2)) ||
        (rc = c->d_pre_n.ensure(8)) || (rc = c->h_pre_klo.ensure(na * 8)) || (rc = c->h_pre_khi.ensure(na * 8)) ||
        (rc = c->h_pre_freq.ensure(na * 2)) || (rc = c->h_pre_n.ensure(8)))
        return rc;
    cudaStream_t s = c->stream;
    if (n) {
        CK(cudaMemsetAsync(c->d_pre_n.p, 0, 8, s));
        k_export_pre<<<c->sm_count * 8, THREADS, 0, s>>>(c->d_t1.as<Slot1>(), c->cap1, c->d_pre_klo.as<u64>(),
                                                          c->d_pre_khi.as<u64>(), c->d_pre_freq.as<u16>(), c->d_pre_n.as<u64>());
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(c->h_pre_klo.p, c->d_pre_klo.p, n * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(c->h_pre_khi.p, c->d_pre_khi.p, n * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(c->h_pre_freq.p, c->d_pre_freq.p, n * 2, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(c->h_pre_n.p, c->d_pre_n.p, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (*c->h_pre_n.as<uint64_t>() != n) return fail(VDJGRAPH_ERR_INTERNAL, "pre-table export count mismatch");
    }
    out->n = n;
    out->kmer_lo = c->h_pre_klo.as<uint64_t>();
    out->kmer_hi = c->h_pre_khi.as<uint64_t>();
    out->frequency = c->h_pre_freq.as<uint16_t>();
    return 0;
}

/* ========================================================================================== */
/* Queries: the node of every k-mer window of caller sequences (k_query_pack, k_query)          */
/* ========================================================================================== */
extern "C" int vdjgraph_query(vdjgraph_ctx *c, const char *seqs, const uint64_t *offsets, size_t nq,
                              uint32_t *out, size_t n_windows, vdjgraph_query_stats *stats) {
    const double t0 = wall_ms();
    int rc = check_state(c, "vdjgraph_query", bit(State::FINISHED));
    if (rc) return rc;
    if (!c->queryable())
        return fail(VDJGRAPH_ERR_STATE, "vdjgraph_query on a graph built over %d ranks: each rank's table holds its own share", c->sh.G);
    if (nq && !offsets) return fail(VDJGRAPH_ERR_PARAM, "offsets is NULL");
    const GraphView &v = c->view;
    const uint64_t k = (uint64_t)v.g.k;
    auto windows_of = [k](uint64_t len) { return len >= k ? len - k + 1 : 0; };
    uint64_t total = 0;
    for (size_t i = 0; i < nq; i++) {
        if (offsets[i + 1] < offsets[i]) return fail(VDJGRAPH_ERR_PARAM, "offsets decrease at query %zu", i);
        total += windows_of(offsets[i + 1] - offsets[i]);
    }
    if (total != n_windows)
        return fail(VDJGRAPH_ERR_PARAM, "n_windows is %zu, the queries have %llu windows", n_windows, (unsigned long long)total);
    const uint64_t t_lo = nq ? offsets[0] : 0, n_bytes = nq ? offsets[nq] - offsets[0] : 0;
    if ((n_bytes && !seqs) || (n_windows && !out)) return fail(VDJGRAPH_ERR_PARAM, "NULL buffer");
    CK(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    QueryBufs &qb = c->q;
    if ((rc = qb.init())) return rc;
    const double chunk_kb = env_double("VDJGRAPH_QUERY_CHUNK_KB", 0);
    const uint64_t CH = chunk_kb > 0 ? std::max<uint64_t>(64, (uint64_t)(chunk_kb * 1024)) : QUERY_CHUNK;
    const uint64_t QMAX = std::max<uint64_t>(1024, CH / 16);   /* queries per chunk (empty ones take no bytes) */
    if ((rc = qb.d_ctr.ensure(16)) || (rc = qb.ctr.ensure(16)) || (rc = qb.d_out.ensure(std::max<size_t>(n_windows, 1) * 4)) ||
        (rc = qb.d_bases.ensure(CH / 4 + 64)) || (rc = qb.d_nmask.ensure(CH / 8 + 64)))
        return rc;
    uint64_t *hc = qb.ctr.as<uint64_t>();   /* [0] windows found, [1] first byte outside ACGTN */
    hc[0] = 0; hc[1] = ~0ull;
    CK(cudaMemcpyAsync(qb.d_ctr.p, hc, 16, cudaMemcpyHostToDevice, s));
    uint64_t h2d = 16, d2h = 0;
    const bool direct = is_page_locked(seqs + t_lo, n_bytes);   /* page-locked text: DMA straight out of it */
    float ms_kernels = 0;
    qb.pending[0] = qb.pending[1] = false;
    auto retire = [&](int b) -> int {   /* chunk kernels behind k_end[b] have finished: add their time */
        if (!qb.pending[b]) return 0;
        CK(cudaEventSynchronize(qb.k_end[b]));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, qb.k_begin[b], qb.k_end[b]));
        ms_kernels += ms;
        qb.pending[b] = false;
        return 0;
    };
    /* chunks of whole queries, at most CH bytes unless one query alone is longer */
    uint64_t w_base = 0;
    for (uint64_t i = 0, chunk = 0; i < nq; chunk++) {
        const int b = (int)(chunk & 1);
        if ((rc = retire(b))) return rc;   /* the kernels of chunk - 2 are done with buffer set b */
        const uint64_t c_lo = offsets[i];
        uint64_t j = i + 1;
        while (j < nq && j - i < QMAX && offsets[j + 1] - c_lo <= CH) j++;
        const uint64_t nb = offsets[j] - c_lo, nqc = j - i, nb_pad = std::max<uint64_t>(64, (nb + 63) & ~63ull);
        const size_t meta_bytes = (2 * nqc + 1) * sizeof(uint64_t);
        if ((rc = qb.meta[b].ensure(meta_bytes)) || (rc = qb.d_meta[b].ensure(meta_bytes)) || (rc = qb.d_text[b].ensure(nb_pad)) ||
            (rc = qb.d_bases.ensure(nb_pad / 4)) || (rc = qb.d_nmask.ensure(nb_pad / 8)) || (!direct && (rc = qb.text[b].ensure(nb))))
            return rc;
        uint64_t *qoff = qb.meta[b].as<uint64_t>(), *woff = qoff + nqc, wn = 0;
        for (uint64_t x = 0; x < nqc; x++) {
            qoff[x] = offsets[i + x] - c_lo;
            woff[x] = wn;
            wn += windows_of(offsets[i + x + 1] - offsets[i + x]);
        }
        woff[nqc] = wn;
        const char *src = seqs + c_lo;
        if (!direct && nb) { memcpy(qb.text[b].p, src, nb); src = qb.text[b].as<char>(); }
        if (nb) CK(cudaMemcpyAsync(qb.d_text[b].p, src, nb, cudaMemcpyHostToDevice, qb.h2d));
        CK(cudaMemcpyAsync(qb.d_meta[b].p, qoff, meta_bytes, cudaMemcpyHostToDevice, qb.h2d));
        CK(cudaEventRecord(qb.copied[b], qb.h2d));
        h2d += nb + meta_bytes;
        CK(cudaStreamWaitEvent(s, qb.copied[b], 0));
        CK(cudaEventRecord(qb.k_begin[b], s));
        u64 *d_ctr = qb.d_ctr.as<u64>();
        if (nb)
            k_query_pack<<<(int)((nb_pad / 64 + THREADS - 1) / THREADS), THREADS, 0, s>>>(
                qb.d_text[b].as<unsigned char>(), nb, c_lo - t_lo, qb.d_bases.as<u64>(), qb.d_nmask.as<u64>(), d_ctr + 1);
        if (wn) {
            QueryArgs qa;
            qa.bases = qb.d_bases.as<u64>(); qa.nmask = qb.d_nmask.as<u64>();
            qa.n_words = nb_pad / 32; qa.n_mwords = nb_pad / 64;
            qa.qoff = qb.d_meta[b].as<u64>(); qa.woff = qa.qoff + nqc;
            qa.nq = nqc; qa.nw = wn;
            qa.table = v.table; qa.cap = v.cap;
            qa.out = qb.d_out.as<u32>() + w_base;
            qa.found = d_ctr;
            const uint64_t per_block = (uint64_t)THREADS * BATCH;
            k_query<<<(int)((wn + per_block - 1) / per_block), THREADS, 0, s>>>(qa, v.g, v.pt);
        }
        CK(cudaGetLastError());
        CK(cudaEventRecord(qb.k_end[b], s));
        qb.pending[b] = true;
        w_base += wn;
        i = j;
    }
    for (int b = 0; b < 2; b++) if ((rc = retire(b))) return rc;
    CK(cudaMemcpyAsync(hc, qb.d_ctr.p, 16, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    d2h += 16;
    if (hc[1] != ~0ull) {
        const uint64_t pos = t_lo + hc[1];
        const size_t qi = (size_t)(std::upper_bound(offsets, offsets + nq + 1, pos) - offsets) - 1;
        return fail(VDJGRAPH_ERR_BASE, "byte %llu of query %zu is outside ACGTN", (unsigned long long)(pos - offsets[qi]), qi);
    }
    /* every chunk passed the alphabet check: the answers to the caller (through page-locked chunks unless
     * its array is page-locked itself) */
    const uint64_t out_bytes = (uint64_t)n_windows * 4;
    if (out_bytes && is_page_locked(out, out_bytes)) {
        CK(cudaMemcpyAsync(out, qb.d_out.p, out_bytes, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
    } else if (out_bytes) {
        if ((rc = qb.text[0].ensure(CH)) || (rc = qb.text[1].ensure(CH))) return rc;
        const uint64_t n_parts = (out_bytes + CH - 1) / CH;
        for (uint64_t part = 0; part <= n_parts; part++) {
            if (part < n_parts) {   /* queue part, then hand over part - 1 while it copies */
                const uint64_t o = part * CH;
                CK(cudaMemcpyAsync(qb.text[part & 1].p, qb.d_out.as<char>() + o, std::min(CH, out_bytes - o), cudaMemcpyDeviceToHost, s));
                CK(cudaEventRecord(qb.copied[part & 1], s));
            }
            if (part > 0) {
                const uint64_t p = part - 1, o = p * CH;
                CK(cudaEventSynchronize(qb.copied[p & 1]));
                memcpy(reinterpret_cast<char *>(out) + o, qb.text[p & 1].p, std::min(CH, out_bytes - o));
            }
        }
    }
    d2h += out_bytes;
    if (stats) {
        stats->n_queries = nq; stats->n_windows = n_windows; stats->n_found = hc[0];
        stats->h2d_bytes = h2d; stats->d2h_bytes = d2h;
        stats->ms_kernels = ms_kernels;
        stats->ms_total = (float)(wall_ms() - t0);
    }
    return 0;
}

/* ========================================================================================== */
/* One graph over several devices of THIS process: the sharded phases above, driven by one host  */
/* thread per device inside the call (what vdjer_b200/shard.py does with one process per GPU).   */
/* ========================================================================================== */
struct vdjgraph_multi {
    int G = 0;
    bool device_barriers = false;           /* distinct devices: the steps of the finish meet in peer memory */
    std::vector<vdjgraph_ctx *> ctx;
    std::vector<int> dev;
    /* what the ranks exchange during a build */
    std::vector<uint64_t> hist;             /* [G][HIST_WORDS] */
    std::vector<uint8_t> hll;               /* [G][HLL_BYTES] */
    std::vector<uint64_t> counts, surv;     /* [G] */
    std::vector<void *> ptrs;               /* [G][NBUF] */
    std::vector<int> rounds;                /* [G]; 0 = this rank's plan failed */
    std::vector<int> rc;
    std::vector<std::string> err;
    std::atomic<int> failed{0};
    /* barrier of the G worker threads */
    std::mutex mu;
    std::condition_variable cv;
    int waiting = 0;
    uint64_t generation = 0;
    void barrier() {
        std::unique_lock<std::mutex> l(mu);
        const uint64_t g = generation;
        if (++waiting == G) { waiting = 0; generation++; cv.notify_all(); }
        else cv.wait(l, [&] { return generation != g; });
    }
};

namespace {

/* rank r's part of a build.  Every rank walks the same sequence of barriers whatever happens: a rank
 * whose library call failed records the status, skips its remaining calls and keeps meeting the others. */
void multi_worker(vdjgraph_multi *m, int r, const char *primary, size_t np, const char *secondary, size_t ns, int fwd) {
    vdjgraph_ctx *c = m->ctx[r];
    const int G = m->G;
    auto step = [&](int rc_) {
        if (rc_ && !m->rc[r]) { m->rc[r] = rc_; m->err[r] = g_err; m->failed = 1; }
        return rc_ == 0;
    };
    auto ok = [&] { return m->failed.load() == 0; };
    /* contiguous record ranges in rank order, even-sized: a read and its reverse complement stay together */
    const size_t rec_bytes = (size_t)2 * (size_t)c->prm.read_length + 1;
    const uint64_t total = ((uint64_t)np + ns) << fwd;
    uint64_t per = (total + G - 1) / G;
    per += per & 1;
    const uint64_t lo = std::min<uint64_t>(total, (uint64_t)r * per), hi = std::min<uint64_t>(total, (uint64_t)(r + 1) * per);
    const uint64_t lo_i = lo >> fwd, hi_i = hi >> fwd;      /* in items of the caller's buffers (records, or forward reads) */
    const uint64_t p_lo = std::min<uint64_t>(lo_i, np), p_hi = std::min<uint64_t>(hi_i, np);
    const uint64_t s_lo = std::max<uint64_t>(lo_i, np) - np, s_hi = std::max<uint64_t>(hi_i, np) - np;
    vdjgraph_shard_info info;
    info.n_ranks = (uint32_t)G; info.rank = (uint32_t)r; info.record_base = lo; info.total_records = total;
    m->counts[r] = hi - lo;
    const char *pp = primary ? primary + p_lo * rec_bytes : nullptr, *sp = secondary ? secondary + s_lo * rec_bytes : nullptr;
    if (ok()) step(fwd ? vdjgraph_shard_stage_forward(c, pp, p_hi - p_lo, sp, s_hi - s_lo, &info)
                       : vdjgraph_shard_stage(c, pp, p_hi - p_lo, sp, s_hi - s_lo, &info));
    if (ok()) step(vdjgraph_shard_count(c, m->hist.data() + (size_t)r * HIST_WORDS, m->hll.data() + (size_t)r * HLL_BYTES));
    m->barrier();
    m->rounds[r] = 0;
    if (ok()) {
        std::vector<uint8_t> merged(m->hll.begin(), m->hll.begin() + HLL_BYTES);   /* registers merge by maximum */
        for (int d = 1; d < G; d++)
            for (size_t i = 0; i < HLL_BYTES; i++) merged[i] = std::max(merged[i], m->hll[(size_t)d * HLL_BYTES + i]);
        if (step(vdjgraph_shard_plan(c, m->hist.data(), merged.data(), m->counts.data()))) m->rounds[r] = vdjgraph_shard_rounds(c);
    }
    if (ok()) step(vdjgraph_shard_buffers(c, m->ptrs.data() + (size_t)r * NBUF, nullptr));
    m->barrier();
    int n_rounds = m->rounds[0];
    for (int d = 0; d < G; d++) n_rounds = std::min(n_rounds, m->rounds[d]);    /* 0 when any rank has failed so far */
    if (n_rounds < 0) n_rounds = 0;
    if (ok()) step(vdjgraph_shard_set_peers(c, m->ptrs.data()));
    m->barrier();                                       /* nobody still uses a buffer that was replaced */
    if (ok()) step(vdjgraph_shard_release_retired(c));
    uint64_t n_surv = 0;
    for (int rnd = 0; rnd < n_rounds; rnd++) {
        if (rnd) m->barrier();                          /* the owners have consumed the previous round's runs */
        if (ok()) step(vdjgraph_shard_scatter(c));
        m->barrier();                                   /* every rank's runs of this round have arrived */
        if (ok()) step(vdjgraph_shard_passes(c, &n_surv));
    }
    m->surv[r] = n_surv;
    m->barrier();
    if (ok()) step(vdjgraph_shard_gather_plan(c, m->surv.data()));
    if (ok()) step(vdjgraph_shard_buffers(c, m->ptrs.data() + (size_t)r * NBUF, nullptr));
    m->barrier();                                       /* every exchange buffer exists, its barrier flags cleared */
    if (ok()) step(vdjgraph_shard_set_peers(c, m->ptrs.data()));
    for (int st = 0; st < 3; st++) {
        if (ok()) step(vdjgraph_shard_finish_step(c, st, m->device_barriers ? 1 : 0));
        if (!m->device_barriers) m->barrier();
    }
    if (ok()) step(vdjgraph_shard_finish(c));
    m->barrier();
    if (ok()) step(vdjgraph_shard_release_retired(c));
}

int multi_build(vdjgraph_multi *m, const char *primary, size_t np, const char *secondary, size_t ns, int fwd, vdjgraph_result *out) {
    if (!m || !out) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    if ((np && !primary) || (ns && !secondary)) return fail(VDJGRAPH_ERR_PARAM, "NULL record buffer");
    const int G = m->G;
    m->failed = 0;
    std::fill(m->rc.begin(), m->rc.end(), 0);
    for (auto &e : m->err) e.clear();
    std::vector<std::thread> th;
    for (int r = 1; r < G; r++) th.emplace_back(multi_worker, m, r, primary, np, secondary, ns, fwd);
    multi_worker(m, 0, primary, np, secondary, ns, fwd);
    for (auto &t : th) t.join();
    for (int r = 0; r < G; r++)
        if (m->rc[r]) return fail(m->rc[r], "device %d (rank %d of %d): %s", m->dev[r], r, G, m->err[r].c_str());
    return vdjgraph_fetch(m->ctx[0], out);
}

} // namespace

extern "C" int vdjgraph_multi_create(const vdjgraph_params *params, const int *devices, uint32_t n_devices, vdjgraph_multi **out) {
    if (!out) return fail(VDJGRAPH_ERR_PARAM, "out is NULL");
    *out = nullptr;
    if (!params || !devices) return fail(VDJGRAPH_ERR_PARAM, "NULL argument");
    if (n_devices < 1 || n_devices > (uint32_t)MAX_DEV || (n_devices & (n_devices - 1)))
        return fail(VDJGRAPH_ERR_PARAM, "n_devices %u must be 1, 2, 4 or 8", n_devices);
    vdjgraph_multi *m = new vdjgraph_multi();
    const int G = (int)n_devices;
    m->G = G;
    m->dev.assign(devices, devices + G);
    bool distinct = true;
    for (int a = 0; a < G; a++)
        for (int b = a + 1; b < G; b++) distinct = distinct && devices[a] != devices[b];
    /* the same device twice (tests on one GPU): host barriers, a kernel that waits for a peer on its own device
     * could keep that peer's kernels from starting */
    m->device_barriers = distinct && G > 1 && env_double("VDJGRAPH_HOST_BARRIERS", 0) == 0;
    m->hist.assign((size_t)G * HIST_WORDS, 0); m->hll.assign((size_t)G * HLL_BYTES, 0);
    m->counts.assign(G, 0); m->surv.assign(G, 0); m->ptrs.assign((size_t)G * NBUF, nullptr);
    m->rounds.assign(G, 0); m->rc.assign(G, 0); m->err.assign(G, std::string());
    int rc = 0;
    for (int r = 0; r < G && !rc; r++) {
        vdjgraph_params prm = *params;
        prm.device = devices[r];
        /* the ranks stage at the same time: they share the host's cores */
        if (!prm.host_threads && G > 1) prm.host_threads = (int32_t)std::max(2u, std::thread::hardware_concurrency() / (unsigned)G);
        vdjgraph_ctx *c = nullptr;
        rc = vdjgraph_create(&prm, &c);
        if (!rc) m->ctx.push_back(c);
    }
    for (int a = 0; a < G && !rc; a++)
        for (int b = 0; b < G && !rc; b++) rc = vdjgraph_enable_peer_access(devices[a], devices[b]);
    if (rc) { vdjgraph_multi_destroy(m); return rc; }
    *out = m;
    return 0;
}

extern "C" void vdjgraph_multi_destroy(vdjgraph_multi *m) {
    if (!m) return;
    for (vdjgraph_ctx *c : m->ctx) vdjgraph_destroy(c);
    delete m;
}

extern "C" int vdjgraph_multi_build(vdjgraph_multi *m, const char *primary, size_t np, const char *secondary, size_t ns,
                                    vdjgraph_result *out) {
    return multi_build(m, primary, np, secondary, ns, 0, out);
}

extern "C" int vdjgraph_multi_build_forward(vdjgraph_multi *m, const char *primary_reads, size_t np, const char *secondary_reads,
                                            size_t ns, vdjgraph_result *out) {
    return multi_build(m, primary_reads, np, secondary_reads, ns, 1, out);
}

extern "C" int vdjgraph_multi_stats(vdjgraph_multi *m, uint32_t rank, vdjgraph_result *out) {
    if (!m || rank >= (uint32_t)m->G) return fail(VDJGRAPH_ERR_PARAM, "bad argument");
    return vdjgraph_stats(m->ctx[rank], out);
}
