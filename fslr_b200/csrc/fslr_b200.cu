// fslr_b200 — B200 (sm_100a) implementation of the read-clustering step of kcleal/fslr.
//
// Replaces, behind the C ABI of include/fslr_b200.h, the reference calls of
// /root/reference/fslr/main.py:233-257,334-342 into /root/reference/fslr/cluster.py:
//   keep_fillings (cluster.py:14-31)           -> k_first_last, k_keep, k_fill_records
//   prepare_data + mask_sequences2 (:89-121)    -> k_mask_flags, k_compact_fillings, radix sort by start, k_build_items
//   query_intervals dict order (:189-191)       -> k_first_dp, k_is_first, scan, sort by query rank
//   build_interval_trees / IntervalMap (:124-130, third-party superintervals)
//                                               -> sort by (chrom, start, end desc, data order), k_ub, prefix-max of ends
//   query_interval_trees (:187-227)             -> k_pair (order-free relation + capped degree) and k_replay
//                                                  (reads that can reach edge_threshold, in query order)
//   different_lengths_or_alignments (:178-183), overall_jaccard_similarity (:140-170),
//   calculate_overlap (:133-136), cutoff lookup (:218-219)
//                                               -> integer thresholds T/Lq/Ln/umax (k_read_info, k_records, host umax)
//   get_subgraphs / networkx (:230-234)         -> k_union_entries, k_union_edges, k_flatten (lock-free union-find,
//                                                  root = smallest query rank = the component's first-inserted node)
//   cluster / n_reads columns (main.py:251-257,334-342) -> k_roots, k_number
//
// Why the sequential reference loop parallelises exactly (DESIGN.md §3): a filling's scan of
// search_values() results covers a contiguous run of sorted positions [stop, ub] walked downwards, so the
// loop state that later queries can observe is one integer per filling.  Reads whose number of passing
// candidates is below edge_threshold can never break: their stop is the chromosome start and their edges follow
// from the order-free relation.  The remaining reads are replayed in query order by a persistent ticket kernel in
// which a warp only ever waits for reads holding smaller tickets.
#include <cuda_runtime.h>
#include "prims.cuh"
#include "tsv.cuh"
#include <string>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <vector>
#include <algorithm>
#include "fslr_b200.h"

#define FSLRC_VERSION 1
#define LMAX FSLRC_MAX_FILLINGS
#define NCNT 56                 // device counters of one call (Pipe::cnt); the error word follows them in the pinned read-back

enum { EF_RANGE = 1, EF_ZERO = 2, EF_TOOMANY = 4, EF_NALN = 8, EF_OVERFLOW = 16 };

// ---------------------------------------------------------------- context
struct fslrc_ctx {
    int device;
    char err[512];
    cudaStream_t stream;
    std::vector<void *> allocs;
    int64_t *h_pin;          // pinned scratch for read-backs (64 x int64)
    cudaEvent_t ev[FSLRC_N_STAGES + 1];
    // pipeline state (kept between the fslrc_mg_* stages)
    struct Pipe *pipe;
    struct TsvState *tsv;    // parsed mappings.bed kept on the device between fslrc_tsv_open and fslrc_tsv_close
    cudaEvent_t ev_block;    // cudaEventBlockingSync event: waits that put the thread to sleep (fslrc_set_blocking_sync)
    int blocking;
    struct BamState *bam;    // table produced from a BAM file, kept on the device between fslrc_bam_open and fslrc_bam_close
    long long launches;      // kernels of this library launched since fslrc_create
    // host calls: the column the first kernels do not read (n_alignments) is uploaded on a second stream BEHIND the others, so the
    // tail of the upload overlaps keep_fillings (ev_c1: the other copies are done; ev_c2: this one is)
    cudaStream_t copy_stream;
    cudaEvent_t ev_c1, ev_c2;
    bool late_pending;
    int edge_capture;        // fslrc_set_edge_capture
    struct EdgeList *edges;  // edge list of the last clustering call (capture on), kept until the next one
    long long tsv_gen;       // bumped by fslrc_tsv_open / fslrc_tsv_delete_false: which parsed table a captured list names
    unsigned char *prim; size_t prim_bytes;   // scratch of the device-wide primitives: one of `allocs`, so free_all drops it
};
// the similarity graph of one clustering call, sorted by (query rank of read1, query rank of read2); device arrays
struct EdgeList {
    int32_t *read1, *read2;
    double *jac;
    int64_t n;
    const int32_t *read_id_col;  // the table's read_id column and ...
    long long tsv_gen;           // ... ctx->tsv_gen at the call: the renderer checks both against the parsed table
};
static void edges_free(fslrc_ctx *ctx) {
    if (!ctx->edges) return;
    void *p[] = {ctx->edges->read1, ctx->edges->read2, ctx->edges->jac};
    for (void *q : p) if (q) cudaFreeAsync(q, ctx->stream);
    delete ctx->edges; ctx->edges = nullptr;
}

static void tsv_free(fslrc_ctx *ctx);
static void bam_free(fslrc_ctx *ctx);
static const int32_t *tsv_read_id(const fslrc_ctx *ctx);

enum { ST_H2D = 0, ST_KEEP, ST_ORDER, ST_QRANK, ST_CHROM, ST_BANDS, ST_CAND, ST_PAIR, ST_HEAVY, ST_SAT, ST_REPLAY, ST_UNION, ST_NUMBER, ST_D2H };
static const char *STAGE_NAMES[FSLRC_N_STAGES] = {
    "h2d", "keep_fillings", "data_order_mask", "query_rank_read_lists", "chrom_sort", "records_bands",
    "candidates", "pair_kernel", "pair_heavy", "saturating_set", "replay", "union_find", "numbering", "d2h"};
static_assert(ST_D2H + 1 == FSLRC_N_STAGES, "stage list");

static int fail(fslrc_ctx *c, int code, const char *fmt, const char *a = "") {
    snprintf(c->err, sizeof(c->err), fmt, a);
    return code;
}
#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            snprintf(ctx->err, sizeof(ctx->err), "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
            return FSLRC_ERR_CUDA;                                                                 \
        }                                                                                          \
    } while (0)

template <typename T>
static int dalloc(fslrc_ctx *ctx, T **p, int64_t n) {
    void *q = nullptr;
    size_t bytes = (size_t)(n > 0 ? n : 1) * sizeof(T);
    CK(cudaMallocAsync(&q, bytes, ctx->stream));
    ctx->allocs.push_back(q);
    *p = (T *)q;
    return 0;
}
static void free_all(fslrc_ctx *ctx) {
    if (ctx->late_pending) { cudaStreamWaitEvent(ctx->stream, ctx->ev_c2, 0); ctx->late_pending = false; }   // (an error path got here first)
    for (void *p : ctx->allocs) cudaFreeAsync(p, ctx->stream);
    ctx->allocs.clear();
    ctx->prim = nullptr; ctx->prim_bytes = 0;
}
#define DA(ptr, n)                                  \
    do {                                            \
        int r__ = dalloc(ctx, &(ptr), (int64_t)(n)); \
        if (r__) return r__;                        \
    } while (0)

// the device arrays of a table kept on the device between calls (TsvState, BamState)
struct Resident {
    std::vector<void *> allocs;
};
template <typename T>
static int res_alloc(fslrc_ctx *ctx, Resident &m, T **p, int64_t n) {
    void *q = nullptr;
    CK(cudaMallocAsync(&q, (size_t)(n > 0 ? n : 1) * sizeof(T), ctx->stream));
    m.allocs.push_back(q);
    *p = (T *)q;
    return 0;
}
#define RA(m, ptr, n) do { int r__ = res_alloc(ctx, (m), &(ptr), (int64_t)(n)); if (r__) return r__; } while (0)
static void res_free(fslrc_ctx *ctx, Resident &m, void *p) {           // one array, stream-ordered
    std::vector<void *>::iterator it = std::find(m.allocs.begin(), m.allocs.end(), p);
    if (it != m.allocs.end()) { m.allocs.erase(it); cudaFreeAsync(p, ctx->stream); }
}
// the context's table *s (ctx->tsv, ctx->bam) and all its arrays
template <typename S>
static void drop_table(fslrc_ctx *ctx, S *&s) {
    if (!s) return;
    for (void *p : s->mem.allocs) cudaFreeAsync(p, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    delete s; s = nullptr;
}
// The cleanup of the calls on a resident table: a failing call frees its scratch and, when it is an open (drop: tsv_free,
// bam_free), the table it was building, so that the context never holds a half-built one.
template <typename F>
static int table_call(fslrc_ctx *ctx, void (*drop)(fslrc_ctx *), F &&body) {
    const int r = body();
    if (r) {
        free_all(ctx);
        if (drop) drop(ctx);
        cudaStreamSynchronize(ctx->stream);
    }
    return r;
}

// every launch of one of OUR kernels goes through KL so that the count can be reported (bench.py "gpu_launches")
#define KL(kernel, grid, block, ...)                         \
    do {                                                     \
        ctx->launches++;                                     \
        kernel<<<(grid), (block), 0, st>>>(__VA_ARGS__);     \
    } while (0)

static inline int nblk(int64_t n, int t) { return (int)((n + t - 1) / t); }

#include "kernels_ingest.cuh"
#include "kernels_pair.cuh"
#include "kernels_hits.cuh"
#include "kernels_replay.cuh"
#include "kernels_graph.cuh"
#include "bam.cuh"
#include "bam_chain.cuh"
#include "crc32.cuh"

// ================================================================ host pipeline
struct Pipe {
    // inputs (device)
    fslrc_table tb;
    fslrc_params pr;
    Widen w_late;            // host calls: the n_alignments column still on its way (ctx->copy_stream); widened by late_columns()
    bool late;
    int A, R, F, D, Q, nP, Tedge, pair_blocks;
    int *err;
    int64_t *cnt;            // device counters: 0 F,1 D,2 Q,3 band,4 tests,5 entry slots,6 nP,7 pedge slots,8 edges,9 ncl,10 forest,
                             //                  11 singletons, 12 runs, 13 entries, 14 tight band, 40-43 partner-record slots / stats,
                             //                  44 tight band of light positions, 45 light partner records, 46 heavy reads, 47 P-pairs (mg),
                             //                  48 largest start (fast ingest)
    int *q_of_rid, *rid_of_q;
    int4 *SR0, *SR1, *RM, *RI;
    int *pmaxS, *s_chrom, *chrom_lo, *chrom_hi;
    int *isP, *plist, *stop, *stopS;
    unsigned *cp;            // per light read: passing partners | partners << 16 | CP_LONG (k_eval), then k_plist's fill counter
    int *rclass, *heavy_list, *plcount, *ploff;
    int hits_blocks;
    int2 *entries, *pedges;
    int4 *PL; PLInfo *plinfo;
    unsigned long long cap_entries, cap_pedges, cap_pl;
    int *parent, *ing;
    unsigned *ticket;
    int stage;              // next event index
    Tab tab;
    UmaxTab um;
};

static int mark(fslrc_ctx *ctx, int stage_end) {   // record the event closing `stage_end`
    CK(cudaEventRecord(ctx->ev[stage_end + 1], ctx->stream));
    return 0;
}
// resident blocks per SM of a persistent (grid-stride) kernel: its grid is one full wave, never a wave and a bit
template <typename K>
static int resident_blocks(K kernel, int threads, size_t dyn_smem = 0) {
    int nb = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, dyn_smem) != cudaSuccess) { cudaGetLastError(); nb = 1; }
    return std::max(nb, 1);
}
static int n_sms(fslrc_ctx *ctx) {
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, ctx->device);
    return n;
}
// ---- device-wide primitives (prims.cuh): look-back status words + ticket live in one reusable scratch region
static int prim_scratch(fslrc_ctx *ctx, size_t status_bytes) {
    const size_t need = status_bytes + 256;
    if (need > ctx->prim_bytes) {
        void *q; const size_t nb = need + (need >> 1);
        CK(cudaMallocAsync(&q, nb, ctx->stream));
        ctx->allocs.push_back(q);
        ctx->prim = (unsigned char *)q; ctx->prim_bytes = nb;
    }
    CK(cudaMemsetAsync(ctx->prim, 0, need, ctx->stream));        // ticket (first 256 bytes) + status words
    return 0;
}
// exclusive sum of int32; *total (device, optional) receives the grand total
static int xscan(fslrc_ctx *ctx, const int *in, int *out, int n, int64_t *total = nullptr) {
    cudaStream_t st = ctx->stream;
    if (n <= 0) { if (total) CK(cudaMemsetAsync(total, 0, sizeof(int64_t), st)); return 0; }
    const int tiles = nblk(n, prims::SC_TILE);
    int r = prim_scratch(ctx, sizeof(unsigned long long) * tiles); if (r) return r;
    KL(prims::k_scan_excl<int>, tiles, prims::SC_THREADS, in, out, n, (unsigned long long *)(ctx->prim + 256), (unsigned *)ctx->prim, (long long *)total);
    return 0;
}
// exclusive sum of int64 (k_reads_fast's packed (count << 32 | L) flags, the line lengths of a text render)
static int xscan64(fslrc_ctx *ctx, const long long *in, long long *out, int n, int64_t *total) {
    cudaStream_t st = ctx->stream;
    if (n <= 0) { if (total) CK(cudaMemsetAsync(total, 0, sizeof(int64_t), st)); return 0; }
    const int tiles = nblk(n, prims::SC_TILE);
    int r = prim_scratch(ctx, sizeof(unsigned long long) * tiles); if (r) return r;
    KL(prims::k_scan_excl<long long>, tiles, prims::SC_THREADS, in, out, n, (unsigned long long *)(ctx->prim + 256), (unsigned *)ctx->prim, (long long *)total);
    return 0;
}
// per-segment inclusive prefix max (seg non-decreasing)
static int segmax_scan(fslrc_ctx *ctx, const int *seg, const int *val, int *out, int n) {
    cudaStream_t st = ctx->stream;
    if (n <= 0) return 0;
    const int tiles = nblk(n, prims::SC_TILE);
    int r = prim_scratch(ctx, sizeof(unsigned long long) * tiles); if (r) return r;
    KL(prims::k_scan_segmax, tiles, prims::SC_THREADS, seg, val, out, n, (unsigned long long *)(ctx->prim + 256), (unsigned *)ctx->prim);
    return 0;
}
// stable LSD radix sort of (key, value) pairs on key bits [b0, b1); the inputs are left untouched.  The last pass hands
// every pair to `last` with its output position; *last_start (optional) receives the start of every digit of that pass.
template <typename Out>
static int sort_pairs_to(fslrc_ctx *ctx, const unsigned *kin, const int *vin, int n, int b0, int b1, Out last,
                         const unsigned **last_start = nullptr) {
    cudaStream_t st = ctx->stream;
    if (n <= 0) return 0;
    const int npass = std::max(1, (b1 - b0 + 7) / 8);
    if (npass > 4) return fail(ctx, FSLRC_ERR_ARG, "radix sort: more than 32 key bits");
    unsigned *hist; DA(hist, 4 * 256);
    CK(cudaMemsetAsync(hist, 0, sizeof(unsigned) * 4 * 256, st));
    prims::PairOut tmp[2] = {};
    for (int k = 0; k < std::min(npass - 1, 2); k++) { DA(tmp[k].kout, n); DA(tmp[k].vout, n); }
    KL(prims::k_rs_hist, std::min(nblk(n, 256 * 16), n_sms(ctx) * 8), 256, kin, n, b0, b1, npass, hist);
    KL(prims::k_rs_scan, npass, 256, hist);
    const int tiles = nblk(n, prims::RS_TILE);
    const unsigned *ks = kin; const int *vs = vin;
    for (int p = 0; p < npass; p++) {
        int r = prim_scratch(ctx, sizeof(unsigned) * 256 * (size_t)tiles); if (r) return r;
        const int nbits = std::min(8, b1 - b0 - 8 * p);
        const unsigned *gb = hist + 256 * p;
        ctx->launches++;
        if (p == npass - 1) {
            prims::k_rs_onesweep<<<tiles, prims::RS_THREADS, sizeof(prims::RsSmem), st>>>(ks, vs, last, n, b0 + 8 * p, (1 << nbits) - 1, gb,
                                                                                          (unsigned *)(ctx->prim + 256), (unsigned *)ctx->prim);
        } else {
            const prims::PairOut o = tmp[p & 1];
            prims::k_rs_onesweep<<<tiles, prims::RS_THREADS, sizeof(prims::RsSmem), st>>>(ks, vs, o, n, b0 + 8 * p, (1 << nbits) - 1, gb,
                                                                                          (unsigned *)(ctx->prim + 256), (unsigned *)ctx->prim);
            ks = o.kout; vs = o.vout;
        }
    }
    if (last_start) *last_start = hist + 256 * (npass - 1);
    return 0;
}
static int sort_pairs(fslrc_ctx *ctx, const unsigned *kin, unsigned *kout, const int *vin, int *vout, int n, int b0, int b1) {
    return sort_pairs_to(ctx, kin, vin, n, b0, b1, prims::PairOut{kout, vout});
}
// wait for the context's stream: spinning (lowest latency) or, for contexts driven from several host threads at once
// (engine.HostPipeline), sleeping on a blocking-sync event so that a waiting thread leaves its core to the others
static cudaError_t ctx_sync(fslrc_ctx *ctx) {
    if (!ctx->blocking) return cudaStreamSynchronize(ctx->stream);
    cudaError_t e = cudaEventRecord(ctx->ev_block, ctx->stream);
    return e != cudaSuccess ? e : cudaEventSynchronize(ctx->ev_block);
}
static int read_counts(fslrc_ctx *ctx, Pipe *P) {   // device counters + error word -> pinned host
    CK(cudaMemcpyAsync(ctx->h_pin, P->cnt, NCNT * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_pin + NCNT, P->err, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx_sync(ctx));
    return 0;
}
static int err_code(fslrc_ctx *ctx) {
    int e = (int)(ctx->h_pin[NCNT] & 0xffffffff);
    if (!e) return 0;
    if (e & EF_RANGE) return fail(ctx, FSLRC_ERR_RANGE, "a table value is out of range (read_id/chrom id, negative coordinate, n_alignments >= 65535 or a bad `order`)");
    if (e & EF_ZERO) return fail(ctx, FSLRC_ERR_ZERO_DIVISOR, "aln_size, qlen2 or n_alignments <= 0 on a filling (the reference raises ZeroDivisionError)");
    if (e & EF_TOOMANY) return fail(ctx, FSLRC_ERR_TOO_MANY_FILLINGS, "a read has more than 64 fillings");
    if (e & EF_NALN) return fail(ctx, FSLRC_ERR_NALN_NOT_CONSTANT, "n_alignments is not constant over the rows of a read");
    return fail(ctx, FSLRC_ERR_OVERFLOW, "internal edge buffer overflow");
}
static int bits_for(int64_t n) { int b = 1; while ((1ll << b) < n && b < 32) b++; return b; }

static int alloc_records(fslrc_ctx *ctx, Pipe *P, int **s_m, int **s_end);
static int pipe_bands(fslrc_ctx *ctx, Pipe *P, const int *s_m, const int *s_end);

// IntervalMap order from data order (stage 4): one stable partition by chromosome + local tie fix, or — long runs of equal
// (chrom, start) — three stable sorts
static int pipe_chrom_order(fslrc_ctx *ctx, Pipe *P, const int4 *IT0, unsigned *tkey, unsigned *tval, bool tie_ok, int *s_dp) {
    cudaStream_t st = ctx->stream;
    const int D = P->D, TB = 256;
    if (D <= 0) return 0;
    if (tie_ok) {
        unsigned *tkey2, *tval2; DA(tkey2, D); DA(tval2, D);
        int r = sort_pairs(ctx, tkey, tkey2, (const int *)tval, (int *)tval2, D, 0, bits_for(P->pr.n_chrom)); if (r) return r;
        KL(k_apply_delta, nblk(D, TB), TB, D, tval2, s_dp);
    } else {
        // (chrom, start, end desc, data order) as three stable sorts from data order: ~end, start, chrom
        unsigned *ek, *ek2; int *v1, *v2, *iotaD;
        DA(ek, D); DA(ek2, D); DA(v1, D); DA(v2, D); DA(iotaD, D);
        KL(k_iota, nblk(D, TB), TB, iotaD, D);
        KL(k_end_keys, nblk(D, TB), TB, D, IT0, ek);
        int r = sort_pairs(ctx, ek, ek2, iotaD, v1, D, 0, 32); if (r) return r;
        KL(k_gather_key, nblk(D, TB), TB, D, v1, IT0, 0, ek);
        r = sort_pairs(ctx, ek, ek2, v1, v2, D, 0, 32); if (r) return r;
        KL(k_gather_key, nblk(D, TB), TB, D, v2, IT0, 1, ek);
        r = sort_pairs(ctx, ek, ek2, v2, s_dp, D, 0, bits_for(P->pr.n_chrom)); if (r) return r;
    }
    return 0;
}

// ---- stages 1-4, fast form (kernels_ingest.cuh: contiguous reads, no caller `order`).  Returns 1 when the table does not
// meet the precondition (nothing useful was computed: the caller runs the general path), 0 on success, < 0 on error.
// the column that was uploaded behind the others (resolve_columns): wait for it and widen it, right before its first reader
static int late_columns(fslrc_ctx *ctx, Pipe *P) {
    if (!P->late) return 0;
    cudaStream_t st = ctx->stream;
    CK(cudaStreamWaitEvent(st, ctx->ev_c2, 0));
    ctx->late_pending = false;
    P->late = false;
    if (P->A > 0) KL(k_widen, nblk(P->A, 256), 256, (int64_t)P->A, P->w_late);
    return 0;
}
static int pipe_ingest_fast(fslrc_ctx *ctx, Pipe *P, const long long *d_clen, const unsigned char *d_cmask) {
    const fslrc_table &tb = P->tb; const fslrc_params &pr = P->pr;
    cudaStream_t st = ctx->stream;
    const int A = P->A, R = P->R, TB = 256;
    int *flagA, *posA, *qlen2;
    long long *QO;                                                          // per read: q << 32 | off, -1 = no interval
    DA(flagA, A); DA(posA, A); DA(qlen2, R); DA(P->q_of_rid, R); DA(QO, R);
    if (R > 0) KL(k_fill<long long>, nblk(R, TB), TB, QO, R, -1ll);
    if (A > 0) {
        KL(k_rows_fast, nblk(A, TB), TB, A, R, tb.read_id, tb.chrom, tb.rstart, tb.rend, tb.qstart, tb.qend, pr.n_chrom, d_clen, d_cmask,
           pr.mask_subtelomere, (long long)pr.subtel, flagA, qlen2, (unsigned long long *)(P->cnt + 0), P->err);
        int r = xscan(ctx, flagA, posA, A, P->cnt + 1); if (r) return r;
    }
    { int r = read_counts(ctx, P); if (r) return r; }
    if (ctx->h_pin[NCNT] & EF_NONMONO) {                                    // rows of a read apart, or ids going down: general path
        CK(cudaMemsetAsync(P->err, 0, sizeof(int), st));
        CK(cudaMemsetAsync(P->cnt, 0, NCNT * sizeof(int64_t), st));
        return 1;
    }
    { int r = err_code(ctx); if (r) return r; }
    P->F = (int)ctx->h_pin[0];
    const int D = P->D = (int)ctx->h_pin[1];
    { int r = mark(ctx, ST_KEEP); if (r) return r; }
    int4 *REC, *IT0, *IT1; unsigned *key, *key2; int *val, *dfill; long long *flag64, *qo64;
    DA(REC, 2 * (int64_t)D); DA(key, D); DA(key2, D); DA(val, D); DA(dfill, D); DA(IT0, D); DA(IT1, D);
    DA(flag64, D); DA(qo64, D);
    unsigned *tkey = nullptr, *tval = nullptr;
    int kbits = 32;
    if (D > 0) {
        if (D >= (1 << 26)) return fail(ctx, FSLRC_ERR_RANGE, "more than 2^26 intervals");
        { int r = late_columns(ctx, P); if (r) return r; }
        KL(k_compact_fast, nblk(A, TB), TB, A, flagA, posA, tb.read_id, tb.chrom, tb.rstart, tb.rend, tb.aln_size, tb.n_alignments,
           REC, key, val, (unsigned long long *)(P->cnt + 48), P->err);
        // the genome bounds the sort key: 4 passes of 8 bits cover any int32 start, fewer when the chromosome lengths say so
        long long mx = 0; bool known = pr.n_chrom > 0;
        for (int c = 0; c < pr.n_chrom; c++) { if (pr.chrom_len[c] <= 0) known = false; mx = std::max<long long>(mx, pr.chrom_len[c]); }
        kbits = (known && mx < 0x7fffffffLL) ? std::min(32, bits_for(mx + 2)) : 32;
        int r = sort_pairs(ctx, key, key2, val, dfill, D, 0, kbits); if (r) return r;
        KL(k_items_fast, nblk(D, TB), TB, D, dfill, REC, IT0, IT1, flag64);
        DA(tkey, D); DA(tval, D);
        KL(k_tie_delta, nblk(D, TB), TB, D, IT0, tkey, tval, (unsigned long long *)(P->cnt + 41), P->err);
    }
    { int r = mark(ctx, ST_ORDER); if (r) return r; }
    // ---- query rank + read-major offsets from one scan over data order
    DA(P->RI, std::min(R, D));
    if (D > 0) {
        int r = xscan64(ctx, flag64, qo64, D, P->cnt + 2); if (r) return r;
        KL(k_firsts_fast, nblk(D, TB), TB, D, flag64, qo64, IT0, IT1, qlen2, pr.qlen_c, pr.naln_c, QO, P->RI, P->err);
    }
    if (R > 0) KL(k_q_of_rid, nblk(R, TB), TB, R, QO, P->q_of_rid);
    { int r = read_counts(ctx, P); if (r) return r; }
    if (kbits < 32 && ((unsigned long long)ctx->h_pin[48] >> kbits) != 0) {   // a start beyond its chromosome's length: the short sort key was
        CK(cudaMemsetAsync(P->err, 0, sizeof(int), st));                      // wrong (and data order with it: k_tie_delta's EF_RANGE), the
        CK(cudaMemsetAsync(P->cnt, 0, NCNT * sizeof(int64_t), st));           // general path sorts on all 32 bits
        return 1;
    }
    { int r = err_code(ctx); if (r) return r; }
    if (D > 0 && (ctx->h_pin[2] & 0xffffffffLL) != D) return fail(ctx, FSLRC_ERR_CUDA, "internal: read-major offsets do not add up");
    P->Q = (int)(ctx->h_pin[2] >> 32);
    { int r = mark(ctx, ST_QRANK); if (r) return r; }
    // ---- IntervalMap order and the records of sorted order
    int *s_m, *s_end;
    { int r = alloc_records(ctx, P, &s_m, &s_end); if (r) return r; }
    const FastRec rec{IT0, IT1, QO, P->RI, pr.overlap, P->SR0, P->SR1, s_m, P->s_chrom, s_end};
    if (D > 0 && ctx->h_pin[41] == 0) {                                      // partition by chromosome, moving the records
        const int cbits = bits_for(pr.n_chrom);
        const unsigned *cstart = nullptr;
        int r = sort_pairs_to(ctx, tkey, (const int *)tval, D, 0, cbits, ChromRecOut{rec}, &cstart); if (r) return r;
        if (cbits <= 8) KL(k_chrom_bounds_digits, 1, 256, pr.n_chrom, D, cstart, P->chrom_lo, P->chrom_hi);
        else KL(k_chrom_bounds, nblk(D, TB), TB, D, P->s_chrom, P->chrom_lo, P->chrom_hi);
    } else if (D > 0) {                                                      // long runs of equal (chrom, start): three full sorts
        int *s_dp; DA(s_dp, D);
        int r = pipe_chrom_order(ctx, P, IT0, tkey, tval, false, s_dp); if (r) return r;
        KL(k_records_fast, nblk(D, TB), TB, D, s_dp, rec);
        KL(k_chrom_bounds, nblk(D, TB), TB, D, P->s_chrom, P->chrom_lo, P->chrom_hi);
    }
    { int r = mark(ctx, ST_CHROM); if (r) return r; }
    return pipe_bands(ctx, P, s_m, s_end);
}

// ---- stage 1 of the general ingest, keep_fillings (cluster.py:14-31): flagA[i] = 1 for every row that is neither the first
// nor the last row of its read by occurrence (the rows of a read need not be contiguous), posA[i] = its filling index in bed
// order, P->cnt[0] = the number of fillings.  qmin / qmax: per read the smallest qstart / largest qend over its kept rows, or
// NULL (the flags only).  A read id outside [0, R) sets EF_RANGE.
static int keep_rows(fslrc_ctx *ctx, Pipe *P, const int *rid, const int *qstart, const int *qend, int *flagA, int *posA,
                     int *qmin, int *qmax) {
    cudaStream_t st = ctx->stream;
    const int A = P->A, R = P->R, TB = 256;
    int *first, *last;
    DA(first, R); DA(last, R);
    if (R > 0) {
        KL(k_fill<int>, nblk(R, TB), TB, first, R, 0x7fffffff);
        KL(k_fill<int>, nblk(R, TB), TB, last, R, -1);
        if (qmin) {
            KL(k_fill<int>, nblk(R, TB), TB, qmin, R, 0x7fffffff);
            KL(k_fill<int>, nblk(R, TB), TB, qmax, R, (int)0x80000000);
        }
    }
    if (A > 0) {
        KL(k_first_last, nblk(A, TB), TB, A, R, rid, first, last, P->err);
        KL(k_keep, nblk(A, TB), TB, A, R, rid, first, last, qstart, qend, flagA, qmin, qmax);
        return xscan(ctx, flagA, posA, A, P->cnt + 0);
    }
    return 0;
}

// ---- stages 1-5: ingestion, orders, records (replicated on every rank)
static int pipe_prepare(fslrc_ctx *ctx, Pipe *P) {
    const fslrc_table &tb = P->tb; const fslrc_params &pr = P->pr;
    cudaStream_t st = ctx->stream;
    const int A = P->A, R = P->R, TB = 256;
    DA(P->err, 1); DA(P->cnt, NCNT);
    CK(cudaMemsetAsync(P->err, 0, sizeof(int), st));
    CK(cudaMemsetAsync(P->cnt, 0, NCNT * sizeof(int64_t), st));
    long long *d_clen; unsigned char *d_cmask;
    DA(d_clen, pr.n_chrom); DA(d_cmask, pr.n_chrom);
    if (pr.n_chrom > 0) {
        CK(cudaMemcpyAsync(d_clen, pr.chrom_len, sizeof(int64_t) * pr.n_chrom, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_cmask, pr.chrom_masked, pr.n_chrom, cudaMemcpyHostToDevice, st));
    }
    if (!tb.order && !getenv("FSLRC_GENERAL_INGEST")) {
        const int r = pipe_ingest_fast(ctx, P, d_clen, d_cmask);
        if (r <= 0) return r;
    }
    // ---- stage 1: keep_fillings
    int *qmin, *qmax, *flagA, *posA;
    DA(qmin, R); DA(qmax, R); DA(flagA, A); DA(posA, A);
    DA(P->q_of_rid, R);
    if (R > 0) KL(k_fill<int>, nblk(R, TB), TB, P->q_of_rid, R, -1);
    { int r = keep_rows(ctx, P, tb.read_id, tb.qstart, tb.qend, flagA, posA, qmin, qmax); if (r) return r; }
    { int r = read_counts(ctx, P); if (r) return r; r = err_code(ctx); if (r) return r; }
    const int F = P->F = (int)ctx->h_pin[0];
    if (tb.order && tb.n_order != F) return fail(ctx, FSLRC_ERR_ARG, "order has the wrong length (must equal the number of fillings)");
    int4 *FR0; int2 *FR1;
    DA(FR0, F); DA(FR1, F);
    { int r = late_columns(ctx, P); if (r) return r; }
    if (A > 0) KL(k_fill_records, nblk(A, TB), TB, A, flagA, posA, tb.read_id, tb.chrom, tb.rstart, tb.rend, tb.aln_size, tb.n_alignments,
                  pr.n_chrom, FR0, FR1, P->err);
    { int r = mark(ctx, ST_KEEP); if (r) return r; }
    // ---- stage 2: mask (cluster.py:89-106; dropping masked fillings before or after the sort is the same list) + data order
    // (cluster.py:114): the caller's permutation, or a stable radix sort by start (ties keep bed order)
    int *flagF, *posF;
    DA(flagF, F); DA(posF, F);
    if (F > 0) {
        KL(k_mask_flags, nblk(F, TB), TB, F, tb.order, FR0, pr.n_chrom, d_clen, d_cmask, pr.mask_subtelomere, (long long)pr.subtel, flagF, P->err);
        int r = xscan(ctx, flagF, posF, F, P->cnt + 1); if (r) return r;
    }
    { int r = read_counts(ctx, P); if (r) return r; r = err_code(ctx); if (r) return r; }
    const int D = P->D = (int)ctx->h_pin[1];
    int *dfill; DA(dfill, D);
    if (tb.order) {
        if (F > 0) KL(k_compact_fillings, nblk(F, TB), TB, F, tb.order, flagF, posF, FR0, (int *)nullptr, dfill);
    } else {
        int *key, *key2, *v; DA(key, D); DA(key2, D); DA(v, D);
        if (F > 0) KL(k_compact_fillings, nblk(F, TB), TB, F, (const int *)nullptr, flagF, posF, FR0, key, v);
        int r = sort_pairs(ctx, (const unsigned *)key, (unsigned *)key2, v, dfill, D, 0, 32); if (r) return r;
    }
    int4 *IT0; int2 *IT1; int *firstdp;
    DA(IT0, D); DA(IT1, D); DA(firstdp, R);
    if (R > 0) KL(k_fill<int>, nblk(R, TB), TB, firstdp, R, 0x7fffffff);
    unsigned *tkey = nullptr, *tkey2 = nullptr, *tval = nullptr, *tval2 = nullptr;
    if (D > 0) KL(k_build_items, nblk(D, TB), TB, D, dfill, FR0, FR1, IT0, IT1, firstdp, P->err);
    if (D > 0 && D < (1 << 26)) {
        DA(tkey, D); DA(tkey2, D); DA(tval, D); DA(tval2, D);
        KL(k_tie_delta, nblk(D, TB), TB, D, IT0, tkey, tval, (unsigned long long *)(P->cnt + 41), P->err);
    }
    { int r = mark(ctx, ST_ORDER); if (r) return r; }
    // ---- stage 3: query rank + per-read lists
    int *flagD, *posD, *it_q;
    DA(flagD, D); DA(posD, D); DA(it_q, D);
    if (D > 0) {
        KL(k_is_first, nblk(D, TB), TB, D, IT0, firstdp, flagD);
        int r = xscan(ctx, flagD, posD, D, P->cnt + 2); if (r) return r;
    }
    { int r = read_counts(ctx, P); if (r) return r; r = err_code(ctx); if (r) return r; }
    const int Q = P->Q = (int)ctx->h_pin[2];
    DA(P->rid_of_q, Q);
    int *qs, *rm_dp, *iotaD, *rmidx, *off, *len_end;
    DA(qs, D); DA(rm_dp, D); DA(iotaD, D); DA(rmidx, D); DA(off, Q); DA(len_end, Q);
    DA(P->RI, Q);
    if (R > 0) KL(k_rank_reads, nblk(R, TB), TB, R, firstdp, posD, P->q_of_rid, P->rid_of_q);
    if (D > 0) {
        KL(k_item_q, nblk(D, TB), TB, D, IT0, P->q_of_rid, it_q);
        KL(k_iota, nblk(D, TB), TB, iotaD, D);
        int r = sort_pairs(ctx, (const unsigned *)it_q, (unsigned *)qs, iotaD, rm_dp, D, 0, bits_for(Q)); if (r) return r;
        KL(k_read_bounds, nblk(D, TB), TB, D, qs, rm_dp, rmidx, off, len_end);
        KL(k_read_info, nblk(Q, TB), TB, Q, P->rid_of_q, off, len_end, rm_dp, IT1, qmin, qmax, pr.qlen_c, pr.naln_c, P->RI, P->err);
    }
    { int r = mark(ctx, ST_QRANK); if (r) return r; }
    // ---- stage 4: IntervalMap order: (chrom, start asc, end desc, data order)
    int *s_dp; DA(s_dp, D);
    { int r = pipe_chrom_order(ctx, P, IT0, tkey, tval, tkey && ctx->h_pin[41] == 0, s_dp); if (r) return r; }   // (flag read back with the stage-3 counters)
    { int r = mark(ctx, ST_CHROM); if (r) return r; }
    int *s_m, *s_end;
    { int r = alloc_records(ctx, P, &s_m, &s_end); if (r) return r; }
    if (D >= (1 << 26)) return fail(ctx, FSLRC_ERR_RANGE, "more than 2^26 intervals");
    if (D > 0) KL(k_records, nblk(D, TB), TB, D, s_dp, rmidx, it_q, IT0, IT1, P->RI, pr.overlap, P->SR0, P->SR1,
                  s_m, P->s_chrom, s_end, P->chrom_lo, P->chrom_hi, P->err);
    return pipe_bands(ctx, P, s_m, s_end);
}

// ---- records of sorted order (written by the ingest that computed the order): SR0, SR1, s_m, s_chrom, s_end, chrom bounds
static int alloc_records(fslrc_ctx *ctx, Pipe *P, int **s_m, int **s_end) {
    const int D = P->D, nc = P->pr.n_chrom;
    cudaStream_t st = ctx->stream;
    DA(P->SR0, D); DA(P->SR1, D); DA(P->s_chrom, D); DA(*s_end, D); DA(*s_m, D);
    DA(P->chrom_lo, nc); DA(P->chrom_hi, nc);
    if (nc > 0) { CK(cudaMemsetAsync(P->chrom_lo, 0, sizeof(int) * nc, st)); CK(cudaMemsetAsync(P->chrom_hi, 0, sizeof(int) * nc, st)); }
    return 0;
}
// ---- stage 5: thresholds, bands; sizes of the pair stage's buffers
static int pipe_bands(fslrc_ctx *ctx, Pipe *P, const int *s_m, const int *s_end) {
    const fslrc_params &pr = P->pr;
    cudaStream_t st = ctx->stream;
    const int D = P->D, Q = P->Q;
    DA(P->RM, 2 * (int64_t)D); DA(P->pmaxS, D); DA(P->rclass, Q);
    if (D > 0) {
        int r = segmax_scan(ctx, P->s_chrom, s_end, P->pmaxS, D); if (r) return r;
        CK(cudaMemsetAsync(P->rclass, 0, sizeof(int) * (size_t)std::max(Q, 1), st));
        KL(k_bands, nblk(D, 256), 256, D, P->SR0, s_m, P->s_chrom, P->pmaxS, P->chrom_lo, P->chrom_hi, P->RM, P->rclass,
           (unsigned long long *)(P->cnt + 3), (unsigned long long *)(P->cnt + 14), (unsigned long long *)(P->cnt + 44));
    }
    { int r = read_counts(ctx, P); if (r) return r; r = err_code(ctx); if (r) return r; }
    long long T = pr.edge_threshold;
    P->Tedge = T > 0x7fffffffLL ? 0x7fffffff : (T < -0x7fffffffLL ? -0x7fffffff : (int)T);
    Tab &t = P->tab;
    t.SR0 = P->SR0; t.SR1 = P->SR1; t.RM = P->RM; t.RI = P->RI; t.pmaxS = P->pmaxS;
    t.chrom_lo = P->chrom_lo; t.chrom_hi = P->chrom_hi; t.sib = nullptr; t.D = D; t.Q = Q; t.Tedge = P->Tedge;
    memcpy(P->um.v, pr.umax, sizeof(P->um.v));
    // hit / relation-entry slots: k_hits lists at most one hit per (light position, tight-band position) pair; k_pair records
    // for a heavy read at most edge_threshold + 7 passing partners (one step past the threshold), each a distinct
    // (filling of a, band position) hit
    const unsigned long long tight = (unsigned long long)ctx->h_pin[14], lightT = (unsigned long long)ctx->h_pin[44];
    unsigned long long capT = P->Tedge > 0 ? (unsigned long long)Q * ((unsigned long long)P->Tedge + 7ull) : 0ull;
    P->pair_blocks = std::max(1, std::min(nblk(Q, PK_GROUPS), n_sms(ctx) * resident_blocks(k_pair<false>, PK_WARPS * 32)));
    P->hits_blocks = std::max(1, std::min(nblk(Q, HK_GROUPS), n_sms(ctx) * resident_blocks(k_hits, HK_WARPS * 32)));
    P->cap_entries = std::min<unsigned long long>(lightT + capT, tight) + (unsigned long long)PK_CHUNK * PK_WARPS * P->pair_blocks +
                     (unsigned long long)HK_CHUNK * HK_WARPS * P->hits_blocks + 64;
    DA(P->entries, P->cap_entries);
    DA(P->cp, Q); DA(P->heavy_list, Q); DA(P->plcount, Q); DA(P->ploff, Q);
    // partner records of saturating reads (replay LIST mode): at most RP_K per read and never more than tight-band hits
    P->cap_pl = std::min<unsigned long long>((unsigned long long)Q * RP_K, tight) + (unsigned long long)PL_CHUNK * PK_WARPS * P->pair_blocks * 2 + 64;
    DA(P->PL, 2 * P->cap_pl); DA(P->plinfo, Q);
    DA(P->isP, Q); DA(P->stop, D); DA(P->stopS, D); DA(P->parent, Q); DA(P->ing, Q); DA(P->ticket, 1);
    if (Q > 0) CK(cudaMemsetAsync(P->isP, 0, sizeof(int) * Q, st));
    return mark(ctx, ST_BANDS);
}


// ---- stage 6: pair stage on one shard: k_hits -> k_eval for the light reads, k_pair for the heavy ones (--overlap <= 0: all)
static int pipe_pair(fslrc_ctx *ctx, Pipe *P, int shard, int nshard) {
    cudaStream_t st = ctx->stream;
    const bool dense = P->Q > 0 && P->pr.overlap > 0.0;
    if (P->Q > 0) CK(cudaMemsetAsync(P->cp, 0, sizeof(unsigned) * (size_t)P->Q, st));
    if (dense) {
        KL(k_heavy_list, nblk(P->Q, 256), 256, P->tab, P->rclass, P->heavy_list, (unsigned *)(P->cnt + 46));
        KL(k_hits, std::max(1, std::min(nblk((P->Q + nshard - 1) / nshard + 256, HK_GROUPS), P->hits_blocks)), HK_WARPS * 32, P->tab, shard, nshard, P->rclass,
           (const unsigned *)(P->cnt + 46), P->entries, (unsigned long long *)(P->cnt + 5), P->cap_entries, P->err);
    }
    { int r = mark(ctx, ST_CAND); if (r) return r; }
    if (dense)
        KL(k_eval, n_sms(ctx) * resident_blocks(k_eval, EV_THREADS), EV_THREADS, P->tab, P->um, P->entries, (const unsigned *)(P->cnt + 46),
           (const unsigned long long *)(P->cnt + 5), P->cap_entries, P->cp,
           (unsigned long long *)(P->cnt + 4), (unsigned long long *)(P->cnt + 13));
    { int r = mark(ctx, ST_PAIR); if (r) return r; }
#define PAIR_ARGS P->isP, P->entries, (unsigned long long *)(P->cnt + 5), P->cap_entries, P->PL, P->plinfo, (unsigned long long *)(P->cnt + 40), \
                  P->cap_pl, (unsigned long long *)(P->cnt + 4), (unsigned long long *)(P->cnt + 13), P->err
    if (dense)
        KL(k_pair<false>, P->pair_blocks, PK_WARPS * 32, P->tab, P->um, shard, nshard, (const int *)P->heavy_list, (const unsigned *)(P->cnt + 46), PAIR_ARGS);
    else if (P->Q > 0)
        KL(k_pair<true>, P->pair_blocks, PK_WARPS * 32, P->tab, P->um, shard, nshard, (const int *)nullptr, (const unsigned *)nullptr, PAIR_ARGS);
#undef PAIR_ARGS
    return mark(ctx, ST_HEAVY);
}
// ---- stage 7a (after the counters are complete): saturating set of the light reads, where their partner records go
static int pipe_sat(fslrc_ctx *ctx, Pipe *P) {
    cudaStream_t st = ctx->stream;
    const int Q = P->Q, TB = 256;
    if (Q > 0 && P->pr.overlap > 0.0) {
        KL(k_light_sat, nblk(Q, TB), TB, P->tab, P->rclass, P->cp, P->isP, P->plinfo, P->plcount, (unsigned long long *)(P->cnt + 40));
        int r = xscan(ctx, P->plcount, P->ploff, Q, P->cnt + 45); if (r) return r;
        KL(k_plinfo, nblk(Q, TB), TB, Q, P->plcount, P->ploff, P->plinfo, (unsigned long long *)(P->cnt + 40), P->cnt + 45, P->cap_pl, P->err);
    }
    return 0;
}

// ---- stages 7-9 (after isP is complete): saturating set, replay, union-find
// pairs / n_pairs: the recorded pairs of light saturating reads of ALL ranks (multi-GPU, after the all-gather); NULL: this
// context's own list holds them all
static int pipe_replay_union(fslrc_ctx *ctx, Pipe *P, int shard, int nshard, const int2 *pairs, unsigned long long n_pairs) {
    cudaStream_t st = ctx->stream;
    const int Q = P->Q, D = P->D, TB = 256;
    int *posQ;
    DA(posQ, Q);
    if (Q > 0 && P->pr.overlap > 0.0) {                                   // partner records of the light saturating reads
        if (pairs) { if (n_pairs > 0) KL(k_plist, std::min(nblk((int64_t)n_pairs, PLT_THREADS), n_sms(ctx) * resident_blocks(k_plist, PLT_THREADS)), PLT_THREADS, P->tab, pairs,
                                       (const unsigned long long *)nullptr, n_pairs, n_pairs, P->plinfo, P->isP, P->cp, P->PL, P->err); }
        else KL(k_plist, n_sms(ctx) * resident_blocks(k_plist, PLT_THREADS), PLT_THREADS, P->tab, (const int2 *)P->entries, (const unsigned long long *)(P->cnt + 5), 0ull,
                P->cap_entries, P->plinfo, P->isP, P->cp, P->PL, P->err);
    }
    if (Q > 0) {
        int r = xscan(ctx, P->isP, posQ, Q, P->cnt + 6); if (r) return r;
    }
    { int r = read_counts(ctx, P); if (r) return r; r = err_code(ctx); if (r) return r; }
    const int nP = P->nP = (int)ctx->h_pin[6];
    DA(P->plist, nP);
    if (Q > 0) KL(k_compact_flagged, nblk(Q, TB), TB, Q, P->isP, posQ, P->plist);
    // stops: a read that never breaks walks every filling's scan to the chromosome start (0 <= any position)
    if (D > 0) { CK(cudaMemsetAsync(P->stop, 0, sizeof(int) * D, st)); CK(cudaMemsetAsync(P->stopS, 0, sizeof(int) * D, st)); }
    CK(cudaMemsetAsync(P->ticket, 0, sizeof(unsigned), st));
    { int r = mark(ctx, ST_SAT); if (r) return r; }
    // a saturating read adds at most edge_threshold edges in the scan that reaches the threshold and one per later filling
    const int replay_blocks_max = n_sms(ctx) * 16;
    const int list_blocks_max = n_sms(ctx) * resident_blocks(k_replay_list, RL_WARPS * 32);
    unsigned long long capp = (unsigned long long)nP * ((unsigned long long)std::max(P->Tedge, 0) + LMAX) + 64;
    unsigned long long alt = 2ull * (unsigned long long)ctx->h_pin[3] + 64;
    P->cap_pedges = std::min(capp, alt) + (unsigned long long)RP_CHUNK * std::max(RG_GROUPS * (replay_blocks_max + 1), RL_WARPS * (list_blocks_max + 1));
    DA(P->pedges, P->cap_pedges);
    if (nP > 0) {
        int *sflag, *spos, *sstart, *rflag, *rpos, *rstart;
        DA(sflag, nP); DA(spos, nP); DA(sstart, nP); DA(rflag, nP); DA(rpos, nP); DA(rstart, nP);
        const bool walk = !(P->pr.overlap > 0.0) || ctx->h_pin[43] != 0;   // some read without partner records?
        int4 *RH = nullptr;
        if (!walk) DA(RH, 3 * (int64_t)nP);
        KL(k_run_flags, nblk(nP, TB), TB, nP, P->plist, P->RI, P->RM, sflag, P->stop, P->stopS, P->plinfo, P->tab.chrom_lo, RH);
        int r = xscan(ctx, sflag, spos, nP, P->cnt + 15); if (r) return r;
        KL(k_compact_flagged, nblk(nP, TB), TB, nP, sflag, spos, sstart);
        KL(k_run_cut, nblk(nP, TB), TB, nP, sflag, spos, sstart, P->cnt + 15, rflag);
        r = xscan(ctx, rflag, rpos, nP, P->cnt + 12); if (r) return r;
        KL(k_compact_flagged, nblk(nP, TB), TB, nP, rflag, rpos, rstart);
        r = read_counts(ctx, P); if (r) return r;
        const int nRuns = (int)ctx->h_pin[12];
        int blocks = std::min(nblk(nRuns, RG_GROUPS), replay_blocks_max);
        int *wboard = nullptr;                                               // job board of the long skip walks (kernels_replay.cuh)
        if (walk) { DA(wboard, WB_SLOTS * WB_STRIDE); CK(cudaMemsetAsync(wboard, 0, sizeof(int) * WB_SLOTS * WB_STRIDE, st)); }
        if (walk && D > 0) {
            int *sib; DA(sib, D);
            KL(k_sib, nblk(D, TB), TB, D, P->SR0, P->SR1, P->RM, sib);
            P->tab.sib = sib;
        }
#define REPLAY_ARGS P->tab, P->um, nP, P->plist, nRuns, rstart, P->isP, P->PL, P->plinfo, P->stop, P->stopS, P->ticket, P->pedges, \
                    (unsigned long long *)(P->cnt + 7), P->cap_pedges, (unsigned long long *)(P->cnt + 4), P->err, (unsigned long long *)(P->cnt + 16), \
                    wboard, (unsigned *)(P->cnt + 51), (unsigned *)(P->cnt + 49), (unsigned long long *)(P->cnt + 50)
        if (!(P->pr.overlap > 0.0)) KL((k_replay<true, true>), blocks, RG_WARPS * 32, REPLAY_ARGS);
        else if (walk) KL((k_replay<false, true>), blocks, RG_WARPS * 32, REPLAY_ARGS);
        else if (getenv("FSLRC_REPLAY_GROUPS")) KL((k_replay<false, false>), std::min(nblk(nRuns, RG_GROUPS), n_sms(ctx) * 16), RG_WARPS * 32, REPLAY_ARGS);
        else KL(k_replay_list, std::min(nblk(nRuns, RL_WARPS), list_blocks_max), RL_WARPS * 32, P->tab, nP, RH, nRuns, rstart, P->isP, P->PL,
                P->stop, P->stopS, P->ticket, P->pedges, (unsigned long long *)(P->cnt + 7), P->cap_pedges, P->err, (unsigned long long *)(P->cnt + 16));
#undef REPLAY_ARGS
    }
    { int r = mark(ctx, ST_REPLAY); if (r) return r; }
    { int r = read_counts(ctx, P); if (r) return r; r = err_code(ctx); if (r) return r; }
    const unsigned long long nent = std::min<unsigned long long>((unsigned long long)ctx->h_pin[5], P->cap_entries);
    const unsigned long long nped = std::min<unsigned long long>((unsigned long long)ctx->h_pin[7], P->cap_pedges);
    if (Q > 0) {
        KL(k_iota, nblk(Q, TB), TB, P->parent, Q);
        CK(cudaMemsetAsync(P->ing, 0, sizeof(int) * Q, st));
    }
    if (nent > 0) KL(k_union_entries, nblk((int64_t)nent, UE_THREADS * UE_PER), UE_THREADS, nent, P->entries, P->isP, P->tab, P->stop, P->parent, P->ing,
                                                                           (unsigned long long *)(P->cnt + 8));
    // replayed edges are identical on every rank; rank 0 contributes them once
    if (nped > 0 && shard == 0) KL(k_union_edges, nblk((int64_t)nped, TB), TB, nped, P->pedges, P->parent, P->ing, (unsigned long long *)(P->cnt + 8));
    (void)nshard;
    return mark(ctx, ST_UNION);
}

// ---- stage 10: numbering
static int pipe_number(fslrc_ctx *ctx, Pipe *P, int *out_cluster, int *out_n) {
    cudaStream_t st = ctx->stream;
    const int Q = P->Q, R = P->R, TB = 256;
    int *isroot, *cidx, *csize, *sflag, *spos;
    DA(isroot, Q); DA(cidx, Q); DA(csize, Q); DA(sflag, R); DA(spos, R);
    if (Q > 0) {
        CK(cudaMemsetAsync(csize, 0, sizeof(int) * Q, st));
        KL(k_flatten, nblk(Q, TB), TB, Q, P->parent, P->ing, isroot, csize);
        int r = xscan(ctx, isroot, cidx, Q, P->cnt + 9); if (r) return r;
    }
    if (R > 0) {
        KL(k_single_flags, nblk(R, TB), TB, R, P->q_of_rid, P->ing, sflag);
        int r = xscan(ctx, sflag, spos, R, P->cnt + 11); if (r) return r;
        KL(k_number, nblk(R, TB), TB, R, P->q_of_rid, P->ing, P->parent, cidx, csize, spos, P->cnt + 9, out_cluster, out_n);
    }
    return mark(ctx, ST_NUMBER);
}

// ---- edge capture (after union-find, before the scratch goes): the directed edges of the relation entries and of the replay,
// which k_union_entries / k_union_edges handed to union-find, with their Jaccard similarity, in query-rank order
static int export_edges(fslrc_ctx *ctx, Pipe *P, const int32_t *read_id_col) {
    cudaStream_t st = ctx->stream;
    const int Q = P->Q, R = P->R, TB = 256;
    { int r = read_counts(ctx, P); if (r) return r; r = err_code(ctx); if (r) return r; }
    const long long E = ctx->h_pin[8];
    if (E > 0x7ffffff0LL) return fail(ctx, FSLRC_ERR_OVERFLOW, "edge capture: more than 2^31 edges");
    const unsigned long long nent = std::min<unsigned long long>((unsigned long long)ctx->h_pin[5], P->cap_entries);
    const unsigned long long nped = std::min<unsigned long long>((unsigned long long)ctx->h_pin[7], P->cap_pedges);
    const int n = (int)E;
    EdgeList *L = new EdgeList();
    memset(L, 0, sizeof(*L));
    L->n = n; L->read_id_col = read_id_col;
    L->tsv_gen = (read_id_col && read_id_col == tsv_read_id(ctx)) ? ctx->tsv_gen : -1;
    ctx->edges = L;
    CK(cudaMallocAsync((void **)&L->read1, sizeof(int32_t) * (size_t)std::max(n, 1), st));
    CK(cudaMallocAsync((void **)&L->read2, sizeof(int32_t) * (size_t)std::max(n, 1), st));
    CK(cudaMallocAsync((void **)&L->jac, sizeof(double) * (size_t)std::max(n, 1), st));
    int2 *dir; unsigned long long *cnt; int *rid_of_q, *iota, *perm1, *perm; unsigned *key, *key2;
    DA(dir, n); DA(cnt, 1); DA(rid_of_q, Q); DA(iota, n); DA(perm1, n); DA(perm, n); DA(key, n); DA(key2, n);
    CK(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), st));
    if (nent > 0) KL(k_edges_of_entries, nblk((int64_t)nent, TB), TB, nent, P->entries, P->isP, P->tab, P->stop, dir, (unsigned long long)n, cnt);
    if (nped > 0) KL(k_edges_of_pedges, nblk((int64_t)nped, TB), TB, nped, P->pedges, dir, (unsigned long long)n, cnt);
    CK(cudaMemcpyAsync(ctx->h_pin + 60, cnt, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(ctx_sync(ctx));
    if (ctx->h_pin[60] != E) return fail(ctx, FSLRC_ERR_OVERFLOW, "internal: the edge export disagrees with the union-find edge count");
    if (R > 0) KL(k_rid_of_q, nblk(R, TB), TB, R, P->q_of_rid, rid_of_q);
    if (n > 0) {
        const int qb = bits_for(Q);
        KL(k_edges_key2, nblk(n, TB), TB, n, dir, key, iota);
        int r = sort_pairs(ctx, key, key2, iota, perm1, n, 0, qb); if (r) return r;
        KL(k_edges_key1, nblk(n, TB), TB, n, dir, perm1, key);
        r = sort_pairs(ctx, key, key2, perm1, perm, n, 0, qb); if (r) return r;
        if (!(P->pr.overlap > 0.0)) KL(k_edges_final<true>, nblk(n, TB), TB, n, P->tab, dir, perm, rid_of_q, L->read1, L->read2, L->jac);
        else KL(k_edges_final<false>, nblk(n, TB), TB, n, P->tab, dir, perm, rid_of_q, L->read1, L->read2, L->jac);
    }
    return 0;
}

static void fill_stats(fslrc_ctx *ctx, Pipe *P, fslrc_stats *s) {
    if (!s) return;
    const int64_t *h = ctx->h_pin;
    memset(s, 0, sizeof(*s));
    s->n_fillings = P->F; s->n_intervals = P->D; s->n_query_reads = P->Q;
    s->band_pairs = h[3]; s->pair_tests = h[4]; s->relation_entries = h[13]; s->saturating_reads = P->nP;
    s->edges = h[8]; s->components = h[9]; s->clustered_reads = (int64_t)P->R - h[11];
    s->partner_records = h[42];
    s->no_clusters = h[9] == 0;
    if (getenv("FSLRC_DEBUG")) fprintf(stderr, "[fslrc] replay: warp-iterations %lld, group-steps %lld, stalled %lld, sleeps %lld, runs %lld, walk-mode reads %lld, skip chunks done by helper warps %lld\n",
                                       (long long)h[16], (long long)h[17], (long long)h[18], (long long)h[19], (long long)h[12], (long long)h[43], (long long)h[50]);
#ifdef FSLRC_WALKPROF
    if (getenv("FSLRC_DEBUG") && h[43]) fprintf(stderr, "[fslrc] walkprof: runs finished after ms (since the first): 50%% %.3f  90%% %.3f  99%% %.3f  99.9%% %.3f  99.99%% %.3f  all %.3f\n",
                                       1e-6 * (double)(h[53] - h[52]), 1e-6 * (double)(h[39] - h[52]), 1e-6 * (double)(h[54] - h[52]), 1e-6 * (double)(h[37] - h[52]),
                                       1e-6 * (double)(h[38] - h[52]), 1e-6 * (double)(h[55] - h[52]));
    if (getenv("FSLRC_DEBUG") && h[28]) fprintf(stderr, "[fslrc] walkprof: %.3f ms; warp-wide steps %lld (%.0f cycles each), other iterations %lld (%.0f cycles each), group-wide steps %lld; inside a warp-wide step: %.0f cycles to the first-round results, %.0f to the sibling results\n",
                                       1e-6 * (double)h[29], (long long)h[30], (double)h[31] / (double)std::max<long long>(h[30], 1), (long long)h[32],
                                       (double)h[33] / (double)std::max<long long>(h[32], 1), (long long)h[34], (double)h[35] / (double)std::max<long long>(h[30], 1), (double)h[36] / (double)std::max<long long>(h[30], 1));
    else
#endif
    if (getenv("FSLRC_DEBUG") && h[28]) fprintf(stderr, "[fslrc] long stall: a %lld waits b %lld stops %d %d base %lld top %lld posf %lld bpos %lld %lld apos2 %lld fi %lld (n=%lld)\n",
                                       (long long)h[29], (long long)h[30], (int)h[31], (int)h[32], (long long)h[33], (long long)h[34], (long long)h[35], (long long)h[36], (long long)h[37], (long long)h[38], (long long)h[39], (long long)h[28]);
    if (getenv("FSLRC_DEBUG") && h[20]) fprintf(stderr, "[fslrc] longest walk: %lld steps (stalled %lld) read %lld filling %lld/%lld band %lld walked %lld edges %lld\n",
                                       (long long)h[20], (long long)h[24], (long long)h[21], (long long)h[22], (long long)h[27], (long long)h[23], (long long)h[25], (long long)h[26]);
    for (int i = 0; i < FSLRC_N_STAGES; i++) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev[i], ctx->ev[i + 1]) != cudaSuccess) { ms = 0.f; cudaGetLastError(); }
        s->stage_ms[i] = ms;
    }
}

static inline bool oc_host_path_ok(const fslrc_table *tb) { return tb->aln_size_is_qspan != 0; }   // aln_size may be omitted then
static int check_args(fslrc_ctx *ctx, const fslrc_table *tb, const fslrc_params *pr, const void *oc, const void *on) {
    if (!ctx) return FSLRC_ERR_ARG;
    if (!tb || !pr || !oc || !on) return fail(ctx, FSLRC_ERR_ARG, "null argument");
    if (tb->n_rows < 0 || tb->n_reads < 0 || tb->n_rows > 0x7ffffff0LL || tb->n_reads > 0x7ffffff0LL) return fail(ctx, FSLRC_ERR_ARG, "table size out of range");
    if (tb->n_rows > 0 && ((!tb->read_id && !tb->rows_per_read_u8) || (!tb->chrom && !tb->chrom_u8) || !tb->rstart || (!tb->rend && !tb->rspan_i16) ||
                           (!tb->aln_size && !oc_host_path_ok(tb)) || (!tb->qstart && !tb->qstart_u16) || (!tb->qend && !tb->qend_u16) ||
                           (!tb->n_alignments && !tb->n_alignments_u16)))
        return fail(ctx, FSLRC_ERR_ARG, "null column");
    if (pr->n_chrom < 0 || pr->n_chrom > (1 << 20) || (pr->n_chrom > 0 && (!pr->chrom_len || !pr->chrom_masked))) return fail(ctx, FSLRC_ERR_ARG, "bad chromosome tables");
    if (pr->overlap != pr->overlap || pr->qlen_c != pr->qlen_c || pr->naln_c != pr->naln_c) return fail(ctx, FSLRC_ERR_ARG, "NaN option");
    return 0;
}

// The int32 device columns the kernels read, from whatever the caller gave: wide or narrow columns, in host memory (copied
// in) or already on the device (used in place; only narrow / derived ones cost a kernel).  `out` receives device pointers.
static int resolve_columns(fslrc_ctx *ctx, Pipe *P, const fslrc_table *in, bool host, fslrc_table *out) {
    cudaStream_t st = ctx->stream;
    const int64_t A = in->n_rows, R = in->n_reads;
    *out = *in;
    out->chrom_u8 = nullptr; out->n_alignments_u16 = nullptr; out->rows_per_read_u8 = nullptr; out->rspan_i16 = nullptr;
    out->qstart_u16 = nullptr; out->qend_u16 = nullptr;
    auto bring = [&](const void *src, size_t bytes, const void **dst) -> int {          // a column as the device sees it
        if (!host || !src || bytes == 0) { *dst = src; return 0; }
        unsigned char *d; DA(d, bytes);
        CK(cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st));
        *dst = d;
        return 0;
    };
#define BRING(src, bytes, dst) do { const void *q__; int r__ = bring((src), (bytes), &q__); if (r__) return r__; (dst) = (decltype(dst))q__; } while (0)
    const size_t a4 = sizeof(int32_t) * (size_t)A;
    // read ids: the column, or run lengths (the rows of read r are contiguous and the reads come in id order: verified by the caller)
    if (in->read_id || A == 0) BRING(in->read_id, a4, out->read_id);
    else {
        const unsigned char *d_r8; int *cnt32, *first, *rid;
        BRING(in->rows_per_read_u8, (size_t)R, d_r8);
        DA(cnt32, R); DA(first, R); DA(rid, A);
        KL(k_widen_u8, nblk(R, 256), 256, R, d_r8, cnt32);
        int r = xscan(ctx, cnt32, first, (int)R); if (r) return r;
        KL(k_rid_from_runs, nblk(R, 256), 256, (int)R, (int)A, first, cnt32, rid);
        out->read_id = rid;
    }
    Widen w; memset(&w, 0, sizeof(w));
    bool any = false;
    BRING(in->rstart, a4, out->rstart);
    w.rstart = out->rstart;
    if (in->chrom || A == 0) BRING(in->chrom, a4, out->chrom);
    else { BRING(in->chrom_u8, (size_t)A, w.c8); DA(w.chrom, A); out->chrom = w.chrom; any = true; }
    if (in->rend || A == 0) BRING(in->rend, a4, out->rend);
    else { BRING(in->rspan_i16, 2 * (size_t)A, w.span16); DA(w.rend, A); out->rend = w.rend; any = true; }
    if (in->qstart || A == 0) BRING(in->qstart, a4, out->qstart);
    else { BRING(in->qstart_u16, 2 * (size_t)A, w.qs16); DA(w.qstart, A); out->qstart = w.qstart; any = true; }
    if (in->qend || A == 0) BRING(in->qend, a4, out->qend);
    else { BRING(in->qend_u16, 2 * (size_t)A, w.qe16); DA(w.qend, A); out->qend = w.qend; any = true; }
    if (in->n_alignments || A == 0) BRING(in->n_alignments, a4, out->n_alignments);
    else if (host && ctx->copy_stream && !ctx->blocking && A >= (1 << 20)) {
        // the first kernels (keep_fillings) do not read this column: its upload goes LAST, on a second stream, and overlaps them
        // (not for the contexts of a HostPipeline — blocking-sync waits —: there the whole upload already overlaps the kernels of
        // the table before; a second copy stream per context would only reorder the DMA queue)
        unsigned char *d16; DA(d16, 2 * (size_t)A); DA(w.naln, A); out->n_alignments = w.naln;
        CK(cudaEventRecord(ctx->ev_c1, st));                                       // (every other column is on its way)
        CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_c1, 0));
        CK(cudaMemcpyAsync(d16, in->n_alignments_u16, 2 * (size_t)A, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(ctx->ev_c2, ctx->copy_stream));
        memset(&P->w_late, 0, sizeof(P->w_late));
        P->w_late.n16 = (const unsigned short *)d16; P->w_late.naln = w.naln;
        P->late = true; ctx->late_pending = true;
    }
    else { BRING(in->n_alignments_u16, 2 * (size_t)A, w.n16); DA(w.naln, A); out->n_alignments = w.naln; any = true; }
    if (in->aln_size || A == 0) BRING(in->aln_size, a4, out->aln_size);
    else {                                                                         // aln_size = qend - qstart (check_args saw the flag)
        DA(w.aln, A); out->aln_size = w.aln; any = true;
        if (!w.qstart) w.qstart = (int *)out->qstart;                              // (read only in that case)
        if (!w.qend) w.qend = (int *)out->qend;
    }
    if (any && A > 0) KL(k_widen, nblk(A, 256), 256, A, w);
    if (in->order) BRING(in->order, sizeof(int32_t) * (size_t)in->n_order, out->order);
#undef BRING
    return 0;
}

static int run_device(fslrc_ctx *ctx, Pipe *P, int32_t *oc, int32_t *on, fslrc_stats *stats) {
    int r = pipe_prepare(ctx, P); if (r) return r;
    r = pipe_pair(ctx, P, 0, 1); if (r) return r;
    r = pipe_sat(ctx, P); if (r) return r;
    r = pipe_replay_union(ctx, P, 0, 1, nullptr, 0); if (r) return r;
    r = pipe_number(ctx, P, oc, on); if (r) return r;
    return 0;
}

// choose_alignment (cluster.py:237-254) on device columns: per read the sum and count of alignment_score over its rows,
// per cluster the read with the highest mean, the one whose first row comes first on ties.  is_rep[r] = 1 for those
// reads; rep_read (nullable) receives each cluster's.  A read id >= R or a cluster id outside [0, C) sets EF_RANGE in *err.
static int choose_alignment_dev(fslrc_ctx *ctx, int A, int R, int C, const int *rid, const int *score, const int *cluster,
                                long long *sum, int *cnt, unsigned char *is_rep, int *rep_read, int *err) {
    cudaStream_t st = ctx->stream;
    const int TB = 256;
    int *first, *minrow; unsigned long long *best;
    DA(first, R); DA(minrow, C); DA(best, C);
    if (R > 0) {
        CK(cudaMemsetAsync(cnt, 0, sizeof(int) * R, st));
        CK(cudaMemsetAsync(sum, 0, sizeof(long long) * R, st));
        KL(k_fill<int>, nblk(R, TB), TB, first, R, 0x7fffffff);
    }
    if (C > 0) {
        CK(cudaMemsetAsync(best, 0, sizeof(unsigned long long) * C, st));
        KL(k_fill<int>, nblk(C, TB), TB, minrow, C, 0x7fffffff);
        if (rep_read) KL(k_fill<int>, nblk(C, TB), TB, rep_read, C, -1);
    }
    CK(cudaMemsetAsync(err, 0, sizeof(int), st));
    if (A > 0) KL(k_ca_rows, nblk(A, TB), TB, A, R, rid, score, sum, cnt, first, err);
    if (R > 0) {
        KL(k_ca_best, nblk(R, TB), TB, R, C, sum, cnt, cluster, best, err);
        KL(k_ca_first, nblk(R, TB), TB, R, C, sum, cnt, first, cluster, best, minrow);
        KL(k_ca_flag, nblk(R, TB), TB, R, C, cnt, first, cluster, minrow, is_rep, rep_read);
    }
    return 0;
}

extern "C" {

int fslrc_version(void) { return FSLRC_VERSION; }
const char *fslrc_stage_name(int s) { return (s >= 0 && s < FSLRC_N_STAGES) ? STAGE_NAMES[s] : ""; }
const char *fslrc_last_error(const fslrc_ctx *ctx) { return ctx ? ctx->err : "null context"; }

int fslrc_create(int device, fslrc_ctx **out) {
    if (!out) return FSLRC_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) { cudaGetLastError(); return FSLRC_ERR_CUDA; }
    if (cudaSetDevice(device) != cudaSuccess) return FSLRC_ERR_CUDA;
    fslrc_ctx *ctx = new fslrc_ctx();
    ctx->device = device; ctx->launches = 0; ctx->err[0] = 0; ctx->stream = nullptr; ctx->pipe = nullptr; ctx->tsv = nullptr; ctx->bam = nullptr; ctx->h_pin = nullptr;
    if (cudaMallocHost((void **)&ctx->h_pin, 64 * sizeof(int64_t)) != cudaSuccess) { delete ctx; return FSLRC_ERR_CUDA; }
    for (int i = 0; i <= FSLRC_N_STAGES; i++) cudaEventCreate(&ctx->ev[i]);
    cudaEventCreateWithFlags(&ctx->ev_block, cudaEventBlockingSync | cudaEventDisableTiming);
    ctx->blocking = 0;
    ctx->copy_stream = nullptr; ctx->late_pending = false;
    ctx->edge_capture = 0; ctx->edges = nullptr; ctx->tsv_gen = 0;
    ctx->prim = nullptr; ctx->prim_bytes = 0;
    if (cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) { ctx->copy_stream = nullptr; cudaGetLastError(); }
    cudaEventCreateWithFlags(&ctx->ev_c1, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->ev_c2, cudaEventDisableTiming);
    cudaFuncSetAttribute(prims::k_rs_onesweep<prims::PairOut>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(prims::RsSmem));
    cudaFuncSetAttribute(prims::k_rs_onesweep<ChromRecOut>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(prims::RsSmem));
    cudaMemPool_t pool;                                   // keep freed scratch cached between calls
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = ctx;
    return 0;
}

void fslrc_destroy(fslrc_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    edges_free(ctx);
    free_all(ctx);
    tsv_free(ctx);
    bam_free(ctx);
    cudaDeviceSynchronize();
    for (int i = 0; i <= FSLRC_N_STAGES; i++) cudaEventDestroy(ctx->ev[i]);
    cudaEventDestroy(ctx->ev_block);
    cudaEventDestroy(ctx->ev_c1); cudaEventDestroy(ctx->ev_c2);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
    delete ctx->pipe;
    delete ctx;
}

// a clustering call drops the edge list of the previous one first (also when it fails)
static void begin_clustering(fslrc_ctx *ctx, void *stream) {
    if (!ctx || !ctx->edges) return;
    cudaSetDevice(ctx->device);
    ctx->stream = (cudaStream_t)stream;
    edges_free(ctx);
}

int fslrc_cluster_device(fslrc_ctx *ctx, const fslrc_table *table, const fslrc_params *params, int32_t *out_cluster,
                         int32_t *out_n_reads, fslrc_stats *stats, void *stream) {
    begin_clustering(ctx, stream);
    int r = check_args(ctx, table, params, out_cluster, out_n_reads); if (r) return r;
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    Pipe P; memset(&P, 0, sizeof(P));
    P.pr = *params; P.A = (int)table->n_rows; P.R = (int)table->n_reads;
    for (int i = 0; i <= FSLRC_N_STAGES; i++) cudaEventRecord(ctx->ev[i], ctx->stream);
    r = resolve_columns(ctx, &P, table, false, &P.tb);
    if (!r) CK(cudaEventRecord(ctx->ev[1], ctx->stream));                  // closes stage 0 (widening of narrow columns, if any)
    if (!r) r = run_device(ctx, &P, out_cluster, out_n_reads, stats);
    if (!r) { r = mark(ctx, ST_D2H); }
    if (!r && ctx->edge_capture) r = export_edges(ctx, &P, table->read_id);
    if (!r) { r = read_counts(ctx, &P); if (!r) r = err_code(ctx); }
    if (!r) fill_stats(ctx, &P, stats);
    free_all(ctx);
    if (r) edges_free(ctx);
    ctx_sync(ctx);
    return r;
}

int fslrc_cluster_host(fslrc_ctx *ctx, const fslrc_table *table, const fslrc_params *params, int32_t *out_cluster,
                       int32_t *out_n_reads, fslrc_stats *stats, void *stream) {
    begin_clustering(ctx, stream);
    int r = check_args(ctx, table, params, out_cluster, out_n_reads); if (r) return r;
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    cudaStream_t st = ctx->stream;
    const int64_t A = table->n_rows, R = table->n_reads;
    for (int i = 0; i <= FSLRC_N_STAGES; i++) cudaEventRecord(ctx->ev[i], st);
    fslrc_table d;
    Pipe P; memset((void *)&P, 0, sizeof(P));
    r = resolve_columns(ctx, &P, table, true, &d); if (r) { free_all(ctx); ctx_sync(ctx); return r; }
    int32_t *d_oc, *d_on;
    DA(d_oc, R); DA(d_on, R);
    CK(cudaEventRecord(ctx->ev[1], st));                                   // closes stage 0 (h2d)
    P.tb = d; P.pr = *params; P.A = (int)A; P.R = (int)R;
    r = run_device(ctx, &P, d_oc, d_on, stats);
    if (!r && R > 0) {
        CK(cudaMemcpyAsync(out_cluster, d_oc, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(out_n_reads, d_on, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, st));
    }
    if (!r) r = mark(ctx, ST_D2H);
    if (!r && ctx->edge_capture) r = export_edges(ctx, &P, nullptr);
    if (!r) { r = read_counts(ctx, &P); if (!r) r = err_code(ctx); }
    if (!r) fill_stats(ctx, &P, stats);
    free_all(ctx);
    if (r) edges_free(ctx);
    ctx_sync(ctx);
    return r;
}

// The column cluster.py:114 sorts, for a host sort with the reference's own call (its tie order is numpy's, not ours): stage 1
// of the general ingest, then one scatter of min(rstart, rend) of the kept rows.  Only the count is read back.
int fslrc_filling_starts(fslrc_ctx *ctx, const fslrc_table *table, int32_t *out_start, int64_t cap, int64_t *n_fillings,
                         void *stream) {
    if (!ctx) return FSLRC_ERR_ARG;
    if (!table || !out_start || !n_fillings) return fail(ctx, FSLRC_ERR_ARG, "null argument");
    const int64_t A = table->n_rows, R = table->n_reads;
    if (A < 0 || R < 0 || A > 0x7ffffff0LL || R > 0x7ffffff0LL) return fail(ctx, FSLRC_ERR_ARG, "table size out of range");
    if (cap < A) return fail(ctx, FSLRC_ERR_ARG, "out_start is smaller than the table (cap < n_rows)");
    if (A > 0 && (!table->read_id || !table->rstart || !table->rend))
        return fail(ctx, FSLRC_ERR_ARG, "the wide device columns read_id, rstart and rend are needed (wire-format-only table)");
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    cudaStream_t st = ctx->stream;
    Pipe P; memset((void *)&P, 0, sizeof(P));
    P.A = (int)A; P.R = (int)R;
    auto run = [&]() -> int {
        int *flagA, *posA;
        DA(P.err, 1); DA(P.cnt, NCNT); DA(flagA, A); DA(posA, A);
        CK(cudaMemsetAsync(P.err, 0, sizeof(int), st));
        CK(cudaMemsetAsync(P.cnt, 0, NCNT * sizeof(int64_t), st));
        int q = keep_rows(ctx, &P, table->read_id, nullptr, nullptr, flagA, posA, nullptr, nullptr); if (q) return q;
        if (A > 0) KL(k_filling_starts, nblk(A, 256), 256, (int)A, flagA, posA, table->rstart, table->rend, out_start);
        q = read_counts(ctx, &P); if (q) return q;
        q = err_code(ctx); if (q) return q;
        *n_fillings = ctx->h_pin[0];
        return 0;
    };
    const int r = run();
    free_all(ctx);
    ctx_sync(ctx);
    return r;
}

// ---------------------------------------------------------------- multi-GPU staging
int fslrc_mg_prepare(fslrc_ctx *ctx, const fslrc_table *table, const fslrc_params *params, void *stream) {
    begin_clustering(ctx, stream);                                      // (the multi-GPU sequence captures no edges)
    int dummy = 0;
    int r = check_args(ctx, table, params, &dummy, &dummy); if (r) return r;
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    free_all(ctx);
    delete ctx->pipe;
    Pipe *P = ctx->pipe = new Pipe(); memset(P, 0, sizeof(*P));
    P->pr = *params; P->A = (int)table->n_rows; P->R = (int)table->n_reads;
    for (int i = 0; i <= FSLRC_N_STAGES; i++) cudaEventRecord(ctx->ev[i], ctx->stream);
    r = resolve_columns(ctx, P, table, false, &P->tb);
    if (!r) CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    if (!r) r = pipe_prepare(ctx, P);
    if (r) { free_all(ctx); cudaStreamSynchronize(ctx->stream); }
    return r;
}
int fslrc_mg_pair(fslrc_ctx *ctx, int rank, int world, int32_t **counts, int64_t *n_counts) {
    if (!ctx || !ctx->pipe || !counts || !n_counts || world < 1 || rank < 0 || rank >= world) return FSLRC_ERR_ARG;
    Pipe *P = ctx->pipe;
    CK(cudaSetDevice(ctx->device));
    int r = pipe_pair(ctx, P, rank, world); if (r) return r;
    CK(cudaStreamSynchronize(ctx->stream));
    *counts = (int32_t *)P->cp; *n_counts = P->Q;
    return 0;
}
int fslrc_mg_partners(fslrc_ctx *ctx, int rank, int world, int32_t **pairs, int64_t *n_pairs) {
    if (!ctx || !ctx->pipe || !pairs || !n_pairs || world < 1 || rank < 0 || rank >= world) return FSLRC_ERR_ARG;
    Pipe *P = ctx->pipe;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    int r = pipe_sat(ctx, P); if (r) return r;
    r = read_counts(ctx, P); if (r) return r;
    r = err_code(ctx); if (r) return r;
    const unsigned long long nent = std::min<unsigned long long>((unsigned long long)ctx->h_pin[5], P->cap_entries);
    int2 *pent; DA(pent, 2 * nent);
    if (nent > 0) KL(k_pent_compact, nblk((int64_t)nent, 256), 256, (const int2 *)P->entries, nent, P->plinfo, pent, (unsigned long long *)(P->cnt + 47));
    r = read_counts(ctx, P); if (r) return r;
    *pairs = (int32_t *)pent; *n_pairs = ctx->h_pin[47];
    return 0;
}
int fslrc_mg_replay(fslrc_ctx *ctx, int rank, int world, const int32_t *all_pairs, int64_t n_all_pairs, int32_t **forest,
                    int64_t *n_forest_edges) {
    if (!ctx || !ctx->pipe || !forest || !n_forest_edges || n_all_pairs < 0 || (n_all_pairs > 0 && !all_pairs)) return FSLRC_ERR_ARG;
    Pipe *P = ctx->pipe;
    CK(cudaSetDevice(ctx->device));
    static const int2 none = {-1, -1};
    int r = pipe_replay_union(ctx, P, rank, world, all_pairs ? (const int2 *)all_pairs : &none, (unsigned long long)n_all_pairs); if (r) return r;
    cudaStream_t st = ctx->stream;
    const int Q = P->Q, TB = 256;
    int *isroot, *csize; int2 *fo;
    DA(isroot, Q); DA(csize, Q); DA(fo, Q);
    if (Q > 0) {
        CK(cudaMemsetAsync(csize, 0, sizeof(int) * Q, st));
        KL(k_flatten, nblk(Q, TB), TB, Q, P->parent, P->ing, isroot, csize);
        KL(k_forest, nblk(Q, TB), TB, Q, P->parent, P->ing, fo, (unsigned long long *)(P->cnt + 10));
    }
    r = read_counts(ctx, P); if (r) return r;
    r = err_code(ctx); if (r) return r;
    *forest = (int32_t *)fo; *n_forest_edges = ctx->h_pin[10];
    return 0;
}
int fslrc_mg_finish(fslrc_ctx *ctx, const int32_t *all_forest, int64_t n_edges, int32_t *out_cluster, int32_t *out_n_reads,
                    fslrc_stats *stats) {
    if (!ctx || !ctx->pipe || !out_cluster || !out_n_reads || n_edges < 0 || (n_edges > 0 && !all_forest)) return FSLRC_ERR_ARG;
    Pipe *P = ctx->pipe;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int Q = P->Q, TB = 256;
    if (Q > 0) {
        KL(k_iota, nblk(Q, TB), TB, P->parent, Q);
        CK(cudaMemsetAsync(P->ing, 0, sizeof(int) * Q, st));
    }
    if (n_edges > 0) KL(k_union_edges, nblk(n_edges, TB), TB, (unsigned long long)n_edges, (const int2 *)all_forest, P->parent, P->ing, (unsigned long long *)nullptr);
    int r = pipe_number(ctx, P, out_cluster, out_n_reads);
    if (!r) r = mark(ctx, ST_D2H);
    if (!r) { r = read_counts(ctx, P); if (!r) r = err_code(ctx); }
    if (!r) fill_stats(ctx, P, stats);
    free_all(ctx);
    cudaStreamSynchronize(st);
    delete ctx->pipe; ctx->pipe = nullptr;
    return r;
}

int fslrc_choose_alignment_host(fslrc_ctx *ctx, int64_t n_rows, int64_t n_reads, int64_t n_clusters, const int32_t *read_id,
                                const int32_t *alignment_score, const int32_t *cluster, uint8_t *out_is_rep, int32_t *out_rep_read,
                                void *stream) {
    if (!ctx) return FSLRC_ERR_ARG;
    if (n_rows < 0 || n_reads < 0 || n_clusters < 0 || n_rows > 0x7ffffff0LL || n_reads > 0x7ffffff0LL || n_clusters > 0x7ffffff0LL ||
        (n_rows > 0 && (!read_id || !alignment_score)) || (n_reads > 0 && (!cluster || !out_is_rep)))
        return fail(ctx, FSLRC_ERR_ARG, "choose_alignment: bad argument");
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    cudaStream_t st = ctx->stream;
    const int A = (int)n_rows, R = (int)n_reads, C = (int)n_clusters;
    int *d_rid, *d_sc, *d_cl, *cnt, *rep, *err; long long *sum; unsigned char *flag;
    DA(d_rid, A); DA(d_sc, A); DA(d_cl, R); DA(cnt, R); DA(rep, C); DA(err, 1); DA(sum, R); DA(flag, R);
    if (A > 0) {
        CK(cudaMemcpyAsync(d_rid, read_id, sizeof(int) * A, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(d_sc, alignment_score, sizeof(int) * A, cudaMemcpyHostToDevice, st));
    }
    if (R > 0) CK(cudaMemcpyAsync(d_cl, cluster, sizeof(int) * R, cudaMemcpyHostToDevice, st));
    { int r = choose_alignment_dev(ctx, A, R, C, d_rid, d_sc, d_cl, sum, cnt, flag, rep, err); if (r) return r; }
    if (R > 0) CK(cudaMemcpyAsync(out_is_rep, flag, R, cudaMemcpyDeviceToHost, st));
    if (C > 0 && out_rep_read) CK(cudaMemcpyAsync(out_rep_read, rep, sizeof(int) * C, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ctx->h_pin + 60, err, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    free_all(ctx);
    cudaStreamSynchronize(st);
    if ((int)(ctx->h_pin[60] & 0xffffffff)) return fail(ctx, FSLRC_ERR_RANGE, "choose_alignment: read id or cluster id out of range");
    return 0;
}

// ---------------------------------------------------------------- mappings.bed ingest / egress on the GPU (tsv.cuh)
}  // extern "C"
struct TsvState {
    Resident mem;            // every device array below (until fslrc_tsv_close or the next fslrc_tsv_open)
    unsigned char *text; long long n; long long *line_start;
    int n_lines, n_rows, n_reads, n_chrom;
    int *read_id, *chrom, *rstart, *rend, *aln, *qstart, *qend, *naln, *score, *first_row;
    long long *q_off; int *q_len;
    long long *line_end;     // nullptr: line l ends at line_start[l + 1] - 1; set once fslrc_tsv_delete_false removed rows
    std::vector<std::string> chrom_names;
};
static const int32_t *tsv_read_id(const fslrc_ctx *ctx) { return ctx->tsv ? ctx->tsv->read_id : nullptr; }
static void tsv_free(fslrc_ctx *ctx) { drop_table(ctx, ctx->tsv); }
// strings -> dense ids in order of first appearance (pandas.factorize); *n_ids receives the number of distinct strings
static int tsv_intern(fslrc_ctx *ctx, const unsigned char *text, int n, const long long *off, const int *len,
                      const unsigned long long *hash, int *id_out, int *first_row_of_id /*nullable, capacity n*/, int *err,
                      int64_t *n_ids_dev) {
    cudaStream_t st = ctx->stream;
    const int TB = 256;
    unsigned cap = 1024; while (cap < 2u * (unsigned)n && cap < (1u << 30)) cap <<= 1;
    unsigned long long *keys; int *first, *slot, *isf, *idat;
    DA(keys, cap); DA(first, cap); DA(slot, n); DA(isf, n); DA(idat, n);
    CK(cudaMemsetAsync(keys, 0xff, sizeof(unsigned long long) * cap, st));
    KL(k_fill<int>, nblk(cap, TB), TB, first, (int64_t)cap, 0x7fffffff);
    KL(tsv::k_tsv_intern_insert, nblk(n, TB), TB, n, hash, keys, first, cap - 1, slot);
    KL(tsv::k_tsv_intern_verify, nblk(n, TB), TB, n, text, off, len, slot, first, isf, err);
    int r = xscan(ctx, isf, idat, n, n_ids_dev); if (r) return r;
    KL(tsv::k_tsv_intern_ids, nblk(n, TB), TB, n, slot, first, idat, id_out, first_row_of_id);
    return 0;
}
static int tsv_open_impl(fslrc_ctx *ctx, const char *text, int64_t n_bytes, uint64_t hash_seed, fslrc_tsv_info *info) {
    cudaStream_t st = ctx->stream;
    tsv_free(ctx);
    // ---- header (host): which field holds which column (names of collect_mapping_info.py:176-181)
    const char *names[tsv::W_N] = {"chrom", "rstart", "rend", "qname", "n_alignments", "aln_size", "qstart", "qend", "alignment_score"};
    tsv::Want w; for (int k = 0; k < tsv::W_N; k++) w.col[k] = -1; w.last = -1;
    {
        int64_t e = 0; while (e < n_bytes && text[e] != '\n') e++;
        int f = 0; int64_t p = 0;
        while (p <= e) {
            int64_t q = p; while (q < e && text[q] != '\t') q++;
            for (int k = 0; k < tsv::W_N; k++)
                if ((int64_t)strlen(names[k]) == q - p && memcmp(names[k], text + p, q - p) == 0) { w.col[k] = f; if (f > w.last) w.last = f; }
            f++; p = q + 1;
        }
        for (int k = 0; k < tsv::W_SCORE; k++) if (w.col[k] < 0) return fail(ctx, FSLRC_ERR_ARG, "tsv: header lacks column %s", names[k]);
    }
    TsvState *T = ctx->tsv = new TsvState();
    ctx->tsv_gen++;
    const bool pad = text[n_bytes - 1] != '\n';
    T->n = n_bytes + (pad ? 1 : 0);
    RA(T->mem, T->text, T->n + 64);
    CK(cudaMemcpyAsync(T->text, text, n_bytes, cudaMemcpyHostToDevice, st));
    if (pad) CK(cudaMemsetAsync(T->text + n_bytes, '\n', 1, st));
    CK(cudaEventRecord(ctx->ev[1], st));
    // ---- lines
    const int TB = 256;
    const int64_t nchunks = (T->n + tsv::CHUNK - 1) / tsv::CHUNK;
    if (nchunks > 0x7ffffff0LL) return fail(ctx, FSLRC_ERR_ARG, "tsv: input too large");
    int *cnt, *pre, *err;
    DA(cnt, nchunks); DA(pre, nchunks); DA(err, 1);
    int64_t *dcount; DA(dcount, 4);
    CK(cudaMemsetAsync(err, 0, sizeof(int), st));
    KL(tsv::k_tsv_count, nblk(nchunks, TB), TB, T->text, (long long)T->n, cnt);
    { int r = xscan(ctx, cnt, pre, (int)nchunks, dcount); if (r) return r; }
    CK(cudaMemcpyAsync(ctx->h_pin, dcount, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (ctx->h_pin[0] > 0x7ffffff0LL) return fail(ctx, FSLRC_ERR_ARG, "tsv: too many lines");
    T->n_lines = (int)ctx->h_pin[0];
    T->n_rows = T->n_lines - 1;
    RA(T->mem, T->line_start, (int64_t)T->n_lines + 1);
    KL(tsv::k_tsv_lines, nblk(nchunks, TB), TB, T->text, (long long)T->n, pre, T->line_start);
    const int n = T->n_rows;
    RA(T->mem, T->read_id, n); RA(T->mem, T->chrom, n); RA(T->mem, T->rstart, n); RA(T->mem, T->rend, n);
    RA(T->mem, T->aln, n); RA(T->mem, T->qstart, n); RA(T->mem, T->qend, n); RA(T->mem, T->naln, n);
    RA(T->mem, T->q_off, n); RA(T->mem, T->q_len, n); RA(T->mem, T->first_row, n);
    T->score = nullptr;
    if (w.col[tsv::W_SCORE] >= 0) RA(T->mem, T->score, n);
    T->n_reads = 0; T->n_chrom = 0;
    if (n > 0) {
        unsigned long long *qh, *ch; long long *coff; int *clen, *cfirst;
        DA(qh, n); DA(ch, n); DA(coff, n); DA(clen, n); DA(cfirst, n);
        KL(tsv::k_tsv_parse, nblk(n, TB), TB, T->text, T->line_start, n, w, (unsigned long long)hash_seed, T->rstart, T->rend, T->naln, T->aln,
           T->qstart, T->qend, T->score, T->q_off, T->q_len, qh, coff, clen, ch, err);
        int r = tsv_intern(ctx, T->text, n, T->q_off, T->q_len, qh, T->read_id, T->first_row, err, dcount + 1); if (r) return r;
        r = tsv_intern(ctx, T->text, n, coff, clen, ch, T->chrom, cfirst, err, dcount + 2); if (r) return r;
        CK(cudaMemcpyAsync(ctx->h_pin, dcount, 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(ctx->h_pin + 8, err, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const int e = (int)(ctx->h_pin[8] & 0xffffffff);
        if (e) {
            if (e & tsv::TE_COLLISION) return fail(ctx, FSLRC_ERR_HASH_COLLISION, "tsv: two different names share a 64-bit hash; call again with another hash_seed");
            if (e & tsv::TE_FIELDS) return fail(ctx, FSLRC_ERR_ARG, "tsv: a line has fewer fields than the header");
            if (e & tsv::TE_RANGE) return fail(ctx, FSLRC_ERR_RANGE, "tsv: an integer field does not fit int32");
            return fail(ctx, FSLRC_ERR_ARG, "tsv: a numeric field is not an integer");
        }
        T->n_reads = (int)ctx->h_pin[1]; T->n_chrom = (int)ctx->h_pin[2];
        // chromosome names (few): offsets of their first rows -> host strings out of the caller's text
        std::vector<int> cf(T->n_chrom);
        CK(cudaMemcpyAsync(cf.data(), cfirst, sizeof(int) * T->n_chrom, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        std::vector<long long> o1(1); std::vector<int> l1(1);
        for (int c = 0; c < T->n_chrom; c++) {
            CK(cudaMemcpyAsync(o1.data(), coff + cf[c], sizeof(long long), cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(l1.data(), clen + cf[c], sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            T->chrom_names.emplace_back(text + o1[0], (size_t)l1[0]);
        }
    }
    CK(cudaEventRecord(ctx->ev[2], st));
    free_all(ctx);
    CK(cudaStreamSynchronize(st));
    memset(info, 0, sizeof(*info));
    info->n_rows = T->n_rows; info->n_reads = T->n_reads; info->n_chrom = T->n_chrom; info->has_score = T->score != nullptr;
    info->read_id = T->read_id; info->chrom = T->chrom; info->rstart = T->rstart; info->rend = T->rend; info->aln_size = T->aln;
    info->qstart = T->qstart; info->qend = T->qend; info->n_alignments = T->naln; info->alignment_score = T->score;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev[0 + 1], ctx->ev[2]) == cudaSuccess) info->parse_ms = ms; else cudaGetLastError();
    return 0;
}
// --filter-false on the parsed table: flag the reads (one thread per read), two exclusive scans give the new read ids and
// the new row positions, one read-back of both totals, and, if any row goes, one compaction into fresh arrays
static int tsv_delete_false_impl(fslrc_ctx *ctx, fslrc_tsv_info *info) {
    cudaStream_t st = ctx->stream;
    TsvState *T = ctx->tsv;
    const int n = T->n_rows, R = T->n_reads, TB = 256;
    ctx->tsv_gen++;
    CK(cudaEventRecord(ctx->ev[1], st));
    if (R > 0) {
        int *keep_read, *new_id, *keep_row, *new_pos; int64_t *tot;
        DA(keep_read, R); DA(new_id, R); DA(keep_row, n); DA(new_pos, n); DA(tot, 2);
        KL(tsv::k_tsv_false, nblk(R, TB), TB, R, T->text, T->first_row, T->q_off, T->q_len, keep_read);
        int r = xscan(ctx, keep_read, new_id, R, tot); if (r) return r;
        KL(tsv::k_tsv_row_keep, nblk(n, TB), TB, n, T->read_id, keep_read, keep_row);
        r = xscan(ctx, keep_row, new_pos, n, tot + 1); if (r) return r;
        CK(cudaMemcpyAsync(ctx->h_pin, tot, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const int R2 = (int)ctx->h_pin[0], n2 = (int)ctx->h_pin[1];
        if (n2 < n) {
            const tsv::Cols s = {T->read_id, T->chrom, T->rstart, T->rend, T->aln, T->qstart, T->qend, T->naln, T->score,
                                 T->q_off, T->q_len, T->line_start, T->line_end};
            tsv::Cols d; memset((void *)&d, 0, sizeof(d));
            int *first_row;
            RA(T->mem, d.read_id, n2); RA(T->mem, d.chrom, n2); RA(T->mem, d.rstart, n2); RA(T->mem, d.rend, n2);
            RA(T->mem, d.aln, n2); RA(T->mem, d.qstart, n2); RA(T->mem, d.qend, n2); RA(T->mem, d.naln, n2);
            RA(T->mem, d.q_off, n2); RA(T->mem, d.q_len, n2); RA(T->mem, d.line_start, (int64_t)n2 + 1); RA(T->mem, d.line_end, (int64_t)n2 + 1);
            RA(T->mem, first_row, R2);
            if (T->score) RA(T->mem, d.score, n2);
            KL(tsv::k_tsv_compact, nblk(n, TB), TB, n, keep_row, new_pos, new_id, T->first_row, s, d, first_row);
            void *old[] = {s.read_id, s.chrom, s.rstart, s.rend, s.aln, s.qstart, s.qend, s.naln, s.score, s.q_off, s.q_len,
                           s.line_start, s.line_end, T->first_row};
            for (void *p : old) if (p) res_free(ctx, T->mem, p);       // (stream-ordered: after the compaction has read them)
            T->read_id = d.read_id; T->chrom = d.chrom; T->rstart = d.rstart; T->rend = d.rend; T->aln = d.aln;
            T->qstart = d.qstart; T->qend = d.qend; T->naln = d.naln; T->score = d.score; T->q_off = d.q_off; T->q_len = d.q_len;
            T->line_start = d.line_start; T->line_end = d.line_end; T->first_row = first_row;
            T->n_rows = n2; T->n_reads = R2; T->n_lines = n2 + 1;
        }
    }
    CK(cudaEventRecord(ctx->ev[2], st));
    free_all(ctx);
    CK(cudaStreamSynchronize(st));
    info->n_rows = T->n_rows; info->n_reads = T->n_reads;
    info->read_id = T->read_id; info->chrom = T->chrom; info->rstart = T->rstart; info->rend = T->rend; info->aln_size = T->aln;
    info->qstart = T->qstart; info->qend = T->qend; info->n_alignments = T->naln; info->alignment_score = T->score;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev[1], ctx->ev[2]) == cudaSuccess) info->filter_ms = ms; else cudaGetLastError();
    return 0;
}
// The second pass of a text render.  len[i] is the byte length of line i (n lines, written by the caller's length kernel); an
// exclusive scan gives every line's offset, and with the optional header *n_out is the size of the file.  out == NULL only
// asks for that size; otherwise emit(off, d_out) writes the lines after the header into a device buffer that goes to `out`.
template <typename Emit>
static int render_text(fslrc_ctx *ctx, const char *who, int n, const long long *len, const std::string *header, char *out,
                       int64_t cap, int64_t *n_out, Emit &&emit) {
    cudaStream_t st = ctx->stream;
    const int64_t nh = header ? (int64_t)header->size() : 0;
    long long *off; int64_t *tot;
    DA(off, n); DA(tot, 1);
    { int r = xscan64(ctx, len, off, n, tot); if (r) return r; }
    CK(cudaMemcpyAsync(ctx->h_pin, tot, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *n_out = ctx->h_pin[0] + nh;
    if (out) {
        if (cap < *n_out) return fail(ctx, FSLRC_ERR_ARG, "%s: output buffer too small", who);
        unsigned char *d_out; DA(d_out, *n_out);
        if (nh > 0) CK(cudaMemcpyAsync(d_out, header->data(), nh, cudaMemcpyHostToDevice, st));
        emit((const long long *)off, d_out);
        CK(cudaMemcpyAsync(out, d_out, *n_out, cudaMemcpyDeviceToHost, st));
    }
    free_all(ctx);
    CK(cudaStreamSynchronize(st));
    return 0;
}
extern "C" {

int fslrc_tsv_open(fslrc_ctx *ctx, const char *text, int64_t n_bytes, uint64_t hash_seed, fslrc_tsv_info *info, void *stream) {
    if (!ctx) return FSLRC_ERR_ARG;
    if (!text || !info || n_bytes <= 0) return fail(ctx, FSLRC_ERR_ARG, "tsv: null or empty input");
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    return table_call(ctx, tsv_free, [&] { return tsv_open_impl(ctx, text, n_bytes, hash_seed, info); });
}
int fslrc_tsv_delete_false(fslrc_ctx *ctx, fslrc_tsv_info *info, void *stream) {
    if (!ctx) return FSLRC_ERR_ARG;
    if (!ctx->tsv || !info) return fail(ctx, FSLRC_ERR_ARG, "tsv: no parsed table (fslrc_tsv_open first) or null info");
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    return table_call(ctx, nullptr, [&] { return tsv_delete_false_impl(ctx, info); });   // (the old arrays stay until the compaction ran)
}
int fslrc_tsv_chrom_name(fslrc_ctx *ctx, int32_t chrom_id, char *buf, int32_t cap) {
    if (!ctx || !ctx->tsv || !buf || chrom_id < 0 || chrom_id >= ctx->tsv->n_chrom) return FSLRC_ERR_ARG;
    const std::string &s = ctx->tsv->chrom_names[chrom_id];
    if ((int)s.size() + 1 > cap) return FSLRC_ERR_ARG;
    memcpy(buf, s.c_str(), s.size() + 1);
    return (int)s.size();
}
int fslrc_tsv_read_names(fslrc_ctx *ctx, int64_t *offsets, int32_t *lengths) {
    if (!ctx || !ctx->tsv || !offsets || !lengths) return FSLRC_ERR_ARG;
    TsvState *T = ctx->tsv;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int R = T->n_reads;
    if (R == 0) return 0;
    std::vector<int> fr(R);
    CK(cudaMemcpyAsync(fr.data(), T->first_row, sizeof(int) * R, cudaMemcpyDeviceToHost, st));
    std::vector<long long> qo(T->n_rows); std::vector<int> ql(T->n_rows);
    CK(cudaMemcpyAsync(qo.data(), T->q_off, sizeof(long long) * T->n_rows, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ql.data(), T->q_len, sizeof(int) * T->n_rows, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int r = 0; r < R; r++) { offsets[r] = qo[fr[r]]; lengths[r] = ql[fr[r]]; }
    return 0;
}
int fslrc_tsv_write_cluster_bed(fslrc_ctx *ctx, const int32_t *cluster_dev, const int32_t *n_reads_dev, char *out, int64_t cap,
                                int64_t *n_out, void *stream) {
    if (!ctx || !ctx->tsv || !cluster_dev || !n_reads_dev || !n_out) return FSLRC_ERR_ARG;
    TsvState *T = ctx->tsv;
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    cudaStream_t st = ctx->stream;
    return table_call(ctx, nullptr, [&]() -> int {
        const int L = T->n_lines, TB = 256;
        long long *len; int *any_single;
        DA(len, L); DA(any_single, 1);
        CK(cudaMemsetAsync(any_single, 0, sizeof(int), st));
        if (T->n_reads > 0) KL(tsv::k_tsv_any_single, nblk(T->n_reads, TB), TB, T->n_reads, n_reads_dev, any_single);
        KL(tsv::k_tsv_outlen, nblk(L, TB), TB, L, T->line_start, T->line_end, T->read_id, cluster_dev, n_reads_dev, any_single, len);
        return render_text(ctx, "tsv", L, len, nullptr, out, cap, n_out, [&](const long long *off, unsigned char *d_out) {
            KL(tsv::k_tsv_emit, nblk((int64_t)L * 32, TB), TB, L, T->text, T->line_start, T->line_end, T->read_id, cluster_dev, n_reads_dev,
               any_single, off, d_out);
        });
    });
}
int fslrc_tsv_write_representative_bed(fslrc_ctx *ctx, const int32_t *cluster_dev, const int32_t *n_reads_dev, char *out,
                                       int64_t cap, int64_t *n_out, void *stream) {
    if (!ctx || !ctx->tsv || !cluster_dev || !n_reads_dev || !n_out) return FSLRC_ERR_ARG;
    TsvState *T = ctx->tsv;
    if (!T->score) return fail(ctx, FSLRC_ERR_ARG, "tsv: the table has no alignment_score column");
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    cudaStream_t st = ctx->stream;
    return table_call(ctx, nullptr, [&]() -> int {
        const int L = T->n_lines, R = T->n_reads, TB = 256;
        long long *sum, *len; int *cnt, *err, *any_single, *txt_len; unsigned char *is_rep; char *txt;
        DA(sum, R); DA(cnt, R); DA(is_rep, R); DA(txt_len, R); DA(txt, (int64_t)R * fmtd::FMT_F64_MAX); DA(err, 1); DA(any_single, 1);
        DA(len, L);
        // cluster ids of the clustering are < n_reads, so n_reads bounds them without a read-back; ids from elsewhere are checked
        { int r = choose_alignment_dev(ctx, T->n_rows, R, R, T->read_id, T->score, cluster_dev, sum, cnt, is_rep, nullptr, err); if (r) return r; }
        CK(cudaMemsetAsync(any_single, 0, sizeof(int), st));
        if (R > 0) {
            KL(tsv::k_tsv_any_single, nblk(R, TB), TB, R, n_reads_dev, any_single);
            KL(tsv::k_tsv_rep_mean, nblk(R, TB), TB, R, is_rep, sum, cnt, txt, txt_len);
        }
        KL(tsv::k_tsv_rep_outlen, nblk(L, TB), TB, L, T->line_start, T->line_end, T->read_id, cluster_dev, n_reads_dev, any_single, is_rep, txt_len, len);
        CK(cudaMemcpyAsync(ctx->h_pin + 1, err, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if ((int)(ctx->h_pin[1] & 0xffffffff)) return fail(ctx, FSLRC_ERR_RANGE, "tsv: a cluster id is negative or not below n_reads");
        return render_text(ctx, "tsv", L, len, nullptr, out, cap, n_out, [&](const long long *off, unsigned char *d_out) {
            KL(tsv::k_tsv_rep_emit, nblk((int64_t)L * 32, TB), TB, L, T->text, T->line_start, T->line_end, T->read_id, cluster_dev, n_reads_dev,
               any_single, is_rep, txt, txt_len, off, d_out);
        });
    });
}
int fslrc_tsv_write_edges(fslrc_ctx *ctx, char *out, int64_t cap, int64_t *n_out, void *stream) {
    if (!ctx) return FSLRC_ERR_ARG;
    if (!n_out) return fail(ctx, FSLRC_ERR_ARG, "tsv: null n_out");
    TsvState *T = ctx->tsv;
    const EdgeList *E = ctx->edges;
    if (!T || !E || E->tsv_gen != ctx->tsv_gen || E->read_id_col != T->read_id)
        return fail(ctx, FSLRC_ERR_ARG, "tsv: no captured edge list of a clustering of the table that is open now "
                                        "(fslrc_set_edge_capture, then fslrc_cluster_device on this table's columns)");
    CK(cudaSetDevice(ctx->device));
    ctx->stream = (cudaStream_t)stream;
    cudaStream_t st = ctx->stream;
    return table_call(ctx, nullptr, [&]() -> int {
        const int n = (int)E->n, L = n + 1, TB = 256;
        long long *len;
        DA(len, L);
        KL(tsv::k_tsv_edge_outlen, nblk(L, TB), TB, n, E->read1, E->read2, E->jac, T->first_row, T->q_len, len);
        return render_text(ctx, "tsv", L, len, nullptr, out, cap, n_out, [&](const long long *off, unsigned char *d_out) {
            KL(tsv::k_tsv_edge_emit, nblk((int64_t)L * 32, TB), TB, n, T->text, E->read1, E->read2, E->jac, T->first_row, T->q_off, T->q_len,
               off, d_out);
        });
    });
}
void fslrc_tsv_close(fslrc_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    tsv_free(ctx);
}

#include "bam_abi.inl"

int fslrc_set_blocking_sync(fslrc_ctx *ctx, int on) {
    if (!ctx) return FSLRC_ERR_ARG;
    ctx->blocking = on != 0;
    return 0;
}

int fslrc_set_edge_capture(fslrc_ctx *ctx, int on) {
    if (!ctx) return FSLRC_ERR_ARG;
    ctx->edge_capture = on != 0;
    if (!on && ctx->edges) {
        CK(cudaSetDevice(ctx->device));
        edges_free(ctx);
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return 0;
}

int fslrc_edges(fslrc_ctx *ctx, int32_t *read1, int32_t *read2, double *jaccard, int64_t cap, int64_t *n_edges, void *stream) {
    if (!ctx) return FSLRC_ERR_ARG;
    if (!n_edges) return fail(ctx, FSLRC_ERR_ARG, "edges: null n_edges");
    const EdgeList *E = ctx->edges;
    if (!E) return fail(ctx, FSLRC_ERR_ARG, "edges: the last clustering call captured no edge list (capture off, the call failed, "
                                            "or it was a fslrc_mg_* sequence)");
    *n_edges = E->n;
    if (!read1 && !read2 && !jaccard) return 0;                          // size query
    if (cap < E->n) return fail(ctx, FSLRC_ERR_ARG, "edges: output buffers too small (cap < n_edges)");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (E->n > 0) {
        if (read1) CK(cudaMemcpyAsync(read1, E->read1, sizeof(int32_t) * E->n, cudaMemcpyDeviceToDevice, st));
        if (read2) CK(cudaMemcpyAsync(read2, E->read2, sizeof(int32_t) * E->n, cudaMemcpyDeviceToDevice, st));
        if (jaccard) CK(cudaMemcpyAsync(jaccard, E->jac, sizeof(double) * E->n, cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

long long fslrc_launch_count(const fslrc_ctx *ctx) { return ctx ? ctx->launches : 0; }

int fslrc_int_peak(fslrc_ctx *ctx, double *lane_ops_per_s) {
    if (!ctx || !lane_ops_per_s) return FSLRC_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    int *d; CK(cudaMalloc(&d, 4));
    const int iters = 4096, blocks = n_sms(ctx) * 8, threads = 256;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    k_int_peak<<<blocks, threads>>>(64, d);
    double best = 0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(e0);
        k_int_peak<<<blocks, threads>>>(iters, d);
        cudaEventRecord(e1);
        CK(cudaEventSynchronize(e1));
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        double ops = (double)blocks * threads * (double)iters * 16.0 * 8.0 * 3.0;     // add + min/max + xor per chain step
        best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *lane_ops_per_s = best;
    return 0;
}

}  // extern "C"
