/* fslr_b200 — C ABI of the B200-native read-clustering step of kcleal/fslr.
 *
 * The reference has no FFI: the boundary it offers is the set of in-process Python calls that
 * /root/reference/fslr/main.py:227-244 makes into /root/reference/fslr/cluster.py.  This header is
 * what a ctypes binding of that step binds instead (INTEGRATION.md shows the stub); each entry
 * point cites the reference interface it replaces.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; return 0 on success, a negative
 * FSLRC_ERR_* otherwise (fslrc_last_error() gives the text); no exception crosses the ABI.  The
 * caller owns every input/output buffer and keeps it alive until the call returns (calls are
 * synchronous with respect to the host: they end with a stream synchronise).  A context belongs to
 * one device and is not re-entrant; separate contexts are independent.  There is NO CPU fallback:
 * every entry point fails with FSLRC_ERR_CUDA when no device is usable.
 */
#ifndef FSLR_B200_H
#define FSLR_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FSLRC_MAX_FILLINGS 64      /* fillings per read after keep_fillings/masking (n_alignments - 2) */
#define FSLRC_N_STAGES 14

enum {
    FSLRC_OK = 0,
    FSLRC_ERR_CUDA = -1,            /* CUDA runtime error, or no device */
    FSLRC_ERR_ARG = -2,             /* null/inconsistent argument */
    FSLRC_ERR_ZERO_DIVISOR = -3,    /* aln_size / qlen2 / n_alignments <= 0 on a filling: the reference raises
                                       ZeroDivisionError at cluster.py:135,179,181 */
    FSLRC_ERR_TOO_MANY_FILLINGS = -4, /* a read has more than FSLRC_MAX_FILLINGS fillings */
    FSLRC_ERR_NALN_NOT_CONSTANT = -5, /* n_alignments differs between rows of one read (the producer,
                                         collect_mapping_info.py:80,122,141, never emits that) */
    FSLRC_ERR_OVERFLOW = -6,        /* internal edge buffer overflow (cannot happen within the stated bounds) */
    FSLRC_ERR_RANGE = -7,           /* a value does not fit the packed device records (n_alignments >= 65536, id out of range) */
    FSLRC_ERR_HASH_COLLISION = -8   /* fslrc_tsv_open: two different names share a 64-bit hash (retry with another seed) */
};

typedef struct fslrc_ctx fslrc_ctx;

/* `<name>.mappings.bed` in columnar form, one entry per alignment row in table order
 * (replaces the DataFrame main.py:209 reads; columns as written by collect_mapping_info.py:176-181).
 * read_id is the dense id of `qname` in order of first appearance, chrom the integer id
 * cluster.rename_chromosomes assigns (cluster.py:34-43; only equality is used). */
typedef struct {
    int64_t n_rows;
    int64_t n_reads;
    const int32_t *read_id;        /* [n_rows] 0..n_reads-1 */
    const int32_t *chrom;          /* [n_rows] 0..n_chrom-1 */
    const int32_t *rstart;         /* [n_rows] */
    const int32_t *rend;           /* [n_rows] */
    const int32_t *aln_size;       /* [n_rows] */
    const int32_t *qstart;         /* [n_rows] */
    const int32_t *qend;           /* [n_rows] */
    const int32_t *n_alignments;   /* [n_rows] */
    /* optional: the permutation cluster.py:114 (`sort_values('start')`, an UNSTABLE sort) applies to the
     * frame keep_fillings returns, as indices into that frame in bed order; NULL = stable sort on the GPU
     * (ties keep bed order).  n_order must equal the number of fillings when given. */
    const int32_t *order;
    int64_t n_order;
    /* optional narrow forms of the columns (the table's wire format: 13.25 instead of 32 bytes per row over PCIe / NVLink):
     * when non-NULL they replace the int32 column of the same name, which may then be NULL, and are widened on the device.
     * Accepted by the host-buffer call and by the device-resident calls alike (pointers of the same kind as the columns). */
    const uint8_t *chrom_u8;       /* [n_rows] chromosome id < 256 */
    const uint16_t *n_alignments_u16; /* [n_rows] */
    const uint8_t *rows_per_read_u8; /* [n_reads] number of rows of every read when the rows of a read are contiguous and the
                                      reads appear in id order (every count in 1..255); `read_id` may then be NULL and is
                                      rebuilt on the device */
    int64_t aln_size_is_qspan;     /* non-zero: every row has aln_size == qend - qstart (what collect_mapping_info.py:88
                                      writes); `aln_size` may then be NULL and is derived on the device */
    const int16_t *rspan_i16;      /* [n_rows] rend - rstart when every difference fits int16: replaces `rend` */
    const uint16_t *qstart_u16;    /* [n_rows] when every qend < 65536: replace `qstart` / `qend` */
    const uint16_t *qend_u16;
} fslrc_table;

/* The options of main.py:33-37,219-223,237 in numeric form.  The three `*_c`/umax fields are computed by the
 * host in the reference's own double arithmetic (Python floats) so no rounding decision is re-made here. */
typedef struct {
    double overlap;                /* --overlap            (main.py:34,220; cluster.py:157) */
    double qlen_c;                 /* 1 - qlen_diff        (cluster.py:179) */
    double naln_c;                 /* 1 - n_alignment_diff (cluster.py:181) */
    int32_t umax[FSLRC_MAX_FILLINGS + 1]; /* umax[n] = largest union with n/union >= cutoff(n), n-1 if none
                                       (cluster.py:165-170,218-219); umax[0] unused */
    int64_t edge_threshold;        /* main.py:221 */
    int32_t n_chrom;
    const int64_t *chrom_len;      /* [n_chrom] host pointer; 0 = chromosome not in the BAM header (cluster.py:99) */
    const uint8_t *chrom_masked;   /* [n_chrom] host pointer; 1 = named in --cluster-mask (cluster.py:96) */
    int32_t mask_subtelomere;      /* 'subtelomere' in mask (cluster.py:98) */
    int64_t subtel;                /* 500000 (main.py:237) */
} fslrc_params;

typedef struct {
    int64_t n_fillings;            /* rows left by keep_fillings (cluster.py:14-31) */
    int64_t n_intervals;           /* after mask_sequences2 (cluster.py:89-106) */
    int64_t n_query_reads;         /* reads with >= 1 interval (cluster.py:189-191) */
    int64_t band_pairs;            /* interval-level candidate pairs {i<j<=ub(i)} (what search_values can return) */
    int64_t pair_tests;            /* full read-pair tests evaluated on the GPU (a10+a11+a13 of SURVEY §8a) */
    int64_t relation_entries;      /* passing (query, other) pairs recorded by the pair stage */
    int64_t saturating_reads;      /* reads that can reach edge_threshold (replayed in query order) */
    int64_t edges;                 /* edges handed to union-find */
    int64_t components;            /* clusters with >= 2 reads */
    int64_t clustered_reads;       /* reads in those clusters */
    int64_t partner_records;       /* partner records the pair kernel left for the replay of saturating reads */
    int32_t no_clusters;           /* main.py:247-249: the reference prints "No clusters were found." and returns */
    int32_t reserved;
    float stage_ms[FSLRC_N_STAGES];/* CUDA-event time per stage, see fslrc_stage_name() */
} fslrc_stats;

int fslrc_create(int device, fslrc_ctx **out);
void fslrc_destroy(fslrc_ctx *ctx);
const char *fslrc_last_error(const fslrc_ctx *ctx);
const char *fslrc_stage_name(int stage);
int fslrc_version(void);
/* number of kernels launched through `ctx` so far (every kernel on the path is this library's own: no CUB / Thrust) */
long long fslrc_launch_count(const fslrc_ctx *ctx);

/* The whole step, main.py:233-257,334-342 (keep_fillings -> prepare_data -> build_interval_trees ->
 * query_interval_trees -> get_subgraphs -> cluster / n_reads columns), on DEVICE-resident columns.
 * out_cluster / out_n_reads: device int32 [n_reads] indexed by read_id: the `cluster` and `n_reads`
 * values the reference writes for that read's rows (as integers; the reference stores them as floats).
 * `stream` is a cudaStream_t (NULL = default stream). */
int fslrc_cluster_device(fslrc_ctx *ctx, const fslrc_table *table, const fslrc_params *params,
                         int32_t *out_cluster, int32_t *out_n_reads, fslrc_stats *stats, void *stream);

/* Same with HOST buffers (pinned recommended): copies the columns in, runs, copies both outputs back. */
int fslrc_cluster_host(fslrc_ctx *ctx, const fslrc_table *table, const fslrc_params *params,
                       int32_t *out_cluster, int32_t *out_n_reads, fslrc_stats *stats, void *stream);

/* The `start` column of the frame keep_fillings returns (cluster.py:14-31,111): min(rstart, rend) of every row that is
 * neither the first nor the last row of its read in table order, in table order.  This is the column cluster.py:114 sorts:
 * sorting it on the host with the reference's own call gives the `order` fslrc_cluster_device takes (the reference's tie
 * order, which depends on the host's numpy and CPU, so it is not reproduced on the device).  The rows of a read need not be
 * contiguous; a read with 1 or 2 rows contributes nothing.
 * `table`: wide DEVICE columns (read_id, rstart, rend; n_rows, n_reads), as fslrc_tsv_open / fslrc_bam_open leave them.
 * out_start: device int32 [cap], cap >= n_rows.  *n_fillings: host.  FSLRC_ERR_ARG: null pointers, cap too small,
 * wire-format-only table.  FSLRC_ERR_RANGE: a read_id outside [0, n_reads). */
int fslrc_filling_starts(fslrc_ctx *ctx, const fslrc_table *table, int32_t *out_start, int64_t cap, int64_t *n_fillings,
                         void *stream);

/* ---- multi-GPU staging (SURVEY §8e): the interval table is replicated, the pair space is sharded ----
 * fslrc_mg_prepare     : ingestion + sort/band on this device (identical on every rank)
 * fslrc_mg_pair        : candidate generation + pair tests for the query reads of shard `rank` of `world`; leaves one
 *                        counter word per query read (passing partners / partners of the reads this rank owns, 0 for the
 *                        others) in a device int32 [n_query_reads] buffer (*counts) that the caller SUM-all-reduces in place
 * fslrc_mg_partners    : after the all-reduce: the saturating set, and this rank's recorded pairs (a, b | flags: int32
 *                        pairs) of the saturating reads whose partner lists the replay needs (*pairs, device); the caller
 *                        all-gathers them — 8 bytes per pair instead of re-evaluating the pairs on every rank
 * fslrc_mg_replay      : takes the all-gathered pairs: partner records, replay of saturating reads (replicated, it is
 *                        sequential) and union-find over this rank's edges; leaves a spanning forest (int32 pairs) in *forest
 * fslrc_mg_finish      : takes the all-gathered forests, final union-find + numbering
 */
int fslrc_mg_prepare(fslrc_ctx *ctx, const fslrc_table *table, const fslrc_params *params, void *stream);
int fslrc_mg_pair(fslrc_ctx *ctx, int rank, int world, int32_t **counts, int64_t *n_counts);
int fslrc_mg_partners(fslrc_ctx *ctx, int rank, int world, int32_t **pairs, int64_t *n_pairs);
int fslrc_mg_replay(fslrc_ctx *ctx, int rank, int world, const int32_t *all_pairs, int64_t n_all_pairs,
                    int32_t **forest, int64_t *n_forest_edges);
int fslrc_mg_finish(fslrc_ctx *ctx, const int32_t *all_forest, int64_t n_edges,
                    int32_t *out_cluster, int32_t *out_n_reads, fslrc_stats *stats);

/* cluster.choose_alignment (cluster.py:237-254; main.py:351-352): the representative read of every cluster = the read with
 * the highest mean alignment_score over its rows (double division of the integer sum by the row count, as pandas'
 * groupby.mean), the read whose first row comes first in the table on ties (DataFrame.idxmax).  HOST buffers.
 * cluster: [n_reads] cluster id per read (0..n_clusters-1; reads without rows are ignored); out_is_rep: [n_reads] 1 for the
 * reads the reference would keep in <base>.mappings.representative.bed; out_rep_read: [n_clusters] or NULL. */
int fslrc_choose_alignment_host(fslrc_ctx *ctx, int64_t n_rows, int64_t n_reads, int64_t n_clusters, const int32_t *read_id,
                                const int32_t *alignment_score, const int32_t *cluster, uint8_t *out_is_rep,
                                int32_t *out_rep_read, void *stream);

/* ---- `<base>.mappings.bed` ingest / egress on the GPU (SURVEY §8f row 1) ----
 * fslrc_tsv_open parses the TSV main.py:209 reads with pandas (header + the columns collect_mapping_info.py:176-181 writes;
 * only chrom, rstart, rend, qname, n_alignments, aln_size, qstart, qend[, alignment_score] are decoded) and leaves the
 * columnar table ON THE DEVICE: `info` holds device pointers that can go straight into fslrc_table for
 * fslrc_cluster_device.  read_id / chrom are dense ids in order of first appearance (pandas.factorize).  The parsed table
 * lives in the context until fslrc_tsv_close (or the next fslrc_tsv_open).
 * fslrc_tsv_write_cluster_bed renders `<base>.mappings.cluster.bed` (main.py:349): every input line followed by the float
 * columns `cluster` and `n_reads` (main.py:334-342), header included, into a HOST buffer (out == NULL: size query). */
typedef struct {
    int64_t n_rows, n_reads;
    int32_t n_chrom, has_score;
    const int32_t *read_id, *chrom, *rstart, *rend, *aln_size, *qstart, *qend, *n_alignments, *alignment_score;  /* device */
    float parse_ms;                /* device time of the parse (after the upload) */
    float filter_ms;               /* device time of fslrc_tsv_delete_false (0 until it runs) */
} fslrc_tsv_info;
int fslrc_tsv_open(fslrc_ctx *ctx, const char *text, int64_t n_bytes, uint64_t hash_seed, fslrc_tsv_info *info, void *stream);
/* fslrc_tsv_delete_false applies --filter-false (main.py:229-230, cluster.py:80-86: bed_file[~qname.str.contains("False")])
 * to the table fslrc_tsv_open left in the context: every row of every read whose qname contains the bytes "False" (case
 * sensitive) leaves the table.  The kept rows keep their order; read ids are renumbered densely in order of first appearance
 * (pandas.factorize of the filtered frame); chromosome ids and names stay those of the unfiltered table (main.py:227 numbers
 * them before the filter).  Rewrites info->n_rows, n_reads, the device column pointers and filter_ms; the pointers an
 * earlier info held are invalid afterwards when rows were removed.  fslrc_tsv_read_names and both renderers then describe
 * the kept rows.  A second call removes nothing.  FSLRC_ERR_ARG without an open table. */
int fslrc_tsv_delete_false(fslrc_ctx *ctx, fslrc_tsv_info *info, void *stream);
int fslrc_tsv_chrom_name(fslrc_ctx *ctx, int32_t chrom_id, char *buf, int32_t cap);     /* returns the length */
int fslrc_tsv_read_names(fslrc_ctx *ctx, int64_t *offsets, int32_t *lengths);           /* [n_reads]: where each qname sits in `text` */
int fslrc_tsv_write_cluster_bed(fslrc_ctx *ctx, const int32_t *cluster_dev, const int32_t *n_reads_dev, char *out, int64_t cap,
                                int64_t *n_out, void *stream);
/* fslrc_tsv_write_representative_bed renders `<base>.mappings.representative.bed` (main.py:351-352, cluster.py:237-254) the
 * same way: the header + "\tcluster\tn_reads\tavg_alignment_score", then, in table order, every line of each cluster's
 * representative read (highest mean alignment_score, the read whose first row comes first on ties) with the two columns
 * above and the read's mean score as Python's repr of the double sum / count.  cluster_dev / n_reads_dev: [n_reads] device
 * arrays, as fslrc_cluster_device leaves them.  FSLRC_ERR_ARG when the table has no alignment_score column;
 * FSLRC_ERR_RANGE when a cluster id is negative or >= n_reads. */
int fslrc_tsv_write_representative_bed(fslrc_ctx *ctx, const int32_t *cluster_dev, const int32_t *n_reads_dev, char *out,
                                       int64_t cap, int64_t *n_out, void *stream);
void fslrc_tsv_close(fslrc_ctx *ctx);

/* ---- The producer of `<base>.mappings.bed` (SURVEY §8f row 4): replaces collect_mapping_info.mapping_info
 * (/root/reference/fslr/collect_mapping_info.py:19-181; called from main.py:181-183).  `bam` is the UNCOMPRESSED BAM stream
 * (BGZF blocks inflated by the caller) in host memory; `first_record` is the offset of the first alignment record (after the
 * header text and the reference list).  Record boundaries are walked on the host, everything else runs on the device:
 * CIGAR / aux parsing, grouping by read name, the primary record, the missing-bread rule for single-alignment reads, the two
 * sorts, short_anchor<50bp, region overlaps.  The table stays on the device (rows in the order of :174) until
 * fslrc_bam_close; `read_id` numbers the reads in order of first appearance in that order, so the columns feed
 * fslrc_cluster_device directly.  Inputs the reference stops on (no primary record, primary without sequence, no AS tag,
 * record without CIGAR, read name without two primer tokens, unknown primer) return FSLRC_ERR_ARG with a message. */
typedef struct {
    int64_t n_records;             /* alignment records in the file */
    int64_t n_mapped;              /* of those, without flag 0x4 */
    int64_t n_reads;               /* distinct read names among them */
    int64_t n_rows;                /* table rows: mapped records + inferred primer rows */
    int32_t n_chrom;               /* chrom ids: [0, n_ref) references, n_ref + k = primer k (inferred rows, :124,143) */
    int32_t overlaps_as_float;     /* regions given and an inferred row exists: pandas holds overlaps_region as float (NaN there) */
    const int32_t *read_id, *chrom, *rstart, *rend, *n_alignments, *aln_size, *qstart, *qend, *strand /* 1 = '-' */,
                  *mapq, *qlen, *alignment_score, *short_anchor, *inferred_by_primer, *overlaps_region /* -1 = absent */;  /* device */
    float parse_ms;
    int32_t reserved;
} fslrc_bam_info;
int fslrc_bam_open(fslrc_ctx *ctx, const uint8_t *bam, int64_t n_bytes, int64_t first_record, int32_t n_ref,
                   const char *primer_names /* n_primers NUL-terminated strings back to back */, const int32_t *primer_seq_len, int32_t n_primers,
                   const int32_t *region_chrom, const int32_t *region_start, const int32_t *region_end, int32_t n_regions /* -1: no regions file */,
                   uint64_t hash_seed, fslrc_bam_info *info, void *stream);
/* The same from the COMPRESSED file bytes: BGZF blocks are inflated on the device (one warp per block) and the record
 * boundaries are found there as well, so only the compressed bytes cross PCIe.  first_record / n_ref come from the caller's
 * parse of the BAM header (the first blocks).  info->reserved is 1 when the device's record-boundary guess failed its chain
 * check and the host walk ran instead (same result).  Every block is checked as htslib checks it: its inflated length
 * against ISIZE (a mismatch is reported as corrupt DEFLATE data), then the CRC-32 of its inflated bytes against the CRC32
 * field of its trailer (on the device, one warp per block).  A CRC mismatch returns FSLRC_ERR_ARG with a message naming the
 * first bad block and its offset in the file; a DEFLATE error is reported before it.  The context stays usable. */
int fslrc_bam_open_bgzf(fslrc_ctx *ctx, const uint8_t *file, int64_t n_bytes, int64_t first_record, int32_t n_ref,
                        const char *primer_names, const int32_t *primer_seq_len, int32_t n_primers,
                        const int32_t *region_chrom, const int32_t *region_start, const int32_t *region_end, int32_t n_regions,
                        uint64_t hash_seed, fslrc_bam_info *info, void *stream);
int fslrc_bam_read_stream(fslrc_ctx *ctx, uint8_t *out, int64_t cap, int64_t *n);   /* the inflated stream (read names live there) */
/* Renders the TSV of :176-181.  chrom_names: n_chrom NUL-terminated strings back to back (references, then primers).
 * With out == NULL only *n_out is computed. */
int fslrc_bam_write_mappings_bed(fslrc_ctx *ctx, const char *chrom_names, const char *fslr_version, char *out, int64_t cap,
                                 int64_t *n_out, void *stream);
int fslrc_bam_read_names(fslrc_ctx *ctx, int64_t *offsets, int32_t *lengths);   /* [n_reads], by read_id: where each qname sits in `bam` */
void fslrc_bam_close(fslrc_ctx *ctx);

/* on != 0: the waits inside fslrc_cluster_host / fslrc_cluster_device put the calling thread to sleep (blocking-sync event)
 * instead of spinning — for contexts driven concurrently from several host threads (one context per thread). */
int fslrc_set_blocking_sync(fslrc_ctx *ctx, int on);

/* ---- The similarity graph (cluster.py:187-227 returns it as match_df and the nx.Graph G) ----
 * on != 0: every later fslrc_cluster_device / fslrc_cluster_host call also builds the list of the edges it handed to
 * union-find (stats.edges of them) and keeps it in the context until the next clustering call, fslrc_destroy, or
 * fslrc_set_edge_capture(ctx, 0), which frees it.  Off (the default), the clustering launches no extra kernel and allocates
 * nothing.  The fslrc_mg_* sequence captures nothing (multi-GPU export is not implemented).
 * Each edge is the directed pair (read1, read2) of read ids: read1 is the read whose query tested the pair (cluster.py:197's
 * query_key, match_df's query1).  jaccard is cluster.py:140-170's intersection / union in that direction (list1 = read1's
 * fillings), as the same IEEE double division.  The list is sorted by (query rank of read1, query rank of read2), query rank
 * = the order in which cluster.py:197 visits the query reads, and does not depend on scheduling. */
int fslrc_set_edge_capture(fslrc_ctx *ctx, int on);
/* Copies the captured list into DEVICE buffers of at least `cap` elements (any of the three may be NULL; all NULL: only
 * *n_edges is set).  FSLRC_ERR_ARG when the last clustering call ran without capture, failed, or was a fslrc_mg_* sequence,
 * and when cap < *n_edges. */
int fslrc_edges(fslrc_ctx *ctx, int32_t *read1, int32_t *read2, double *jaccard, int64_t cap, int64_t *n_edges, void *stream);
/* Renders the captured list as match_df.to_csv(sep="\t", index=False) writes it: the header "query1\tquery2\tjaccard_similarity"
 * and one line per edge, "<qname>\t<qname>\t<repr(jaccard)>", into a HOST buffer (out == NULL: size query), with the qnames of
 * the parsed table.  FSLRC_ERR_ARG unless the list was captured by a clustering of the columns of the table that is open
 * now (not before a later fslrc_tsv_open or fslrc_tsv_delete_false). */
int fslrc_tsv_write_edges(fslrc_ctx *ctx, char *out, int64_t cap, int64_t *n_out, void *stream);

/* Integer-issue microbenchmark used as the pair-kernel roofline denominator (SURVEY §8d): returns the measured
 * dependent-free IADD3/LOP3/VIMNMX lane-ops per second on this device. */
int fslrc_int_peak(fslrc_ctx *ctx, double *lane_ops_per_s);

#ifdef __cplusplus
}
#endif
#endif
