// GPU ingest / egress of `<base>.mappings.bed` (SURVEY §8f row 1): the TSV main.py:209 reads with pandas
// (columns written by collect_mapping_info.py:176-181) and the `<base>.mappings.cluster.bed` main.py:349 writes.
//
//   k_tsv_count / k_tsv_lines   newline positions -> line starts (one pass over the bytes + an exclusive scan)
//   k_tsv_parse                 one thread per line walks the first fields only (the long `seq` column is never touched):
//                               decimal ints of the wanted columns, (offset, length, FNV-1a hash) of qname and chrom
//   k_tsv_intern_*              open-addressing hash table keyed by the 64-bit hash: first row of every distinct string,
//                               byte-for-byte verification against that row, dense ids in order of first appearance
//                               (= pandas.factorize = the singleton numbering order of main.py:336-341)
//   k_tsv_false / k_tsv_row_keep / k_tsv_compact
//                               --filter-false (main.py:229-230, cluster.py:80-86): the reads whose qname contains "False"
//                               leave the table; the kept rows move down in table order and the reads are renumbered densely
//   k_tsv_outlen / k_tsv_emit   every input line + "\t<cluster>.0\t<n_reads>.0" (the float columns of main.py:334-342)
//   k_tsv_rep_mean / k_tsv_rep_outlen / k_tsv_rep_emit
//                               `<base>.mappings.representative.bed` (main.py:351-352): the lines of every cluster's
//                               representative read only, + the same two columns + repr(mean alignment_score)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "fmt_double.cuh"

namespace tsv {

constexpr int CHUNK = 64;                 // bytes per thread in the newline pass
enum { TE_FIELDS = 1, TE_INT = 2, TE_COLLISION = 4, TE_RANGE = 8 };
enum { W_CHROM = 0, W_RSTART, W_REND, W_QNAME, W_NALN, W_ALN, W_QSTART, W_QEND, W_SCORE, W_N };

struct Want { int col[W_N]; int last; };   // field index of every wanted column (-1: absent), highest wanted index

__global__ void k_tsv_count(const unsigned char *__restrict__ text, long long n, int *cnt) {
    const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long b0 = c * CHUNK;
    if (b0 >= n) return;
    int k = 0;
    if (b0 + CHUNK <= n) {
#pragma unroll
        for (int j = 0; j < CHUNK / 16; j++) {
            const uint4 v = __ldg((const uint4 *)(text + b0) + j);
            const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const unsigned x = w[q] ^ 0x0a0a0a0au;                 // bytes equal to '\n' become 0
                k += __popc(((x - 0x01010101u) & ~x & 0x80808080u));
            }
        }
    } else {
        for (long long i = b0; i < n; i++) k += text[i] == '\n';
    }
    cnt[c] = k;
}
// line_start[l] = offset of the first byte of line l (line 0 starts at 0; every '\n' at p starts a line at p + 1)
__global__ void k_tsv_lines(const unsigned char *__restrict__ text, long long n, const int *__restrict__ pre, long long *line_start) {
    const long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long b0 = c * CHUNK;
    if (b0 >= n) return;
    int l = pre[c] + 1;
    const long long b1 = b0 + CHUNK < n ? b0 + CHUNK : n;
    for (long long i = b0; i < b1; i++)
        if (text[i] == '\n') line_start[l++] = i + 1;
    if (c == 0) line_start[0] = 0;
}
__device__ __forceinline__ unsigned long long fnv1a(const unsigned char *p, int len, unsigned long long seed) {
    unsigned long long h = 1469598103934665603ull ^ seed;
    for (int i = 0; i < len; i++) { h ^= p[i]; h *= 1099511628211ull; }
    return h == ~0ull ? 0x1234567ull : h;                              // ~0 marks an empty slot
}
// rows = data lines (line 0 is the header): row r is line r + 1
__global__ void k_tsv_parse(const unsigned char *__restrict__ text, const long long *__restrict__ line_start, int n_rows, Want w,
                            unsigned long long seed, int *rstart, int *rend,
                            int *naln, int *aln, int *qstart, int *qend, int *score, long long *q_off, int *q_len,
                            unsigned long long *q_hash, long long *c_off, int *c_len, unsigned long long *c_hash, int *err) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const long long s = line_start[r + 1], e = line_start[r + 2] - 1;   // [s, e): the line without its '\n'
    long long p = s;
    int vals[W_N];
#pragma unroll
    for (int k = 0; k < W_N; k++) vals[k] = 0;
    int bad = 0;
    for (int f = 0; f <= w.last; f++) {
        long long fe = p;
        while (fe < e && text[fe] != '\t') fe++;
        if (p > e) { bad |= TE_FIELDS; break; }
        int which = -1;
#pragma unroll
        for (int k = 0; k < W_N; k++) if (w.col[k] == f) which = k;
        if (which == W_QNAME) { q_off[r] = p; q_len[r] = (int)(fe - p); q_hash[r] = fnv1a(text + p, (int)(fe - p), seed); }
        else if (which == W_CHROM) { c_off[r] = p; c_len[r] = (int)(fe - p); c_hash[r] = fnv1a(text + p, (int)(fe - p), seed); }
        else if (which >= 0) {
            long long i = p;
            bool neg = false;
            if (i < fe && text[i] == '-') { neg = true; i++; }
            long long v = 0;
            if (i == fe) bad |= TE_INT;
            for (; i < fe; i++) {
                const int d = text[i] - '0';
                if ((unsigned)d > 9u) {                                 // "12.0": a pandas float column that holds integers
                    if (text[i] == '.') { for (long long j = i + 1; j < fe; j++) if (text[j] != '0') bad |= TE_INT; }
                    else bad |= TE_INT;
                    break;
                }
                v = v * 10 + d;
                if (v > 0x7fffffffLL) { bad |= TE_RANGE; v = 0; }
            }
            vals[which] = (int)(neg ? -v : v);
        }
        p = fe + 1;
    }
    if (bad) atomicOr(err, bad);
    rstart[r] = vals[W_RSTART]; rend[r] = vals[W_REND]; naln[r] = vals[W_NALN]; aln[r] = vals[W_ALN];
    qstart[r] = vals[W_QSTART]; qend[r] = vals[W_QEND];
    if (score) score[r] = vals[W_SCORE];
}
// ---- interning: slot table {hash, first row}; capacity is a power of two
__global__ void k_tsv_intern_insert(int n_rows, const unsigned long long *__restrict__ hash, unsigned long long *keys, int *first,
                                    unsigned mask, int *slot_of_row) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const unsigned long long h = hash[r];
    unsigned s = (unsigned)(h ^ (h >> 32)) & mask;
    for (;;) {
        const unsigned long long cur = atomicCAS(&keys[s], ~0ull, h);
        if (cur == ~0ull || cur == h) break;
        s = (s + 1) & mask;
    }
    atomicMin(&first[s], r);
    slot_of_row[r] = s;
}
// every row's string must equal, byte for byte, the string of the first row of its slot (a 64-bit hash collision between
// two different names is reported, never silently merged); is_first flags the first appearance of every distinct string
__global__ void k_tsv_intern_verify(int n_rows, const unsigned char *__restrict__ text, const long long *__restrict__ off,
                                    const int *__restrict__ len, const int *__restrict__ slot_of_row, const int *__restrict__ first,
                                    int *is_first, int *err) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int f = first[slot_of_row[r]];
    is_first[r] = f == r;
    if (f != r) {
        const int l = len[r];
        bool same = len[f] == l;
        const unsigned char *a = text + off[r], *b = text + off[f];
        for (int i = 0; same && i < l; i++) same = a[i] == b[i];
        if (!same) atomicOr(err, TE_COLLISION);
    }
}
__global__ void k_tsv_intern_ids(int n_rows, const int *__restrict__ slot_of_row, const int *__restrict__ first,
                                 const int *__restrict__ id_at_row, int *id, int *first_row_of_id) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int f = first[slot_of_row[r]];
    const int i = id_at_row[f];
    id[r] = i;
    if (f == r && first_row_of_id) first_row_of_id[i] = r;
}
// ---- --filter-false: bed_file[~bed_file["qname"].str.contains("False")] on the parsed table
// every row of a read carries the same name bytes (k_tsv_intern_verify), so the read's first row decides for all of them;
// "False" has no regex metacharacter, so str.contains is a case-sensitive substring search
__global__ void k_tsv_false(int n_reads, const unsigned char *__restrict__ text, const int *__restrict__ first_row,
                            const long long *__restrict__ q_off, const int *__restrict__ q_len, int *keep) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const int f = first_row[r];
    const unsigned char *p = text + q_off[f];
    const int l = q_len[f];
    bool hit = false;
    for (int i = 0; i + 5 <= l && !hit; i++)
        hit = p[i] == 'F' && p[i + 1] == 'a' && p[i + 2] == 'l' && p[i + 3] == 's' && p[i + 4] == 'e';
    keep[r] = !hit;
}
__global__ void k_tsv_row_keep(int n_rows, const int *__restrict__ rid, const int *__restrict__ keep_read, int *keep_row) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_rows) keep_row[r] = keep_read[rid[r]];
}
// the per-row columns of the parsed table; line_start / line_end describe lines (line 0 is the header, row r is line r + 1)
struct Cols {
    int *read_id, *chrom, *rstart, *rend, *aln, *qstart, *qend, *naln, *score;   // score: nullable
    long long *q_off; int *q_len;
    long long *line_start, *line_end;                                           // line_end: nullable (= line_start[l + 1] - 1)
};
// kept row r goes to new_pos[r]; read ids become new_id[read_id] (the kept reads in order of first appearance, which is
// pandas.factorize of the filtered frame).  Chromosome ids keep the numbering of the unfiltered table (main.py:227 numbers
// the chromosomes before :229-230 filters).  The kept lines are no longer contiguous in the text, so every line gets its end.
__global__ void k_tsv_compact(int n_rows, const int *__restrict__ keep_row, const int *__restrict__ new_pos,
                              const int *__restrict__ new_id, const int *__restrict__ first_row, Cols s, Cols d, int *first_row_out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    if (r == 0) { d.line_start[0] = s.line_start[0]; d.line_end[0] = s.line_end ? s.line_end[0] : s.line_start[1] - 1; }
    if (!keep_row[r]) return;
    const int p = new_pos[r], q = s.read_id[r], id = new_id[q];
    d.read_id[p] = id; d.chrom[p] = s.chrom[r]; d.rstart[p] = s.rstart[r]; d.rend[p] = s.rend[r]; d.aln[p] = s.aln[r];
    d.qstart[p] = s.qstart[r]; d.qend[p] = s.qend[r]; d.naln[p] = s.naln[r];
    if (s.score) d.score[p] = s.score[r];
    d.q_off[p] = s.q_off[r]; d.q_len[p] = s.q_len[r];
    d.line_start[p + 1] = s.line_start[r + 1];
    d.line_end[p + 1] = s.line_end ? s.line_end[r + 1] : s.line_start[r + 2] - 1;
    if (first_row[q] == r) first_row_out[id] = p;
}
// ---- egress
// line l without its '\n' is [line_start[l], line_end(l)); line_end == nullptr: the lines are contiguous in the text
__device__ __forceinline__ long long line_end_of(const long long *__restrict__ line_start, const long long *__restrict__ line_end, int l) {
    return line_end ? line_end[l] : line_start[l + 1] - 1;
}
__device__ __forceinline__ int dec_digits(int v) {
    int d = 1;
    unsigned u = v < 0 ? (unsigned)(-(long long)v) : (unsigned)v;
    while (u >= 10u) { u /= 10u; d++; }
    return d + (v < 0);
}
__device__ __forceinline__ unsigned char *put_dec(unsigned char *o, int v) {
    const int nd = dec_digits(v);
    unsigned u = v < 0 ? (unsigned)(-(long long)v) : (unsigned)v;
    if (v < 0) o[0] = '-';
    for (int k = nd - 1; k >= (v < 0); k--) { o[k] = (unsigned char)('0' + u % 10u); u /= 10u; }
    return o + nd;
}
// main.py:334-342: the left merge leaves NaN for singletons, which makes `cluster` / `n_reads` float columns ("12.0");
// a table in which every read ended in a cluster has no NaN and keeps integer columns ("12").  *any_single != 0 <=> floats.
__global__ void k_tsv_any_single(int n_reads, const int *__restrict__ nreads, int *any_single) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const bool s = r < n_reads && nreads[r] == 1;
    if (__syncthreads_or(s) && threadIdx.x == 0) *any_single = 1;
}
// the columns both files append to a data line: "\t<c>.0\t<n>.0" (floats) or "\t<c>\t<n>"
__device__ __forceinline__ int cluster_cols_len(int c, int n, bool fl) { return 2 + dec_digits(c) + dec_digits(n) + (fl ? 4 : 0); }
__device__ __forceinline__ unsigned char *put_cluster_cols(unsigned char *q, int c, int n, bool fl) {
    *q++ = '\t'; q = put_dec(q, c); if (fl) { *q++ = '.'; *q++ = '0'; }
    *q++ = '\t'; q = put_dec(q, n); if (fl) { *q++ = '.'; *q++ = '0'; }
    return q;
}
__device__ __forceinline__ unsigned char *put_str(unsigned char *q, const char *h) { while (*h) *q++ = (unsigned char)*h++; return q; }
// output length of every line: header + "\tcluster\tn_reads\n"; row: line + "\t<c>.0\t<n>.0\n" (floats) or "\t<c>\t<n>\n"
__global__ void k_tsv_outlen(int n_lines, const long long *__restrict__ line_start, const long long *__restrict__ line_end,
                             const int *__restrict__ rid, const int *__restrict__ cluster, const int *__restrict__ nreads,
                             const int *__restrict__ any_single, long long *len) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_lines) return;
    const long long body = line_end_of(line_start, line_end, l) - line_start[l];
    if (l == 0) len[l] = body + 17;                                     // "\tcluster\tn_reads\n"
    else { const int r = rid[l - 1]; len[l] = body + cluster_cols_len(cluster[r], nreads[r], *any_single != 0) + 1; }
}
// one warp per line: coalesced byte copy, lane 0 appends the two columns
__global__ void k_tsv_emit(int n_lines, const unsigned char *__restrict__ text, const long long *__restrict__ line_start,
                           const long long *__restrict__ line_end, const int *__restrict__ rid, const int *__restrict__ cluster,
                           const int *__restrict__ nreads, const int *__restrict__ any_single, const long long *__restrict__ out_off,
                           unsigned char *out) {
    const long long wg = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wg >= n_lines) return;
    const int l = (int)wg;
    const long long s = line_start[l], body = line_end_of(line_start, line_end, l) - s;
    unsigned char *o = out + out_off[l];
    for (long long i = lane; i < body; i += 32) o[i] = text[s + i];
    if (lane == 0) {
        unsigned char *q = o + body;
        if (l == 0) put_str(q, "\tcluster\tn_reads\n");
        else { const int r = rid[l - 1]; q = put_cluster_cols(q, cluster[r], nreads[r], *any_single != 0); *q = '\n'; }
    }
}
// ---- mappings.representative.bed (cluster.py:237-254): is_rep / sum / cnt per read come from the k_ca_* kernels
constexpr int REP_HEADER_LEN = 37;                                      // "\tcluster\tn_reads\tavg_alignment_score\n"
// the mean of every representative read, formatted once per read into a fixed slot: repr(sum / cnt) (pandas' to_csv of
// the float64 column; the same IEEE division k_ca_best ranks the reads by)
__global__ void k_tsv_rep_mean(int n_reads, const unsigned char *__restrict__ is_rep, const long long *__restrict__ sum,
                               const int *__restrict__ cnt, char *txt, int *txt_len) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads || !is_rep[r]) return;
    txt_len[r] = fmtd::fmt_repr_f64(__ddiv_rn((double)sum[r], (double)cnt[r]), txt + (long long)r * fmtd::FMT_F64_MAX);
}
// output length of every line: 0 for the lines of a read that is not its cluster's representative
__global__ void k_tsv_rep_outlen(int n_lines, const long long *__restrict__ line_start, const long long *__restrict__ line_end,
                                 const int *__restrict__ rid, const int *__restrict__ cluster, const int *__restrict__ nreads,
                                 const int *__restrict__ any_single, const unsigned char *__restrict__ is_rep,
                                 const int *__restrict__ txt_len, long long *len) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_lines) return;
    const long long body = line_end_of(line_start, line_end, l) - line_start[l];
    if (l == 0) { len[l] = body + REP_HEADER_LEN; return; }
    const int r = rid[l - 1];
    len[l] = is_rep[r] ? body + cluster_cols_len(cluster[r], nreads[r], *any_single != 0) + 1 + txt_len[r] + 1 : 0;
}
// one warp per kept line: coalesced byte copy, lane 0 appends the cluster columns and the formatted mean
__global__ void k_tsv_rep_emit(int n_lines, const unsigned char *__restrict__ text, const long long *__restrict__ line_start,
                               const long long *__restrict__ line_end, const int *__restrict__ rid,
                               const int *__restrict__ cluster, const int *__restrict__ nreads,
                               const int *__restrict__ any_single, const unsigned char *__restrict__ is_rep,
                               const char *__restrict__ txt, const int *__restrict__ txt_len, const long long *__restrict__ out_off,
                               unsigned char *out) {
    const long long wg = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wg >= n_lines) return;
    const int l = (int)wg;
    const int r = l > 0 ? rid[l - 1] : -1;
    if (l > 0 && !is_rep[r]) return;
    const long long s = line_start[l], body = line_end_of(line_start, line_end, l) - s;
    unsigned char *o = out + out_off[l];
    for (long long i = lane; i < body; i += 32) o[i] = text[s + i];
    if (lane == 0) {
        unsigned char *q = o + body;
        if (l == 0) put_str(q, "\tcluster\tn_reads\tavg_alignment_score\n");
        else {
            q = put_cluster_cols(q, cluster[r], nreads[r], *any_single != 0);
            *q++ = '\t';
            const char *m = txt + (long long)r * fmtd::FMT_F64_MAX;
            for (int i = 0; i < txt_len[r]; i++) *q++ = (unsigned char)m[i];
            *q = '\n';
        }
    }
}

// ---- the similarity graph's edges (fslrc_tsv_write_edges): match_df.to_csv(sep="\t", index=False) of cluster.py:226's frame
constexpr int EDGE_HEADER_LEN = 33;                                     // "query1\tquery2\tjaccard_similarity\n"
// line 0: the header; line l > 0: edge l - 1 = "<qname of read1>\t<qname of read2>\t<repr(jaccard)>\n"
__global__ void k_tsv_edge_outlen(int n_edges, const int *__restrict__ read1, const int *__restrict__ read2, const double *__restrict__ jac,
                                  const int *__restrict__ first_row, const int *__restrict__ q_len, long long *len) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > n_edges) return;
    if (l == 0) { len[0] = EDGE_HEADER_LEN; return; }
    char buf[fmtd::FMT_F64_MAX];
    const int e = l - 1;
    len[l] = (long long)q_len[first_row[read1[e]]] + q_len[first_row[read2[e]]] + fmtd::fmt_repr_f64(jac[e], buf) + 3;
}
// one warp per line: coalesced copies of both names, lane 0 writes the separators and the formatted value
__global__ void k_tsv_edge_emit(int n_edges, const unsigned char *__restrict__ text, const int *__restrict__ read1,
                                const int *__restrict__ read2, const double *__restrict__ jac, const int *__restrict__ first_row,
                                const long long *__restrict__ q_off, const int *__restrict__ q_len, const long long *__restrict__ out_off,
                                unsigned char *out) {
    const long long wg = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wg > n_edges) return;
    const int l = (int)wg;
    unsigned char *o = out + out_off[l];
    if (l == 0) { if (lane == 0) put_str(o, "query1\tquery2\tjaccard_similarity\n"); return; }
    const int e = l - 1, f1 = first_row[read1[e]], f2 = first_row[read2[e]];
    const long long s1 = q_off[f1], s2 = q_off[f2];
    const int n1 = q_len[f1], n2 = q_len[f2];
    for (int i = lane; i < n1; i += 32) o[i] = text[s1 + i];
    for (int i = lane; i < n2; i += 32) o[n1 + 1 + i] = text[s2 + i];
    if (lane == 0) {
        char buf[fmtd::FMT_F64_MAX];
        const int nj = fmtd::fmt_repr_f64(jac[e], buf);
        o[n1] = '\t';
        unsigned char *q = o + n1 + 1 + n2;
        *q++ = '\t';
        for (int i = 0; i < nj; i++) *q++ = (unsigned char)buf[i];
        *q = '\n';
    }
}

}  // namespace tsv
