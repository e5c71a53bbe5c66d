// Part of fslr_b200.cu (one translation unit; included after the error flags, LMAX and fslr_b200.h are defined).
// Kernels of the ingest stages 1-5: keep_fillings, data order + mask, query rank and per-read lists, IntervalMap order,
// sorted / read-major records and bands.
#pragma once

// ---------------------------------------------------------------- small utility kernels
template <typename T>
__global__ void k_fill(T *p, int64_t n, T v) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
// narrow wire columns -> the int32 columns the kernels read (any source pointer may be NULL: that column is wide already)
struct Widen {
    const unsigned char *c8; const unsigned short *n16, *qs16, *qe16; const short *span16;
    int *chrom, *naln, *qstart, *qend, *rend, *aln;      // destinations (NULL = nothing to do); aln = qend - qstart
    const int *rstart;
};
__global__ void k_widen(int64_t n, Widen w) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (w.c8) w.chrom[i] = w.c8[i];
    if (w.n16) w.naln[i] = w.n16[i];
    if (w.qs16) w.qstart[i] = w.qs16[i];
    if (w.qe16) w.qend[i] = w.qe16[i];
    if (w.span16) w.rend[i] = w.rstart[i] + (int)w.span16[i];
    if (w.aln) w.aln[i] = w.qend[i] - w.qstart[i];                     // aln_size = qend - qstart (collect_mapping_info.py:88)
}
__global__ void k_widen_u8(int64_t n, const unsigned char *__restrict__ in, int *out) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}
// read ids from run lengths (host calls with rows_per_read): read r owns the rows [first[r], first[r] + cnt[r])
__global__ void k_rid_from_runs(int R, int A, const int *__restrict__ first, const int *__restrict__ cnt, int *rid) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int f = first[r], n = cnt[r];
    for (int j = 0; j < n; j++) if (f + j < A) rid[f + j] = r;
}
__global__ void k_iota(int *p, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = i;
}

// exact threshold in the reference's double arithmetic: min{o >= 0 : fl(o/a) >= p}  (cluster.py:133-136,179,181)
__device__ __forceinline__ int thr_f64(int a, double p) {
    if (!(p > 0.0)) return 0;
    double da = (double)a;
    double x = ceil(__dmul_rn(p, da));
    if (x >= 2147483000.0) return 2147483647;
    long long o = (long long)x;
    while (o > 0 && __ddiv_rn((double)(o - 1), da) >= p) --o;
    while (__ddiv_rn((double)o, da) < p) ++o;
    return (int)o;
}

// ---------------------------------------------------------------- stage 1: keep_fillings (cluster.py:14-31)
__global__ void k_first_last(int A, int R, const int *__restrict__ rid, int *first, int *last, int *err) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A) return;
    int r = rid[i];
    if ((unsigned)r >= (unsigned)R) { atomicOr(err, EF_RANGE); return; }
    atomicMin(&first[r], i);
    atomicMax(&last[r], i);
}
__global__ void k_keep(int A, int R, const int *__restrict__ rid, const int *__restrict__ first, const int *__restrict__ last,
                       const int *__restrict__ qstart, const int *__restrict__ qend, int *flag, int *qmin, int *qmax) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A) return;
    int r = rid[i];
    int keep = 0;
    if ((unsigned)r < (unsigned)R) {
        keep = (i != first[r] && i != last[r]);
        if (keep && qmin) { atomicMax(&qmax[r], qend[i]); atomicMin(&qmin[r], qstart[i]); }   // (qmin == NULL: flags only)
    }
    flag[i] = keep;
}
// the `start` column of the fillings frame (cluster.py:111), in bed order: min(rstart, rend) of every kept row at its filling index
__global__ void k_filling_starts(int A, const int *__restrict__ flag, const int *__restrict__ pos, const int *__restrict__ rstart,
                                 const int *__restrict__ rend, int *start) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < A && flag[i]) start[pos[i]] = min(rstart[i], rend[i]);
}
// fillings in bed order as packed records: FR0[k] = {read_id, chrom, start, end}, FR1[k] = {aln_size, n_alignments}
// (start/end = min/max of rstart, rend: cluster.py:111-112).  One coalesced pass over the kept rows.
__global__ void k_fill_records(int A, const int *__restrict__ flag, const int *__restrict__ pos, const int *__restrict__ rid,
                               const int *__restrict__ chrom, const int *__restrict__ rstart, const int *__restrict__ rend,
                               const int *__restrict__ aln, const int *__restrict__ naln, int n_chrom, int4 *FR0, int2 *FR1, int *err) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A || !flag[i]) return;
    const int k = pos[i];
    const int c = chrom[i], rs = rstart[i], re = rend[i];
    if ((unsigned)c >= (unsigned)n_chrom || min(rs, re) < 0) atomicOr(err, EF_RANGE);
    FR0[k] = make_int4(rid[i], c, min(rs, re), max(rs, re));
    FR1[k] = make_int2(aln[i], naln[i]);
}

// ---------------------------------------------------------------- stage 2: prepare_data + mask (cluster.py:109-121, 89-106)
__device__ __forceinline__ bool is_masked(const int4 f, int n_chrom, const long long *__restrict__ clen,
                                          const unsigned char *__restrict__ cmasked, int sub_on, long long subtel) {
    if ((unsigned)f.y >= (unsigned)n_chrom) return true;
    bool masked = cmasked[f.y] != 0;                                          // cluster.py:96
    const long long cl = clen[f.y];
    if (sub_on && cl > 1000000 && ((long long)f.z < subtel || cl - (long long)f.w < subtel)) masked = true;   // :94,98-100
    return masked;
}
// flags over the fillings taken in the order `perm` (NULL = bed order)
__global__ void k_mask_flags(int F, const int *__restrict__ perm, const int4 *__restrict__ FR0, int n_chrom,
                             const long long *__restrict__ clen, const unsigned char *__restrict__ cmasked, int sub_on,
                             long long subtel, int *flag, int *err) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= F) return;
    int fk = k;
    if (perm) { fk = perm[k]; if ((unsigned)fk >= (unsigned)F) { atomicOr(err, EF_RANGE); flag[k] = 0; return; } }
    flag[k] = is_masked(FR0[fk], n_chrom, clen, cmasked, sub_on, subtel) ? 0 : 1;
}
// unmasked fillings, compacted: sort key (start) + filling index, or directly the data-order list when perm is given
__global__ void k_compact_fillings(int F, const int *__restrict__ perm, const int *__restrict__ flag, const int *__restrict__ pos,
                                   const int4 *__restrict__ FR0, int *key, int *val) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= F || !flag[k]) return;
    const int fk = perm ? perm[k] : k;
    const int u = pos[k];
    if (key) key[u] = FR0[fk].z;
    val[u] = fk;
}
// data items in data order: IT0[d] = {read_id, chrom, start, end}, IT1[d] = {aln_size, n_alignments}
__global__ void k_build_items(int D, const int *__restrict__ dfill, const int4 *__restrict__ FR0, const int2 *__restrict__ FR1,
                              int4 *IT0, int2 *IT1, int *firstdp, int *err) {
    int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const int fk = dfill[d];
    const int4 f0 = FR0[fk];
    const int2 f1 = FR1[fk];
    IT0[d] = f0; IT1[d] = f1;
    if (f1.x <= 0 || f1.y <= 0) atomicOr(err, EF_ZERO);
    if (f1.y >= 65535) atomicOr(err, EF_RANGE);
    atomicMin(&firstdp[f0.x], d);
}

// ---------------------------------------------------------------- stage 3: query rank (cluster.py:189-191) + per-read lists
__global__ void k_is_first(int D, const int4 *__restrict__ IT0, const int *__restrict__ firstdp, int *flag) {
    int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < D) flag[d] = (firstdp[IT0[d].x] == d);
}
__global__ void k_rank_reads(int R, const int *__restrict__ firstdp, const int *__restrict__ rank_at, int *q_of_rid, int *rid_of_q) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    int f = firstdp[r];
    int q = -1;
    if (f != 0x7fffffff) { q = rank_at[f]; rid_of_q[q] = r; }
    q_of_rid[r] = q;
}
__global__ void k_item_q(int D, const int4 *__restrict__ IT0, const int *__restrict__ q_of_rid, int *it_q) {
    int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < D) it_q[d] = q_of_rid[IT0[d].x];
}
// rm order: items grouped by query rank, data order inside a read
__global__ void k_read_bounds(int D, const int *__restrict__ qs /*sorted q*/, const int *__restrict__ rm_dp, int *rmidx, int *off, int *len_end) {
    int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= D) return;
    int q = qs[m];
    rmidx[rm_dp[m]] = m;
    if (m == 0 || qs[m - 1] != q) off[q] = m;
    if (m == D - 1 || qs[m + 1] != q) len_end[q] = m + 1;
}
// per read: RI[q] = {qlen2, Lq, n_alignments | Ln << 16, off << 6 | (L - 1)}: the ratio thresholds of
// cluster.py:26-29,178-183 and where the read's fillings live in read-major order
__global__ void k_read_info(int Q, const int *__restrict__ rid_of_q, const int *__restrict__ off, const int *__restrict__ len_end,
                            const int *__restrict__ rm_dp, const int2 *__restrict__ IT1, const int *__restrict__ qmin,
                            const int *__restrict__ qmax, double qlen_c, double naln_c, int4 *RI, int *err) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    int r = rid_of_q[q], o = off[q], L = len_end[q] - o;
    if (L > LMAX) { atomicOr(err, EF_TOOMANY); L = LMAX; }
    long long ql = (long long)qmax[r] - (long long)qmin[r];
    int na = IT1[rm_dp[o]].y;
    if (ql <= 0 || na <= 0) { atomicOr(err, EF_ZERO); ql = ql <= 0 ? 1 : ql; na = na <= 0 ? 1 : na; }
    if (ql > 0x7fffffffLL) { atomicOr(err, EF_RANGE); ql = 1; }
    int Ln = thr_f64(na, naln_c);
    if (Ln > 65535) Ln = 65535;
    RI[q] = make_int4((int)ql, thr_f64((int)ql, qlen_c), (na & 0xffff) | (Ln << 16), (int)(((unsigned)o << 6) | (unsigned)((L - 1) & 63)));
}
// ---------------------------------------------------------------- stage 4/5: IntervalMap order + records + bands
__global__ void k_end_keys(int D, const int4 *__restrict__ IT0, unsigned *key) {
    int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < D) key[d] = ~(unsigned)IT0[d].w;                        // ascending ~end == end descending
}
__global__ void k_gather_key(int D, const int *__restrict__ dp_in, const int4 *__restrict__ IT0, int which, unsigned *key) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < D) { const int4 it = IT0[dp_in[k]]; key[k] = (unsigned)(which ? it.y : it.z); }      // start / chromosome of the item
}
// IntervalMap order without sorting by start again: data order is already sorted by start, so a STABLE partition by
// chromosome yields (chrom, start, data order); what is missing is "end descending" inside runs of equal (chrom, start).
// Those runs are short (PCR duplicates), and in data order their members sit in one block of equal starts: every item
// counts, with coalesced neighbour reads, how many members of its run precede it in data order (idx) and how many must
// precede it in the final order (rank: larger end, or equal end and earlier in data order).  The partition moves the run
// as a block, so the item's final position is its partition position + (rank - idx).  val[d] = d | (rank - idx + 32) << 26.
// Runs that do not fit the window raise `overflow` and the caller falls back to the two full radix sorts.
#define TIE_WIN 48
__global__ void k_tie_delta(int D, const int4 *__restrict__ IT0, unsigned *ckey, unsigned *val,
                            unsigned long long *overflow, int *err) {
    int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const int4 me = IT0[d];
    if (d > 0 && IT0[d - 1].z > me.z) atomicOr(err, EF_RANGE);       // a caller-supplied `order` that does not sort by start
    int idx = 0, rank = 0;
    bool ovf = false;
    for (int k = 1;; k++) {                                          // earlier in data order
        if (d - k < 0) break;
        const int4 o = IT0[d - k];
        if (o.z != me.z) break;
        if (k > TIE_WIN) { ovf = true; break; }
        if (o.y == me.y) { idx++; rank += o.w >= me.w; }
    }
    for (int k = 1;; k++) {                                          // later in data order
        if (d + k >= D) break;
        const int4 o = IT0[d + k];
        if (o.z != me.z) break;
        if (k > TIE_WIN) { ovf = true; break; }
        if (o.y == me.y) rank += o.w > me.w;
    }
    if (idx > 31 || rank > 31) ovf = true;
    if (ovf) { atomicAdd(overflow, 1ull); rank = idx; }
    ckey[d] = (unsigned)me.y;
    val[d] = (unsigned)d | ((unsigned)(rank - idx + 32) << 26);
}
__global__ void k_apply_delta(int D, const unsigned *__restrict__ val, int *s_dp) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= D) return;
    const unsigned v = val[p];
    s_dp[p + (int)(v >> 26) - 32] = (int)(v & 0x3ffffffu);
}
// SR0[p] = {start, end, T, q | fi << 26} (fi = index of the filling in its read's list); SR1[p] = the read's RI record;
// RM[2m] = {chrom, start, end, T}, RM[2m+1] = {pos, ub (closed band, replay), lbT, ubT (tight band, pair kernel)}: one
// 32-byte sector per filling in read-major order, written once by k_bands
#define QMASK 0x3ffffff
#define PCAP 128                // a sorted position whose tight band is longer makes its read "heavy" (kernels_hits.cuh)
#define EB_NOPASS 0x80000000u   // entry.y bit 31: b is a partner of a (n > 0) but a -> b fails the Jaccard cutoff
#define EB_HEAVY 0x40000000u    // entry.y bit 30: recorded by k_pair for a heavy read (its partner records exist already)
#define EB_SYM 0x20000000u      // entry.y bit 29: symmetric mode, the slot also stands for the reverse directed pair (b, a) ...
#define EB_NOPASS2 0x10000000u  // entry.y bit 28: ... which fails the Jaccard cutoff (the greedy count is not symmetric)
// per-read word `cp` (light reads): bits 0-15 passing partners, bits 16-30 partners, bit 31 a partner has > 4 fillings
#define CP_LONG 0x80000000u
__global__ void k_records(int D, const int *__restrict__ s_dp, const int *__restrict__ rmidx, const int *__restrict__ it_q,
                          const int4 *__restrict__ IT0, const int2 *__restrict__ IT1, const int4 *__restrict__ RI,
                          double overlap, int4 *SR0, int4 *SR1, int *s_m,
                          int *s_chrom, int *s_end, int *chrom_lo, int *chrom_hi, int *err) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= D) return;
    const int d = s_dp[p], m = rmidx[d], q = it_q[d];
    const int4 it = IT0[d];
    const int c = it.y, s = it.z, e = it.w;
    const int2 i1 = IT1[d];
    const int T = thr_f64(max(i1.x, 1), overlap);
    const int4 ri = RI[q];
    if ((ri.z & 0xffff) != i1.y) atomicOr(err, EF_NALN);            // n_alignments must be constant over the rows of a read
    const int fi = m - (int)((unsigned)ri.w >> 6);                   // index of this filling in its read's list
    SR0[p] = make_int4(s, e, T, (int)((unsigned)q | ((unsigned)fi << 26)));
    SR1[p] = ri;
    s_m[p] = m;
    s_chrom[p] = c; s_end[p] = e;
    const int cprev = p > 0 ? IT0[s_dp[p - 1]].y : -1;
    const int cnext = p < D - 1 ? IT0[s_dp[p + 1]].y : -1;
    if (cprev != c) chrom_lo[c] = p;
    if (cnext != c) chrom_hi[c] = p + 1;
}
// Bands of sorted position p, and the read-major record of its filling.
// ub(p): last sorted position on the chromosome with start <= end_p (IntervalMap upper bound; SURVEY §8a), by galloping
// from p (the band is short: ~2 log2(band) probes instead of log2(D)).  Tight band [lbT, ubT]: the positions whose
// interval can reciprocally overlap p by >= T_p (cluster.py:157): above p, start <= end_p - T_p (inside [p, ub]); below p,
// nothing before the first position whose prefix-max end reaches start_p + T_p.
__global__ void k_bands(int D, const int4 *__restrict__ SR0, const int *__restrict__ s_m, const int *__restrict__ s_chrom,
                        const int *__restrict__ pmaxS, const int *__restrict__ chrom_lo, const int *__restrict__ chrom_hi,
                        int4 *RM, int *rclass, unsigned long long *band_pairs, unsigned long long *tight_pairs,
                        unsigned long long *light_pairs) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    long long mine = 0, mineT = 0, mineL = 0;
    if (p < D) {
        const int4 me = SR0[p];
        const int c = s_chrom[p];
        const int e = me.y, lim = chrom_hi[c], clo = chrom_lo[c];
        int lo = p, step = 1;                                        // invariant: start[lo] <= e
        while (lo + step < lim && SR0[lo + step].x <= e) { lo += step; step <<= 1; }
        int hi = min(lo + step, lim);                                // start[hi] > e, or hi == lim
        while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (SR0[mid].x <= e) lo = mid; else hi = mid; }
        const long long et = (long long)e - (long long)me.z;        // T = 0 (overlap <= 0): the closed band
        int tl = p, th = lo + 1;                                     // start[tl] <= et or tl == p; start[th] > et or th == ub + 1
        while (th - tl > 1) { int mid = (tl + th) >> 1; if ((long long)SR0[mid].x <= et) tl = mid; else th = mid; }
        const long long st = (long long)me.x + (long long)me.z;
        int lb = p;
        if (p > clo && (long long)pmaxS[p - 1] >= st) {
            lb = p - 1;
            int stp = 1;                                             // invariant: pmaxS[lb] >= st
            while (lb - stp >= clo && (long long)pmaxS[lb - stp] >= st) { lb -= stp; stp <<= 1; }
            int l2 = max(lb - stp, clo - 1);                         // pmaxS[l2] < st, or l2 == clo - 1
            while (lb - l2 > 1) { int mid = (l2 + lb) >> 1; if ((long long)pmaxS[mid] >= st) lb = mid; else l2 = mid; }
        }
        const int m = s_m[p];
        RM[2 * m] = make_int4(c, me.x, me.y, me.z);
        RM[2 * m + 1] = make_int4(p, lo, lb, tl);
        mine = lo - p;
        mineT = tl - lb;
        if (mineT > PCAP) atomicOr(&rclass[me.w & QMASK], 1);        // hotspot: its read goes through k_pair (early exit)
        else mineL = mineT;                                          // upper bound of the hits k_hits can list for this position
    }
    __shared__ long long s_sum[3][8];                                 // one triple of global atomics per block
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        mine += __shfl_down_sync(0xffffffffu, mine, o); mineT += __shfl_down_sync(0xffffffffu, mineT, o);
        mineL += __shfl_down_sync(0xffffffffu, mineL, o);
    }
    if ((threadIdx.x & 31) == 0) { s_sum[0][threadIdx.x >> 5] = mine; s_sum[1][threadIdx.x >> 5] = mineT; s_sum[2][threadIdx.x >> 5] = mineL; }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long a = 0, b = 0, c = 0;
        for (int w = 0; w < 8; w++) { a += s_sum[0][w]; b += s_sum[1][w]; c += s_sum[2][w]; }
        if (a) atomicAdd(band_pairs, (unsigned long long)a);
        if (b) atomicAdd(tight_pairs, (unsigned long long)b);
        if (c) atomicAdd(light_pairs, (unsigned long long)c);
    }
}

// ================================================================ fast ingest (stages 1-3 when the rows of every read are
// contiguous and the read ids never decrease along the table — what collect_mapping_info.py:174 writes and what
// pandas.factorize(qname) numbers — and the caller gives no `order`).  Same results as the general kernels above with
//   * no per-read atomics: a read's first / last row are the rows whose neighbour belongs to another read (cluster.py:14-24),
//     its qlen2 (cluster.py:26-29) is folded by the thread of its first row;
//   * no sort by query rank: a read's fillings are contiguous in bed order, so after the one sort by start every filling finds
//     its read's first item in data order (= the dict order of cluster.py:189-191) among its neighbours, and ONE 64-bit scan
//     over data order of (1, L) at those first items yields both the query rank and the read-major offset.
// A table that violates the precondition raises EF_NONMONO and the general path runs instead.
#define EF_NONMONO 0x40000000
__global__ void k_rows_fast(int A, int R, const int *__restrict__ rid_, const int *__restrict__ chrom, const int *__restrict__ rstart,
                            const int *__restrict__ rend, const int *__restrict__ qstart, const int *__restrict__ qend, int n_chrom,
                            const long long *__restrict__ clen, const unsigned char *__restrict__ cmasked, int sub_on, long long subtel,
                            int *flag, int *qlen2, unsigned long long *n_fillings, int *err) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int kept = 0;
    if (i < A) {
        const int rid = rid_[i];
        const int prev = i > 0 ? rid_[i - 1] : -1, next = i + 1 < A ? rid_[i + 1] : -1;
        int f = 0;
        if ((unsigned)rid >= (unsigned)R) atomicOr(err, EF_RANGE);
        else {
            if (rid < prev) atomicOr(err, EF_NONMONO);
            const bool first = rid != prev, last = rid != next;
            if (!first && !last) {                                                  // a filling (cluster.py:14-24)
                kept = 1;
                const int c = chrom[i], rs = rstart[i], re = rend[i];
                if ((unsigned)c >= (unsigned)n_chrom || min(rs, re) < 0) atomicOr(err, EF_RANGE);
                else f = is_masked(make_int4(rid, c, min(rs, re), max(rs, re)), n_chrom, clen, cmasked, sub_on, subtel) ? 0 : 1;
            }
            if (first) {                                                            // qlen2 over the read's kept rows (cluster.py:26-29)
                int qmn = 0x7fffffff, qmx = (int)0x80000000;
                for (int j = i + 1; j + 1 < A && rid_[j + 1] == rid; j++) { qmn = min(qmn, qstart[j]); qmx = max(qmx, qend[j]); }
                long long ql = qmx >= qmn ? (long long)qmx - (long long)qmn : 0;
                if (ql > 0x7fffffffLL) { atomicOr(err, EF_RANGE); ql = 1; }
                qlen2[rid] = (int)ql;
            }
        }
        flag[i] = f;
    }
    const int cnt = __syncthreads_count(kept);
    if (threadIdx.x == 0 && cnt) atomicAdd(n_fillings, (unsigned long long)cnt);
}
// unmasked fillings in bed order, one 32-byte sector each: REC[2u] = {read_id, chrom, start, end},
// REC[2u+1] = {aln_size, n_alignments, fi, L}; sort key = start
__global__ void k_compact_fast(int A, const int *__restrict__ flag, const int *__restrict__ pos, const int *__restrict__ rid,
                               const int *__restrict__ chrom, const int *__restrict__ rstart, const int *__restrict__ rend,
                               const int *__restrict__ aln, const int *__restrict__ naln, int4 *REC, unsigned *key, int *val,
                               unsigned long long *max_start, int *err) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int s = 0;
    if (i < A && flag[i]) {
        const int u = pos[i];
        const int r = rid[i], rs = rstart[i], re = rend[i], a = aln[i], na = naln[i];
        s = min(rs, re);
        if (a <= 0 || na <= 0) atomicOr(err, EF_ZERO);
        if (na >= 65535) atomicOr(err, EF_RANGE);
        // Data order = the stable sort of the unmasked fillings by start, so two fillings of a read compare in data order like
        // (start, row): the index fi of this filling among its read's fillings in data order, and the read's filling count L,
        // are known here, before the sort, from the neighbouring rows of the table (the read's rows are contiguous).
        int fi = 0, L = 1;
        bool over = false;
        for (int j = i - 1; j >= 0 && rid[j] == r; j--) {
            if (!flag[j]) continue;
            if (++L > LMAX) { over = true; break; }
            fi += min(rstart[j], rend[j]) <= s;                                     // (start', row') < (start, row) with row' < row
            if (naln[j] != na) atomicOr(err, EF_NALN);                              // n_alignments constant over a read's rows
        }
        for (int j = i + 1; !over && j < A && rid[j] == r; j++) {
            if (!flag[j]) continue;
            if (++L > LMAX) { over = true; break; }
            fi += min(rstart[j], rend[j]) < s;
        }
        if (over) { atomicOr(err, EF_TOOMANY); L = LMAX; fi &= 63; }
        REC[2 * u] = make_int4(r, chrom[i], s, max(rs, re));
        REC[2 * u + 1] = make_int4(a, na, fi, L);
        key[u] = (unsigned)s; val[u] = u;
    }
    __shared__ int s_max;                                                           // one atomic per block, and only when it can matter
    if (threadIdx.x == 0) s_max = 0;
    __syncthreads();
    s = __reduce_max_sync(0xffffffffu, s);
    if ((threadIdx.x & 31) == 0 && s > 0) atomicMax(&s_max, s);
    __syncthreads();
    if (threadIdx.x == 0 && (unsigned long long)s_max > *(volatile unsigned long long *)max_start) atomicMax(max_start, (unsigned long long)s_max);
}
// per data position d (filling u = dfill[d]): the filling's record, gathered as one sector — the one random permutation of
// the fast ingest — and written out coalesced in data order (IT0[d] = REC[2u], IT1[d] = REC[2u+1]);
// flag64[d] = (1 << 32 | L) when the filling is its read's first item in data order (fi == 0), else 0
__global__ void k_items_fast(int D, const int *__restrict__ dfill, const int4 *__restrict__ REC, int4 *IT0, int4 *IT1, long long *flag64) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const int u = dfill[d];
    const int4 r0 = REC[2 * u], r1 = REC[2 * u + 1];                                // (one sector) r1 = {aln_size, n_alignments, fi, L}
    IT0[d] = r0;
    IT1[d] = r1;
    flag64[d] = r1.z == 0 ? ((1ll << 32) | (long long)r1.w) : 0ll;
}
// the read's first item in data order knows the read's query rank q and read-major offset `off` (the scan at its position):
// QO[read_id] = (q << 32 | off) — the only scattered write of the fast ingest, one per query read — and RI[q]
// (k_read_info; consecutive first items write consecutive q)
__global__ void k_firsts_fast(int D, const long long *__restrict__ flag64, const long long *__restrict__ qo64, const int4 *__restrict__ IT0,
                              const int4 *__restrict__ IT1, const int *__restrict__ qlen2, double qlen_c,
                              double naln_c, long long *QO, int4 *RI, int *err) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const long long fl = flag64[d];
    if (!fl) return;
    const long long qo = qo64[d];
    const int q = (int)(qo >> 32), off = (int)(qo & 0xffffffffll), L = (int)(fl & 0xffffffffll), rid = IT0[d].x;
    QO[rid] = qo;
    int ql = qlen2[rid], na = IT1[d].y;
    if (ql <= 0 || na <= 0) { atomicOr(err, EF_ZERO); ql = ql <= 0 ? 1 : ql; na = na <= 0 ? 1 : na; }
    int Ln = thr_f64(na, naln_c);
    if (Ln > 65535) Ln = 65535;
    RI[q] = make_int4(ql, thr_f64(ql, qlen_c), (na & 0xffff) | (Ln << 16), (int)(((unsigned)off << 6) | (unsigned)((L - 1) & 63)));
}
// q_of_rid from QO (filled with -1 beforehand), coalesced: a second scattered 4-byte write in k_firsts_fast costs ~10x this
__global__ void k_q_of_rid(int R, const long long *__restrict__ QO, int *q_of_rid) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < R) q_of_rid[r] = (int)(QO[r] >> 32);
}
// sorted position p of data position d: SR0[p] = {start, end, T, q | fi << 26}, SR1[p] = RI[q], s_m[p] = m = off + fi
// (the read's query rank and read-major offset come from QO: 8 bytes per read, mostly L2 hits)
struct FastRec {
    const int4 *IT0, *IT1; const long long *QO; const int4 *RI; double overlap;
    int4 *SR0, *SR1; int *s_m, *s_chrom, *s_end;
    __device__ __forceinline__ void operator()(int p, int d) const {
        const int4 r0 = __ldg(&IT0[d]), r1 = __ldg(&IT1[d]);                         // r1 = {aln_size, n_alignments, fi, L}
        const long long qo = __ldg(&QO[r0.x]);
        const int q = (int)(qo >> 32), off = (int)(qo & 0xffffffffll);
        SR0[p] = make_int4(r0.z, r0.w, thr_f64(max(r1.x, 1), overlap), (int)((unsigned)q | ((unsigned)(r1.z & 63) << 26)));
        SR1[p] = __ldg(&RI[q]);
        s_m[p] = off + r1.z;
        s_chrom[p] = r0.y; s_end[p] = r0.w;
    }
};
// IntervalMap order in one move of the records: the last pass of the stable partition of data order by chromosome
// (key = chrom, val = k_tie_delta's d | (shift + 32) << 26) writes the record of d straight to its final position, the
// partition position moved by the tie shift.  The pass hands over global partition positions, so a run of equal
// (chrom, start) that straddles tiles lands exactly where k_tie_delta's shift expects it.
struct ChromRecOut {
    FastRec rec;
    __device__ __forceinline__ void operator()(unsigned g, unsigned, int val) const {
        rec((int)g + (int)((unsigned)val >> 26) - 32, val & QMASK);
    }
};
// the same records from a list of data positions (IntervalMap order by the three full sorts)
__global__ void k_records_fast(int D, const int *__restrict__ s_dp, FastRec rec) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < D) rec(p, s_dp[p]);
}
__global__ void k_chrom_bounds(int D, const int *__restrict__ s_chrom, int *chrom_lo, int *chrom_hi) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= D) return;
    const int c = s_chrom[p];
    if (p == 0 || s_chrom[p - 1] != c) chrom_lo[c] = p;
    if (p == D - 1 || s_chrom[p + 1] != c) chrom_hi[c] = p + 1;
}
// the same bounds from the digit starts of a one-pass partition by chromosome (start[c]: first position of chromosome c)
__global__ void k_chrom_bounds_digits(int n_chrom, int D, const unsigned *__restrict__ start, int *chrom_lo, int *chrom_hi) {
    const int c = threadIdx.x;
    if (c >= n_chrom) return;
    const unsigned e = c + 1 < 256 ? start[c + 1] : (unsigned)D;
    if (e > start[c]) { chrom_lo[c] = (int)start[c]; chrom_hi[c] = (int)e; }
}

