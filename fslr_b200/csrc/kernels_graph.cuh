// Part of fslr_b200.cu (one translation unit; included after the error flags, LMAX and fslr_b200.h are defined).
// Stages 9-10 and the rows around the path: union-find, cluster numbering, choose_alignment, integer-issue microbenchmark.
#pragma once

// ---------------------------------------------------------------- stage 9: union-find (root = smallest query rank)
__device__ __forceinline__ int uf_find(int *parent, int x) {
    for (;;) {
        int p = *(volatile int *)&parent[x];
        if (p == x) return x;
        int gp = *(volatile int *)&parent[p];
        if (gp != p) atomicMin(&parent[x], gp);                                      // path halving, keeps parent <= index
        x = p;
    }
}
__device__ __forceinline__ void uf_union(int *parent, int a, int b) {
    if (*(volatile int *)&parent[a] == *(volatile int *)&parent[b]) return;         // (both loads in flight at once) same tree already:
    for (;;) {                                                                      //  most pairs of a PCR family after its first unions
        a = uf_find(parent, a); b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { int tmp = a; a = b; b = tmp; }                                  // hook the larger root under the smaller
        if (atomicCAS(&parent[a], a, b) == a) return;
    }
}
// entries (a, b) recorded by k_eval / k_pair (a -> b evaluated; only the passing ones matter here): a not saturating;
// b > a -> a tested it (edge); b < a -> edge only if b is saturating and its scan stopped before reaching a (then a's
// query tested the pair, direction a -> b).  The rules live in the three functions below, which k_union_entries and the
// edge export (k_edges_of_entries) share.
// the directed pairs a slot stands for that pass the Jaccard cutoff: (a, b), and in symmetric mode (b, a)
__device__ __forceinline__ bool slot_fwd(const int2 ab) { return ab.x >= 0 && !((unsigned)ab.y & EB_NOPASS); }
__device__ __forceinline__ bool slot_rev(const int2 ab) {
    return ab.x >= 0 && ((unsigned)ab.y & EB_SYM) && !((unsigned)ab.y & EB_NOPASS2);
}
// a -> b passes and a is not saturating: is it an edge of the reference's graph, i.e. did a's query test the pair?
__device__ __forceinline__ bool directed_is_edge(const Tab &t, const int *isP, const int *stop, int a, int b) {
    if (b > a) return true;
    if (!isP[b]) return false;
    const int wa = t.RI[a].w, wb = t.RI[b].w;
    const int offa = (int)((unsigned)wa >> 6), La = (wa & 63) + 1, offb = (int)((unsigned)wb >> 6), Lb = (wb & 63) + 1;
    for (int f = 0; f < Lb; f++) {                                                  // some scan of b got down to a: b's query saw it
        const int4 bf = rm0(t, offb + f);
        const int ubf = rm1(t, offb + f).y, sf = stop[offb + f];
        for (int g = 0; g < La; g++) {
            const int4 ag = rm0(t, offa + g);
            const int pg = rm1(t, offa + g).x;
            if (ag.x == bf.x && sf <= pg && pg <= ubf && ag.z >= bf.y) return false;
        }
    }
    return true;
}
#define UE_PER 4
#define UE_THREADS 256
// Only about a third of the list's slots are edges (the rest: padding, pairs of saturating reads, pairs that do not pass), and
// union-find is pointer chasing: what counts is how many chases are in flight.  Every block filters its 1024 slots (entry and
// isP loads batched), compacts the survivors in shared memory and walks them with all lanes busy.
__global__ void __launch_bounds__(UE_THREADS) k_union_entries(unsigned long long n, const int2 *__restrict__ entries, const int *__restrict__ isP,
                                                              Tab t, const int *stop, int *parent, int *ing, unsigned long long *n_edges) {
    __shared__ int2 sE[UE_THREADS * UE_PER * 2];                                    // (a symmetric slot stands for two directed pairs)
    __shared__ int s_warp[UE_THREADS / 32];
    __shared__ int s_ne;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long k0 = (unsigned long long)blockIdx.x * (UE_THREADS * UE_PER) + tid;
    if (tid == 0) s_ne = 0;
    int2 ab[UE_PER];
    int pa[UE_PER], pb[UE_PER];
#pragma unroll
    for (int u = 0; u < UE_PER; u++) {                                              // all entries, then all flags: loads in flight together
        const unsigned long long k = k0 + (unsigned long long)u * UE_THREADS;
        ab[u] = k < n ? __ldg(&entries[k]) : make_int2(-1, -1);
    }
#pragma unroll
    for (int u = 0; u < UE_PER; u++) {                                              // 1: nothing to do for that direction
        const unsigned y = (unsigned)ab[u].y;
        pa[u] = slot_fwd(ab[u]) ? __ldg(&isP[ab[u].x]) : 1;
        pb[u] = slot_rev(ab[u]) ? __ldg(&isP[y & QMASK]) : 1;
    }
    int mine = 0;
#pragma unroll
    for (int u = 0; u < UE_PER; u++) mine += !pa[u] + !pb[u];
    int incl = mine;                                                                // block-wide exclusive scan of the survivor counts
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < UE_THREADS / 32; w++) { const int c = s_warp[w]; if (w < warp) wbase += c; total += c; }
    int at = wbase + incl - mine;
#pragma unroll
    for (int u = 0; u < UE_PER; u++) {                                              // y: b | EB_NOPASS | EB_HEAVY | EB_SYM | EB_NOPASS2
        if (!pa[u]) sE[at++] = make_int2(ab[u].x, ab[u].y & QMASK);
        if (!pb[u]) sE[at++] = make_int2(ab[u].y & QMASK, ab[u].x);
    }
    __syncthreads();
    int ne = 0;
    for (int idx = tid; idx < total; idx += UE_THREADS) {
        const int a = sE[idx].x, b = sE[idx].y;
        if (directed_is_edge(t, isP, stop, a, b)) { ing[a] = 1; ing[b] = 1; uf_union(parent, a, b); ne++; }
    }
    for (int o = 16; o; o >>= 1) ne += __shfl_down_sync(0xffffffffu, ne, o);
    if (lane == 0 && ne) atomicAdd(&s_ne, ne);
    __syncthreads();
    if (tid == 0 && s_ne) atomicAdd(n_edges, (unsigned long long)s_ne);             // one counter update per block
}
__global__ void k_union_edges(unsigned long long n, const int2 *__restrict__ edges, int *parent, int *ing, unsigned long long *n_edges) {
    unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    bool e = false;
    if (k < n) {
        const int2 ab = edges[k];
        if (ab.x >= 0) {                                                            // skip chunk padding
            e = true;
            ing[ab.x] = 1; ing[ab.y] = 1;
            uf_union(parent, ab.x, ab.y);
        }
    }
    const int cnt = __syncthreads_count(e);
    if (threadIdx.x == 0 && cnt && n_edges) atomicAdd(n_edges, (unsigned long long)cnt);
}
// ---------------------------------------------------------------- edge export (fslrc_set_edge_capture)
// Every edge union-find was handed, as the directed pair (query read, other read): the first read is the one whose query
// tested the pair (cluster.py:197-220's query_key).  Appended in any order; k_edges_final puts them in a fixed one.
__device__ __forceinline__ unsigned long long warp_reserve(int c, unsigned long long *n_out) {   // warp-aggregated append
    const int lane = threadIdx.x & 31;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    unsigned long long base = 0;
    if (lane == 31 && incl) base = atomicAdd(n_out, (unsigned long long)incl);
    return __shfl_sync(0xffffffffu, base, 31) + (unsigned long long)(incl - c);
}
__global__ void k_edges_of_entries(unsigned long long n, const int2 *__restrict__ entries, const int *__restrict__ isP, Tab t,
                                   const int *stop, int2 *out, unsigned long long cap, unsigned long long *n_out) {
    const unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    const int2 ab = k < n ? entries[k] : make_int2(-1, -1);
    const int a = ab.x, b = ab.y & QMASK;
    const bool e1 = slot_fwd(ab) && !isP[a] && directed_is_edge(t, isP, stop, a, b);
    const bool e2 = slot_rev(ab) && !isP[b] && directed_is_edge(t, isP, stop, b, a);
    unsigned long long at = warp_reserve((int)e1 + (int)e2, n_out);
    if (e1) { if (at < cap) out[at] = make_int2(a, b); at++; }
    if (e2 && at < cap) out[at] = make_int2(b, a);
}
__global__ void k_edges_of_pedges(unsigned long long n, const int2 *__restrict__ pedges, int2 *out, unsigned long long cap,
                                  unsigned long long *n_out) {
    const unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    const int2 ab = k < n ? pedges[k] : make_int2(-1, -1);
    const bool e = ab.x >= 0;                                                       // skip chunk padding
    const unsigned long long at = warp_reserve((int)e, n_out);
    if (e && at < cap) out[at] = ab;
}
// radix keys of the two stable passes: first by the second read's query rank, then (gathered) by the first read's
__global__ void k_edges_key2(int n, const int2 *__restrict__ dir, unsigned *key, int *iota) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    key[i] = (unsigned)dir[i].y; iota[i] = i;
}
__global__ void k_edges_key1(int n, const int2 *__restrict__ dir, const int *__restrict__ perm, unsigned *key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    key[i] = (unsigned)dir[perm[i]].x;
}
__global__ void k_rid_of_q(int R, const int *__restrict__ q_of_rid, int *rid_of_q) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const int q = q_of_rid[r];
    if (q >= 0) rid_of_q[q] = r;
}
// cluster.py:140-170 in the edge's direction: list1 = the query read's fillings in data order, list2 = the other's; each
// filling of list1 takes the first free matching filling of list2 (k_eval's predicate, ALLMATCH for --overlap <= 0)
template <bool ALLMATCH>
__device__ int greedy_count(const Tab &t, int q1, int q2, int *L1, int *L2) {
    const int w1 = __ldg(&t.RI[q1]).w, w2 = __ldg(&t.RI[q2]).w;
    const int off1 = (int)((unsigned)w1 >> 6), La = (w1 & 63) + 1, off2 = (int)((unsigned)w2 >> 6), Lb = (w2 & 63) + 1;
    unsigned long long used = 0;
    int n = 0;
    for (int fa = 0; fa < La; fa++) {
        const int4 a = rm0(t, off1 + fa);
        for (int fb = 0; fb < Lb; fb++)
            if (!((used >> fb) & 1ull) && matchT<ALLMATCH>(a, rm0(t, off2 + fb))) { used |= 1ull << fb; n++; break; }
    }
    *L1 = La; *L2 = Lb;
    return n;
}
// the sorted list: read ids and the Jaccard similarity n / (L1 + L2 - n), the IEEE division CPython does
template <bool ALLMATCH>
__global__ void k_edges_final(int n, Tab t, const int2 *__restrict__ dir, const int *__restrict__ perm, const int *__restrict__ rid_of_q,
                              int *read1, int *read2, double *jac) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int2 e = dir[perm[i]];
    int L1, L2;
    const int c = greedy_count<ALLMATCH>(t, e.x, e.y, &L1, &L2);
    read1[i] = rid_of_q[e.x]; read2[i] = rid_of_q[e.y];
    jac[i] = __ddiv_rn((double)c, (double)(L1 + L2 - c));
}
__global__ void k_flatten(int Q, int *parent, const int *__restrict__ ing, int *isroot, int *csize) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    int r = uf_find(parent, q);
    parent[q] = r;                                                                  // safe: r is a root and stays one
    isroot[q] = (ing[q] && r == q);
    if (ing[q]) atomicAdd(&csize[r], 1);
}
// spanning forest of the local components (multi-GPU exchange, SURVEY §8e)
__global__ void k_forest(int Q, const int *__restrict__ parent, const int *__restrict__ ing, int2 *forest, unsigned long long *n) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    bool e = q < Q && ing[q] && parent[q] != q;
    const unsigned m = __ballot_sync(0xffffffffu, e);
    unsigned long long at = 0;
    if ((threadIdx.x & 31) == 0 && m) at = atomicAdd(n, (unsigned long long)__popc(m));
    at = __shfl_sync(0xffffffffu, at, 0);
    if (e) forest[at + __popc(m & ((1u << (threadIdx.x & 31)) - 1u))] = make_int2(q, parent[q]);
}

// ---------------------------------------------------------------- stage 10: cluster / n_reads (main.py:251-257,334-342)
__global__ void k_single_flags(int R, const int *__restrict__ q_of_rid, const int *__restrict__ ing, int *flag) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    int q = q_of_rid[r];
    flag[r] = !(q >= 0 && ing[q]);
}
__global__ void k_number(int R, const int *__restrict__ q_of_rid, const int *__restrict__ ing, const int *__restrict__ root,
                         const int *__restrict__ cidx, const int *__restrict__ csize, const int *__restrict__ spos,
                         const int64_t *__restrict__ ncl, int *out_cluster, int *out_n) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    int q = q_of_rid[r];
    if (q >= 0 && ing[q]) { int rt = root[q]; out_cluster[r] = cidx[rt]; out_n[r] = csize[rt]; }
    else { out_cluster[r] = (int)(*ncl) + spos[r]; out_n[r] = 1; }                   // singletons after the clusters, bed order
}

// ---------------------------------------------------------------- choose_alignment (cluster.py:237-254, main.py:351-352)
// per read: sum and count of alignment_score over its rows, first row; per cluster: the read with the highest mean
// (IEEE double division, as pandas' groupby.mean of an integer column), first row in table order on ties (idxmax)
__device__ __forceinline__ unsigned long long order_f64(double x) {   // monotone map double -> uint64
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__global__ void k_ca_rows(int A, int R, const int *__restrict__ rid, const int *__restrict__ score, long long *sum, int *cnt, int *first, int *err) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A) return;
    const int r = rid[i];
    if ((unsigned)r >= (unsigned)R) { atomicOr(err, EF_RANGE); return; }
    atomicAdd((unsigned long long *)&sum[r], (unsigned long long)(long long)score[i]);
    atomicAdd(&cnt[r], 1);
    atomicMin(&first[r], i);
}
__global__ void k_ca_best(int R, int C, const long long *__restrict__ sum, const int *__restrict__ cnt, const int *__restrict__ cluster,
                          unsigned long long *best, int *err) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R || cnt[r] == 0) return;
    const int c = cluster[r];
    if ((unsigned)c >= (unsigned)C) { atomicOr(err, EF_RANGE); return; }
    atomicMax(&best[c], order_f64(__ddiv_rn((double)sum[r], (double)cnt[r])));
}
__global__ void k_ca_first(int R, int C, const long long *__restrict__ sum, const int *__restrict__ cnt, const int *__restrict__ first,
                           const int *__restrict__ cluster, const unsigned long long *__restrict__ best, int *minrow) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R || cnt[r] == 0) return;
    const int c = cluster[r];
    if ((unsigned)c >= (unsigned)C) return;
    if (order_f64(__ddiv_rn((double)sum[r], (double)cnt[r])) == best[c]) atomicMin(&minrow[c], first[r]);
}
__global__ void k_ca_flag(int R, int C, const int *__restrict__ cnt, const int *__restrict__ first, const int *__restrict__ cluster,
                          const int *__restrict__ minrow, unsigned char *is_rep, int *rep_read) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    unsigned char f = 0;
    if (cnt[r] > 0) {
        const int c = cluster[r];
        if ((unsigned)c < (unsigned)C && minrow[c] == first[r]) { f = 1; if (rep_read) rep_read[c] = r; }
    }
    is_rep[r] = f;
}

// ---------------------------------------------------------------- integer-issue microbenchmark (roofline denominator)
__global__ void k_int_peak(int iters, int *out) {
    int a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 5, a5 = a0 + 7, a6 = a0 + 11, a7 = a0 + 13;
    const int k = blockIdx.x | 1;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 16; j++) {                                               // 8 independent chains x 2 ops: min/max + add/xor
            a0 = max(a0 + k, a1) ^ j; a1 = min(a1 - k, a2) ^ j; a2 = max(a2 + k, a3) ^ j; a3 = min(a3 - k, a4) ^ j;
            a4 = max(a4 + k, a5) ^ j; a5 = min(a5 - k, a6) ^ j; a6 = max(a6 + k, a7) ^ j; a7 = min(a7 - k, a0) ^ j;
        }
    }
    if ((a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7) == 0x12345678) out[0] = a0;
}
