// Device-wide primitives of the ingest stages, hand-written for sm_100a: single-pass scans and a one-sweep LSD radix
// sort, both with decoupled look-back (one read + one write of the data per pass; tiles are handed out by an atomic
// ticket so that a tile only ever waits for tiles that are already running).
//
//   scan_excl_i32     exclusive prefix sum of int32 (flags / counts), optional grand total
//   scan_incl_max_u64 inclusive prefix max of uint64 (segmented max as (segment << 32 | value))
//   radix_sort_pairs  stable LSD sort of (uint32 key, int32 value) pairs on bits [b0, b1), 8 bits per pass
//
// Status words carry value and validity in ONE 64-bit (scan) / 32-bit (sort) word, so no fence is needed between a
// tile's partial result and its flag.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace prims {

constexpr int SC_THREADS = 256;
constexpr int SC_ITEMS = 16;
constexpr int SC_TILE = SC_THREADS * SC_ITEMS;
constexpr unsigned long long ST_AGG = 1ull << 62, ST_INC = 2ull << 62, ST_MASK = (1ull << 62) - 1ull;

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u32(unsigned *p, unsigned v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

struct OpAdd { __device__ __forceinline__ unsigned long long operator()(unsigned long long a, unsigned long long b) const { return a + b; } };
struct OpMax { __device__ __forceinline__ unsigned long long operator()(unsigned long long a, unsigned long long b) const { return a > b ? a : b; } };

// Look-back of warp 0: combines the aggregates of the preceding tiles, 32 at a time, down to the nearest tile whose
// inclusive prefix is known.  Values are < 2^62.
template <typename Op>
__device__ __forceinline__ unsigned long long lookback(const unsigned long long *status, int tile, int lane, Op op, unsigned long long identity) {
    unsigned long long excl = identity;
    int p = tile - 1;
    for (;;) {
        const int idx = p - lane;
        unsigned long long w;
        do {                                                          // every predecessor holds a smaller ticket: it is running
            w = idx >= 0 ? ld_relaxed_u64(&status[idx]) : (ST_INC | identity);
        } while (__any_sync(0xffffffffu, (w >> 62) == 0));
        const unsigned inc = __ballot_sync(0xffffffffu, (w >> 62) == 2);
        const int first = inc ? __ffs(inc) - 1 : 31;                  // nearest predecessor with an inclusive prefix
        unsigned long long v = lane <= first ? (w & ST_MASK) : identity;
#pragma unroll
        for (int o = 16; o; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
        excl = op(excl, v);
        if (inc) break;
        p -= 32;
    }
    return excl;
}

// ---------------------------------------------------------------- exclusive sum (int32, or int64 for byte offsets)
template <typename T>
__global__ void __launch_bounds__(SC_THREADS) k_scan_excl(const T *__restrict__ in, T *__restrict__ out, int n,
                                                          unsigned long long *status, unsigned *ticket, long long *total) {
    __shared__ unsigned s_tile;
    __shared__ long long s_warp[SC_THREADS / 32];
    __shared__ long long s_excl;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile;
    const int base = tile * SC_TILE + tid * SC_ITEMS;
    T v[SC_ITEMS];
    if (sizeof(T) == 4 && base + SC_ITEMS <= n && (((uintptr_t)(in + base)) & 15) == 0) {
#pragma unroll
        for (int k = 0; k < SC_ITEMS / 4; k++) {
            const int4 q = __ldg((const int4 *)(in + base) + k);
            v[4 * k] = (T)q.x; v[4 * k + 1] = (T)q.y; v[4 * k + 2] = (T)q.z; v[4 * k + 3] = (T)q.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++) v[k] = base + k < n ? in[base + k] : (T)0;
    }
    long long tsum = 0;
#pragma unroll
    for (int k = 0; k < SC_ITEMS; k++) tsum += v[k];
    long long incl = tsum;                                            // inclusive scan of the thread sums inside the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    long long wbase = 0, tile_sum = 0;
#pragma unroll
    for (int w = 0; w < SC_THREADS / 32; w++) { const long long x = s_warp[w]; if (w < warp) wbase += x; tile_sum += x; }
    if (warp == 0) {
        if (lane == 0) st_relaxed_u64(&status[tile], (tile == 0 ? ST_INC : ST_AGG) | ((unsigned long long)tile_sum & ST_MASK));
        unsigned long long excl = 0;
        if (tile > 0) {
            excl = lookback(status, tile, lane, OpAdd(), 0ull);
            if (lane == 0) st_relaxed_u64(&status[tile], ST_INC | ((excl + (unsigned long long)tile_sum) & ST_MASK));
        }
        if (lane == 0) {
            s_excl = (long long)excl;
            if (total && (long long)(tile + 1) * SC_TILE >= n) *total = (long long)excl + tile_sum;
        }
    }
    __syncthreads();
    long long run = s_excl + wbase + incl - tsum;
    if (sizeof(T) == 4 && base + SC_ITEMS <= n && (((uintptr_t)(out + base)) & 15) == 0) {
#pragma unroll
        for (int k = 0; k < SC_ITEMS / 4; k++) {
            int4 q;
            q.x = (int)run; run += v[4 * k]; q.y = (int)run; run += v[4 * k + 1]; q.z = (int)run; run += v[4 * k + 2]; q.w = (int)run; run += v[4 * k + 3];
            *((int4 *)(out + base) + k) = q;
        }
    } else {
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++) { if (base + k < n) out[base + k] = (T)run; run += v[k]; }
    }
}

// ---------------------------------------------------------------- inclusive max of (seg << 32 | value): per-segment prefix max
// seg[] must be non-decreasing along the array (sorted by chromosome); out[i] = max of val over the items of seg[i] up to i
__global__ void __launch_bounds__(SC_THREADS) k_scan_segmax(const int *__restrict__ seg, const int *__restrict__ val, int *__restrict__ out,
                                                            int n, unsigned long long *status, unsigned *ticket) {
    __shared__ unsigned s_tile;
    __shared__ unsigned long long s_warp[SC_THREADS / 32];
    __shared__ unsigned long long s_excl;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile;
    const int base = tile * SC_TILE + tid * SC_ITEMS;
    unsigned long long v[SC_ITEMS];
    unsigned long long tmax = 0;
    if (base + SC_ITEMS <= n && ((((uintptr_t)(seg + base)) | ((uintptr_t)(val + base))) & 15) == 0) {
#pragma unroll
        for (int k = 0; k < SC_ITEMS / 4; k++) {
            const int4 sg = __ldg((const int4 *)(seg + base) + k), vl = __ldg((const int4 *)(val + base) + k);
            v[4 * k] = ((unsigned long long)(unsigned)sg.x << 32) | (unsigned)vl.x;
            v[4 * k + 1] = ((unsigned long long)(unsigned)sg.y << 32) | (unsigned)vl.y;
            v[4 * k + 2] = ((unsigned long long)(unsigned)sg.z << 32) | (unsigned)vl.z;
            v[4 * k + 3] = ((unsigned long long)(unsigned)sg.w << 32) | (unsigned)vl.w;
        }
    } else {
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++)
            v[k] = base + k < n ? (((unsigned long long)(unsigned)seg[base + k] << 32) | (unsigned)val[base + k]) : 0ull;
    }
#pragma unroll
    for (int k = 0; k < SC_ITEMS; k++) tmax = v[k] > tmax ? v[k] : tmax;
    unsigned long long incl = tmax;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned long long y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o && y > incl) incl = y; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned long long wbase = 0, tile_max = 0;
#pragma unroll
    for (int w = 0; w < SC_THREADS / 32; w++) { const unsigned long long x = s_warp[w]; if (w < warp && x > wbase) wbase = x; if (x > tile_max) tile_max = x; }
    if (warp == 0) {
        if (lane == 0) st_relaxed_u64(&status[tile], (tile == 0 ? ST_INC : ST_AGG) | tile_max);
        unsigned long long excl = 0;
        if (tile > 0) {
            excl = lookback(status, tile, lane, OpMax(), 0ull);
            if (lane == 0) st_relaxed_u64(&status[tile], ST_INC | (excl > tile_max ? excl : tile_max));
        }
        if (lane == 0) s_excl = excl;
    }
    __syncthreads();
    unsigned long long run = s_excl > wbase ? s_excl : wbase;         // max over everything before this thread's items
    const unsigned long long prev = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane > 0 && prev > run) run = prev;
    if (base + SC_ITEMS <= n && (((uintptr_t)(out + base)) & 15) == 0) {
#pragma unroll
        for (int k = 0; k < SC_ITEMS / 4; k++) {
            int4 q;                                                    // low word = max inside the item's own segment
            if (v[4 * k] > run) run = v[4 * k];         q.x = (int)(unsigned)run;
            if (v[4 * k + 1] > run) run = v[4 * k + 1]; q.y = (int)(unsigned)run;
            if (v[4 * k + 2] > run) run = v[4 * k + 2]; q.z = (int)(unsigned)run;
            if (v[4 * k + 3] > run) run = v[4 * k + 3]; q.w = (int)(unsigned)run;
            *((int4 *)(out + base) + k) = q;
        }
    } else {
#pragma unroll
        for (int k = 0; k < SC_ITEMS; k++) {
            if (v[k] > run) run = v[k];
            if (base + k < n) out[base + k] = (int)(unsigned)(run & 0xffffffffull);
        }
    }
}

// ---------------------------------------------------------------- one-sweep LSD radix sort of (u32 key, i32 value) pairs
#ifndef RS_THREADS_
#define RS_THREADS_ 512
#endif
#ifndef RS_ITEMS_
#define RS_ITEMS_ 12
#endif
#ifndef RS_MINB
#define RS_MINB 2
#endif
constexpr int RS_THREADS = RS_THREADS_;     // (>= 256: thread t < 256 owns digit t)
constexpr int RS_ITEMS = RS_ITEMS_;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;       // 8192 pairs per tile
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr unsigned RS_AGG = 1u << 30, RS_INC = 2u << 30, RS_MASK = (1u << 30) - 1u;

// histograms of all passes in one read of the keys: hist[pass][256]
__global__ void __launch_bounds__(256) k_rs_hist(const unsigned *__restrict__ keys, int n, int b0, int b1, int npass, unsigned *hist) {
    __shared__ unsigned sh[4][256];
    for (int k = threadIdx.x; k < 4 * 256; k += 256) (&sh[0][0])[k] = 0;
    __syncthreads();
    for (long long i = blockIdx.x * 256ll + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        const unsigned key = __ldg(&keys[i]);
#pragma unroll
        for (int p = 0; p < 4; p++)
            if (p < npass) atomicAdd(&sh[p][(key >> (b0 + 8 * p)) & ((1u << min(8, b1 - b0 - 8 * p)) - 1u)], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < npass * 256; k += 256) { const unsigned c = (&sh[0][0])[k]; if (c) atomicAdd(&hist[k], c); }
}
// exclusive scan of each pass's 256 counters (in place): global start of every digit's bucket
__global__ void __launch_bounds__(256) k_rs_scan(unsigned *hist) {
    __shared__ unsigned s[256];
    unsigned *h = hist + blockIdx.x * 256;
    const unsigned c = h[threadIdx.x];
    s[threadIdx.x] = c;
    __syncthreads();
    unsigned sum = 0;
    for (int k = 0; k < (int)threadIdx.x; k++) sum += s[k];
    h[threadIdx.x] = sum;
}
// one pass: every tile ranks its pairs by digit (stable), publishes its digit counts, looks back for the counts of the
// preceding tiles and scatters through shared memory (so that the global writes of a bucket are contiguous: 8192 pairs
// per tile = runs of ~32 pairs = whole 128-byte lines per digit)
struct RsSmem {
    unsigned cnt[RS_WARPS][256];      // per-warp digit counts, then per-warp exclusive bases inside the tile
    unsigned dbase[256];              // start of each digit inside the tile
    unsigned gofs[256];               // global address of the digit's first pair of this tile, minus dbase
    unsigned wt[8];
    unsigned tile;
    unsigned keys[RS_TILE];
    int vals[RS_TILE];
};
// where a pass puts pair (key, val) of output position g: the next pass's key / value arrays, or (last pass) a caller's sink
struct PairOut {
    unsigned *kout; int *vout;
    __device__ __forceinline__ void operator()(unsigned g, unsigned key, int val) const { kout[g] = key; vout[g] = val; }
};
template <typename Out>
__global__ void __launch_bounds__(RS_THREADS, RS_MINB) k_rs_onesweep(const unsigned *__restrict__ kin, const int *__restrict__ vin, Out out,
                                                            int n, int shift, int mask, const unsigned *__restrict__ gbase,
                                                            unsigned *status, unsigned *ticket) {
    extern __shared__ __align__(16) unsigned char rs_raw[];
    RsSmem &sm = *reinterpret_cast<RsSmem *>(rs_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) sm.tile = atomicAdd(ticket, 1u);
    for (int k = tid; k < RS_WARPS * 256; k += RS_THREADS) (&sm.cnt[0][0])[k] = 0;
    __syncthreads();
    const int tile = (int)sm.tile;
    const long long tbase = (long long)tile * RS_TILE;
    // ---- load (warp-striped: item i of lane l of warp w is pair tbase + w*32*ITEMS + i*32 + l) and rank inside the warp
    unsigned key[RS_ITEMS];
    int val[RS_ITEMS];
    unsigned short rk[RS_ITEMS];
    const unsigned ltmask = (1u << lane) - 1u;
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const long long idx = tbase + warp * (32 * RS_ITEMS) + i * 32 + lane;
        key[i] = idx < n ? __ldg(&kin[idx]) : 0xffffffffu;            // padding sorts last inside the last tile and is never written
        val[i] = idx < n ? __ldg(&vin[idx]) : 0;
    }
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const unsigned d = (key[i] >> shift) & (unsigned)mask;
        unsigned m = 0xffffffffu;                                      // lanes holding the same digit: 8 ballots (MATCH.ANY is far slower)
#pragma unroll
        for (int b = 0; b < 8; b++) {
            const unsigned vote = __ballot_sync(0xffffffffu, (d >> b) & 1u);
            m &= ((d >> b) & 1u) ? vote : ~vote;
        }
        const unsigned old = sm.cnt[warp][d];
        __syncwarp();
        rk[i] = (unsigned short)(old + __popc(m & ltmask));
        if ((m & ltmask) == 0) sm.cnt[warp][d] = old + __popc(m);     // the lowest lane of the digit group
        __syncwarp();
    }
    __syncthreads();
    // ---- tile digit counts; thread t < 256 owns digit t
    unsigned cnt = 0, pub = 0, excl = 0;
    unsigned *st = status + (size_t)tile * 256;
    if (tid < 256) {
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) { const unsigned c = sm.cnt[w][tid]; sm.cnt[w][tid] = cnt; cnt += c; }
        // padding of the last tile was counted in digit `mask` (all ones): take it out of the published count
        pub = cnt;
        if (tid == mask && tbase + RS_TILE > n) pub -= (unsigned)(tbase + RS_TILE - n);
        st_relaxed_u32(&st[tid], (tile == 0 ? RS_INC : RS_AGG) | pub);
        unsigned incl = cnt;                                            // exclusive scan of the digit counts inside the tile
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
        if (lane == 31) sm.wt[warp] = incl;
        sm.dbase[tid] = incl - cnt;
    }
    __syncthreads();
    if (tid < 256) {
        unsigned wb = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) if (w < warp) wb += sm.wt[w];
        sm.dbase[tid] += wb;
        // ---- look-back: pairs with digit `tid` in the preceding tiles
        if (tile > 0) {
            int p = tile - 1;
            for (;;) {
                const unsigned w = ld_relaxed_u32(&status[(size_t)p * 256 + tid]);
                if (w & RS_INC) { excl += w & RS_MASK; break; }
                if (w & RS_AGG) { excl += w & RS_MASK; if (--p < 0) break; }
            }
            st_relaxed_u32(&st[tid], RS_INC | (excl + pub));
        }
        sm.gofs[tid] = __ldg(&gbase[tid]) + excl - sm.dbase[tid];
    }
    __syncthreads();
    // ---- scatter into shared memory in sorted order, then contiguous global writes
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const unsigned d = (key[i] >> shift) & (unsigned)mask;
        const unsigned pos = sm.dbase[d] + sm.cnt[warp][d] + rk[i];
        sm.keys[pos] = key[i];
        sm.vals[pos] = val[i];
    }
    __syncthreads();
    const int valid = (int)((tbase + RS_TILE <= n) ? RS_TILE : (n - tbase));
#pragma unroll
    for (int i = 0; i < RS_ITEMS; i++) {
        const int pos = i * RS_THREADS + tid;
        if (pos < valid) {
            const unsigned k = sm.keys[pos];
            const unsigned d = (k >> shift) & (unsigned)mask;
            out(sm.gofs[d] + (unsigned)pos, k, sm.vals[pos]);
        }
    }
}

}  // namespace prims
