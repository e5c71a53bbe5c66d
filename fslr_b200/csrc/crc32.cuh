// CRC-32 of gzip (RFC 1952: reflected polynomial 0xEDB88320, initial value and final xor 0xFFFFFFFF), used to check every
// BGZF block's inflated bytes against the CRC32 field of its trailer, as htslib does when it reads a BAM file.
//
// The update is table driven, eight bytes per step (slice-by-8).  The CRC register is affine in the data, so a block can
// be split into segments whose remainders are computed independently and combined: a segment's remainder followed by
// n more bytes is the remainder times x^(8n) modulo the polynomial (`multmodp` / `x2nmodp`, as zlib's crc32_combine
// defines them).  k_bgzf_crc gives each lane of a warp one segment of a block.
//
// Plain functions compiled for host and device (FSLR_HD), like inflate.cuh: the host build is what
// tests/test_crc32_host.py checks against zlib, including the kernel's per-lane layout.  The tables are constant
// expressions, computed once by the compiler.
#pragma once
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define FSLR_HD __host__ __device__ __forceinline__
#else
#define FSLR_HD inline
#endif

namespace crc32 {

constexpr uint32_t POLY = 0xEDB88320u;
constexpr int LANES = 32;
constexpr int SEG = 2048;                        // bytes per lane: 32 x 2048 = 65536, the largest BGZF block

// a * b modulo the CRC polynomial, in the reflected bit order (bit 31 = x^0)
FSLR_HD constexpr uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (uint32_t m = 1u << 31; m; m >>= 1) {
        if (a & m) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ POLY : b >> 1;
    }
    return p;
}
// x^(n * 2^k) modulo the polynomial; x2nmodp(n, 3) shifts a remainder by n zero bytes
FSLR_HD constexpr uint32_t x2nmodp(long long n, unsigned k) {
    uint32_t sq = 1u << 30;                      // x^(2^0)
    for (unsigned i = 0; i < k; i++) sq = multmodp(sq, sq);
    uint32_t p = 1u << 31;                       // x^0
    for (; n; n >>= 1) {
        if (n & 1) p = multmodp(sq, p);
        sq = multmodp(sq, sq);
    }
    return p;
}

struct Tables {
    uint32_t t[8][256];                          // t[0]: one byte; t[j][b]: byte b followed by j zero bytes
    uint32_t shift[LANES];                       // shift[j] = x^(8 * j * SEG): lane l's remainder is followed by (31 - l) segments
};
FSLR_HD constexpr Tables make_tables() {
    Tables T{};
    for (uint32_t b = 0; b < 256; b++) {
        uint32_t c = b;
        for (int i = 0; i < 8; i++) c = (c & 1u) ? (c >> 1) ^ POLY : c >> 1;
        T.t[0][b] = c;
    }
    for (int j = 1; j < 8; j++)
        for (int b = 0; b < 256; b++) T.t[j][b] = (T.t[j - 1][b] >> 8) ^ T.t[0][T.t[j - 1][b] & 0xffu];
    for (int j = 0; j < LANES; j++) T.shift[j] = x2nmodp((long long)j * SEG, 3);
    return T;
}

typedef uint32_t Tab[256];
FSLR_HD uint32_t bytes(uint32_t c, const unsigned char *p, long long n, const Tab *t) {
    for (long long i = 0; i < n; i++) c = t[0][(c ^ p[i]) & 0xffu] ^ (c >> 8);
    return c;
}
FSLR_HD uint32_t step8(uint32_t c, uint32_t lo, uint32_t hi, const Tab *t) {   // eight bytes, little-endian words
    lo ^= c;
    return t[7][lo & 0xffu] ^ t[6][(lo >> 8) & 0xffu] ^ t[5][(lo >> 16) & 0xffu] ^ t[4][lo >> 24] ^
           t[3][hi & 0xffu] ^ t[2][(hi >> 8) & 0xffu] ^ t[1][(hi >> 16) & 0xffu] ^ t[0][hi >> 24];
}
// raw register update (no initial value, no final xor) over p[0, n); p has any alignment: bytes one at a time up to a
// 16-byte boundary, then 16-byte loads
FSLR_HD uint32_t update(uint32_t c, const unsigned char *p, long long n, const Tab *t) {
    const long long head = (long long)((16u - ((unsigned)(uintptr_t)p & 15u)) & 15u);
    const long long h = head < n ? head : n;
    c = bytes(c, p, h, t);
    p += h; n -= h;
#pragma unroll 4
    for (; n >= 16; p += 16, n -= 16) {
#ifdef __CUDA_ARCH__
        const uint4 v = __ldg((const uint4 *)p);
        c = step8(c, v.x, v.y, t);
        c = step8(c, v.z, v.w, t);
#else
        uint32_t v[4];
        memcpy(v, p, 16);
        c = step8(c, v[0], v[1], t);
        c = step8(c, v[2], v[3], t);
#endif
    }
    return bytes(c, p, n, t);
}
// gzip's CRC-32 of p[0, n), sequentially
FSLR_HD uint32_t crc(const unsigned char *p, long long n, const Tab *t) { return update(0xFFFFFFFFu, p, n, t) ^ 0xFFFFFFFFu; }

// Lane `lane`'s share of the CRC of a block of n <= 65536 bytes.  Segments are aligned to the block's END: lane l covers
// [max(0, n - (32 - l) * SEG), max(0, n - (31 - l) * SEG)), so every lane's remainder is followed by exactly (31 - l) * SEG
// bytes and one multiply by shift[31 - l] puts it in place.  The lane holding byte 0 starts from 0xFFFFFFFF (the initial
// value, which the shift carries through the whole block), the others from 0; lanes with an empty segment give 0.  The
// XOR of all 32 shares, passed through `finish`, is the block's CRC.
FSLR_HD uint32_t lane_share(const unsigned char *blk, int n, int lane, const Tab *t, const uint32_t *shift) {
    const int lo = n - (LANES - lane) * SEG > 0 ? n - (LANES - lane) * SEG : 0;
    const int hi = n - (LANES - 1 - lane) * SEG > 0 ? n - (LANES - 1 - lane) * SEG : 0;
    if (hi == 0) return 0;
    const uint32_t c = update(lo == 0 ? 0xFFFFFFFFu : 0u, blk + lo, hi - lo, t);
    return multmodp(shift[LANES - 1 - lane], c);
}
FSLR_HD uint32_t finish(uint32_t x, int n) { return n ? x ^ 0xFFFFFFFFu : 0u; }   // the CRC of no bytes is 0

}  // namespace crc32

#ifdef __CUDACC__
namespace crc32 {
__constant__ Tables TABLES = make_tables();
constexpr int CRC_WARPS = 8;                     // BGZF blocks per CTA
// one warp per BGZF block of the inflated stream (out_off / out_len as k_inflate wrote it); want[blk] = the CRC32 field of
// the block's trailer.  A mismatch lowers *bad to the block's index, so the smallest bad index survives any schedule.
__global__ void __launch_bounds__(CRC_WARPS * 32) k_bgzf_crc(const unsigned char *__restrict__ text, const long long *__restrict__ out_off,
                                                             const int *__restrict__ out_len, const uint32_t *__restrict__ want,
                                                             int n_blocks, unsigned *bad) {
    __shared__ uint32_t t[8][256];
    __shared__ uint32_t shift[LANES];
    for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) t[i >> 8][i & 255] = TABLES.t[i >> 8][i & 255];
    if (threadIdx.x < LANES) shift[threadIdx.x] = TABLES.shift[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31, blk = blockIdx.x * CRC_WARPS + (threadIdx.x >> 5);
    if (blk >= n_blocks) return;
    const int n = out_len[blk];
    uint32_t x = lane_share(text + out_off[blk], n, lane, t, shift);
#pragma unroll
    for (int o = 16; o; o >>= 1) x ^= __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0 && finish(x, n) != want[blk]) atomicMin(bad, (unsigned)blk);
}
}  // namespace crc32
#endif
