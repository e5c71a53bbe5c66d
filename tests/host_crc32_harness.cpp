// Host build of fslr_b200/csrc/crc32.cuh for tests/test_crc32_host.py (g++; the same source runs on the device).
#include "../fslr_b200/csrc/crc32.cuh"
static constexpr crc32::Tables TAB = crc32::make_tables();

extern "C" uint32_t host_crc32(const unsigned char *p, long long n) { return crc32::crc(p, n, TAB.t); }
// k_bgzf_crc's arithmetic, one lane after the other: the XOR of the 32 lane shares, finished
extern "C" uint32_t host_crc32_lanes(const unsigned char *p, int n) {
    uint32_t x = 0;
    for (int lane = 0; lane < crc32::LANES; lane++) x ^= crc32::lane_share(p, n, lane, TAB.t, TAB.shift);
    return crc32::finish(x, n);
}
extern "C" uint32_t host_multmodp(uint32_t a, uint32_t b) { return crc32::multmodp(a, b); }
extern "C" uint32_t host_shift(int j) { return TAB.shift[j]; }
