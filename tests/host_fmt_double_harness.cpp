// Host build of fslr_b200/csrc/fmt_double.cuh for tests/test_fmt_double_host.py: formats n doubles into fixed 32-byte
// slots and their lengths.
#include "../fslr_b200/csrc/fmt_double.cuh"

extern "C" void host_fmt_many(const double *x, long long n, char *out, int *len) {
    for (long long i = 0; i < n; i++) len[i] = fmtd::fmt_repr_f64(x[i], out + i * fmtd::FMT_F64_MAX);
}
