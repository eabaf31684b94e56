// CPU check of glibc_log1pf (sage_b200/csrc/glibc_log.cuh) against this host's libm log1pf on EVERY float (compiled by tests/test_glibc_log.py).
#include "glibc_log.cuh"

#include <cmath>
#include <cstdio>

int main() {
    unsigned long long bad = 0, n = 0;
#pragma omp parallel for reduction(+ : bad, n) schedule(static)
    for (long long b = 0; b < (1ll << 32); b++) {
        const uint32_t u = (uint32_t)b;
        float x;
        memcpy(&x, &u, 4);
        volatile float vx = x;
        const float ref = log1pf(vx), got = sb::glog::glibc_log1pf(x);
        n++;
        bad += memcmp(&ref, &got, 4) != 0;   // NaN results too: sign and payload as the host's SSE arithmetic leaves them
    }
    printf("tested %llu bad %llu\n", n, bad);
    return bad != 0;
}
