// check_polya_math.cu — nanopolish_b200/csrc/polya_math.cuh against the C library of the machine it runs on (test infrastructure).
//   device (default): expf_glibc on EVERY float x <= 0 (-0, the normal and subnormal negatives, -inf) and logf_glibc on EVERY
//                     float x >= 0 (+0, subnormals, normals, +inf), each compared bit for bit with libm's expf / logf
//   --host-only N:    the host copies of both functions on N pseudo-random inputs of each domain (plus the edge values)
// Prints the mismatch counts; exit code 0 iff both are 0.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <vector>
#include <cuda_runtime.h>
#include "../../nanopolish_b200/csrc/polya_math.cuh"

using namespace nph_polya_math;

static bool same(float a, float b) { return f2u(a) == f2u(b) || (std::isnan(a) && std::isnan(b)); }

__global__ void eval_kernel(uint32_t first_bits, uint32_t n, int which, float* out)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float x = u2f(first_bits + i);
        out[i] = which == 0 ? expf_glibc(x) : logf_glibc(x);
    }
}

// [lo, hi] bit patterns: expf over 0x80000000 (-0) .. 0xff800000 (-inf), logf over 0 (+0) .. 0x7f800000 (+inf)
static unsigned long long run_device(int which, uint32_t lo, uint32_t hi)
{
    const uint32_t chunk = 1u << 26;
    float* d = nullptr;
    if (cudaMalloc(&d, sizeof(float) * chunk) != cudaSuccess) { fprintf(stderr, "cudaMalloc failed\n"); exit(2); }
    std::vector<float> h(chunk);
    unsigned long long bad = 0;
    for (uint64_t b = lo; b <= hi; b += chunk) {
        const uint32_t n = (uint32_t)std::min<uint64_t>(chunk, (uint64_t)hi - b + 1);
        eval_kernel<<<1024, 256>>>((uint32_t)b, n, which, d);
        if (cudaMemcpy(h.data(), d, sizeof(float) * n, cudaMemcpyDeviceToHost) != cudaSuccess) { fprintf(stderr, "kernel failed\n"); exit(2); }
        #pragma omp parallel for reduction(+:bad) schedule(static)
        for (long long i = 0; i < (long long)n; ++i) {
            const float x = u2f((uint32_t)(b + i));
            const float want = which == 0 ? expf(x) : logf(x);
            if (!same(h[i], want)) {
                if (bad < 5) fprintf(stderr, "%s(%a): device %a, libm %a\n", which == 0 ? "expf" : "logf", x, h[i], want);
                ++bad;
            }
        }
    }
    cudaFree(d);
    return bad;
}

static unsigned long long run_host(int which, uint64_t n, uint32_t lo, uint32_t hi, unsigned long long* tried)
{
    const float edges[] = {0.0f, -0.0f, INFINITY, -INFINITY, 1.0f, -0x1.f8cbb2p+5f, -0x1.9fe368p6f, -0x1.9fe366p6f, -88.0f, 0x1p-149f, 0x1p-126f,
                           0x1.fffffep-127f, 100.0f, -103.0f, -104.0f, 3.4028235e38f};
    unsigned long long bad = 0, cnt = 0;
    for (float x : edges) {
        if (which == 0 ? !(x <= 0.0f) : !(x >= 0.0f)) continue;
        const float got = which == 0 ? expf_glibc(x) : logf_glibc(x), want = which == 0 ? expf(x) : logf(x);
        ++cnt;
        if (!same(got, want)) { fprintf(stderr, "%s(%a): restated %a, libm %a\n", which == 0 ? "expf" : "logf", x, got, want); ++bad; }
    }
    const uint64_t span = (uint64_t)hi - lo + 1;
    #pragma omp parallel for reduction(+:bad, cnt) schedule(static)
    for (long long i = 0; i < (long long)n; ++i) {
        uint64_t s = 0x9E3779B97F4A7C15ull * (uint64_t)(i + 1) + (uint64_t)which;
        s ^= s >> 31; s *= 0xBF58476D1CE4E5B9ull; s ^= s >> 27;
        uint32_t bits = lo + (uint32_t)(s % span);
        if ((i & 3) == 0 && which == 0) bits = f2u(-(float)((s >> 40) % 120000) * 1e-3f - (float)((s >> 20) & 1023) * 1e-7f);   // the emission range
        const float x = u2f(bits);
        const float got = which == 0 ? expf_glibc(x) : logf_glibc(x), want = which == 0 ? expf(x) : logf(x);
        ++cnt;
        if (!same(got, want)) ++bad;
    }
    *tried += cnt;
    return bad;
}

int main(int argc, char** argv)
{
    const uint32_t e_lo = 0x80000000u, e_hi = 0xff800000u, l_lo = 0u, l_hi = 0x7f800000u;
    if (argc > 2 && strcmp(argv[1], "--host-only") == 0) {
        const uint64_t n = strtoull(argv[2], nullptr, 10);
        unsigned long long te = 0, tl = 0;
        const unsigned long long be = run_host(0, n, e_lo, e_hi, &te), bl = run_host(1, n, l_lo, l_hi, &tl);
        printf("host: expf %llu bad of %llu, logf %llu bad of %llu\n", be, te, bl, tl);
        return (be || bl) ? 1 : 0;
    }
    const unsigned long long be = run_device(0, e_lo, e_hi), bl = run_device(1, l_lo, l_hi);
    printf("device: expf %llu bad of %llu, logf %llu bad of %llu\n", be, (unsigned long long)(e_hi - e_lo) + 1, bl, (unsigned long long)(l_hi - l_lo) + 1);
    return (be || bl) ? 1 : 0;
}
