// Microbenchmark: how many random 2-byte lookups per second can one B200 sustain on a
// unidic-sized connection matrix (15626 x 15388 i16 = 459 MiB) when the ids follow the same
// Zipf(1.0) law as the synthetic dictionary, (a) with ids in random order, (b) frequency-sorted?
// This is the practical ceiling for K3's dominant access pattern.
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o tools/gather_bench tools/gather_bench.cu
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <numeric>
#include <random>
#include <vector>

#define CK(x)                                                                      \
    do {                                                                           \
        cudaError_t e = (x);                                                       \
        if (e != cudaSuccess) {                                                    \
            std::printf("%s: %s\n", #x, cudaGetErrorString(e));                    \
            return 1;                                                              \
        }                                                                          \
    } while (0)

template <int MODE>
__global__ void k_gather(const int16_t* __restrict__ M, uint32_t NR, const uint32_t* __restrict__ lr, size_t n,
                         long long* out) {
    size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    size_t stride = size_t(gridDim.x) * blockDim.x;
    long long acc = 0;
    for (; i + 3 * stride < n; i += 4 * stride) {
        uint32_t a = lr[i], b = lr[i + stride], c = lr[i + 2 * stride], d = lr[i + 3 * stride];
        const int16_t* pa = M + size_t(a & 0xFFFF) * NR + (a >> 16);
        const int16_t* pb = M + size_t(b & 0xFFFF) * NR + (b >> 16);
        const int16_t* pc = M + size_t(c & 0xFFFF) * NR + (c >> 16);
        const int16_t* pd = M + size_t(d & 0xFFFF) * NR + (d >> 16);
        int va, vb, vc, vd;
        if (MODE == 0) {
            va = __ldg(pa), vb = __ldg(pb), vc = __ldg(pc), vd = __ldg(pd);
        } else {
            asm volatile("ld.global.nc.L1::no_allocate.s16 %0, [%1];" : "=r"(va) : "l"(pa));
            asm volatile("ld.global.nc.L1::no_allocate.s16 %0, [%1];" : "=r"(vb) : "l"(pb));
            asm volatile("ld.global.nc.L1::no_allocate.s16 %0, [%1];" : "=r"(vc) : "l"(pc));
            asm volatile("ld.global.nc.L1::no_allocate.s16 %0, [%1];" : "=r"(vd) : "l"(pd));
        }
        acc += va + vb + vc + vd;
    }
    if (acc == 0x7fffffffffffll) *out = acc;
}

int main() {
    const uint32_t NL = 15626, NR = 15388;
    const size_t n = size_t(1) << 28;  // 268M lookups per launch
    std::mt19937_64 rng(1);
    auto zipf_cdf = [](uint32_t k) {
        std::vector<double> c(k);
        double s = 0;
        for (uint32_t i = 0; i < k; ++i) c[i] = (s += 1.0 / (i + 1));
        for (auto& v : c) v /= s;
        return c;
    };
    std::vector<double> cl = zipf_cdf(NL - 1), cr = zipf_cdf(NR - 1);
    std::vector<uint32_t> lperm(NL - 1), rperm(NR - 1);
    std::iota(lperm.begin(), lperm.end(), 0);
    std::iota(rperm.begin(), rperm.end(), 0);
    std::shuffle(lperm.begin(), lperm.end(), rng);
    std::shuffle(rperm.begin(), rperm.end(), rng);
    std::vector<uint32_t> sorted(n), shuffled(n), uniform(n);
    std::uniform_real_distribution<double> U(0, 1);
    for (size_t i = 0; i < n; ++i) {
        uint32_t l = uint32_t(std::lower_bound(cl.begin(), cl.end(), U(rng)) - cl.begin());
        uint32_t r = uint32_t(std::lower_bound(cr.begin(), cr.end(), U(rng)) - cr.begin());
        sorted[i] = (l + 1) | ((r + 1) << 16);
        shuffled[i] = (lperm[l] + 1) | ((rperm[r] + 1) << 16);
        uniform[i] = uint32_t(rng() % NL) | (uint32_t(rng() % NR) << 16);
    }
    int16_t* M;
    uint32_t* d_lr;
    long long* d_out;
    CK(cudaMalloc(&M, size_t(NL) * NR * 2));
    CK(cudaMemset(M, 1, size_t(NL) * NR * 2));
    CK(cudaMalloc(&d_lr, n * 4));
    CK(cudaMalloc(&d_out, 8));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const char* names[3] = {"zipf ids frequency-sorted", "zipf ids in random order", "uniform ids"};
    const std::vector<uint32_t>* sets[3] = {&sorted, &shuffled, &uniform};
    for (int s = 0; s < 3; ++s) {
        CK(cudaMemcpy(d_lr, sets[s]->data(), n * 4, cudaMemcpyHostToDevice));
        for (int mode = 0; mode < 2; ++mode) {
            float best = 1e9;
            for (int rep = 0; rep < 4; ++rep) {
                cudaEventRecord(e0);
                if (mode == 0)
                    k_gather<0><<<148 * 16, 256>>>(M, NR, d_lr, n, d_out);
                else
                    k_gather<1><<<148 * 16, 256>>>(M, NR, d_lr, n, d_out);
                cudaEventRecord(e1);
                CK(cudaEventSynchronize(e1));
                float ms;
                cudaEventElapsedTime(&ms, e0, e1);
                best = std::min(best, ms);
            }
            std::printf("%-28s %-22s %8.3f ms  %7.1f G lookups/s\n", names[s], mode ? "ld.nc.L1::no_allocate" : "ld.nc (L1 allocate)",
                        best, double(n) / best / 1e6);
        }
    }
    return 0;
}
