// probe_l2_read.cu -- L2 read bandwidth: every SM reads the same 128-KiB buffer over and over (ld.global.cg: cached in
// L2 only, so no request is served by L1; 16 bytes per lane, whole 32-byte sectors), so after the first pass every
// request is an L2 hit and no byte comes from HBM.  The
// denominator of a streamed tensor-path operand (tools/streamed_operand_bench.py).
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a probe_l2_read.cu -o probe_l2_read && ./probe_l2_read
// prints one JSON line: bytes read, best time of five launches, TB/s.
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>

#define CHECK(expr)                                                                                        \
    do {                                                                                                   \
        const cudaError_t e_ = (expr);                                                                     \
        if (e_ != cudaSuccess) {                                                                           \
            fprintf(stderr, "%s failed: %s\n", #expr, cudaGetErrorString(e_));                             \
            exit(1);                                                                                       \
        }                                                                                                  \
    } while (0)

__global__ void __launch_bounds__(512) l2_read_kernel(const double2 *buf, int n2, int iters, double *sink)
{
    double a = 0.0, b = 0.0;
    const int step = blockDim.x;                               // a block sweeps the buffer, 8 KiB per iteration
    int i = (blockIdx.x * blockDim.x + threadIdx.x) % n2;
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
#pragma unroll 8
        for (int k = 0; k < 8; k++) {
            double2 v;
            asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(buf + i));
            a += v.x;
            b += v.y;
            i += step;
            i = i >= n2 ? i - n2 : i;
        }
    }
    if (a + b == 1.2345) sink[0] = a + b;
}

int main()
{
    const int bytes = 128 * 1024, n2 = bytes / 16;
    int sms = 0;
    CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    double2 *buf;
    double *sink;
    CHECK(cudaMalloc(&buf, bytes));
    CHECK(cudaMalloc(&sink, 8));
    CHECK(cudaMemset(buf, 0, bytes));
    const int blocks = 4 * sms, threads = 512, iters = 2000;
    cudaEvent_t e0, e1;
    CHECK(cudaEventCreate(&e0));
    CHECK(cudaEventCreate(&e1));
    l2_read_kernel<<<blocks, threads>>>(buf, n2, 50, sink);              // warm-up: the buffer into L2
    CHECK(cudaGetLastError());
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        CHECK(cudaEventRecord(e0));
        l2_read_kernel<<<blocks, threads>>>(buf, n2, iters, sink);
        CHECK(cudaGetLastError());
        CHECK(cudaEventRecord(e1));
        CHECK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CHECK(cudaEventElapsedTime(&ms, e0, e1));
        best = ms < best ? ms : best;
    }
    const double read = 16.0 * 8.0 * iters * (double)blocks * threads;
    printf("{\"buffer_bytes\": %d, \"bytes_read\": %.0f, \"best_ms\": %.4f, \"tb_per_s\": %.3f, \"blocks\": %d, "
           "\"threads\": %d}\n", bytes, read, best, read / (best * 1e-3) / 1e12, blocks, threads);
    cudaFree(buf);
    cudaFree(sink);
    return 0;
}
