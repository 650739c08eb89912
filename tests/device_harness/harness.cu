// Device harness of the kernel headers (TEST INFRASTRUCTURE ONLY, built by tests/test_device_bounds.py into a shared
// library in a temporary directory, one per shipped define set; never linked into libzkpair.so).  Runs the bodies of
// bodies.cuh on raw Montgomery representatives, one lane pair per element as the product kernels do.
#include <cuda_runtime.h>

#include "bodies.cuh"

using namespace zkp;

#define HARNESS_TPB 128

__global__ void __launch_bounds__(HARNESS_TPB) k_body(int body, const uint64_t *in, uint64_t *out, int n) {
    int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 1);
    // converged builds: every lane of the block takes the same path (ZKP_CODE_SYNC is a __syncthreads()), so tail
    // lanes recompute the last element and store nothing, as k_pairing does
    const bool live = i < n;
    if (!live) i = n - 1;
    body_one(body, in + (size_t)i * BODY_U64, out + (size_t)i * BODY_U64, live);
}

// n elements of BODY_U64 u64 each, host buffers in and out.  Returns 0 or the CUDA error code.
extern "C" int harness_run(int body, int n, const uint64_t *in, uint64_t *out) {
    if (n <= 0) return 0;
    const size_t bytes = (size_t)n * BODY_U64 * sizeof(uint64_t);
    uint64_t *d_in = nullptr, *d_out = nullptr;
    cudaError_t e = cudaMalloc(&d_in, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d_out, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(d_in, in, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(d_out, 0, bytes);
    if (e == cudaSuccess) {
        const int blocks = (int)((2 * (size_t)n + HARNESS_TPB - 1) / HARNESS_TPB);
        k_body<<<blocks, HARNESS_TPB>>>(body, d_in, d_out, n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out, bytes, cudaMemcpyDeviceToHost);
    cudaFree(d_in);
    cudaFree(d_out);
    return (int)e;
}
