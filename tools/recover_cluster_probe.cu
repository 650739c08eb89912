// Prints what the CUDA runtime reports for k_cells_recover as the library configures it: registers, shared memory and
// cudaOccupancyMaxActiveClusters (one cluster = two blocks of 512 threads with 128 KiB of dynamic shared memory each).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o build/recover_cluster_probe
//        tools/recover_cluster_probe.cu zkvm_pairings_b200/csrc/pairing_kernel.cu zkvm_pairings_b200/csrc/fe_kernel.cu
#include "../zkvm_pairings_b200/csrc/kernels.cu"

int main() {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, 0) != cudaSuccess) return 1;
    cudaError_t e = cudaFuncSetAttribute(k_cells_recover, cudaFuncAttributeMaxDynamicSharedMemorySize, ZKP_RECOVER_HALF * sizeof(Fr));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2);
    cfg.blockDim = dim3(ZKP_CELLS_TPB);
    cfg.dynamicSmemBytes = ZKP_RECOVER_HALF * sizeof(Fr);
    int clusters = -1;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveClusters(&clusters, k_cells_recover, &cfg);
    cudaFuncAttributes a = {};
    cudaFuncGetAttributes(&a, k_cells_recover);
    printf("%s, %d SMs: k_cells_recover %d registers, %zu B static + %zu B dynamic shared memory per block; "
           "cudaOccupancyMaxActiveClusters = %d (%s)\n", p.name, p.multiProcessorCount, a.numRegs, a.sharedSizeBytes,
           (size_t)cfg.dynamicSmemBytes, clusters, cudaGetErrorString(e));
    return e == cudaSuccess ? 0 : 1;
}
