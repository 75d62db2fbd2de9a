// Kernel 2 — solve + fused epilogue: persistent CTAs pull instances from a work counter; each
// instance is solved entirely by one CTA with its working set in shared memory (spilling to the
// CTA's global scratch slot only when it does not fit), then the target / cosine loss /
// d loss / d pred epilogue runs in the same kernel (solver_core.cuh).
// Kernel 3 — finalize: fixed-order reduction of the per-instance losses (mean / sum) and dtype
// conversion of the per-instance outputs.
#include <cuda_runtime.h>
#include <stdint.h>
#include "layout.cuh"
#include "solve_kernel.cuh"

namespace cave {

template <class TIO>
__global__ void __launch_bounds__(1024) finalize_kernel(FinalizeParams p) {
    __shared__ double part[1024];
    const int tid = threadIdx.x;
    TIO* loss_i = (TIO*)p.loss_i;
    TIO* rnorm = (TIO*)p.rnorm;
    double acc = 0.0;
    for (int i = tid; i < p.B; i += 1024) {
        const double l = p.loss64[i];
        acc += l;
        loss_i[i] = (TIO)l;
        if (rnorm) rnorm[i] = (TIO)p.rnorm64[i];
        if (p.status_out) p.status_out[i] = p.status[i];
        if (p.iters_out) p.iters_out[i] = p.iters[i];
    }
    part[tid] = acc;
    __syncthreads();
    for (int s = 512; s > 0; s >>= 1) {
        if (tid < s) part[tid] += part[tid + s];
        __syncthreads();
    }
    if (tid == 0 && p.loss && p.reduction != 2)
        *(TIO*)p.loss = (TIO)(p.reduction == 0 ? part[0] / (double)p.B : part[0]);
}

template <class T, class TIO>
cudaError_t launch_solve_t(const SolveParams& p, int grid, int threads, cudaStream_t stream);     // solve_inst_*.cu
extern template cudaError_t launch_solve_t<float, float>(const SolveParams&, int, int, cudaStream_t);
extern template cudaError_t launch_solve_t<float, double>(const SolveParams&, int, int, cudaStream_t);
extern template cudaError_t launch_solve_t<double, float>(const SolveParams&, int, int, cudaStream_t);
extern template cudaError_t launch_solve_t<double, double>(const SolveParams&, int, int, cudaStream_t);

template <class T, class TIO>
cudaError_t solve_static_smem_t(size_t* out);                                                   // solve_inst_*.cu
extern template cudaError_t solve_static_smem_t<float, float>(size_t*);
extern template cudaError_t solve_static_smem_t<float, double>(size_t*);
extern template cudaError_t solve_static_smem_t<double, float>(size_t*);
extern template cudaError_t solve_static_smem_t<double, double>(size_t*);

cudaError_t solve_wide_smem_bytes(int* out) {
    int dev = 0, optin = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    size_t st = 0, s[4] = {0, 0, 0, 0};
    if (e == cudaSuccess) e = solve_static_smem_t<float, float>(&s[0]);
    if (e == cudaSuccess) e = solve_static_smem_t<float, double>(&s[1]);
    if (e == cudaSuccess) e = solve_static_smem_t<double, float>(&s[2]);
    if (e == cudaSuccess) e = solve_static_smem_t<double, double>(&s[3]);
    if (e != cudaSuccess) return e;
    for (size_t v : s) st = v > st ? v : st;
    // one figure for every instantiation: the pack's plan records it before the call's precision is known
    *out = (int)(((size_t)optin - st) & ~(size_t)15);
    return cudaSuccess;
}

cudaError_t launch_solve(const SolveParams& p, int compute_f32, int io_f32, int grid, int threads, cudaStream_t stream) {
    if (compute_f32) return io_f32 ? launch_solve_t<float, float>(p, grid, threads, stream)
                                   : launch_solve_t<float, double>(p, grid, threads, stream);
    return io_f32 ? launch_solve_t<double, float>(p, grid, threads, stream)
                  : launch_solve_t<double, double>(p, grid, threads, stream);
}

cudaError_t launch_finalize(const FinalizeParams& p, int io_f32, cudaStream_t stream) {
    if (io_f32) finalize_kernel<float><<<1, 1024, 0, stream>>>(p);
    else finalize_kernel<double><<<1, 1024, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace cave
