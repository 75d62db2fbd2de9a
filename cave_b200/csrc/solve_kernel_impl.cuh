// Solve kernel template and its launcher; instantiated once per (factor dtype, I/O dtype) in solve_inst_*.cu so
// that the four variants compile in parallel.  Each comes in two kernels: with and without the warm-start code.
#pragma once
#ifndef CAVE_LB_T
#define CAVE_LB_T 256      // launch bounds of the solve kernel: 256 x 2 = 128 registers per thread
#define CAVE_LB_C 2
#endif
#include <cuda_runtime.h>
#include <stdint.h>
#include "layout.cuh"
#include "solve_kernel.cuh"
#include "solver_core.cuh"

namespace cave {

// WARM: the variant for calls with a warm-start buffer (p.warm); the other one compiles none of the warm-start code.
template <class T, class TIO, bool WARM>
__global__ void __launch_bounds__(CAVE_LB_T, CAVE_LB_C) solve_kernel(SolveParams p) {
    extern __shared__ __align__(16) char smem[];
    __shared__ double red[64];
    __shared__ int s_b, s_large;
    // >= 0: the warm start of instance s_b failed after this many iterations; it is solved once more from zero instead of
    // taking the next instance (so a warm start can cost time but never end worse than a cold solve)
    __shared__ int s_retry;
    if (p.cfg_id >= 0 && choose_solve_config(p.plan, sizeof(T), sizeof(TIO) == 8 ? (size_t)p.d * 4 : 0) != p.cfg_id) return;
    Ctx cx(red);
    char* slot = p.slots + (size_t)blockIdx.x * p.slot_bytes;
    EpiParams ep; ep.mode = p.mode; ep.inner_ratio = p.inner_ratio; ep.sign = p.sign; ep.gscale = p.gscale;
    SolveOpts opt; opt.max_iter = p.max_iter; opt.max_ls = p.max_ls; opt.tol = p.tol;
    const TIO* pred = (const TIO*)p.pred;
    TIO* grad = (TIO*)p.grad;
    TIO* proj = (TIO*)p.proj;
    if (WARM && cx.tid == 0) s_retry = -1;
    for (;;) {
        if (cx.tid == 0 && (!WARM || s_retry < 0)) s_b = atomicAdd(p.counter, 1);
        __syncthreads();
        const int slot_b = s_b, retry = WARM ? s_retry : -1;
        __syncthreads();
        if (slot_b >= p.B) break;
        const int b = p.order ? p.order[slot_b] : slot_b;
        if (p.dense_flag && p.dense_flag[b]) continue;                            // solved by the dense (Gram) path
        const long long qi = p.inst_index ? (long long)p.inst_index[b] : (long long)b;
        if (qi < 0 || qi >= p.n_packed || (p.mode != MODE_EXACT && p.plan[PLAN_NO_AVG] != 0ull)) {
            // an index outside the pack (stale permutation, another shard's index): report, never read out of bounds;
            // likewise a pack without the average unit normal used by a mode that pushes towards it
            if (cx.tid == 0) { p.loss64[b] = NAN; p.rnorm64[b] = NAN; p.status[b] = ST_BADINPUT; p.iters[b] = 0; }
            for (int k = cx.tid; k < p.d; k += cx.nthr) { grad[(size_t)b * p.d + k] = (TIO)NAN; if (proj) proj[(size_t)b * p.d + k] = (TIO)NAN; }
            continue;
        }
        const size_t q = (size_t)qi;     // instance of the pack / of A
        Instance in;
        in.A = p.A ? p.A + q * p.m_max * p.d : nullptr;
        in.gen = p.gen + q * p.m_max;
        in.ctype = p.ctype + q * p.dpad;
        in.avg = p.avg + q * p.dpad;
        in.d = p.d; in.ngen = p.ngen[q]; in.gen_nnz = p.gennnz[q]; in.nvalid = p.nvalid[q]; in.nsingc = p.nsingc[q];
        in.csr_ok = p.csr_ok[q]; in.maxl1 = p.maxl1[q]; in.maxl2 = p.maxl2[q];
        in.ghash = p.ghash + q * p.m_max;
        in.pcol = p.csr_col + q * p.cap_nnz;
        in.pval = p.csr_val + q * p.cap_nnz;
        in.setup = p.setup ? p.setup + q * (size_t)p.setup_stride : nullptr;
        in.warm = (WARM && p.warm) ? p.warm + q * (size_t)p.warm_stride : nullptr; in.warm_cap = p.warm_cap; in.warm_from_slot = retry < 0;
        // an instance whose working set cannot fit this CTA's slot borrows one of the worst-case slots under a lock
        char* islot = slot; size_t islot_bytes = p.slot_bytes;
        int held = -1;
        if (p.n_large > 0 && in.ngen > 0 && instance_slot_bytes(p.d, in.ngen, in.gen_nnz, in.nsingc == 0, 8) > p.slot_bytes) {
            if (cx.tid == 0) {
                int got = -1;
                unsigned ns = 64;
                for (int probe = (int)(blockIdx.x % (unsigned)p.n_large); got < 0; probe = (probe + 1) % p.n_large) {
                    if (atomicCAS(p.counter + 8 + probe, 0, 1) == 0) got = probe;
                    else if (probe == (int)(blockIdx.x % (unsigned)p.n_large)) { __nanosleep(ns); ns = ns < 4096 ? ns * 2 : ns; }
                }
                __threadfence();
                s_large = got;
            }
            __syncthreads();
            held = s_large;
            islot = p.large + (size_t)held * p.large_bytes; islot_bytes = p.large_bytes;
        }
        solve_instance<T, TIO, WARM>(cx, in, smem, (size_t)p.smem_bytes, islot, islot_bytes, pred + (size_t)b * p.d, ep, opt, grad + (size_t)b * p.d,
                               proj ? proj + (size_t)b * p.d : nullptr, p.loss64 + b, p.rnorm64 + b,
                               p.status + b, p.iters + b);
        __syncthreads();
        if (held >= 0 && cx.tid == 0) { __threadfence(); atomicExch(p.counter + 8 + held, 0); }
        if (WARM && cx.tid == 0) {          // (status and iters of b were written by this thread)
            const int st = p.status[b];
            if (retry >= 0) { p.iters[b] += retry; s_retry = -1; }
            else if ((st & ST_WARM) && ((st & 0xff) == ST_ITER_CAP || (st & 0xff) == ST_STALLED)) s_retry = p.iters[b];
        }
    }
}

template <class T, class TIO, bool WARM>
cudaError_t launch_solve_v(const SolveParams& p, int grid, int threads, cudaStream_t stream) {
    // the attribute is per device (and cheap to set): no process-wide cache, so a second GPU in the same process works
    static int configured[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = -1;
    if (dev < 0 || configured[dev] < p.smem_bytes) {
        cudaError_t e = cudaFuncSetAttribute(solve_kernel<T, TIO, WARM>, cudaFuncAttributeMaxDynamicSharedMemorySize, p.smem_bytes);
        if (e != cudaSuccess) return e;
        if (dev >= 0) configured[dev] = p.smem_bytes;
    }
    solve_kernel<T, TIO, WARM><<<grid, threads, p.smem_bytes, stream>>>(p);
    return cudaGetLastError();
}

template <class T, class TIO>
cudaError_t launch_solve_t(const SolveParams& p, int grid, int threads, cudaStream_t stream) {
    return p.warm ? launch_solve_v<T, TIO, true>(p, grid, threads, stream) : launch_solve_v<T, TIO, false>(p, grid, threads, stream);
}

// static shared memory of the two kernels of this (factor, I/O) pair, the larger one (the wide configuration's dynamic shared
// memory is the per-block maximum less this)
template <class T, class TIO>
cudaError_t solve_static_smem_t(size_t* out) {
    cudaFuncAttributes a, w;
    cudaError_t e = cudaFuncGetAttributes(&a, solve_kernel<T, TIO, false>);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&w, solve_kernel<T, TIO, true>);
    if (e == cudaSuccess) *out = a.sharedSizeBytes > w.sharedSizeBytes ? a.sharedSizeBytes : w.sharedSizeBytes;
    return e;
}

}  // namespace cave
