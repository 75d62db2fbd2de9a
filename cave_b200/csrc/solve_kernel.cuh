#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cave {

struct SolveParams {
    const float* A;
    const void* pred;
    void* grad;
    void* proj;            // nullable
    int B, m_max, d;
    int64_t dpad;
    // pack
    const int *nvalid, *ngen, *gennnz, *nsingc;
    const int4* gen;
    const unsigned char* ctype;
    const float* avg;
    const int* csr_ok;
    const float *maxl1, *maxl2;
    const ulonglong2* ghash;
    const uint16_t* csr_col;
    const float* csr_val;
    int64_t cap_nnz;
    // scratch
    int* counter;
    double *loss64, *rnorm64;
    int *status, *iters;
    char* slots;
    size_t slot_bytes;
    char* large; size_t large_bytes; int n_large;      // worst-case slots, taken under a lock (counter[8 + i]) when needed
    int smem_bytes;
    // epilogue / options
    int mode;
    double inner_ratio, sign, gscale;
    int max_iter, max_ls;
    double tol;
    const int* inst_index; // nullable: batch position -> instance of the (dataset-wide) pack and of A
    // launch plan: this launch is configuration cfg_id of layout.cuh's table and runs only if the pack's plan
    // statistics select it (cfg_id < 0: forced, no check)
    int cfg_id;
    const unsigned long long* plan;
    const int* order;      // nullable: work-queue position -> instance (most expensive first)
    const int* dense_flag; // nullable: [B] 1 = the dense (Gram) path owns this batch position, skip it here
    long long n_packed;    // instances in the pack (inst_index values must be below it)
    const char* setup;     // nullable: cached per-instance setup blocks of the pack (layout.cuh SetupBlock)
    long long setup_stride;
    char* warm;            // nullable: warm-start slots, one per pack instance (layout.cuh warm_slot_bytes)
    long long warm_stride;
    int warm_cap;          // most variables a slot holds
};

struct FinalizeParams {
    int B, reduction;
    const double *loss64, *rnorm64;
    const int *status, *iters;
    void *loss, *loss_i, *rnorm;
    int *status_out, *iters_out;
};

cudaError_t launch_solve(const SolveParams& p, int compute_f32, int io_f32, int grid, int threads, cudaStream_t stream);
// dynamic shared memory of the wide configuration (layout.cuh kWideConfig) on the current device: the per-block maximum less
// the largest static shared memory of the solve kernels, rounded down to 16 bytes
cudaError_t solve_wide_smem_bytes(int* out);
cudaError_t launch_finalize(const FinalizeParams& p, int io_f32, cudaStream_t stream);

}  // namespace cave
