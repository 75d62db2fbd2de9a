#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cave {

struct ScanParams {
    const float* A;
    const int* m_rows;      // nullable
    int B, m_max, d;
    int R, stages;          // filled by launch_scan
    size_t stage_stride;    // filled by launch_scan
    int64_t dpad;
    int *nvalid, *navg, *ngen, *gennnz, *nsingc;
    int4* gen4;             // per general row: (row, nnz, offset in the packed CSR, 0), ascending row
    unsigned char* ctype;
    float* avg;
    // packed CSR of the general rows (per instance capacity cap_nnz) + row hashes for +-row matching
    ulonglong2* ghash;
    uint16_t* csr_col;
    float* csr_val;
    int cap_nnz;
    int* csr_ok;            // 1 if every general row of the instance fitted into the packed CSR
    float *maxl1, *maxl2;   // max_i ||a_i||_1 and max_i ||a_i||_2^2 over the general rows
    int skip_avg;           // 1: the average of the normalised rows is not needed (one-shot pack of an exact-mode call: the
                            // exact loss has no push-inside step, src/cave.py:84-129); avg is then written as the singleton part only
};

cudaError_t launch_scan(const ScanParams& p, cudaStream_t stream);
// sparse ingestion: the same pack from per-instance CSR input (device pointers); p.A is unused
cudaError_t launch_scan_sparse(const ScanParams& p, const long long* inst_off, const long long* row_ptr, const int* col,
                               const float* val, cudaStream_t stream);

struct PlanParams {
    int B, m_max, d;
    const int *nvalid, *ngen, *gennnz, *nsingc, *csr_ok;
    const int4* gen4;
    const ulonglong2* ghash;
    unsigned long long* plan;   // zeroed by the caller on the same stream
    int* okey;                  // [B] cost estimate per instance
    int* order;                 // [B] instances by descending cost (filled by the order kernel)
    // setup kernel (cached per-instance solver setup, layout.cuh SetupBlock)
    const uint16_t* csr_col; const float* csr_val; int64_t cap_nnz;
    char* setup; int64_t setup_stride, setup_cap_v;
    int wide_smem;              // dynamic shared memory of the wide solve configuration (solve_wide_smem_bytes)
};
cudaError_t launch_plan(const PlanParams& p, cudaStream_t stream);
cudaError_t launch_clear_setup(char* setup, long long stride, int B, cudaStream_t stream);

}  // namespace cave
