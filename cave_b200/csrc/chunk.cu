// Chunked calls (cave_forward_backward_chunk): the offset rebase of a per-instance CSR chunk cut out of a larger batch, so that
// the sparse pack of every chunk is built from the chunk's own copy without a host pass over its offsets.
#include <cuda_runtime.h>
#include <stdint.h>

namespace cave {

__global__ void csr_rebase_kernel(long long* inst_off, long long n_inst_off, long long row_base, long long* row_ptr,
                                  long long n_row_ptr, long long nnz_base) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_inst_off + n_row_ptr; i += stride) {
        if (i < n_inst_off) inst_off[i] -= row_base;
        else row_ptr[i - n_inst_off] -= nnz_base;
    }
}

cudaError_t launch_csr_rebase(long long* inst_off, long long n_inst_off, long long row_base, long long* row_ptr,
                              long long n_row_ptr, long long nnz_base, cudaStream_t stream) {
    const long long n = n_inst_off + n_row_ptr;
    long long blocks = (n + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    csr_rebase_kernel<<<(int)blocks, 256, 0, stream>>>(inst_off, n_inst_off, row_base, row_ptr, n_row_ptr, nnz_base);
    return cudaGetLastError();
}

}  // namespace cave
