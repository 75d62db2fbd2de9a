// Instantiation of the solve kernel: factor precision float, I/O dtype float.
#include "solve_kernel_impl.cuh"
namespace cave {
template cudaError_t launch_solve_t<float, float>(const SolveParams&, int, int, cudaStream_t);
template cudaError_t solve_static_smem_t<float, float>(size_t*);
}
