// Dense regime (instances without singleton rows and with enough rows that G = A A^T is a real contraction):
// shared declarations of the prep / Gram / Gram-space solve kernels and of their workspace layout.
//
// Per round of at most n_slots dense instances (all on the caller's stream, no host round trip):
//   dense_prep_kernel   reads the valid rows of A once, writes them split into two TF32 planes (hi = rn_tf32(a),
//                       lo = rn_tf32(a - hi)), zero padded to [m_pad, d_pad], plus b = A c (float64) and ||a_i||_1
//   dense_gram_kernel   G~ = hi hi^T + hi lo^T + lo hi^T ("3xTF32") on the 5th-generation tensor cores: TMA
//                       (cp.async.bulk.tensor) tiles into 128B-swizzled shared memory, tcgen05.mma with float32
//                       accumulators in TMEM, epilogue tcgen05.ld -> registers -> both triangles of G~ in global memory
//   dense_solve_kernel  one CTA per instance: projected Newton on min 1/2 lam^T G~ lam - b^T lam, lam >= 0, with a
//                       blocked float32 Cholesky of G~_FF in the instance's workspace and float64 iterates; then the
//                       iterate is polished against A itself in float64 (true gradient A (A^T lam - c)), so the
//                       result is anchored to A and G~ only acts as the metric; fused loss / gradient epilogue.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "layout.cuh"

namespace cave {

constexpr int kDenseMinRows = 128;      // below this the in-shared-memory Lawson-Hanson path is the better tool

// Workspace of the dense path inside the caller's scratch buffer.
struct DenseLayout {
    size_t ctrl;        // int[16]: [0] number of dense instances of the call, [1] work counter of the solve kernel
    size_t list;        // int[B]  batch positions of the dense instances, ascending
    size_t flag;        // int[B]  1: the dense path owns this instance (cleared again when it hands it back)
    size_t planes;      // float[n_slots][2][m_pad][d_pad]   TF32 hi / lo planes (one 2-D TMA tensor)
    size_t G;           // float[n_slots][m_pad][m_pad]      Gram matrix, both triangles
    size_t W;           // float[n_slots][m_pad][m_pad]      Cholesky workspace of the free block
    size_t bvec;        // double[n_slots][m_pad]            b = A c
    size_t l1;          // float[n_slots][m_pad]             ||a_i||_1
    size_t vec;         // double[n_slots][vec_doubles]      spill area for the solver's vectors
    size_t vec_doubles;
    int64_t m_pad, d_pad, n_slots;
    size_t total;
};

CAVE_HD int64_t dense_m_pad(int64_t m_max) { return (int64_t)align_up((size_t)m_max, 128); }
CAVE_HD int64_t dense_d_pad(int64_t d) { return (int64_t)align_up((size_t)d, 32); }
CAVE_HD size_t dense_slot_bytes(int64_t m_max, int64_t d) {
    const size_t mp = (size_t)dense_m_pad(m_max), dp = (size_t)dense_d_pad(d);
    return 2 * mp * dp * 4 + 2 * mp * mp * 4 + mp * 12 + (8 * mp + 3 * dp + 64) * 8;
}
CAVE_HD DenseLayout make_dense_layout(int64_t B, int64_t m_max, int64_t d, int64_t n_slots, size_t base) {
    DenseLayout L;
    L.m_pad = dense_m_pad(m_max); L.d_pad = dense_d_pad(d); L.n_slots = n_slots;
    const size_t mp = (size_t)L.m_pad, dp = (size_t)L.d_pad, ns = (size_t)n_slots;
    L.vec_doubles = 8 * mp + 3 * dp + 64;
    size_t o = align_up(base, 1024);
    L.ctrl = o;   o = align_up(o + 512, 256);     // 16 ints, then 16 x uint64 phase clocks (CAVE_DENSE_PROFILE builds)
    L.list = o;   o = align_up(o + (size_t)B * 4, 256);
    L.flag = o;   o = align_up(o + (size_t)B * 4, 256);
    L.planes = o = align_up(o, 1024); o += ns * 2 * mp * dp * 4;
    L.G = o = align_up(o, 1024);      o += ns * mp * mp * 4;
    L.W = o = align_up(o, 1024);      o += ns * mp * mp * 4;
    L.bvec = o = align_up(o, 256);    o += ns * mp * 8;
    L.l1 = o = align_up(o, 256);      o += ns * mp * 4;
    L.vec = o = align_up(o, 256);     o += ns * L.vec_doubles * 8;
    L.total = align_up(o, 256);
    return L;
}

// tiles of the upper block triangle of an nI x nI block matrix (128-row blocks), 128 x (128 | 256) each
CAVE_HD int dense_tiles(int nI) {
    int t = 0;
    for (int I = 0; I < nI; ++I) t += (nI - I + 1) / 2;
    return t;
}

struct DenseParams {
    // inputs
    const float* A;             // [*, m_max, d]
    const void* pred;           // [B, d] io dtype
    int B, m_max, d;
    const int* inst_index;      // nullable
    long long n_packed;         // instances in the pack (bound of inst_index values)
    const int *nvalid, *ngen, *nsingc;
    const int4* gen;            // [*, m_max]
    const unsigned char* ctype; // [*, dpad]
    const float* avg;           // [*, dpad]
    int64_t dpad;               // padded d of the pack (ctype / avg stride)
    const unsigned long long* plan;   // the pack's plan block (PLAN_NO_AVG), nullable
    // workspace
    char* ws;                   // scratch base
    DenseLayout L;
    int round;                  // this launch handles dense instances [round * n_slots, (round + 1) * n_slots)
    int trace_b;                // diagnostics (CAVE_DENSE_TRACE=<batch index>): per-iteration printf of that instance, -1 off
    int no_handback;            // diagnostics (CAVE_DENSE_NO_HANDBACK=1): keep the result of an instance that would be handed back,
                                // status |= reason << 16 (1 phase-1 cap, 2 phase-1 stall, 3 phase-2 cap, 4 phase-2 stall) | phase << 12
    int force;                  // 1: every instance without singleton rows and >= kDenseMinRows rows qualifies
    // outputs
    void* grad; void* proj;
    double *loss64, *rnorm64;
    int *status, *iters;
    // options
    int mode; double inner_ratio, sign, gscale;
    int max_iter, max_ls; double tol;
    int io_f32;
    int nk;                     // d_pad / 32
    int tc_update;              // set by launch_dense_solve: the Cholesky block-column update runs on the tensor cores (shared memory permitting)
    char* warm;                 // nullable: warm-start slots, one per pack instance (layout.cuh dense_warm_slot_bytes)
    long long warm_stride;
    int warm_cap;               // most rows a slot holds
};

cudaError_t launch_dense_list(const DenseParams& p, cudaStream_t stream);
cudaError_t launch_dense_prep(const DenseParams& p, cudaStream_t stream);
cudaError_t launch_dense_gram(const DenseParams& p, cudaStream_t stream);
cudaError_t launch_dense_solve(const DenseParams& p, cudaStream_t stream);
const char* dense_last_error();

}  // namespace cave
