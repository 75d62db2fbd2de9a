// Dense regime, kernels 1-3: instance list, TF32 split ("prep") and the batched Gram contraction G = A A^T on the
// 5th-generation tensor cores (north_star item 1; SURVEY.md section 8d "Algorithmic flops").
//
// dense_gram_kernel is a persistent, warp-specialised sm_100a kernel, one CTA per SM:
//   warp 0      TMA producer: cp.async.bulk.tensor.2d tiles of the hi / lo planes (box 32 x 128 float32 = one
//               128-byte swizzle span per row) into a 2-stage shared-memory ring, completion on mbarriers
//   warp 1      MMA issuer (one elected lane): per 32-wide k-slab 4 x 3 tcgen05.mma.kind::tf32 instructions
//               (hi*hi + hi*lo + lo*hi, K = 8 each) into a 128 x (128|256) float32 accumulator in TMEM;
//               tcgen05.commit releases the shared-memory stage / publishes the accumulator
//   warps 2-5   epilogue: tcgen05.ld of the accumulator (each warp its 32 TMEM lanes), both orientations of the
//               tile written to G (exactly symmetric: the diagonal block is mirrored from its lower triangle)
// TMEM holds two accumulator stages (2 x 256 columns), so the epilogue of tile t overlaps the MMAs of tile t + 1.
// Only tiles on or above the block diagonal are computed.  Operand precision: a = hi + lo exactly to 2^-22 |a|, so
// G~ carries float32-level rounding (accumulation in the tensor core); the solver treats it as the metric of its
// Newton steps and anchors the result to A itself (dense_solve.cu).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include "dense.cuh"
#include "tc05.cuh"

namespace cave {

namespace {
thread_local std::string g_dense_err;
}
const char* dense_last_error() { return g_dense_err.c_str(); }

// ------------------------------------------------------------------ instance list
// One CTA: ordered compaction of the batch positions that take the dense path.
__global__ void __launch_bounds__(1024) dense_list_kernel(DenseParams p) {
    __shared__ int wsum[32];
    __shared__ int base_s;
    int* ctrl = (int*)(p.ws + p.L.ctrl);
    int* list = (int*)(p.ws + p.L.list);
    int* flag = (int*)(p.ws + p.L.flag);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    for (int b0 = 0; b0 < p.B; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        bool take = false;
        if (b < p.B && p.mode != 2) {
            const long long q = p.inst_index ? (long long)p.inst_index[b] : (long long)b;
            if (q >= 0 && q < p.n_packed) {           // (out-of-range indices are reported by the general kernel)
                take = dense_qualifies(p.nvalid, p.ngen, p.nsingc, q, p.force, p.d);
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, take);
        if (lane == 0) wsum[warp] = __popc(m);
        __syncthreads();
        int off = base_s;
        for (int w = 0; w < warp; ++w) off += wsum[w];
        if (take) list[off + __popc(m & ((1u << lane) - 1u))] = b;
        if (b < p.B) flag[b] = take ? 1 : 0;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 32; ++w) t += wsum[w]; base_s += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { ctrl[0] = base_s; ctrl[1] = 0; ctrl[2] = 0; ctrl[3] = 0; }
    if (threadIdx.x < 16) ((unsigned long long*)(ctrl + 16))[threadIdx.x] = 0ull;       // phase clocks of profile builds
}

cudaError_t launch_dense_list(const DenseParams& p, cudaStream_t stream) {
    dense_list_kernel<<<1, 1024, 0, stream>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------ prep: TF32 split, b = A c, row 1-norms
// PLANES = false (calls with a Gram cache): the same loop without the plane stores, so b and ||a_i||_1 are bit-identical.

template <class TIO, bool PLANES>
__global__ void __launch_bounds__(256) dense_prep_kernel(DenseParams p) {
    const int* ctrl = (const int*)(p.ws + p.L.ctrl);
    const int* list = (const int*)(p.ws + p.L.list);
    const int m_pad = (int)p.L.m_pad, d_pad = (int)p.L.d_pad;
    const int chunks = m_pad / 8;
    const int s = blockIdx.x / chunks;
    const int j = p.round * (int)p.L.n_slots + s;
    if (j >= ctrl[0]) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) ((int*)(p.ws + p.L.ctrl))[1] = 0;       // work counter of this round's solve kernel
    const int v = (blockIdx.x - s * chunks) * 8 + warp;
    const int b = list[j];
    const size_t q = p.inst_index ? (size_t)p.inst_index[b] : (size_t)b;
    const int ng = p.ngen[q];
    if (v >= ((ng + 127) & ~127)) return;
    float* hi = (float*)(p.ws + p.L.planes) + ((size_t)s * 2 * m_pad + v) * d_pad;
    float* lo = hi + (size_t)m_pad * d_pad;
    const bool live = v < ng;
    const float* src = live ? p.A + ((size_t)q * p.m_max + (size_t)p.gen[q * p.m_max + v].x) * p.d : nullptr;
    const TIO* pred = (const TIO*)p.pred + (size_t)b * p.d;
    double dot = 0.0;
    float l1 = 0.f;
    for (int k0 = 0; k0 < d_pad; k0 += 128) {
        float x[4]; TIO c[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + u * 32 + lane;
            const bool in = live && k < p.d;
            x[u] = in ? __ldg(src + k) : 0.f;
            c[u] = in ? pred[k] : (TIO)0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + u * 32 + lane;
            if (k < d_pad) {
                if constexpr (PLANES) {
                    const float h = tf32_rn(x[u]);
                    hi[k] = h;
                    lo[k] = tf32_rn(x[u] - h);
                }
                dot += (double)x[u] * (double)(TIO)(p.sign * (double)c[u]);
                l1 += fabsf(x[u]);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { dot += __shfl_xor_sync(0xffffffffu, dot, o); l1 += __shfl_xor_sync(0xffffffffu, l1, o); }
    if (lane == 0) {
        ((double*)(p.ws + p.L.bvec))[(size_t)s * m_pad + v] = dot;
        ((float*)(p.ws + p.L.l1))[(size_t)s * m_pad + v] = l1;
    }
}

cudaError_t launch_dense_prep(const DenseParams& p, cudaStream_t stream) {
    const unsigned grid = (unsigned)(p.L.n_slots * (p.L.m_pad / 8));
    if (p.gram) {
        if (p.io_f32) dense_prep_kernel<float, false><<<grid, 256, 0, stream>>>(p);
        else dense_prep_kernel<double, false><<<grid, 256, 0, stream>>>(p);
    } else {
        if (p.io_f32) dense_prep_kernel<float, true><<<grid, 256, 0, stream>>>(p);
        else dense_prep_kernel<double, true><<<grid, 256, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------ Gram cache of a resident dataset (dense.cuh)
// One CTA: ordered compaction of the pack instances the dense path could take (dense_qualifies with force semantics).
__global__ void __launch_bounds__(1024) gram_cache_map_kernel(const int* nvalid, const int* ngen, const int* nsingc, int N,
                                                              int m_pad, int* map, int* n_cached, int* header) {
    __shared__ int wsum[32];
    __shared__ int base_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    for (int q0 = 0; q0 < N; q0 += 1024) {
        const int q = q0 + threadIdx.x;
        const bool take = q < N && dense_qualifies(nvalid, ngen, nsingc, q, 1, 0);
        const unsigned m = __ballot_sync(0xffffffffu, take);
        if (lane == 0) wsum[warp] = __popc(m);
        __syncthreads();
        int off = base_s;
        for (int w = 0; w < warp; ++w) off += wsum[w];
        if (map && q < N) map[q] = take ? off + __popc(m & ((1u << lane) - 1u)) : -1;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 32; ++w) t += wsum[w]; base_s += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (n_cached) *n_cached = base_s;
        if (header) { header[0] = 0; header[1] = base_s; header[2] = m_pad; header[3] = N; }
    }
}

cudaError_t launch_gram_cache_map(const int* nvalid, const int* ngen, const int* nsingc, int N, int m_pad, int* map,
                                  int* n_cached, int* header, cudaStream_t stream) {
    gram_cache_map_kernel<<<1, 1024, 0, stream>>>(nvalid, ngen, nsingc, N, m_pad, map, n_cached, header);
    return cudaGetLastError();
}

// One warp per row of a slot, grid as dense_prep_kernel: the instance's leading square of G~ is copied, the rest of the
// cache slot is zeroed (those entries of a DenseLayout::G slot are never written).
__global__ void __launch_bounds__(256) gram_cache_copy_kernel(DenseParams p, char* cache, long long cap) {
    const int* ctrl = (const int*)(p.ws + p.L.ctrl);
    const int* list = (const int*)(p.ws + p.L.list);
    const int m_pad = (int)p.L.m_pad;
    const int chunks = m_pad / 8;
    const int s = blockIdx.x / chunks;
    const int j = p.round * (int)p.L.n_slots + s;
    if (j >= ctrl[0]) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int row = (blockIdx.x - s * chunks) * 8 + warp;
    const int q = list[j];
    const int slot = ((const int*)(cache + 16))[q];
    if (slot < 0 || slot >= cap) return;
    const int lim = (p.ngen[q] + 127) & ~127;
    const float4* src = (const float4*)((const float*)(p.ws + p.L.G) + ((size_t)s * m_pad + row) * m_pad);
    float4* dst = (float4*)((float*)(cache + gram_cache_base(p.n_packed)) + ((size_t)slot * m_pad + row) * m_pad);
    for (int c = lane; c < m_pad / 4; c += 32)
        dst[c] = (row < lim && 4 * c < lim) ? src[c] : make_float4(0.f, 0.f, 0.f, 0.f);
}

cudaError_t launch_gram_cache_copy(const DenseParams& p, char* cache, long long cap, cudaStream_t stream) {
    const unsigned grid = (unsigned)(p.L.n_slots * (p.L.m_pad / 8));
    gram_cache_copy_kernel<<<grid, 256, 0, stream>>>(p, cache, cap);
    return cudaGetLastError();
}

__global__ void gram_cache_seal_kernel(int* header, long long cap) {
    if (header[1] <= cap) header[0] = 1;
}

cudaError_t launch_gram_cache_seal(char* cache, long long cap, cudaStream_t stream) {
    gram_cache_seal_kernel<<<1, 1, 0, stream>>>((int*)cache, cap);
    return cudaGetLastError();
}


constexpr int kGramThreads = 192;
constexpr int kGramStages = 2;
constexpr int kTileA = 128 * 128;                       // bytes: 128 rows x 32 float32
constexpr int kStageBytes = 2 * kTileA + 2 * 2 * kTileA;   // A hi, A lo, B hi (256 rows), B lo (256 rows)
constexpr int kGramSmem = kGramStages * kStageBytes + 1024;

struct GramItem { int s, I, J, w, valid; };

// item -> (slot, tile): tiles are enumerated per instance over the upper block triangle, 128 x (128|256)
__device__ __forceinline__ GramItem gram_item(const DenseParams& p, const int* list, int item, int tmax) {
    GramItem g;
    g.s = item / tmax;
    int t = item - g.s * tmax;
    const int b = list[p.round * (int)p.L.n_slots + g.s];
    const size_t q = p.inst_index ? (size_t)p.inst_index[b] : (size_t)b;
    const int nI = (p.ngen[q] + 127) >> 7;
    g.valid = 0; g.I = 0; g.J = 0; g.w = 1;
    for (int I = 0; I < nI; ++I) {
        const int cnt = (nI - I + 1) >> 1;
        if (t < cnt) { g.I = I; g.J = I + 2 * t; g.w = nI - g.J >= 2 ? 2 : 1; g.valid = 1; break; }
        t -= cnt;
    }
    return g;
}

__global__ void __launch_bounds__(kGramThreads, 1) dense_gram_kernel(const __grid_constant__ CUtensorMap tmap, DenseParams p) {
    extern __shared__ uint8_t gram_smem_raw[];
    __shared__ uint64_t full_bar[kGramStages], empty_bar[kGramStages], tfull_bar[2], tempty_bar[2];
    __shared__ uint32_t tmem_base_s;
    const int* ctrl = (const int*)(p.ws + p.L.ctrl);
    const int* list = (const int*)(p.ws + p.L.list);
    const int n_slots = (int)p.L.n_slots, m_pad = (int)p.L.m_pad;
    int n_round = ctrl[0] - p.round * n_slots;
    n_round = n_round < n_slots ? n_round : n_slots;
    const int tmax = dense_tiles(m_pad >> 7);
    const int n_items = n_round * tmax;
    if ((int)blockIdx.x >= n_items) return;                       // nothing to do (before any allocation)
    uint8_t* smem = (uint8_t*)(((uintptr_t)gram_smem_raw + 1023) & ~(uintptr_t)1023);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kGramStages; ++i) { tc::mbar_init(&full_bar[i], 1); tc::mbar_init(&empty_bar[i], 1); }
        for (int i = 0; i < 2; ++i) { tc::mbar_init(&tfull_bar[i], 1); tc::mbar_init(&tempty_bar[i], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tc::smem_u32(&tmem_base_s)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc::fence_before();
    __syncthreads();
    tc::fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 0) {
        // ---------------- TMA producer
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
                const GramItem g = gram_item(p, list, item, tmax);
                if (!g.valid) continue;
                const int rowB = (g.s * 2) * m_pad + g.J * 128;
                const int rowA = (g.s * 2) * m_pad + g.I * 128;
                const bool diag = g.J == g.I;
                const uint32_t bytes = (uint32_t)((diag ? 0 : 2 * kTileA) + 2 * g.w * kTileA);
                for (int ks = 0; ks < p.nk; ++ks) {
                    tc::mbar_wait(&empty_bar[stage], phase ^ 1u);
                    tc::mbar_expect_tx(&full_bar[stage], bytes);
                    uint8_t* base = smem + stage * kStageBytes;
                    const int x = ks * 32;
                    if (!diag) {
                        tc::tma_load_2d(base, &tmap, x, rowA, &full_bar[stage]);
                        tc::tma_load_2d(base + kTileA, &tmap, x, rowA + m_pad, &full_bar[stage]);
                    }
                    tc::tma_load_2d(base + 2 * kTileA, &tmap, x, rowB, &full_bar[stage]);
                    tc::tma_load_2d(base + 4 * kTileA, &tmap, x, rowB + m_pad, &full_bar[stage]);
                    if (g.w == 2) {
                        tc::tma_load_2d(base + 3 * kTileA, &tmap, x, rowB + 128, &full_bar[stage]);
                        tc::tma_load_2d(base + 5 * kTileA, &tmap, x, rowB + m_pad + 128, &full_bar[stage]);
                    }
                    if (++stage == kGramStages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer
        int stage = 0; uint32_t phase = 0;
        int acc = 0; uint32_t accphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            const GramItem g = gram_item(p, list, item, tmax);
            if (!g.valid) continue;
            const bool diag = g.J == g.I;
            const uint32_t idesc = tc::instr_desc(g.w * 128);
            tc::mbar_wait(&tempty_bar[acc], accphase ^ 1u);
            tc::fence_after();
            for (int ks = 0; ks < p.nk; ++ks) {
                tc::mbar_wait(&full_bar[stage], phase);
                tc::fence_after();
                if (lane == 0) {
                    const uint32_t base = tc::smem_u32(smem + stage * kStageBytes);
                    const uint32_t bHi = base + 2 * kTileA, bLo = base + 4 * kTileA;
                    const uint32_t aHi = diag ? bHi : base, aLo = diag ? bLo : base + kTileA;
                    const uint32_t d = tmem_base + (uint32_t)acc * 256u;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint64_t dAh = tc::smem_desc(aHi + kk * 32), dAl = tc::smem_desc(aLo + kk * 32);
                        const uint64_t dBh = tc::smem_desc(bHi + kk * 32), dBl = tc::smem_desc(bLo + kk * 32);
                        tc::mma_tf32(d, dAl, dBh, idesc, (ks | kk) != 0 ? 1u : 0u);
                        tc::mma_tf32(d, dAh, dBl, idesc, 1u);
                        tc::mma_tf32(d, dAh, dBh, idesc, 1u);
                    }
                    tc::mma_commit(&empty_bar[stage]);
                    if (ks == p.nk - 1) tc::mma_commit(&tfull_bar[acc]);
                }
                __syncwarp();
                if (++stage == kGramStages) { stage = 0; phase ^= 1u; }
            }
            if (++acc == 2) { acc = 0; accphase ^= 1u; }
        }
    } else {
        // ---------------- epilogue: TMEM -> registers -> G (both orientations)
        const int qg = warp & 3;                       // this warp's TMEM lane group
        int acc = 0; uint32_t accphase = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            const GramItem g = gram_item(p, list, item, tmax);
            if (!g.valid) continue;
            float* G = (float*)(p.ws + p.L.G) + (size_t)g.s * m_pad * m_pad;
            tc::mbar_wait(&tfull_bar[acc], accphase);
            tc::fence_after();
            const int rl = qg * 32 + lane;             // row inside the 128-row block
            const int r = g.I * 128 + rl;
            for (int cc = 0; cc < g.w * 4; ++cc) {
                uint32_t v[32];
                tc::tmem_ld32(tmem_base + (uint32_t)acc * 256u + (uint32_t)cc * 32u + ((uint32_t)(qg * 32) << 16), v);
                const int col0 = g.J * 128 + cc * 32;
                const bool dblk = (g.J + (cc >> 2)) == g.I;      // this 128-column block is the diagonal block
                const int cl0 = (cc & 3) * 32;                   // first column inside its block
                if (!dblk) {
                    float4* dst = reinterpret_cast<float4*>(G + (size_t)r * m_pad + col0);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                             __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
#pragma unroll
                    for (int j = 0; j < 32; ++j) G[(size_t)(col0 + j) * m_pad + r] = __uint_as_float(v[j]);
                } else {
                    // diagonal block: the lower triangle (column <= row) is written and mirrored, so G is exactly symmetric
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        if (cl0 + j <= rl) {
                            const float x = __uint_as_float(v[j]);
                            G[(size_t)r * m_pad + col0 + j] = x;
                            if (cl0 + j < rl) G[(size_t)(col0 + j) * m_pad + r] = x;
                        }
                    }
                }
            }
            tc::fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&tempty_bar[acc]);
            if (++acc == 2) { acc = 0; accphase ^= 1u; }
        }
    }
    tc::fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ------------------------------------------------------------------ host side
namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qr) != cudaSuccess || !ptr) {
        (void)cudaGetLastError();
        return nullptr;
    }
    fn = (EncodeTiledFn)ptr;
    return fn;
}
}  // namespace

cudaError_t launch_dense_gram(const DenseParams& p, cudaStream_t stream) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) { g_dense_err = "cuTensorMapEncodeTiled is not available from the driver"; return cudaErrorNotSupported; }
    alignas(64) CUtensorMap tmap;
    const cuuint64_t dims[2] = {(cuuint64_t)p.L.d_pad, (cuuint64_t)(p.L.n_slots * 2 * p.L.m_pad)};
    const cuuint64_t strides[1] = {(cuuint64_t)p.L.d_pad * 4};
    const cuuint32_t box[2] = {32, 128};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)(p.ws + p.L.planes), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char buf[160];
        snprintf(buf, sizeof(buf), "cuTensorMapEncodeTiled failed with CUresult %d (d_pad %lld, rows %lld)", (int)r,
                 (long long)p.L.d_pad, (long long)(p.L.n_slots * 2 * p.L.m_pad));
        g_dense_err = buf;
        return cudaErrorInvalidValue;
    }
    cudaError_t e = cudaFuncSetAttribute(dense_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGramSmem);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long items = (long long)p.L.n_slots * dense_tiles((int)(p.L.m_pad >> 7));
    const unsigned grid = (unsigned)(items < sms ? items : sms);
    dense_gram_kernel<<<grid, kGramThreads, kGramSmem, stream>>>(tmap, p);
    return cudaGetLastError();
}

}  // namespace cave
