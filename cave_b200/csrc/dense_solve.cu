// Dense regime, kernel 4: one CTA per instance solves  min_{lam >= 0} 1/2 ||A^T lam - c||^2  in Gram space.
//
// Phase 1 (Gram space, reads only G~ and b): Bertsekas' two-metric projected Newton on q(lam) = 1/2 lam^T G~ lam - b^T lam.
//   Free set F = variables that are not epsilon-binding; Newton system (G~_FF + reg I) x = g_F by a blocked left-looking
//   float32 Cholesky in the instance's global workspace (register-tiled 8 x 8 FFMA kernel fed from shared memory, 64-column
//   block columns, 32 x 32 diagonal blocks factored in registers by one warp), Armijo search along the projection arc.
//   The gradient of the accepted trial point is the G~ matvec that evaluated it.  Stops at 1e-6 of the KKT scale: G~
//   (3xTF32) is not more accurate than that.
// Phase 2 (anchors the result to A, float64): the same iteration with the TRUE gradient g = A (A^T lam - c), i.e. two passes
//   over the rows of A per step, and the Cholesky factor of phase 1 as the metric (refactored only if F changes).  Each
//   step contracts the error by about cond(G_FF) * 1e-6, so one or two steps reach the float64 KKT tolerance that the
//   Lawson-Hanson path and scipy.optimize.nnls (src/cave.py:307) reach.
// An instance that does not converge (e.g. m > d with the cone the whole space: G singular, the solution not unique)
// is handed back: its flag is cleared and the Lawson-Hanson path of the general solve kernel, launched afterwards, takes it.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include "dense.cuh"
#include "tc05.cuh"
#include "solver_core.cuh"

namespace cave {

constexpr int kDT = 512;            // threads per CTA
constexpr int kRC = 512;            // rows per chunk of the block-column update (one row per thread when staging)
constexpr int kNB = 64;             // block-column width
constexpr int kKS = 16;             // k-slab of the update

struct DenseSmem {
    double *lam, *lamt, *g, *gt, *dir, *bb;
    double *lamp;                   // the trial point, 32 x 4 transposed inside every 128-block: conflict-free reads in the matvec
    int *fl, *flp;
    int *arow, *sup;                // row of A behind every variable; support list of the point being evaluated
    float *As, *Bs, *D, *Dt, *invd;
    float *xs;                      // [m_pad] float32 right-hand side / solution of the triangular solves
    unsigned long long* prof;       // phase clocks (profile builds only, else nullptr)
};
#ifdef CAVE_DENSE_PROFILE
#define CPROF_BEGIN() long long cprof_t = clock64()
#define CPROF(ph) do { __syncthreads(); if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd(S.prof + (ph), (unsigned long long)(t_ - cprof_t)); cprof_t = t_; } } while (0)
#else
#define CPROF_BEGIN() do {} while (0)
#define CPROF(ph) do {} while (0)
#endif

// tensor-core update: operand planes of one 32-wide k-slab, K-major with the 128-byte swizzle of the UMMA descriptors:
// A hi / lo (256 rows x 128 bytes each), B hi / lo (64 rows)
#ifndef CAVE_TC_INLINE
#define CAVE_TC_INLINE __noinline__
#endif
#ifndef CAVE_TC_MASKSPLIT
#define CAVE_TC_MASKSPLIT 0
#endif
#ifndef CAVE_TC_KMAJOR
#define CAVE_TC_KMAJOR 0
#endif
#ifndef CAVE_TC_PD
#define CAVE_TC_PD 1
#endif
#ifndef CAVE_TC_L2AHEAD
#define CAVE_TC_L2AHEAD 3
#endif
constexpr int kTcL2Ahead = CAVE_TC_L2AHEAD;     // items whose operands are pulled into the L2 ahead of the register prefetch
// State of the tensor-core update in static shared memory (no kernel-lifetime registers: the solver's matvec loops sit at the
// register limit): mbarrier of the tcgen05.commit, its phase, TMEM base address (256 columns).
__shared__ uint64_t tc_bar_s;
__shared__ uint32_t tc_phase_s, tmem_base_s;
constexpr int kTcRows = 256;
constexpr int kTcA = kTcRows * 128;
constexpr int kTcB = kNB * 128;
constexpr int kTcBytes = 2 * kTcA + 2 * kTcB;
constexpr int kStageSimt = (kKS * kRC + kKS * kNB) * 4;      // As, Bs of the FFMA update

__host__ __device__ inline size_t dense_solve_smem(int64_t m_pad, bool tc) {
    size_t o = 0;
    o += 7 * (size_t)m_pad * 8;                 // lam lamt g gt dir bb lamp
    o += 4 * (size_t)m_pad * 4;                 // free lists, arow, sup
    o += (size_t)m_pad * 4;                     // xs
    o += tc ? (size_t)kTcBytes + 1024 : (size_t)kStageSimt;     // As, Bs / the tensor-core operand planes over them
    o += (size_t)kNB * (kNB + 1) * 4 + (size_t)kNB * kNB * 4 + kNB * 4; // D, Dt, invd
    return o + 256;
}

// Factor the kNB x kNB diagonal block held in D (row stride kNB + 1, lower triangle valid, zero above it) in place; nb valid
// rows.  Right-looking in panels of 8 columns: warp 0 factors a panel entirely in registers (rows lane and lane + 32, the
// pivot row broadcast by shuffles, rsqrt pivots), then all warps apply the rank-8 update to the trailing block — two CTA
// barriers per panel and no 32-step dependent chain.  Entries above the diagonal collect garbage in the registers; they are
// never stored.  All threads call; ends with a barrier.  invd[c] = 1 / L[c][c].
__device__ void factor_diag(float* D, float* invd, int nb, float floor_, int tid) {
    constexpr int LD = kNB + 1, PB = 8;
    const int lane = tid & 31, warp = tid >> 5;
    // rows / columns >= nb: identity, so the 64-wide code below needs no bounds
    for (int t = tid; t < kNB * kNB; t += kDT) {
        const int i = t / kNB, j = t - i * kNB;
        if (i >= nb || j >= nb) D[i * LD + j] = i == j ? 1.0f : 0.0f;
    }
    __syncthreads();
    for (int j0 = 0; j0 < kNB; j0 += PB) {
        if (warp == 0) {
            const bool hi = j0 >= 32;                   // a panel never straddles row 32: its pivot rows sit in one register set
            float a0[PB], a1[PB];                       // rows lane and lane + 32
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                a0[c] = lane >= j0 ? D[lane * LD + j0 + c] : 0.0f;
                a1[c] = D[(lane + 32) * LD + j0 + c];
            }
#pragma unroll
            for (int jj = 0; jj < PB; ++jj) {
                const int j = j0 + jj;
                const float piv = __shfl_sync(0xffffffffu, hi ? a1[jj] : a0[jj], j & 31);
                const float pv = piv > floor_ ? piv : floor_;
                float inv = rsqrtf(pv);
                inv = inv * (1.5f - 0.5f * pv * inv * inv);         // one Newton step: full float32 accuracy
                const float l = pv * inv;
                if (lane == 0) invd[j] = inv;
                a0[jj] = (lane == j) ? l : a0[jj] * inv;
                a1[jj] = (lane + 32 == j) ? l : a1[jj] * inv;
#pragma unroll
                for (int c = jj + 1; c < PB; ++c) {
                    const float t = __shfl_sync(0xffffffffu, hi ? a1[jj] : a0[jj], (j0 + c) & 31);   // L[j0 + c][j]
                    a0[c] = fmaf(-a0[jj], t, a0[c]);
                    a1[c] = fmaf(-a1[jj], t, a1[c]);
                }
            }
#pragma unroll
            for (int c = 0; c < PB; ++c) {
                if (lane >= j0 + c) D[lane * LD + j0 + c] = a0[c];
                if (lane + 32 >= j0 + c) D[(lane + 32) * LD + j0 + c] = a1[c];
            }
        }
        __syncthreads();
        const int t0 = j0 + PB, n = kNB - t0;           // trailing block: D[i][k] -= sum_c L[i][j0 + c] L[k][j0 + c], k <= i
        for (int t = tid; t < n * n; t += kDT) {
            const int i = t0 + t / n, k = t0 + t % n;
            if (k <= i) {
                float acc = D[i * LD + k];
#pragma unroll
                for (int c = 0; c < PB; ++c) acc = fmaf(-D[i * LD + j0 + c], D[k * LD + j0 + c], acc);
                D[i * LD + k] = acc;
            }
        }
        __syncthreads();
    }
}

// One chunk of the block-column update of the left-looking Cholesky: rows [r0, r0 + 64 RM) x columns [j0, j0 + 64) of W get
// -= L[rows, 0:j0] L[j0:j0+64, 0:j0]^T.  512 threads, each a micro-tile of RM rows x 8 columns; the k-slabs of both operands
// go through shared memory k-major (one row per staging thread, next slab prefetched into registers).  RM = 8 interleaves two
// groups of four rows per thread so that the 128-bit operand loads of a quarter-warp fall into distinct banks.
template <int RM>
__device__ __forceinline__ void chol_update_chunk(float* __restrict__ W, int ldw, int nf, int j0, int r0, const DenseSmem& S, int tid) {
    constexpr int ROWS = 64 * RM;
    // warp tile = 8 row groups x 4 column groups (not 32 x 1): the four 128-bit operand loads of a k-step then touch 128 + 128 +
    // 64 + 64 distinct bytes per warp (lanes that share an address are served by one multicast) instead of 2 x 512 + 2 x 16
    const int warp_ = tid >> 5, lane_ = tid & 31;
    const int tr = (warp_ & 7) * 8 + (lane_ & 7), tcg = (warp_ >> 3) * 4 + (lane_ >> 3);
    float acc[RM][8];
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
    // staging: the A operand one row per thread (16 k-values), the 64 x 16 B operand two values per thread (all threads), so
    // that the prefetch costs 18 registers and the k-loop can keep the next step's operands in flight
    const bool stage_a = tid < ROWS;
    const int myrow = r0 + tid < nf ? r0 + tid : nf - 1;                // clamped
    const int bq_row = tid >> 3, bq_k = (tid & 7) * 2;
    const int mybrow = j0 + bq_row < nf ? j0 + bq_row : nf - 1;
    const float* arow = W + (size_t)myrow * ldw;
    const float* brow = W + (size_t)mybrow * ldw + bq_k;
    // Prefetch ring of PD k-slabs in registers: a slab's loads have PD compute phases to arrive.  The loads come from L2 / HBM
    // (~4000 cycles under load), a compute phase is 4096 / 2048 / 1024 / 512 FFMA-cycles for RM = 8 / 4 / 2 / 1: with a
    // distance of one slab the short tiles ran at the pace of the memory latency, not of the arithmetic.
    constexpr int PD = RM == 8 ? 1 : (RM == 4 ? 2 : 4);
    float4 pa[PD][4]; float2 pb[PD];
#pragma unroll
    for (int sl = 0; sl < PD; ++sl) {
        if (sl * kKS < j0) {
#pragma unroll
            for (int u = 0; u < 4; ++u) pa[sl][u] = stage_a ? *reinterpret_cast<const float4*>(arow + sl * kKS + u * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            pb[sl] = *reinterpret_cast<const float2*>(brow + sl * kKS);
        }
    }
    auto load_ops = [&](int k, float (&av)[RM], float (&bv)[8]) {
        if (RM == 8) {
            const float4 a0 = *reinterpret_cast<const float4*>(S.As + k * kRC + tr * 4);
            const float4 a1 = *reinterpret_cast<const float4*>(S.As + k * kRC + 256 + tr * 4);
            av[0] = a0.x; av[1 % RM] = a0.y; av[2 % RM] = a0.z; av[3 % RM] = a0.w;
            av[4 % RM] = a1.x; av[5 % RM] = a1.y; av[6 % RM] = a1.z; av[7 % RM] = a1.w;
        } else if (RM == 4) {
            const float4 a0 = *reinterpret_cast<const float4*>(S.As + k * kRC + tr * 4);
            av[0] = a0.x; av[1 % RM] = a0.y; av[2 % RM] = a0.z; av[3 % RM] = a0.w;
        } else if (RM == 2) {
            const float2 a0 = *reinterpret_cast<const float2*>(S.As + k * kRC + tr * 2);
            av[0] = a0.x; av[1 % RM] = a0.y;
        } else {
            av[0] = S.As[k * kRC + tr];
        }
        const float4 b0 = *reinterpret_cast<const float4*>(S.Bs + k * kNB + tcg * 8);
        const float4 b1 = *reinterpret_cast<const float4*>(S.Bs + k * kNB + tcg * 8 + 4);
        bv[0] = b0.x; bv[1] = b0.y; bv[2] = b0.z; bv[3] = b0.w; bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
    };
    for (int p0 = 0; p0 < j0; p0 += kKS * PD) {
#pragma unroll
        for (int sl = 0; sl < PD; ++sl) {
            const int p = p0 + sl * kKS;
            if (p < j0) {                       // (uniform across the CTA)
                __syncthreads();                // previous slab consumed
                if (stage_a) {
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        S.As[(u * 4 + 0) * kRC + tid] = pa[sl][u].x; S.As[(u * 4 + 1) * kRC + tid] = pa[sl][u].y;
                        S.As[(u * 4 + 2) * kRC + tid] = pa[sl][u].z; S.As[(u * 4 + 3) * kRC + tid] = pa[sl][u].w;
                    }
                }
                S.Bs[bq_k * kNB + bq_row] = pb[sl].x; S.Bs[(bq_k + 1) * kNB + bq_row] = pb[sl].y;
                __syncthreads();
                if (p + PD * kKS < j0) {
                    if (stage_a) {
#pragma unroll
                        for (int u = 0; u < 4; ++u) pa[sl][u] = *reinterpret_cast<const float4*>(arow + p + PD * kKS + u * 4);
                    }
                    pb[sl] = *reinterpret_cast<const float2*>(brow + p + PD * kKS);
                }
                float av[2][RM], bv[2][8];
                load_ops(0, av[0], bv[0]);
#pragma unroll
                for (int k = 0; k < kKS; ++k) {
                    if (k + 1 < kKS) load_ops(k + 1, av[(k + 1) & 1], bv[(k + 1) & 1]);       // next step's operands while this one multiplies
#pragma unroll
                    for (int i = 0; i < RM; ++i)
#pragma unroll
                        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[k & 1][i], bv[k & 1][j], acc[i][j]);
                }
            }
        }
    }
    // ---- W[r, j0 + c] -= acc
#pragma unroll
    for (int i = 0; i < RM; ++i) {
        const int rl = RM == 8 ? (i < 4 ? tr * 4 + i : 256 + tr * 4 + (i - 4)) : tr * RM + i;
        const int r = r0 + rl;
        if (r < nf) {
            float* w = W + (size_t)r * ldw + j0 + tcg * 8;
            float4 w0 = *reinterpret_cast<float4*>(w), w1 = *reinterpret_cast<float4*>(w + 4);
            w0.x -= acc[i][0]; w0.y -= acc[i][1]; w0.z -= acc[i][2]; w0.w -= acc[i][3];
            w1.x -= acc[i][4]; w1.y -= acc[i][5]; w1.z -= acc[i][6]; w1.w -= acc[i][7];
            *reinterpret_cast<float4*>(w) = w0; *reinterpret_cast<float4*>(w + 4) = w1;
        }
    }
}

// The same update on the tensor cores (3 x TF32, float32 accumulation in TMEM): rows [r0, r0 + rows), rows <= 512, as up to
// four 128-row tiles (two per 256-row half; the halves share the staging planes and follow each other in one pipeline).  Per 32-wide k-slab all threads split their 16-byte pieces of L[rows, k..k+32) and L[j0.., k..k+32) into
// hi / lo TF32 planes, written K-major with the 128-byte swizzle the UMMA descriptor expects (16-byte chunk index XOR row & 7;
// a quarter-warp writes one full 128-byte row: conflict-free); one thread then issues 4 k-steps x (lo*hi + hi*lo + hi*hi) per
// tile and commits to the mbarrier; the next slab's global loads are in flight meanwhile and its stores wait for the commit.
// Epilogue: every warp reads its TMEM lane quarter (tcgen05.ld 32x32b.x32) and subtracts from W.  All threads call.
__device__ __forceinline__ void tc_store_split(unsigned char* hi, unsigned char* lo, int row, int chunk, const float4& v) {
    const uint32_t off = (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
    float4 h, l;
#if CAVE_TC_MASKSPLIT
    // hi = the upper 19 bits (truncation), lo = x - hi exactly; the tensor core reads only the TF32 bits of either, i.e. lo is
    // truncated to 11 significant bits by the hardware: 2 instructions per value instead of ~10 for two cvt.rna.tf32
    h.x = __uint_as_float(__float_as_uint(v.x) & 0xffffe000u); h.y = __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
    h.z = __uint_as_float(__float_as_uint(v.z) & 0xffffe000u); h.w = __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
    l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
#else
    h.x = tf32_rn(v.x); h.y = tf32_rn(v.y); h.z = tf32_rn(v.z); h.w = tf32_rn(v.w);
    l.x = tf32_rn(v.x - h.x); l.y = tf32_rn(v.y - h.y); l.z = tf32_rn(v.z - h.z); l.w = tf32_rn(v.w - h.w);
#endif
    *reinterpret_cast<float4*>(hi + off) = h;
    *reinterpret_cast<float4*>(lo + off) = l;
}

// Not inlined: its registers then do not compete with the solver's live state.
__device__ CAVE_TC_INLINE void chol_update_tc(float* __restrict__ W, int ldw, int nf, int j0, int r0, int rows, float* stage, int tid) {
    unsigned char* tcbuf = (unsigned char*)(((uintptr_t)stage + 1023) & ~(uintptr_t)1023);
    uint64_t* tc_bar = &tc_bar_s;
    uint32_t phase = tc_phase_s;
    const uint32_t tmem = tmem_base_s;
    // Work items = (256-row half, k-slab).  The factors of the instances in flight (148 x 1.25 MB) do not fit the L2 and a load
    // from HBM takes ~4000 cycles under load while an item computes for ~1000: operands are pulled into the L2 kTcL2Ahead items
    // ahead (prefetch.global.L2, no registers) and into registers PD items ahead.
    constexpr int PD = CAVE_TC_PD;
    const int nslab = j0 >> 5;
    const int nh = (rows + kTcRows - 1) / kTcRows;
    const int nitem = nh * nslab;
    const int srow = tid >> 3, chunk = tid & 7;
    unsigned char* Ah = tcbuf; unsigned char* Al = Ah + kTcA; unsigned char* Bh = Al + kTcA; unsigned char* Bl = Bh + kTcB;
    const int rb = j0 + srow < nf ? j0 + srow : nf - 1;
    const float* bsrc = W + (size_t)rb * ldw + chunk * 4;
    const uint32_t idesc = tc::instr_desc(kNB);
    auto tiles_of = [&](int h) { const int rh = rows - h * kTcRows; return rh > 128 ? 2 : 1; };
    // item -> this thread's 16-byte pieces; pf: only an L2 prefetch (every 32-byte sector once: even chunks)
    auto fetch = [&](int it, float4 (&a)[4], float4& b, bool pf) {
        const int h = it >= nslab ? 1 : 0, s = it - h * nslab;
        const int na = tiles_of(h) * 2;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (u < na) {
                int r = r0 + h * kTcRows + srow + u * 64;
                r = r < nf ? r : nf - 1;                // clamped: finite operands, the rows are not stored
                const float* src = W + (size_t)r * ldw + chunk * 4 + s * 32;
                if (!pf) a[u] = *reinterpret_cast<const float4*>(src);
                else if (!(chunk & 1)) asm volatile("prefetch.global.L2 [%0];" ::"l"(src));
            }
        }
        if (!pf) b = *reinterpret_cast<const float4*>(bsrc + s * 32);
        else if (!(chunk & 1) && h == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(bsrc + s * 32));
    };
    float4 pa[PD][4], pb[PD];
#pragma unroll
    for (int sl = 0; sl < PD; ++sl)
        if (sl < nitem) fetch(sl, pa[sl], pb[sl], false);
    for (int it = PD; it < PD + kTcL2Ahead && it < nitem; ++it) fetch(it, pa[0], pb[0], true);
    for (int it0 = 0; it0 < nitem; it0 += PD) {
#pragma unroll
        for (int sl = 0; sl < PD; ++sl) {
            const int it = it0 + sl;
            if (it < nitem) {                                                   // (uniform across the CTA)
                const int h = it >= nslab ? 1 : 0, s = it - h * nslab;
                const int nt = tiles_of(h);
                if (it > 0) { tc::mbar_wait(tc_bar, phase); phase ^= 1u; }    // the MMAs of the previous item have read the planes
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (u < nt * 2) tc_store_split(Ah, Al, srow + u * 64, chunk, pa[sl][u]);
                tc_store_split(Bh, Bl, srow, chunk, pb[sl]);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncthreads();
                if (tid == 0) {
                    tc::fence_after();
                    const uint32_t aH = tc::smem_u32(Ah), aL = tc::smem_u32(Al), bH = tc::smem_u32(Bh), bL = tc::smem_u32(Bl);
#if CAVE_TC_KMAJOR
                    // k-step outermost: consecutive instructions alternate between the two tiles' accumulators
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint64_t dBh = tc::smem_desc(bH + kk * 32), dBl = tc::smem_desc(bL + kk * 32);
                        for (int t = 0; t < nt; ++t) {
                            const uint32_t dcol = tmem + (uint32_t)(h * 2 + t) * kNB;
                            const uint64_t dAh = tc::smem_desc(aH + t * 16384 + kk * 32), dAl = tc::smem_desc(aL + t * 16384 + kk * 32);
                            tc::mma_tf32(dcol, dAl, dBh, idesc, (s | kk) != 0 ? 1u : 0u);
                            tc::mma_tf32(dcol, dAh, dBl, idesc, 1u);
                            tc::mma_tf32(dcol, dAh, dBh, idesc, 1u);
                        }
                    }
#else
                    for (int t = 0; t < nt; ++t) {
                        const uint32_t dcol = tmem + (uint32_t)(h * 2 + t) * kNB;
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            const uint64_t dAh = tc::smem_desc(aH + t * 16384 + kk * 32), dAl = tc::smem_desc(aL + t * 16384 + kk * 32);
                            const uint64_t dBh = tc::smem_desc(bH + kk * 32), dBl = tc::smem_desc(bL + kk * 32);
                            tc::mma_tf32(dcol, dAl, dBh, idesc, (s | kk) != 0 ? 1u : 0u);
                            tc::mma_tf32(dcol, dAh, dBl, idesc, 1u);
                            tc::mma_tf32(dcol, dAh, dBh, idesc, 1u);
                        }
                    }
#endif
                    tc::mma_commit(tc_bar);
                }
                if (it + PD < nitem) fetch(it + PD, pa[sl], pb[sl], false);
                if (it + PD + kTcL2Ahead < nitem) fetch(it + PD + kTcL2Ahead, pa[sl], pb[sl], true);
            }
        }
    }
    // ---- W[r, j0 + c] -= acc: warp -> (tile, TMEM lane quarter, 32-column half); the first half's W values are loaded while the
    // last MMAs run (one half at a time: 32 + 32 registers)
    const int warp = tid >> 5, lane = tid & 31;
    const int tile = (warp >> 2) & 1, qd = warp & 3, ch = warp >> 3;
    const int rl = tile * 128 + qd * 32 + lane;
    float4 wv[8];
    auto load_w = [&](int h) {
        if (h * kTcRows + rl < rows) {
            const float* w = W + (size_t)(r0 + h * kTcRows + rl) * ldw + j0 + ch * 32;
#pragma unroll
            for (int j = 0; j < 8; ++j) wv[j] = *reinterpret_cast<const float4*>(w + 4 * j);
        }
    };
    load_w(0);
    tc::mbar_wait(tc_bar, phase); phase ^= 1u;
    tc::fence_after();
    for (int h = 0; h < nh; ++h) {
        if (h > 0) load_w(h);
        if (tile < tiles_of(h)) {                                               // (uniform across the warp)
            uint32_t v[32];
            tc::tmem_ld32(tmem + (uint32_t)((h * 2 + tile) * kNB + ch * 32) + ((uint32_t)(qd * 32) << 16), v);
            if (h * kTcRows + rl < rows) {
                float* w = W + (size_t)(r0 + h * kTcRows + rl) * ldw + j0 + ch * 32;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float4 x = wv[j];
                    x.x -= __uint_as_float(v[4 * j]); x.y -= __uint_as_float(v[4 * j + 1]);
                    x.z -= __uint_as_float(v[4 * j + 2]); x.w -= __uint_as_float(v[4 * j + 3]);
                    *reinterpret_cast<float4*>(w + 4 * j) = x;
                }
            }
        }
    }
    tc::fence_before();
    __syncthreads();
    if (tid == 0) tc_phase_s = phase;               // (read again after the barriers of the diagonal block / row solves)
}

// Blocked left-looking Cholesky of the nf x nf lower triangle in W (row stride ldw): W <- L.
template <bool TC>
__device__ void chol_blocked(float* __restrict__ W, int ldw, int nf, float floor_, const DenseSmem& S, int tid) {
    constexpr int LD = kNB + 1;
    CPROF_BEGIN();
    for (int j0 = 0; j0 < nf; j0 += kNB) {
        const int nb = nf - j0 < kNB ? nf - j0 : kNB;
        for (int r0 = j0; r0 < nf;) {
            const int rem = nf - r0;
            const int rows = rem > 256 ? 512 : (rem > 128 ? 256 : (rem > 64 ? 128 : 64));      // rows of this chunk
            if constexpr (TC) {
                if (j0 > 0)
                    chol_update_tc(W, ldw, nf, j0, r0, rows < nf - r0 ? rows : nf - r0, S.As, tid);
            } else if (j0 > 0) {
                if (rows == 512) chol_update_chunk<8>(W, ldw, nf, j0, r0, S, tid);
                else if (rows == 256) chol_update_chunk<4>(W, ldw, nf, j0, r0, S, tid);
                else if (rows == 128) chol_update_chunk<2>(W, ldw, nf, j0, r0, S, tid);
                else chol_update_chunk<1>(W, ldw, nf, j0, r0, S, tid);
            }
            __syncthreads();
            CPROF(13);
            if (r0 == j0) {
                // ---- diagonal block: factor in shared memory, write L_jj back; Dt = aligned copy for the row solves
                for (int t = tid; t < kNB * kNB; t += kDT) {
                    const int i = t / kNB, j = t - i * kNB;
                    S.D[i * LD + j] = (i < nb && j <= i) ? W[(size_t)(j0 + i) * ldw + j0 + j] : 0.0f;
                }
                __syncthreads();
                factor_diag(S.D, S.invd, nb, floor_, tid);
                for (int t = tid; t < kNB * kNB; t += kDT) {
                    const int i = t / kNB, j = t - i * kNB;
                    const float v = S.D[i * LD + j];
                    S.Dt[t] = j < i ? v : 0.0f;
                    if (i < nb && j <= i) W[(size_t)(j0 + i) * ldw + j0 + j] = v;
                }
                __syncthreads();
                CPROF(14);
            }
            // ---- rows below the diagonal block: x <- x L_jj^-T, one row per thread
            {
                const int r = r0 + tid;
                if (tid < rows && r >= j0 + kNB && r < nf) {
                    float* w = W + (size_t)r * ldw + j0;
                    float x[kNB];
#pragma unroll
                    for (int u = 0; u < kNB / 4; ++u) {
                        const float4 v = *reinterpret_cast<const float4*>(w + u * 4);
                        x[u * 4] = v.x; x[u * 4 + 1] = v.y; x[u * 4 + 2] = v.z; x[u * 4 + 3] = v.w;
                    }
#pragma unroll
                    for (int c = 0; c < kNB; ++c) {
                        float s = x[c];
#pragma unroll
                        for (int q4 = 0; q4 < (c + 3) / 4; ++q4) {      // Dt is zero on and above the diagonal
                            const float4 l4 = *reinterpret_cast<const float4*>(S.Dt + c * kNB + q4 * 4);
                            s = fmaf(-x[q4 * 4], l4.x, s); s = fmaf(-x[q4 * 4 + 1], l4.y, s);
                            s = fmaf(-x[q4 * 4 + 2], l4.z, s); s = fmaf(-x[q4 * 4 + 3], l4.w, s);
                        }
                        x[c] = s * S.invd[c];
                    }
#pragma unroll
                    for (int u = 0; u < kNB / 4; ++u)
                        *reinterpret_cast<float4*>(w + u * 4) = make_float4(x[u * 4], x[u * 4 + 1], x[u * 4 + 2], x[u * 4 + 3]);
                }
            }
            __syncthreads();
            CPROF(15);
            r0 += rows;
        }
    }
}

// Solve L L^T x = rhs for the factor in W; rhs in S.xs (float32, length nf), solution returned there.
__device__ void chol_solve_blocked(const float* __restrict__ W, int ldw, int nf, const DenseSmem& S, int tid) {
    constexpr int LD = kNB + 1;
    const int lane = tid & 31, warp = tid >> 5;
    float* x = S.xs;
    // forward: L y = rhs
    for (int j0 = 0; j0 < nf; j0 += kNB) {
        const int nb = nf - j0 < kNB ? nf - j0 : kNB;
        for (int t = tid; t < kNB * kNB; t += kDT) {
            const int i = t / kNB, j = t - i * kNB;
            S.D[i * LD + j] = (i < nb && j <= i) ? W[(size_t)(j0 + i) * ldw + j0 + j] : (i == j ? 1.0f : 0.0f);
        }
        {   // s_i = sum_{p < j0} L[i][p] y[p]: the four rows of a warp (i = warp + 16 t) together, so that their loads (from L2 /
            // HBM) are in flight at once instead of one row after the other
            const float* rows[4];
            float s[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int i = warp + t * (kDT / 32);
                rows[t] = W + (size_t)(j0 + (i < nb ? i : 0)) * ldw;
            }
#pragma unroll 2
            for (int q = lane * 4; q < j0; q += 128) {
                float4 l4[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) l4[t] = *reinterpret_cast<const float4*>(rows[t] + q);
                const float x0 = x[q], x1 = x[q + 1], x2 = x[q + 2], x3 = x[q + 3];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    s[t] = fmaf(l4[t].x, x0, s[t]); s[t] = fmaf(l4[t].y, x1, s[t]);
                    s[t] = fmaf(l4[t].z, x2, s[t]); s[t] = fmaf(l4[t].w, x3, s[t]);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int t = 0; t < 4; ++t) s[t] += __shfl_xor_sync(0xffffffffu, s[t], o);
            }
            if (lane == 0) {
#pragma unroll
                for (int t = 0; t < 4; ++t) { const int i = warp + t * (kDT / 32); if (i < nb) S.invd[i] = s[t]; }
            }
        }
        __syncthreads();
        if (warp == 0) {                                    // 64-step substitution, two rows per lane
            float t0 = lane < nb ? x[j0 + lane] - S.invd[lane] : 0.0f;
            float t1 = lane + 32 < nb ? x[j0 + lane + 32] - S.invd[lane + 32] : 0.0f;
            const float i0 = 1.0f / S.D[lane * LD + lane], i1 = 1.0f / S.D[(lane + 32) * LD + lane + 32];
            for (int c = 0; c < nb; ++c) {
                const float yc = __shfl_sync(0xffffffffu, c < 32 ? t0 * i0 : t1 * i1, c & 31);
                if (lane == (c & 31)) { if (c < 32) t0 = yc; else t1 = yc; }
                if (lane > c) t0 = fmaf(-S.D[lane * LD + c], yc, t0);
                if (lane + 32 > c) t1 = fmaf(-S.D[(lane + 32) * LD + c], yc, t1);
            }
            if (lane < nb) x[j0 + lane] = t0;
            if (lane + 32 < nb) x[j0 + lane + 32] = t1;
        }
        __syncthreads();
    }
    // backward: L^T x = y
    for (int j0 = ((nf - 1) / kNB) * kNB; j0 >= 0; j0 -= kNB) {
        const int nb = nf - j0 < kNB ? nf - j0 : kNB;
        for (int t = tid; t < kNB * kNB; t += kDT) {
            const int i = t / kNB, j = t - i * kNB;
            S.D[i * LD + j] = (i < nb && j <= i) ? W[(size_t)(j0 + i) * ldw + j0 + j] : (i == j ? 1.0f : 0.0f);
        }
        // s_c = sum_{i >= j0 + nb} L[i][j0 + c] x[i]: warps over rows i, lanes over the block's columns (two each)
        float s0 = 0.0f, s1 = 0.0f;
        {
            int i = j0 + nb + warp;
            for (; i + 7 * (kDT / 32) < nf; i += 8 * (kDT / 32)) {          // eight rows (sixteen loads) in flight per lane
                float a0[8], a1[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float* row = W + (size_t)(i + u * (kDT / 32)) * ldw + j0;
                    a0[u] = row[lane]; a1[u] = row[lane + 32];
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) { const float xi = x[i + u * (kDT / 32)]; s0 = fmaf(a0[u], xi, s0); s1 = fmaf(a1[u], xi, s1); }
            }
            for (; i < nf; i += kDT / 32) {
                const float xi = x[i];
                const float* row = W + (size_t)i * ldw + j0;
                s0 = fmaf(row[lane], xi, s0);
                s1 = fmaf(row[lane + 32], xi, s1);
            }
        }
        S.As[warp * kNB + lane] = s0; S.As[warp * kNB + lane + 32] = s1;
        __syncthreads();
        if (warp == 0) {
            float a0 = 0.0f, a1 = 0.0f;
            for (int w = 0; w < kDT / 32; ++w) { a0 += S.As[w * kNB + lane]; a1 += S.As[w * kNB + lane + 32]; }
            float t0 = lane < nb ? x[j0 + lane] - a0 : 0.0f;
            float t1 = lane + 32 < nb ? x[j0 + lane + 32] - a1 : 0.0f;
            const float i0 = 1.0f / S.D[lane * LD + lane], i1 = 1.0f / S.D[(lane + 32) * LD + lane + 32];
            for (int c = nb - 1; c >= 0; --c) {
                const float xc = __shfl_sync(0xffffffffu, c < 32 ? t0 * i0 : t1 * i1, c & 31);
                if (lane == (c & 31)) { if (c < 32) t0 = xc; else t1 = xc; }
                if (lane < c) t0 = fmaf(-S.D[c * LD + lane], xc, t0);
                if (lane + 32 < c) t1 = fmaf(-S.D[c * LD + lane + 32], xc, t1);
            }
            if (lane < nb) x[j0 + lane] = t0;
            if (lane + 32 < nb) x[j0 + lane + 32] = t1;
        }
        __syncthreads();
    }
}

// gt = G lamt - bb over all m rows (float64 accumulation); returns lamt^T gt and bb^T lamt.  The rows come from L2 / HBM with
// a latency of microseconds under load, so every warp keeps two rows = up to sixteen 16-byte loads per lane in flight.
__device__ void gram_matvec(const float* __restrict__ G, int ldg, int m, const double* lamt, const double* lamp, const double* bb,
                            double* gt, Ctx& cx, double& lg, double& lb) {
    double a_lg = 0.0, a_lb = 0.0;
    for (int v0 = 2 * cx.warp; v0 < m; v0 += 2 * cx.nwarp) {
        const bool two = v0 + 1 < m;
        const float* row0 = G + (size_t)v0 * ldg;
        const float* row1 = G + (size_t)(two ? v0 + 1 : v0) * ldg;
        double s0 = 0.0, s1 = 0.0;
        for (int j0 = cx.lane * 4; j0 < m; j0 += 1024) {    // columns up to the next multiple of 128 are zero in G and in lamt
            float4 g0[8], g1[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const bool in = j0 + u * 128 < m;
                g0[u] = in ? __ldg(reinterpret_cast<const float4*>(row0 + j0 + u * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
                g1[u] = in ? __ldg(reinterpret_cast<const float4*>(row1 + j0 + u * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int j = j0 + u * 128;
                if (j < m) {
                    // lamp holds column (base + 4 lane + c) at base + 32 c + lane: consecutive lanes, consecutive words
                    const int pb = (j & ~127) + cx.lane;
                    const double l0 = lamp[pb], l1 = lamp[pb + 32], l2 = lamp[pb + 64], l3 = lamp[pb + 96];
                    s0 += (double)g0[u].x * l0 + (double)g0[u].y * l1 + (double)g0[u].z * l2 + (double)g0[u].w * l3;
                    s1 += (double)g1[u].x * l0 + (double)g1[u].y * l1 + (double)g1[u].z * l2 + (double)g1[u].w * l3;
                }
            }
        }
        s0 = cx.warp_sum(s0); s1 = cx.warp_sum(s1);
        if (cx.lane == 0) {
            const double gv0 = s0 - bb[v0];
            gt[v0] = gv0; a_lg += lamt[v0] * gv0; a_lb += bb[v0] * lamt[v0];
            if (two) { const double gv1 = s1 - bb[v0 + 1]; gt[v0 + 1] = gv1; a_lg += lamt[v0 + 1] * gv1; a_lb += bb[v0 + 1] * lamt[v0 + 1]; }
        }
    }
    cx.block_sum2(a_lg, a_lb);
    lg = a_lg; lb = a_lb;
}

// rout = c - A^T x through the rows of A (float64), returns ||rout||^2.  The support of x is compacted first so that the
// column loop has no branch; four rows in flight per thread.
template <class TIO>
__device__ double true_residual(const float* __restrict__ Ainst, int d, int m, const double* x, const TIO* c, double* rout,
                                const DenseSmem& S, Ctx& cx, int* s_cnt) {
    if (cx.warp == 0) {
        int cnt = 0;
        for (int v0 = 0; v0 < m; v0 += 32) {
            const int v = v0 + cx.lane;
            const bool on = v < m && x[v] != 0.0;
            const unsigned mk = __ballot_sync(0xffffffffu, on);
            if (on) S.sup[cnt + __popc(mk & ((1u << cx.lane) - 1u))] = v;
            cnt += __popc(mk);
        }
        if (cx.lane == 0) *s_cnt = cnt;
    }
    __syncthreads();
    const int ns = *s_cnt;
    double ff = 0.0;
    for (int k = cx.tid; k < d; k += cx.nthr) {
        double acc = (double)c[k];
        int i = 0;
        for (; i + 32 <= ns; i += 32) {                     // 32 rows in flight per thread (the rows come from L2 / HBM)
            float a[32];
#pragma unroll
            for (int u = 0; u < 32; ++u) a[u] = __ldg(Ainst + (size_t)S.arow[S.sup[i + u]] * d + k);
#pragma unroll
            for (int u = 0; u < 32; ++u) acc -= x[S.sup[i + u]] * (double)a[u];
        }
        for (; i + 8 <= ns; i += 8) {
            float a[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) a[u] = __ldg(Ainst + (size_t)S.arow[S.sup[i + u]] * d + k);
#pragma unroll
            for (int u = 0; u < 8; ++u) acc -= x[S.sup[i + u]] * (double)a[u];
        }
        for (; i < ns; ++i) { const int v = S.sup[i]; acc -= x[v] * (double)__ldg(Ainst + (size_t)S.arow[v] * d + k); }
        rout[k] = acc; ff += acc * acc;
    }
    return cx.block_sum(ff);        // (barriers inside: rout is visible afterwards)
}

// g = -A r over all rows (one warp per row, kTgU 4-byte loads in flight per lane: the rows of A come from HBM)
#ifndef CAVE_TG_U
#define CAVE_TG_U 40      // (d = 1225 then is a single pass per row; 16 -> 40 measured +1 % at 1225 x 1024, neutral at d = 4950)
#endif
constexpr int kTgU = CAVE_TG_U;
__device__ void true_gradient(const float* __restrict__ Ainst, int d, int m, const double* r, double* g, const DenseSmem& S, Ctx& cx) {
    for (int v = cx.warp; v < m; v += cx.nwarp) {
        const float* row = Ainst + (size_t)S.arow[v] * d;
        double acc = 0.0;
        for (int k0 = 0; k0 < d; k0 += 32 * kTgU) {
            float a[kTgU];
#pragma unroll
            for (int u = 0; u < kTgU; ++u) { const int k = k0 + u * 32 + cx.lane; a[u] = k < d ? __ldg(row + k) : 0.f; }
#pragma unroll
            for (int u = 0; u < kTgU; ++u) { const int k = k0 + u * 32 + cx.lane; if (k < d) acc += (double)a[u] * r[k]; }
        }
        acc = cx.warp_sum(acc);
        if (cx.lane == 0) g[v] = -acc;
    }
    __syncthreads();
}

__device__ double kkt_residual(const double* lam, const double* g, int m, Ctx& cx) {
    double res = 0.0;
    for (int v = cx.tid; v < m; v += cx.nthr) {
        double t = lam[v] - g[v];
        t = t < 0.0 ? 0.0 : t;
        const double w = fabs(lam[v] - t);
        res = w > res ? w : res;
    }
    return cx.block_max(res);
}

// ---- Outlined shells (by-value arguments only, so nothing of the caller lives in memory): each heavy phase gets a register
// allocation of its own.  Inside the 128-register kernel ptxas sized the load batches of these loops by whatever else was
// live at the call site (e.g. the 32 loads in flight of true_residual came out as 10 + 9 + 8 in one instantiation and the
// phase ran three times slower), which made every phase depend on unrelated code.
#ifndef OUT_RES
#define OUT_RES 1
#endif
#ifndef OUT_GRAD
#define OUT_GRAD 1
#endif
#ifndef OUT_MV
#define OUT_MV 1
#endif
#ifndef OUT_TRI
#define OUT_TRI 0
#endif
#ifndef OUT_CHOL
#define OUT_CHOL 0
#endif
struct Pair64 { double a, b; };
template <class TIO>
__device__ __noinline__ double true_residual_o(const float* Ainst, int d, int m, const double* x, const TIO* c, double* rout, int* sup,
                                               int* arow, double* red, int* s_cnt) {
    DenseSmem S; S.sup = sup; S.arow = arow;
    Ctx cx(red);
    return true_residual<TIO>(Ainst, d, m, x, c, rout, S, cx, s_cnt);
}
__device__ __noinline__ void true_gradient_o(const float* Ainst, int d, int m, const double* r, double* g, int* arow, double* red) {
    DenseSmem S; S.arow = arow;
    Ctx cx(red);
    true_gradient(Ainst, d, m, r, g, S, cx);
}
__device__ __noinline__ Pair64 gram_matvec_o(const float* G, int ldg, int m, const double* lamt, const double* lamp, const double* bb,
                                             double* gt, double* red) {
    Ctx cx(red);
    Pair64 r;
    gram_matvec(G, ldg, m, lamt, lamp, bb, gt, cx, r.a, r.b);
    return r;
}
__device__ __noinline__ void chol_solve_o(const float* W, int ldw, int nf, float* As, float* D, float* invd, float* xs, int tid) {
    DenseSmem S; S.As = As; S.D = D; S.invd = invd; S.xs = xs;
    chol_solve_blocked(W, ldw, nf, S, tid);
}
template <bool TC>
__device__ __noinline__ void chol_blocked_o(float* W, int ldw, int nf, float floor_, float* As, float* Bs, float* D, float* Dt, float* invd,
                                            unsigned long long* prof, int tid) {
    DenseSmem S; S.As = As; S.Bs = Bs; S.D = D; S.Dt = Dt; S.invd = invd; S.prof = prof;
    chol_blocked<TC>(W, ldw, nf, floor_, S, tid);
}

// ---- Warm start (layout.cuh dense_warm_slot_bytes).  As for the structured solve (solver_core.cuh warm_read), a slot is
// only ever a starting guess: an index may hold an instance twice, so another CTA may write a slot while it is read.  The
// helpers run once per instance, outside the iteration, and are outlined with by-value arguments like the phases above.
// Hash of m and of every general row's index and length, by one warp (every lane gets the value).
__device__ uint32_t dense_warm_tag(const int4* gen, int m, int lane) {
    uint64_t h = 0;
    for (int v = lane; v < m; v += 32) {
        const int4 gv = gen[v];
        h += mix64(((uint64_t)v << 40) ^ ((uint64_t)(uint32_t)gv.y << 20) ^ (uint64_t)(uint32_t)gv.x);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
    return (uint32_t)(h ^ (h >> 32)) ^ (uint32_t)m;
}
// lam[0, m) <- the slot's multipliers if the slot holds a solution of this instance (same m and tag), with non-finite values
// replaced by 0 and negative ones clamped to 0; lam is left as it is otherwise.  Returns the slot's flags, or -1 if it was
// not used: the same on every thread (decided by thread 0, broadcast through *word, a word of shared memory).  All threads
// call; ends with a barrier.
__device__ __noinline__ int dense_warm_read(const char* slot, const int4* gen, int m, double* lam, int* word) {
    const int tid = threadIdx.x;
    if (tid < 32) {
        const uint32_t tag = dense_warm_tag(gen, m, tid);
        if (tid == 0) {
            const int4 h = __ldcg((const int4*)slot);
            *word = (h.x == 1 && h.y == m && (uint32_t)h.z == tag) ? (h.w & 1) : -1;
        }
    }
    __syncthreads();
    const int flags = *word;
    if (flags >= 0) {
        const double* val = (const double*)(slot + 16);
        for (int v = tid; v < m; v += kDT) {
            double x = __ldcg(val + v);
            if (!(x - x == 0.0) || x < 0.0) x = 0.0;        // NaN / Inf, negative
            lam[v] = x;
        }
    }
    __syncthreads();
    return flags;
}
// Stores lam[0, m) and flags as the slot's solution: the values first, the header after a fence and a barrier (a reader that
// sees the new header with older values still only gets a starting guess).  All threads call.
__device__ __noinline__ void dense_warm_write(char* slot, const int4* gen, int m, const double* lam, int flags) {
    const int tid = threadIdx.x;
    double* val = (double*)(slot + 16);
    for (int v = tid; v < m; v += kDT) val[v] = lam[v];
    uint32_t tag = 0;
    if (tid < 32) tag = dense_warm_tag(gen, m, tid);
    __threadfence();
    __syncthreads();
    if (tid == 0) *(int4*)slot = make_int4(1, m, (int)tag, flags);
}

// Coarse phase clocks (thread 0, clock64 deltas summed over instances): only in -DCAVE_DENSE_PROFILE builds.
#ifdef CAVE_DENSE_PROFILE
#define DPROF_BEGIN() long long dprof_t = clock64()
#define DPROF(ph) do { if (threadIdx.x == 0) { const long long t_ = clock64(); atomicAdd(prof + (ph), (unsigned long long)(t_ - dprof_t)); dprof_t = t_; } } while (0)
#else
#define DPROF_BEGIN() do {} while (0)
#define DPROF(ph) do {} while (0)
#endif
enum { DP_SETUP = 0, DP_KKT = 1, DP_FREESET = 2, DP_GATHER = 3, DP_CHOL = 4, DP_TRISOLVE = 5, DP_LS_GRAM = 6, DP_LS_TRUE = 7,
       DP_TRUEGRAD = 8, DP_EPILOGUE = 9, DP_SWITCH = 10, DP_NFACT = 11, DP_NITER = 12 };

// TC: the Cholesky block-column update runs on the tensor cores (a separate instantiation, so that the register allocation of
// each variant only sees the update it uses).  WARM: the variant for calls with a warm-start buffer (p.warm); the other one
// compiles none of the warm-start code.
template <class TIO, bool TC, bool WARM>
__global__ void __launch_bounds__(kDT, 1) dense_solve_kernel(DenseParams p) {
    extern __shared__ __align__(16) char dsm[];
    __shared__ double red[64];
    __shared__ int s_next, s_nf, s_same, s_cnt;
    int* ctrl = (int*)(p.ws + p.L.ctrl);
#ifdef CAVE_DENSE_PROFILE
    unsigned long long* prof = (unsigned long long*)(p.ws + p.L.ctrl + 64);
#endif
    const int* list = (const int*)(p.ws + p.L.list);
    int* flag = (int*)(p.ws + p.L.flag);
    const int n_slots = (int)p.L.n_slots, mp = (int)p.L.m_pad;
    int n_round = ctrl[0] - p.round * n_slots;
    n_round = n_round < n_slots ? n_round : n_slots;
    if (n_round <= 0) return;
    Ctx cx(red);
    const int tid = cx.tid;
    DenseSmem S;
    {
        char* o = dsm;
        S.lam = (double*)o; o += (size_t)mp * 8; S.lamt = (double*)o; o += (size_t)mp * 8;
        S.g = (double*)o; o += (size_t)mp * 8; S.gt = (double*)o; o += (size_t)mp * 8;
        S.dir = (double*)o; o += (size_t)mp * 8; S.bb = (double*)o; o += (size_t)mp * 8;
        S.lamp = (double*)o; o += (size_t)mp * 8;
        S.fl = (int*)o; o += (size_t)mp * 4; S.flp = (int*)o; o += (size_t)mp * 4;
        S.arow = (int*)o; o += (size_t)mp * 4; S.sup = (int*)o; o += (size_t)mp * 4;
        S.xs = (float*)o; o += (size_t)mp * 4;
        S.As = (float*)o; S.Bs = S.As + (size_t)kKS * kRC;
        o += TC ? (size_t)kTcBytes + 1024 : (size_t)kStageSimt;    // (TC: the 1024-byte aligned operand planes lie over As / Bs)
        S.Dt = (float*)o; o += (size_t)kNB * kNB * 4;
        S.D = (float*)o; o += (size_t)kNB * (kNB + 1) * 4; S.invd = (float*)o;
#ifdef CAVE_DENSE_PROFILE
        S.prof = prof;
#else
        S.prof = nullptr;
#endif
    }
    if constexpr (TC) {
        // TMEM: 256 columns = four 128 x 64 float32 accumulator tiles of the Cholesky update (one CTA per SM: no contention)
        if (tid == 0) {
            tc::mbar_init(&tc_bar_s, 1);
            tc_phase_s = 0;
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        if (tid < 32) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(tc::smem_u32(&tmem_base_s)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tc::fence_before();
        __syncthreads();
        tc::fence_after();
    }
    const TIO* pred_all = (const TIO*)p.pred;
    TIO* grad_all = (TIO*)p.grad;
    TIO* proj_all = (TIO*)p.proj;
    EpiParams ep; ep.mode = p.mode; ep.inner_ratio = p.inner_ratio; ep.sign = p.sign; ep.gscale = p.gscale;
    constexpr double kEps = 2.220446049250313e-16;

    for (;;) {
        if (tid == 0) s_next = atomicAdd(&ctrl[1], 1);
        __syncthreads();
        const int s = s_next;
        __syncthreads();
        if (s >= n_round) break;
        DPROF_BEGIN();
        const int b = list[p.round * n_slots + s];
        const size_t q = p.inst_index ? (size_t)p.inst_index[b] : (size_t)b;
        const int m = p.ngen[q], d = p.d;
        const float* Ainst = p.A + q * (size_t)p.m_max * d;
        const int4* gen = p.gen + q * (size_t)p.m_max;
        const float* G = (const float*)(p.ws + p.L.G) + (size_t)s * mp * mp;
        float* W = (float*)(p.ws + p.L.W) + (size_t)s * mp * mp;
        const double* bsrc = (const double*)(p.ws + p.L.bvec) + (size_t)s * mp;
        const float* l1src = (const float*)(p.ws + p.L.l1) + (size_t)s * mp;
        double* vec = (double*)(p.ws + p.L.vec) + (size_t)s * p.L.vec_doubles;
        double* r = vec;                                        // [d]  r = c - A^T lam
        double* rt = vec + p.L.d_pad;                           // [d]  trial residual
        TIO* c = (TIO*)(vec + 2 * p.L.d_pad);                   // [d]  c = sign * pred
        const TIO* pred = pred_all + (size_t)b * d;

        // ---- setup
        double cc = 0.0, l1m = 0.0, dmax = 0.0, dsum = 0.0, osum = 0.0;
        double* dgv = vec + 3 * p.L.d_pad;                      // [m]  diagonal of G~ (scaling of the binding block)
        for (int k = tid; k < d; k += kDT) { const TIO vc = (TIO)(p.sign * (double)pred[k]); c[k] = vc; r[k] = (double)vc; cc += (double)vc * (double)vc; }
        for (int v = tid; v < mp; v += kDT) {
            const bool in = v < m;
            S.bb[v] = in ? bsrc[v] : 0.0; S.lam[v] = 0.0; S.lamt[v] = 0.0; S.g[v] = in ? -bsrc[v] : 0.0; S.gt[v] = 0.0; S.dir[v] = 0.0;
            S.arow[v] = in ? gen[v].x : 0;
            if (in) {
                const double l = (double)l1src[v]; l1m = l > l1m ? l : l1m;
                const float* grow = G + (size_t)v * mp;
                const double gd = (double)grow[v]; dmax = gd > dmax ? gd : dmax; dsum += gd;
                dgv[v] = gd > 0.0 ? gd : 1.0;
                // a sample of the off-diagonal magnitudes: how good a model of G~ its diagonal is
                osum += fabs((double)grow[(v + 1) % m]) + fabs((double)grow[(v + 7) % m]) + fabs((double)grow[(v + m / 2) % m]) + fabs((double)grow[(v + m / 3 + 1) % m]);
            }
        }
        cc = cx.block_sum(cc);
        cx.block_max2(l1m, dmax);
        cx.block_sum2(dsum, osum);
        // Scaling M of the binding block in Bertsekas' two-metric projection: diag(G~)^-1 when G~ is weakly coupled (Gaussian-like
        // rows: the 1-D Newton step is then the right step for a nearly active variable and epsilon lives in lambda units), the
        // identity when the rows are strongly correlated (e.g. positive matrices, where almost everything ends up bound and the
        // aggressive identity-scaled rule identifies it in a few iterations).  An instance switches to the diagonal scaling for good
        // when a line search has to cut the step to the order of 1 / G_vv (the signature of the identity scaling overshooting).
        bool scaled = osum * 0.25 < 0.25 * dsum;
        const double cnorm = sqrt(cc);
        const bool finite_in = cc < 1e300 && !(p.mode != MODE_EXACT && p.plan && p.plan[PLAN_NO_AVG] != 0ull);   // (or a pack without the average in a mode that needs it)
        DPROF(DP_SETUP);
        int status = ST_BADINPUT, iters = 0;
        bool handed_back = false;
        int why = 0, why_phase = 0;
        if (finite_in) {
            const double scale = (l1m > 1.0 ? l1m : 1.0) * (cnorm > 1e-30 ? cnorm : 1e-30);
            const double tol = (p.tol > 0 ? p.tol : 1e-12) * scale;
            const double tolG = 1e-6 * scale > tol ? 1e-6 * scale : tol;
            const int max_it1 = p.max_iter > 0 ? p.max_iter : 60, max_it2 = 40;
            const int max_ls = p.max_ls > 0 ? p.max_ls : 40;
            // Tikhonov term above the accuracy of G~ (3xTF32 operands, truncating float32 accumulation: ~1.5e-5 relative on the
            // diagonal at d = 1225), so that the factored matrix is positive definite even where G_FF is singular (|F| > d)
            const float regf = (float)(4e-5 * dmax), floorf_ = (float)(1e-6 * dmax);
            // Warm start: lam from the instance's slot if it holds a solution of this instance.  Such a start skips the
            // Gram-space phase (it would pull lam towards the float32-accurate optimum of G~, while the stored lam is anchored
            // to A) and resumes with the metric the stored solve ended with.
            char* wslot = (WARM && p.warm && m <= p.warm_cap) ? p.warm + q * (size_t)p.warm_stride : nullptr;
            bool warm_try = false;
            const bool scaled0 = scaled;
            if (WARM && wslot) {
                const int wf = dense_warm_read(wslot, gen, m, S.lam, &s_nf);
                warm_try = wf >= 0;
                if (warm_try) scaled = (wf & 1) != 0;
            }
            double* lam = S.lam; double* lamt = S.lamt; double* g = S.g; double* gt = S.gt;
            double* rc = r; double* rtr = rt;
            for (;;) {      // (WARM: a failed warm start is solved once more from zero; otherwise one pass)
            int nf_fact = -1;                           // size of the free set the factor in W belongs to (-1: none)
            double f = 0.0;                             // phase 1: q(lam);  phase 2: 1/2 ||r||^2
            int phase = 1, since_best = 0, it1 = (WARM && warm_try) ? max_it1 : 0, it2 = 0;     // (a warm start switches at once)
            double res_best = 1e300;
            status = ST_ITER_CAP;
            for (;;) {
                double res = kkt_residual(lam, g, m, cx);
                DPROF(DP_KKT);
                if (phase == 1 && (res <= tolG || it1 >= max_it1)) {
                    if (res > 1e-4 * scale && !(WARM && warm_try)) { handed_back = true; why = 1; why_phase = 1; break; }       // the Gram-space iteration did not settle
                    // ---- switch to the true problem: r = c - A^T lam, g = -A r
                    phase = 2; since_best = 0; res_best = 1e300;
                    f = 0.5 * (OUT_RES ? true_residual_o<TIO>(Ainst, d, m, lam, c, rc, S.sup, S.arow, red, &s_cnt)
                                                  : true_residual<TIO>(Ainst, d, m, lam, c, rc, S, cx, &s_cnt));
                    // a warm point that fits worse than lam = 0 (or overflows) is not worth starting from
                    if (WARM && warm_try && !(f <= 0.5 * cc)) { status = ST_STALLED; break; }
                    if (OUT_GRAD) true_gradient_o(Ainst, d, m, rc, g, S.arow, red); else true_gradient(Ainst, d, m, rc, g, S, cx);
                    res = kkt_residual(lam, g, m, cx);
                    DPROF(DP_SWITCH);
                }
                if (phase == 2) {
                    if (!(res > tol)) { status = ST_CONVERGED; break; }
                    if (res < 0.5 * res_best) { res_best = res; since_best = 0; }
                    else if (++since_best >= 4 && res <= 1e3 * tol) { status = ST_CONVERGED; break; }
                    if (it2 >= max_it2) {
                        status = res <= 1e3 * tol ? ST_CONVERGED : ST_ITER_CAP;
                        if (res > 1e-8 * scale) { handed_back = true; why = 3; why_phase = 2; }
                        break;
                    }
                    ++it2;
                } else {
                    ++it1;
                }
                ++iters;
                // ---- free set (ordered); binding variables take a gradient step
                const double epsb = res < 1e-3 ? res : 1e-3;
                if (cx.warp == 0) {
                    int cnt = 0; bool same = true;
                    for (int v0 = 0; v0 < m; v0 += 32) {
                        const int v = v0 + cx.lane;
                        const bool isf = v < m && !(lam[v] <= (scaled ? epsb / dgv[v] : epsb) && g[v] > 0.0);
                        const unsigned mk = __ballot_sync(0xffffffffu, isf);
                        if (isf) {
                            const int pos = cnt + __popc(mk & ((1u << cx.lane) - 1u));
                            if (pos >= nf_fact || S.flp[pos] != v) same = false;
                            S.fl[pos] = v;
                        }
                        cnt += __popc(mk);
                    }
                    same = __all_sync(0xffffffffu, same) && cnt == nf_fact;
                    if (cx.lane == 0) { s_nf = cnt; s_same = same ? 1 : 0; }
                }
                for (int v = tid; v < m; v += kDT) S.dir[v] = scaled ? g[v] / dgv[v] : g[v];
                __syncthreads();
                const int nf = s_nf;
                const bool same = s_same != 0;
                DPROF(DP_FREESET);
                if (nf > 0) {
                    if (!same) {
                        // gather the free block: W[a][b'] = G[F[a]][F[b']] (b' <= a) + reg on the diagonal, then factor
                        for (int a = cx.warp; a < nf; a += cx.nwarp) {
                            const float* grow = G + (size_t)S.fl[a] * mp;
                            float* wrow = W + (size_t)a * mp;
                            for (int b0 = cx.lane; b0 <= a; b0 += 256) {        // eight gathers in flight per lane
                                float gv[8];
#pragma unroll
                                for (int u = 0; u < 8; ++u) { const int bq = b0 + u * 32; gv[u] = bq <= a ? __ldg(grow + S.fl[bq]) : 0.0f; }
#pragma unroll
                                for (int u = 0; u < 8; ++u) { const int bq = b0 + u * 32; if (bq <= a) wrow[bq] = gv[u] + (bq == a ? regf : 0.0f); }
                            }
                        }
                        for (int a = tid; a < nf; a += kDT) S.flp[a] = S.fl[a];
                        __syncthreads();
                        DPROF(DP_GATHER);
                        if (OUT_CHOL) chol_blocked_o<TC>(W, mp, nf, floorf_, S.As, S.Bs, S.D, S.Dt, S.invd, S.prof, tid);
                        else chol_blocked<TC>(W, mp, nf, floorf_, S, tid);
                        nf_fact = nf;
                        DPROF(DP_CHOL);
#ifdef CAVE_DENSE_PROFILE
                        if (tid == 0) atomicAdd(prof + DP_NFACT, 1ull);
#endif
                    }
                    for (int a = tid; a < nf; a += kDT) S.xs[a] = (float)g[S.fl[a]];
                    __syncthreads();
                    if (OUT_TRI) chol_solve_o(W, mp, nf, S.As, S.D, S.invd, S.xs, tid); else chol_solve_blocked(W, mp, nf, S, tid);
                    for (int a = tid; a < nf; a += kDT) S.dir[S.fl[a]] = (double)S.xs[a];
                }
                __syncthreads();
                DPROF(DP_TRISOLVE);
#ifdef CAVE_DENSE_PROFILE
                if (tid == 0) atomicAdd(prof + DP_NITER, 1ull);
#endif
                // ---- Armijo along the projection arc
                double alpha = 1.0, ft = f;
                bool ok = false, at_floor = false;
                for (int ls = 0; ls < max_ls; ++ls) {
                    double dec = 0.0;
                    for (int v = tid; v < mp; v += kDT) {
                        double t = 0.0;
                        if (v < m) { t = lam[v] - alpha * S.dir[v]; if (t < 0.0) t = 0.0; dec += g[v] * (lam[v] - t); }
                        lamt[v] = t;
                        S.lamp[(v & ~127) + ((v & 3) << 5) + ((v >> 2) & 31)] = t;
                    }
                    dec = cx.block_sum(dec);
                    if (phase == 1) {
                        double lg, lb;
                        if (OUT_MV) { const Pair64 pr = gram_matvec_o(G, mp, m, lamt, S.lamp, S.bb, gt, red); lg = pr.a; lb = pr.b; }
                        else gram_matvec(G, mp, m, lamt, S.lamp, S.bb, gt, cx, lg, lb);
                        ft = 0.5 * lg - 0.5 * lb;
                        DPROF(DP_LS_GRAM);
                    } else {
                        ft = 0.5 * (OUT_RES ? true_residual_o<TIO>(Ainst, d, m, lamt, c, rtr, S.sup, S.arow, red, &s_cnt)
                                                       : true_residual<TIO>(Ainst, d, m, lamt, c, rtr, S, cx, &s_cnt));
                        DPROF(DP_LS_TRUE);
                    }
                    const double fa = fabs(f);
                    if (ls == 0 && fabs(dec) <= 16.0 * kEps * fa && fabs(ft - f) <= 16.0 * kEps * fa) { ok = true; at_floor = true; break; }
                    if (ft <= f - 1e-4 * dec + 4.0 * kEps * fa) { ok = true; break; }
                    alpha *= 0.5;
                }
                if (p.trace_b == b && tid == 0)
                    printf("dense trace b=%d phase %d it1 %d it2 %d res/scale %.3e nf %d same %d alpha %.3e f %.15e ft %.15e ok %d floor %d\n", b, phase, it1, it2,
                           res / scale, nf, (int)same, alpha, f, ft, (int)ok, (int)at_floor);
                if (!ok && !scaled) { scaled = true; continue; }      // identity scaling failed outright: retry this point with the diagonal one
                if (!ok) {
                    // the current point stays; in phase 1 a stall close to the solution still goes on to the true problem
                    if (phase == 1 && res <= 1e-4 * scale) { it1 = max_it1; continue; }
                    status = (phase == 2 && res <= 1e3 * tol) ? ST_CONVERGED : ST_STALLED;
                    if (phase == 1 || res > 1e-8 * scale) { handed_back = true; why = phase == 1 ? 2 : 4; why_phase = phase; }
                    break;
                }
                if (alpha < 1.0 / 64.0) scaled = true;
                { double* t1 = lam; lam = lamt; lamt = t1; }
                f = ft;
                if (phase == 1) { double* t2 = g; g = gt; gt = t2; }
                else {
                    { double* t3 = rc; rc = rtr; rtr = t3; }
                    if (OUT_GRAD) true_gradient_o(Ainst, d, m, rc, g, S.arow, red); else true_gradient(Ainst, d, m, rc, g, S, cx);
                    DPROF(DP_TRUEGRAD);
                    if (at_floor) { status = ST_CONVERGED; break; }
                }
                __syncthreads();
            }
            __syncthreads();
            if (!(WARM && warm_try && (handed_back || status == ST_ITER_CAP || status == ST_STALLED))) break;
            // ---- the warm start failed: back to the state the setup above left (iterations add up; only this cold
            // solve may hand the instance back to Lawson-Hanson)
            warm_try = false; handed_back = false; why = 0; why_phase = 0; scaled = scaled0;
            lam = S.lam; lamt = S.lamt; g = S.g; gt = S.gt; rc = r; rtr = rt;
            for (int k = tid; k < d; k += kDT) r[k] = (double)c[k];
            for (int v = tid; v < mp; v += kDT) {
                S.lam[v] = 0.0; S.lamt[v] = 0.0; S.g[v] = v < m ? -bsrc[v] : 0.0; S.gt[v] = 0.0; S.dir[v] = 0.0;
            }
            __syncthreads();
            }
            if (!handed_back && rc != r) {          // the epilogue reads r
                for (int k = tid; k < d; k += kDT) r[k] = rc[k];
            }
            __syncthreads();
            if (WARM && wslot && !handed_back && status == ST_CONVERGED) dense_warm_write(wslot, gen, m, lam, scaled ? 1 : 0);
            if (WARM && warm_try) status |= ST_WARM;
        }
        if (handed_back && p.no_handback) { handed_back = false; status |= (why << 16) | (why_phase << 12); }
        if (handed_back) {
            if (tid == 0) flag[b] = 0;               // the Lawson-Hanson path (general solve kernel, launched next) takes it
        } else if (!finite_in) {                     // NaN / Inf prediction: reported, never a silent number
            for (int k = tid; k < d; k += kDT) { grad_all[(size_t)b * d + k] = (TIO)NAN; if (proj_all) proj_all[(size_t)b * d + k] = (TIO)NAN; }
            if (tid == 0) { p.loss64[b] = NAN; p.rnorm64[b] = NAN; p.status[b] = ST_BADINPUT | ST_PATH_GRAM; p.iters[b] = 0; }
        } else {
            Instance in;
            in.A = Ainst; in.gen = (const gen_t*)gen; in.ctype = p.ctype + q * p.dpad; in.avg = p.avg + q * p.dpad;
            in.d = d; in.ngen = m; in.gen_nnz = 0; in.nvalid = m; in.nsingc = 0; in.csr_ok = 0;
            in.ghash = nullptr; in.pcol = nullptr; in.pval = nullptr; in.maxl1 = 0.f; in.maxl2 = 0.f; in.setup = nullptr;
            in.warm = nullptr; in.warm_cap = 0;
            epilogue<double, TIO, const TIO*>(cx, in, ep, c, r, p.mode != MODE_HEURISTIC, false, grad_all + (size_t)b * d,
                                              proj_all ? proj_all + (size_t)b * d : nullptr, p.loss64 + b, p.rnorm64 + b);
            if (tid == 0) { p.status[b] = status | ST_PATH_GRAM; p.iters[b] = iters; }
        }
        __syncthreads();
        DPROF(DP_EPILOGUE);
    }
    if constexpr (TC) {
        tc::fence_before();
        __syncthreads();
        if (tid < 32) {
            tc::fence_after();
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base_s) : "memory");
        }
    }
}

cudaError_t launch_dense_solve(const DenseParams& p_in, cudaStream_t stream) {
    DenseParams p = p_in;
    // static shared memory of the kernel (reduction scratch, counters, mbarrier): 1.6 KB
    const size_t budget = 227 * 1024 - 2048;
    // Default when its operand planes fit beside the solver's vectors (m_pad <= 1408); CAVE_DENSE_TC=0 keeps the FFMA update.
    // Measured on B200 at 1225 x 1024: update 3.5 -> 1.8 Mclk per instance, 18.5 k -> 20.0 k inst/s.  (It only pays with the
    // outlined phases + -rdc: inlined into the 128-register kernel, ptxas sized the load batches of the residual / matvec /
    // triangular-solve loops by what the call site left free and the other phases lost what the update gained: DESIGN.md 4.3.)
    const char* e_tc = getenv("CAVE_DENSE_TC");
    p.tc_update = (!e_tc || atoi(e_tc) != 0) && dense_solve_smem(p.L.m_pad, true) <= budget ? 1 : 0;
    size_t smem = dense_solve_smem(p.L.m_pad, p.tc_update != 0);
    if (smem > budget) return cudaErrorInvalidValue;
    if (const char* e_pad = getenv("CAVE_DENSE_SMEM_PAD")) {  // diagnostics: unused extra shared memory (moves the L1 / shared-memory split)
        const size_t want = smem + (size_t)atoi(e_pad);
        smem = want < budget ? want : budget;
    }
    void (*kern)(DenseParams) =
        p.warm ? (p.tc_update ? (p.io_f32 ? dense_solve_kernel<float, true, true> : dense_solve_kernel<double, true, true>)
                              : (p.io_f32 ? dense_solve_kernel<float, false, true> : dense_solve_kernel<double, false, true>))
               : (p.tc_update ? (p.io_f32 ? dense_solve_kernel<float, true, false> : dense_solve_kernel<double, true, false>)
                              : (p.io_f32 ? dense_solve_kernel<float, false, false> : dense_solve_kernel<double, false, false>));
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned grid = (unsigned)(p.L.n_slots < sms ? p.L.n_slots : sms);
    kern<<<grid, kDT, smem, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace cave
