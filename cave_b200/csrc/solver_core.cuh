// Per-instance cone projection solver + fused loss/backward epilogue, written against cave::Ctx
// (one CTA per instance on the device; single thread under CAVE_HOST_SIM).
//
// Problem (SURVEY.md App. A; reference src/cave.py:298-309): for the valid rows a_i of A,
//     lambda* = argmin_{lambda >= 0} || sum_i lambda_i a_i - c ||^2 ,  p = sum_i lambda*_i a_i .
// Rows with exactly one non-zero ("singleton" rows alpha*e_k; src/dataset.py:198-211 emits one per
// variable) generate a product of 1-D cones, against which the distance is separable:
//     psi_k(r) = r - proj_{I_k}(r),  I_k in { {0}, [0,inf), (-inf,0], R }   (ctype 0,1,2,3).
// With B the remaining "general" rows the projection reduces exactly to
//     min_{nu >= 0} f(nu) = 1/2 || psi(c - B^T nu) ||^2 ,    p = c - psi(c - B^T nu*)
// a convex piecewise quadratic in dim(nu) = #general rows (~110 instead of ~1335 at TSP-50).
//
//  * Structured instances (some coordinate has a singleton row): projected semismooth Newton
//    (Bertsekas' two-metric projection with the generalised Hessian B_F W B_F^T, W = diag(psi')),
//    Armijo search along the projection arc.  Rows b_j = -b_i (an equality split into +- rows,
//    src/dataset.py:182-184) are merged into one sign-free variable first.
//  * Pure general instances (no singleton row at all, e.g. the dense rand/randn matrices of
//    test/test_func.py:34-43): Lawson-Hanson active set in Gram form with an appended Cholesky
//    row per pivot — the same algorithm family as scipy.optimize.nnls which the reference calls.
//
// Nothing here is first order: no step-size/momentum pair that could reproduce the FISTA
// divergence documented in the reference README (README.md:40).
#pragma once
#if defined(CAVE_NW_TRACE)
#include <stdio.h>
#endif
#include "ctx.cuh"

namespace cave {

#ifdef CAVE_HOST_SIM
struct int4_ { int x, y, z, w; };
typedef int4_ gen_t;
struct u64x2_ { uint64_t x, y; };
typedef u64x2_ hash_t;
struct float4_ { float x, y, z, w; };
typedef float4_ f4_t;
#else
typedef int4 gen_t;
typedef float4 f4_t;
typedef ulonglong2 hash_t;
#endif

struct alignas(16) G16 { uint32_t x, y, z, w; };      // one 16-byte granule (bulk copies of byte / halfword arrays)
// Bulk copy of n granules by the whole CTA, four loads in flight per thread.  Deliberately not inlined: it runs once per
// instance and must not add to the register pressure of the solver it is called from.
#ifdef CAVE_HOST_SIM
inline void copy_granules(G16* dst, const G16* src, int n, int tid, int nthr) { for (int e = tid; e < n; e += nthr) dst[e] = src[e]; }
#else
static __device__ __noinline__ void copy_granules(G16* dst, const G16* src, int n, int tid, int nthr) {
    for (int e0 = 0; e0 < n; e0 += 4 * nthr) {
        G16 a[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { const int e = e0 + u * nthr + tid; if (e < n) a[u] = src[e]; }
#pragma unroll
        for (int u = 0; u < 4; ++u) { const int e = e0 + u * nthr + tid; if (e < n) dst[e] = a[u]; }
    }
}
#endif

enum { ST_CONVERGED = 0, ST_ITER_CAP = 1, ST_STALLED = 2, ST_NOSPACE = 3, ST_SKIPPED = 4, ST_BADINPUT = 5, ST_PATH_LH = 0x100, ST_PATH_GRAM = 0x200,
       ST_WARM = 0x400 };
enum { MODE_EXACT = 0, MODE_INNER = 1, MODE_HEURISTIC = 2 };

struct SolveOpts {
    int max_iter;      // <= 0: default
    int max_ls;
    double tol;        // relative KKT tolerance
};

// Bump allocator over the CTA's shared memory and its global scratch slot.
//   get_sm : "hot" arrays (vectors, Hessian, factor).  Shared memory only, taken from the front; the
//            returned pointer is shared-base + offset with no generic select, so the compiler keeps the
//            shared address space and emits LDS/STS/ATOMS for them.
//   get    : "cold" arrays (sparse rows, setup scratch).  Taken from the back of shared memory while it
//            lasts, then from the global slot; accessed through generic pointers.
struct Arena {
    char* sm; size_t sm_front, sm_back;
    char* gl; size_t gl_cap, gl_off;
    bool overflow, hot_overflow;
    CAVE_DEV void init(char* s, size_t sc, char* g, size_t gc) {
        sm = s; sm_front = 0; sm_back = sc & ~(size_t)15; gl = g; gl_cap = gc; gl_off = 0; overflow = false; hot_overflow = false;
    }
    template <class U> CAVE_DEV U* get_sm(size_t n) {
        const size_t bytes = (n * sizeof(U) + 15) & ~(size_t)15;
        U* p = (U*)(sm + sm_front);
        if (sm_front + bytes <= sm_back) sm_front += bytes; else { hot_overflow = true; overflow = true; }
        return p;      // callers check `overflow` before touching memory
    }
    template <class U> CAVE_DEV U* get(size_t n) {
        const size_t bytes = (n * sizeof(U) + 15) & ~(size_t)15;
        if (sm_front + bytes <= sm_back) { sm_back -= bytes; return (U*)(sm + sm_back); }
        if (gl_off + bytes <= gl_cap) { U* p = (U*)(gl + gl_off); gl_off += bytes; return p; }
        overflow = true;
        return (U*)gl;
    }
    // setup-only scratch: always from the global slot (keeps shared memory for the iteration's arrays)
    template <class U> CAVE_DEV U* get_gl(size_t n) {
        const size_t bytes = (n * sizeof(U) + 15) & ~(size_t)15;
        if (gl_off + bytes <= gl_cap) { U* p = (U*)(gl + gl_off); gl_off += bytes; return p; }
        overflow = true;
        return (U*)gl;
    }
    template <bool HOT, class U> CAVE_DEV HPtr<U, HOT> geth(size_t n) {
        if (HOT) return HPtr<U, HOT>(get_sm<U>(n));
        return HPtr<U, HOT>(get<U>(n));
    }
};

// Bump allocator over a borrowed region (an array that is idle during setup); falls back to the arena's cold side.
struct SubArena {
    char* base; size_t cap, off;
    CAVE_DEV void init(char* b, size_t c) { base = b; cap = c & ~(size_t)15; off = 0; }
    template <class U> CAVE_DEV U* get(Arena& ar, size_t n) {
        const size_t bytes = (n * sizeof(U) + 15) & ~(size_t)15;
        if (off + bytes <= cap) { U* p = (U*)(base + off); off += bytes; return p; }
        return ar.get<U>(n);
    }
};

// ctype bit0: a row +a*e_k exists (positive residual absorbed); bit1: a row -a*e_k exists (negative absorbed)
template <class T> CAVE_DEV bool psi_active(T r, int t) {
    return t == 0 ? true : (r > (T)0 ? !(t & 1) : (r < (T)0 ? !(t & 2) : false));
}
template <class T> CAVE_DEV T psi(T r, int t) { return psi_active(r, t) ? r : (T)0; }
template <class T> CAVE_DEV T cabs(T v) { return v < (T)0 ? -v : v; }
// start of row i in a row-packed lower triangle (row i holds columns 0..i)
CAVE_DEV uint32_t tri(int i) { return ((uint32_t)i * (uint32_t)(i + 1)) >> 1; }
// Reciprocal of a positive pivot: it sits on the critical path of every LDL^T column.  Measured dependent latency
// on B200 (tools/ubench/rcp.cu): 1.0/x 80 cycles, MUFU seed + Newton steps 47 (f64, full precision) / 22 (f32).
CAVE_DEV float fast_rcp(float x) {
#ifdef CAVE_HOST_SIM
    return 1.0f / x;
#else
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    const float e = fmaf(-x, y, 1.0f);
    return fmaf(y, e, y);
#endif
}
CAVE_DEV double fast_rcp(double x) {
#ifdef CAVE_HOST_SIM
    return 1.0 / x;
#else
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));     // >= 20 bits
    double e = fma(-x, y, 1.0); y = fma(y, e, y);
    e = fma(-x, y, 1.0);
    return fma(y, e, y);
#endif
}
template <class T> CAVE_DEV T eps_mach();
template <> CAVE_DEV double eps_mach<double>() { return 2.220446049250313e-16; }
template <> CAVE_DEV float eps_mach<float>() { return 1.1920929e-7f; }

CAVE_DEV uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

// ------------------------------------------------------------------ dense Cholesky helpers
// In-place right-looking Cholesky of the lower triangle of H (row-major, leading dim ld).  The
// diagonal of L goes to diagL; H's own diagonal is left untouched.  Pivots are floored at
// `floor_` so that semidefinite systems stay solvable (the Tikhonov term makes them consistent).
template <class T>
CAVE_DEV void chol_factor(Ctx& cx, T* H, int n, int ld, T* diagL, T floor_) {
    for (int j = 0; j < n; ++j) {
        cx.sync();
        T piv = H[(size_t)j * ld + j];
        T ljj = (T)sqrt((double)(piv > floor_ ? piv : floor_));
        if (cx.tid == 0) diagL[j] = ljj;
        T inv = (T)1 / ljj;
        for (int i = j + 1 + cx.tid; i < n; i += cx.nthr) H[(size_t)i * ld + j] *= inv;
        cx.sync();
        for (int i = j + 1 + cx.warp; i < n; i += cx.nwarp) {
            T lij = H[(size_t)i * ld + j];
            for (int k = j + 1 + cx.lane; k <= i; k += Ctx::WS)
                H[(size_t)i * ld + k] -= lij * H[(size_t)k * ld + j];
        }
    }
    cx.sync();
}

// Forward substitution L y = x in place for rows [0, n) (warp 0 only; caller syncs afterwards).
template <class T>
CAVE_DEV void tri_forward_w0(Ctx& cx, const T* L, int n, int ld, const T* diagL, T* x) {
    for (int j = 0; j < n; ++j) {
        T yj = x[j] / diagL[j];
        cx.syncwarp();
        if (cx.lane == 0) x[j] = yj;
        for (int i = j + 1 + cx.lane; i < n; i += Ctx::WS) x[i] -= L[(size_t)i * ld + j] * yj;
        cx.syncwarp();
    }
}
template <class T>
CAVE_DEV void tri_backward_w0(Ctx& cx, const T* L, int n, int ld, const T* diagL, T* x) {
    for (int j = n - 1; j >= 0; --j) {
        T zj = x[j] / diagL[j];
        cx.syncwarp();
        if (cx.lane == 0) x[j] = zj;
        for (int i = cx.lane; i < j; i += Ctx::WS) x[i] -= L[(size_t)j * ld + i] * zj;
        cx.syncwarp();
    }
}
template <class T>
CAVE_DEV void chol_solve(Ctx& cx, const T* L, int n, int ld, const T* diagL, T* x) {
    cx.sync();
    if (cx.warp == 0) {
        tri_forward_w0(cx, L, n, ld, diagL, x);
        tri_backward_w0(cx, L, n, ld, diagL, x);
    }
    cx.sync();
}


// ------------------------------------------------------------------ blocked LDL^T (Newton systems)
// In-place LDL^T of the row-packed lower triangle L (row i at tri(i)) with unscaled columns (S_ik = l_ik d_k) and one
// extra row L[nf] holding the right-hand side, which the elimination turns into z = L^-1 g.
// invd[j] receives 1/d_j.  Panels of 8 columns: warp 0 factors a panel entirely in registers
// (rows on lanes, shuffles for the pivot column), then all warps apply the rank-8 update to the
// trailing block — two CTA barriers per panel instead of one or two per column.
#ifndef CAVE_HOST_SIM
// One panel of ldlt_blocked, by one warp: rows j0 + lane (+ 32) in registers, NS = 1 when no row lies beyond j0 + 31.
// Entries above the diagonal (and columns >= pw) are loaded as zero and then left to collect garbage: nothing valid
// ever reads them and they are not stored, which keeps the elimination free of per-element predicates.
template <class TH, class PL, int NS>
CAVE_DEV void ldlt_panel(Ctx& cx, PL L, int nf, PL invd, TH piv_floor, int j0, int pw) {
    constexpr int PB = 8;
    TH a[NS][PB];
    int cmax[NS];                 // row i holds the valid columns c < cmax (its part of the lower triangle / the rhs row)
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int i = j0 + cx.lane + 32 * s;
        const int w = i == nf ? pw : (i - j0 + 1 < pw ? i - j0 + 1 : pw);
        cmax[s] = i <= nf ? w : 0;
        const PL li = L + (tri(i <= nf ? i : nf) + j0);
#pragma unroll
        for (int c = 0; c < PB; ++c) a[s][c] = c < cmax[s] ? (TH)li[c] : (TH)0;
    }
#pragma unroll
    for (int jj = 0; jj < PB; ++jj) {
        if (jj < pw) {
            const TH dj = __shfl_sync(0xffffffffu, a[0][jj], jj);
            const TH inv = fast_rcp(dj > piv_floor ? dj : piv_floor);
            if (cx.lane == 0) invd[j0 + jj] = inv;
            TH pc[PB];
#pragma unroll
            for (int c = jj + 1; c < PB; ++c) pc[c] = __shfl_sync(0xffffffffu, a[0][jj], c);
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const TH f = a[s][jj] * inv;
#pragma unroll
                for (int c = jj + 1; c < PB; ++c) a[s][c] -= f * pc[c];
            }
        }
    }
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int i = j0 + cx.lane + 32 * s;
        const PL li = L + (tri(i <= nf ? i : nf) + j0);
#pragma unroll
        for (int c = 0; c < PB; ++c)
            if (c < cmax[s]) li[c] = a[s][c];
    }
}
#endif

template <class TH, class PL>
CAVE_DEV void ldlt_blocked(Ctx& cx, PL L, int nf, PL invd, TH piv_floor) {
    constexpr int PB = 8;
    if (nf + 1 <= 2 * Ctx::WS || Ctx::WS == 1) {
        for (int j0 = 0; j0 < nf; j0 += PB) {
            const int pw = nf - j0 < PB ? nf - j0 : PB;
            if (cx.warp == 0) {
#ifdef CAVE_HOST_SIM
                // single-thread restatement of the panel factorisation
                for (int jj = 0; jj < pw; ++jj) {
                    const int j = j0 + jj;
                    TH dj = L[tri(j) + j];
                    const TH inv = (TH)1 / (dj > piv_floor ? dj : piv_floor);
                    invd[j] = inv;
                    for (int i = j + 1; i <= nf; ++i) {
                        const TH f = (TH)L[tri(i) + j] * inv;
                        for (int c = jj + 1; c < pw; ++c)
                            if (j0 + c <= i || i == nf) L[tri(i) + j0 + c] -= f * (TH)L[tri(j0 + c) + j];
                    }
                }
#else
                if (j0 + Ctx::WS <= nf) ldlt_panel<TH, PL, 2>(cx, L, nf, invd, piv_floor, j0, pw);
                else ldlt_panel<TH, PL, 1>(cx, L, nf, invd, piv_floor, j0, pw);
#endif
            }
            cx.sync();
            // rank-pw update of the trailing block: rows over warps, k over lanes
            const int t0 = j0 + pw;
            if (t0 <= nf - 1) {
                for (int kc = t0; kc <= nf - 1; kc += Ctx::WS) {
                    const int k = kc + cx.lane;
                    const bool kin = k <= nf - 1;
                    TH pk[PB];
#pragma unroll
                    for (int c = 0; c < PB; ++c) pk[c] = (kin && c < pw) ? (TH)L[tri(k) + j0 + c] * (TH)invd[j0 + c] : (TH)0;
                    for (int i = kc + cx.warp; i <= nf; i += cx.nwarp) {
                        const PL li = L + tri(i);
                        if (kin && (k <= i || i == nf)) {
                            TH x = li[k];
                            TH f[PB];
#pragma unroll
                            for (int c = 0; c < PB; ++c) f[c] = c < pw ? (TH)li[j0 + c] : (TH)0;
#pragma unroll
                            for (int c = 0; c < PB; ++c) x -= f[c] * pk[c];
                            li[k] = x;
                        }
                    }
                }
            }
            cx.sync();
        }
        return;
    }
    // generic path (nf >= 64): one column at a time
    for (int j = 0; j < nf; ++j) {
        cx.sync();
        TH dj = L[tri(j) + j];
        const TH inv = (TH)1 / (dj > piv_floor ? dj : piv_floor);
        if (cx.tid == 0) invd[j] = inv;
        for (int i = j + 1 + cx.warp; i <= nf; i += cx.nwarp) {
            const TH lij = (TH)L[tri(i) + j] * inv;
            const int kend = i < nf ? i : nf - 1;
            for (int k = j + 1 + cx.lane; k <= kend; k += Ctx::WS) L[tri(i) + k] -= lij * (TH)L[tri(k) + j];
        }
    }
    cx.sync();
}

// ------------------------------------------------------------------ instance description
struct Instance {
    const float* A;         // this instance's rows, [m_max, d] row-major (global)
    const gen_t* gen;       // general rows: (row index, nnz, offset in the packed CSR, 0), ascending row
    const uint8_t* ctype;   // [d] singleton cone type per coordinate            (from the pack)
    const float* avg;       // [d] average unit normal (src/cave.py:222-228)     (from the pack)
    int d, ngen, gen_nnz, nvalid, nsingc;
    // packed CSR of the general rows written by the scan kernel (valid iff csr_ok & 1; bit 1: all int8)
    int csr_ok;
    const hash_t* ghash;    // indexed by row: hash(row), hash(-row)   (general rows only)
    const uint16_t* pcol;
    const float* pval;
    float maxl1, maxl2;     // max ||a_i||_1, max ||a_i||_2^2 over the general rows
    // cached setup block of the pack (layout.cuh SetupBlock) or nullptr; its header holds the byte offsets of its arrays
    const char* setup;
    // this instance's warm-start slot (layout.cuh warm_slot_bytes) or nullptr; it holds at most warm_cap variables.
    // warm_from_slot = false: start from zero all the same (the cold re-solve after a failed warm start) but store the result.
    char* warm;
    int warm_cap;
    bool warm_from_slot;
};

template <class T>
struct Result {
    T* r;          // [d] r = c - B^T nu at the solution; the residual is q = psi(r)
    int iters;
    int status;
};

// ------------------------------------------------------------------ Newton path
template <class T, class TH, class TC, bool HOT>
struct NewtonWork {
    int d, mB, nv;
    HPtr<TC, HOT> c;                              // c = sign * pred, exact in the I/O dtype
    HPtr<T, HOT> r;
    HPtr<uint8_t, HOT> ctype;
    int* rptr; uint16_t* rcol; void* rval;       // CSR of the general rows (values float, or int8 if i8)
    bool i8;
    int* grow;                                    // general row -> row index in A
    uint8_t* rtype;                               // 0 bounded, 1 free (merged +-), 2 dropped
    int* vrow;                                    // variable -> CSR row
    HPtr<uint8_t, HOT> vfree;                     // variable is sign-free
    int* cptr; uint16_t* crow; void* cval;       // CSC over variables
    HPtr<T, HOT> nu, g, dir, nut;
    HPtr<T, HOT> wmax;                            // [32] per-warp partial maxima
    HPtr<int, HOT> flist;                         // free-set variable ids
    HPtr<int, HOT> fpos;                          // variable -> position in flist or -1
    int* cur;                                     // [d] CSC fill cursors (setup only)
    HPtr<uint8_t, HOT> wflag;                     // [d] psi'(r_k) currently folded into H
    HPtr<uint8_t, HOT> act;                       // [d] psi'(r_k) of the last evaluated point
    HPtr<uint16_t, HOT> flipk;                    // [d] coordinates whose activity changed (bit 15: now active)
    HPtr<int, HOT> fcnt;                          // [1] length of flipk, zero between Hessian updates
    HPtr<TH, HOT> H;                              // [nv, nv] lower triangle of B W B^T, kept up to date
    HPtr<int, HOT> Hi;                            // ... as exact 32-bit integers when the rows are int8 (i8)
    HPtr<TH, HOT> L;                              // [(nf+1), ldl] LDL^T work array with the rhs as last row
    HPtr<TH, HOT> xs;                             // scratch; reciprocal pivots 1/d_j live at xs + nv + 2
};

template <class VT, class T, class TH, class TC, bool HOT>
CAVE_DEV void nw_eval2_t(Ctx& cx, const NewtonWork<T, TH, TC, HOT>& W, HPtr<T, HOT> nu, HPtr<T, HOT> rout, T& f, T& extra) {
    const VT* cval = (const VT*)W.cval;
    T acc = (T)0;
    for (int k = cx.tid; k < W.d; k += cx.nthr) {
        T rk = (T)(TC)W.c[k];
        const int e1 = W.cptr[k + 1];
        // four gathers in flight per thread (the shared-memory accessors are ordered, so the compiler will not
        // overlap them by itself); entries past the column end are read as 0 * nu[0]: the subtraction order and
        // the result are those of the plain loop
        for (int e = W.cptr[k]; e < e1; e += 4) {
            const bool p1 = e + 1 < e1, p2 = e + 2 < e1, p3 = e + 3 < e1;
            const int i0 = W.crow[e], i1 = p1 ? W.crow[e + 1] : 0, i2 = p2 ? W.crow[e + 2] : 0, i3 = p3 ? W.crow[e + 3] : 0;
            const T v0 = (T)cval[e], v1 = p1 ? (T)cval[e + 1] : (T)0, v2 = p2 ? (T)cval[e + 2] : (T)0, v3 = p3 ? (T)cval[e + 3] : (T)0;
            const T n0 = nu[i0], n1 = nu[i1], n2 = nu[i2], n3 = nu[i3];
            rk -= v0 * n0; rk -= v1 * n1; rk -= v2 * n2; rk -= v3 * n3;
        }
        // the array holds q = psi(r) (all that the gradient and the epilogue need; psi is idempotent) and the
        // activity flag psi'(r) goes to its own byte array for the Hessian update
        const int t = (int)(uint8_t)W.ctype[k];
        const bool on = psi_active(rk, t);
        const T q = on ? rk : (T)0;
        rout[k] = q;
        W.act[k] = (uint8_t)(on ? 1 : 0);
        acc += q * q;
    }
    cx.block_sum2(acc, extra);
    f = (T)0.5 * acc;
}
template <class T, class TH, class TC, bool HOT>
CAVE_DEV void nw_eval2(Ctx& cx, const NewtonWork<T, TH, TC, HOT>& W, HPtr<T, HOT> nu, HPtr<T, HOT> rout, T& f, T& extra) {
    if (W.i8) nw_eval2_t<int8_t>(cx, W, nu, rout, f, extra); else nw_eval2_t<float>(cx, W, nu, rout, f, extra);
}

// g = -B psi(r), and in the same pass the projected-gradient fixed-point residual
// max_v |nu_v - P(nu_v - g_v)| (returned to every thread; one barrier in total)
template <class VT, class T, class TH, class TC, bool HOT>
CAVE_DEV T nw_grad_t(Ctx& cx, const NewtonWork<T, TH, TC, HOT>& W, HPtr<T, HOT> r, HPtr<T, HOT> g, HPtr<T, HOT> nu) {
    const VT* rval = (const VT*)W.rval;
    T wres = (T)0;
    for (int v = cx.warp; v < W.nv; v += cx.nwarp) {
        int row = W.vrow[v];
        T acc = (T)0;
        int e = W.rptr[row] + cx.lane;
        const int e1 = W.rptr[row + 1];
        for (; e < e1; e += 4 * Ctx::WS) {                     // guarded: up to four gathers in flight per lane, same order
            const bool p1 = e + Ctx::WS < e1, p2 = e + 2 * Ctx::WS < e1, p3 = e + 3 * Ctx::WS < e1;
            const int k0 = W.rcol[e], k1 = p1 ? (int)W.rcol[e + Ctx::WS] : 0, k2 = p2 ? (int)W.rcol[e + 2 * Ctx::WS] : 0, k3 = p3 ? (int)W.rcol[e + 3 * Ctx::WS] : 0;
            const T v0 = (T)rval[e], v1 = p1 ? (T)rval[e + Ctx::WS] : (T)0, v2 = p2 ? (T)rval[e + 2 * Ctx::WS] : (T)0, v3 = p3 ? (T)rval[e + 3 * Ctx::WS] : (T)0;
            const T r0 = r[k0], r1 = r[k1], r2 = r[k2], r3 = r[k3];          // r holds psi(r) already (nw_eval2)
            acc += v0 * r0; acc += v1 * r1; acc += v2 * r2; acc += v3 * r3;
        }
        acc = cx.warp_sum(acc);
        const T gv = -acc, nv_ = nu[v];
        if (cx.lane == 0) g[v] = gv;
        T t = nv_ - gv;
        if (!(uint8_t)W.vfree[v] && t < (T)0) t = (T)0;
        const T w = cabs(nv_ - t);
        wres = w > wres ? w : wres;
    }
    if (cx.lane == 0) W.wmax[cx.warp] = wres;
    cx.sync();
    T res = (T)0;
    for (int w2 = 0; w2 < cx.nwarp; ++w2) { const T x = W.wmax[w2]; res = x > res ? x : res; }
    return res;
}
template <class T, class TH, class TC, bool HOT>
CAVE_DEV T nw_grad(Ctx& cx, const NewtonWork<T, TH, TC, HOT>& W, HPtr<T, HOT> r, HPtr<T, HOT> g, HPtr<T, HOT> nu) {
    return W.i8 ? nw_grad_t<int8_t>(cx, W, r, g, nu) : nw_grad_t<float>(cx, W, r, g, nu);
}

// Fold the columns whose activity psi'(r_k) changed since the last call into H = B W B^T
// (lower triangle over ALL variables): H += +-b_k b_k^T with shared-memory atomics.  After the
// first iterations only a handful of coordinates change sign, so this is almost free.
template <class VT, class T, class TH, class TC, bool HOT>
CAVE_DEV void nw_hessian_update_t(Ctx& cx, const NewtonWork<T, TH, TC, HOT>& W, HPtr<T, HOT> r) {
    const VT* cval = (const VT*)W.cval;
    // phase 1: the coordinates whose activity changed, compacted into a list (order irrelevant: the integer
    // Hessian is exact, and a float Hessian was order dependent before as well)
    for (int k0 = 0; k0 < W.d; k0 += cx.nthr) {
        const int k = k0 + cx.tid;
        bool flip = false;
        uint8_t now = 0;
        if (k < W.d) {
            now = (uint8_t)W.act[k];
            flip = now != (uint8_t)W.wflag[k];
            if (flip) W.wflag[k] = now;
        }
        const unsigned m = cx.ballot(flip);
        if (m) {
            int base = 0;
            if (cx.lane == 0) base = W.fcnt.fetch_add(0, cx.popc(m));
            base = cx.shfl(base, 0);
            if (flip) W.flipk[base + cx.lanes_below(m)] = (uint16_t)(k | (now ? 0x8000 : 0));
        }
    }
    cx.sync();
    const int n = W.fcnt[0];
    // phase 2: G threads per flipped column (G a power of two, about nthr / n) share its pairs, so a handful
    // of flips late in the solve still occupies whole warps and thousands of them in the first iterations
    // are spread one per thread
    int G = 1;
    while (G < Ctx::WS && n * (G * 2) <= cx.nthr) G *= 2;
    const int sub = cx.tid & (G - 1);
    for (int fi = cx.tid / G; fi < n; fi += cx.nthr / G) {
        const int kk = (int)(uint16_t)W.flipk[fi];
        const int k = kk & 0x3fff;
        const int s = W.cptr[k], cnt = W.cptr[k + 1] - s;
        const int sgi = (kk & 0x8000) ? 1 : -1;
        // pair p <-> (e1 >= e2): walk the rows of the triangle, starting where this thread's first pair lies
        int e1 = 0, rowstart = 0;
        const int npairs = (cnt * (cnt + 1)) >> 1;
        for (int p = sub; p < npairs; p += G) {
            while (rowstart + e1 + 1 <= p) { rowstart += e1 + 1; ++e1; }
            const int e2 = p - rowstart;
            const int a = W.crow[s + e1], b = W.crow[s + e2];
            const int hi = a > b ? a : b, lo = a > b ? b : a;
            if (sizeof(VT) == 1) W.Hi.atomic_add(tri(hi) + lo, sgi * (int)cval[s + e1] * (int)cval[s + e2]);
            else W.H.atomic_add(tri(hi) + lo, ((TH)sgi * (TH)cval[s + e1]) * (TH)cval[s + e2]);
        }
    }
    cx.sync();
    if (cx.tid == 0) W.fcnt[0] = 0;       // invariant: zero between calls (the next use is several barriers away)
}
template <class T, class TH, class TC, bool HOT>
CAVE_DEV void nw_hessian_update(Ctx& cx, const NewtonWork<T, TH, TC, HOT>& W, HPtr<T, HOT> r) {
    if (W.i8) nw_hessian_update_t<int8_t>(cx, W, r); else nw_hessian_update_t<float>(cx, W, r);
}

// Inclusive scan of x[0..n) in place by warp 0 (callers synchronise before and after).
CAVE_DEV void warp0_inclusive_scan(Ctx& cx, int* x, int n) {
    if (cx.warp != 0) return;
    int carry = 0;
    for (int i0 = 0; i0 < n; i0 += Ctx::WS) {
        const int i = i0 + cx.lane;
        int v = i < n ? x[i] : 0;
#ifndef CAVE_HOST_SIM
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int u = __shfl_up_sync(0xffffffffu, v, o); if (cx.lane >= o) v += u; }
#endif
        v += carry;
        if (i < n) x[i] = v;
        carry = cx.shfl(v, Ctx::WS - 1);
    }
}

// Inclusive scan of x[0..n) in place by the whole CTA: every warp scans a contiguous segment, the segment totals
// go through scr[nwarp].  Callers synchronise before; ends with a barrier.
CAVE_DEV void block_inclusive_scan(Ctx& cx, int* x, int n, int* scr) {
    if (Ctx::WS == 1 || n < 8 * Ctx::WS) {
        warp0_inclusive_scan(cx, x, n);
        cx.sync();
        return;
    }
#ifndef CAVE_HOST_SIM
    const int seg = ((n + cx.nwarp - 1) / cx.nwarp + 31) & ~31;
    const int s0 = cx.warp * seg, s1 = s0 + seg < n ? s0 + seg : n;
    int carry = 0;
    for (int i0 = s0; i0 < s1; i0 += 32) {
        const int i = i0 + cx.lane;
        int v = i < s1 ? x[i] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, v, o); if (cx.lane >= o) v += u; }
        v += carry;
        if (i < s1) x[i] = v;
        carry = __shfl_sync(0xffffffffu, v, 31);
    }
    if (cx.lane == 0) scr[cx.warp] = carry;
    cx.sync();
    int off = 0;
    for (int w = 0; w < cx.warp; ++w) off += scr[w];
    if (off) for (int i = s0 + cx.lane; i < s1; i += 32) x[i] += off;
    cx.sync();
#endif
}

// Setup of one structured instance: merge +- rows, build the variable list, bring the CSR of the kept
// general rows into the arena (from the scan kernel's pack, or by reading the rows of A when the pack
// could not hold them) and build the CSC.  HOT selects shared-memory-only allocation for the arrays of
// the Newton iteration.  Returns false if the instance does not fit (ar.hot_overflow tells which side).
template <class T, class TH, class TC, bool HOT>
CAVE_DEV bool nw_setup(Ctx& cx, const Instance& in, Arena& ar, NewtonWork<T, TH, TC, HOT>& W, T* maxrow_l1, T* maxrow_l2sq) {
    const int d = in.d, mB = in.ngen;
    W.d = d; W.mB = mB;
    // hot: vectors of the iteration
    W.nu = ar.geth<HOT, T>(mB + 1); W.g = ar.geth<HOT, T>(mB + 1); W.dir = ar.geth<HOT, T>(mB + 1); W.nut = ar.geth<HOT, T>(mB + 1);
    W.xs = ar.geth<HOT, TH>(2 * mB + 6);          // reciprocal pivots (and scratch)
    W.wmax = ar.geth<HOT, T>(32);
    W.flist = ar.geth<HOT, int>(mB + 2);
    W.fpos = ar.geth<HOT, int>(mB + 2);
    W.vfree = ar.geth<HOT, uint8_t>(mB + 1);
    W.wflag = ar.geth<HOT, uint8_t>(d + 1);
    W.act = ar.geth<HOT, uint8_t>(d + 1);
    W.flipk = ar.geth<HOT, uint16_t>(d + 1);
    W.fcnt = ar.geth<HOT, int>(4);
    HPtr<uint8_t, HOT> ctype_s = ar.geth<HOT, uint8_t>(d + 1);
    W.rptr = ar.get<int>(mB + 2);
    W.vrow = ar.get<int>(mB + 1);
    // cold: sparse structure first (it is read in every iteration), then the setup-only scratch, which takes
    // whatever shared memory is left and otherwise lives in the global slot
    W.cptr = ar.get<int>(d + 2);
    // setup-only scratch lives in r (free until the first evaluation writes it) when it fits there
    SubArena sa; sa.init((char*)W.r.raw(), (size_t)d * sizeof(T));
    uint64_t* hpos = sa.get<uint64_t>(ar, mB + 1);
    uint64_t* hneg = sa.get<uint64_t>(ar, mB + 1);
    int* goff = sa.get<int>(ar, mB + 2);          // row offsets in the source CSR (pack, or the one built here)
    int* gcnt = sa.get<int>(ar, mB + 2);          // non-zeros per general row
    W.grow = sa.get<int>(ar, mB + 1);
    int* cand = sa.get<int>(ar, mB + 1);
    W.cur = sa.get<int>(ar, d + 1);
    W.rtype = sa.get<uint8_t>(ar, mB + 1);
    if (ar.overflow) return false;
    for (int k0 = 0; k0 < d; k0 += 8 * cx.nthr) {       // global loads first, then the (ordered) shared stores
        uint8_t t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int k = k0 + u * cx.nthr + cx.tid; t[u] = k < d ? in.ctype[k] : (uint8_t)0; }
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int k = k0 + u * cx.nthr + cx.tid; if (k < d) { ctype_s[k] = t[u]; W.wflag[k] = 0; } }
    }
    W.ctype = ctype_s;
    if (cx.tid == 0) W.fcnt[0] = 0;
#ifndef CAVE_NO_SETUP_CACHE
    if (in.setup && ((const int*)in.setup)[0] == 1) {
        // ---- cached setup (emitted once per pack by the setup kernel): everything below is a copy-in
        const int* hdr = (const int*)in.setup;
        const int nv = hdr[1], nnzc = hdr[2];
        W.nv = nv; W.i8 = true;
        W.Hi = ar.geth<HOT, int>((size_t)tri(nv) + 1);
        W.L = ar.geth<HOT, TH>((size_t)tri(nv + 2) + 1);
        W.crow = ar.get<uint16_t>(nnzc + 1);
        W.cval = ar.get<int8_t>(nnzc + 1);
        W.rcol = ar.get<uint16_t>(nnzc + 8);
        W.rval = ar.get<int8_t>(nnzc + 4);
        if (ar.overflow) return false;
        *maxrow_l1 = (T)in.maxl1; *maxrow_l2sq = (T)in.maxl2;
        const uint8_t* c_vfree = (const uint8_t*)(in.setup + hdr[3]);
        const int* c_rptr = (const int*)(in.setup + hdr[4]);
        const int* c_cptr = (const int*)(in.setup + hdr[5]);
        for (int v = cx.tid; v <= nv; v += cx.nthr) { W.rptr[v] = c_rptr[v]; if (v < nv) { W.vfree[v] = c_vfree[v]; W.vrow[v] = v; } }
        for (int k0 = 0; k0 <= d; k0 += 8 * cx.nthr) {
            int t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) { const int k = k0 + u * cx.nthr + cx.tid; t[u] = k <= d ? c_cptr[k] : 0; }
#pragma unroll
            for (int u = 0; u < 8; ++u) { const int k = k0 + u * cx.nthr + cx.tid; if (k <= d) W.cptr[k] = t[u]; }
        }
        // the four non-zero arrays: 16-byte granules (the block's arrays are 16-byte aligned and padded; so are the arena's)
        const int n2 = (nnzc * 2 + 15) >> 4, n1 = (nnzc + 15) >> 4;
        copy_granules((G16*)W.rcol, (const G16*)(in.setup + hdr[6]), n2, cx.tid, cx.nthr);
        copy_granules((G16*)W.crow, (const G16*)(in.setup + hdr[7]), n2, cx.tid, cx.nthr);
        copy_granules((G16*)W.rval, (const G16*)(in.setup + hdr[8]), n1, cx.tid, cx.nthr);
        copy_granules((G16*)W.cval, (const G16*)(in.setup + hdr[9]), n1, cx.tid, cx.nthr);
        for (uint32_t t = cx.tid; t < tri(nv); t += cx.nthr) W.Hi[t] = 0;
        cx.sync();
        return true;
    }
#endif
    for (int i = cx.tid; i < mB; i += cx.nthr) {
        gen_t g = in.gen[i]; W.grow[i] = g.x; gcnt[i] = g.y; goff[i] = g.z;
        if (in.csr_ok) { hash_t h = in.ghash[g.x]; hpos[i] = h.x; hneg[i] = h.y; }
    }
    cx.sync();
    const uint16_t* mcol = in.pcol;     // where the merge verification reads the rows from
    const float* mval = in.pval;
    if (!in.csr_ok && !in.A) { ar.overflow = true; return false; }     // rows neither packed nor resident
    if (!in.csr_ok) {
        // offsets of the CSR built here = exclusive scan of the counts
        if (cx.tid == 0) goff[0] = 0;
        for (int i = cx.tid; i < mB; i += cx.nthr) goff[i + 1] = gcnt[i];
        cx.sync();
        warp0_inclusive_scan(cx, goff + 1, mB);
        cx.sync();
        // fallback: build the CSR of ALL general rows from A (one warp per row, ballot compaction keeps
        // the columns sorted), computing the hashes and norms the scan kernel could not deliver
        W.rcol = ar.get<uint16_t>(in.gen_nnz + 8);
        float* rvalf = ar.get<float>(in.gen_nnz + 4);
        W.rval = rvalf;
        if (ar.overflow) return false;
        T l1max = (T)0, l2max = (T)0;
        for (int i = cx.warp; i < mB; i += cx.nwarp) {
            const float* row = in.A + (size_t)W.grow[i] * d;
            int off = goff[i];
            uint64_t hp = 0, hn = 0;
            float l1 = 0.f, l2 = 0.f;
            for (int k0 = 0; k0 < d; k0 += Ctx::WS * 8) {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    int k = k0 + u * Ctx::WS + cx.lane;
                    v[u] = k < d ? ld_stream(row + k) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    int k = k0 + u * Ctx::WS + cx.lane;
                    bool nz = v[u] != 0.f;
                    unsigned m = cx.ballot(nz);
                    if (nz) {
                        int p = off + cx.lanes_below(m);
                        W.rcol[p] = (uint16_t)k; rvalf[p] = v[u];
                        union { float f; uint32_t u; } cv; cv.f = v[u];
                        hp += mix64(((uint64_t)k << 32) | cv.u);
                        hn += mix64(((uint64_t)k << 32) | (cv.u ^ 0x80000000u));
                        l1 += v[u] < 0.f ? -v[u] : v[u];
                        l2 += v[u] * v[u];
                    }
                    off += cx.popc(m);
                }
            }
            hp = cx.warp_sum_u64(hp); hn = cx.warp_sum_u64(hn);
            l1 = cx.warp_sum(l1); l2 = cx.warp_sum(l2);
            if (cx.lane == 0) { hpos[i] = hp; hneg[i] = hn; }
            if ((T)l1 > l1max) l1max = (T)l1;
            if ((T)l2 > l2max) l2max = (T)l2;
        }
        cx.block_max2(l1max, l2max);    // (barriers inside make the CSR visible)
        *maxrow_l1 = l1max; *maxrow_l2sq = l2max;
        mcol = W.rcol; mval = rvalf;
    } else {
        *maxrow_l1 = (T)in.maxl1; *maxrow_l2sq = (T)in.maxl2;
    }
    // merge b_j = -b_i : cand[i] = smallest j != i with row_j == -row_i (hash match, then an exact
    // comparison); merged iff the choice is mutual.  One warp per row.
    for (int i = cx.warp; i < mB; i += cx.nwarp) {
        const int pi = goff[i], ni = gcnt[i];
        const uint64_t want = hneg[i];
        int c0 = -1;
        for (int j0 = 0; j0 < mB && c0 < 0; j0 += Ctx::WS) {
            const int j = j0 + cx.lane;
            bool hit = j < mB && j != i && hpos[j] == want && gcnt[j] == ni;
            unsigned m = cx.ballot(hit);
            while (m && c0 < 0) {
#ifdef CAVE_HOST_SIM
                const int jj = j0;
#else
                const int jj = j0 + __ffs(m) - 1;
#endif
                const int pj = goff[jj];
                bool ok = true;
                for (int e0 = 0; e0 < ni; e0 += 4 * Ctx::WS) {     // all loads of a batch issued before any compare
                    uint16_t ci[4], cj[4]; float vi[4], vj[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int e = e0 + u * Ctx::WS + cx.lane;
                        const bool in_row = e < ni;
                        ci[u] = in_row ? mcol[pi + e] : (uint16_t)0; cj[u] = in_row ? mcol[pj + e] : (uint16_t)0;
                        vi[u] = in_row ? mval[pi + e] : 0.f; vj[u] = in_row ? mval[pj + e] : 0.f;
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) ok = ok & (ci[u] == cj[u]) & (vi[u] == -vj[u]);
                }
                const unsigned bad = cx.ballot(!ok);
                if (!bad) c0 = jj;
                m &= m - 1;
            }
        }
        if (cx.lane == 0) cand[i] = c0;
    }
    cx.sync();
    for (int i = cx.tid; i < mB; i += cx.nthr) {
        int j = cand[i];
        W.rtype[i] = (j >= 0 && cand[j] == i) ? (i < j ? 1 : 2) : 0;
    }
    cx.sync();
    // variables = rows that were not dropped (ordered compaction by warp 0).  With a packed CSR only the
    // kept rows are copied in (rptr over variables, vrow = identity); in fallback mode the CSR holds every
    // general row and vrow maps a variable to its row.
    if (cx.warp == 0) {
        int nvb = 0, nz = 0;
        for (int i0 = 0; i0 < mB; i0 += Ctx::WS) {
            const int i = i0 + cx.lane;
            const bool keep = i < mB && W.rtype[i] != 2;
            const unsigned m = cx.ballot(keep);
            if (keep) {
                const int v = nvb + cx.lanes_below(m);
                W.vrow[v] = i; W.vfree[v] = (uint8_t)(W.rtype[i] == 1);
                nz += gcnt[i];
            }
            nvb += cx.popc(m);
        }
        nz = cx.warp_sum(nz);
        if (cx.lane == 0) { W.flist[0] = nvb; W.flist[1] = nz; }   // broadcast through memory
    }
    cx.sync();
    W.nv = W.flist[0];
    const int nnzc = W.flist[1];
    cx.sync();
    const int nv = W.nv;
    // Integer-valued rows (every shipped model) are kept as int8, and their Hessian as exact int32.
    W.i8 = (in.csr_ok & 3) == 3;
    if (W.i8) W.Hi = ar.geth<HOT, int>((size_t)tri(nv) + 1);      // row-packed lower triangles
    else W.H = ar.geth<HOT, TH>((size_t)tri(nv) + 1);
    W.L = ar.geth<HOT, TH>((size_t)tri(nv + 2) + 1);
    // the CSC feeds eval (several times per iteration) and the Hessian update, the CSR only the gradient:
    // the CSC gets shared memory first.
    W.crow = ar.get<uint16_t>(nnzc + 1);
    if (W.i8) W.cval = ar.get<int8_t>(nnzc + 1); else W.cval = ar.get<float>(nnzc + 1);
    if (in.csr_ok) {
        W.rcol = ar.get<uint16_t>(nnzc + 8);
        if (W.i8) W.rval = ar.get<int8_t>(nnzc + 4); else W.rval = ar.get<float>(nnzc + 4);
    }
    if (ar.overflow) return false;
    if (in.csr_ok) {
        // rptr over variables, then one warp per kept row copies its non-zeros from the pack
        if (cx.tid == 0) W.rptr[0] = 0;
        for (int v = cx.tid; v < nv; v += cx.nthr) W.rptr[v + 1] = gcnt[W.vrow[v]];
        cx.sync();
        warp0_inclusive_scan(cx, W.rptr + 1, nv);
        cx.sync();
        for (int v = cx.warp; v < nv; v += cx.nwarp) {
            const int src = goff[W.vrow[v]], dst = W.rptr[v], n = W.rptr[v + 1] - dst;
            for (int e0 = 0; e0 < n; e0 += 8 * Ctx::WS) {       // eight loads per lane in flight
                uint16_t cc[8]; float vv[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int e = e0 + u * Ctx::WS + cx.lane;
                    cc[u] = e < n ? in.pcol[src + e] : (uint16_t)0; vv[u] = e < n ? in.pval[src + e] : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int e = e0 + u * Ctx::WS + cx.lane;
                    if (e < n) {
                        W.rcol[dst + e] = cc[u];
                        if (W.i8) ((int8_t*)W.rval)[dst + e] = (int8_t)vv[u]; else ((float*)W.rval)[dst + e] = vv[u];
                    }
                }
            }
        }
        cx.sync();
        for (int v = cx.tid; v < nv; v += cx.nthr) W.vrow[v] = v;
    } else {
        for (int i = cx.tid; i < mB; i += cx.nthr) W.rptr[i] = goff[i];
        if (cx.tid == 0) W.rptr[mB] = goff[mB - 1] + gcnt[mB - 1];
    }
    // CSC: count, scan, fill with a cursor, then order every column by variable id
    for (int k = cx.tid; k <= d; k += cx.nthr) W.cptr[k] = 0;
    if (W.i8) for (uint32_t t = cx.tid; t < tri(nv); t += cx.nthr) W.Hi[t] = 0;
    else for (uint32_t t = cx.tid; t < tri(nv); t += cx.nthr) W.H[t] = (TH)0;
    cx.sync();
    for (int v = cx.warp; v < nv; v += cx.nwarp) {
        int row = W.vrow[v];
        for (int e = W.rptr[row] + cx.lane; e < W.rptr[row + 1]; e += Ctx::WS) cx.atomic_add(&W.cptr[W.rcol[e] + 1], 1);
    }
    cx.sync();
    block_inclusive_scan(cx, W.cptr + 1, d, (int*)W.wmax.raw());      // wmax (32 doubles) is idle during setup
    for (int k = cx.tid; k < d; k += cx.nthr) W.cur[k] = W.cptr[k];
    cx.sync();
    for (int v = cx.warp; v < nv; v += cx.nwarp) {
        int row = W.vrow[v];
        for (int e = W.rptr[row] + cx.lane; e < W.rptr[row + 1]; e += Ctx::WS) {
            int p = cx.atomic_add(&W.cur[W.rcol[e]], 1);
            W.crow[p] = (uint16_t)v;
            if (W.i8) ((int8_t*)W.cval)[p] = ((const int8_t*)W.rval)[e]; else ((float*)W.cval)[p] = ((const float*)W.rval)[e];
        }
    }
    cx.sync();
    for (int k = cx.tid; k < d; k += cx.nthr) {      // insertion sort: deterministic summation order
        int s = W.cptr[k], e = W.cptr[k + 1];
        if (e - s <= 64)
            for (int a = s + 1; a < e; ++a) {
                uint16_t rr = W.crow[a]; int b = a - 1;
                if (W.i8) {
                    int8_t* cv = (int8_t*)W.cval; int8_t vv = cv[a];
                    while (b >= s && W.crow[b] > rr) { W.crow[b + 1] = W.crow[b]; cv[b + 1] = cv[b]; --b; }
                    W.crow[b + 1] = rr; cv[b + 1] = vv;
                } else {
                    float* cv = (float*)W.cval; float vv = cv[a];
                    while (b >= s && W.crow[b] > rr) { W.crow[b + 1] = W.crow[b]; cv[b + 1] = cv[b]; --b; }
                    W.crow[b + 1] = rr; cv[b + 1] = vv;
                }
            }
    }
    cx.sync();
    return true;
}

// ------------------------------------------------------------------ warm start (layout.cuh warm_slot_bytes)
// A slot is only ever a starting guess: another CTA of the same launch may write it while it is read (an index may hold an
// instance twice), so nothing read from it is trusted beyond what the Newton iteration itself checks.  The helpers run
// once per instance and are not inlined, like copy_granules, so they add nothing to the registers of the iteration.
#ifdef CAVE_HOST_SIM
#define CAVE_NOINLINE inline
#else
#define CAVE_NOINLINE static __device__ __noinline__
#endif
struct alignas(16) WarmHeader { int32_t valid, nv; uint32_t tag, pad; };

// Hash of the variable -> row map (length and first column of every variable's row) and of the sign-free flags, computed
// by every warp on its own (at most a few hundred variables): the same value on every thread without a barrier.
CAVE_DEV uint32_t warm_tag(Ctx& cx, int nv, const uint8_t* vfree, const int* rptr, const int* vrow, const uint16_t* rcol) {
    uint64_t h = 0;
    for (int v = cx.lane; v < nv; v += Ctx::WS) {
        const int row = vrow[v], s = rptr[row], n = rptr[row + 1] - s;
        h += mix64(((uint64_t)v << 40) ^ ((uint64_t)vfree[v] << 36) ^ ((uint64_t)(uint32_t)n << 16) ^ (uint64_t)(n > 0 ? rcol[s] : 0));
    }
    h = cx.warp_sum_u64(h);
    return (uint32_t)(h ^ (h >> 32)) ^ (uint32_t)nv;
}

// nu <- the slot's multipliers if the slot is valid for this instance (same nv and tag), with non-finite entries replaced by
// zero and bounded variables clamped to >= 0; nu <- 0 otherwise.  Returns 1 if the slot was used (the same on every
// thread: decided by thread 0 and broadcast through *flag, a word of shared memory, which is left at 1 or 0 accordingly).
// Ends with a barrier.
CAVE_NOINLINE int warm_read(Ctx cx, const char* slot, int nv, const uint8_t* vfree, const int* rptr, const int* vrow,
                            const uint16_t* rcol, double* nu, int* flag) {
    const uint32_t tag = warm_tag(cx, nv, vfree, rptr, vrow, rcol);
    if (cx.tid == 0) {
#ifdef CAVE_HOST_SIM
        const WarmHeader h = *(const WarmHeader*)slot;
#else
        const int4 hv = __ldcg((const int4*)slot);
        WarmHeader h; h.valid = hv.x; h.nv = hv.y; h.tag = (uint32_t)hv.z;
#endif
        *flag = (h.valid == 1 && h.nv == nv && h.tag == tag) ? 1 : 0;
    }
    cx.sync();
    const int use = *flag;
    const double* val = (const double*)(slot + sizeof(WarmHeader));
    for (int v = cx.tid; v < nv; v += cx.nthr) {
        double x = 0.0;
        if (use) {
#ifdef CAVE_HOST_SIM
            x = val[v];
#else
            x = __ldcg(val + v);
#endif
            if (!(x - x == 0.0)) x = 0.0;                  // NaN / Inf
            if (!vfree[v] && x < 0.0) x = 0.0;
        }
        nu[v] = x;
    }
    cx.sync();
    return use;
}

// Stores nu as the slot's multipliers: the values first, the header after a barrier (a reader that sees the header of this
// write and older values still only gets a starting guess).
CAVE_NOINLINE void warm_write(Ctx cx, char* slot, int nv, const uint8_t* vfree, const int* rptr, const int* vrow,
                              const uint16_t* rcol, const double* nu) {
    const uint32_t tag = warm_tag(cx, nv, vfree, rptr, vrow, rcol);
    double* val = (double*)(slot + sizeof(WarmHeader));
    for (int v = cx.tid; v < nv; v += cx.nthr) val[v] = nu[v];
#ifndef CAVE_HOST_SIM
    __threadfence();
#endif
    cx.sync();
    if (cx.tid == 0) {
        WarmHeader h; h.valid = 1; h.nv = nv; h.tag = tag; h.pad = 0;
        *(WarmHeader*)slot = h;
    }
}

template <class T, class TH, class TC, bool HOT, bool WARM>
CAVE_DEV void newton_solve(Ctx& cx, const Instance& in, Arena& ar, HPtr<TC, HOT> c, HPtr<T, HOT> r, T cnorm,
                           const SolveOpts& opt, Result<T>& out) {
    NewtonWork<T, TH, TC, HOT> W;
    W.c = c; W.r = r;
    T l1max, l2max;
    if (!nw_setup<T, TH, TC, HOT>(cx, in, ar, W, &l1max, &l2max)) { out.status = ST_NOSPACE; out.iters = 0; out.r = r.raw(); return; }
    const int nv = W.nv;
    const T scale = (l1max > (T)1 ? l1max : (T)1) * (cnorm > (T)1e-30 ? cnorm : (T)1e-30);
    const T tol = (T)(opt.tol > 0 ? opt.tol : 1e-12) * scale;   // tight: the rnorm < 1e-7 inside-the-cone test depends on it
    const int max_iter = opt.max_iter > 0 ? opt.max_iter : 200;
    const int max_ls = opt.max_ls > 0 ? opt.max_ls : 40;
    // Tikhonov term: relative to the largest possible diagonal entry of B W B^T (max_i ||b_i||^2)
    const TH reg = (sizeof(TH) == 8 ? (TH)1e-11 : (TH)2e-6) * (TH)(l2max > (T)0 ? l2max : (T)1);
    const TH piv_floor = eps_mach<TH>() * (TH)(l2max > (T)0 ? l2max : (T)1);

    // Warm start (WARM: the kernel variant launched with a warm-start buffer; without one, none of this is compiled in):
    // nu from the instance's slot if it holds a solution of this instance.  Whether it did stays in fcnt[1] (a word of
    // shared memory) rather than in a register live through the iteration.
    if (WARM && in.warm && in.warm_from_slot && nv <= in.warm_cap) warm_read(cx, in.warm, nv, W.vfree.raw(), W.rptr, W.vrow, W.rcol, W.nu.raw(), W.fcnt.raw() + 1);
    else {
        if (WARM && in.warm && cx.tid == 0) W.fcnt[1] = 0;
        for (int v = cx.tid; v < nv; v += cx.nthr) W.nu[v] = (T)0;
        cx.sync();
    }
    HPtr<T, HOT> nu = W.nu, nut = W.nut;
    const HPtr<T, HOT> rc = W.r;       // r is updated in place by every trial evaluation
    T f, dummy = (T)0;
    nw_eval2(cx, W, nu, rc, f, dummy);
    int status = ST_ITER_CAP, it = 0, since_best = 0, flat = 0;
    T res_best = (T)1e300;
    for (; it < max_iter; ++it) {
        const T res = nw_grad(cx, W, rc, W.g, nu);
#if defined(CAVE_NW_TRACE) && !defined(CAVE_HOST_SIM)
        if (cx.tid == 0 && it < 40) printf("it %d res %.6e tol %.3e f %.17g res_best %.3e since %d\n", it, (double)res, (double)tol, (double)f, (double)res_best, since_best);
#endif
        if (!(res > tol)) { status = ST_CONVERGED; break; }
        // stagnation at the floating-point floor: the KKT residual is already tiny and has not halved for five
        // iterations (it hovers a hair above the tolerance) -> converged, not an iteration-cap failure
        if (res < (T)0.5 * res_best) { res_best = res; since_best = 0; }
        else if (++since_best >= 5 && res <= (T)8 * tol) { status = ST_CONVERGED; break; }
        const T epsb = res < (T)1e-3 ? res : (T)1e-3;
        // Ordered free list (every variable that is not epsilon-binding).  Every warp evaluates all chunks of
        // 32 variables (a handful of ballots) and writes the slice it owns, so nf is known to every thread
        // without a broadcast and no warp is held up; very wide problems fall back to warp 0.
        int nf = 0;
        const int nchunk = (nv + Ctx::WS - 1) / Ctx::WS;
        if (nchunk <= cx.nwarp) {
            for (int ci = 0; ci < nchunk; ++ci) {
                const int v = ci * Ctx::WS + cx.lane;
                const bool isf = v < nv && !(!(uint8_t)W.vfree[v] && (T)nu[v] <= epsb && (T)W.g[v] > (T)0);
                const unsigned m = cx.ballot(isf);
                if (ci == cx.warp && v < nv) {
                    const int pos = nf + cx.lanes_below(m);
                    W.fpos[v] = isf ? pos : -1;
                    if (isf) W.flist[pos] = v; else W.dir[v] = W.g[v];      // binding set: gradient step
                }
                nf += cx.popc(m);
            }
            nw_hessian_update(cx, W, rc);      // (ends with a barrier: flist / fpos / dir visible too)
        } else {
            if (cx.warp == 0) {
                int nfb = 0;
                for (int v0 = 0; v0 < nv; v0 += Ctx::WS) {
                    const int v = v0 + cx.lane;
                    const bool isf = v < nv && !(!(uint8_t)W.vfree[v] && (T)nu[v] <= epsb && (T)W.g[v] > (T)0);
                    const unsigned m = cx.ballot(isf);
                    if (v < nv) {
                        const int pos = nfb + cx.lanes_below(m);
                        W.fpos[v] = isf ? pos : -1;
                        if (isf) W.flist[pos] = v; else W.dir[v] = W.g[v];
                    }
                    nfb += cx.popc(m);
                }
                if (cx.lane == 0) W.fpos[nv] = nfb;
            }
            nw_hessian_update(cx, W, rc);
            nf = (int)W.fpos[nv];
        }
        // L <- [H_FF + reg I ; g_F^T]
        if (Ctx::WS == 32 && nf <= 2 * Ctx::WS) {
            // the free list in registers (two entries per lane): one gather hop per element instead of two
            const int l = cx.lane;
            const int f0 = l < nf ? (int)W.flist[l] : 0, f1 = l + 32 < nf ? (int)W.flist[l + 32] : 0;
            for (int a = cx.warp; a <= nf; a += cx.nwarp) {
                const HPtr<TH, HOT> la = W.L + tri(a);
                if (a == nf) {
                    if (l < nf) la[l] = (TH)(T)W.g[f0];
                    if (l + 32 < nf) la[l + 32] = (TH)(T)W.g[f1];
                } else {
                    const int fa = (int)W.flist[a];                  // flist ascending => flist[a] >= flist[b]
                    TH h0 = (TH)0, h1 = (TH)0;
                    if (W.i8) {
                        const HPtr<int, HOT> ha = W.Hi + tri(fa);
                        if (l <= a) h0 = (TH)(int)ha[f0];
                        if (l + 32 <= a) h1 = (TH)(int)ha[f1];
                    } else {
                        const HPtr<TH, HOT> ha = W.H + tri(fa);
                        if (l <= a) h0 = (TH)ha[f0];
                        if (l + 32 <= a) h1 = (TH)ha[f1];
                    }
                    if (l <= a) la[l] = h0 + (a == l ? reg : (TH)0);
                    if (l + 32 <= a) la[l + 32] = h1 + (a == l + 32 ? reg : (TH)0);
                }
            }
        } else
        for (int a = cx.warp; a <= nf; a += cx.nwarp) {
            const HPtr<TH, HOT> la = W.L + tri(a);
            if (a == nf) {
                for (int b = cx.lane; b < nf; b += Ctx::WS) la[b] = (TH)(T)W.g[(int)W.flist[b]];
            } else if (W.i8) {
                const HPtr<int, HOT> ha = W.Hi + tri((int)W.flist[a]);          // flist ascending => flist[a] >= flist[b]
                for (int b = cx.lane; b <= a; b += Ctx::WS) la[b] = (TH)(int)ha[(int)W.flist[b]] + (a == b ? reg : (TH)0);
            } else {
                const HPtr<TH, HOT> ha = W.H + tri((int)W.flist[a]);
                for (int b = cx.lane; b <= a; b += Ctx::WS) la[b] = (TH)ha[(int)W.flist[b]] + (a == b ? reg : (TH)0);
            }
        }
        cx.sync();
        const HPtr<TH, HOT> invd = W.xs + (nv + 2);
        ldlt_blocked<TH, HPtr<TH, HOT> >(cx, W.L, nf, invd, piv_floor);
        // back substitution D L^T x = z by warp 0 (column oriented, no reductions, no divisions)
        if (cx.warp == 0) {
            const HPtr<TH, HOT> z = W.L + tri(nf);
#ifndef CAVE_HOST_SIM
            if (nf <= 2 * Ctx::WS) {
                // z, 1/d and the solution stay in registers (two per lane); one shuffle per step broadcasts x_j and the
                // next row of L is fetched while the current one is applied
                const int l = cx.lane;
                TH z0 = l < nf ? (TH)z[l] : (TH)0, z1 = l + 32 < nf ? (TH)z[l + 32] : (TH)0;
                const TH d0 = l < nf ? (TH)invd[l] : (TH)0, d1 = l + 32 < nf ? (TH)invd[l + 32] : (TH)0;
                int j = nf - 1;
                uint32_t tj = tri(j);                       // start of row j; row j - 1 starts j entries earlier
                TH l0 = l < j ? (TH)W.L[tj + l] : (TH)0, l1 = l + 32 < j ? (TH)W.L[tj + l + 32] : (TH)0;
                // rows 32 .. nf-1: x_j comes from the upper register, both halves of z are updated
                for (; j >= 32; --j) {
                    const uint32_t tn = tj - (uint32_t)j;
                    const TH n0 = l < j - 1 ? (TH)W.L[tn + l] : (TH)0;
                    const TH n1 = l + 32 < j - 1 ? (TH)W.L[tn + l + 32] : (TH)0;
                    const TH xj = __shfl_sync(0xffffffffu, z1 * d1, j & 31);
                    if (l == 0) z[j] = xj;                  // the solution overwrites z in place
                    z0 -= l0 * xj; z1 -= l1 * xj;
                    l0 = n0; l1 = n1; tj = tn;
                }
                for (; j >= 0; --j) {
                    const uint32_t tn = tj - (uint32_t)j;
                    const TH n0 = l < j - 1 ? (TH)W.L[tn + l] : (TH)0;
                    const TH xj = __shfl_sync(0xffffffffu, z0 * d0, j);
                    if (l == 0) z[j] = xj;
                    z0 -= l0 * xj;
                    l0 = n0; tj = tn;
                }
                cx.syncwarp();
                if (l < nf) W.dir[(int)W.flist[l]] = (T)(TH)z[l];
                if (l + 32 < nf) W.dir[(int)W.flist[l + 32]] = (T)(TH)z[l + 32];
            } else
#endif
            for (int j = nf - 1; j >= 0; --j) {
                const TH xj = (TH)z[j] * (TH)invd[j];
                cx.syncwarp();
                if (cx.lane == 0) W.dir[(int)W.flist[j]] = (T)xj;
                for (int i = cx.lane; i < j; i += Ctx::WS) z[i] -= (TH)W.L[tri(j) + i] * xj;
                cx.syncwarp();
            }
        }
        cx.sync();
        // Armijo along the projection arc
        T alpha = (T)1, ft = f;
        bool ok = false, at_floor = false;
        for (int ls = 0; ls < max_ls; ++ls) {
            T dec = (T)0;
            for (int v = cx.tid; v < nv; v += cx.nthr) {
                const T nv_ = nu[v];
                T t = nv_ - alpha * (T)W.dir[v];
                if (!(uint8_t)W.vfree[v] && t < (T)0) t = (T)0;
                nut[v] = t;
                dec += (T)W.g[v] * (nv_ - t);
            }
            cx.sync();
            nw_eval2(cx, W, nut, rc, ft, dec);
            // Predicted AND actual change below the rounding level of f: no further progress is representable; the trial
            // point is as good as the current one (r already belongs to it), so take it and stop.
            if (ls == 0 && cabs(dec) <= (T)16 * eps_mach<T>() * f && cabs(ft - f) <= (T)16 * eps_mach<T>() * f) { ok = true; at_floor = true; break; }
            if (ft <= f - (T)1e-4 * dec + (T)4 * eps_mach<T>() * f) { ok = true; break; }
            alpha *= (T)0.5;
        }
#if defined(CAVE_NW_TRACE) && !defined(CAVE_HOST_SIM)
        if (cx.tid == 0 && it < 40) printf("   nf %d alpha %.3e ft %.17g ok %d floor %d\n", nf, (double)alpha, (double)ft, (int)ok, (int)at_floor);
#endif
        if (!ok) {                    // r holds the last rejected trial: restore it for the current iterate
            T d0 = (T)0;
            nw_eval2(cx, W, nu, rc, f, d0);
            status = ST_STALLED;
            break;
        }
        HPtr<T, HOT> t1 = nu; nu = nut; nut = t1;
        // Accepted steps that no longer decrease f by a representable amount (the Armijo slack lets a step of length ~2^-24
        // through after two dozen halvings): the iterate sits at the floating-point floor of a degenerate instance with the
        // KKT residual a few tens of tol above the tolerance.  Three in a row end the solve instead of running to the
        // iteration cap (SP 5x5, seed 1001 #3905: 200 iterations x 25 evaluations = 5 ms for one 90 x 40 instance).
        // (only steps that were cut below 2^-10: a full step along a degenerate pivot may leave f unchanged and still move on)
        flat = (alpha > (T)0.0009765625 || ft < f - (T)16 * eps_mach<T>() * f) ? 0 : flat + 1;
        f = ft;
        if (at_floor) { status = ST_CONVERGED; ++it; break; }
        if (flat >= 3) {    // (the residual is re-evaluated here rather than kept live through the iteration: two registers)
            const T res_now = nw_grad(cx, W, rc, W.g, nu);
            status = res_now <= (T)1000 * tol ? ST_CONVERGED : ST_STALLED; ++it; break;
        }
    }
    out.r = rc.raw(); out.iters = it; out.status = status;
    if (WARM && in.warm && (int)W.fcnt[1] == 1) out.status |= ST_WARM;
    if (WARM && in.warm && nv <= in.warm_cap && status == ST_CONVERGED) warm_write(cx, in.warm, nv, W.vfree.raw(), W.rptr, W.vrow, W.rcol, nu.raw());
}

// ------------------------------------------------------------------ Lawson-Hanson path (dense rows)
template <class T>
CAVE_DEV T row_dot(Ctx& cx, const float* row, const T* x, int d) {   // one warp, result on all lanes
    T acc = (T)0;
    for (int k0 = 0; k0 < d; k0 += Ctx::WS * 4) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { int k = k0 + u * Ctx::WS + cx.lane; v[u] = k < d ? ld_stream(row + k) : 0.f; }
#pragma unroll
        for (int u = 0; u < 4; ++u) { int k = k0 + u * Ctx::WS + cx.lane; if (k < d) acc += (T)v[u] * x[k]; }
    }
    return cx.warp_sum(acc);
}

template <class T, class TH>
CAVE_DEV void lh_solve(Ctx& cx, const Instance& in, Arena& ar, T* c, T* r, T cnorm,
                       const SolveOpts& opt, Result<T>& out) {
    const int d = in.d, mB = in.ngen;
    const int kmax = mB < d ? mB : d;
    const int ld = kmax;
    T* xP = ar.get<T>(kmax + 1); TH* s = ar.get<TH>(kmax + 1); T* bP = ar.get<T>(kmax + 1);
    TH* tmp = ar.get<TH>(kmax + 2); TH* diagL = ar.get<TH>(kmax + 1);
    int* P = ar.get<int>(kmax + 1); int* map = ar.get<int>(kmax + 2);
    uint8_t* st = ar.get<uint8_t>(mB + 1);
    int* grow = ar.get<int>(mB + 1);
    T* rowv = ar.get<T>(d);                 // staged entering row
    TH* L = ar.get<TH>((size_t)kmax * kmax + 1);
    TH* Gp = ar.get<TH>((size_t)kmax * kmax + 1);
    out.r = r; out.iters = 0;
    if (ar.overflow || !in.A) { out.status = ST_NOSPACE | ST_PATH_LH; return; }    // dense rows are read from A

    for (int i = cx.tid; i < mB; i += cx.nthr) { st[i] = 0; grow[i] = in.gen[i].x; }
    for (int k = cx.tid; k < d; k += cx.nthr) r[k] = c[k];
    cx.sync();
    // scale = max_i ||a_i||_1 * ||c||
    T l1max = (T)0;
    for (int i = cx.warp; i < mB; i += cx.nwarp) {
        const float* row = in.A + (size_t)grow[i] * d;
        T acc = (T)0;
        for (int k = cx.lane; k < d; k += Ctx::WS) { float v = ld_stream(row + k); acc += (T)(v < 0.f ? -v : v); }
        acc = cx.warp_sum(acc);
        l1max = acc > l1max ? acc : l1max;
    }
    l1max = cx.block_max(l1max);
    const T scale = (l1max > (T)1 ? l1max : (T)1) * (cnorm > (T)1e-30 ? cnorm : (T)1e-30);
    const T tolw = (T)(opt.tol > 0 ? opt.tol : (sizeof(T) == 8 ? 1e-12 : 2e-6)) * scale;
    const int cap = opt.max_iter > 0 ? opt.max_iter : 3 * mB + 10;
    const TH dep_tol = sizeof(TH) == 8 ? (TH)1e-11 : (TH)1e-5;
    int k = 0, iters = 0, status = ST_CONVERGED;

    for (;;) {
        // dual vector on the zero set: w_i = a_i . r ; pick the largest
        T best = (T)0; int bi = -1;
        for (int i = cx.warp; i < mB; i += cx.nwarp) {
            if (st[i] != 0) continue;
            T w = row_dot(cx, in.A + (size_t)grow[i] * d, r, d);
            if (bi < 0 || w > best) { best = w; bi = i; }
        }
        cx.block_argmax(best, bi);
        if (bi < 0 || !(best > tolw) || k >= kmax) break;
        if (iters++ >= cap) { status = ST_ITER_CAP; break; }
        const int j = bi;
        const float* rowj = in.A + (size_t)grow[j] * d;
        T gjj = (T)0, bj = (T)0;
        for (int q = cx.tid; q < d; q += cx.nthr) { T v = (T)ld_stream(rowj + q); rowv[q] = v; gjj += v * v; bj += v * c[q]; }
        gjj = cx.block_sum(gjj); bj = cx.block_sum(bj);
        for (int idx = cx.warp; idx < k; idx += cx.nwarp) {
            T h = row_dot(cx, in.A + (size_t)grow[P[idx]] * d, rowv, d);
            if (cx.lane == 0) { Gp[(size_t)k * ld + idx] = (TH)h; tmp[idx] = (TH)h; }
        }
        cx.sync();
        if (cx.warp == 0) {   // append a Cholesky row: L z = h, rho^2 = g_jj - z.z
            tri_forward_w0(cx, L, k, ld, diagL, tmp);
            TH zz = (TH)0;
            for (int idx = cx.lane; idx < k; idx += Ctx::WS) zz += tmp[idx] * tmp[idx];
            zz = cx.warp_sum(zz);
            if (cx.lane == 0) tmp[k] = (TH)gjj - zz;
        }
        cx.sync();
        TH rho2 = tmp[k];
        cx.sync();
        if (!(rho2 > dep_tol * (TH)gjj)) {     // numerically dependent on the passive set: skip for this round
            if (cx.tid == 0) st[j] = 2;
            cx.sync();
            continue;
        }
        for (int idx = cx.tid; idx < k; idx += cx.nthr) L[(size_t)k * ld + idx] = tmp[idx];
        if (cx.tid == 0) {
            diagL[k] = (TH)sqrt((double)rho2); Gp[(size_t)k * ld + k] = (TH)gjj; L[(size_t)k * ld + k] = (TH)gjj;
            P[k] = j; st[j] = 1; bP[k] = bj; xP[k] = (T)0;
        }
        cx.sync();
        ++k;
        for (int idx = cx.tid; idx < k; idx += cx.nthr) s[idx] = (TH)bP[idx];
        chol_solve(cx, L, k, ld, diagL, s);
        if (!(s[k - 1] > (TH)0)) {           // Lawson-Hanson step 6 safeguard
            cx.sync();
            --k;
            if (cx.tid == 0) st[j] = 2;
            cx.sync();
            continue;
        }
        bool capped = false;
        for (;;) {                          // inner loop: step back to feasibility, drop zeros
            TH smin = (TH)1;
            for (int idx = cx.tid; idx < k; idx += cx.nthr) smin = s[idx] < smin ? s[idx] : smin;
            smin = cx.block_min(smin);
            if (smin > (TH)0) break;
            if (iters++ >= cap) { capped = true; break; }
            T al = (T)2; int ai = -1;
            for (int idx = cx.tid; idx < k; idx += cx.nthr)
                if (!(s[idx] > (TH)0)) { T a = xP[idx] / (xP[idx] - (T)s[idx]); if (ai < 0 || a < al) { al = a; ai = idx; } }
            cx.block_argmin(al, ai);
            if (!(al >= (T)0)) al = (T)0;
            T xmax = (T)0;
            for (int idx = cx.tid; idx < k; idx += cx.nthr) {
                T xn = xP[idx] + al * ((T)s[idx] - xP[idx]);
                xP[idx] = xn;
                xmax = xn > xmax ? xn : xmax;
            }
            xmax = cx.block_max(xmax);
            if (cx.tid == 0) {              // compaction map (ordered)
                int kn = 0;
                for (int idx = 0; idx < k; ++idx) {
                    bool rem = idx == ai || (!(s[idx] > (TH)0) && !(xP[idx] > (T)1e-14 * xmax));
                    if (rem) st[P[idx]] = 0; else map[kn++] = idx;
                }
                map[kmax + 1] = kn;
            }
            cx.sync();
            const int kn = map[kmax + 1];
            // L <- compacted Gram (scratch), then Gp <- L, then factor L in place
            for (int t = cx.tid; t < kn * kn; t += cx.nthr) {
                int a = t / kn, b = t - a * kn;
                if (b <= a) L[(size_t)a * ld + b] = Gp[(size_t)map[a] * ld + map[b]];
            }
            cx.sync();
            for (int t = cx.tid; t < kn * kn; t += cx.nthr) {
                int a = t / kn, b = t - a * kn;
                if (b <= a) Gp[(size_t)a * ld + b] = L[(size_t)a * ld + b];
            }
            if (cx.tid == 0)
                for (int a = 0; a < kn; ++a) { int o = map[a]; P[a] = P[o]; xP[a] = xP[o]; bP[a] = bP[o]; }
            cx.sync();
            k = kn;
            TH dmax = (TH)0;
            for (int a = cx.tid; a < k; a += cx.nthr) { TH h = Gp[(size_t)a * ld + a]; dmax = h > dmax ? h : dmax; }
            dmax = cx.block_max(dmax);
            chol_factor(cx, L, k, ld, diagL, eps_mach<TH>() * dmax);
            for (int idx = cx.tid; idx < k; idx += cx.nthr) s[idx] = (TH)bP[idx];
            chol_solve(cx, L, k, ld, diagL, s);
            if (k == 0) break;
        }
        if (capped) { status = ST_ITER_CAP; break; }
        for (int idx = cx.tid; idx < k; idx += cx.nthr) xP[idx] = (T)s[idx];
        for (int i = cx.tid; i < mB; i += cx.nthr) if (st[i] == 2) st[i] = 0;
        cx.sync();
        for (int q = cx.tid; q < d; q += cx.nthr) {     // r = c - sum_P x_i a_i
            T acc = c[q];
            for (int idx = 0; idx < k; ++idx) acc -= xP[idx] * (T)in.A[(size_t)grow[P[idx]] * d + q];
            r[q] = acc;
        }
        cx.sync();
    }
    if (sizeof(TH) < sizeof(T) && k > 0) {
        // mixed precision: two rounds of iterative refinement of the passive-set least squares with
        // the residual formed in T through A itself and the TH Cholesky factor as the solver
        for (int round = 0; round < 2; ++round) {
            for (int idx = cx.warp; idx < k; idx += cx.nwarp) {
                T h = row_dot(cx, in.A + (size_t)grow[P[idx]] * d, r, d);
                if (cx.lane == 0) s[idx] = (TH)h;
            }
            chol_solve(cx, L, k, ld, diagL, s);
            for (int idx = cx.tid; idx < k; idx += cx.nthr) { T xn = xP[idx] + (T)s[idx]; xP[idx] = xn > (T)0 ? xn : (T)0; }
            cx.sync();
            for (int q = cx.tid; q < d; q += cx.nthr) {
                T acc = c[q];
                for (int idx = 0; idx < k; ++idx) acc -= xP[idx] * (T)in.A[(size_t)grow[P[idx]] * d + q];
                r[q] = acc;
            }
            cx.sync();
        }
    }
    out.iters = iters; out.status = status | ST_PATH_LH;
}

// ------------------------------------------------------------------ fused epilogue
// target (src/cave.py:121-129, 197-219), loss = 1 - cos (src/cave.py:72), d loss / d pred.
struct EpiParams {
    int mode;
    double inner_ratio, sign, gscale;   // gscale = 1/B for 'mean', 1 otherwise
};

template <class T, class TIO, class PC>
CAVE_DEV void epilogue(Ctx& cx, const Instance& in, const EpiParams& ep, PC c, const T* r,
                       bool have_proj, bool empty_cone,
                       TIO* grad_out, TIO* proj_out, double* loss_out, double* rnorm_out) {
    const int d = in.d;
    constexpr int U = 8;        // global loads (ctype, avg) of U strides are issued together, ahead of the ordered shared loads
    const bool use_q = have_proj && !empty_cone;
    double pp = 0.0, qq = 0.0, cc = 0.0;
    for (int k0 = 0; k0 < d; k0 += U * cx.nthr) {
        int ty[U];
#pragma unroll
        for (int u = 0; u < U; ++u) { const int k = k0 + u * cx.nthr + cx.tid; ty[u] = (use_q && k < d) ? (int)in.ctype[k] : 0; }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int k = k0 + u * cx.nthr + cx.tid;
            if (k < d) {
                const double ck = (double)c[k];
                const double q = use_q ? (double)psi(r[k], ty[u]) : 0.0;
                const double p = ck - q;
                pp += p * p; qq += q * q; cc += ck * ck;
            }
        }
    }
    pp = cx.block_sum(pp); qq = cx.block_sum(qq); cc = cx.block_sum(cc);
    const double rnorm = sqrt(qq), pnorm = sqrt(pp), cnorm = sqrt(cc);
    const double pden = pnorm > 1e-8 ? pnorm : 1e-8;
    const double cden = cnorm > 1e-8 ? cnorm : 1e-8;
    const double rr = ep.inner_ratio;
    const bool push = ep.mode == MODE_INNER && !(rnorm < 1e-7);
    const bool heur = ep.mode == MODE_HEURISTIC;
    const bool need_avg = heur || push;
    // target t_k (recomputed in the last pass instead of being stored: no d-vector of scratch)
    auto target = [&](int k, double ck, int ty, double av) -> double {
        if (heur) return (1.0 - rr) * (ck / cden) + rr * av;
        const double q = empty_cone ? 0.0 : (double)psi(r[k], ty);
        const double ph = (ck - q) / pden;
        return push ? (1.0 - rr) * ph + rr * av : ph;
    };
    double tt = 0.0, ct = 0.0;
    for (int k0 = 0; k0 < d; k0 += U * cx.nthr) {
        int ty[U]; float av[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int k = k0 + u * cx.nthr + cx.tid;
            ty[u] = (!heur && !empty_cone && k < d) ? (int)in.ctype[k] : 0;
            av[u] = (need_avg && k < d) ? in.avg[k] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int k = k0 + u * cx.nthr + cx.tid;
            if (k < d) {
                const double ck = (double)c[k];
                const double t = target(k, ck, ty[u], (double)av[u]);
                if (proj_out && !heur) proj_out[k] = (TIO)(ck - (empty_cone ? 0.0 : (double)psi(r[k], ty[u])));
                tt += t * t; ct += ck * t;
            }
        }
    }
    tt = cx.block_sum(tt); ct = cx.block_sum(ct);
    const double tnorm = sqrt(tt);
    const double tden = tnorm > 1e-8 ? tnorm : 1e-8;
    const double cosv = ct / (cden * tden);
    const double invc = cnorm > 0.0 ? 1.0 / cnorm : 0.0;
    const double gs = ep.gscale * ep.sign;
    for (int k0 = 0; k0 < d; k0 += U * cx.nthr) {
        int ty[U]; float av[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int k = k0 + u * cx.nthr + cx.tid;
            ty[u] = (!heur && !empty_cone && k < d) ? (int)in.ctype[k] : 0;
            av[u] = (need_avg && k < d) ? in.avg[k] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int k = k0 + u * cx.nthr + cx.tid;
            if (k < d) {
                const double ck = (double)c[k];
                const double v = target(k, ck, ty[u], (double)av[u]) / tden;
                const double w = ck * invc;
                grad_out[k] = (TIO)(gs * (-(v - cosv * w) / cden));
            }
        }
    }
    if (cx.tid == 0) { *loss_out = 1.0 - cosv; *rnorm_out = (ep.mode == MODE_HEURISTIC) ? 0.0 : rnorm; }
}

// ------------------------------------------------------------------ one instance, start to finish
template <class TH, class TIO, bool HOT, bool WARM>
CAVE_DEV bool solve_instance_t(Ctx& cx, const Instance& in, Arena& ar, const TIO* pred, const EpiParams& ep,
                               const SolveOpts& opt, TIO* grad_out, TIO* proj_out,
                               double* loss_out, double* rnorm_out, int* status_out, int* iters_out) {
    typedef double T;      // state vectors are always double; TH is the Hessian / factor precision
    const int d = in.d;
    HPtr<TIO, HOT> c = ar.geth<HOT, TIO>(d);      // c = sign * pred is exact in the I/O dtype
    HPtr<T, HOT> r = ar.geth<HOT, T>(d);
    if (HOT && ar.hot_overflow) return false;         // retry with generic placement
    bool nospace = ar.overflow;                         // cannot even hold the cost vector
    Result<T> res; res.r = r.raw(); res.iters = 0; res.status = ST_SKIPPED;
    const bool empty = in.nvalid == 0;
    if (!nospace) {
        T cc = (T)0;
        for (int k0 = 0; k0 < d; k0 += 8 * cx.nthr) {       // global loads first, then the (ordered) shared stores
            TIO pv[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) { const int k = k0 + u * cx.nthr + cx.tid; pv[u] = k < d ? pred[k] : (TIO)0; }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int k = k0 + u * cx.nthr + cx.tid;
                if (k < d) { const TIO vc = (TIO)(ep.sign * (double)pv[u]); const T v = (T)vc; c[k] = vc; r[k] = v; cc += v * v; }
            }
        }
        cc = cx.block_sum(cc);
        const T cnorm = (T)sqrt((double)cc);
        const bool finite_in = cc < (T)1e300;              // false for NaN / Inf predictions
        const bool solve = ep.mode != MODE_HEURISTIC && !empty && finite_in;
        if (!finite_in) res.status = ST_BADINPUT;
        if (solve && in.ngen > 0) {
            if (in.nsingc == 0) {
                T* cd = ar.get<T>(d);         // Lawson-Hanson works on a float64 copy of c (generic placement)
                if (!ar.overflow) {
                    for (int k = cx.tid; k < d; k += cx.nthr) cd[k] = (T)(TIO)c[k];
                    cx.sync();
                }
                lh_solve<T, T>(cx, in, ar, cd, r.raw(), cnorm, opt, res);    // dense path: float64 factor in both modes
            } else {
                newton_solve<T, TH, TIO, HOT, WARM>(cx, in, ar, c, r, cnorm, opt, res);
            }
        } else if (solve) {
            res.status = ST_CONVERGED;      // only singleton rows: closed form, r = c
        }
        cx.sync();
        if ((res.status & 0xff) == ST_NOSPACE) {
            if (HOT && ar.hot_overflow) return false;   // the shared-memory-only layout did not fit
            nospace = true;
        }
    }
    if (nospace) {          // report, never a silent number
        if (cx.tid == 0) { *loss_out = NAN; *rnorm_out = NAN; *status_out = ST_NOSPACE | (res.status & ST_PATH_LH); *iters_out = 0; }
        for (int k = cx.tid; k < d; k += cx.nthr) { grad_out[k] = (TIO)NAN; if (proj_out) proj_out[k] = (TIO)NAN; }
        return true;
    }
    epilogue<T, TIO, HPtr<TIO, HOT> >(cx, in, ep, c, res.r, ep.mode != MODE_HEURISTIC, empty, grad_out, proj_out, loss_out, rnorm_out);
    if (cx.tid == 0) { *status_out = res.status; *iters_out = res.iters; }
    return true;
}

// One instance, start to finish.  First with the iteration's arrays pinned to shared memory (the
// fast layout); if they do not fit (very large d or very many general rows) once more with generic
// placement, where everything may spill to the CTA's global scratch slot.  WARM = false compiles none of the warm-start
// code (Instance::warm and the fields after it are then never read).
template <class TH, class TIO, bool WARM = false>
CAVE_DEV void solve_instance(Ctx& cx, const Instance& in, char* smem, size_t smem_bytes, char* slot, size_t slot_bytes,
                             const TIO* pred, const EpiParams& ep, const SolveOpts& opt, TIO* grad_out, TIO* proj_out,
                             double* loss_out, double* rnorm_out, int* status_out, int* iters_out) {
    Arena ar;
    ar.init(smem, smem_bytes, slot, slot_bytes);
    if (solve_instance_t<TH, TIO, true, WARM>(cx, in, ar, pred, ep, opt, grad_out, proj_out, loss_out, rnorm_out, status_out, iters_out))
        return;
    cx.sync();
    ar.init(smem, smem_bytes, slot, slot_bytes);
    solve_instance_t<TH, TIO, false, WARM>(cx, in, ar, pred, ep, opt, grad_out, proj_out, loss_out, rnorm_out, status_out, iters_out);
}

}  // namespace cave
