// Kernel 1 — scan/pack: ONE streaming pass over A (the HBM-bound part of the path).  One CTA per instance.
//
// Two variants, chosen by row length (launch_scan):
//  * scan_rows_kernel (rows up to a few KB — every shipped model): warp-streaming, see its comment below;
//    measured 5.4 TB/s = 83 % of the measured HBM copy peak at TSP-50 (profiles/r1_ncu_summary.txt).
//  * scan_kernel (any row length up to the ABI limit): row tiles go through a CTA-wide shared-memory ring fed by
//    1-D TMA bulk copies (cp.async.bulk ... mbarrier::complete_tx) issued by one thread; phase A: one warp per
//    row, aligned 128-bit shared loads with a warp-uniform all-zero test, per-row non-zero count / sum|a| /
//    sum a^2; phase B: one thread does the ordered bookkeeping of singleton rows, all threads accumulate
//    a/||a|| column-parallel over the general rows, one warp per general row compacts it into the packed CSR
//    and hashes it.
// Both produce everything `_average_ctrs` (src/cave.py:222-228) and the row mask of `_project_nnls`
// (src/cave.py:303) recompute on the host for every call, in one read of A, plus what the solver needs: per
// coordinate singleton cone types, the general-row list with a packed CSR, and two order-free 64-bit row
// hashes for +-row matching.  Accumulation orders are fixed (or exact integer arithmetic), so the pack is
// bit-reproducible run to run.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include "layout.cuh"
#include "scan_kernel.cuh"

namespace cave {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ uint64_t mix64d(uint64_t x) {      // same mixer as solver_core.cuh
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

struct RowAcc {
    float l1, l2, lv;
    int lk, n;
    __device__ __forceinline__ void add(float v, int k) {
        l1 += fabsf(v);
        l2 = fmaf(v, v, l2);
        lk = k; lv = v; ++n;
    }
};

template <int NT>
__global__ void __launch_bounds__(NT) scan_kernel(ScanParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    const int d = p.d, R = p.R, S = p.stages;
    const int b = blockIdx.x;

    unsigned char* ring = smem;
    float* avg_gen = (float*)(smem + (size_t)S * p.stage_stride);
    int* sing = (int*)(avg_gen + d);
    uint64_t* full = (uint64_t*)align_up((size_t)(sing + d), 8);
    float* r_l1 = (float*)(full + S);
    float* r_nrm = r_l1 + R;
    float* r_inv = r_nrm + R;
    float* r_val = r_inv + R;
    int* r_cnt = (int*)(r_val + R);
    int* r_k = r_cnt + R;
    int* s_cnt = r_k + R;                                   // [8]
    unsigned char* ctype = (unsigned char*)align_up((size_t)(s_cnt + 8), 16);   // [dpad]

    const int m_b = p.m_rows ? min(max(p.m_rows[b], 0), p.m_max) : p.m_max;
    const int ntiles = (m_b + R - 1) / R;
    const float* A_b = p.A + (size_t)b * p.m_max * d;

    for (int k = tid; k < d; k += NT) { avg_gen[k] = 0.f; sing[k] = 0; }
    for (int k = tid; k < (int)p.dpad; k += NT) ctype[k] = 0;
    if (tid < 8) s_cnt[tid] = 0;
    if (tid == 0) {
        for (int s = 0; s < S; ++s) mbar_init(full + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto issue = [&](int t) {
        const int s = t % S;
        const int rows = min(R, m_b - t * R);
        const uintptr_t a = (uintptr_t)(A_b + (size_t)t * R * d);
        const uintptr_t a0 = a & ~(uintptr_t)15;
        const uintptr_t a1 = (a + (size_t)rows * d * 4 + 15) & ~(uintptr_t)15;
        const uint32_t bytes = (uint32_t)(a1 - a0);
        mbar_expect_tx(full + s, bytes);
        tma_bulk_g2s(ring + (size_t)s * p.stage_stride, (const void*)a0, bytes, full + s);
    };
    if (tid == 0)
        for (int t = 0; t < S && t < ntiles; ++t) issue(t);

    // running totals, replicated in every thread (identical arithmetic everywhere)
    int t_ngen = 0, t_gennnz = 0;
    float t_l1max = 0.f, t_l2max = 0.f;
    // bookkeeper-only counters (thread NT-1)
    int c_nvalid = 0, c_navg = 0;
    int overflow = 0;
    int4* gen_out = p.gen4 + (size_t)b * p.m_max;
    ulonglong2* hash_out = p.ghash + (size_t)b * p.m_max;      // row-indexed
    uint16_t* col_out = p.csr_col + (size_t)b * p.cap_nnz;
    float* val_out = p.csr_val + (size_t)b * p.cap_nnz;

    for (int t = 0; t < ntiles; ++t) {
        const int s = t % S;
        const int rows = min(R, m_b - t * R);
        const uintptr_t a = (uintptr_t)(A_b + (size_t)t * R * d);
        const int shift = (int)((a & 15) >> 2);
        const float* base = (const float*)(ring + (size_t)s * p.stage_stride);   // 16-byte aligned
        const float* tile = base + shift;
        mbar_wait(full + s, (uint32_t)((t / S) & 1));

        // ---- phase A: per-row statistics, one warp per row
        for (int rr = warp; rr < rows; rr += NW) {
            const int e0 = shift + rr * d, e1 = e0 + d;         // element range in `base` coordinates
            const int q0 = (e0 + 3) >> 2, q1 = e1 >> 2;         // whole float4 words inside the row
            RowAcc acc; acc.l1 = 0.f; acc.l2 = 0.f; acc.lv = 0.f; acc.lk = -1; acc.n = 0;
            int cnt = 0;
            if (q0 <= q1) {
                if (lane < 4) {                                  // ragged head and tail (< 4 elements each)
                    const int kh = e0 + lane;
                    if (kh < (q0 << 2) && kh < e1) { float v = base[kh]; if (v != 0.f) acc.add(v, kh - e0); }
                    const int kt = (q1 << 2) + lane;
                    if (kt >= (q0 << 2) && kt < e1) { float v = base[kt]; if (v != 0.f) acc.add(v, kt - e0); }
                }
                const float4* b4 = (const float4*)base;
                for (int q = q0 + lane; q < q1 + lane; q += 32) {       // uniform trip count
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (q < q1) v = b4[q];
                    const uint32_t any = (__float_as_uint(v.x) | __float_as_uint(v.y) | __float_as_uint(v.z) | __float_as_uint(v.w)) << 1;
                    if (__ballot_sync(0xffffffffu, any != 0u) == 0u) continue;      // all 128 words are zero
                    if (any != 0u) {
                        const int k = (q << 2) - e0;
                        if (v.x != 0.f) acc.add(v.x, k);
                        if (v.y != 0.f) acc.add(v.y, k + 1);
                        if (v.z != 0.f) acc.add(v.z, k + 2);
                        if (v.w != 0.f) acc.add(v.w, k + 3);
                    }
                }
            } else {                                             // row shorter than one aligned word
                for (int k = e0 + lane; k < e1; k += 32) { float v = base[k]; if (v != 0.f) acc.add(v, k - e0); }
            }
            // exact non-zero count of the row (lanes that saw nothing are skipped with one ballot)
            const unsigned sawm = __ballot_sync(0xffffffffu, acc.n > 0);
            if (sawm) {
                if ((sawm & (sawm - 1)) == 0u) {
                    cnt = __shfl_sync(0xffffffffu, acc.n, __ffs(sawm) - 1);
                } else {
                    cnt = acc.n;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
                }
            }
            float l1 = 0.f, nrm = 0.f, v1 = 0.f;
            int k1 = -1;
            if (cnt == 1) {
                const int src = __ffs(sawm) - 1;
                k1 = __shfl_sync(0xffffffffu, acc.lk, src);
                v1 = __shfl_sync(0xffffffffu, acc.lv, src);
                l1 = fabsf(v1); nrm = sqrtf(v1 * v1);
            } else if (cnt >= 2) {
                float a1 = acc.l1, a2 = acc.l2;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    a1 += __shfl_xor_sync(0xffffffffu, a1, o);
                    a2 += __shfl_xor_sync(0xffffffffu, a2, o);
                }
                l1 = a1; nrm = sqrtf(a2);
            }
            if (lane == 0) {
                r_l1[rr] = l1; r_nrm[rr] = nrm;
                r_inv[rr] = nrm > 1e-7f ? 1.f / fmaxf(nrm, 1e-8f) : 0.f;
                r_cnt[rr] = cnt; r_k[rr] = k1; r_val[rr] = v1;
            }
        }
        __syncthreads();

        // ---- phase B
        // every thread: masks of the tile's general rows (valid for the solver / valid for the average)
        unsigned gmask = 0, amask = 0;
        for (int rr = 0; rr < rows; ++rr) {
            const bool gen = r_cnt[rr] >= 2;
            if (gen && r_l1[rr] > 1e-7f) gmask |= 1u << rr;          // src/cave.py:303
            if (gen && r_inv[rr] != 0.f) amask |= 1u << rr;          // src/cave.py:224-225
        }
        if (tid == NT - 1) {                                         // ordered bookkeeping of the other rows
            for (int rr = 0; rr < rows; ++rr) {
                const bool nv = r_l1[rr] > 1e-7f, av = r_inv[rr] != 0.f;
                c_nvalid += nv; c_navg += av;
                if (r_cnt[rr] == 1) {
                    const int k = r_k[rr];
                    const bool pos = r_val[rr] > 0.f;
                    if (nv) ctype[k] |= pos ? 1 : 2;
                    if (av) sing[k] += pos ? 1 : -1;
                }
            }
        }
        if (amask) {                                                 // a / ||a|| over the general rows
            for (int k = tid; k < d; k += NT) {
                float acc = 0.f;
                for (unsigned m = amask; m; m &= m - 1) {
                    const int rr = __ffs(m) - 1;
                    acc = fmaf(tile[(size_t)rr * d + k], r_inv[rr], acc);
                }
                avg_gen[k] += acc;
            }
        }
        if (gmask) {                                                 // pack the general rows (CSR)
            int ord = 0, off = t_gennnz;
            for (unsigned m = gmask; m; m &= m - 1, ++ord) {
                const int rr = __ffs(m) - 1;
                const int cnt = r_cnt[rr];
                if (ord % NW == warp) {
                    uint64_t hp = 0, hn = 0;
                    if (off + cnt <= p.cap_nnz) {
                        const float* row = tile + (size_t)rr * d;
                        int w = off;
                        for (int k0 = 0; k0 < d; k0 += 32) {
                            const int k = k0 + lane;
                            const float v = k < d ? row[k] : 0.f;
                            const unsigned nzm = __ballot_sync(0xffffffffu, v != 0.f);
                            if (v != 0.f) {
                                const int pos = w + __popc(nzm & ((1u << lane) - 1u));
                                col_out[pos] = (uint16_t)k; val_out[pos] = v;
                                if (!(v == (float)(int)v && fabsf(v) <= 127.f)) s_cnt[7] = 1;
                                const uint32_t bits = __float_as_uint(v);
                                hp += mix64d(((uint64_t)k << 32) | bits);
                                hn += mix64d(((uint64_t)k << 32) | (bits ^ 0x80000000u));
                            }
                            w += __popc(nzm);
                        }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            hp += __shfl_xor_sync(0xffffffffu, hp, o);
                            hn += __shfl_xor_sync(0xffffffffu, hn, o);
                        }
                    }
                    if (lane == 0) {
                        gen_out[t_ngen + ord] = make_int4(t * R + rr, cnt, off, 0);
                        hash_out[t * R + rr] = make_ulonglong2(hp, hn);
                    }
                }
                if (off + cnt > p.cap_nnz) overflow = 1;
                off += cnt;
                t_l1max = fmaxf(t_l1max, r_l1[rr]);
                t_l2max = fmaxf(t_l2max, r_nrm[rr] * r_nrm[rr]);
            }
            t_ngen += ord; t_gennnz = off;
        }
        __syncthreads();
        if (tid == 0 && t + S < ntiles) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(t + S);
        }
    }

    if (tid == NT - 1) { s_cnt[0] = c_nvalid; s_cnt[1] = c_navg; }
    __syncthreads();
    int nsc = 0;
    for (int k = tid; k < d; k += NT) nsc += ctype[k] != 0;
    for (int o = 16; o > 0; o >>= 1) nsc += __shfl_xor_sync(0xffffffffu, nsc, o);
    if (lane == 0 && nsc) atomicAdd(&s_cnt[4], nsc);
    __syncthreads();
    const float ninv = 1.f / (float)max(s_cnt[1], 1);
    float* avg_out = p.avg + (size_t)b * p.dpad;
    for (int k = tid; k < (int)p.dpad; k += NT) avg_out[k] = k < d ? (avg_gen[k] + (float)sing[k]) * ninv : 0.f;
    uint32_t* ct_out = (uint32_t*)(p.ctype + (size_t)b * p.dpad);
    for (int k = tid; k < (int)(p.dpad / 4); k += NT) ct_out[k] = ((const uint32_t*)ctype)[k];
    if (tid == 0) {
        p.nvalid[b] = s_cnt[0]; p.navg[b] = s_cnt[1]; p.ngen[b] = t_ngen; p.gennnz[b] = t_gennnz; p.nsingc[b] = s_cnt[4];
        p.csr_ok[b] = overflow ? 0 : (s_cnt[7] ? 1 : 3);
        p.maxl1[b] = t_l1max; p.maxl2[b] = t_l2max;
    }
}


// one non-zero of a general row: its 2^-40 fixed-point share of the average, the int8 test and the two row hashes
template <bool SKIPAVG>
__device__ __forceinline__ void gen_elem(float v, int k, bool av, bool fits, float inv, unsigned long long* avg_fx, int* s_cnt,
                                         uint64_t& hp, uint64_t& hn) {
    if (av && !SKIPAVG) atomicAdd(&avg_fx[k], (unsigned long long)__double2ll_rn((double)v * (double)inv * 1099511627776.0));
    if (fits) {
        if (!(v == (float)(int)v && fabsf(v) <= 127.f)) s_cnt[7] = 1;      // not an int8 value
        const uint32_t bits = __float_as_uint(v);
        hp += mix64d(((uint64_t)k << 32) | bits);
        hn += mix64d(((uint64_t)k << 32) | (bits ^ 0x80000000u));
    }
}

// ---------------------------------------------------------------------------------------------
// Warp-streaming variant (rows up to a few KB: every shipped model).  No CTA barrier in the steady
// state: warp w owns rows w, w+8, ... of the instance and a private ring of row buffers that its lane 0
// refills with TMA bulk copies, so eight independent row streams are in flight per CTA.  Cross-row
// state is either warp-private (fixed order => reproducible) or exact under reordering (integer
// atomics); the ordered general-row list is assembled once per instance after a single barrier.
// Per row: one pass of 128-bit loads folded into one bit per non-zero word and one ballot; only the non-zero words are
// read again.  92 % of the rows of a TSP-50 instance are singletons, so that slot is refilled as soon as the row is
// classified; a general row refills after its CSR / hash pass, which visits the non-zero words only.
// SKIPAVG: instantiation for packs that need no average (ScanParams::skip_avg); the default instantiation is textually the
// round-1 kernel (a run-time test in the row loop changed its register allocation, 56 -> 48, and cost the TSP-50 scan 4 %).
template <int NT, int S, bool SKIPAVG = false>
__global__ void __launch_bounds__(NT, 2) scan_rows_kernel(ScanParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NT / 32;
    const int d = p.d;
    const int b = blockIdx.x;
    const size_t rowbuf = p.stage_stride;

    unsigned char* ring = smem;                                             // [NW][S][rowbuf]
    // average of a/||a|| over the general rows: 2^-40 fixed point in 64-bit integers, so that the shared
    // accumulator is exact (hence reproducible) under any interleaving of the warps
    unsigned long long* avg_fx = (unsigned long long*)(smem + (size_t)NW * S * rowbuf);   // [d]
    int* sing = (int*)(avg_fx + d);                                          // [d]
    int2* rowinfo = (int2*)align_up((size_t)(sing + d), 8);                 // [m_max] (cnt, off); cnt = 0: not general
    uint64_t* full = (uint64_t*)(rowinfo + p.m_max);                        // [NW*S]
    int* s_cnt = (int*)(full + NW * S);                                     // [16]
    float* s_max = (float*)(s_cnt + 16);                                    // [2*NW]
    unsigned* ctype_w = (unsigned*)align_up((size_t)(s_max + 2 * NW), 16);  // [dpad/4] words of 4 cone types

    const int m_b = p.m_rows ? min(max(p.m_rows[b], 0), p.m_max) : p.m_max;
    const float* A_b = p.A + (size_t)b * p.m_max * d;

    for (int k = tid; k < d; k += NT) avg_fx[k] = 0ull;
    for (int k = tid; k < d; k += NT) sing[k] = 0;
    for (int k = tid; k < (int)(p.dpad / 4); k += NT) ctype_w[k] = 0u;
    for (int k = tid; k < p.m_max; k += NT) rowinfo[k] = make_int2(0, 0);
    if (tid < 16) s_cnt[tid] = 0;
    if (tid == 0) {
        for (int i = 0; i < NW * S; ++i) mbar_init(full + i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    unsigned char* myring = ring + (size_t)warp * S * rowbuf;
    uint64_t* mybar = full + warp * S;
    auto issue = [&](int it) {          // lane 0 only
        const int s = it % S;
        const int row = warp + NW * it;
        const uintptr_t a = (uintptr_t)(A_b + (size_t)row * d);
        const uintptr_t a0 = a & ~(uintptr_t)15;
        const uintptr_t a1 = (a + (size_t)d * 4 + 15) & ~(uintptr_t)15;
        const uint32_t bytes = (uint32_t)(a1 - a0);
        mbar_expect_tx(mybar + s, bytes);
        tma_bulk_g2s(myring + (size_t)s * rowbuf, (const void*)a0, bytes, mybar + s);
    };
    const int nit = m_b > warp ? (m_b - warp + NW - 1) / NW : 0;
    if (lane == 0)
        for (int it = 0; it < S && it < nit; ++it) issue(it);

    int w_nvalid = 0, w_navg = 0, w_gennnz = 0, w_ngen = 0;
    float w_l1max = 0.f, w_l2max = 0.f;
    uint16_t* col_out = p.csr_col + (size_t)b * p.cap_nnz;
    float* val_out = p.csr_val + (size_t)b * p.cap_nnz;
    ulonglong2* hash_out = p.ghash + (size_t)b * p.m_max;       // row-indexed

    for (int it = 0; it < nit; ++it) {
        const int s = it % S;
        const int row_id = warp + NW * it;
        const uintptr_t a = (uintptr_t)(A_b + (size_t)row_id * d);
        const int shift = (int)((a & 15) >> 2);
        const float* base = (const float*)(myring + (size_t)s * rowbuf);
        mbar_wait(mybar + s, (uint32_t)((it / S) & 1));

        // The row is split into units: lanes 0-3 each own one element of the ragged head (before the first whole 128-bit
        // word) and one of the ragged tail, and lane L owns the whole words q0 + L + 32 j.  Pass 1 loads every unit and
        // keeps one bit per non-zero unit (bit 0 head, bit 1 tail, bit 2 + j word j); one ballot then classifies the row.
        // Only the non-zero units are visited again, in bit order, which is the per-lane order of the sums below.
        const int e0 = shift, e1 = e0 + d;
        const int q0 = (e0 + 3) >> 2, q1 = e1 >> 2;         // [q0, q1): whole words; q0 > q1 only for d < 4 (head only)
        const float4* b4 = (const float4*)base;
        uint32_t nzw = 0;
        if (lane < 4) {
            const int kh = e0 + lane, kt = (q1 << 2) + lane;
            if (kh < min(q0 << 2, e1) && (__float_as_uint(base[kh]) << 1) != 0u) nzw = 1u;      // (<< 1: -0.0 is a zero)
            if (kt >= (q0 << 2) && kt < e1 && (__float_as_uint(base[kt]) << 1) != 0u) nzw |= 2u;
        }
        for (int q = q0 + lane, j = 2; q < q1 + lane; q += 128, j += 4) {     // uniform trip count; j < 20 (launch_scan: d < 2100)
            uint32_t nib = 0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (q + 32 * u < q1) {
                    const float4 v = b4[q + 32 * u];
                    if (((__float_as_uint(v.x) | __float_as_uint(v.y) | __float_as_uint(v.z) | __float_as_uint(v.w)) << 1) != 0u)
                        nib |= 1u << u;
                }
            }
            nzw |= nib << j;
        }
        const unsigned sawm = __ballot_sync(0xffffffffu, nzw != 0u);
        // exact non-zero count, |a|_1, |a|_2^2 and the last non-zero of every lane, in the lane's unit order
        RowAcc acc; acc.l1 = 0.f; acc.l2 = 0.f; acc.lv = 0.f; acc.lk = -1; acc.n = 0;
        for (uint32_t m = nzw; m; m &= m - 1) {
            const int bit = __ffs(m) - 1;
            if (bit < 2) {
                const int e = bit == 0 ? e0 + lane : (q1 << 2) + lane;
                acc.add(base[e], e - e0);
            } else {
                const int q = q0 + lane + 32 * (bit - 2), k = (q << 2) - e0;
                const float4 v = b4[q];
                if (v.x != 0.f) acc.add(v.x, k);
                if (v.y != 0.f) acc.add(v.y, k + 1);
                if (v.z != 0.f) acc.add(v.z, k + 2);
                if (v.w != 0.f) acc.add(v.w, k + 3);
            }
        }
        int cnt = 0;
        if (sawm) {
            if ((sawm & (sawm - 1)) == 0u) {
                cnt = __shfl_sync(0xffffffffu, acc.n, __ffs(sawm) - 1);
            } else {
                cnt = acc.n;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            }
        }
        if (cnt < 2) {
            // an empty or singleton row is in registers now: its ring slot can take the next row before the bookkeeping
            __syncwarp();
            if (lane == 0 && it + S < nit) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue(it + S);
            }
        }
        if (cnt == 1) {
            const int src = __ffs(sawm) - 1;
            const float v1 = __shfl_sync(0xffffffffu, acc.lv, src);
            const bool nv = fabsf(v1) > 1e-7f, av = sqrtf(v1 * v1) > 1e-7f;
            w_nvalid += nv; w_navg += av;
            if (lane == src) {
                const int k1 = acc.lk;
                if (nv) atomicOr(&ctype_w[k1 >> 2], (v1 > 0.f ? 1u : 2u) << ((k1 & 3) * 8));
                if (av) atomicAdd(&sing[k1], v1 > 0.f ? 1 : -1);
            }
        } else if (cnt >= 2) {
            float a1 = acc.l1, a2 = acc.l2;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                a1 += __shfl_xor_sync(0xffffffffu, a1, o);
                a2 += __shfl_xor_sync(0xffffffffu, a2, o);
            }
            const float nrm = sqrtf(a2);
            const bool nv = a1 > 1e-7f, av = nrm > 1e-7f;
            const float inv = av ? 1.f / fmaxf(nrm, 1e-8f) : 0.f;
            w_nvalid += nv; w_navg += av;
            int off = 0;
            bool fits = false;
            if (nv) {
                if (lane == 0) off = atomicAdd(&s_cnt[5], cnt);
                off = __shfl_sync(0xffffffffu, off, 0);
                fits = off + cnt <= p.cap_nnz;
                if (!fits && lane == 0) s_cnt[6] = 1;
                w_gennnz += cnt; ++w_ngen;
                w_l1max = fmaxf(w_l1max, a1); w_l2max = fmaxf(w_l2max, a2);
            }
            if (fits) {
                // packed CSR in column order: head units, then the words by (j, lane), then tail units; a lane's position
                // inside each group is the warp prefix of the non-zero counts (three ballots of the 0..4 count per word)
                const unsigned lt = (1u << lane) - 1u;
                const unsigned hm = __ballot_sync(0xffffffffu, nzw & 1u);
                if (nzw & 1u) {
                    const int pos = off + __popc(hm & lt);
                    col_out[pos] = (uint16_t)lane; val_out[pos] = base[e0 + lane];
                }
                int w = off + __popc(hm);
                for (uint32_t jm = __reduce_or_sync(0xffffffffu, nzw & ~3u); jm; jm &= jm - 1) {
                    const int bit = __ffs(jm) - 1;
                    const int q = q0 + lane + 32 * (bit - 2);
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if ((nzw >> bit) & 1u) v = b4[q];
                    const int n = (v.x != 0.f) + (v.y != 0.f) + (v.z != 0.f) + (v.w != 0.f);
                    const unsigned c0 = __ballot_sync(0xffffffffu, n & 1), c1 = __ballot_sync(0xffffffffu, n & 2),
                                   c2 = __ballot_sync(0xffffffffu, n & 4);
                    int pos = w + __popc(c0 & lt) + 2 * __popc(c1 & lt) + 4 * __popc(c2 & lt);
                    w += __popc(c0) + 2 * __popc(c1) + 4 * __popc(c2);
                    if (n) {
                        const int k = (q << 2) - e0;
                        if (v.x != 0.f) { col_out[pos] = (uint16_t)k; val_out[pos++] = v.x; }
                        if (v.y != 0.f) { col_out[pos] = (uint16_t)(k + 1); val_out[pos++] = v.y; }
                        if (v.z != 0.f) { col_out[pos] = (uint16_t)(k + 2); val_out[pos++] = v.z; }
                        if (v.w != 0.f) { col_out[pos] = (uint16_t)(k + 3); val_out[pos] = v.w; }
                    }
                }
                const unsigned tm = __ballot_sync(0xffffffffu, nzw & 2u);
                if (nzw & 2u) {
                    const int e = (q1 << 2) + lane;
                    const int pos = w + __popc(tm & lt);
                    col_out[pos] = (uint16_t)(e - e0); val_out[pos] = base[e];
                }
            }
            // average, int8 test and hashes: order-free, so every lane walks its own non-zero units
            // (SKIPAVG: a row that does not fit the packed CSR has nothing left to do here: 1.25 M shared 64-bit atomics per
            // 1024 x 1225 dense instance otherwise)
            uint64_t hp = 0, hn = 0;
            for (uint32_t m = (SKIPAVG && !fits) ? 0u : nzw; m; m &= m - 1) {
                const int bit = __ffs(m) - 1;
                if (bit < 2) {
                    const int e = bit == 0 ? e0 + lane : (q1 << 2) + lane;
                    gen_elem<SKIPAVG>(base[e], e - e0, av, fits, inv, avg_fx, s_cnt, hp, hn);
                } else {
                    const int q = q0 + lane + 32 * (bit - 2), k = (q << 2) - e0;
                    const float4 v = b4[q];
                    if (v.x != 0.f) gen_elem<SKIPAVG>(v.x, k, av, fits, inv, avg_fx, s_cnt, hp, hn);
                    if (v.y != 0.f) gen_elem<SKIPAVG>(v.y, k + 1, av, fits, inv, avg_fx, s_cnt, hp, hn);
                    if (v.z != 0.f) gen_elem<SKIPAVG>(v.z, k + 2, av, fits, inv, avg_fx, s_cnt, hp, hn);
                    if (v.w != 0.f) gen_elem<SKIPAVG>(v.w, k + 3, av, fits, inv, avg_fx, s_cnt, hp, hn);
                }
            }
            if (nv) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    hp += __shfl_xor_sync(0xffffffffu, hp, o);
                    hn += __shfl_xor_sync(0xffffffffu, hn, o);
                }
                if (lane == 0) {
                    rowinfo[row_id] = make_int2(cnt, off);
                    hash_out[row_id] = make_ulonglong2(hp, hn);
                }
            }
            __syncwarp();       // a general row reads its slot until here
            if (lane == 0 && it + S < nit) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue(it + S);
            }
        }
    }

    // ---- once per instance: totals and the ordered general-row list
    if (lane == 0) {
        atomicAdd(&s_cnt[0], w_nvalid); atomicAdd(&s_cnt[1], w_navg);
        atomicAdd(&s_cnt[2], w_ngen); atomicAdd(&s_cnt[3], w_gennnz);
        s_max[warp] = w_l1max; s_max[NW + warp] = w_l2max;
    }
    __syncthreads();
    {   // rows are split into NW contiguous chunks; warp-ballot compaction inside, chunk bases via s_cnt[8..]
        const int chunk = (p.m_max + NW - 1) / NW;
        const int r0 = warp * chunk, r1 = min(r0 + chunk, p.m_max);
        int mine = 0;
        for (int r = r0 + lane; r < r1 + lane; r += 32) {
            const bool g = r < r1 && rowinfo[r].x > 0;
            mine += __popc(__ballot_sync(0xffffffffu, g));
        }
        if (lane == 0) s_cnt[8 + warp] = mine;
        __syncthreads();
        int basei = 0;
        for (int w2 = 0; w2 < warp; ++w2) basei += s_cnt[8 + w2];
        int4* gen_out = p.gen4 + (size_t)b * p.m_max;
        for (int r = r0 + lane; r < r1 + lane; r += 32) {
            const bool g = r < r1 && rowinfo[r].x > 0;
            const unsigned m = __ballot_sync(0xffffffffu, g);
            if (g) {
                const int2 ri = rowinfo[r];
                gen_out[basei + __popc(m & ((1u << lane) - 1u))] = make_int4(r, ri.x, ri.y, 0);
            }
            basei += __popc(m);
        }
    }
    int nsc = 0;
    for (int k = tid; k < (int)(p.dpad / 4); k += NT) {
        const unsigned wv = ctype_w[k];
        nsc += ((wv & 0xffu) != 0) + ((wv & 0xff00u) != 0) + ((wv & 0xff0000u) != 0) + ((wv & 0xff000000u) != 0);
    }
    for (int o = 16; o > 0; o >>= 1) nsc += __shfl_xor_sync(0xffffffffu, nsc, o);
    if (lane == 0 && nsc) atomicAdd(&s_cnt[4], nsc);
    __syncthreads();
    const float ninv = 1.f / (float)max(s_cnt[1], 1);
    float* avg_out = p.avg + (size_t)b * p.dpad;
    for (int k = tid; k < (int)p.dpad; k += NT) {
        float acc = 0.f;
        if (k < d) acc = ((float)((double)(long long)avg_fx[k] * (1.0 / 1099511627776.0)) + (float)sing[k]) * ninv;
        avg_out[k] = acc;
    }
    uint32_t* ct_out = (uint32_t*)(p.ctype + (size_t)b * p.dpad);
    for (int k = tid; k < (int)(p.dpad / 4); k += NT) ct_out[k] = ctype_w[k];
    if (tid == 0) {
        float m1 = 0.f, m2 = 0.f;
        for (int w2 = 0; w2 < NW; ++w2) { m1 = fmaxf(m1, s_max[w2]); m2 = fmaxf(m2, s_max[NW + w2]); }
        p.nvalid[b] = s_cnt[0]; p.navg[b] = s_cnt[1]; p.ngen[b] = s_cnt[2]; p.gennnz[b] = s_cnt[3]; p.nsingc[b] = s_cnt[4];
        p.csr_ok[b] = s_cnt[6] ? 0 : (s_cnt[7] ? 1 : 3);       // bit 1: every packed value is an int8
        p.maxl1[b] = m1; p.maxl2[b] = m2;
    }
}

size_t scan_rows_smem_bytes(int d, int m_max, int NW, int S, size_t* rowbuf_out) {
    const size_t rowbuf = align_up((size_t)d * 4 + 32, 128);
    const int64_t dpad = (int64_t)align_up((size_t)d, 16);
    size_t o = (size_t)NW * S * rowbuf + (size_t)d * 8 + (size_t)d * 4 + 8;
    o += (size_t)m_max * 8 + (size_t)NW * S * 8 + 16 * 4 + 2 * NW * 4 + 16 + (size_t)dpad;
    if (rowbuf_out) *rowbuf_out = rowbuf;
    return align_up(o, 16);
}

size_t scan_smem_bytes(int d, int R, int stages, size_t* stage_stride_out) {
    const size_t stride = align_up((size_t)R * d * 4 + 32, 128);
    const int64_t dpad = (int64_t)align_up((size_t)d, 16);
    size_t o = (size_t)stages * stride;
    o += (size_t)d * 8 + 8;             // avg_gen, sing (+ alignment)
    o += (size_t)stages * 8;            // mbarriers
    o += (size_t)R * 24;                // row arrays
    o += 8 * 4 + 16;                    // counters (+ alignment)
    o += (size_t)dpad;                  // ctype
    if (stage_stride_out) *stage_stride_out = stride;
    return align_up(o, 16);
}

cudaError_t launch_scan(const ScanParams& p0, cudaStream_t stream) {
    ScanParams p = p0;
    constexpr int NT = 256;
    {   // warp-streaming kernel whenever eight row rings fit in shared memory: depth 2 with two CTAs
        // per SM if that fits (more independent row streams), else depth 3 with one CTA per SM
        const char* force = getenv("CAVE_SCAN_KERNEL");
        const char* sdepth = getenv("CAVE_SCAN_STAGES");
        size_t rowbuf = 0;
        int S = 2;
        size_t smem = scan_rows_smem_bytes(p.d, p.m_max, NT / 32, 2, &rowbuf);
        if (smem > 113 * 1024 || (sdepth && sdepth[0] == '3')) { S = 3; smem = scan_rows_smem_bytes(p.d, p.m_max, NT / 32, 3, &rowbuf); }
        if (smem <= 220 * 1024 && !(force && force[0] == 't')) {
            p.stage_stride = rowbuf; p.R = 1; p.stages = S;
            static size_t configured2[64] = {0}, configured3[64] = {0};     // per device: the attribute is a per-device property
            int dev = 0;
            if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
            size_t& conf = S == 2 ? configured2[dev] : configured3[dev];
            void (*kern)(ScanParams) = p.skip_avg ? (S == 2 ? scan_rows_kernel<NT, 2, true> : scan_rows_kernel<NT, 3, true>)
                                                  : (S == 2 ? scan_rows_kernel<NT, 2> : scan_rows_kernel<NT, 3>);
            if (smem > conf || p.skip_avg) {        // (the skip-average instantiations are rare: set their attribute every time)
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
                if (!p.skip_avg) conf = smem;
            }
            kern<<<dim3((unsigned)p.B), dim3(NT), smem, stream>>>(p);
            return cudaGetLastError();
        }
    }
    // tile = R rows, about 20 KB; ring depth 4 unless shared memory runs out
    int R = (int)(20480 / ((size_t)p.d * 4));
    R = R < 1 ? 1 : (R > 32 ? 32 : R);
    int stages = 4;
    size_t stride = 0, smem = scan_smem_bytes(p.d, R, stages, &stride);
    while (smem > 200 * 1024 && stages > 2) { --stages; smem = scan_smem_bytes(p.d, R, stages, &stride); }
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    p.R = R; p.stages = stages; p.stage_stride = stride;
    static size_t configured[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
    if (smem > configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(scan_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured[dev] = smem;
    }
    scan_kernel<NT><<<dim3((unsigned)p.B), dim3(NT), smem, stream>>>(p);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Sparse ingestion: the same pack, built from the non-zeros of the rows (CSR per instance) instead of the dense
// [B, m_max, d] tensor — 90 KB instead of 6.5 MB per TSP-50 instance cross PCIe / HBM.  Row classification, thresholds,
// the 2^-40 fixed-point average, hashes and the packed CSR are those of scan_rows_kernel (for integer-valued rows the
// pack content is identical; for other values the row norms may differ in the last bit: different summation order).
// One CTA per instance, one warp per row.  Columns inside a row must be ascending; explicit zeros are skipped.
struct SparseScanParams {
    const long long* inst_off;      // [B + 1] first row of every instance in row_ptr
    const long long* row_ptr;       // [R + 1]
    const int* col; const float* val;
    ScanParams pk;                  // pack pointers (A unused)
};
constexpr int kSparseThreads = 256;
__host__ __device__ inline size_t sparse_scan_smem_bytes(int d, int m_max, int64_t dpad) {
    return (size_t)d * 12 + 16 + (size_t)m_max * 8 + 64 + 16 * 4 + 2 * (kSparseThreads / 32) * 4 + 16 + (size_t)dpad + 64;
}
__global__ void __launch_bounds__(kSparseThreads) scan_sparse_kernel(SparseScanParams q) {
    extern __shared__ __align__(128) unsigned char smem[];
    const ScanParams& p = q.pk;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NT = kSparseThreads, NW = NT / 32;
    const int d = p.d, b = blockIdx.x;
    unsigned long long* avg_fx = (unsigned long long*)smem;                          // [d]
    int* sing = (int*)(avg_fx + d);                                                  // [d]
    int2* rowinfo = (int2*)align_up((size_t)(sing + d), 8);                         // [m_max]
    int* s_cnt = (int*)(rowinfo + p.m_max);                                         // [16 + NW]
    float* s_max = (float*)(s_cnt + 16 + NW);                                       // [2 * NW]
    unsigned* ctype_w = (unsigned*)align_up((size_t)(s_max + 2 * NW), 16);          // [dpad / 4]
    const long long r_first = q.inst_off[b];
    long long nrows = q.inst_off[b + 1] - r_first;
    const int m_b = (int)(nrows < 0 ? 0 : (nrows > p.m_max ? p.m_max : nrows));
    for (int k = tid; k < d; k += NT) { avg_fx[k] = 0ull; sing[k] = 0; }
    for (int k = tid; k < (int)(p.dpad / 4); k += NT) ctype_w[k] = 0u;
    for (int k = tid; k < p.m_max; k += NT) rowinfo[k] = make_int2(0, 0);
    if (tid < 16 + NW) s_cnt[tid] = 0;
    __syncthreads();
    int w_nvalid = 0, w_navg = 0, w_gennnz = 0, w_ngen = 0;
    float w_l1max = 0.f, w_l2max = 0.f;
    uint16_t* col_out = p.csr_col + (size_t)b * p.cap_nnz;
    float* val_out = p.csr_val + (size_t)b * p.cap_nnz;
    ulonglong2* hash_out = p.ghash + (size_t)b * p.m_max;
    for (int row_id = warp; row_id < m_b; row_id += NW) {
        const long long e0 = q.row_ptr[r_first + row_id], e1 = q.row_ptr[r_first + row_id + 1];
        RowAcc acc; acc.l1 = 0.f; acc.l2 = 0.f; acc.lv = 0.f; acc.lk = -1; acc.n = 0;
        for (long long e = e0 + lane; e < e1; e += 32) {
            const float v = q.val[e];
            const int k = q.col[e];
            if (v != 0.f && k >= 0 && k < d) acc.add(v, k);
        }
        int cnt = acc.n;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        const unsigned sawm = __ballot_sync(0xffffffffu, acc.n > 0);
        if (cnt == 1) {
            const int src = __ffs(sawm) - 1;
            const int k1 = __shfl_sync(0xffffffffu, acc.lk, src);
            const float v1 = __shfl_sync(0xffffffffu, acc.lv, src);
            const bool nv = fabsf(v1) > 1e-7f, av = sqrtf(v1 * v1) > 1e-7f;
            w_nvalid += nv; w_navg += av;
            if (lane == 0) {
                if (nv) atomicOr(&ctype_w[k1 >> 2], (v1 > 0.f ? 1u : 2u) << ((k1 & 3) * 8));
                if (av) atomicAdd(&sing[k1], v1 > 0.f ? 1 : -1);
            }
        } else if (cnt >= 2) {
            float a1 = acc.l1, a2 = acc.l2;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { a1 += __shfl_xor_sync(0xffffffffu, a1, o); a2 += __shfl_xor_sync(0xffffffffu, a2, o); }
            const float nrm = sqrtf(a2);
            const bool nv = a1 > 1e-7f, av = nrm > 1e-7f;
            const float inv = av ? 1.f / fmaxf(nrm, 1e-8f) : 0.f;
            w_nvalid += nv; w_navg += av;
            int off = 0;
            bool fits = false;
            if (nv) {
                if (lane == 0) off = atomicAdd(&s_cnt[5], cnt);
                off = __shfl_sync(0xffffffffu, off, 0);
                fits = off + cnt <= p.cap_nnz;
                if (!fits && lane == 0) s_cnt[6] = 1;
                w_gennnz += cnt; ++w_ngen;
                w_l1max = fmaxf(w_l1max, a1); w_l2max = fmaxf(w_l2max, a2);
            }
            uint64_t hp = 0, hn = 0;
            int w = off;
            for (long long eb = e0; eb < e1; eb += 32) {
                const long long e = eb + lane;
                float v = 0.f; int k = 0;
                if (e < e1) { v = q.val[e]; k = q.col[e]; if (k < 0 || k >= d) v = 0.f; }
                const unsigned nzm = __ballot_sync(0xffffffffu, v != 0.f);
                if (v != 0.f) {
                    if (av) atomicAdd(&avg_fx[k], (unsigned long long)__double2ll_rn((double)v * (double)inv * 1099511627776.0));
                    if (fits) {
                        const int pos = w + __popc(nzm & ((1u << lane) - 1u));
                        col_out[pos] = (uint16_t)k; val_out[pos] = v;
                        if (!(v == (float)(int)v && fabsf(v) <= 127.f)) s_cnt[7] = 1;
                        const uint32_t bits = __float_as_uint(v);
                        hp += mix64d(((uint64_t)k << 32) | bits);
                        hn += mix64d(((uint64_t)k << 32) | (bits ^ 0x80000000u));
                    }
                }
                w += __popc(nzm);
            }
            if (nv) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { hp += __shfl_xor_sync(0xffffffffu, hp, o); hn += __shfl_xor_sync(0xffffffffu, hn, o); }
                if (lane == 0) { rowinfo[row_id] = make_int2(cnt, off); hash_out[row_id] = make_ulonglong2(hp, hn); }
            }
        }
        __syncwarp();
    }
    // ---- once per instance: totals and the ordered general-row list (as in scan_rows_kernel)
    if (lane == 0) {
        atomicAdd(&s_cnt[0], w_nvalid); atomicAdd(&s_cnt[1], w_navg);
        atomicAdd(&s_cnt[2], w_ngen); atomicAdd(&s_cnt[3], w_gennnz);
        s_max[warp] = w_l1max; s_max[NW + warp] = w_l2max;
    }
    __syncthreads();
    {
        const int chunk = (p.m_max + NW - 1) / NW;
        const int r0 = warp * chunk, r1 = min(r0 + chunk, p.m_max);
        int mine = 0;
        for (int r = r0 + lane; r < r1 + lane; r += 32) {
            const bool g = r < r1 && rowinfo[r].x > 0;
            mine += __popc(__ballot_sync(0xffffffffu, g));
        }
        if (lane == 0) s_cnt[16 + warp] = mine;
        __syncthreads();
        int basei = 0;
        for (int w2 = 0; w2 < warp; ++w2) basei += s_cnt[16 + w2];
        int4* gen_out = p.gen4 + (size_t)b * p.m_max;
        for (int r = r0 + lane; r < r1 + lane; r += 32) {
            const bool g = r < r1 && rowinfo[r].x > 0;
            const unsigned m = __ballot_sync(0xffffffffu, g);
            if (g) {
                const int2 ri = rowinfo[r];
                gen_out[basei + __popc(m & ((1u << lane) - 1u))] = make_int4(r, ri.x, ri.y, 0);
            }
            basei += __popc(m);
        }
    }
    int nsc = 0;
    for (int k = tid; k < (int)(p.dpad / 4); k += NT) {
        const unsigned wv = ctype_w[k];
        nsc += ((wv & 0xffu) != 0) + ((wv & 0xff00u) != 0) + ((wv & 0xff0000u) != 0) + ((wv & 0xff000000u) != 0);
    }
    for (int o = 16; o > 0; o >>= 1) nsc += __shfl_xor_sync(0xffffffffu, nsc, o);
    if (lane == 0 && nsc) atomicAdd(&s_cnt[4], nsc);
    __syncthreads();
    const float ninv = 1.f / (float)max(s_cnt[1], 1);
    float* avg_out = p.avg + (size_t)b * p.dpad;
    for (int k = tid; k < (int)p.dpad; k += NT) {
        float acc = 0.f;
        if (k < d) acc = ((float)((double)(long long)avg_fx[k] * (1.0 / 1099511627776.0)) + (float)sing[k]) * ninv;
        avg_out[k] = acc;
    }
    uint32_t* ct_out = (uint32_t*)(p.ctype + (size_t)b * p.dpad);
    for (int k = tid; k < (int)(p.dpad / 4); k += NT) ct_out[k] = ctype_w[k];
    if (tid == 0) {
        float m1 = 0.f, m2 = 0.f;
        for (int w2 = 0; w2 < NW; ++w2) { m1 = fmaxf(m1, s_max[w2]); m2 = fmaxf(m2, s_max[NW + w2]); }
        p.nvalid[b] = s_cnt[0]; p.navg[b] = s_cnt[1]; p.ngen[b] = s_cnt[2]; p.gennnz[b] = s_cnt[3]; p.nsingc[b] = s_cnt[4];
        p.csr_ok[b] = s_cnt[6] ? 0 : (s_cnt[7] ? 1 : 3);
        p.maxl1[b] = m1; p.maxl2[b] = m2;
    }
}

cudaError_t launch_scan_sparse(const ScanParams& pk, const long long* inst_off, const long long* row_ptr, const int* col,
                               const float* val, cudaStream_t stream) {
    SparseScanParams q;
    q.inst_off = inst_off; q.row_ptr = row_ptr; q.col = col; q.val = val; q.pk = pk;
    const size_t smem = sparse_scan_smem_bytes(pk.d, pk.m_max, pk.dpad);
    if (smem > 220 * 1024) return cudaErrorInvalidValue;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(scan_sparse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    scan_sparse_kernel<<<dim3((unsigned)pk.B), dim3(kSparseThreads), smem, stream>>>(q);
    return cudaGetLastError();
}

// ---- plan kernel: one warp per instance estimates the solver's shared-memory footprint (general rows, rows
// that will merge into +- pairs by hash, non-zeros kept) and reduces it into the batch statistics from which
// the solve kernel's launch configuration is chosen on the device (layout.cuh).  Integer sums and maxima:
// order independent, hence reproducible.
constexpr int kPlanMaxRows = 512;       // hashes staged per warp; beyond that the pair estimate is skipped
__global__ void __launch_bounds__(256) plan_kernel(PlanParams p) {
    __shared__ unsigned long long hp[8][kPlanMaxRows];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int b = blockIdx.x * 8 + w;
    if (b == 0 && lane == 0) p.plan[PLAN_WIDE] = wide_config_enabled(p.m_max, p.d) ? (unsigned long long)p.wide_smem : 0ull;
    if (b >= p.B) return;
    const int ngen = p.ngen[b], nnz = p.gennnz[b], ok = p.csr_ok[b];
    const bool dense_path = p.nsingc[b] == 0;
    int paired = 0;
    if (ngen > 0 && !dense_path && (ok & 1) && ngen <= kPlanMaxRows) {
        const int4* gen = p.gen4 + (size_t)b * p.m_max;
        const ulonglong2* gh = p.ghash + (size_t)b * p.m_max;
        unsigned long long want[kPlanMaxRows / 32];
#pragma unroll
        for (int u = 0; u < kPlanMaxRows / 32; ++u) {
            const int i = u * 32 + lane;
            want[u] = 0;
            if (i < ngen) { const ulonglong2 h = gh[gen[i].x]; hp[w][i] = h.x; want[u] = h.y; }
        }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < kPlanMaxRows / 32; ++u) {
            const int i = u * 32 + lane;
            if (u * 32 < ngen) {
                bool hit = false;
                for (int j = 0; j < ngen; ++j) hit |= (j != i) & (hp[w][j] == want[u]);
                paired += (i < ngen && hit) ? 1 : 0;
            }
        }
        for (int o = 16; o > 0; o >>= 1) paired += __shfl_xor_sync(0xffffffffu, paired, o);
    }
    if (lane == 0) {
        const int nv = ngen - paired / 2;
        const long long nnz_kept = ngen > 0 ? (long long)nnz * nv / ngen : 0;
        const bool skip = p.nvalid[b] == 0;
        size_t hot8, work8, hot4, work4;
        instance_footprint(p.d, skip ? 0 : ngen, nv, nnz_kept, (ok & 3) == 3, dense_path, 8, &hot8, &work8);
        instance_footprint(p.d, skip ? 0 : ngen, nv, nnz_kept, (ok & 3) == 3, dense_path, 4, &hot4, &work4);
        // cost estimate for the work queue order: non-zeros swept per iteration + the dense part of the Newton system
        long long key = skip ? 0 : (dense_path ? (long long)ngen * p.d : nnz_kept + 16ll * nv);
        p.okey[b] = (int)(key > 0x7fffffffll ? 0x7fffffffll : key);
        atomicAdd(p.plan + PLAN_N, 1ull);
        atomicAdd(p.plan + PLAN_SUM8, (unsigned long long)work8);
        atomicAdd(p.plan + PLAN_SUM4, (unsigned long long)work4);
        atomicMax(p.plan + PLAN_MAXHOT8, (unsigned long long)hot8);
        atomicMax(p.plan + PLAN_MAXHOT4, (unsigned long long)hot4);
    }
}

// ---- order kernel: order[rank] = b with rank(b) = number of instances that cost more (ties: lower index first).
// Rank by counting, one warp per instance, O(B^2) comparisons in total: a few microseconds at the batch sizes
// where the order matters; larger batches keep the index order.
__global__ void __launch_bounds__(256) order_kernel(PlanParams p) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= p.B) return;
    if (p.B > kOrderMaxBatch) { if (lane == 0) p.order[b] = b; return; }
    const int mine = p.okey[b];
    int rank = 0;
    for (int j = lane; j < p.B; j += 32) {
        const int k = p.okey[j];
        rank += (k > mine) | ((k == mine) & (j < b));
    }
    for (int o = 16; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
    if (lane == 0) p.order[rank] = b;
}

// ---- setup kernel: the per-instance setup of the Newton path, computed ONCE per pack (A_i is constant across epochs,
// SURVEY.md 7.2) instead of in every solve: +- merge of the general rows (hash match + exact comparison), the kept rows
// as int8 CSR over variables, and the CSC (count, scan, cursor fill, per-column sort by variable => fixed summation
// order).  One CTA per instance; results go to the instance's SetupBlock in the pack (layout.cuh); the solver's
// nw_setup turns into a copy-in.  Only integer-valued instances with a complete packed CSR are cached (every shipped
// model); the others keep the in-solver setup.
constexpr int kSetupThreads = 128;
__host__ __device__ inline size_t setup_smem_bytes(int64_t cap_v, int64_t d) {
    return (size_t)cap_v * (8 + 8 + 4 + 4 + 4 + 4 + 1) + 64 + (size_t)(d + 2) * 8 + 64;
}
__global__ void __launch_bounds__(kSetupThreads) setup_kernel(PlanParams p, int enabled) {
    extern __shared__ __align__(16) char ssm[];
    __shared__ int s_nv, s_nz;
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = kSetupThreads / 32;
    char* blk = p.setup + (size_t)b * p.setup_stride;
    int* hdr = (int*)blk;
    const int mB = p.ngen[b], d = p.d;
    const bool eligible = enabled && p.nsingc[b] > 0 && mB > 0 && (p.csr_ok[b] & 3) == 3 && mB <= p.setup_cap_v && p.nvalid[b] > 0;
    if (!eligible) { if (tid == 0) hdr[0] = 0; return; }
    const SetupBlock SB = make_setup_block(p.setup_cap_v, p.cap_nnz, d);
    const int cv = (int)p.setup_cap_v;
    unsigned long long* hpos = (unsigned long long*)ssm;
    unsigned long long* hneg = hpos + cv;
    int* goff = (int*)(hneg + cv);
    int* gcnt = goff + cv + 1;
    int* cand = gcnt + cv + 1;          // later: row pointers over variables
    int* keep = cand + cv + 2;          // variable -> general row
    int* cnt = keep + cv + 1;           // [d + 2] column counts / pointers
    int* cur = cnt + d + 2;             // [d + 1] fill cursors
    unsigned char* rtype = (unsigned char*)(cur + d + 1);
    const int4* gen = p.gen4 + (size_t)b * p.m_max;
    const ulonglong2* gh = p.ghash + (size_t)b * p.m_max;
    const uint16_t* pcol = p.csr_col + (size_t)b * p.cap_nnz;
    const float* pval = p.csr_val + (size_t)b * p.cap_nnz;
    for (int i = tid; i < mB; i += kSetupThreads) {
        const int4 g = gen[i]; gcnt[i] = g.y; goff[i] = g.z;
        const ulonglong2 h = gh[g.x]; hpos[i] = h.x; hneg[i] = h.y;
    }
    for (int k = tid; k <= d + 1; k += kSetupThreads) cnt[k] = 0;
    __syncthreads();
    // merge b_j = -b_i: cand[i] = smallest j != i with row_j == -row_i; merged iff the choice is mutual
    for (int i = warp; i < mB; i += NW) {
        const int pi = goff[i], ni = gcnt[i];
        const unsigned long long want = hneg[i];
        int c0 = -1;
        for (int j0 = 0; j0 < mB && c0 < 0; j0 += 32) {
            const int j = j0 + lane;
            const bool hit = j < mB && j != i && hpos[j] == want && gcnt[j] == ni;
            unsigned m = __ballot_sync(0xffffffffu, hit);
            while (m && c0 < 0) {
                const int jj = j0 + __ffs(m) - 1;
                const int pj = goff[jj];
                bool ok = true;
                for (int e = lane; e < ni; e += 32) ok = ok & (pcol[pi + e] == pcol[pj + e]) & (pval[pi + e] == -pval[pj + e]);
                if (!__ballot_sync(0xffffffffu, !ok)) c0 = jj;
                m &= m - 1;
            }
        }
        if (lane == 0) cand[i] = c0;
    }
    __syncthreads();
    for (int i = tid; i < mB; i += kSetupThreads) {
        const int j = cand[i];
        rtype[i] = (j >= 0 && cand[j] == i) ? (i < j ? 1 : 2) : 0;
    }
    __syncthreads();
    unsigned char* o_vfree = (unsigned char*)(blk + SB.vfree);
    int* o_rptr = (int*)(blk + SB.rptr);
    int* o_cptr = (int*)(blk + SB.cptr);
    uint16_t* o_rcol = (uint16_t*)(blk + SB.rcol);
    uint16_t* o_crow = (uint16_t*)(blk + SB.crow);
    signed char* o_rval = (signed char*)(blk + SB.rval);
    signed char* o_cval = (signed char*)(blk + SB.cval);
    int* rp = cand;                     // reused: row pointers over variables
    if (warp == 0) {                    // ordered compaction of the kept rows + exclusive scan of their lengths
        int nvb = 0, run = 0;
        for (int i0 = 0; i0 < mB; i0 += 32) {
            const int i = i0 + lane;
            const bool kp = i < mB && rtype[i] != 2;
            const unsigned m = __ballot_sync(0xffffffffu, kp);
            int len = kp ? gcnt[i] : 0, incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
            if (kp) {
                const int v = nvb + __popc(m & ((1u << lane) - 1u));
                keep[v] = i; o_vfree[v] = (unsigned char)(rtype[i] == 1);
                const int start = run + incl - len;
                rp[v] = start; o_rptr[v] = start;
            }
            nvb += __popc(m);
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) { rp[nvb] = run; o_rptr[nvb] = run; s_nv = nvb; s_nz = run; }
    }
    __syncthreads();
    const int nv = s_nv, nz = s_nz;
    // kept rows -> int8 CSR of the block; column counts
    for (int v = warp; v < nv; v += NW) {
        const int src = goff[keep[v]], dst = rp[v], n = rp[v + 1] - dst;
        for (int e = lane; e < n; e += 32) {
            const uint16_t c = pcol[src + e];
            o_rcol[dst + e] = c; o_rval[dst + e] = (signed char)pval[src + e];
            atomicAdd(&cnt[c + 1], 1);
        }
    }
    __syncthreads();
    if (warp == 0) {                    // inclusive scan of cnt[1..d]: cnt[k] becomes the column pointer
        int carry = 0;
        for (int k0 = 1; k0 <= d; k0 += 32) {
            const int k = k0 + lane;
            int v = k <= d ? cnt[k] : 0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += u; }
            v += carry;
            if (k <= d) cnt[k] = v;
            carry = __shfl_sync(0xffffffffu, v, 31);
        }
    }
    __syncthreads();
    for (int k = tid; k <= d; k += kSetupThreads) { o_cptr[k] = cnt[k]; if (k < d) cur[k] = cnt[k]; }
    __syncthreads();
    // CSC fill, ordered by construction: every warp owns a range of columns and walks the kept rows in ascending variable
    // order, placing the entries whose column falls into its range (the columns of one row are distinct, so the cursors need
    // no atomics and every column comes out sorted by variable: no sort, a fixed summation order for the solver).  The next
    // row's entries are fetched while the current one is placed (rows of up to 256 non-zeros; longer rows take the loop).
    {
        const int c_lo = (int)(((long long)d * warp) / NW), c_hi = (int)(((long long)d * (warp + 1)) / NW);
        constexpr int U = 8;
        int cc[U]; float vv[U];
        auto fetch = [&](int v) {
            const int src = goff[keep[v]], n = rp[v + 1] - rp[v];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int e = lane + 32 * u;
                cc[u] = e < n ? (int)pcol[src + e] : -1;
                vv[u] = e < n ? pval[src + e] : 0.f;
            }
        };
        if (nv > 0) fetch(0);
        for (int v = 0; v < nv; ++v) {
            int c0[U]; float v0[U];
#pragma unroll
            for (int u = 0; u < U; ++u) { c0[u] = cc[u]; v0[u] = vv[u]; }
            const int n = rp[v + 1] - rp[v];
            if (v + 1 < nv) fetch(v + 1);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (c0[u] >= c_lo && c0[u] < c_hi) {
                    const int q = cur[c0[u]]; cur[c0[u]] = q + 1;
                    o_crow[q] = (uint16_t)v; o_cval[q] = (signed char)v0[u];
                }
            }
            if (n > 32 * U) {
                const int src = goff[keep[v]];
                for (int e = 32 * U + lane; e < n; e += 32) {
                    const int c = pcol[src + e];
                    if (c >= c_lo && c < c_hi) { const int q = cur[c]; cur[c] = q + 1; o_crow[q] = (uint16_t)v; o_cval[q] = (signed char)pval[src + e]; }
                }
            }
            __syncwarp();
        }
    }
    if (tid == 0) {
        hdr[1] = nv; hdr[2] = nz;
        hdr[3] = (int)SB.vfree; hdr[4] = (int)SB.rptr; hdr[5] = (int)SB.cptr; hdr[6] = (int)SB.rcol; hdr[7] = (int)SB.crow;
        hdr[8] = (int)SB.rval; hdr[9] = (int)SB.cval;
        hdr[0] = 1;
    }
}

__global__ void clear_setup_kernel(char* setup, long long stride, int B) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) *(int*)(setup + (size_t)b * (size_t)stride) = 0;
}
// packs without a cached setup: the valid word of every instance's setup block says so
cudaError_t launch_clear_setup(char* setup, long long stride, int B, cudaStream_t stream) {
    clear_setup_kernel<<<(unsigned)((B + 255) / 256), 256, 0, stream>>>(setup, stride, B);
    return cudaGetLastError();
}

cudaError_t launch_plan(const PlanParams& p, cudaStream_t stream) {
    plan_kernel<<<dim3((unsigned)((p.B + 7) / 8)), dim3(256), 0, stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    order_kernel<<<dim3((unsigned)((p.B + 7) / 8)), dim3(256), 0, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess || !p.setup) return e;
    const size_t smem = setup_smem_bytes(p.setup_cap_v, p.d);
    const char* off = getenv("CAVE_SETUP_CACHE");
    const int enabled = (smem <= 200 * 1024 && !(off && off[0] == '0')) ? 1 : 0;
    const size_t use = enabled ? smem : 0;
    if (use > 48 * 1024) {
        e = cudaFuncSetAttribute(setup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)use);
        if (e != cudaSuccess) return e;
    }
    setup_kernel<<<dim3((unsigned)p.B), dim3(kSetupThreads), use, stream>>>(p, enabled);
    return cudaGetLastError();
}

}  // namespace cave
