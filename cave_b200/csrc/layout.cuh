// Device-resident layouts shared by the scan kernel, the solve kernel and the C ABI.
#pragma once
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define CAVE_HD __host__ __device__ inline
#else
#define CAVE_HD inline
#endif

namespace cave {

CAVE_HD size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// The "pack": everything the solver needs to know about A besides the general rows themselves.
//   nvalid[B]   rows with sum|a| > 1e-7            (the NNLS row mask, src/cave.py:303)
//   navg[B]     rows with ||a||_2 > 1e-7           (the average's row mask, src/cave.py:224-225)
//   ngen[B]     valid rows with >= 2 non-zeros     ("general" rows)
//   gennnz[B]   non-zeros in the general rows
//   nsingc[B]   coordinates that own at least one singleton row
//   gen[B, m_max]   int4 (row index, nnz, offset into the packed CSR, 0) of every general row, ascending row
//                   (offsets need not be monotone: rows are placed as they are scanned)
//   ctype[B, dpad]  per coordinate: bit0 = a row +a*e_k exists, bit1 = a row -a*e_k exists
//   avg[B, dpad]    float32 average unit normal     (src/cave.py:222-228)
//   csrok[B], maxl1[B], maxl2[B]   packed-CSR complete flag; max ||a||_1, max ||a||_2^2 over general rows
//   ghash[B, m_max]   indexed by ROW: order-free 64-bit hashes of the row and of its negation (general rows only)
//   csr_col/val[B, cap_nnz]   the general rows' non-zeros, row after row, columns ascending
//   plan[8]     uint64 batch statistics written by the plan kernel (see PlanStats): the solve kernel's
//               launch configuration is chosen from them on the device, without a host round trip
//   okey[B], order[B]   per-instance cost estimate and the instances sorted by it, most expensive first: the order
//               in which the solve kernel's persistent CTAs take them (shortens the drain at the end of the kernel)
//   setup[B, setup_stride]   per-instance solver setup emitted once by the setup kernel (A_i is constant across epochs:
//               SURVEY.md 7.2): +- merge result, the kept rows as int8 CSR and the CSC over variables, i.e. everything
//               nw_setup would otherwise recompute in every call; see SetupBlock
struct PackLayout {
    size_t nvalid, navg, ngen, gennnz, nsingc, gen, ctype, avg, csrok, maxl1, maxl2, ghash, csr_col, csr_val, plan, okey, order, setup, total;
    int64_t dpad, cap_nnz, setup_stride, setup_cap_v;
};

// Cached setup of one structured instance (integer-valued rows only: every shipped model).  Byte offsets inside the block:
//   [0]   int32 header: valid, nv (variables after the +- merge), nnz (non-zeros kept), then the byte offsets of the
//         seven arrays below (64 bytes)
//   vfree u8[cap_v]      variable is sign-free (a merged +- pair)
//   rptr  i32[cap_v + 1] CSR row pointers over variables
//   cptr  i32[d + 1]     CSC column pointers
//   rcol  u16[cap_z]  crow u16[cap_z]  rval i8[cap_z]  cval i8[cap_z]
struct SetupBlock { size_t vfree, rptr, cptr, rcol, crow, rval, cval, total; };
// instances with more general rows than this keep the in-solver setup (every shipped model has far fewer: TSP-50 ~110,
// TSP-100 ~210); a small cap keeps the setup kernel's shared memory small, i.e. many instances in flight per SM
CAVE_HD int64_t setup_cap_v(int64_t m_max) { return m_max < 256 ? m_max : 256; }
CAVE_HD SetupBlock make_setup_block(int64_t cap_v, int64_t cap_z, int64_t d) {
    SetupBlock S;
    size_t o = 64;
    S.vfree = o; o = align_up(o + (size_t)cap_v, 16);
    S.rptr = o;  o = align_up(o + (size_t)(cap_v + 1) * 4, 16);
    S.cptr = o;  o = align_up(o + (size_t)(d + 1) * 4, 16);
    S.rcol = o;  o = align_up(o + (size_t)cap_z * 2, 16);
    S.crow = o;  o = align_up(o + (size_t)cap_z * 2, 16);
    S.rval = o;  o = align_up(o + (size_t)cap_z, 16);
    S.cval = o;  o = align_up(o + (size_t)cap_z, 16);
    S.total = align_up(o, 256);
    return S;
}

// Warm-start state of a resident pack (cave_forward_backward_warm): one slot per pack instance, in a caller-owned buffer.
//   [0]  int32 header: valid (1), nv (variables after the +- merge), tag (hash of the variable -> row map and of the
//        sign-free flags, solver_core.cuh warm_tag), 0
//   [16] float64 nu[cap_v]: the multipliers of the last converged Newton solve, in the solver's variable order
// An all-zero buffer is a buffer of empty slots.  Instances with more variables than cap_v are never stored.
CAVE_HD int64_t warm_cap_v(int64_t m_max) { return m_max < 256 ? m_max : 256; }
CAVE_HD size_t warm_slot_bytes(int64_t m_max) { return align_up(16 + (size_t)warm_cap_v(m_max) * 8, 16); }
// Warm-start state of the dense Gram-space Newton solve (cave_forward_backward_warm_ex), a second caller-owned buffer with
// one slot per pack instance:
//   [0]  int32 header: valid (1), m (general rows), tag (hash of m and of every row's index and length, dense_solve.cu
//        dense_warm_tag), flags (bit 0: the solve ended with the diagonal metric)
//   [16] float64 lam[cap]: the multipliers of the last converged dense solve, in the instance's general-row order
// An all-zero buffer is a buffer of empty slots.  The dense path takes at most 2048 rows, so every dense instance fits.
CAVE_HD int64_t dense_warm_cap(int64_t m_max) { return m_max < 2048 ? m_max : 2048; }
CAVE_HD size_t dense_warm_slot_bytes(int64_t m_max) { return align_up(16 + (size_t)dense_warm_cap(m_max) * 8, 16); }

// per-instance capacity of the packed CSR: every shipped model (TSP/VRP/SP) fits; instances that do
// not (dense general rows) are flagged and the solver reads their rows from A instead
CAVE_HD int64_t pack_cap_nnz(int64_t m_max, int64_t d) {
    int64_t full = m_max * d, c = 16 * d + 4096;
    return (c < full ? c : full + 1) / 8 * 8 + 8;
}

CAVE_HD PackLayout make_pack_layout(int64_t B, int64_t m_max, int64_t d) {
    PackLayout L;
    L.dpad = (int64_t)align_up((size_t)d, 16);
    size_t o = 0;
    L.nvalid = o; o = align_up(o + (size_t)B * 4, 256);
    L.navg = o;   o = align_up(o + (size_t)B * 4, 256);
    L.ngen = o;   o = align_up(o + (size_t)B * 4, 256);
    L.gennnz = o; o = align_up(o + (size_t)B * 4, 256);
    L.nsingc = o; o = align_up(o + (size_t)B * 4, 256);
    L.gen = o;    o = align_up(o + (size_t)B * (size_t)m_max * 16, 256);
    L.ctype = o;  o = align_up(o + (size_t)B * (size_t)L.dpad, 256);
    L.avg = o;    o = align_up(o + (size_t)B * (size_t)L.dpad * 4, 256);
    L.cap_nnz = pack_cap_nnz(m_max, d);
    L.csrok = o;  o = align_up(o + (size_t)B * 4, 256);
    L.maxl1 = o;  o = align_up(o + (size_t)B * 4, 256);
    L.maxl2 = o;  o = align_up(o + (size_t)B * 4, 256);
    L.ghash = o;  o = align_up(o + (size_t)B * (size_t)m_max * 16, 256);
    L.csr_col = o; o = align_up(o + (size_t)B * (size_t)L.cap_nnz * 2, 256);
    L.csr_val = o; o = align_up(o + (size_t)B * (size_t)L.cap_nnz * 4, 256);
    L.plan = o;   o = align_up(o + 64, 256);
    L.okey = o;   o = align_up(o + (size_t)B * 4, 256);
    L.order = o;  o = align_up(o + (size_t)B * 4, 256);
    L.setup_cap_v = setup_cap_v(m_max);
    L.setup_stride = (int64_t)make_setup_block(L.setup_cap_v, L.cap_nnz, d).total;
    L.setup = o;  o = align_up(o + (size_t)B * (size_t)L.setup_stride, 256);
    L.total = o;
    return L;
}

// ---- launch plan of the solve kernel
// The solver is latency bound, so small instances want many small CTAs per SM and large ones few big CTAs.
// Which one applies depends on the data (general rows, +- pairs, non-zeros), which only the device knows
// after the scan; the plan kernel therefore reduces per-instance shared-memory footprints into PlanStats and
// every candidate configuration is launched — the ones the statistics do not select exit at once.  The wide
// configuration (one CTA per SM) is a candidate only for the shapes wide_config_enabled admits.
enum { PLAN_N = 0, PLAN_SUM8 = 1, PLAN_SUM4 = 2, PLAN_MAXHOT8 = 3, PLAN_MAXHOT4 = 4,   // indices into plan[]
       PLAN_WIDE = 5,       // dynamic shared memory of the one-CTA-per-SM configuration if the shape enqueues it, else 0
       PLAN_NO_AVG = 7 };   // != 0: the pack was written without the average unit normal (one-shot pack of an exact-mode call)
constexpr int kOrderMaxBatch = 16384;     // beyond this the drain is negligible and instances are taken in index order
struct SolveConfig { int threads, ctas_per_sm, smem_bytes; };
constexpr int kNumSolveConfigs = 5;
constexpr int kWideConfig = 4;            // 256 threads x 1 CTA/SM
CAVE_HD SolveConfig solve_config(int i) {
    // 4 x 128 x 128 registers fills the register file; shared memory per CTA leaves room for the static part.  The wide
    // configuration gets what one CTA may have, the per-block maximum less the kernel's static shared memory: a property of
    // the device and of the compiled kernel, read at run time (solve_wide_smem_bytes, plan[PLAN_WIDE]), hence 0 here.
    const SolveConfig t[kNumSolveConfigs] = {{64, 8, 27520}, {128, 4, 56320}, {160, 3, 75776}, {256, 2, 112640}, {256, 1, 0}};
    return t[i];
}
// Whether a shape enqueues the wide configuration (the ABI's launch loop, the plan kernel's PLAN_WIDE word and, through that
// word, the device rule and cave_plan_choice all follow this one function).  m_max > d is the structured regime: a bound row
// per variable (the dense path's gate relies on the same test).  d > 2048: every shipped model up to TSP-50 (d = 1225) and
// VRP-20 fits its largest hot set into 256 x 2 and keeps exactly the launches it had; from TSP-80 (d = 3160) on the hot set
// of a Newton solve (the Hessian of ~d/50 variables and its factor) outgrows the 110 KiB of that configuration.
CAVE_HD bool wide_config_enabled(int64_t m_max, int64_t d) { return m_max > d && d > 2048; }
CAVE_HD size_t a16(size_t v) { return (v + 15) & ~(size_t)15; }
// Shared-memory footprint of one instance (bytes), mirroring the Arena requests of solver_core.cuh.
//   hot  : arrays that must be in shared memory for the fast layout
//   work : hot + the CSC and the pointer arrays + half of the CSR (which may spill to the global slot at little cost)
CAVE_HD void instance_footprint(int64_t d, int64_t ngen, int64_t nv, int64_t nnz_kept, bool i8, bool dense_path,
                                size_t th, size_t* hot, size_t* work) {
    const size_t D = (size_t)d, M = (size_t)ngen, V = (size_t)nv, Z = (size_t)nnz_kept;
    size_t h = a16(D * 4) + a16(D * 8);                             // c (I/O dtype, 4 assumed here) and r
    if (ngen == 0) { *hot = h; *work = h; return; }
    if (dense_path) {                                               // Lawson-Hanson: Gram + factor, three d-vectors
        const size_t k = (M < D ? M : D) + 1;
        size_t w = h + 2 * a16(D * 8) + 2 * a16(k * k * 8) + 8 * a16(k * 8) + a16(M * 5);
        *hot = h; *work = w; return;
    }
    h += 4 * a16((M + 1) * 8) + a16((2 * M + 6) * th) + 256 + 2 * a16((M + 2) * 4) + a16(M + 1) + 3 * a16(D + 1) + a16((D + 1) * 2) + 16;
    h += a16((V * (V + 1) / 2 + 1) * (i8 ? 4 : th)) + a16(((V + 2) * (V + 3) / 2 + 1) * th);
    size_t w = h + a16((M + 2) * 4) + a16((M + 1) * 4) + a16((D + 2) * 4) + a16((Z + 1) * 2) + a16((Z + 1) * (i8 ? 1 : 4));
    w += (a16((Z + 8) * 2) + a16((Z + 4) * (i8 ? 1 : 4))) / 2;        // half of the CSR: spilling it costs little, not nothing
    *hot = h; *work = w;
}
// Smallest configuration whose shared memory holds the average working set with 5 % to spare and the largest
// hot set outright; 256 x 2 otherwise, unless the largest hot set does not fit there but fits the wide configuration
// and the shape enqueued it (plan[PLAN_WIDE] != 0).  io_extra: bytes added when c is stored in float64.
CAVE_HD int choose_solve_config(const unsigned long long* plan, size_t th, size_t io_extra) {
    const unsigned long long n = plan[PLAN_N];
    if (n == 0) return kWideConfig - 1;
    const size_t avg = (size_t)((th == 8 ? plan[PLAN_SUM8] : plan[PLAN_SUM4]) / n) + io_extra;
    const size_t mx = (size_t)(th == 8 ? plan[PLAN_MAXHOT8] : plan[PLAN_MAXHOT4]) + io_extra;
    for (int i = 0; i < kWideConfig - 1; ++i) {
        const size_t cap = (size_t)solve_config(i).smem_bytes;
        if (avg * 20 <= cap * 19 && mx + 1024 <= cap) return i;
    }
    const size_t wide = (size_t)plan[PLAN_WIDE];
    if (wide != 0 && mx + 1024 > (size_t)solve_config(kWideConfig - 1).smem_bytes && mx + 1024 <= wide) return kWideConfig;
    return kWideConfig - 1;
}

// Solver scratch: [work counter + large-slot locks][loss64 B][rnorm64 B][status B][iters B][one small slot per CTA]
// [n_large worst-case slots].  A CTA spills into its own small slot (sized for the structured instances every shipped model
// produces); an instance whose working set cannot fit there takes one of the few worst-case slots under a device-side
// lock for the duration of its solve (the holders never wait for anybody, so the waiters always get served).
constexpr int kMaxLargeSlots = 48;
struct ScratchLayout {
    size_t counter, loss64, rnorm64, status, iters, slots, slot_bytes, large, large_bytes, total;
    int64_t n_slots, n_large;
};

// Newton path (upper bound over every Arena::get in nw_setup / newton_solve) for `rows` general rows with `nnz` non-zeros
CAVE_HD size_t newton_slot_bytes(int64_t d, int64_t rows, int64_t nnz, size_t T) {
    const size_t r = (size_t)rows + 2, dd = (size_t)d + 2;
    return 3 * dd * T + 4 * dd + 4 * dd + 4 * dd + 64 + r * (6 * T + 4 + 4 + 1 + 4 + 1 + 4 + 4 + 8 + 4)
           + (size_t)(nnz + 2) * 12 + (r * (r + 1) / 2 + (r + 2) * (r + 3) / 2 + 8) * T;
}
// Lawson-Hanson path: `rows` general rows, passive set of at most kcap = min(rows, d) columns
CAVE_HD size_t lh_slot_bytes(int64_t d, int64_t rows, size_t T, int64_t kcap = -1) {
    const size_t r = (size_t)rows + 2, dd = (size_t)d + 2;
    int64_t kk = rows < d ? rows : d;
    if (kcap >= 0 && kk > kcap) kk = kcap;
    const size_t k = (size_t)kk + 2;
    return 3 * dd * T + dd * T + k * (5 * T + 8) + r * 5 + 2 * k * k * T;
}
CAVE_HD size_t solver_slot_bytes(int64_t d, int64_t cap_rows, int64_t cap_nnz, size_t T) {
    const size_t nw = newton_slot_bytes(d, cap_rows, cap_nnz, T), lh = lh_slot_bytes(d, cap_rows, T);
    return align_up((nw > lh ? nw : lh) + 64 * 16 + 1024, 256);
}
// what ONE instance needs from its slot, by the path it will take (no singleton row: Lawson-Hanson, else Newton)
CAVE_HD size_t instance_slot_bytes(int64_t d, int64_t ngen, int64_t gen_nnz, bool lh_path, size_t T) {
    return align_up((lh_path ? lh_slot_bytes(d, ngen, T) : newton_slot_bytes(d, ngen, gen_nnz, T)) + 64 * 16 + 1024, 256);
}

CAVE_HD ScratchLayout make_scratch_layout(int64_t B, int64_t d, int64_t cap_rows, int64_t cap_nnz, size_t T,
                                          int64_t n_slots, int64_t n_large = 0, size_t large_bytes = 0, size_t small_bytes = 0) {
    ScratchLayout L;
    size_t o = 0;
    L.counter = o; o = align_up(o + 256, 256);          // int[0] work counter, int[8 .. 8 + n_large) slot locks
    L.loss64 = o;  o = align_up(o + (size_t)B * 8, 256);
    L.rnorm64 = o; o = align_up(o + (size_t)B * 8, 256);
    L.status = o;  o = align_up(o + (size_t)B * 4, 256);
    L.iters = o;   o = align_up(o + (size_t)B * 4, 256);
    L.slot_bytes = small_bytes ? small_bytes : solver_slot_bytes(d, cap_rows, cap_nnz, T);
    L.n_slots = n_slots;
    L.slots = o;   o += L.slot_bytes * (size_t)n_slots;
    L.n_large = n_large; L.large_bytes = large_bytes;
    L.large = o;   o += large_bytes * (size_t)n_large;
    L.total = o;
    return L;
}

}  // namespace cave
