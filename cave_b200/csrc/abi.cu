// extern "C" entry points declared in include/cave_b200.h.  Plain pointers and sizes only; no
// allocation, no synchronisation, no exceptions across the boundary.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <string>

#include "../../include/cave_b200.h"
#include "layout.cuh"
#include "scan_kernel.cuh"
#include "solve_kernel.cuh"
#include "dense.cuh"

namespace cave {       // tsp_dp.cu (auxiliary: exact TSP for regret evaluation)
size_t tsp_slot_floats(int n);
cudaError_t launch_tsp(const float* cost, int N, int n, int* tour, double* obj, void* scratch, int n_slots, cudaStream_t stream);
}

namespace {

thread_local std::string g_err;
std::atomic<unsigned long long> g_launches{0};      // kernels launched by this library in this process (cave_launch_count)

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

const int64_t kMaxD = 12288;        // shared-memory bound of the scan ring / u16 column ids
const int64_t kMaxM = 65535;        // u16 variable ids in the CSC
const int64_t kMaxB = 0x7fffffff;

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

int sm_count() {                    // of the CURRENT device (cached per device: a process may drive several GPUs)
    static int cached[64] = {0};
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64) {
        if (cached[dev] > 0) return cached[dev];
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
            cached[dev] = n;
            return n;
        }
    }
    (void)cudaGetLastError();
    return 148;                     // B200; used only for sizing when no device is visible
}

// dynamic shared memory of the wide solve configuration on the current device (cached per device, as sm_count)
cudaError_t wide_smem(int* out) {
    static int cached[64] = {0};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && cached[dev] > 0) { *out = cached[dev]; return cudaSuccess; }
    e = cave::solve_wide_smem_bytes(out);
    if (e == cudaSuccess && dev >= 0 && dev < 64) cached[dev] = *out;
    return e;
}

bool solve_forced() {     // experiments: a single launch with explicit thread / CTA / shared-memory settings
    return getenv("CAVE_SOLVE_THREADS") || getenv("CAVE_SOLVE_CTAS_PER_SM") || getenv("CAVE_SOLVE_SMEM");
}

// Scratch slots (one per resident CTA of the widest-grid configuration that may run), bounded so that the
// worst-case slots of a large shape do not take more than 16 GiB; the two-CTAs-per-SM grid is always served.
int64_t solver_slots(int64_t B, size_t slot_bytes) {
    const int64_t sms = sm_count();
    int64_t n = sms * (solve_forced() ? env_int("CAVE_SOLVE_CTAS_PER_SM", 2) : cave::solve_config(0).ctas_per_sm);
    const int64_t cap = (int64_t)(((size_t)16 << 30) / (slot_bytes ? slot_bytes : 1));
    if (!solve_forced() && n > cap) n = cap > 2 * sms ? cap : 2 * sms;
    return B < n ? B : n;
}

int check_shape(int64_t B, int64_t m_max, int64_t d) {
    if (B <= 0 || m_max <= 0 || d <= 0) return fail(CAVE_EINVAL, "B, m_max and d must be positive (got %lld, %lld, %lld)",
                                                    (long long)B, (long long)m_max, (long long)d);
    if (d > kMaxD) return fail(CAVE_ELIMIT, "d = %lld exceeds the supported maximum %lld", (long long)d, (long long)kMaxD);
    if (m_max > kMaxM) return fail(CAVE_ELIMIT, "m_max = %lld exceeds the supported maximum %lld", (long long)m_max, (long long)kMaxM);
    if (B > kMaxB) return fail(CAVE_ELIMIT, "B = %lld exceeds the supported maximum", (long long)B);
    return CAVE_OK;
}

// Caps of the per-CTA ("small") slot.  Explicit caps keep their old meaning (instances beyond them report CAVE_ST_NOSPACE, no
// worst-case slots).  By default the small slot is sized for structured instances (<= 192 general rows, non-zeros within the
// packed-CSR capacity) and a few worst-case slots serve everything else.
bool resolve_caps(const cave_solver_opts* o, int64_t m_max, int64_t d, int64_t* cap_rows, int64_t* cap_nnz) {
    const bool explicit_caps = o && (o->cap_rows > 0 || o->cap_nnz > 0);
    int64_t r = (o && o->cap_rows > 0) ? o->cap_rows : (explicit_caps ? m_max : (m_max < 192 ? m_max : 192));
    if (r > m_max) r = m_max;
    int64_t z = (o && o->cap_nnz > 0) ? o->cap_nnz : (explicit_caps ? r * d : cave::pack_cap_nnz(m_max, d));
    if (z > r * d) z = r * d;
    *cap_rows = r; *cap_nnz = z;
    return explicit_caps;
}

struct ScratchPlan { int64_t cr, cz, n_slots, n_large; size_t large_bytes, small_bytes; };
ScratchPlan plan_scratch(const cave_solver_opts* o, int64_t B, int64_t m_max, int64_t d);

ScratchPlan plan_scratch(const cave_solver_opts* o, int64_t B, int64_t m_max, int64_t d) {
    ScratchPlan P;
    const bool explicit_caps = resolve_caps(o, m_max, d, &P.cr, &P.cz);
    size_t small = cave::solver_slot_bytes(d, P.cr, P.cz, 8);
    if (!explicit_caps) {
        // Lawson-Hanson instances with many rows but a passive set of at most 192 columns (e.g. d = 190, m = 1024) stay in
        // the small slot as well
        const size_t lh_many_rows = cave::align_up(cave::lh_slot_bytes(d, m_max, 8, 192) + 64 * 16 + 1024, 256);
        if (lh_many_rows > small) small = lh_many_rows;
    }
    P.small_bytes = small;
    P.n_slots = solver_slots(B, small);
    P.n_large = 0; P.large_bytes = 0;
    if (!explicit_caps) {
        const size_t worst = cave::solver_slot_bytes(d, m_max, m_max * d, 8);
        if (worst > small) {
            // a 1 GiB scratch in total where that leaves at least 8 worst-case slots; never more than one per CTA of the 2/SM grid
            const size_t used = small * (size_t)P.n_slots;
            int64_t n = used < ((size_t)1 << 30) ? (int64_t)((((size_t)1 << 30) - used) / worst) : 0;
            if (n < 8) n = 8;
            if (n > cave::kMaxLargeSlots) n = cave::kMaxLargeSlots;
            if (n > B) n = B;
            P.n_large = n; P.large_bytes = worst;
        }
    }
    return P;
}

// ---- dense (tensor-core Gram) path: host-side gate and workspace sizing
bool dense_enabled(const cave_solver_opts* o, const float* A, int64_t m_max, int64_t d, int mode) {
    const int dm = o ? o->dense_mode : 0;
    if (dm < 0 || !A || mode == CAVE_MODE_HEURISTIC) return false;
    if (m_max < cave::kDenseMinRows || cave::dense_m_pad(m_max) > 2048) return false;
    return dm > 0 || m_max <= d;      // auto: structured models (one bound row per variable) always have m > d
}

int64_t dense_slots(const cave_solver_opts* o, int64_t B, int64_t m_max, int64_t d) {
    int64_t n;
    if (o && o->dense_slots > 0) n = o->dense_slots;
    else {
        const int64_t sms = sm_count();
        const int64_t by_budget = (int64_t)(((size_t)24 << 30) / cave::dense_slot_bytes(m_max, d));
        n = 8 * sms < by_budget ? 8 * sms : by_budget;       // more instances per round: a shorter relative tail in the solve kernel
        if (n < sms) n = sms;
    }
    return n < B ? n : B;
}

}  // namespace

extern "C" {

int cave_abi_version(void) { return CAVE_B200_ABI_VERSION; }

unsigned long long cave_launch_count(void) { return g_launches.load(); }

const char* cave_last_error(void) { return g_err.c_str(); }

int cave_get_limits(cave_limits* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    out->max_d = kMaxD; out->max_m = kMaxM; out->max_batch = kMaxB;
    return CAVE_OK;
}

int cave_pack_bytes(int64_t B, int64_t m_max, int64_t d, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (int e = check_shape(B, m_max, d)) return e;
    *out = cave::make_pack_layout(B, m_max, d).total;
    return CAVE_OK;
}

int cave_plan_offset(int64_t B, int64_t m_max, int64_t d, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (int e = check_shape(B, m_max, d)) return e;
    *out = cave::make_pack_layout(B, m_max, d).plan;
    return CAVE_OK;
}

int cave_dense_ctrl_offset(int64_t B, int64_t m_max, int64_t d, const cave_solver_opts* opts, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (int e = check_shape(B, m_max, d)) return e;
    const ScratchPlan SPn = plan_scratch(opts, B, m_max, d);
    const cave::ScratchLayout SL = cave::make_scratch_layout(B, d, SPn.cr, SPn.cz, 8, SPn.n_slots, SPn.n_large, SPn.large_bytes, SPn.small_bytes);
    *out = cave::make_dense_layout(B, m_max, d, dense_slots(opts, B, m_max, d), SL.total).ctrl;
    return CAVE_OK;
}

int cave_plan_choice(const uint64_t* plan_host, int64_t d, int io_dtype, int compute_dtype,
                     int* threads, int* ctas_per_sm, int* smem_bytes) {
    if (!plan_host) return fail(CAVE_EINVAL, "plan_host is null");
    unsigned long long pl[8];
    for (int i = 0; i < 8; ++i) pl[i] = plan_host[i];
    const int c = cave::choose_solve_config(pl, compute_dtype == CAVE_F32 ? 4 : 8, io_dtype == CAVE_F64 ? (size_t)d * 4 : 0);
    const cave::SolveConfig cfg = cave::solve_config(c);
    if (threads) *threads = cfg.threads;
    if (ctas_per_sm) *ctas_per_sm = cfg.ctas_per_sm;
    if (smem_bytes) *smem_bytes = c == cave::kWideConfig ? (int)pl[cave::PLAN_WIDE] : cfg.smem_bytes;
    return c;
}

int cave_scratch_bytes(int64_t B, int64_t m_max, int64_t d, int compute_dtype, const cave_solver_opts* opts, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (int e = check_shape(B, m_max, d)) return e;
    if (compute_dtype != CAVE_F32 && compute_dtype != CAVE_F64) return fail(CAVE_EINVAL, "bad compute_dtype %d", compute_dtype);
    const ScratchPlan SPn = plan_scratch(opts, B, m_max, d);
    size_t total = cave::make_scratch_layout(B, d, SPn.cr, SPn.cz, 8, SPn.n_slots, SPn.n_large, SPn.large_bytes, SPn.small_bytes).total;
    // mode and A are not known here: sized for the case that the call takes the dense path
    static const float kSomeA = 0.f;
    if (dense_enabled(opts, &kSomeA, m_max, d, CAVE_MODE_EXACT))
        total = cave::make_dense_layout(B, m_max, d, dense_slots(opts, B, m_max, d), total).total;
    *out = total;
    return CAVE_OK;
}

struct SparseIn { const long long* inst_off; const long long* row_ptr; const int* col; const float* val; };
static int pack_impl(const float* A, const int32_t* m_rows, int64_t B, int64_t m_max, int64_t d, void* pack, size_t pack_bytes,
                     void* stream, bool emit_setup, const SparseIn* sparse = nullptr, bool skip_avg = false) {
    if ((!A && !sparse) || !pack) return fail(CAVE_EINVAL, "A and pack must not be null");
    if (int e = check_shape(B, m_max, d)) return e;
    const cave::PackLayout L = cave::make_pack_layout(B, m_max, d);
    if (pack_bytes < L.total) return fail(CAVE_ENOSPC, "pack buffer has %zu bytes, %zu needed", pack_bytes, L.total);
    if (((uintptr_t)pack & 255) != 0) return fail(CAVE_EINVAL, "pack must be 256-byte aligned");
    char* base = (char*)pack;
    cave::ScanParams p;
    memset(&p, 0, sizeof(p));
    p.A = A; p.m_rows = m_rows; p.B = (int)B; p.m_max = (int)m_max; p.d = (int)d; p.dpad = L.dpad;
    p.nvalid = (int*)(base + L.nvalid); p.navg = (int*)(base + L.navg); p.ngen = (int*)(base + L.ngen);
    p.gennnz = (int*)(base + L.gennnz); p.nsingc = (int*)(base + L.nsingc);
    p.gen4 = (int4*)(base + L.gen); p.ctype = (unsigned char*)(base + L.ctype); p.avg = (float*)(base + L.avg);
    p.ghash = (ulonglong2*)(base + L.ghash); p.csr_col = (uint16_t*)(base + L.csr_col); p.csr_val = (float*)(base + L.csr_val);
    p.cap_nnz = (int)L.cap_nnz; p.csr_ok = (int*)(base + L.csrok); p.maxl1 = (float*)(base + L.maxl1); p.maxl2 = (float*)(base + L.maxl2);
    p.skip_avg = skip_avg ? 1 : 0;
    cudaError_t e = cudaMemsetAsync(base + L.plan, 0, 64, (cudaStream_t)stream);
    // marked in the pack: a later warm call in another mode reports CAVE_ST_BADINPUT instead of pushing towards a zero average
    if (e == cudaSuccess && skip_avg) e = cudaMemsetAsync(base + L.plan + 8 * cave::PLAN_NO_AVG, 1, 1, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(CAVE_ECUDA, "cudaMemsetAsync failed: %s", cudaGetErrorString(e));
    e = sparse ? cave::launch_scan_sparse(p, sparse->inst_off, sparse->row_ptr, sparse->col, sparse->val, (cudaStream_t)stream)
               : cave::launch_scan(p, (cudaStream_t)stream);
    g_launches += 1;
    if (e != cudaSuccess) return fail(CAVE_ECUDA, "scan kernel launch failed: %s", cudaGetErrorString(e));
    cave::PlanParams pp;
    memset(&pp, 0, sizeof(pp));
    pp.B = (int)B; pp.m_max = (int)m_max; pp.d = (int)d;
    pp.nvalid = p.nvalid; pp.ngen = p.ngen; pp.gennnz = p.gennnz; pp.nsingc = p.nsingc; pp.csr_ok = p.csr_ok;
    pp.gen4 = p.gen4; pp.ghash = p.ghash; pp.plan = (unsigned long long*)(base + L.plan);
    pp.okey = (int*)(base + L.okey); pp.order = (int*)(base + L.order);
    pp.csr_col = p.csr_col; pp.csr_val = p.csr_val; pp.cap_nnz = L.cap_nnz;
    // the cached solver setup pays off when the pack is reused (warm / dataset packs: cave_pack); a pack that lives for one
    // call (cold cave_forward_backward) keeps the in-solver setup: the setup kernel would cost what it saves
    pp.setup = emit_setup ? base + L.setup : nullptr; pp.setup_stride = L.setup_stride; pp.setup_cap_v = L.setup_cap_v;
    if (cave::wide_config_enabled(m_max, d)) {
        e = wide_smem(&pp.wide_smem);
        if (e != cudaSuccess) return fail(CAVE_ECUDA, "solve kernel attributes: %s", cudaGetErrorString(e));
    }
    if (!emit_setup) {
        // no cached setup in this pack: the valid word of every instance's setup block must say so (the pack buffer is the
        // caller's uninitialised memory, possibly a recycled pack)
        e = cave::launch_clear_setup(base + L.setup, (long long)L.setup_stride, (int)B, (cudaStream_t)stream);
        if (e != cudaSuccess) return fail(CAVE_ECUDA, "clear-setup kernel launch failed: %s", cudaGetErrorString(e));
    }
    e = cave::launch_plan(pp, (cudaStream_t)stream);
    g_launches += 3;      // plan, order, and the setup kernel or the kernel that clears the setup blocks' valid words
    if (e != cudaSuccess) return fail(CAVE_ECUDA, "plan kernel launch failed: %s", cudaGetErrorString(e));
    return CAVE_OK;
}

int cave_pack(const float* A, const int32_t* m_rows, int64_t B, int64_t m_max, int64_t d, void* pack, size_t pack_bytes,
              void* stream) {
    return pack_impl(A, m_rows, B, m_max, d, pack, pack_bytes, stream, true);
}

int cave_pack_ex(const float* A, const int32_t* m_rows, int64_t B, int64_t m_max, int64_t d, int32_t flags, void* pack,
                 size_t pack_bytes, void* stream) {
    return pack_impl(A, m_rows, B, m_max, d, pack, pack_bytes, stream, (flags & 1) != 0);
}

int cave_pack_sparse(const int64_t* inst_off, const int64_t* row_ptr, const int32_t* col, const float* val, int64_t B,
                     int64_t m_max, int64_t d, int32_t flags, void* pack, size_t pack_bytes, void* stream) {
    if (!inst_off || !row_ptr || !col || !val) return fail(CAVE_EINVAL, "inst_off, row_ptr, col and val must not be null");
    SparseIn in;
    in.inst_off = (const long long*)inst_off; in.row_ptr = (const long long*)row_ptr; in.col = col; in.val = val;
    return pack_impl(nullptr, nullptr, B, m_max, d, pack, pack_bytes, stream, (flags & 1) != 0, &in);
}

int cave_warm_bytes(int64_t n_instances, int64_t m_max, int64_t d, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (int e = check_shape(n_instances, m_max, d)) return e;
    *out = (size_t)n_instances * cave::warm_slot_bytes(m_max);
    return CAVE_OK;
}

int cave_dense_warm_bytes(int64_t n_instances, int64_t m_max, int64_t d, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (int e = check_shape(n_instances, m_max, d)) return e;
    *out = (size_t)n_instances * cave::dense_warm_slot_bytes(m_max);
    return CAVE_OK;
}

// cave_forward_backward and its warm-start variants: warm / warm_dense are null for the former, checked buffers (either
// may be null) for the latter
static int forward_backward_impl(const float* A, const int32_t* m_rows, const void* pred, int64_t B, int64_t m_max, int64_t d,
                                 double sign, int mode, double inner_ratio, int reduction, int io_dtype, int compute_dtype,
                                 const cave_solver_opts* opts, void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                                 int32_t* status, int32_t* iters, void* pack, size_t pack_bytes, void* scratch,
                                 size_t scratch_bytes, void* warm, size_t warm_bytes, void* warm_dense,
                                 size_t warm_dense_bytes, const void* gram, size_t gram_bytes, void* stream) {
    const bool indexed = opts && opts->inst_index;
    if ((!A && !indexed) || !pred || !loss_i || !grad || !pack || !scratch) return fail(CAVE_EINVAL, "A, pred, loss_i, grad, pack, scratch must not be null");
    if (indexed && !opts->warm_pack) return fail(CAVE_EINVAL, "inst_index needs warm_pack (a pack built over the whole dataset)");
    if (indexed && opts->n_packed <= 0) return fail(CAVE_EINVAL, "n_packed must be positive with inst_index");
    if (int e = check_shape(B, m_max, d)) return e;
    if (mode < CAVE_MODE_EXACT || mode > CAVE_MODE_HEURISTIC) return fail(CAVE_EINVAL, "bad mode %d", mode);
    if (reduction < CAVE_REDUCE_MEAN || reduction > CAVE_REDUCE_NONE) return fail(CAVE_EINVAL, "bad reduction %d", reduction);
    if ((io_dtype != CAVE_F32 && io_dtype != CAVE_F64) || (compute_dtype != CAVE_F32 && compute_dtype != CAVE_F64))
        return fail(CAVE_EINVAL, "bad dtype (io %d, compute %d)", io_dtype, compute_dtype);
    if (!(sign == 1.0 || sign == -1.0)) return fail(CAVE_EINVAL, "sign must be +1 or -1");
    if (!(inner_ratio >= 0.0 && inner_ratio <= 1.0)) return fail(CAVE_EINVAL, "inner_ratio must be in [0, 1]");
    if (reduction != CAVE_REDUCE_NONE && !loss) return fail(CAVE_EINVAL, "loss must not be null for mean/sum");
    if (((uintptr_t)scratch & 255) != 0 || ((uintptr_t)pack & 255) != 0) return fail(CAVE_EINVAL, "pack and scratch must be 256-byte aligned");

    const int64_t Bpack = indexed ? opts->n_packed : B;
    if (int e = check_shape(Bpack, m_max, d)) return e;
    const cave::PackLayout PL = cave::make_pack_layout(Bpack, m_max, d);
    if (pack_bytes < PL.total) return fail(CAVE_ENOSPC, "pack buffer has %zu bytes, %zu needed", pack_bytes, PL.total);
    const ScratchPlan SPn = plan_scratch(opts, B, m_max, d);
    const size_t T = 8;   // state vectors are double in both modes; sized for the f64 factor
    const int64_t n_slots = SPn.n_slots;
    const cave::ScratchLayout SL = cave::make_scratch_layout(B, d, SPn.cr, SPn.cz, T, n_slots, SPn.n_large, SPn.large_bytes, SPn.small_bytes);
    const bool dense = dense_enabled(opts, A, m_max, d, mode);
    cave::DenseLayout DL;
    memset(&DL, 0, sizeof(DL));
    if (dense) DL = cave::make_dense_layout(B, m_max, d, dense_slots(opts, B, m_max, d), SL.total);
    const size_t need = dense ? DL.total : SL.total;
    if (scratch_bytes < need) return fail(CAVE_ENOSPC, "scratch buffer has %zu bytes, %zu needed", scratch_bytes, need);
    if (warm) {
        const size_t wneed = (size_t)Bpack * cave::warm_slot_bytes(m_max);
        if (warm_bytes < wneed) return fail(CAVE_ENOSPC, "warm-start buffer has %zu bytes, %zu needed (cave_warm_bytes of %lld instances)",
                                            warm_bytes, wneed, (long long)Bpack);
        if (((uintptr_t)warm & 15) != 0) return fail(CAVE_EINVAL, "warm-start buffer must be 16-byte aligned");
    }
    if (warm_dense) {
        const size_t wneed = (size_t)Bpack * cave::dense_warm_slot_bytes(m_max);
        if (warm_dense_bytes < wneed)
            return fail(CAVE_ENOSPC, "dense warm-start buffer has %zu bytes, %zu needed (cave_dense_warm_bytes of %lld instances)",
                        warm_dense_bytes, wneed, (long long)Bpack);
        if (((uintptr_t)warm_dense & 15) != 0) return fail(CAVE_EINVAL, "dense warm-start buffer must be 16-byte aligned");
    }
    if (gram) {
        if (!A) return fail(CAVE_EINVAL, "a Gram cache needs A (the dense path reads the rows of A)");
        if (((uintptr_t)gram & 15) != 0) return fail(CAVE_EINVAL, "Gram cache must be 16-byte aligned");
        const size_t gneed = cave::gram_cache_bytes(Bpack, 0, m_max);
        if (gram_bytes < gneed)
            return fail(CAVE_ENOSPC, "Gram cache has %zu bytes, at least %zu needed (cave_gram_cache_bytes of %lld instances)",
                        gram_bytes, gneed, (long long)Bpack);
    }

    cudaStream_t st = (cudaStream_t)stream;
    if (!(opts && opts->warm_pack)) {
        // one-shot pack: the exact loss never reads the average of the normalised rows
        if (int e = pack_impl(A, m_rows, B, m_max, d, pack, pack_bytes, stream, env_int("CAVE_COLD_SETUP", 0) != 0, nullptr,
                              mode == CAVE_MODE_EXACT)) return e;
    }
    char* pb = (char*)pack;
    char* sb = (char*)scratch;
    cudaError_t ce = cudaMemsetAsync(sb + SL.counter, 0, 256, st);
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "cudaMemsetAsync failed: %s", cudaGetErrorString(ce));

    cave::SolveParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.A = A; sp.pred = pred; sp.grad = grad; sp.proj = proj;
    sp.B = (int)B; sp.m_max = (int)m_max; sp.d = (int)d; sp.dpad = PL.dpad;
    sp.nvalid = (const int*)(pb + PL.nvalid); sp.ngen = (const int*)(pb + PL.ngen);
    sp.gennnz = (const int*)(pb + PL.gennnz); sp.nsingc = (const int*)(pb + PL.nsingc);
    sp.gen = (const int4*)(pb + PL.gen); sp.ctype = (const unsigned char*)(pb + PL.ctype); sp.avg = (const float*)(pb + PL.avg);
    sp.csr_ok = (const int*)(pb + PL.csrok); sp.maxl1 = (const float*)(pb + PL.maxl1); sp.maxl2 = (const float*)(pb + PL.maxl2);
    sp.ghash = (const ulonglong2*)(pb + PL.ghash); sp.csr_col = (const uint16_t*)(pb + PL.csr_col);
    sp.csr_val = (const float*)(pb + PL.csr_val); sp.cap_nnz = PL.cap_nnz;
    sp.counter = (int*)(sb + SL.counter); sp.loss64 = (double*)(sb + SL.loss64); sp.rnorm64 = (double*)(sb + SL.rnorm64);
    sp.status = (int*)(sb + SL.status); sp.iters = (int*)(sb + SL.iters);
    sp.slots = sb + SL.slots; sp.slot_bytes = SL.slot_bytes;
    sp.large = sb + SL.large; sp.large_bytes = SL.large_bytes; sp.n_large = (int)SL.n_large;
    sp.mode = mode; sp.inner_ratio = inner_ratio; sp.sign = sign;
    sp.gscale = reduction == CAVE_REDUCE_MEAN ? 1.0 / (double)B : 1.0;
    sp.max_iter = opts ? opts->max_iter : 0; sp.max_ls = opts ? opts->max_linesearch : 0; sp.tol = opts ? opts->tol : 0.0;
    sp.inst_index = indexed ? opts->inst_index : nullptr;
    sp.plan = (const unsigned long long*)(pb + PL.plan);
    sp.order = (indexed || env_int("CAVE_SOLVE_ORDER", 1) == 0) ? nullptr : (const int*)(pb + PL.order);       // the order of a dataset-wide pack does not apply to a batch
    sp.n_packed = Bpack;
    sp.setup = (((opts && opts->warm_pack) || env_int("CAVE_COLD_SETUP", 0)) && env_int("CAVE_SETUP_CACHE", 1)) ? pb + PL.setup : nullptr;
    sp.setup_stride = PL.setup_stride;
    sp.warm = (char*)warm; sp.warm_stride = (long long)cave::warm_slot_bytes(m_max); sp.warm_cap = (int)cave::warm_cap_v(m_max);
    sp.dense_flag = nullptr;
    if (dense) {
        // Dense regime first: instance list, then per round of n_slots instances the TF32 split, the tensor-core Gram and
        // the Gram-space solve.  Everything is decided on the device; a batch without dense instances costs the list
        // kernel and 3 x rounds launches that return at once.  Instances the Gram-space solver hands back are taken by
        // the general solve kernel below (Lawson-Hanson).
        cave::DenseParams dp;
        memset(&dp, 0, sizeof(dp));
        dp.A = A; dp.pred = pred; dp.B = (int)B; dp.m_max = (int)m_max; dp.d = (int)d;
        dp.inst_index = sp.inst_index; dp.n_packed = Bpack; dp.nvalid = sp.nvalid; dp.ngen = sp.ngen; dp.nsingc = sp.nsingc; dp.gen = sp.gen;
        dp.ctype = sp.ctype; dp.avg = sp.avg; dp.dpad = PL.dpad;
        dp.plan = (const unsigned long long*)(pb + PL.plan); dp.ws = sb; dp.L = DL; dp.force = (opts && opts->dense_mode > 0) ? 1 : 0; dp.no_handback = env_int("CAVE_DENSE_NO_HANDBACK", 0); dp.trace_b = env_int("CAVE_DENSE_TRACE", -1);
        dp.grad = grad; dp.proj = proj; dp.loss64 = sp.loss64; dp.rnorm64 = sp.rnorm64; dp.status = sp.status; dp.iters = sp.iters;
        dp.mode = mode; dp.inner_ratio = inner_ratio; dp.sign = sign; dp.gscale = sp.gscale;
        dp.max_iter = 0; dp.max_ls = sp.max_ls; dp.tol = sp.tol; dp.io_f32 = io_dtype == CAVE_F32; dp.nk = (int)(DL.d_pad / 32);
        dp.warm = (char*)warm_dense; dp.warm_stride = (long long)cave::dense_warm_slot_bytes(m_max); dp.warm_cap = (int)cave::dense_warm_cap(m_max);
        // with the pack's Gram cache the prep kernel writes no TF32 planes and the Gram kernel is not launched
        dp.gram = (const char*)gram; dp.gram_bytes = gram_bytes;
        ce = cave::launch_dense_list(dp, st);
        g_launches += 1;
        if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense list kernel launch failed: %s", cudaGetErrorString(ce));
        const int64_t rounds = (B + DL.n_slots - 1) / DL.n_slots;
        for (int64_t r = 0; r < rounds; ++r) {
            dp.round = (int)r;
            ce = cave::launch_dense_prep(dp, st);
            if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense prep kernel launch failed: %s", cudaGetErrorString(ce));
            if (!gram) {
                ce = cave::launch_dense_gram(dp, st);
                if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense Gram kernel launch failed: %s (%s)", cudaGetErrorString(ce), cave::dense_last_error());
            }
            ce = cave::launch_dense_solve(dp, st);
            g_launches += gram ? 2 : 3;
            if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense solve kernel launch failed: %s", cudaGetErrorString(ce));
        }
        sp.dense_flag = (const int*)(sb + DL.flag);
    }
    if (solve_forced()) {
        sp.smem_bytes = env_int("CAVE_SOLVE_SMEM", 110 * 1024);
        int threads = env_int("CAVE_SOLVE_THREADS", 256);
        if (threads < 32 || threads > 256 || threads % 32) threads = 256;
        sp.cfg_id = -1;
        ce = cave::launch_solve(sp, compute_dtype == CAVE_F32, io_dtype == CAVE_F32, (int)n_slots, threads, st);
        g_launches += 1;
        if (ce != cudaSuccess) return fail(CAVE_ECUDA, "solve kernel launch failed: %s", cudaGetErrorString(ce));
    } else {
        // every candidate configuration is enqueued; the pack's plan statistics select exactly one on the device
        // and the others return immediately (no host round trip, a few microseconds of launch overhead).  The wide
        // configuration is a candidate for the shapes wide_config_enabled admits (the plan kernel recorded the same test).
        const int only = env_int("CAVE_SOLVE_CFG", -1);
        const bool forced = only >= 0 && only < cave::kNumSolveConfigs;
        for (int i = 0; i < cave::kNumSolveConfigs; ++i) {
            const cave::SolveConfig cfg = cave::solve_config(i);
            if (forced && i != only) continue;
            if (i == cave::kWideConfig && !forced && !cave::wide_config_enabled(m_max, d)) continue;
            int64_t grid = (int64_t)sm_count() * cfg.ctas_per_sm;
            if (grid > n_slots) grid = n_slots;
            sp.smem_bytes = cfg.smem_bytes;
            if (i == cave::kWideConfig) {
                ce = wide_smem(&sp.smem_bytes);
                if (ce != cudaSuccess) return fail(CAVE_ECUDA, "solve kernel attributes: %s", cudaGetErrorString(ce));
            }
            sp.cfg_id = forced ? -1 : i;
            ce = cave::launch_solve(sp, compute_dtype == CAVE_F32, io_dtype == CAVE_F32, (int)grid, cfg.threads, st);
            g_launches += 1;
            if (ce != cudaSuccess) return fail(CAVE_ECUDA, "solve kernel launch failed: %s", cudaGetErrorString(ce));
        }
    }

    cave::FinalizeParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.B = (int)B; fp.reduction = reduction; fp.loss64 = sp.loss64; fp.rnorm64 = sp.rnorm64; fp.status = sp.status; fp.iters = sp.iters;
    fp.loss = loss; fp.loss_i = loss_i; fp.rnorm = rnorm; fp.status_out = status; fp.iters_out = iters;
    ce = cave::launch_finalize(fp, io_dtype == CAVE_F32, st);
    g_launches += 1;
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "finalize kernel launch failed: %s", cudaGetErrorString(ce));
    return CAVE_OK;
}

int cave_forward_backward(const float* A, const int32_t* m_rows, const void* pred, int64_t B, int64_t m_max, int64_t d,
                          double sign, int mode, double inner_ratio, int reduction, int io_dtype, int compute_dtype,
                          const cave_solver_opts* opts, void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                          int32_t* status, int32_t* iters, void* pack, size_t pack_bytes, void* scratch,
                          size_t scratch_bytes, void* stream) {
    return forward_backward_impl(A, m_rows, pred, B, m_max, d, sign, mode, inner_ratio, reduction, io_dtype, compute_dtype, opts,
                                 loss, loss_i, grad, proj, rnorm, status, iters, pack, pack_bytes, scratch, scratch_bytes,
                                 nullptr, 0, nullptr, 0, nullptr, 0, stream);
}

int cave_forward_backward_warm(const float* A, const int32_t* m_rows, const void* pred, int64_t B, int64_t m_max, int64_t d,
                               double sign, int mode, double inner_ratio, int reduction, int io_dtype, int compute_dtype,
                               const cave_solver_opts* opts, void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                               int32_t* status, int32_t* iters, void* pack, size_t pack_bytes, void* scratch,
                               size_t scratch_bytes, void* warm, size_t warm_bytes, void* stream) {
    if (!warm) return fail(CAVE_EINVAL, "warm must not be null (use cave_forward_backward for a call without warm-start state)");
    if (!(opts && opts->warm_pack))
        return fail(CAVE_EINVAL, "warm-start state needs opts->warm_pack = 1: it belongs to a pack built beforehand by cave_pack()");
    return forward_backward_impl(A, m_rows, pred, B, m_max, d, sign, mode, inner_ratio, reduction, io_dtype, compute_dtype, opts,
                                 loss, loss_i, grad, proj, rnorm, status, iters, pack, pack_bytes, scratch, scratch_bytes,
                                 warm, warm_bytes, nullptr, 0, nullptr, 0, stream);
}

int cave_forward_backward_warm_ex(const float* A, const int32_t* m_rows, const void* pred, int64_t B, int64_t m_max, int64_t d,
                                  double sign, int mode, double inner_ratio, int reduction, int io_dtype, int compute_dtype,
                                  const cave_solver_opts* opts, void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                                  int32_t* status, int32_t* iters, void* pack, size_t pack_bytes, void* scratch,
                                  size_t scratch_bytes, void* warm, size_t warm_bytes, void* warm_dense, size_t warm_dense_bytes,
                                  void* stream) {
    if (!warm && !warm_dense)
        return fail(CAVE_EINVAL, "warm and warm_dense must not both be null (use cave_forward_backward for a call without warm-start state)");
    if (!(opts && opts->warm_pack))
        return fail(CAVE_EINVAL, "warm-start state needs opts->warm_pack = 1: it belongs to a pack built beforehand by cave_pack()");
    return forward_backward_impl(A, m_rows, pred, B, m_max, d, sign, mode, inner_ratio, reduction, io_dtype, compute_dtype, opts,
                                 loss, loss_i, grad, proj, rnorm, status, iters, pack, pack_bytes, scratch, scratch_bytes,
                                 warm, warm_bytes, warm_dense, warm_dense_bytes, nullptr, 0, stream);
}

int cave_forward_backward_resident(const float* A, const int32_t* m_rows, const void* pred, int64_t B, int64_t m_max, int64_t d,
                                   double sign, int mode, double inner_ratio, int reduction, int io_dtype, int compute_dtype,
                                   const cave_solver_opts* opts, void* loss, void* loss_i, void* grad, void* proj, void* rnorm,
                                   int32_t* status, int32_t* iters, void* pack, size_t pack_bytes, void* scratch,
                                   size_t scratch_bytes, void* warm, size_t warm_bytes, void* warm_dense, size_t warm_dense_bytes,
                                   const void* gram, size_t gram_bytes, void* stream) {
    if (!warm && !warm_dense && !gram)
        return fail(CAVE_EINVAL, "warm, warm_dense and gram must not all be null (use cave_forward_backward for a call without them)");
    if (!(opts && opts->warm_pack))
        return fail(CAVE_EINVAL, "warm-start state and Gram cache need opts->warm_pack = 1: they belong to a pack built beforehand by cave_pack()");
    return forward_backward_impl(A, m_rows, pred, B, m_max, d, sign, mode, inner_ratio, reduction, io_dtype, compute_dtype, opts,
                                 loss, loss_i, grad, proj, rnorm, status, iters, pack, pack_bytes, scratch, scratch_bytes,
                                 warm, warm_bytes, warm_dense, warm_dense_bytes, gram, gram_bytes, stream);
}

int cave_gram_cache_bytes(int64_t N, int64_t n_cached, int64_t m_max, int64_t d, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (int e = check_shape(N, m_max, d)) return e;
    if (n_cached < 0 || n_cached > N) return fail(CAVE_EINVAL, "n_cached = %lld must be in [0, N = %lld]", (long long)n_cached, (long long)N);
    *out = cave::gram_cache_bytes(N, n_cached, m_max);
    return CAVE_OK;
}

int cave_gram_cache_count(const void* pack, size_t pack_bytes, int64_t N, int64_t m_max, int64_t d, int32_t* n_cached_dev,
                          void* stream) {
    if (!pack || !n_cached_dev) return fail(CAVE_EINVAL, "pack and n_cached_dev must not be null");
    if (int e = check_shape(N, m_max, d)) return e;
    const cave::PackLayout PL = cave::make_pack_layout(N, m_max, d);
    if (pack_bytes < PL.total) return fail(CAVE_ENOSPC, "pack buffer has %zu bytes, %zu needed", pack_bytes, PL.total);
    if (((uintptr_t)pack & 255) != 0) return fail(CAVE_EINVAL, "pack must be 256-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t ce;
    static const float kSomeA = 0.f;
    cave_solver_opts o;
    memset(&o, 0, sizeof(o));
    o.dense_mode = 1;
    if (!dense_enabled(&o, &kSomeA, m_max, d, CAVE_MODE_EXACT)) {
        ce = cudaMemsetAsync(n_cached_dev, 0, 4, st);       // a shape the dense path never takes: nothing to cache
    } else {
        const char* pb = (const char*)pack;
        ce = cave::launch_gram_cache_map((const int*)(pb + PL.nvalid), (const int*)(pb + PL.ngen), (const int*)(pb + PL.nsingc),
                                         (int)N, (int)cave::dense_m_pad(m_max), nullptr, n_cached_dev, nullptr, st);
        g_launches += 1;
    }
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "Gram cache count failed: %s", cudaGetErrorString(ce));
    return CAVE_OK;
}

int cave_gram_cache_build(const float* A, int64_t N, int64_t m_max, int64_t d, const cave_solver_opts* opts, void* cache,
                          size_t cache_bytes, const void* pack, size_t pack_bytes, void* scratch, size_t scratch_bytes,
                          void* stream) {
    if (!A || !cache || !pack || !scratch) return fail(CAVE_EINVAL, "A, cache, pack, scratch must not be null");
    if (int e = check_shape(N, m_max, d)) return e;
    cave_solver_opts o;
    memset(&o, 0, sizeof(o));
    if (opts) o = *opts;
    o.dense_mode = 1; o.inst_index = nullptr; o.n_packed = 0;
    if (!dense_enabled(&o, A, m_max, d, CAVE_MODE_EXACT)) return fail(CAVE_ELIMIT, "shape outside the dense path (128 <= m_max <= 2048)");
    if (((uintptr_t)scratch & 255) != 0 || ((uintptr_t)pack & 255) != 0) return fail(CAVE_EINVAL, "pack and scratch must be 256-byte aligned");
    if (((uintptr_t)cache & 15) != 0) return fail(CAVE_EINVAL, "Gram cache must be 16-byte aligned");
    const size_t cneed = cave::gram_cache_bytes(N, 0, m_max);
    if (cache_bytes < cneed)
        return fail(CAVE_ENOSPC, "Gram cache has %zu bytes, at least %zu needed (cave_gram_cache_bytes of %lld instances)",
                    cache_bytes, cneed, (long long)N);
    const cave::PackLayout PL = cave::make_pack_layout(N, m_max, d);
    if (pack_bytes < PL.total) return fail(CAVE_ENOSPC, "pack buffer has %zu bytes, %zu needed", pack_bytes, PL.total);
    const ScratchPlan SPn = plan_scratch(&o, N, m_max, d);
    const cave::ScratchLayout SL = cave::make_scratch_layout(N, d, SPn.cr, SPn.cz, 8, SPn.n_slots, SPn.n_large, SPn.large_bytes, SPn.small_bytes);
    const cave::DenseLayout DL = cave::make_dense_layout(N, m_max, d, dense_slots(&o, N, m_max, d), SL.total);
    if (scratch_bytes < DL.total) return fail(CAVE_ENOSPC, "scratch buffer has %zu bytes, %zu needed", scratch_bytes, DL.total);
    const char* pb = (const char*)pack;
    char* cb = (char*)cache;
    cudaStream_t st = (cudaStream_t)stream;
    // slots the buffer holds: a buffer sized for fewer instances than the pack has stays invalid (header valid = 0)
    const long long cap = (long long)((cache_bytes - cave::gram_cache_base(N)) / ((size_t)DL.m_pad * DL.m_pad * 4));
    cave::DenseParams dp;
    memset(&dp, 0, sizeof(dp));
    dp.A = A; dp.B = (int)N; dp.m_max = (int)m_max; dp.d = (int)d; dp.n_packed = N;
    dp.nvalid = (const int*)(pb + PL.nvalid); dp.ngen = (const int*)(pb + PL.ngen); dp.nsingc = (const int*)(pb + PL.nsingc);
    dp.gen = (const int4*)(pb + PL.gen); dp.ctype = (const unsigned char*)(pb + PL.ctype); dp.avg = (const float*)(pb + PL.avg);
    dp.dpad = PL.dpad; dp.ws = (char*)scratch; dp.L = DL; dp.force = 1; dp.trace_b = -1; dp.sign = 0.0; dp.io_f32 = 1; dp.nk = (int)(DL.d_pad / 32);
    dp.pred = A;       // prep also forms b = A c: any finite data will do (as in cave_dense_gram)
    cudaError_t ce = cave::launch_gram_cache_map(dp.nvalid, dp.ngen, dp.nsingc, (int)N, (int)DL.m_pad, (int*)(cb + 16), nullptr,
                                                 (int*)cb, st);
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "Gram cache map kernel launch failed: %s", cudaGetErrorString(ce));
    ce = cave::launch_dense_list(dp, st);
    g_launches += 2;
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense list kernel launch failed: %s", cudaGetErrorString(ce));
    // the same list -> prep -> Gram sequence as a call (dense_mode = 1, every pack instance), round by round
    const int64_t rounds = (N + DL.n_slots - 1) / DL.n_slots;
    for (int64_t r = 0; r < rounds; ++r) {
        dp.round = (int)r;
        ce = cave::launch_dense_prep(dp, st);
        if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense prep kernel launch failed: %s", cudaGetErrorString(ce));
        ce = cave::launch_dense_gram(dp, st);
        if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense Gram kernel launch failed: %s (%s)", cudaGetErrorString(ce), cave::dense_last_error());
        ce = cave::launch_gram_cache_copy(dp, cb, cap, st);
        g_launches += 3;
        if (ce != cudaSuccess) return fail(CAVE_ECUDA, "Gram cache copy kernel launch failed: %s", cudaGetErrorString(ce));
    }
    ce = cave::launch_gram_cache_seal(cb, cap, st);
    g_launches += 1;
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "Gram cache seal kernel launch failed: %s", cudaGetErrorString(ce));
    return CAVE_OK;
}

int cave_tsp_scratch_bytes(int64_t N, int32_t n_nodes, size_t* out) {
    if (!out) return fail(CAVE_EINVAL, "out is null");
    if (N <= 0 || n_nodes < 3 || n_nodes > 20) return fail(CAVE_ELIMIT, "Held-Karp needs 3 <= n_nodes <= 20 and N > 0");
    const int64_t slots = N < sm_count() ? N : sm_count();
    *out = (size_t)slots * cave::tsp_slot_floats(n_nodes) * 4;
    return CAVE_OK;
}

int cave_tsp_solve(const float* cost, int64_t N, int32_t n_nodes, int32_t* tour, double* obj, void* scratch, size_t scratch_bytes,
                   void* stream) {
    if (!cost || !tour || !obj || !scratch) return fail(CAVE_EINVAL, "cost, tour, obj and scratch must not be null");
    size_t need = 0;
    if (int e = cave_tsp_scratch_bytes(N, n_nodes, &need)) return e;
    if (scratch_bytes < need) return fail(CAVE_ENOSPC, "scratch buffer has %zu bytes, %zu needed", scratch_bytes, need);
    const int64_t slots = N < sm_count() ? N : sm_count();
    cudaError_t ce = cave::launch_tsp(cost, (int)N, n_nodes, tour, obj, scratch, (int)slots, (cudaStream_t)stream);
    g_launches += 1;
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "Held-Karp kernel launch failed: %s", cudaGetErrorString(ce));
    return CAVE_OK;
}

int cave_dense_gram(const float* A, int64_t B, int64_t m_max, int64_t d, const cave_solver_opts* opts, float* G_out,
                    int32_t* n_dense_out, void* pack, size_t pack_bytes, void* scratch, size_t scratch_bytes, void* stream) {
    if (!A || !G_out || !pack || !scratch) return fail(CAVE_EINVAL, "A, G_out, pack, scratch must not be null");
    if (int e = check_shape(B, m_max, d)) return e;
    cave_solver_opts o;
    memset(&o, 0, sizeof(o));
    if (opts) o = *opts;
    o.dense_mode = 1;
    if (!dense_enabled(&o, A, m_max, d, CAVE_MODE_EXACT)) return fail(CAVE_ELIMIT, "shape outside the dense path (128 <= m_max <= 2048)");
    if (((uintptr_t)scratch & 255) != 0 || ((uintptr_t)pack & 255) != 0) return fail(CAVE_EINVAL, "pack and scratch must be 256-byte aligned");
    if (!o.warm_pack) { if (int e = cave_pack(A, nullptr, B, m_max, d, pack, pack_bytes, stream)) return e; }
    const cave::PackLayout PL = cave::make_pack_layout(B, m_max, d);
    if (pack_bytes < PL.total) return fail(CAVE_ENOSPC, "pack buffer has %zu bytes, %zu needed", pack_bytes, PL.total);
    const ScratchPlan SPn = plan_scratch(&o, B, m_max, d);
    const cave::ScratchLayout SL = cave::make_scratch_layout(B, d, SPn.cr, SPn.cz, 8, SPn.n_slots, SPn.n_large, SPn.large_bytes, SPn.small_bytes);
    const cave::DenseLayout DL = cave::make_dense_layout(B, m_max, d, dense_slots(&o, B, m_max, d), SL.total);
    if (scratch_bytes < DL.total) return fail(CAVE_ENOSPC, "scratch buffer has %zu bytes, %zu needed", scratch_bytes, DL.total);
    char* pb = (char*)pack;
    char* sb = (char*)scratch;
    cudaStream_t st = (cudaStream_t)stream;
    cave::DenseParams dp;
    memset(&dp, 0, sizeof(dp));
    static const float kZero = 0.f;
    dp.A = A; dp.pred = &kZero; dp.B = (int)B; dp.m_max = (int)m_max; dp.d = (int)d; dp.n_packed = B;
    dp.nvalid = (const int*)(pb + PL.nvalid); dp.ngen = (const int*)(pb + PL.ngen); dp.nsingc = (const int*)(pb + PL.nsingc);
    dp.gen = (const int4*)(pb + PL.gen); dp.ctype = (const unsigned char*)(pb + PL.ctype); dp.avg = (const float*)(pb + PL.avg);
    dp.dpad = PL.dpad; dp.ws = sb; dp.L = DL; dp.force = 1; dp.trace_b = -1; dp.sign = 0.0; dp.io_f32 = 1; dp.nk = (int)(DL.d_pad / 32);
    // prep reads pred[b * d + k] for the right-hand side b = A c: point it at A's first rows (any finite data will do)
    dp.pred = A;
    cudaError_t ce = cave::launch_dense_list(dp, st);
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense list kernel launch failed: %s", cudaGetErrorString(ce));
    dp.round = 0;
    ce = cave::launch_dense_prep(dp, st);
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense prep kernel launch failed: %s", cudaGetErrorString(ce));
    ce = cave::launch_dense_gram(dp, st);
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "dense Gram kernel launch failed: %s (%s)", cudaGetErrorString(ce), cave::dense_last_error());
    const int64_t n = DL.n_slots < B ? DL.n_slots : B;
    ce = cudaMemcpyAsync(G_out, sb + DL.G, (size_t)n * DL.m_pad * DL.m_pad * 4, cudaMemcpyDeviceToDevice, st);
    if (ce != cudaSuccess) return fail(CAVE_ECUDA, "copy of G failed: %s", cudaGetErrorString(ce));
    if (n_dense_out) {
        ce = cudaMemcpyAsync(n_dense_out, sb + DL.ctrl, 4, cudaMemcpyDeviceToDevice, st);
        if (ce != cudaSuccess) return fail(CAVE_ECUDA, "copy of the dense count failed: %s", cudaGetErrorString(ce));
    }
    return CAVE_OK;
}

}  // extern "C"
