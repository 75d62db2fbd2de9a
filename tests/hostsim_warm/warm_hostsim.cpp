// CPU build of the solver core with the warm-start state (CAVE_HOST_SIM: one thread, warp width 1).  TEST
// INFRASTRUCTURE ONLY: built by tests/hostsim_warm/warm_sim.py, loaded by tests/test_warm_start_host.py, never by
// cave_b200/.  The pack restatement (host_pack) comes from tests/hostsim/hostsim.cpp; the instance loop below adds what
// the WARM variant of the solve kernel (solve_kernel_impl.cuh) adds to it: the slot of each instance and the cold
// re-solve after a failed warm start.
#include "../hostsim/hostsim.cpp"
#include "../../cave_b200/csrc/layout.cuh"

template <class T>
static void run_warm(const float* A, int B, int m, int d, const double* pred, double sign, int mode, double inner_ratio,
                     double gscale, int force_path, int max_iter, const int* index, char* warm, double* loss_i, double* grad,
                     double* proj, double* rnorm, int* status, int* iters) {
    size_t cap = (size_t)64 << 20;
    char* buf = (char*)malloc(cap);
    for (int b = 0; b < B; ++b) {
        const int q = index ? index[b] : b;            // instance of A and of the warm-start buffer
        HostPack pk; host_pack(A + (size_t)q * m * d, m, d, pk);
        Instance in; in.A = A + (size_t)q * m * d; in.gen = pk.gen.data(); in.ctype = pk.ctype.data(); in.avg = pk.avg.data();
        in.d = d; in.ngen = (int)pk.gen.size(); in.gen_nnz = pk.gen_nnz; in.nvalid = pk.nvalid; in.nsingc = pk.nsingc;
        bool all8 = true; for (float v : pk.val) all8 = all8 && v == (float)(int)v && fabsf(v) <= 127.f;
        in.csr_ok = (force_path & 2) ? 0 : (all8 ? 3 : 1);                                  // bit 1: rebuild the CSR from A
        in.ghash = pk.ghash.data(); in.pcol = pk.col.data(); in.pval = pk.val.data(); in.maxl1 = pk.maxl1; in.maxl2 = pk.maxl2;
        in.setup = nullptr;
        in.warm = warm ? warm + (size_t)q * warm_slot_bytes(m) : nullptr; in.warm_cap = (int)warm_cap_v(m); in.warm_from_slot = true;
        if (force_path & 1) in.nsingc = 0 == in.nsingc ? 1 : in.nsingc;       // bit 0: force the Newton path
        Ctx cx; EpiParams ep; ep.mode = mode; ep.inner_ratio = inner_ratio; ep.sign = sign; ep.gscale = gscale;
        SolveOpts opt; opt.max_iter = max_iter; opt.max_ls = 0; opt.tol = 0;
        static char fake_smem[96 * 1024];
        // as the solve kernel: a warm start that fails is followed by one cold solve of the same instance
        for (int retry = -1;;) {
            in.warm_from_slot = retry < 0;
            solve_instance<T, double, true>(cx, in, fake_smem, sizeof(fake_smem), buf, cap, pred + (size_t)b * d, ep, opt,
                                            grad + (size_t)b * d, proj + (size_t)b * d, loss_i + b, rnorm + b, status + b, iters + b);
            const int st = status[b];
            if (!warm) break;
            if (retry >= 0) { iters[b] += retry; break; }
            if (!((st & ST_WARM) && ((st & 0xff) == ST_ITER_CAP || (st & 0xff) == ST_STALLED))) break;
            retry = iters[b];
        }
    }
    free(buf);
}

// A: [N, m, d] with N = B without an index; index: optional int32[B] batch row -> instance of A; warm: optional warm-start
// buffer of N slots (layout.cuh warm_slot_bytes), read and written as the solve kernel does
extern "C" void hostsim_forward_backward_warm(const float* A, int B, int m, int d, const double* pred, double sign, int mode,
                                              double inner_ratio, double gscale, int compute_f32, int force_path, int max_iter,
                                              const int* index, char* warm, double* loss_i, double* grad, double* proj,
                                              double* rnorm, int* status, int* iters) {
    if (compute_f32) run_warm<float>(A, B, m, d, pred, sign, mode, inner_ratio, gscale, force_path, max_iter, index, warm, loss_i, grad, proj, rnorm, status, iters);
    else run_warm<double>(A, B, m, d, pred, sign, mode, inner_ratio, gscale, force_path, max_iter, index, warm, loss_i, grad, proj, rnorm, status, iters);
}

extern "C" size_t hostsim_warm_slot_bytes(int m) { return warm_slot_bytes(m); }
