"""Seeded adversarial instances for the structured (Newton) path of the solver: test infrastructure, pure numpy.

Every family aims at one branch of the Newton setup (nw_setup in cave_b200/csrc/solver_core.cuh, setup_kernel in
scan_kernel.cu) that the synthetic TSP / VRP / SP instances never reach; its docstring names that branch.  A family is a
float32 ``[B, m_max, d]`` array with zero padding rows.  Every instance of a structured family holds at least one
singleton row, so it takes the Newton path; only ``mixed_batch`` adds pure-general (Lawson-Hanson) instances.  Sizes stay
within d <= 400 and m <= 700, so the float64 oracle (scipy nnls on all of A) takes well under a second per instance.

``batch(name)`` repeats a family once per prediction regime (``REGIMES``) and returns the predictions with it, so one
call of the solver covers every regime of every instance."""
import numpy as np

REGIMES = ("uniform", "near", "inside", "polar", "tiny", "huge")
FAMILIES = ("pm_pairs", "int8_edges", "long_column", "cone_types", "setup_cap", "csr_overflow", "no_general", "mixed_batch")


# ------------------------------------------------------------------ building blocks
def _row(d, cols, vals):
    r = np.zeros(d, np.float32)
    r[np.asarray(cols)] = np.asarray(vals, np.float32)
    return r


def _general(rng, d, n, nnz=(2, 5), vals=(1, -1, 1, -1, 2, -2, 3), cols=None):
    """n general rows (>= 2 non-zeros) with integer values drawn from `vals`."""
    out = []
    for _ in range(n):
        k = rng.choice(d if cols is None else cols, size=int(rng.integers(nnz[0], nnz[1] + 1)), replace=False)
        out.append(_row(d, k, rng.choice(vals, size=len(k))))
    return out


def _singletons(rng, d, p=(0.5, 0.15, 0.2, 0.15), mags=(1.0,)):
    """Singleton rows: per coordinate +e_k, -e_k, both (the coordinate is free) or none, scaled by one of `mags`."""
    out = []
    for k, t in enumerate(rng.choice(4, size=d, p=p)):
        if t in (0, 2):
            out.append(_row(d, [k], [rng.choice(mags)]))
        if t in (1, 2):
            out.append(_row(d, [k], [-rng.choice(mags)]))
    if not out:
        out.append(_row(d, [0], [1.0]))
    return out


def _instance(rng, rows, shuffle=True):
    A = np.stack(rows).astype(np.float32)
    return A[rng.permutation(len(A))] if shuffle else A


def _pad(insts, extra=0):
    d = insts[0].shape[1]
    m = max(a.shape[0] for a in insts) + extra
    out = np.zeros((len(insts), m, d), np.float32)
    for b, a in enumerate(insts):
        out[b, :a.shape[0]] = a
    return out


def pack_cap_nnz(m_max, d):
    """layout.cuh pack_cap_nnz: non-zeros of general rows the packed CSR holds per instance."""
    full, c = m_max * d, 16 * d + 4096
    return (c if c < full else full + 1) // 8 * 8 + 8


def general_rows(a):
    """Rows with at least two non-zeros (the solver's general rows; -0.0 counts as zero)."""
    return a[(a != 0).sum(axis=1) >= 2]


def is_int8(a, m_max):
    """True iff the solver keeps this instance's rows as int8 (packed CSR complete, every general value an integer in
    [-127, 127]): the instances whose results the code promises bit for bit across routes."""
    g = general_rows(a)
    v = g[g != 0]
    return len(v) <= pack_cap_nnz(m_max, a.shape[1]) and bool(np.all((v == np.round(v)) & (np.abs(v) <= 127)))


def has_singletons(a):
    return bool(((a != 0).sum(axis=1) == 1).any())


# ------------------------------------------------------------------ families
def pm_pairs(rng, d=40):
    """+- merge (hash match, exact compare, mutual choice): a with -a; the pair twice (a, a, -a, -a); a triple
    (a, -a, a); a with -2a (spans the line, not merged); a with -a' where a' differs from a in one value, in one column
    or by one extra non-zero (near misses: the order-free hash or the non-zero count already rejects them, so the
    exact compare's accept path is exercised and its reject path, which only a 64-bit hash collision reaches, is not).
    One instance has float rows (merged through the float compare), one keeps its rows in order."""
    out = []
    for variant in range(6):
        base = _general(rng, d, 14)
        a = [_general(rng, d, 1, nnz=(3, 6))[0] for _ in range(8)]
        extra = [a[0], -a[0],                                  # a, -a
                 a[1], a[1], -a[1], -a[1],                     # the same pair twice
                 a[2], -a[2], a[2],                            # a triple
                 a[3], -2 * a[3]]                              # a and -2a: not merged
        near = a[4].copy(); k = np.flatnonzero(near)[0]; near[k] += 1 if near[k] != -1 else -1
        extra += [a[4], -near]                                 # one value differs
        near = a[5].copy(); nz = np.flatnonzero(near); z = np.flatnonzero(near == 0)
        near[z[0]], near[nz[-1]] = near[nz[-1]], 0
        extra += [a[5], -near]                                 # one column differs, same non-zero count
        near = a[6].copy(); near[np.flatnonzero(near == 0)[1]] = 1
        extra += [a[6], -near]                                 # one extra non-zero
        extra += [-a[7], a[7]]                                 # the negative first
        rows = base + extra
        if variant == 4:
            rows = [r * np.float32(0.37) for r in rows]       # float rows: merged by the float compare, float Hessian
        out.append(_instance(rng, rows + _singletons(rng, d), shuffle=variant != 5))
    return _pad(out)


def int8_edges(rng, d=40):
    """The int8 test of the packed CSR (csr_ok bit 1): integer rows with values +-127 (int8: exact int32 Hessian);
    instances where one row holds 128, -128 or 0.5 (the whole instance goes to the float path); negative zeros in
    general rows and a row of negative zeros amid the valid rows (zero, not a non-zero; the latter is padding)."""
    out = []
    for variant in range(6):
        rows = _general(rng, d, 16, vals=(127, -127, 1, -1, 64))
        if variant == 1:
            rows[3][np.flatnonzero(rows[3])[0]] = 128.0
        elif variant == 2:
            rows[5][np.flatnonzero(rows[5])[-1]] = -128.0
        elif variant == 3:
            rows[7][np.flatnonzero(rows[7])[0]] = 0.5
        elif variant == 4:
            for r in rows[:8]:
                r[np.flatnonzero(r == 0)[:3]] = -0.0
            rows.append(np.full(d, -0.0, np.float32))
        elif variant == 5:
            rows += [-rows[0], np.sign(rows[1]) * np.float32(127)]
        out.append(_instance(rng, rows + _singletons(rng, d)))
    return _pad(out)


def long_column(rng, d=300, lengths=(65, 100, 250), n_float=1):
    """CSC columns longer than 64 general-row entries (the in-solver setup's per-column sort used to stop there,
    leaving such a column in the order the warps' atomic cursor filled it): one column hit by 65, one by 100 and one by
    250 general rows.  One general row with more than 256 non-zeros (the loop branch of setup_kernel's CSC fill, whose
    unrolled part covers 256).  The last instance has float rows."""
    out = []
    n_int = 2
    for b in range(n_int + n_float):
        n = max(lengths)
        cols = rng.permutation(d)
        hot = cols[:len(lengths)]
        rows = _general(rng, d, n, nnz=(1, 3), cols=cols[len(lengths):])
        for c, L in zip(hot, lengths):
            for i in rng.permutation(n)[:L]:
                rows[i][c] = rng.choice((1, -1, 2))
        k = rng.choice(cols[len(lengths):], size=min(d - 20, 280), replace=False)
        rows.append(_row(d, k, rng.choice((1, -1), size=len(k))))
        if b >= n_int:
            rows = [r * np.float32(0.5) for r in rows]
        out.append(_instance(rng, rows + _singletons(rng, d, p=(0.75, 0.1, 0.05, 0.1))))
    return _pad(out)


def cone_types(rng, d=30):
    """The singleton cone type of every coordinate (ctype, psi): no singleton row ({0}), only +e_k, only -e_k, both (R),
    duplicated singletons (the same row twice, and +e_k beside 2.5 e_k), and singleton magnitudes 1e-3, 0.5, 2.5 and
    127 (magnitudes of singleton rows do not enter the int8 test of the general rows)."""
    out = []
    for variant in range(4):
        mags = ((1.0,), (1e-3, 0.5, 2.5, 127.0), (1e-3,), (127.0, 2.5))[variant]
        p = ((0.25, 0.25, 0.25, 0.25), (0.4, 0.2, 0.2, 0.2), (0.0, 0.0, 1.0, 0.0), (0.2, 0.3, 0.1, 0.4))[variant]
        sing = _singletons(rng, d, p=p, mags=mags)
        sing += [sing[0].copy(), sing[-1].copy()]
        sing.append(_row(d, [int(np.flatnonzero(sing[1])[0])], [2.5]))
        out.append(_instance(rng, _general(rng, d, 12) + sing))
    return _pad(out)


def setup_cap(rng, d=300):
    """The limits of the cached setup and of the small solver slot: 192, 193, 256 and 257 general rows before merging
    (setup_cap_v = min(m_max, 256) decides between the cached and the in-solver setup, cap_rows = 192 between the small
    and the worst-case slot), and 257 rows that merge into 255 variables (still above the cache's row limit)."""
    out = []
    for n in (192, 193, 256, 257):
        out.append(_instance(rng, _general(rng, d, n, nnz=(2, 4)) + _singletons(rng, d, p=(0.7, 0.1, 0.1, 0.1))))
    rows = _general(rng, d, 255, nnz=(2, 4))
    rows += [-rows[0], -rows[1]]
    out.append(_instance(rng, rows + _singletons(rng, d, p=(0.7, 0.1, 0.1, 0.1))))
    return _pad(out)


def csr_overflow(rng, d=200):
    """General rows with more non-zeros than the packed CSR holds (pack_cap_nnz, csr_ok = 0): the solver reads its rows
    back from A (float path, hashes and norms computed in the solver), or reports ST_NOSPACE when the pack keeps no
    dense rows.  Integer and float values, and one instance that fits beside them."""
    out = []
    n = pack_cap_nnz(2 * d, d) // int(0.95 * d) + 2
    for variant in range(3):
        rows = []
        for _ in range(n if variant < 2 else 8):
            k = rng.choice(d, size=int(0.95 * d), replace=False)
            v = rng.choice((1, -1, 2, -2, 3), size=len(k)).astype(np.float32)
            rows.append(_row(d, k, v * (np.float32(0.3) if variant == 1 else 1)))
        out.append(_instance(rng, rows + _singletons(rng, d, p=(0.7, 0.1, 0.1, 0.1))))
    A = _pad(out)
    assert A.shape[1] <= 2 * d
    return A


def no_general(rng, d=50):
    """Singleton rows only (ngen = 0): the closed form r = c, no Newton iteration."""
    out = []
    for p in ((0.25, 0.25, 0.25, 0.25), (1.0, 0.0, 0.0, 0.0), (0.0, 0.0, 0.5, 0.5)):
        sing = _singletons(rng, d, p=p, mags=(1.0, 2.5))
        out.append(_instance(rng, sing + [sing[0].copy()]))
    return _pad(out)


def pure_general(rng, d, m):
    """No singleton row: the Lawson-Hanson path (dense float rows)."""
    return rng.standard_normal((m, d)).astype(np.float32)


def mixed_batch(rng, d=300):
    """Instances of every family at one d, pure-general instances (Lawson-Hanson) and extra padding, shuffled into
    one batch: the cost-ordered work queue (order_kernel) must write every result back to its own instance, whatever
    path, slot and setup each one takes."""
    parts = [pm_pairs(rng, d)[[0, 4]], int8_edges(rng, d)[[0, 3]], long_column(rng, d)[[0, 2]], cone_types(rng, d)[[1]],
             setup_cap(rng, d)[[1, 4]], csr_overflow(rng, d)[[0]], no_general(rng, d)[[0]]]
    insts = [a[(a != 0).any(axis=1)] for part in parts for a in part]
    insts += [pure_general(rng, d, 40), pure_general(rng, d, 90)]
    order = rng.permutation(len(insts))
    return _pad([insts[i] for i in order], extra=7)


_MAKERS = dict(pm_pairs=pm_pairs, int8_edges=int8_edges, long_column=long_column, cone_types=cone_types,
               setup_cap=setup_cap, csr_overflow=csr_overflow, no_general=no_general, mixed_batch=mixed_batch)


def family(name, seed=0):
    """float32 [B, m_max, d] with zero padding rows."""
    return _MAKERS[name](np.random.default_rng([seed, FAMILIES.index(name)]))


# ------------------------------------------------------------------ predictions
def _polar_point(rng, a):
    """A point of the polar cone {q : A q <= 0}: the Moreau residual c0 - P(c0) of a random c0 (certified float64
    projection of the oracle)."""
    from oracle import cave_oracle as O
    c0 = rng.standard_normal(a.shape[1])
    return c0 - O.project_nnls(c0, a.astype(np.float64), fp64_out=True, certify=True)[0]


def predictions(A, regime, seed=0):
    """Predicted costs [B, d] float32 for minimisation (the solver projects c = -pred):
    'uniform' U(0, 1)^d and 'near' (noisy costs around a random 0/1 solution) in the manner of synth.predictions;
    'inside' c = A^T lam with lam > 0 on every row (inside the cone); 'polar' c in the polar cone (projection 0);
    'tiny' / 'huge' the uniform costs scaled by 1e-4 / 1e4."""
    rng = np.random.default_rng([seed, REGIMES.index(regime)])
    B, m, d = A.shape
    if regime in ("uniform", "tiny", "huge"):
        p = rng.random((B, d))
        return (p * {"uniform": 1.0, "tiny": 1e-4, "huge": 1e4}[regime]).astype(np.float32)
    if regime == "near":
        sol = rng.random((B, d)) < 0.3
        c_true = np.where(sol, 0.2, 1.0) * (0.5 + rng.random((B, d)))
        return (c_true * (1.0 + 0.5 * rng.standard_normal((B, d)))).astype(np.float32)
    if regime == "inside":
        lam = 0.05 + rng.random((B, m))
        return (-np.einsum("bm,bmd->bd", lam, A.astype(np.float64))).astype(np.float32)
    return np.stack([-_polar_point(rng, A[b]) for b in range(B)]).astype(np.float32)


def batch(name, seed=0):
    """(A [R*B, m, d], pred [R*B, d], regime [R*B]): the family once per regime of REGIMES."""
    A = family(name, seed)
    preds = [predictions(A, r, seed) for r in REGIMES]
    regime = np.repeat(np.arange(len(REGIMES)), A.shape[0])
    return np.concatenate([A] * len(REGIMES)), np.concatenate(preds), regime
