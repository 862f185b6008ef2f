"""Every batched linearisation instance against an exact QR reference.

lin_kernel (csrc/blsq_lin.cuh) turns [J | f] of every running problem into the
record the round kernel works from (LinRec<N>): R packed row-major from 0, Q^T f
at NT, g = J^T f at NT + N and f.f at NT + 2N.  launch_lin picks one of
8 N x 4 lane-group classes x 3 Jacobian modes x {dense, ROWS} instances; the
checks below call blsq_linearise_batched[_rows] directly at both sides of every
class edge for every N.

Reference: the (n+1) x (n+1) Gram matrix of [J | f] formed exactly in Python
integers (every double is an integer times a power of two), then its Cholesky
factor at 256 bits in mpmath.  Its first n columns are R (positive diagonal),
column n is Q^T f; the Gram matrix itself holds g and f.f.  Rank-deficient
problems (an exactly zero pivot) are gated backward: R^T R against J^T J.

Every check takes ``lib`` and a torch device: the unmarked tests run it on the
host emulation (tests/host_emul/emul.cpp, a serial Gram-Schmidt: they validate
the reference and the gates), the ``gpu``-marked ones on libblsq_b200.so.
"""
import ctypes as C
import math
from fractions import Fraction

import mpmath
import numpy as np
import pytest
import torch

import hostemul

U = 2.0 ** -53
A_BATCH = 37                      # the last warp and block are partly filled
SENTINEL = np.array([0x7FF4DEADBEEF0001], dtype=np.int64).view(np.float64)[0]
CLASSES = ("G8", "G16", "G32", "MULTI")
FAMILIES = ("random", "kappa6", "graded", "dup_col", "kappa12", "zero_col", "f_zero",
            "rows3_zero")


def rpl(N):
    """Rows per lane of lin_kernel (LinCfg<N>::RPL)."""
    return 8 if N <= 6 else 4


def lin_class(N, m):
    """The lane-group class launch_lin picks: the smallest group whose
    registers hold all m rows, else 32 lanes folding chunks (MULTI)."""
    for G, name in ((8, "G8"), (16, "G16"), (32, "G32")):
        if m <= G * rpl(N):
            return name
    return "MULTI"


def group_size(lib, cls):
    """Rows are spread over G lanes on the GPU; the host emulation sums them
    serially (one 'lane')."""
    if not lib.requires_cuda:
        return 1
    return {"G8": 8, "G16": 16, "G32": 32, "MULTI": 32}[cls]


def widths(N):
    """m at both sides of every class edge of N, plus m < n and m = n."""
    edges = ((63, 64, 65, 127, 128, 129, 255, 256, 257, 512, 513, 1100) if N <= 6 else
             (32, 33, 64, 65, 128, 129, 256, 257, 1100))
    return sorted({m for m in (1, N - 1, N) + edges if m >= 1})


def tri(N, i, j):
    return i * N - (i * (i - 1)) // 2 + (j - i)


def decode(rec, N):
    """(R upper N x N, qtf, g, f.f) of one LinRec<N>."""
    NT = N * (N + 1) // 2
    R = np.zeros((N, N))
    for i in range(N):
        for j in range(i, N):
            R[i, j] = rec[tri(N, i, j)]
    return R, rec[NT:NT + N].copy(), rec[NT + N:NT + 2 * N].copy(), rec[NT + 2 * N]


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


# ---------------------------------------------------------------- reference --

def exact_gram(M):
    """M^T M of a finite float64 matrix exactly: integer matrix Gi and column
    exponents e with (M^T M)_ij = Gi_ij 2^(e_i + e_j)."""
    mant, ex = np.frexp(M)
    Mi = (mant * 2.0 ** 53).astype(np.int64)          # exact: 53-bit mantissas
    ex = ex.astype(np.int64) - 53
    nz = Mi != 0
    e0 = np.where(nz, ex, np.iinfo(np.int64).max).min(axis=0)
    e0 = np.where(nz.any(axis=0), e0, 0)
    sh = np.where(nz, ex - e0, 0)
    X = np.empty(M.shape, dtype=object)
    for (i, j), v in np.ndenumerate(Mi):
        X[i, j] = int(v) << int(sh[i, j])
    return X.T @ X, [int(v) for v in e0]


def reference(J, f):
    """Exact-Gram / 256-bit Cholesky reference of one problem.  R and qtf are
    None when the Cholesky meets a zero pivot (rank deficient, or m < n)."""
    m, n = J.shape
    Gi, e = exact_gram(np.concatenate([J, f[:, None]], axis=1))
    k = n + 1
    with mpmath.workprec(256):
        G = [[mpmath.ldexp(mpmath.mpf(int(Gi[i, j])), e[i] + e[j]) for j in range(k)]
             for i in range(k)]
        Rf = [[mpmath.mpf(0)] * k for _ in range(n)]
        full = True
        for i in range(n):
            d = G[i][i] - mpmath.fsum(Rf[p][i] ** 2 for p in range(i))
            if d <= G[i][i] * mpmath.mpf(2) ** -200 or G[i][i] == 0:
                full = False
                break
            Rf[i][i] = mpmath.sqrt(d)
            for j in range(i + 1, k):
                Rf[i][j] = (G[i][j] - mpmath.fsum(Rf[p][i] * Rf[p][j] for p in range(i))) / Rf[i][i]
        out = dict(
            full=full,
            gram=[[Fraction(int(Gi[i, j])) * Fraction(2) ** (e[i] + e[j]) for j in range(k)]
                  for i in range(k)],
            norms=np.array([float(mpmath.sqrt(G[j][j])) for j in range(k)]),
            g=np.array([float(G[j][n]) for j in range(n)]),
            ff=float(G[n][n]))
        if full:
            out["R"] = np.array([[float(Rf[i][j]) for j in range(n)] for i in range(n)])
            out["qtf"] = np.array([float(Rf[i][n]) for i in range(n)])
    out["absjf"] = np.abs(J * f[:, None]).sum(axis=0)
    if full:
        # Householder (LAPACK) on the same input: the Q^T f gate is relative to it
        Rh = np.linalg.qr(np.concatenate([J, f[:, None]], axis=1), mode="r")
        s = np.sign(np.diag(Rh)[:n])
        out["qtf_lapack_err"] = float(np.abs(s * Rh[:n, n] - out["qtf"]).max())
        out["qtf_mgs_err"] = float(np.abs(mgs_qtf(J, f) - out["qtf"]).max())
        out["kappa"] = float(np.linalg.cond(J))
    return out


def mgs_qtf(J, f):
    """Q^T f of a textbook modified Gram-Schmidt on [J | f] in float64.  At
    m = n the last directions of Q are the orthogonal complement, which
    Householder gets to O(u) and Gram-Schmidt only to O(kappa u): the Q^T f
    gate allows the larger of the two errors, and kappa u |f| (first-order
    bound of a backward-stable QR)."""
    a = np.concatenate([J, f[:, None]], axis=1).copy()
    n = J.shape[1]
    q = np.zeros(n)
    for k in range(n):
        d = a[:, k] @ a[:, k]
        r = math.sqrt(d)
        for j in range(k + 1, n + 1):
            dj = a[:, k] @ a[:, j]
            if j == n:
                q[k] = dj / r
            a[:, j] -= (dj / d) * a[:, k]
    return q


def exact(v):
    return Fraction(float(v))


def backward_errors(R, q, ref):
    """Worst |R^T R - J^T J|_ij / (u |a_i| |a_j|) and |R^T q - J^T f|_j /
    (u |a_j| |f|), both formed exactly."""
    n = R.shape[0]
    G, nrm = ref["gram"], ref["norms"]
    Rx = [[exact(R[i, j]) for j in range(n)] for i in range(n)]
    qx = [exact(v) for v in q]
    ew, eq = 0.0, 0.0
    for j in range(n):
        for i in range(j + 1):
            d = sum(Rx[p][i] * Rx[p][j] for p in range(n)) - G[i][j]
            sc = nrm[i] * nrm[j]
            ew = max(ew, float(abs(d)) / (U * sc) if sc > 0 else (0.0 if d == 0 else math.inf))
        d = sum(Rx[p][j] * qx[p] for p in range(n)) - G[j][n]
        sc = nrm[j] * nrm[n]
        eq = max(eq, float(abs(d)) / (U * sc) if sc > 0 else (0.0 if d == 0 else math.inf))
    return ew, eq


def gate_record(rec, N, m, G, ref, fam, stats, fails, key):
    """All gates of one record; worst error / gate unit into stats[key]."""
    R, q, g, ff = decode(rec, N)
    st = stats.setdefault(key, dict(R=0.0, qtf=0.0, qtf_bwd=0.0, g=0.0, ff=0.0, gram_bwd=0.0))
    k = math.ceil(m / G) + 6
    nrm = ref["norms"]

    def worse(name, v, gate):
        st[name] = max(st[name], v)
        if not v <= gate:
            fails.append((key, name, m, v, gate))
    if not (np.isfinite(R).all() and np.isfinite(q).all() and np.isfinite(g).all()
            and np.isfinite(ff)):
        fails.append((key, "non-finite record", None, None))
        return
    den = np.maximum(U * ref["absjf"], 1e-300)
    worse("g", float((np.abs(g - ref["g"]) / den).max()) if (ref["absjf"] > 0).any() or
          (g != 0).any() else 0.0, k)
    worse("ff", abs(ff - ref["ff"]) / (U * ref["ff"]) if ref["ff"] > 0 else
          (0.0 if ff == 0 else math.inf), k)
    ew, eq = backward_errors(R, q, ref)
    worse("qtf_bwd", eq, 16)
    if ref["full"]:
        colu = U * nrm[:N]
        worse("R", float((np.abs(np.triu(R - ref["R"])) / colu[None, :]).max()), 64)
        err = float(np.abs(q - ref["qtf"]).max())
        gate = max(4 * ref["qtf_lapack_err"], 4 * ref["qtf_mgs_err"],
                   max(16, ref["kappa"]) * U * nrm[N])
        worse("qtf", err / (U * nrm[N]) if nrm[N] > 0 else (0.0 if err == 0 else math.inf),
              gate / (U * nrm[N]) if nrm[N] > 0 else 0.0)
    else:
        worse("gram_bwd", ew, 64)
    # an exactly zero column keeps an exactly zero diagonal and row of R.  An
    # exact copy of column 0 does so in the serial emulation (coefficient
    # d / d = 1); lin_kernel forms the coefficient as d * (1/sqrt(d))^2, which
    # need not be 1, and leaves a diagonal of a few u |a_j| (DESIGN 5)
    if fam == "zero_col" and N >= 2 and m >= N:
        j = N // 2
        if not (np.all(R[j, j:] == 0.0) and np.all(R[:j, j] == 0.0) and q[j] == 0.0):
            fails.append((key, "zero column: exact zero row", m, float(R[j, j]), 0.0))
    if fam == "dup_col" and N >= 2 and m >= N:
        j = N - 1
        v = abs(R[j, j]) / (U * nrm[j])
        st["dup_diag"] = max(st.get("dup_diag", 0.0), v)
        if not (v == 0.0 if G == 1 else v <= 16):
            fails.append((key, "duplicate column: diagonal", m, v, 0.0 if G == 1 else 16))


# --------------------------------------------------------------- test data --

def make_problem(rng, fam, m, N):
    """J (m, N), f (m) of one input family.  Entries of the plain families have
    magnitudes in [0.5, 1.5]: dropping or repeating any one row moves f.f and
    every g_j far outside their gates."""
    def mag(*shape):
        return rng.uniform(0.5, 1.5, shape) * rng.choice([-1.0, 1.0], shape)
    J, f = mag(m, N), mag(m)
    if fam in ("kappa6", "kappa12") and m >= N and N >= 2:
        kap = 1e6 if fam == "kappa6" else 1e12
        Uo = np.linalg.qr(rng.standard_normal((m, N)))[0]
        Vo = np.linalg.qr(rng.standard_normal((N, N)))[0]
        J = (Uo * np.logspace(0, -np.log10(kap), N)) @ Vo.T
    elif fam == "graded":
        J = J * np.ldexp(1.0, rng.integers(-60, 61, N))[None, :]
        f = f * np.ldexp(1.0, int(rng.integers(-60, 61)))
    elif fam == "dup_col" and N >= 2:
        J[:, N - 1] = J[:, 0]
    elif fam == "zero_col":
        J[:, N // 2] = 0.0
    elif fam == "f_zero":
        f[:] = 0.0
    elif fam == "rows3_zero":
        J[::3] = 0.0
        f[::3] = 0.0
    return J, f


def make_batch(N, m, seed):
    rng = np.random.default_rng(seed)
    fams = [FAMILIES[b % len(FAMILIES)] for b in range(A_BATCH)]
    Js, fs = zip(*[make_problem(rng, fam, m, N) for fam in fams])
    return np.stack(Js), np.stack(fs), fams


class Runner:
    """Calls the linearisation entry points of ``lib`` on ``dev`` and counts
    the (N, class, mode) instances it launched."""

    def __init__(self, lib, dev):
        self.lib, self.dev = lib, dev
        self.dense, self.rows = set(), set()

    def T(self, a, dtype=torch.float64):
        return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(self.dev)

    def run(self, N, m, running, F, J=None, Fp=None, dx=None, idx=None, rows=None):
        """Records (A, SIZE) with lin prefilled with SENTINEL; `running` is the
        status mask indexed by problem id, F / J / Fp by slot."""
        lib = self.lib
        A = F.shape[0]
        mode = 0 if Fp is None else (1 if len(Fp) == N else 2)
        LS = lib.lin_record_size(N)
        nprob = len(running)
        ist = np.zeros((nprob, 8), dtype=np.int32)
        ist[:, 0] = np.where(running, -1, 0)
        ist_t = self.T(ist, torch.int32)
        lin = self.T(np.full((A, LS), SENTINEL))
        Ft = self.T(F)
        keep = [Ft, ist_t, lin]
        Jp = None
        if J is not None:
            Jt = self.T(J)
            keep.append(Jt)
            Jp = Jt.data_ptr()
        plist, dxp = None, None
        if Fp is not None:
            Fpt = [self.T(a) for a in Fp]
            dxt = self.T(dx)
            keep += Fpt + [dxt]
            arr = (C.c_void_p * len(Fpt))(*[t.data_ptr() for t in Fpt])
            plist, dxp = C.cast(arr, C.c_void_p), dxt.data_ptr()
        ip = None
        if idx is not None:
            it = self.T(idx, torch.int32)
            keep.append(it)
            ip = it.data_ptr()
        st = lib.stream(ist_t)
        if rows is None:
            lib.call("blsq_linearise_batched", A, ip, m, N, Ft.data_ptr(), Jp, plist, dxp,
                     mode, ist_t.data_ptr(), lin.data_ptr(), st)
            self.dense.add((N, lin_class(N, m), mode))
        else:
            rt = self.T(rows, torch.int32)
            keep.append(rt)
            lib.call("blsq_linearise_batched_rows", A, ip, m, N, Ft.data_ptr(), Jp, plist,
                     dxp, mode, ist_t.data_ptr(), lin.data_ptr(), rt.data_ptr(), st)
            self.rows.add((N, lin_class(N, m), mode))
        return lin.cpu().numpy()


def fd_inputs(rng, J, F, mode):
    """Fpert, dx for mode 1 / 2 and the Jacobian NumPy forms from them
    (scipy _dense_difference), with quotients near the subnormal and the
    overflow ends on some problems."""
    A, m, N = J.shape
    dx = np.ldexp(rng.uniform(0.5, 1.0, (A, N)), rng.integers(-30, -20, (A, N)))
    dx[2::5, 0] = 3e-8
    D = J * dx[:, None, :]                           # the differences f1 - f0
    dx[0::5] = 1e-300                                # quotients near 1e8, every 4th
    D[0::5] = np.clip(J[0::5], -1, 1) * 1e-292       # row near 1e307 (below overflow)
    D[0::5, ::4] = np.clip(J[0::5, ::4], -1, 1) * 1e7
    dx[1::5] = 1e300                                 # subnormal quotients
    D[1::5] = J[1::5] * 1e-10
    if mode == 1:
        Fp = [F + D[:, :, j] for j in range(N)]
        Jfd = np.stack([(Fp[j] - F) / dx[:, None, j] for j in range(N)], axis=2)
        return Fp, dx, Jfd
    one = rng.random((A, N)) < 0.5
    Fp = []
    for j in range(N):
        f1 = F + 0.5 * D[:, :, j]
        f2 = F + D[:, :, j] * np.where(one[:, j:j + 1], 1.0, -1.0)
        Fp += [f1, f2]
    Jfd = np.empty_like(J)
    for j in range(N):
        f1, f2 = Fp[2 * j], Fp[2 * j + 1]
        d1 = ((-3 * F + 4 * f1) - f2) / dx[:, None, j]
        d2 = (f2 - f1) / dx[:, None, j]
        Jfd[:, :, j] = np.where(one[:, j:j + 1], d1, d2)
    return Fp, np.concatenate([dx, one.astype(np.float64)], axis=1), Jfd


# ------------------------------------------------------------------ checks --

def check_every_instance(lib, dev, Ns=range(1, 9)):
    """Gates against the reference at every class edge of every N, dense and
    (where the library has it) ROWS, the three Jacobian modes, and the
    bit-exact invariances."""
    run = Runner(lib, dev)
    has_rows = lib.has("blsq_linearise_batched_rows")
    stats, fails, nref = {}, [], 0
    for N in Ns:
        for m in widths(N):
            cls = lin_class(N, m)
            G = group_size(lib, cls)
            seed = 1000 * N + m
            rng = np.random.default_rng(seed + 7)
            J, F, fams = make_batch(N, m, seed)
            refs = [reference(J[b], F[b]) for b in range(A_BATCH)]
            nref += A_BATCH
            run1 = np.arange(A_BATCH) % 3 != 1               # a third not running
            base = run.run(N, m, run1, F, J)
            for b in range(A_BATCH):
                key = (N, cls, fams[b])
                if run1[b]:
                    gate_record(base[b], N, m, G, refs[b], fams[b], stats, fails, key)
                elif not same_bits(base[b], np.full_like(base[b], SENTINEL)):
                    fails.append((key, "record of a stopped problem written", m, b))
            # shuffled idx, another running set: slot s holds problem perm[s]
            perm = rng.permutation(A_BATCH)
            run2 = np.arange(A_BATCH) % 3 != 2
            sh = run.run(N, m, run2, F[perm], J[perm], idx=perm)
            for s, p in enumerate(perm):
                if not run2[p]:
                    if not same_bits(sh[s], np.full_like(sh[s], SENTINEL)):
                        fails.append(((N, cls), "stopped record written (idx)", m, s))
                elif run1[p]:
                    if not same_bits(sh[s], base[p]):
                        fails.append(((N, cls), "slot / warp-mates / idx changed bits", m, p))
                else:
                    gate_record(sh[s], N, m, G, refs[p], fams[p], stats, fails,
                                (N, cls, fams[p]))
            # a smaller batch A = 11 of other problems in another order
            sub = rng.choice(np.nonzero(run1)[0], 11, replace=False)
            sm = run.run(N, m, np.ones(11, bool), F[sub], J[sub])
            for s, p in enumerate(sub):
                if not same_bits(sm[s], base[p]):
                    fails.append(((N, cls), "A changed bits", m, int(p)))
            # NaN / Inf in one running problem's J leaves every other record
            # alone: slot 5 of the base pass (slot 6 of its G = 8 warp runs
            # too), and slot 1 of the A = 11 pass, where every problem runs
            # (the G = 8 and 16 warps of slot 1 take the whole-chunk path
            # wherever m fills the chunk)
            assert run1[5] and run1[6]
            for poison in (np.nan, np.inf):
                Jb = J.copy()
                Jb[5, m - 1, N - 1] = poison
                pb = run.run(N, m, run1, F, Jb)
                if not same_bits(np.delete(pb, 5, axis=0), np.delete(base, 5, axis=0)):
                    fails.append(((N, cls), f"{poison} leaked into other records", m, 5))
                if np.isfinite(decode(pb[5], N)[2]).all():        # g holds the poison
                    fails.append(((N, cls), f"{poison} not read", m, 5))
                Js = J[sub].copy()
                Js[1, m - 1, N - 1] = poison
                ps = run.run(N, m, np.ones(11, bool), F[sub], Js)
                if not same_bits(np.delete(ps, 1, axis=0), np.delete(sm, 1, axis=0)):
                    fails.append(((N, cls), f"{poison} leaked into warp mates", m, 1))
                if np.isfinite(decode(ps[1], N)[2]).all():
                    fails.append(((N, cls), f"{poison} not read (A = 11)", m, 1))
            if has_rows:
                rr = run.run(N, m, run1, F, J, rows=np.full(A_BATCH, m))
                if not same_bits(rr, base):
                    fails.append(((N, cls), "ROWS with rows = m differs from dense", m, 0))
            # finite-difference modes == mode 0 on the NumPy-formed Jacobian
            for mode in (1, 2):
                Fp, dx, Jfd = fd_inputs(rng, J, F, mode)
                fd = run.run(N, m, run1, F, Fp=Fp, dx=dx)
                an = run.run(N, m, run1, F, Jfd)
                if not same_bits(fd, an):
                    bad = [b for b in range(A_BATCH) if not same_bits(fd[b], an[b])]
                    fails.append(((N, cls), f"mode {mode} != mode 0 on its Jacobian", m, bad))
                if has_rows:
                    fr = run.run(N, m, run1, F, Fp=Fp, dx=dx, rows=np.full(A_BATCH, m))
                    if not same_bits(fr, fd):
                        fails.append(((N, cls), f"ROWS mode {mode} differs from dense", m, 0))
    report = dict(dense=len(run.dense), rows=len(run.rows), references=nref)
    print("\nworst error / gate unit per (N, class, family):")
    print("  (R: u|a_j|, qtf and backward checks: u|a_j||f|, g: u sum|J_ij f_i|, f.f: u f.f; "
          "gates R 64, qtf_bwd 16, gram_bwd 64, g and f.f ceil(m/G) + 6)")
    for key in sorted(stats):
        print("  ", key, {k: float(f"{v:.3g}") for k, v in stats[key].items()})
    print("instances:", report)
    for f in fails[:40]:
        print("FAIL", f)
    assert not fails, f"{len(fails)} failures, first: {fails[0]}"
    return report, run


def check_all_instances_launched(lib, dev):
    report, run = check_every_instance(lib, dev)
    want = {(N, c, mo) for N in range(1, 9) for c in CLASSES for mo in (0, 1, 2)}
    assert run.dense == want and len(want) == 96, sorted(want - run.dense)
    if lib.requires_cuda:
        assert run.rows == want, sorted(want - run.rows)
    return report


def check_power_of_two_scaling(lib, dev):
    """Scaling column j of J by 2^c_j and f by 2^c_f scales column j of R by
    exactly 2^c_j, Q^T f by 2^c_f, g_j by 2^(c_j + c_f) and f.f by 4^c_f, for
    c in [-400, 400]: Gram-Schmidt is covariant and norm_terms' reciprocal
    square root is too."""
    run = Runner(lib, dev)
    rng = np.random.default_rng(11)
    worst = 0
    for N in range(1, 9):
        for m in ((64, 128, 256, 513) if N <= 6 else (32, 64, 128, 257)):
            J, F, _ = make_batch(N, m, 5000 + N * m)
            J[:, :, :], F[:] = make_problem(rng, "random", m * A_BATCH, N)[0].reshape(
                A_BATCH, m, N), make_problem(rng, "random", m * A_BATCH, 1)[1].reshape(A_BATCH, m)
            run1 = np.ones(A_BATCH, bool)
            base = run.run(N, m, run1, F, J)
            c = rng.integers(-400, 401, (A_BATCH, N))
            cf = rng.integers(-400, 401, A_BATCH)
            sc = run.run(N, m, run1, np.ldexp(F, cf[:, None]),
                         np.ldexp(J, c[:, None, :]))
            for b in range(A_BATCH):
                R0, q0, g0, f0 = decode(base[b], N)
                R1, q1, g1, f1 = decode(sc[b], N)
                want = (np.ldexp(R0, c[b][None, :]), np.ldexp(q0, cf[b]),
                        np.ldexp(g0, c[b] + cf[b]), np.ldexp(f0, 2 * cf[b]))
                for got, w in zip((R1, q1, g1, f1), want):
                    d = np.abs(np.asarray(got).view(np.int64) - np.asarray(w).view(np.int64))
                    worst = max(worst, int(np.max(d)))
    print("power-of-two scaling: worst deviation", worst, "ulp")
    assert worst == 0
    return worst


def check_scale_range(lib, dev):
    """The range the batched linearisation is valid in: [J | f] scaled by 2^c.
    Sums of squares are formed in double, so once squared entries leave the
    normal range the record is lost.  Pinned: c = -500 and c = +500 meet every
    gate; at c = -540 the squares underflow (R wrong far beyond its gate), at
    c = +520 they overflow (record not finite)."""
    with np.errstate(all="ignore"):             # the references of the lost records
        return _scale_range(Runner(lib, dev))


def _scale_range(run):
    lib = run.lib
    out = {}
    for N in (2, 5, 8):
        for m in (N + 3, 257, 513):
            cls = lin_class(N, m)
            rng = np.random.default_rng(N * m)
            J, F = make_problem(rng, "random", m * A_BATCH, N)
            J, F = J.reshape(A_BATCH, m, N), F[:m * A_BATCH].reshape(A_BATCH, m)
            for c in (-500, 500, -540, 520):
                Js, Fs = np.ldexp(J, c), np.ldexp(F, c)
                rec = run.run(N, m, np.ones(A_BATCH, bool), Fs, Js)
                stats, fails = {}, []
                for b in range(0, A_BATCH, 9):
                    ref = reference(Js[b], Fs[b])
                    gate_record(rec[b], N, m, group_size(lib, cls), ref, "random", stats,
                                fails, c)
                # the fields of each record (the padding words are never written)
                nfin = sum(all(np.isfinite(v).all() for v in decode(rec[b], N))
                           for b in range(A_BATCH))
                out[(N, m, c)] = (stats.get(c, {}).get("R"), nfin)
                if abs(c) == 500:
                    assert not fails and nfin == A_BATCH, ((N, m, c), fails[:3], nfin)
                elif c < 0:
                    assert stats[c]["R"] > 1e6, ((N, m, c), stats)
                else:
                    assert nfin == 0, (N, m, c, nfin)
    print("scale range (N, m, c) -> (worst R error / u|a_j|, finite records of 37):", out)
    return out


def check_covariance(lib, dev):
    """blsq_covariance ((R^T R)^-1 from R) against an exact-integer inverse of
    the given double R: packed records for n = 1..8, dense (the tall path) for
    n = 9, 33, 64, 129, 256.  Gate: 4 x the error of inv(R) @ inv(R).T in
    NumPy plus 4 n u max|C*|.  The singular threshold is pinned: a pivot of
    exactly 16 n eps max|r_ii| gives NaN, one ulp above it a finite matrix."""
    T = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64).to(dev)  # noqa
    rng = np.random.default_rng(21)
    out = {}

    def cov(Rs, packed):
        B, n = Rs.shape[0], Rs.shape[1]
        if packed:
            NT = n * (n + 1) // 2
            rec = np.zeros((B, NT + 3))                # stride != NT
            for b in range(B):
                rec[b, :NT] = [Rs[b, i, j] for i in range(n) for j in range(i, n)]
            stride = NT + 3
        else:
            rec, stride = Rs.reshape(B, n * n), n * n
        rt = T(rec)
        ct = torch.empty((B, n, n), dtype=torch.float64, device=dev)
        lib.call("blsq_covariance", B, n, rt.data_ptr(), stride, 0, int(packed),
                 ct.data_ptr(), lib.stream(rt))
        return ct.cpu().numpy()

    for n, packed in [(n, True) for n in range(1, 9)] + [(n, False) for n in
                                                         (9, 33, 64, 129, 256)]:
        B = 12 if packed else 1
        Rs = np.triu(rng.standard_normal((B, n, n)))
        for b in range(B):
            # diagonals positive, 2^-8 .. 2^8: condition numbers up to ~1e6
            Rs[b][np.diag_indices(n)] = np.ldexp(rng.uniform(1, 2, n), rng.integers(-8, 9, n))
        got = cov(Rs, packed)
        worst = 0.0
        for b in range(B):
            Cs = exact_cov(Rs[b])
            Ri = np.linalg.inv(Rs[b])
            err_np = np.abs(Ri @ Ri.T - Cs).max()
            err = np.abs(got[b] - Cs).max()
            gate = 4 * err_np + 4 * n * U * np.abs(Cs).max()
            worst = max(worst, err / gate)
            assert err <= gate, (n, packed, b, err, gate)
        out[(n, packed)] = round(worst, 3)
        if n >= 2 and n <= 9:
            # the singular threshold: pivot == 16 n eps dmax -> NaN
            Rd = np.eye(n)[None].repeat(2, axis=0)
            t = 16.0 * n * 2.220446049250313e-16 * 1.0
            Rd[0, n - 1, n - 1] = t
            Rd[1, n - 1, n - 1] = np.nextafter(t, np.inf)
            c = cov(Rd, packed)
            assert np.isnan(c[0]).all() and np.isfinite(c[1]).all(), (n, packed)
    print("covariance worst error / gate:", out)
    return out


def exact_cov(R):
    """R^-1 R^-T of a double upper-triangular R with a positive diagonal, in
    Python integers: R = Ri 2^-E exactly, X = round(2^K Ri^-1) by back
    substitution, C = 2^(2E - 2K) X X^T."""
    n = R.shape[0]
    E = int(53 - np.frexp(R[R != 0])[1].min())
    Ri = np.empty((n, n), dtype=object)
    for (i, j), v in np.ndenumerate(R):
        Ri[i, j] = int(np.ldexp(v, E))                  # exact: E covers the smallest ulp
    K = 400 + E
    S = 1 << K
    X = np.zeros((n, n), dtype=object)
    for i in range(n - 1, -1, -1):
        rhs = np.zeros(n - i, dtype=object)
        rhs[0] = S
        if i < n - 1:
            rhs = rhs - Ri[i, i + 1:] @ X[i + 1:, i:]
        d = Ri[i, i]
        X[i, i:] = [(2 * v + d) // (2 * d) for v in rhs]
    P = X @ X.T
    s = 2 * K - 2 * E
    return np.array([[v / (1 << s) for v in row] for row in P], dtype=np.float64)


# ------------------------------------------------------- GPU-only checks --

def check_misaligned_views(dev):
    """A callback that returns F and J carved out of one buffer (J starting at
    an 8-byte offset): the batched solve gives the bits of the aligned solve
    (n = 2, 4, 6, 8), the tall solve too, and a direct ABI call with such a J
    returns BLSQ_E_BADARG."""
    from bounded_lsq_b200 import least_squares, least_squares_batched, PerProblem, get_lib
    from bounded_lsq_b200._lib import BlsqError
    lib = get_lib()
    rng = np.random.default_rng(4)
    A, m = 37, 9                                        # A m odd: J is 8 bytes off
    for n in (2, 4, 6, 8):
        Dm = torch.as_tensor(rng.standard_normal((m, n)), device=dev)
        Y = torch.as_tensor(rng.standard_normal((A, m)), device=dev)

        def fun(X, y):
            return torch.sin(X) @ Dm.T - y

        def jac(X, y):
            return torch.cos(X)[:, None, :] * Dm[None]

        def fun_v(X, y):
            k = X.shape[0]
            buf = torch.empty(k * m + k * m * n + 8, dtype=torch.float64, device=dev)
            F = buf[1:1 + k * m].view(k, m)
            F.copy_(fun(X, y))
            return F

        def jac_v(X, y):
            k = X.shape[0]
            buf = torch.empty(k * m + k * m * n + 8, dtype=torch.float64, device=dev)
            s = k * m + 1 + (k * m) % 2                # an odd number of doubles in
            Jv = buf[s:s + k * m * n].view(k, m, n)
            assert Jv.data_ptr() % 16 == 8
            Jv.copy_(jac(X, y))
            return Jv
        X0 = torch.zeros((A, n), dtype=torch.float64, device=dev)
        args = (PerProblem(Y),)
        r0 = least_squares_batched(fun, X0, jac=jac, args=args)
        r1 = least_squares_batched(fun_v, X0, jac=jac_v, args=args)
        for f in ("x", "obj_value", "status", "nfev"):
            assert same_bits(getattr(r0, f).cpu().numpy(), getattr(r1, f).cpu().numpy()), (n, f)
        # the ABI refuses the misaligned J before any launch
        ist = torch.full((A, 8), -1, dtype=torch.int32, device=dev)
        lin = torch.zeros((A, lib.lin_record_size(n)), dtype=torch.float64, device=dev)
        buf = torch.zeros(A * m * n + 8, dtype=torch.float64, device=dev)
        Fz = torch.zeros((A, m), dtype=torch.float64, device=dev)
        for off in ((1, 2, 3) if n % 4 == 0 else (1,)):
            with pytest.raises(BlsqError, match="invalid argument"):
                lib.call("blsq_linearise_batched", A, None, m, n, Fz.data_ptr(),
                         buf[off:].data_ptr(), None, None, 0, ist.data_ptr(),
                         lin.data_ptr(), lib.stream(ist))
        torch.cuda.synchronize()
    # tall mode: f and J views 8 bytes off an aligned allocation
    mt, nt = 600, 12
    Dt = torch.as_tensor(rng.standard_normal((mt, nt)), device=dev)
    yt = torch.as_tensor(rng.standard_normal(mt), device=dev)

    def tfun(x):
        return torch.sin(x) @ Dt.T - yt

    def tjac(x):
        return Dt * torch.cos(x)[None, :]

    def tfun_v(x):
        buf = torch.empty(mt + 2, dtype=torch.float64, device=dev)
        buf[1:1 + mt] = tfun(x)
        return buf[1:1 + mt]

    def tjac_v(x):
        buf = torch.empty(mt * nt + 2, dtype=torch.float64, device=dev)
        Jv = buf[1:1 + mt * nt].view(mt, nt)
        Jv.copy_(tjac(x))
        return Jv
    x0 = torch.full((nt,), 0.1, dtype=torch.float64, device=dev)
    t0 = least_squares(tfun, x0, jac=tjac)
    t1 = least_squares(tfun_v, x0, jac=tjac_v)
    assert same_bits(t0.x.cpu().numpy(), t1.x.cpu().numpy())
    assert t0.nfev == t1.nfev and t0.status == t1.status


def check_64bit_indexing(lib, dev):
    """N = 8, m = 257 (MULTI, 256-bit loads) with A m N > 2^31 elements: the
    records of the first and last 64 slots against the reference."""
    N, m = 8, 257
    A = (1 << 31) // (m * N) + 5000
    assert A * m * N > 2 ** 31
    need = (A * m * (N + 1) + A * lib.lin_record_size(N)) * 8 + A * 32
    if torch.cuda.mem_get_info(dev)[0] < max(need + (2 << 30), 24 << 30):
        pytest.skip("needs 24 GB of free device memory")
    g = torch.Generator(device=dev)
    g.manual_seed(8)
    try:
        # in place: one 17 GB tensor, not two
        J = torch.rand((A, m, N), dtype=torch.float64, device=dev, generator=g).add_(0.5)
        F = torch.rand((A, m), dtype=torch.float64, device=dev, generator=g).sub_(1.5)
        ist = torch.zeros((A, 8), dtype=torch.int32, device=dev)
        ist[:, 0] = -1
        LS = lib.lin_record_size(N)
        lin = torch.zeros((A, LS), dtype=torch.float64, device=dev)
        lib.call("blsq_linearise_batched", A, None, m, N, F.data_ptr(), J.data_ptr(),
                 None, None, 0, ist.data_ptr(), lin.data_ptr(), lib.stream(ist))
        sel = list(range(64)) + list(range(A - 64, A))
        Jh, Fh, rec = J[sel].cpu().numpy(), F[sel].cpu().numpy(), lin[sel].cpu().numpy()
    finally:
        J = F = ist = lin = None
        torch.cuda.empty_cache()
    stats, fails = {}, []
    for b in range(len(sel)):
        gate_record(rec[b], N, m, 32, reference(Jh[b], Fh[b]), "random", stats, fails,
                    "64-bit")
    print("64-bit indexing, A =", A, stats)
    assert not fails, fails[:3]


# ------------------------------------------------------------------ tests --

CPU = torch.device("cpu")
CHECKS = [check_all_instances_launched, check_power_of_two_scaling, check_scale_range,
          check_covariance]


@pytest.fixture(scope="module")
def cuda_lib():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from bounded_lsq_b200 import get_lib
    return get_lib()


@pytest.mark.parametrize("check", CHECKS, ids=lambda c: c.__name__[6:])
def test_hostemul(check):
    print(check(hostemul.get(), CPU))


@pytest.mark.gpu
@pytest.mark.parametrize("check", CHECKS, ids=lambda c: c.__name__[6:])
def test_gpu(cuda_lib, check):
    print(check(cuda_lib, torch.device("cuda:0")))


@pytest.mark.gpu
def test_gpu_misaligned_views(cuda_lib):
    check_misaligned_views(torch.device("cuda:0"))


@pytest.mark.gpu
def test_gpu_64bit_indexing(cuda_lib):
    check_64bit_indexing(cuda_lib, torch.device("cuda:0"))
