"""CPU "CG+AMG" solver of the oracle -- TEST / BASELINE INFRASTRUCTURE ONLY.

The reference's iterative path is  Krylov.cg(G, b; M = aspreconditioner(
smoothed_aggregation(G; coarse_solver = Pinv, presmoother = GaussSeidel(),
postsmoother = GaussSeidel())), rtol = 1e-6, itmax = 100_000)  (src/core.jl:164-167,
639).  Krylov.jl 0.10 and AlgebraicMultigrid.jl 1.2 are registry packages that are
NOT vendored under /root/reference (Project.toml:25,32; no Manifest), so this file
restates their *published* algorithms (Vanek-Mandel-Brezina smoothed aggregation as
implemented by PyAMG/AlgebraicMultigrid.jl: symmetric strength theta = 0, standard
aggregation, constant near-null-space candidate, Jacobi prolongation smoothing
omega = 4/3, symmetric Gauss-Seidel pre/post smoothing, pseudo-inverse coarse
solve, V-cycle; textbook preconditioned CG with Krylov.jl's stop test
sqrt(r'z) <= atol + rtol*sqrt(r0'z0), atol = sqrt(eps)).
Parity status: pinned at the *solution* level (it must reproduce the same golden
vectors as the direct oracle: tests/test_oracle_golden.py::test_cg_amg_*);
unpinned at the AMG-internals level (hierarchy shapes / iteration counts are not
asserted by any reference test).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import scipy.sparse as sp

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_ref", "liboracle_amg.so")
_lib = None


_SRC = os.path.join(_HERE, "csrc", "amg_kernels.c")


def _stale(so):
    return not os.path.isfile(so) or os.path.getmtime(so) < os.path.getmtime(_SRC)


def build(force=False, so=_SO):
    """gcc -O3 the sequential kernels into `so` (called by __graft_entry__.build())."""
    os.makedirs(os.path.dirname(so), exist_ok=True)
    if force or _stale(so):
        import subprocess
        subprocess.check_call(["gcc", "-O3", "-march=x86-64-v2", "-shared", "-fPIC", "-o", so, _SRC])
    return so


def _load():
    global _lib
    if _lib is None:
        so = _SO
        if _stale(so):      # not built or out of date: compile a private copy, the source tree may be read-only
            import tempfile
            so = build(so=os.path.join(tempfile.mkdtemp(prefix="oracle_amg_"), "liboracle_amg.so"))
        lib = C.CDLL(so)
        i32p, f64p = C.POINTER(C.c_int32), C.POINTER(C.c_double)
        lib.csr_matvec.argtypes = [C.c_int64, i32p, i32p, f64p, f64p, f64p]
        lib.gauss_seidel.argtypes = [C.c_int64, i32p, i32p, f64p, f64p, f64p, C.c_int]
        lib.standard_aggregation.argtypes = [C.c_int64, i32p, i32p, i32p]
        lib.standard_aggregation.restype = C.c_int64
        _lib = lib
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class Level:
    def __init__(self, A):
        A = sp.csr_matrix(A, dtype=np.float64)
        A.sort_indices()
        self.A = A
        self.ip = np.ascontiguousarray(A.indptr, dtype=np.int32)
        self.ix = np.ascontiguousarray(A.indices, dtype=np.int32)
        self.a = np.ascontiguousarray(A.data, dtype=np.float64)
        self.n = A.shape[0]
        self.P = None
        self.R = None

    def matvec(self, x):
        y = np.empty(self.n)
        _load().csr_matvec(self.n, _p(self.ip, C.c_int32), _p(self.ix, C.c_int32), _p(self.a, C.c_double),
                           _p(x, C.c_double), _p(y, C.c_double))
        return y

    def gs(self, x, b, direction):
        _load().gauss_seidel(self.n, _p(self.ip, C.c_int32), _p(self.ix, C.c_int32), _p(self.a, C.c_double),
                             _p(x, C.c_double), _p(b, C.c_double), direction)


class MultiLevel:
    def __init__(self, levels, coarse_pinv):
        self.levels = levels
        self.coarse_pinv = coarse_pinv

    def operator_complexity(self):
        return sum(l.A.nnz for l in self.levels) / self.levels[0].A.nnz


def _spectral_radius_DinvA(A, iters=15, seed=0):
    """power iteration estimate of rho(D^-1 A) (PyAMG uses a short Arnoldi run)."""
    d = A.diagonal()
    dinv = np.where(d != 0, 1.0 / np.where(d != 0, d, 1.0), 0.0)
    x = np.random.default_rng(seed).random(A.shape[0])
    lam = 1.0
    for _ in range(iters):
        y = dinv * (A @ x)
        lam = np.linalg.norm(y)
        if lam == 0:
            return 1.0
        x = y / lam
    return lam


def smoothed_aggregation(A, max_levels=10, max_coarse=10, omega=4.0 / 3.0):
    lib = _load()
    levels = [Level(A)]
    while len(levels) < max_levels and levels[-1].n > max_coarse:
        lvl = levels[-1]
        Acsr = lvl.A
        n = lvl.n
        # strength: symmetric, theta = 0 -> every off-diagonal nonzero entry
        S = Acsr.copy()
        S.data = (S.data != 0).astype(np.float64)
        S.setdiag(0)
        S.eliminate_zeros()
        S.sort_indices()
        agg = np.empty(n, dtype=np.int32)
        nagg = lib.standard_aggregation(n, _p(np.ascontiguousarray(S.indptr, dtype=np.int32), C.c_int32),
                                        _p(np.ascontiguousarray(S.indices, dtype=np.int32), C.c_int32),
                                        _p(agg, C.c_int32))
        if nagg == 0 or nagg >= n:
            break
        keep = agg >= 0
        rows = np.nonzero(keep)[0]
        counts = np.bincount(agg[keep], minlength=nagg).astype(np.float64)
        T = sp.csr_matrix((1.0 / np.sqrt(counts[agg[keep]]), (rows, agg[keep])), shape=(n, nagg))
        d = Acsr.diagonal()
        dinv = np.where(d != 0, 1.0 / np.where(d != 0, d, 1.0), 0.0)
        rho = _spectral_radius_DinvA(Acsr)
        P = (T - (omega / rho) * (sp.diags(dinv) @ (Acsr @ T))).tocsr()
        R = P.T.tocsr()
        Ac = (R @ Acsr @ P).tocsr()
        lvl.P, lvl.R = P, R
        levels.append(Level(Ac))
    coarse = np.linalg.pinv(levels[-1].A.toarray())
    return MultiLevel(levels, coarse)


def vcycle(ml, b, lvl=0):
    """one V(1,1) cycle with symmetric Gauss-Seidel, zero initial guess."""
    L = ml.levels[lvl]
    if lvl == len(ml.levels) - 1:
        return ml.coarse_pinv @ b
    x = np.zeros(L.n)
    L.gs(x, b, +1); L.gs(x, b, -1)                       # presmoother (symmetric sweep)
    r = b - L.matvec(x)
    xc = vcycle(ml, np.ascontiguousarray(L.R @ r), lvl + 1)
    x += L.P @ xc
    L.gs(x, b, +1); L.gs(x, b, -1)                       # postsmoother
    return x


def pcg(A, b, ml, rtol=1e-6, atol=None, itmax=100_000, x0=None):
    """Preconditioned CG with Krylov.jl's `cg` stop rule.  Returns (x, iterations)."""
    # the hierarchy may have been built on a (regularised) copy: the operator applied is always A
    top = ml.levels[0] if (ml is not None and A is ml.levels[0].A) else Level(A)
    if atol is None:
        atol = np.sqrt(np.finfo(np.float64).eps)
    n = len(b)
    x = np.zeros(n)
    r = np.array(b, dtype=np.float64)
    z = vcycle(ml, r) if ml is not None else r.copy()
    p = z.copy()
    gamma = float(r @ z)
    rnorm = np.sqrt(abs(gamma))
    eps = atol + rtol * rnorm
    it = 0
    while rnorm > eps and it < itmax:
        Ap = top.matvec(p)
        pAp = float(p @ Ap)
        if pAp <= 0:
            break
        alpha = gamma / pAp
        x += alpha * p
        r -= alpha * Ap
        z = vcycle(ml, r) if ml is not None else r.copy()
        gnew = float(r @ z)
        beta = gnew / gamma
        gamma = gnew
        p = z + beta * p
        rnorm = np.sqrt(abs(gamma))
        it += 1
    return x, it
