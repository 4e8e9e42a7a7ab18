"""Host-side mirror of the reference's solver interface for the enumeration path.

``Canonical`` keeps the reference's getter names (reference:
src/ProblemTypes/Canonical.h:10-49, Canonical.cpp:126-154) and constructor
validation (Canonical.cpp:27-46); ``EnumerationSolver`` has the call shape of
the reference's ``Solver`` (src/SimplexSolover.h:285-288): construct from a
Canonical, ``solve()`` returns the first ``GetOriginalVariablesCount()``
components of the optimal x (SimplexSolover.h:435-439) and raises
``RuntimeError`` when the LP has no feasible basis (cf. SimplexSolover.h:371).

All numerical work happens in libenumgpu (CUDA, sm_100a) behind the C ABI of
include/enumgpu.h; this module only marshals buffers.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Optional, Sequence

import numpy as np

from . import _abi
from ._lib import EnumGpuError, last_error, lib


class Canonical:
    """min/max c'x, Ax = b, x >= 0 with a designated basis (reference Canonical)."""

    def __init__(self, A, b, c, basisIndices: Sequence[int], minimize: bool = True):
        A = np.asarray(A, dtype=np.float64)
        b = np.asarray(b, dtype=np.float64).reshape(-1)
        c = np.asarray(c, dtype=np.float64).reshape(-1)
        if A.ndim != 2:
            raise ValueError("A must be a matrix")
        # same checks, same order, as Canonical.cpp:27-46
        if A.shape[0] != b.size:
            raise ValueError("dimensions of A and b do not match")
        if A.shape[1] != c.size:
            raise ValueError("dimensions of A and c do not match")
        if len(basisIndices) != A.shape[0]:
            raise ValueError("number of basis indices differs from the number of rows of A")
        for idx in basisIndices:
            if idx < 0 or idx >= A.shape[1]:
                raise ValueError("basis index out of range")
        self._A = np.asfortranarray(A)          # Eigen default storage: column-major
        self._b = np.ascontiguousarray(b)
        self._c = np.ascontiguousarray(c)
        self._basis = [int(i) for i in basisIndices]
        self._minimize = bool(minimize)
        self._n_orig = int(c.size)              # Canonical.cpp:25

    # -- reference getters (Canonical.cpp:126-154) -------------------------
    def GetConstraintsMatrix(self): return self._A
    def GetRightHandSide(self): return self._b
    def GetObjectiveCoefficients(self): return self._c
    def IsMaximization(self): return not self._minimize
    def GetBasisIndices(self): return self._basis
    def GetOriginalVariablesCount(self): return self._n_orig

    def SetOriginalVariablesCount(self, count: int):
        if count <= 0 or count > self._c.size:      # Canonical.cpp:156-163
            raise ValueError("invalid number of original variables")
        self._n_orig = int(count)

    def Evaluate(self, solution) -> float:
        x = np.asarray(solution, dtype=np.float64).reshape(-1)
        if x.size != self._c.size:                  # Canonical.cpp:81-84
            raise ValueError("solution size differs from the number of variables")
        return float(self._c @ x)


    def GetDual(self) -> "Canonical":
        """Canonical form of the dual, built like the reference (Canonical.cpp:305-364):
        variables y = y' - y'' and one slack per dual row: A_d = [A' | -A' | I] (n x (2m+n)),
        b_d = c, c_d = [b | -b | 0], slack basis, opposite sense, 2m original variables.
        (Like the reference's, the construction is the dual of a MIN primal.)"""
        m, n = self._A.shape
        Ad = np.zeros((n, 2 * m + n), order="F")
        Ad[:, :m] = self._A.T
        Ad[:, m:2 * m] = -self._A.T
        Ad[:, 2 * m:] = np.eye(n)
        cd = np.concatenate([self._b, -self._b, np.zeros(n)])
        dual = Canonical(Ad, self._c.copy(), cd, [2 * m + i for i in range(n)], minimize=not self._minimize)
        dual.SetOriginalVariablesCount(2 * m)
        return dual

    # -- back to the other forms, original variables only (Canonical.cpp:199-303) --
    def ToCommon(self):
        """Rows stay equalities, variables >= 0 (reference Canonical.cpp:199-228)."""
        from .problem_types import Common, ConstraintType, VariableType
        m, n = self._A.shape[0], self._n_orig
        return Common(self._A[:, :n], self._b, self._c[:n], [ConstraintType.Equal] * m, [VariableType.NonNegative] * n,
                      not self._minimize)

    def ToSymmetrical(self):
        """Each equality becomes the pair (row, -row) with the sense's inequality (reference Canonical.cpp:230-303)."""
        from .problem_types import Symmetrical
        m, n = self._A.shape[0], self._n_orig
        A = np.empty((2 * m, n))
        A[0::2] = self._A[:, :n]
        A[1::2] = -self._A[:, :n]
        b = np.empty(2 * m)
        b[0::2] = self._b
        b[1::2] = -self._b
        return Symmetrical(A, b, self._c[:n], not self._minimize)

    def PrintText(self) -> str:
        """The text the reference's Canonical::Print() writes (Canonical.cpp:88-123)."""
        from .problem_types import _lp_text
        return _lp_text("=== Каноническая форма задачи ЛП ===", not self._minimize, self._A, self._b, self._c,
                        "При ограничениях (Ax = b):", "*", lambda i: " = ") + \
            "\nВсе переменные неотрицательны: x_i >= 0\n\nБазисные переменные: " + \
            ", ".join(f"x{j + 1}" for j in self._basis) + \
            f"\nКоличество исходных переменных: {self._n_orig}\nДополнительных переменных: {self._c.size - self._n_orig}\n"

    def Print(self):
        print(self.PrintText(), end="")

    # -- per-basis numerics: on the GPU, through enumgpu_eval_basis ---------
    def _eval_designated(self):
        ps = _problem_struct(self._A, self._b, self._c, not self._minimize)
        m = self._A.shape[0]
        basis = (C.c_int32 * m)(*self._basis)
        x = (C.c_double * m)()
        z, cls = C.c_double(), C.c_int32()
        _check(lib().enumgpu_eval_basis(C.byref(ps), None, basis, x, C.byref(z), C.byref(cls)))
        return cls.value, list(x), z.value

    def GetBasicSolution(self):
        """x (length n) of the designated basis (reference Canonical.cpp:179-197), for a Canonical of any size and
        any index list the constructor accepted.  One documented deviation: the reference's QR solve returns
        *some* vector for a singular basis without signalling; here a singular basis (repeated indices included)
        raises RuntimeError("Singular basis matrix"), the convention of the reference's other per-basis solve
        (Solver::computeBFS, SimplexSolover.h:124-126).  IsFeasibleBasis() never raises: singular -> False."""
        cls, xB, _ = self._eval_designated()
        if cls == 2:
            raise RuntimeError("Singular basis matrix")
        x = np.zeros(self._c.size)
        for j, v in zip(self._basis, xB):
            x[j] = v
        return x

    def IsFeasibleBasis(self) -> bool:
        """All basic values >= -1e-9 (reference Canonical.cpp:165-177)."""
        return self._eval_designated()[0] == 0


def _problem_struct(A, b, c, maximize):
    m, n = A.shape
    return _abi.Problem(m, n, A.strides[1] // 8 if n > 1 else m, int(bool(maximize)),
                        A.ctypes.data, b.ctypes.data, c.ctypes.data)


def _check(rc: int):
    if rc == _abi.ERR_CUDA:
        raise EnumGpuError(last_error())
    if rc in (_abi.ERR_ARG, _abi.ERR_RANGE, _abi.ERR_NONFINITE):
        raise ValueError(last_error())


class CostRanges(NamedTuple):
    """Cost ranging of EnumerationSolver.costRanges(): for each canonical column j, c_j can fall by decrease[j] or
    rise by increase[j] (np.inf: without limit) and the optimal vertex stays optimal.  *_rank[j] is the basis that
    takes over at that end (UINT64_MAX: none); where *_ray[j] is True it is an extreme ray, a rank among the
    C(n, m+1) bases of the auxiliary LP.  status is CERT_OPTIMAL (exact) or CERT_UNDECIDED (m = 16: no rays
    enumerated; the ranges on the side rays can limit are upper bounds)."""
    status: int
    decrease: np.ndarray
    increase: np.ndarray
    decrease_rank: np.ndarray
    increase_rank: np.ndarray
    decrease_ray: np.ndarray
    increase_ray: np.ndarray
    n_vertex_bases: int
    n_ray_bases: int
    kernel_ms: float


class RhsRanges(NamedTuple):
    """Right-hand-side ranging of EnumerationSolver.rhsRanges(): for each row i, b_i can fall by decrease[i] or rise
    by increase[i] (np.inf: without limit) and the dual values stay optimal; over that interval the objective is
    objective + delta * shadow_price[i].  *_rank[i] is the basis (a rank among the C(n, m) bases) that attains the
    limit (UINT64_MAX: none).  tight: the columns whose reduced cost is tight at the duals, the basis included;
    n_bases = C(len(tight), m) bases were looked at, n_singular of them singular.  status is CERT_OPTIMAL, or
    CERT_BOUNDED / CERT_UNDECIDED when no dual-feasible basis was found (every range NaN)."""
    status: int
    shadow_price: np.ndarray
    decrease: np.ndarray
    increase: np.ndarray
    decrease_rank: np.ndarray
    increase_rank: np.ndarray
    tight: list
    n_bases: int
    n_singular: int
    kernel_ms: float


class EnumerationSolver:
    """Solve a Canonical LP by enumerating all C(n, m) bases on the GPU(s).

    >>> x = EnumerationSolver(canonical).solve()          # like Solver(problem).solve()
    """

    def __init__(self, problem: Canonical, devices: Optional[Sequence[int]] = None,
                 algo: int = _abi.ALGO_AUTO, eps_feas: float = 1e-9, eps_piv: float = -1.0,
                 pivot_rule: int = _abi.PIVOT_ABSOLUTE, check_unbounded: bool = False, optimal_duals: bool = False):
        """check_unbounded: solve() certifies the enumeration's optimum (certify()) and raises
        RuntimeError("objective is unbounded") on an unbounded LP, as the reference's Solver does
        (SimplexSolover.h:443).  Off by default: enumerating vertices alone cannot see unboundedness.
        optimal_duals: certify() (and dualValues, reducedCosts, unboundedRay, check_unbounded) searches all optimal
        bases for a dual-feasible one when the winner's certificate is undecided (enumgpu_certify_optimum); the
        certificate then belongs to certificateBasis(), which may differ from optimalBasis().  Off by default: it
        costs one more enumeration on a degenerate optimum."""
        A = problem.GetConstraintsMatrix()
        m, n = A.shape
        if m > n:
            raise ValueError(f"m={m} > n={n}: no basis exists")
        if m > _abi.MAX_M or n > _abi.MAX_N:
            raise ValueError(f"(m,n)=({m},{n}) above the library limits ({_abi.MAX_M},{_abi.MAX_N})")
        self._problem = problem                      # reference copies (SimplexSolover.h:12,285); arrays are not mutated here
        self._devices = None if devices is None else [int(d) for d in devices]
        self._algo = int(algo)
        self._eps = (float(eps_feas), float(eps_piv))      # eps_piv < 0: the rule's default (1e-9 absolute, m*2^-52 relative)
        self._rule = int(pivot_rule)
        self._check_unbounded = bool(check_unbounded)
        self._optimal_duals = bool(optimal_duals)
        self._res: Optional[_abi.Result] = None
        self._cert: Optional[_abi.Certificate] = None
        self._cert_basis: Optional[list] = None
        self._handles = None                         # enumgpu_handle per device, created at the first solve, kept

    # -- handles: stream, events, pinned staging, device buffers live as long as the solver (include/enumgpu.h) --
    def _get_handles(self):
        if self._handles is None:
            hs = []
            try:
                for d in (self._devices if self._devices else [-1]):
                    h = C.c_void_p()
                    _check(lib().enumgpu_create(int(d), C.byref(h)))
                    hs.append(h)
            except BaseException:
                for h in hs:
                    lib().enumgpu_destroy(h)
                raise
            self._handles = hs
        return self._handles

    def close(self):
        if self._handles:
            for h in self._handles:
                lib().enumgpu_destroy(h)
        self._handles = None

    def __del__(self):
        try:
            self.close()
        except Exception:            # interpreter shutdown
            pass

    def _options(self, rank_begin=0, rank_end=0, shard_index=0, shard_count=0):
        return _abi.Options(self._eps[0], self._eps[1], rank_begin, rank_end, 0, self._algo, None, None,
                            shard_index, shard_count, self._rule, 0)

    # -- the reference call shape ------------------------------------------
    def solve(self, rank_begin: int = 0, rank_end: int = 0) -> np.ndarray:
        p = self._problem
        if self._check_unbounded and (rank_begin, rank_end) != (0, 0):
            m, n = p.GetConstraintsMatrix().shape
            if (rank_begin, rank_end) != (0, lib().enumgpu_binomial(n, m)):
                raise ValueError("check_unbounded needs the whole rank range: its conclusion rests on the global optimum")
        res = self.enumerate(rank_begin, rank_end)
        if res.status == _abi.NO_FEASIBLE:
            raise RuntimeError("the problem has no feasible basic solution")
        if self._check_unbounded and self.certify().status == _abi.CERT_UNBOUNDED:
            raise RuntimeError("objective is unbounded")
        x = np.zeros(p.GetObjectiveCoefficients().size)
        for i in range(res.m):
            x[res.basis[i]] = res.x_B[i]
        return x[: p.GetOriginalVariablesCount()].copy()

    def enumerate(self, rank_begin: int = 0, rank_end: int = 0, shard_index: int = 0, shard_count: int = 0) -> _abi.Result:
        """Run the enumeration and return the raw result struct (no exception on NO_FEASIBLE).

        shard_index/shard_count select the interleaved rank windows of one shard
        (one process per GPU); the partial results merge with enumgpu_merge_partial."""
        p = self._problem
        A, b, c = p.GetConstraintsMatrix(), p.GetRightHandSide(), p.GetObjectiveCoefficients()
        ps = _problem_struct(A, b, c, p.IsMaximization())
        o = self._options(rank_begin, rank_end, shard_index, shard_count)
        res = _abi.Result()
        if lib().enumgpu_device_count() < 1:          # no device: let the library say so (no CPU fallback)
            _check(lib().enumgpu_solve(C.byref(ps), C.byref(o), C.byref(res)))
        hs = self._get_handles()
        arr = (C.c_void_p * len(hs))(*[h.value for h in hs])
        rc = lib().enumgpu_solve_hv(arr, len(hs), C.byref(ps), C.byref(o), C.byref(res))
        _check(rc)
        self._res = res
        self._cert = self._cert_basis = None
        return res

    # -- many cost vectors over one feasible set (enumgpu_solve_objectives) ----------------------
    def enumerateObjectives(self, costs, rank_begin: int = 0, rank_end: int = 0, max_list: int = 0):
        """The raw result structs of every cost vector, from one enumeration: costs is a (k, n) array whose rows are
        cost vectors (the problem's own sense for all of them; the problem's c is not used).  Entry i is what
        enumerate() returns for the problem with c = costs[i], bit for bit; kernel_ms and n_launches describe the
        whole call.  Runs on the current CUDA device.  max_list: feasible ranks held on the device (0 = 2^26)."""
        p = self._problem
        A = p.GetConstraintsMatrix()
        n = A.shape[1]
        costs = np.ascontiguousarray(np.asarray(costs, dtype=np.float64))   # C-contiguous (k, n) = column-major n x k
        if costs.ndim != 2 or costs.shape[1] != n:
            raise ValueError(f"costs must be a (k, {n}) array, one cost vector per row; got shape {costs.shape}")
        k = costs.shape[0]
        ps = _problem_struct(A, p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        out = (_abi.Result * max(k, 1))()
        _check(lib().enumgpu_solve_objectives(C.byref(ps), C.byref(self._options(rank_begin, rank_end)), k,
                                              costs.ctypes.data_as(C.POINTER(C.c_double)), n, int(max_list), out))
        return [out[i] for i in range(k)]

    def solveObjectives(self, costs, rank_begin: int = 0, rank_end: int = 0) -> np.ndarray:
        """solve() for every row of costs (a (k, n) array of cost vectors) with one enumeration: row i of the
        (k, GetOriginalVariablesCount()) result is what solve() returns with c = costs[i].  Raises RuntimeError if
        some cost vector has no optimum (no feasible basis), as solve() does."""
        res = self.enumerateObjectives(costs, rank_begin, rank_end)
        n = self._problem.GetObjectiveCoefficients().size
        X = np.zeros((len(res), n))
        for i, r in enumerate(res):
            if r.status == _abi.NO_FEASIBLE:
                raise RuntimeError("the problem has no feasible basic solution")
            X[i, list(r.basis)[:r.m]] = list(r.x_B)[:r.m]
        return X[:, : self._problem.GetOriginalVariablesCount()].copy()

    # -- certificate of the optimum: duals, reduced costs, unboundedness (enumgpu_certify) --------
    def _device_options(self):
        """Options for the handle-free entries: the solver's device list, tolerances, kernel and rule."""
        o = self._options()
        if self._devices:
            self._dev_arr = (C.c_int32 * len(self._devices))(*self._devices)
            o.n_devices, o.devices = len(self._devices), self._dev_arr
        return o

    def certify(self, eps_opt: float = 1e-9) -> _abi.Certificate:
        """Certificate of the last enumeration's optimal basis (enumerates first if nothing has been).
        .status is CERT_OPTIMAL (y dual feasible), CERT_BOUNDED (degenerate vertex: no ray exists, y not dual
        feasible), CERT_UNBOUNDED (.ray is a ray) or CERT_UNDECIDED (degenerate vertex at m = 16).
        With optimal_duals the certificate is that of the lowest-rank dual-feasible optimal basis when the winner's is
        undecided and one exists (enumgpu_certify_optimum); certificateBasis() names its basis."""
        res = self._res if self._res is not None else self.enumerate()
        if res.status != _abi.OK:
            raise RuntimeError("the problem has no feasible basic solution")
        p = self._problem
        ps = _problem_struct(p.GetConstraintsMatrix(), p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        if self._optimal_duals:
            opt = _abi.Optimum()
            _check(lib().enumgpu_certify_optimum(C.byref(ps), C.byref(self._device_options()), C.byref(res), float(eps_opt),
                                                 0, C.byref(opt)))
            cert, basis = opt.cert, list(opt.basis)[:res.m]
        else:
            basis = list(res.basis)[:res.m]
            cert = _abi.Certificate()
            _check(lib().enumgpu_certify(C.byref(ps), C.byref(self._device_options()), (C.c_int32 * res.m)(*basis),
                                         float(eps_opt), C.byref(cert)))
        self._cert, self._cert_basis = cert, [int(j) for j in basis]
        return cert

    def costRanges(self, eps_opt: float = 1e-9, max_list: int = 0) -> CostRanges:
        """Cost ranging of the optimum (enumgpu_cost_ranges): how far each c_j can move, all else fixed, before the
        optimal vertex stops being optimal, exact at degenerate vertices (every feasible basis and every extreme ray
        is looked at).  Enumerates first if nothing has been.  Runs on the current CUDA device.  Raises
        RuntimeError("objective is unbounded") on an unbounded LP.  max_list: ranks held on the device (0 = 2^26)."""
        res = self._res if self._res is not None else self.enumerate()
        if res.status != _abi.OK:
            raise RuntimeError("the problem has no feasible basic solution")
        p = self._problem
        ps = _problem_struct(p.GetConstraintsMatrix(), p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        out = _abi.Ranging()
        _check(lib().enumgpu_cost_ranges(C.byref(ps), C.byref(self._options()), C.byref(res), float(eps_opt), int(max_list),
                                         C.byref(out)))
        if out.status == _abi.CERT_UNBOUNDED:
            raise RuntimeError("objective is unbounded")
        r = out.range[: out.n]
        return CostRanges(int(out.status),
                          np.array([v.decrease for v in r]), np.array([v.increase for v in r]),
                          np.array([v.decrease_rank for v in r], dtype=np.uint64),
                          np.array([v.increase_rank for v in r], dtype=np.uint64),
                          np.array([bool(v.decrease_ray) for v in r]), np.array([bool(v.increase_ray) for v in r]),
                          int(out.n_vertex_bases), int(out.n_ray_bases), float(out.kernel_ms))

    def rhsRanges(self, eps_opt: float = 1e-9) -> RhsRanges:
        """Right-hand-side ranging of the optimum (enumgpu_rhs_ranges): how far each b_i can move, all else fixed,
        while the dual values stay optimal, exact under dual degeneracy (every nonsingular basis of the tight columns
        is looked at, feasible at b or not).  The duals are those of a dual-feasible optimal basis
        (enumgpu_certify_optimum), whatever optimal_duals is set to.  Enumerates first if nothing has been.  Runs on
        the current CUDA device.  Raises RuntimeError("objective is unbounded") on an unbounded LP."""
        res = self._res if self._res is not None else self.enumerate()
        if res.status != _abi.OK:
            raise RuntimeError("the problem has no feasible basic solution")
        p = self._problem
        ps = _problem_struct(p.GetConstraintsMatrix(), p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        o = self._options()
        opt = _abi.Optimum()
        _check(lib().enumgpu_certify_optimum(C.byref(ps), C.byref(o), C.byref(res), float(eps_opt), 0, C.byref(opt)))
        if opt.cert.status == _abi.CERT_UNBOUNDED:
            raise RuntimeError("objective is unbounded")
        out = _abi.RhsRanging()
        _check(lib().enumgpu_rhs_ranges(C.byref(ps), C.byref(o), C.byref(opt), float(eps_opt), C.byref(out)))
        r = out.range[: out.m]
        return RhsRanges(int(out.status), np.array([v.shadow_price for v in r]),
                         np.array([v.decrease for v in r]), np.array([v.increase for v in r]),
                         np.array([v.decrease_rank for v in r], dtype=np.uint64),
                         np.array([v.increase_rank for v in r], dtype=np.uint64),
                         [int(j) for j in out.tight[: out.n_tight]], int(out.n_bases), int(out.n_singular),
                         float(out.kernel_ms))

    def certificateBasis(self):
        """The columns (ascending) of the basis the certificate belongs to: the enumeration's optimal basis, or with
        optimal_duals the dual-feasible optimal basis certify() found."""
        self._need_cert()
        return list(self._cert_basis)

    def optimalBases(self, capacity: int = 1 << 22, eps_opt: float = 1e-9):
        """Ranks (ascending, uint64 array) of the optimal bases, at most `capacity` of them: the feasible bases whose
        key (the objective, negated when maximising) is at most key* + eps_opt * max(1, |key*|), key* the optimum's
        (enumgpu_list_window).  Enumerates first if nothing has been."""
        res = self._res if self._res is not None else self.enumerate()
        if res.status != _abi.OK:
            raise RuntimeError("the problem has no feasible basic solution")
        eps = 1e-9 if not eps_opt >= 0 else float(eps_opt) + 0.0      # as enumgpu_certify: < 0 the default, -0.0 is 0
        key_max = res.key + eps * max(1.0, abs(res.key))
        p = self._problem
        ps = _problem_struct(p.GetConstraintsMatrix(), p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        ranks = np.zeros(max(int(capacity), 1), dtype=np.uint64)
        n_listed = C.c_uint64()
        out = _abi.Result()
        _check(lib().enumgpu_list_window(C.byref(ps), C.byref(self._options()), key_max,
                                         ranks.ctypes.data_as(C.POINTER(C.c_uint64)), int(capacity), C.byref(n_listed),
                                         C.byref(out)))
        return ranks[: n_listed.value].copy()

    def findRay(self) -> _abi.Result:
        """enumgpu_find_ray: the extreme rays of {d >= 0, A d = 0} with c.d < 0 (> 0 when maximising), enumerated as
        the feasible bases of the auxiliary LP of include/enumgpu.h.  status OK: basis/x_B of the lowest-rank ray."""
        p = self._problem
        ps = _problem_struct(p.GetConstraintsMatrix(), p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        res = _abi.Result()
        _check(lib().enumgpu_find_ray(C.byref(ps), C.byref(self._device_options()), C.byref(res)))
        return res

    def _need_cert(self) -> _abi.Certificate:
        return self._cert if self._cert is not None else self.certify()

    def dualValues(self) -> np.ndarray:
        """y = B^-T c_B at the optimal basis (shadow prices, true sense)."""
        c = self._need_cert(); return np.array(c.y[: c.m])

    def reducedCosts(self) -> np.ndarray:
        """r_j = c_j - y.a_j for every column (true sense; ~0 on the basic ones)."""
        c = self._need_cert(); return np.array(c.reduced_cost[: c.n])

    def unboundedRay(self) -> Optional[np.ndarray]:
        """A ray d >= 0, A d = 0 along which the objective improves without bound, or None if the LP is bounded
        (or, at m = 16 on a degenerate vertex, undecided)."""
        c = self._need_cert()
        return np.array(c.ray[: c.n]) if c.status == _abi.CERT_UNBOUNDED else None

    # -- the extreme points themselves (README step 9 of the reference) -------
    def listFeasibleBases(self, capacity: int = 1 << 22):
        """Ranks (ascending, uint64 array) of the feasible bases, at most `capacity` of them; the result
        struct of the same enumeration is kept (feasibleCount() is the full count)."""
        p = self._problem
        ps = _problem_struct(p.GetConstraintsMatrix(), p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        o = self._options()
        ranks = np.zeros(max(int(capacity), 1), dtype=np.uint64)
        n_listed = C.c_uint64()
        res = _abi.Result()
        rc = lib().enumgpu_list_feasible(C.byref(ps), C.byref(o), ranks.ctypes.data_as(C.POINTER(C.c_uint64)),
                                         int(capacity), C.byref(n_listed), C.byref(res))
        _check(rc)
        self._res = res
        return ranks[: n_listed.value].copy()

    def evaluateBases(self, ranks):
        """(bases [k, m] int, x_B [k, m], objective [k], class [k]) of the bases with the given ranks, on the GPU."""
        p = self._problem
        A = p.GetConstraintsMatrix()
        m, n = A.shape
        ranks = np.ascontiguousarray(np.asarray(ranks, dtype=np.uint64))
        k = ranks.size
        xB = np.zeros((k, m)); z = np.zeros(k); cls = np.zeros(k, dtype=np.int32)
        ps = _problem_struct(A, p.GetRightHandSide(), p.GetObjectiveCoefficients(), p.IsMaximization())
        o = self._options()
        _check(lib().enumgpu_eval_ranks(C.byref(ps), C.byref(o), ranks.ctypes.data_as(C.POINTER(C.c_uint64)), k,
                                        xB.ctypes.data_as(C.POINTER(C.c_double)), z.ctypes.data_as(C.POINTER(C.c_double)),
                                        cls.ctypes.data_as(C.POINTER(C.c_int32))))
        bases = np.zeros((k, m), dtype=np.int32)
        buf = (C.c_int32 * m)()
        for i, r in enumerate(ranks):
            lib().enumgpu_unrank(n, m, int(r), buf)
            bases[i] = buf[:]
        return bases, xB, z, cls

    def feasibleVertices(self, capacity: int = 1 << 20, decimals: int = 9):
        """Distinct feasible vertices x (rows, length n) and their objective values: degenerate vertices are
        reached by several bases; rows are merged when they agree to `decimals` digits (host-side grouping)."""
        ranks = self.listFeasibleBases(capacity)
        bases, xB, z, _ = self.evaluateBases(ranks)
        n = self._problem.GetObjectiveCoefficients().size
        X = np.zeros((ranks.size, n))
        np.put_along_axis(X, bases.astype(np.int64), xB, axis=1)
        _, first = np.unique(np.round(X, decimals) + 0.0, axis=0, return_index=True)
        first.sort()
        return X[first], z[first]

    # -- accessors the parity metric needs (not in the reference) -----------
    def _need(self) -> _abi.Result:
        if self._res is None:
            raise RuntimeError("solve() has not been called")
        return self._res

    def optimalBasis(self): r = self._need(); return [int(r.basis[i]) for i in range(r.m)]
    def basicValues(self): r = self._need(); return [float(r.x_B[i]) for i in range(r.m)]
    def objective(self): return float(self._need().objective)
    def bestRank(self): return int(self._need().best_rank)
    def basesEvaluated(self): return int(self._need().n_bases)
    def singularCount(self): return int(self._need().n_singular)
    def infeasibleCount(self): return int(self._need().n_infeasible)
    def feasibleCount(self): return int(self._need().n_feasible)
    def kernelMilliseconds(self): return float(self._need().kernel_ms)
    def launches(self): return int(self._need().n_launches)
