"""Host-side mirror of the reference's ClpSimplex interface for the dual path.

Method names, argument meaning and status codes follow ClpSimplex / ClpModel
(/root/reference/src/ClpSimplex.hpp, ClpModel.hpp): ``loadProblem``, ``readMps``, ``dual``,
``status`` (0 optimal, 1 primal infeasible, 2 dual infeasible, 3 stopped, 4 errors),
``objectiveValue``, ``primalColumnSolution`` ... Everything computational happens behind the
C ABI of include/clp_b200.h in hand-written sm_100a CUDA; this module only marshals arrays.
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _capi
from ._capi import c_double_p, c_int_p, c_ubyte_p


class NoDeviceError(RuntimeError):
    pass


def _dp(a):
    return a.ctypes.data_as(c_double_p)


def _ip(a):
    return a.ctypes.data_as(c_int_p)


def _up(a):
    return a.ctypes.data_as(c_ubyte_p)




def denseInvert(a):
    """Inverse of a dense matrix by the refactorization kernels (blocked LU with partial
    pivoting + blocked substitution).  Returns (info, inverse)."""
    a = np.asfortranarray(a, dtype=np.float64)
    k = a.shape[0]
    x = np.zeros((k, k), dtype=np.float64, order="F")
    info = _capi.lib().Clpb_denseInvert(int(k), _dp(a), _dp(x))
    if info == _capi.NO_DEVICE:
        raise NoDeviceError("clp_b200 needs a CUDA device (no CPU fallback)")
    return info, x


class ClpSimplex:
    # ClpSimplex::Status (ClpSimplex.hpp:119-126)
    isFree, basic, atUpperBound, atLowerBound, superBasic, isFixed = range(6)

    def __init__(self):
        self._L = _capi.lib()
        self._h = self._L.Clpb_newModel()
        self._keep = None

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._L.Clpb_deleteModel(h)
            self._h = None

    # ---- ClpModel::loadProblem (column-major matrix without gaps) ----
    def loadProblem(self, numberColumns, numberRows, start, index, value, collb=None, colub=None,
                    obj=None, rowlb=None, rowub=None):
        c = lambda a, t: None if a is None else np.ascontiguousarray(a, dtype=t)
        keep = [c(start, np.int32), c(index, np.int32), c(value, np.float64), c(collb, np.float64),
                c(colub, np.float64), c(obj, np.float64), c(rowlb, np.float64), c(rowub, np.float64)]
        p = lambda a, f: None if a is None else f(a)
        rc = self._L.Clpb_loadProblem(self._h, int(numberColumns), int(numberRows), _ip(keep[0]),
                                      _ip(keep[1]), _dp(keep[2]), p(keep[3], _dp), p(keep[4], _dp),
                                      p(keep[5], _dp), p(keep[6], _dp), p(keep[7], _dp))
        if rc != 0:
            raise ValueError(f"loadProblem failed ({rc})")
        return rc

    def loadLP(self, lp):
        return self.loadProblem(lp.n, lp.m, lp.col_start, lp.row_index, lp.element, lp.col_lower,
                                lp.col_upper, lp.objective, lp.row_lower, lp.row_upper)

    # ---- ClpModel::readMps ----
    def readMps(self, fileName, keepNames=False, ignoreErrors=False):
        return self._L.Clpb_readMps(self._h, str(fileName).encode(), int(keepNames), int(ignoreErrors))

    # ---- ClpPresolve::presolvedModel / postsolve (elementary actions) ----
    def presolvedModel(self):
        """Returns (status, reduced ClpSimplex or None); status 0 ok, 1 infeasible, 2 unbounded."""
        st = ctypes.c_int(0)
        h = self._L.Clpb_presolvedModel(self._h, ctypes.byref(st))
        if not h:
            return st.value, None
        red = ClpSimplex.__new__(ClpSimplex)
        red._L, red._h, red._keep = self._L, h, None
        return 0, red

    def postsolve(self, reduced):
        return self._L.Clpb_postsolve(self._h, reduced._h)

    def setSolution(self, x, rowPrice, status, problemStatus=0):
        x = np.ascontiguousarray(x, dtype=np.float64); pi = np.ascontiguousarray(rowPrice, dtype=np.float64)
        st = np.ascontiguousarray(status, dtype=np.uint8)
        self._L.Clpb_setSolution(self._h, _dp(x), _dp(pi), _up(st), int(problemStatus))

    def initialSolve(self, presolve=True):
        """ClpSimplex::initialSolve with the dual algorithm: presolve -> dual -> postsolve."""
        if not presolve:
            return self.dual()
        st, red = self.presolvedModel()
        if red is None:
            return st
        rc = red.dual()
        self.postsolve(red)  # also hands a non-optimal status back to this model
        return rc

    def initialPrimalSolve(self, presolve=True):
        """ClpSimplex::initialSolve with the primal algorithm: presolve -> primal -> postsolve."""
        if not presolve:
            return self.primal()
        st, red = self.presolvedModel()
        if red is None:
            return st
        rc = red.primal()
        self.postsolve(red)
        return rc

    def writeMps(self, fileName, formatType=1, numberAcross=1, objSense=0.0):
        return self._L.Clpb_writeMps(self._h, str(fileName).encode(), int(formatType), int(numberAcross), float(objSense))

    def numberRows(self):
        return self._L.Clpb_numberRows(self._h)

    def numberColumns(self):
        return self._L.Clpb_numberColumns(self._h)

    def getNumElements(self):
        return self._L.Clpb_getNumElements(self._h)

    def getProblem(self):
        """Returns the loaded problem as a generators.LP (what readMps parsed)."""
        from .generators import LP

        n, m, nnz = self.numberColumns(), self.numberRows(), self.getNumElements()
        st = np.zeros(n + 1, np.int32); ix = np.zeros(nnz, np.int32); va = np.zeros(nnz)
        cl = np.zeros(n); cu = np.zeros(n); ob = np.zeros(n); rl = np.zeros(m); ru = np.zeros(m)
        self._L.Clpb_getProblem(self._h, _ip(st), _ip(ix), _dp(va), _dp(cl), _dp(cu), _dp(ob),
                                _dp(rl), _dp(ru))
        return LP("from-engine", m, n, st, ix, va, cl, cu, ob, rl, ru)

    # ---- parameters ----
    def _set(self, key, value):
        if self._L.Clpb_setParameter(self._h, key.encode(), float(value)) != 0:
            raise KeyError(key)

    def setPrimalTolerance(self, v): self._set("primalTolerance", v)
    def setDualTolerance(self, v): self._set("dualTolerance", v)
    def setDualBound(self, v): self._set("dualBound", v)
    def setMaximumIterations(self, v): self._set("maximumIterations", v)
    def setMaximumSeconds(self, v): self._set("maximumSeconds", v)
    def setLogLevel(self, v): self._set("logLevel", v)
    def setFactorizationFrequency(self, v): self._set("factorizationFrequency", v)
    def setParameter(self, key, v): self._set(key, v)

    def setPerturbation(self, value):
        """ClpSimplex::setPerturbation: 50 perturb costs, 100 automatic, 102 off (default here)."""
        self._set("perturbation", value)

    def perturbedCosts(self):
        """(rc, cost[n]) -- host-only preview of ClpSimplexDual::perturb for the current settings."""
        c = np.zeros(self.numberColumns())
        rc = self._L.Clpb_perturbedCosts(self._h, _dp(c))
        return rc, c

    def scaling(self, mode):
        """ClpModel::scaling(mode): 0 off, 1 equilibrium, 2 geometric, 3 automatic, 4 dynamic."""
        self._L.Clpb_scaling(self._h, int(mode))

    def scaleFactors(self):
        """(rc, rowScale, columnScale) of ClpPackedMatrix::scale for the current mode (host only)."""
        r = np.ones(self.numberRows()); c = np.ones(self.numberColumns())
        rc = self._L.Clpb_scaleFactors(self._h, _dp(r), _dp(c))
        return rc, r, c

    def copyinStatus(self, status):
        st = np.ascontiguousarray(status, dtype=np.uint8)
        self._L.Clpb_copyinStatus(self._h, _up(st))

    # ---- ClpSimplex::writeBasis / readBasis ----
    def writeBasis(self, fileName, writeValues=False, formatType=0):
        return self._L.Clpb_writeBasis(self._h, str(fileName).encode(), int(writeValues), int(formatType))

    def readBasis(self, fileName):
        return self._L.Clpb_readBasis(self._h, str(fileName).encode())

    # ---- ClpSimplex::dual ----
    def chgColumnLower(self, v): self._L.Clpb_chgColumnLower(self._h, _dp(np.ascontiguousarray(v, dtype=np.float64)))
    def chgColumnUpper(self, v): self._L.Clpb_chgColumnUpper(self._h, _dp(np.ascontiguousarray(v, dtype=np.float64)))
    def chgRowLower(self, v): self._L.Clpb_chgRowLower(self._h, _dp(np.ascontiguousarray(v, dtype=np.float64)))
    def chgRowUpper(self, v): self._L.Clpb_chgRowUpper(self._h, _dp(np.ascontiguousarray(v, dtype=np.float64)))
    def lastSolveWasHot(self): return bool(self._L.Clpb_lastSolveWasHot(self._h))
    def refactorizationInterval(self, nucleusSize): return self._L.Clpb_refactorizationInterval(self._h, int(nucleusSize))

    def fastDual(self):
        """ClpSimplexDual::fastDual: dual() that keeps the device-resident factors of the previous solve"""
        self._set("hotStart", 1)
        try:
            return self.dual()
        finally:
            self._set("hotStart", 0)

    def dual(self, ifValuesPass=0):
        rc = self._L.Clpb_dual(self._h, int(ifValuesPass))
        if rc == _capi.NO_DEVICE:
            raise NoDeviceError("clp_b200 needs a CUDA device (no CPU fallback)")
        if rc == -99:
            raise RuntimeError("clp_b200: CUDA failure inside dual()")
        return rc

    # ---- ClpSimplex::primal ----
    def primal(self, ifValuesPass=0):
        """ClpSimplex::primal (phase 1 sum of infeasibilities, Devex or Dantzig pricing)."""
        rc = self._L.Clpb_primal(self._h, int(ifValuesPass))
        if rc == _capi.NO_DEVICE:
            raise NoDeviceError("clp_b200 needs a CUDA device (no CPU fallback)")
        if rc == -99:
            raise RuntimeError("clp_b200: CUDA failure inside primal()")
        return rc

    def chgObjCoefficients(self, obj):
        """Clp_chgObjCoefficients: replace the loaded objective (n entries)."""
        o = np.ascontiguousarray(obj, dtype=np.float64)
        if o.shape != (self.numberColumns(),):
            raise ValueError("chgObjCoefficients needs one cost per column")
        self._L.Clpb_chgObjCoefficients(self._h, _dp(o))

    def setPrimalColumnPivotAlgorithm(self, mode):
        """0 exact Devex (default), 1 Dantzig."""
        self._set("primalColumnPivot", mode)

    def status(self): return self._L.Clpb_status(self._h)
    def isProvenOptimal(self): return self.status() == 0
    def isProvenPrimalInfeasible(self): return self.status() == 1
    def isProvenDualInfeasible(self): return self.status() == 2
    def objectiveValue(self): return self._L.Clpb_objectiveValue(self._h)
    def numberIterations(self): return self._L.Clpb_numberIterations(self._h)
    def numberRefactorizations(self): return self._L.Clpb_numberRefactorizations(self._h)
    def secondsInLoop(self): return self._L.Clpb_secondsInLoop(self._h)
    def kernelLaunches(self): return self._L.Clpb_kernelLaunches(self._h)
    def nucleusSize(self): return self._L.Clpb_nucleusSize(self._h)

    def timedWindow(self):
        ms = ctypes.c_double(0.0); it = ctypes.c_int(0)
        self._L.Clpb_timedWindow(self._h, ctypes.byref(ms), ctypes.byref(it))
        return ms.value, it.value

    def phaseTimes(self):
        o = np.zeros(14)
        self._L.Clpb_phaseTimes(self._h, _dp(o))
        keys = ["chuzr", "btran", "price", "chuzc", "dualUpdate", "ftran", "update", "refactor", "samples",
                "priceKernel", "ftranGemv", "btranGemv", "ftranGemvBytes", "btranGemvBytes"]
        return dict(zip(keys, o.tolist()))

    def _vec(self, fn, size, dtype=np.float64):
        out = np.zeros(size, dtype=dtype)
        fn(self._h, _dp(out) if dtype == np.float64 else _up(out))
        return out

    def primalColumnSolution(self): return self._vec(self._L.Clpb_primalColumnSolution, self.numberColumns())
    def primalRowSolution(self): return self._vec(self._L.Clpb_primalRowSolution, self.numberRows())
    def dualColumnSolution(self): return self._vec(self._L.Clpb_dualColumnSolution, self.numberColumns())
    def dualRowSolution(self): return self._vec(self._L.Clpb_dualRowSolution, self.numberRows())
    def statusArray(self): return self._vec(self._L.Clpb_statusArray, self.numberColumns() + self.numberRows(), np.uint8)

    # ---- column sharding ----
    def initSharding(self, rank, world_size, unique_id):
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        rc = self._L.Clpb_initSharding(self._h, int(rank), int(world_size), _up(uid))
        if rc != 0:
            raise RuntimeError(f"NCCL communicator init failed ({rc})")

    @staticmethod
    def ncclUniqueId():
        uid = np.zeros(128, dtype=np.uint8)
        rc = _capi.lib().Clpb_ncclUniqueId(_up(uid))
        if rc != 0:
            raise RuntimeError(f"ncclGetUniqueId failed ({rc})")
        return uid

    # ---- plug-in level (ClpFactorization / ClpMatrixBase / ClpDualRowPivot interfaces) ----
    def _chk(self, rc):
        if rc == _capi.NO_DEVICE:
            raise NoDeviceError("clp_b200 needs a CUDA device (no CPU fallback)")
        if rc == -99:
            raise RuntimeError("clp_b200: CUDA failure")
        return rc

    def factorize(self, basicSequence):
        b = np.ascontiguousarray(basicSequence, dtype=np.int32)
        pv = np.zeros(self.numberRows(), dtype=np.int32)
        rc = self._chk(self._L.Clpb_factorize(self._h, _ip(b), _ip(pv)))
        return rc, pv

    def updateColumn(self, region):
        v = np.array(region, dtype=np.float64)
        self._chk(self._L.Clpb_updateColumn(self._h, _dp(v)))
        return v

    def updateColumnTranspose(self, region):
        v = np.array(region, dtype=np.float64)
        self._chk(self._L.Clpb_updateColumnTranspose(self._h, _dp(v)))
        return v

    def replaceColumn(self, sequenceIn, pivotRow):
        return self._chk(self._L.Clpb_replaceColumn(self._h, int(sequenceIn), int(pivotRow)))

    def transposeTimes(self, scalar, pi):
        pi = np.ascontiguousarray(pi, dtype=np.float64)
        z = np.zeros(self.numberColumns())
        self._chk(self._L.Clpb_transposeTimes(self._h, float(scalar), _dp(pi), _dp(z)))
        return z

    def times(self, scalar, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.zeros(self.numberRows())
        self._chk(self._L.Clpb_times(self._h, float(scalar), _dp(x), _dp(y)))
        return y

    def dualColumn(self, alphaRow, dj, status, direction, infeasibility):
        a = np.ascontiguousarray(alphaRow, dtype=np.float64)
        d = np.ascontiguousarray(dj, dtype=np.float64)
        s = np.ascontiguousarray(status, dtype=np.uint8)
        theta = ctypes.c_double(0.0)
        q = self._chk(self._L.Clpb_dualColumn(self._h, _dp(a), _dp(d), _up(s), int(direction),
                                              float(infeasibility), ctypes.byref(theta)))
        return q, theta.value

    def dualColumnRowPass(self, alphaRow, dj, status, direction, infeasibility):
        a = np.ascontiguousarray(alphaRow, dtype=np.float64)
        d = np.ascontiguousarray(dj, dtype=np.float64)
        s = np.ascontiguousarray(status, dtype=np.uint8)
        theta = ctypes.c_double(0.0)
        q = self._chk(self._L.Clpb_dualColumnRowPass(self._h, _dp(a), _dp(d), _up(s), int(direction),
                                                     float(infeasibility), ctypes.byref(theta)))
        return q, theta.value

    # ---- ClpDualRowPivot surface, one iteration at a time (include/clp_b200.h)
    def pivotRow(self):
        """ClpDualRowPivot::pivotRow -> (row or -1/-2, sequenceOut, direction, infeasibility)"""
        so, di, inf = ctypes.c_int(-1), ctypes.c_int(0), ctypes.c_double(0.0)
        r = self._chk(self._L.Clpb_pivotRow(self._h, ctypes.byref(so), ctypes.byref(di), ctypes.byref(inf)))
        return r, so.value, di.value, inf.value

    def updateColumnTransposeAndPrice(self):
        rho, row = np.zeros(self.numberRows()), np.zeros(self.numberColumns())
        nz = self._chk(self._L.Clpb_updateColumnTransposeAndPrice(self._h, _dp(rho), _dp(row)))
        return nz, rho, row

    def dualColumnDevice(self):
        th, al = ctypes.c_double(0.0), ctypes.c_double(0.0)
        q = self._chk(self._L.Clpb_dualColumnDevice(self._h, ctypes.byref(th), ctypes.byref(al)))
        return q, th.value, al.value

    def updateWeights(self):
        rc = ctypes.c_int(0)
        alpha = self._L.Clpb_updateWeights(self._h, ctypes.byref(rc))
        return alpha, rc.value

    def unrollWeights(self): return self._L.Clpb_unrollWeights(self._h)

    def updatePrimalSolution(self):
        ch = ctypes.c_double(0.0)
        t = self._chk(self._L.Clpb_updatePrimalSolution(self._h, ctypes.byref(ch)))
        return t, ch.value

    def saveWeights(self, mode): return self._chk(self._L.Clpb_saveWeights(self._h, int(mode)))

    def updateColumnFT(self, region):
        r = np.ascontiguousarray(region, dtype=np.float64).copy()
        nz = self._chk(self._L.Clpb_updateColumnFT(self._h, _dp(r)))
        return nz, r

    def updateTwoColumnsFT(self, regionFT, regionOther):
        a = np.ascontiguousarray(regionFT, dtype=np.float64).copy()
        b = np.ascontiguousarray(regionOther, dtype=np.float64).copy()
        nz = self._chk(self._L.Clpb_updateTwoColumnsFT(self._h, _dp(a), _dp(b)))
        return nz, a, b

    def replaceColumnChecked(self, sequenceIn, pivotRow, pivotCheck, acceptablePivot=1e-8):
        return self._L.Clpb_replaceColumnChecked(self._h, int(sequenceIn), int(pivotRow), float(pivotCheck),
                                                 float(acceptablePivot))

    def _packed(self, fn, indices, elements, cap):
        idx = np.zeros(cap, dtype=np.int32); el = np.zeros(cap)
        k = len(indices)
        idx[:k] = indices; el[:k] = elements
        num = ctypes.c_int(k)
        self._chk(fn(self._h, ctypes.byref(num), _ip(idx), _dp(el)))
        return idx[:num.value].copy(), el[:num.value].copy()

    def updateColumnPacked(self, indices, elements):
        return self._packed(self._L.Clpb_updateColumnPacked, indices, elements, self.numberRows())

    def updateColumnTransposePacked(self, indices, elements):
        return self._packed(self._L.Clpb_updateColumnTransposePacked, indices, elements, self.numberRows())

    def transposeTimesPacked(self, scalar, indices, elements):
        ip = np.ascontiguousarray(indices, dtype=np.int32); ep = np.ascontiguousarray(elements, dtype=np.float64)
        iz = np.zeros(self.numberColumns(), dtype=np.int32); ez = np.zeros(self.numberColumns())
        nz = ctypes.c_int(0)
        self._chk(self._L.Clpb_transposeTimesPacked(self._h, float(scalar), len(ip), _ip(ip), _dp(ep),
                                                    ctypes.byref(nz), _ip(iz), _dp(ez)))
        return iz[:nz.value].copy(), ez[:nz.value].copy()

    def primalColumnPivot(self, dj, status, weights, mode=0):
        """ClpPrimalColumnPivot::pivotColumn on explicit dj / status / weights (n+m each) -> sequence or -1"""
        d = np.ascontiguousarray(dj, dtype=np.float64)
        s = np.ascontiguousarray(status, dtype=np.uint8)
        w = np.ascontiguousarray(weights, dtype=np.float64)
        return self._chk(self._L.Clpb_primalColumnPivot(self._h, _dp(d), _up(s), _dp(w), int(mode)))

    def primalRow(self, alpha, xB, lowerB, upperB, direction, enteringRange, phase=2):
        """ClpSimplexPrimal::primalRow on explicit vectors (m each) -> (row, -1 no block or -2 flip; theta)"""
        a, x, lo, up = (np.ascontiguousarray(v, dtype=np.float64) for v in (alpha, xB, lowerB, upperB))
        theta = ctypes.c_double(0.0)
        r = self._chk(self._L.Clpb_primalRow(self._h, _dp(a), _dp(x), _dp(lo), _dp(up), int(direction),
                                             float(enteringRange), int(phase), ctypes.byref(theta)))
        return r, theta.value

    def startup(self): return self._chk(self._L.Clpb_startup(self._h))
    def iterate(self, count): return self._chk(self._L.Clpb_iterate(self._h, int(count)))

    def weights(self):
        w = np.zeros(self.numberRows())
        self._L.Clpb_getWeights(self._h, _dp(w))
        return w

    def deviceVector(self, name):
        n, m = self.numberColumns(), self.numberRows()
        size = {"sol": n + m, "dj": n + m, "rho": m, "alphaRow": n + m, "pivotVariable": m,
                "status": n + m}[name]
        out = np.zeros(size)
        self._L.Clpb_getDeviceVector(self._h, name.encode(), _dp(out))
        return out
