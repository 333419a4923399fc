"""ctypes loader of the C-ABI library (include/clp_b200.h).

The library is built in-tree by ``clp_b200/csrc/Makefile`` into ``clp_b200/_lib/``.  There is
no fallback: if the shared object is missing the import of any solver entry point raises.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libclp_b200.so")
NO_DEVICE = -100

_lib = None

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)
c_ubyte_p = ctypes.POINTER(ctypes.c_ubyte)

# name -> (restype, argtypes); mirrors include/clp_b200.h one to one
SIGNATURES = {
    "Clpb_newModel": (ctypes.c_void_p, []),
    "Clpb_deleteModel": (None, [ctypes.c_void_p]),
    "Clpb_loadProblem": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_int_p, c_int_p,
                                        c_double_p, c_double_p, c_double_p, c_double_p, c_double_p,
                                        c_double_p]),
    "Clpb_readMps": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]),
    "Clpb_presolvedModel": (ctypes.c_void_p, [ctypes.c_void_p, c_int_p]),
    "Clpb_postsolve": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "Clpb_setSolution": (None, [ctypes.c_void_p, c_double_p, c_double_p, c_ubyte_p, ctypes.c_int]),
    "Clpb_writeMps": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_double]),
    "Clpb_numberRows": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_numberColumns": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_getNumElements": (ctypes.c_longlong, [ctypes.c_void_p]),
    "Clpb_getProblem": (None, [ctypes.c_void_p, c_int_p, c_int_p, c_double_p, c_double_p, c_double_p,
                               c_double_p, c_double_p, c_double_p]),
    "Clpb_setParameter": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_double]),
    "Clpb_scaling": (None, [ctypes.c_void_p, ctypes.c_int]),
    "Clpb_scaleFactors": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p]),
    "Clpb_perturbedCosts": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "Clpb_copyinStatus": (None, [ctypes.c_void_p, c_ubyte_p]),
    "Clpb_writeBasis": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int, ctypes.c_int]),
    "Clpb_readBasis": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p]),
    "Clpb_chgColumnLower": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_chgColumnUpper": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_chgRowLower": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_chgRowUpper": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_lastSolveWasHot": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_refactorizationInterval": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "Clpb_dual": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "Clpb_primal": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "Clpb_chgObjCoefficients": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_primalColumnPivot": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_ubyte_p, c_double_p, ctypes.c_int]),
    "Clpb_primalRow": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p, c_double_p, c_double_p, ctypes.c_int,
                                      ctypes.c_double, ctypes.c_int, c_double_p]),
    "Clpb_status": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_objectiveValue": (ctypes.c_double, [ctypes.c_void_p]),
    "Clpb_numberIterations": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_numberRefactorizations": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_primalColumnSolution": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_primalRowSolution": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_dualColumnSolution": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_dualRowSolution": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_statusArray": (None, [ctypes.c_void_p, c_ubyte_p]),
    "Clpb_secondsInLoop": (ctypes.c_double, [ctypes.c_void_p]),
    "Clpb_kernelLaunches": (ctypes.c_longlong, [ctypes.c_void_p]),
    "Clpb_phaseTimes": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_nucleusSize": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_timedWindow": (None, [ctypes.c_void_p, c_double_p, c_int_p]),
    "Clpb_ncclUniqueId": (ctypes.c_int, [c_ubyte_p]),
    "Clpb_initSharding": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, c_ubyte_p]),
    "Clpb_factorize": (ctypes.c_int, [ctypes.c_void_p, c_int_p, c_int_p]),
    "Clpb_updateColumn": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "Clpb_updateColumnTranspose": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "Clpb_replaceColumn": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "Clpb_transposeTimes": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_double, c_double_p, c_double_p]),
    "Clpb_times": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_double, c_double_p, c_double_p]),
    "Clpb_dualColumn": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p, c_ubyte_p, ctypes.c_int,
                                       ctypes.c_double, c_double_p]),
    "Clpb_dualColumnRowPass": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p, c_ubyte_p, ctypes.c_int,
                                              ctypes.c_double, c_double_p]),
    "Clpb_denseInvert": (ctypes.c_int, [ctypes.c_int, c_double_p, c_double_p]),
    "Clpb_pivotRow": (ctypes.c_int, [ctypes.c_void_p, c_int_p, c_int_p, c_double_p]),
    "Clpb_updateColumnTransposeAndPrice": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p]),
    "Clpb_dualColumnDevice": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p]),
    "Clpb_updateWeights": (ctypes.c_double, [ctypes.c_void_p, c_int_p]),
    "Clpb_unrollWeights": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_updatePrimalSolution": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "Clpb_saveWeights": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "Clpb_updateColumnFT": (ctypes.c_int, [ctypes.c_void_p, c_double_p]),
    "Clpb_updateTwoColumnsFT": (ctypes.c_int, [ctypes.c_void_p, c_double_p, c_double_p]),
    "Clpb_replaceColumnChecked": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double]),
    "Clpb_updateColumnPacked": (ctypes.c_int, [ctypes.c_void_p, c_int_p, c_int_p, c_double_p]),
    "Clpb_updateColumnTransposePacked": (ctypes.c_int, [ctypes.c_void_p, c_int_p, c_int_p, c_double_p]),
    "Clpb_transposeTimesPacked": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_double, ctypes.c_int, c_int_p, c_double_p,
                                                 c_int_p, c_int_p, c_double_p]),
    "Clpb_startup": (ctypes.c_int, [ctypes.c_void_p]),
    "Clpb_iterate": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "Clpb_getWeights": (None, [ctypes.c_void_p, c_double_p]),
    "Clpb_getDeviceVector": (None, [ctypes.c_void_p, ctypes.c_char_p, c_double_p]),
}


def build(force: bool = False) -> str:
    """Compile the CUDA sources for sm_100a (nvcc cross-compiles without a GPU)."""
    args = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
    if force:
        args.append("-B")
    subprocess.check_call(args)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C clp_b200/csrc` "
                "(clp_b200 has no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
