"""ctypes mirrors of the plain-data structs in csrc/pip_types.h and include/piplib_b200.h."""
import ctypes as C

import numpy as np

ST_OK, ST_VOID, ST_FATAL, ST_FAULT = 0, 1, 1000, 2000
ST_PENDING, ST_CAPACITY, ST_UNSUPPORTED = 4000, 4001, 4002
F_INT, F_DUAL, F_DEEPEST = 1, 2, 4


class PipProblem(C.Structure):
    _fields_ = [("nvar", C.c_int), ("nparm", C.c_int), ("ni", C.c_int), ("nc", C.c_int),
                ("bigparm", C.c_int), ("flags", C.c_int), ("off", C.c_longlong)]


class PipResult(C.Structure):
    _fields_ = [("status", C.c_int), ("ncells", C.c_int), ("cell_off", C.c_longlong),
                ("pivots", C.c_uint), ("cuts", C.c_uint), ("subsolves", C.c_uint),
                ("splits", C.c_uint), ("max_rows", C.c_uint), ("max_cols", C.c_uint),
                ("ser_words", C.c_uint), ("elem_updates_lo", C.c_uint), ("elem_updates_hi", C.c_uint),
                ("pad", C.c_uint)]


class PipCell(C.Structure):
    _fields_ = [("kind", C.c_int), ("pad", C.c_int), ("p1", C.c_longlong), ("p2", C.c_longlong)]


PROBLEM_DTYPE = np.dtype([("nvar", "i4"), ("nparm", "i4"), ("ni", "i4"), ("nc", "i4"),
                          ("bigparm", "i4"), ("flags", "i4"), ("off", "i8")])
RESULT_DTYPE = np.dtype([("status", "i4"), ("ncells", "i4"), ("cell_off", "i8"), ("pivots", "u4"),
                         ("cuts", "u4"), ("subsolves", "u4"), ("splits", "u4"), ("max_rows", "u4"),
                         ("max_cols", "u4"), ("ser_words", "u4"), ("elem_updates_lo", "u4"),
                         ("elem_updates_hi", "u4"), ("pad", "u4")])
CELL_DTYPE = np.dtype([("kind", "i4"), ("pad", "i4"), ("p1", "i8"), ("p2", "i8")])
# PipProblemInfo_dp (include/piplib_b200.h): the per-problem solve report of a dense batch
INFO_DTYPE = np.dtype([("flags", "u4"), ("pivots", "u4"), ("cuts", "u4"), ("splits", "u4"), ("max_rows", "u4"),
                       ("max_cols", "u4"), ("spare", "u4", (2,))])
assert PROBLEM_DTYPE.itemsize == C.sizeof(PipProblem) == 32
assert RESULT_DTYPE.itemsize == C.sizeof(PipResult) == 56
assert CELL_DTYPE.itemsize == C.sizeof(PipCell) == 24
assert INFO_DTYPE.itemsize == 32


def pack_tableau_problems(cases):
    """cases: iterable of dicts with nvar,nparm,ni,nc,bigparm,nq,tab,ctx (the .dat view).
    Returns (problems[PROBLEM_DTYPE], pool[int64])."""
    cases = list(cases)
    probs = np.zeros(len(cases), dtype=PROBLEM_DTYPE)
    chunks, off = [], 0
    for i, c in enumerate(cases):
        tab = np.asarray(c["tab"], dtype=np.int64).reshape(-1)
        ctx = np.asarray(c["ctx"], dtype=np.int64).reshape(-1)
        assert tab.size == c["ni"] * (c["nvar"] + c["nparm"] + 1)
        assert ctx.size == c["nc"] * (c["nparm"] + 1)
        probs[i] = (c["nvar"], c["nparm"], c["ni"], c["nc"], c["bigparm"],
                    (F_INT if c["nq"] & 1 else (2 if c["nq"] & 2 else 0)) | (4 if c["nq"] & 4 else 0), off)
        chunks += [tab, ctx]
        off += tab.size + ctx.size
    pool = np.concatenate(chunks) if chunks else np.zeros(0, dtype=np.int64)
    if pool.size == 0:
        pool = np.zeros(1, dtype=np.int64)
    return probs, np.ascontiguousarray(pool, dtype=np.int64)
