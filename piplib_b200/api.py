"""Python mirror of the C-ABI (ctypes).  Thin by design: the product is the shared library
piplib_b200/lib/libpiplib_dp.so; this module only marshals numpy arrays into it so that the
parity tests and bench.py read like the reference's own drivers (example/example.c, maind.c).

There is no CPU path: if the library is missing, or no sm_100 device is present when a solve
is requested, the call fails loudly.
"""
import ctypes as C
import os

import numpy as np

from .ctypes_defs import CELL_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PIPLIB_B200_LIB") or os.path.join(HERE, "lib", "libpiplib_dp.so")
PHASES = ["load", "sort", "scan", "buildsub", "choose", "update", "swap", "cut", "frame", "emit", "other",
          "u_head", "u_pass1", "u_gcd", "u_div", "u_wait"]      # u_*: lane 0's share inside "update"

I64P = C.POINTER(C.c_longlong)


class PipMatrix(C.Structure):
    _fields_ = [("NbRows", C.c_uint), ("NbColumns", C.c_uint), ("p", C.POINTER(I64P)),
                ("p_Init", I64P), ("p_Init_size", C.c_int)]


class PipOptions(C.Structure):
    _fields_ = [("Nq", C.c_int), ("Verbose", C.c_int), ("Simplify", C.c_int),
                ("Deepest_cut", C.c_int), ("Maximize", C.c_int), ("Urs_parms", C.c_int),
                ("Urs_unknowns", C.c_int), ("Compute_dual", C.c_int)]


class PipTableauHeader(C.Structure):
    _fields_ = [("nvar", C.c_int), ("nparm", C.c_int), ("ni", C.c_int), ("nc", C.c_int),
                ("bigparm", C.c_int), ("nq", C.c_int)]


class PipBatchStats(C.Structure):
    _fields_ = [("pivots", C.c_ulonglong), ("cuts", C.c_ulonglong), ("subsolves", C.c_ulonglong),
                ("splits", C.c_ulonglong), ("elem_updates", C.c_ulonglong),
                ("max_rows", C.c_uint), ("max_cols", C.c_uint),
                ("seconds_h2d", C.c_double), ("seconds_kernel", C.c_double),
                ("seconds_d2h", C.c_double), ("seconds_host", C.c_double),
                ("device_ms", C.c_float), ("launches", C.c_int), ("rounds", C.c_int),
                ("h2d_bytes", C.c_ulonglong), ("d2h_bytes", C.c_ulonglong),
                ("cells", C.c_ulonglong), ("phase_cycles", C.c_ulonglong * 16), ("wrapped", C.c_ulonglong)]


_lib = None


def lib():
    """load the CUDA library; raises if it has not been built (no fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("piplib_b200: %s is missing -- run `python -m piplib_b200.build`; "
                               "there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.pip_matrix_alloc_dp.restype = C.POINTER(PipMatrix)
        L.pip_matrix_alloc_dp.argtypes = [C.c_uint, C.c_uint]
        L.pip_matrix_free_dp.argtypes = [C.POINTER(PipMatrix)]
        L.pip_options_init_dp.restype = C.POINTER(PipOptions)
        L.pip_options_free_dp.argtypes = [C.POINTER(PipOptions)]
        L.pip_solve_dp.restype = C.c_void_p
        L.pip_solve_dp.argtypes = [C.POINTER(PipMatrix), C.POINTER(PipMatrix), C.c_int,
                                   C.POINTER(PipOptions)]
        L.pip_solve_batch_dp.restype = C.c_int
        L.pip_quast_free_dp.argtypes = [C.c_void_p]
        L.pip_quast_serialize_dp.restype = C.c_long
        L.pip_quast_serialize_dp.argtypes = [C.c_void_p, I64P, C.c_long]
        L.pip_quast_print_dp.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.pip_traiter_batch_dp.restype = C.c_int
        L.pip_solve_dense_dp.restype = C.c_int
        L.pip_device_batch_create.restype = C.c_void_p
        L.pip_device_batch_run.restype = C.c_int
        L.pip_device_batch_run.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float)]
        L.pip_device_batch_results.restype = C.c_int
        L.pip_device_batch_results.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.pip_device_batch_destroy.argtypes = [C.c_void_p]
        L.pip_large_create_dp.restype = C.c_void_p
        L.pip_large_run_dp.restype = C.c_int
        L.pip_large_run_dp.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.pip_large_fetch_dp.restype = C.c_int
        L.pip_large_fetch_dp.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_int,
                                         C.POINTER(C.c_int), C.POINTER(C.c_longlong)]
        L.pip_large_destroy_dp.argtypes = [C.c_void_p]
        L.pip_last_batch_stats_dp.argtypes = [C.POINTER(PipBatchStats)]
        L.pip_set_device_dp.restype = C.c_int
        L.pip_last_batch_flags_dp.restype = C.c_longlong
        L.pip_last_batch_flags_dp.argtypes = [C.c_void_p, C.c_longlong]
        L.pip_set_devices_dp.restype = C.c_int
        L.pip_pin_buffer_dp.restype = C.c_int
        L.pip_pin_buffer_dp.argtypes = [C.c_void_p, C.c_size_t]
        L.pip_unpin_buffer_dp.restype = C.c_int
        L.pip_unpin_buffer_dp.argtypes = [C.c_void_p]
        L.pip_b200_version.restype = C.c_char_p
        _lib = L
    return _lib


def set_device(dev):
    return lib().pip_set_device_dp(int(dev))


def set_devices(devs):
    """devices pip_solve_dense_dp spreads its chunks over (one process, several GPUs); [] = default"""
    arr = (C.c_int * max(1, len(devs)))(*devs)
    rc = lib().pip_set_devices_dp(len(devs), arr)
    if rc != 0:
        raise RuntimeError("pip_set_devices_dp failed")


def pin(a):
    """page-lock a numpy array in place (cudaHostRegister): pip_solve_dense_dp then moves it by DMA alone"""
    if a is None or a.nbytes == 0:
        return a
    if lib().pip_pin_buffer_dp(a.ctypes.data, a.nbytes) != 0:
        raise RuntimeError("pip_pin_buffer_dp failed")
    return a


_pinned_allocs = {}


def pinned_empty(shape, dtype):
    """numpy array over page-locked memory from the driver (pip_alloc_pinned_dp); free with pinned_free"""
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) * dt.itemsize
    L = lib()
    L.pip_alloc_pinned_dp.restype = C.c_void_p
    L.pip_alloc_pinned_dp.argtypes = [C.c_size_t]
    L.pip_free_pinned_dp.argtypes = [C.c_void_p]
    p = L.pip_alloc_pinned_dp(max(n, 1))
    if not p:
        raise RuntimeError("pip_alloc_pinned_dp failed")
    buf = (C.c_char * max(n, 1)).from_address(p)
    a = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)
    _pinned_allocs[a.ctypes.data] = p
    return a


def pinned_copy(a):
    b = pinned_empty(a.shape, a.dtype)
    b[...] = a
    return b


def pinned_free(a):
    p = _pinned_allocs.pop(a.ctypes.data, None)
    if p:
        lib().pip_free_pinned_dp(p)


def unpin(a):
    if a is not None and a.nbytes:
        lib().pip_unpin_buffer_dp(a.ctypes.data)


def last_flags():
    """per-problem flags of the last batch / traiter call on this thread (bit 0: a 128-bit product wrapped)"""
    n = lib().pip_last_batch_flags_dp(None, C.c_longlong(0))
    out = np.zeros(max(int(n), 1), dtype=np.uint32)
    lib().pip_last_batch_flags_dp(out.ctypes.data_as(C.c_void_p), C.c_longlong(int(n)))
    return out[:int(n)]


def last_stats():
    s = PipBatchStats()
    lib().pip_last_batch_stats_dp(C.byref(s))
    return s


def make_options(**kw):
    o = PipOptions(1, 0, 0, 0, 0, 0, 0, 0)
    for k, v in kw.items():
        setattr(o, k, int(v))
    return o


def _matrix(rows, cols, data):
    L = lib()
    m = L.pip_matrix_alloc_dp(rows, cols)
    if rows and cols:
        a = np.ascontiguousarray(data, dtype=np.int64).reshape(rows * cols)
        C.memmove(m.contents.p_Init, a.ctypes.data, a.nbytes)
    return m


def _serialize(q):
    L = lib()
    n = L.pip_quast_serialize_dp(q, None, 0)
    buf = np.zeros(max(n, 1), dtype=np.int64)
    L.pip_quast_serialize_dp(q, buf.ctypes.data_as(I64P), n)
    return [int(x) for x in buf[:n]]


def solve_batch(problems, **opts):
    """problems: list of dict(dom=2-D list, ctx=2-D list or None, ctx_cols=int, bignum=int).
    One pip_solve_batch_dp call.  Returns [(status, serialised quast)]."""
    L = lib()
    n = len(problems)
    doms = (C.POINTER(PipMatrix) * n)()
    ctxs = (C.POINTER(PipMatrix) * n)()
    bgs = (C.c_int * n)()
    for i, p in enumerate(problems):
        d = np.asarray(p["dom"], dtype=np.int64)
        doms[i] = _matrix(d.shape[0], d.shape[1], d)
        if p.get("ctx") is not None:
            c = np.asarray(p["ctx"], dtype=np.int64)
            if c.ndim != 2:
                c = c.reshape(0, p["ctx_cols"])
            ctxs[i] = _matrix(c.shape[0], c.shape[1], c)
        bgs[i] = int(p.get("bignum", -1))
    out = (C.c_void_p * n)()
    status = (C.c_int * n)()
    o = make_options(**opts)
    rc = L.pip_solve_batch_dp(n, doms, ctxs, bgs, C.byref(o), out, status)
    if rc != 0:
        raise RuntimeError("pip_solve_batch_dp failed: %d" % rc)
    res = []
    for i in range(n):
        st = int(status[i])
        ser = _serialize(out[i]) if st in (0, 1) else []
        if out[i]:
            L.pip_quast_free_dp(out[i])
        res.append((st, ser))
        L.pip_matrix_free_dp(doms[i])
        if ctxs[i]:
            L.pip_matrix_free_dp(ctxs[i])
    return res


def time_solve_batch(dom, ctx, bignum=-1, reps=2, **opts):
    """pip_solve_batch_dp (PipMatrix objects in, malloc'd PipQuast trees out) on a dense numpy batch: the
    matrices are built before and the trees freed after the timed call.  Returns (best seconds, statuses)."""
    import time
    L = lib()
    n = dom.shape[0]
    doms = (C.POINTER(PipMatrix) * n)()
    ctxs = (C.POINTER(PipMatrix) * n)()
    bgs = (C.c_int * n)(*([int(bignum)] * n))
    for i in range(n):
        doms[i] = _matrix(dom.shape[1], dom.shape[2], dom[i])
        if ctx is not None:
            ctxs[i] = _matrix(ctx.shape[1], ctx.shape[2], ctx[i])
    out = (C.c_void_p * n)()
    status = (C.c_int * n)()
    o = make_options(**opts)
    best = 1e30
    for _ in range(reps):
        t = time.perf_counter()
        rc = L.pip_solve_batch_dp(n, doms, ctxs, bgs, C.byref(o), out, status)
        best = min(best, time.perf_counter() - t)
        if rc != 0:
            raise RuntimeError("pip_solve_batch_dp failed: %d" % rc)
        for i in range(n):
            if out[i]:
                L.pip_quast_free_dp(out[i])
    for i in range(n):
        L.pip_matrix_free_dp(doms[i])
        if ctxs[i]:
            L.pip_matrix_free_dp(ctxs[i])
    return best, np.asarray(list(status), dtype=np.int32)


def solve(dom, ctx, bg, ctx_cols=None, **opts):
    """one problem through the batch entry point (pip_solve_dp itself exits on fatal verdicts)."""
    return solve_batch([dict(dom=dom, ctx=ctx, ctx_cols=ctx_cols, bignum=bg)], **opts)[0]


def traiter_batch(cases):
    """cases: dicts with nvar,nparm,ni,nc,bigparm,nq,tab,ctx (the .dat view).
    Returns [(status, [[kind,p1,p2],...])]."""
    L = lib()
    n = len(cases)
    hdr = (PipTableauHeader * n)()
    tabs = (I64P * n)()
    ctxs = (I64P * n)()
    keep = []
    for i, c in enumerate(cases):
        hdr[i] = PipTableauHeader(c["nvar"], c["nparm"], c["ni"], c["nc"], c["bigparm"], c["nq"])
        t = np.ascontiguousarray(np.asarray(c["tab"], dtype=np.int64).reshape(-1))
        x = np.ascontiguousarray(np.asarray(c["ctx"], dtype=np.int64).reshape(-1))
        if t.size == 0:
            t = np.zeros(1, dtype=np.int64)
        if x.size == 0:
            x = np.zeros(1, dtype=np.int64)
        keep += [t, x]
        tabs[i] = t.ctypes.data_as(I64P)
        ctxs[i] = x.ctypes.data_as(I64P)
    status = np.zeros(n, dtype=np.int32)
    ncells = np.zeros(n, dtype=np.int32)
    off = np.zeros(n, dtype=np.int64)
    need = C.c_longlong(0)
    cap = 4096 * min(n, 64) + 4096
    while True:
        cells = np.zeros(cap, dtype=CELL_DTYPE)
        rc = L.pip_traiter_batch_dp(n, hdr, tabs, ctxs, status.ctypes.data_as(C.c_void_p),
                                    cells.ctypes.data_as(C.c_void_p), C.c_longlong(cap),
                                    off.ctypes.data_as(C.c_void_p), ncells.ctypes.data_as(C.c_void_p),
                                    C.byref(need))
        if rc == -2:
            cap = int(need.value) + 16
            continue
        if rc != 0:
            raise RuntimeError("pip_traiter_batch_dp failed: %d" % rc)
        break
    out = []
    for i in range(n):
        c = cells[off[i]:off[i] + ncells[i]]
        out.append((int(status[i]), [[int(x["kind"]), int(x["p1"]), int(x["p2"])] for x in c]))
    return out


def _ptr(a):
    """address of a numpy array, or of a torch tensor's data (host or device memory)"""
    return C.c_void_p(a.data_ptr()) if hasattr(a, "data_ptr") else a.ctypes.data_as(C.c_void_p)


def _ready(*arrays):
    """the library works on CUDA streams of its own: whatever torch queued on the current stream of a device that
    holds one of the arrays (producing the inputs, clearing the outputs) must be complete before the call"""
    devices = {a.device for a in arrays if getattr(a, "is_cuda", False)}
    if devices:
        import torch
        for d in devices:
            torch.cuda.current_stream(d).synchronize()


class _HostArrays:
    """solve_dense on numpy arrays (pageable or page-locked host memory)"""

    def input(self, a):
        return np.ascontiguousarray(a, dtype=np.int64)

    def zeros(self, n, dtype):
        return np.zeros(n, dtype=np.uint64 if dtype == "u64" else dtype)

    def empty(self, n):
        return np.empty(n, dtype=np.int64)


class _CudaTensors:
    """solve_dense on torch CUDA tensors: the library reads the rows and writes the results in device memory,
    on the device that holds them.  Hashes come back as int64 tensors holding the uint64 bits."""

    def __init__(self, like):
        import torch
        self.torch, self.device = torch, like.device

    def input(self, a):
        if not getattr(a, "is_cuda", False) or a.device != self.device:
            raise ValueError("solve_dense: dom and ctx must both be CUDA tensors on one device, or both host arrays")
        return a.to(self.torch.int64).contiguous()

    def zeros(self, n, dtype):
        return self.torch.zeros(n, dtype=self.torch.int32 if dtype == np.int32 else self.torch.int64, device=self.device)

    def empty(self, n):
        return self.torch.empty(n, dtype=self.torch.int64, device=self.device)


def solve_dense(dom, ctx, bignum=-1, want_hashes=True, want_ser=False, ser_cap_hint=None, out=None, **opts):
    """dom: [n, rows, cols] int64; ctx: [n, rows, cols] or None.  Host arrays (numpy), or torch CUDA tensors:
    these are read and the results written in GPU memory, and the results are CUDA tensors (status int32,
    hashes / ser / ser_off / ser_len int64; hashes hold the uint64 bits).
    Returns dict(status, hashes, ser, ser_off, ser_len)."""
    L = lib()
    B = _CudaTensors(dom) if getattr(dom, "is_cuda", False) else _HostArrays()
    dom = B.input(dom)
    n, dr, dc = dom.shape
    if ctx is None:
        has, cr, cc, cp = 0, 0, 0, None
    else:
        ctx = B.input(ctx)
        has, cr, cc = 1, ctx.shape[1], ctx.shape[2]
        cp = _ptr(ctx)
    # `out` = the dict returned by an earlier call of the same shape: its (caller-owned) result
    # buffers are reused instead of allocating and page-faulting gigabytes again
    reuse = out is not None and out["status"].shape[0] == n
    status = out["status"] if reuse else B.zeros(n, np.int32)
    hashes = None
    if want_hashes:
        hashes = out["hashes"] if reuse and out.get("hashes") is not None else B.zeros(n, "u64")
    o = make_options(**opts)
    ser = ser_off = ser_len = None
    cap = 0
    if want_ser:
        if reuse and out.get("ser") is not None:
            ser, ser_off, ser_len = out["ser"], out["ser_off"], out["ser_len"]
            cap = ser.shape[0]
        else:
            ser_off = B.zeros(n + 1, np.int64)
            ser_len = B.zeros(n, np.int64)
            cap = (ser_cap_hint or 448) * n + 1024
            ser = B.empty(cap)
    while True:
        _ready(dom, ctx, status, hashes, ser, ser_off, ser_len)
        rc = L.pip_solve_dense_dp(C.c_longlong(n), dr, dc, _ptr(dom), has, cr, cc, cp,
                                  int(bignum), C.byref(o), _ptr(status),
                                  _ptr(hashes) if want_hashes else None,
                                  _ptr(ser) if want_ser else None,
                                  C.c_longlong(cap),
                                  _ptr(ser_off) if want_ser else None,
                                  _ptr(ser_len) if want_ser else None)
        if rc == -2:
            was_pinned = reuse and out.get("ser") is ser and isinstance(ser, np.ndarray)
            cap = int(ser_off[n]) + 16
            ser = ser.new_empty(cap) if hasattr(ser, "new_empty") else np.empty(cap, dtype=np.int64)
            if was_pinned:
                pin(ser)
            continue
        if rc == -3:
            raise RuntimeError("pip_solve_dense_dp refused the device-resident buffers (-3): they are on different "
                               "devices, mix host and device memory, or meet an option the host decoder serves")
        if rc != 0:
            raise RuntimeError("pip_solve_dense_dp failed: %d" % rc)
        break
    return dict(status=status, hashes=hashes, ser=ser, ser_off=ser_off, ser_len=ser_len)


def alloc_result(n, words_per_problem=448, pinned=False):
    """caller-owned result buffers for solve_dense(out=...); pinned=True page-locks the quast stream so
    that the device writes it by DMA"""
    cap = words_per_problem * n + 1024
    out = dict(status=np.zeros(n, dtype=np.int32), hashes=np.zeros(n, dtype=np.uint64),
               ser=pinned_empty((cap,), np.int64) if pinned == "alloc" else np.empty(cap, dtype=np.int64),
               ser_off=np.zeros(n + 1, dtype=np.int64), ser_len=np.zeros(n, dtype=np.int64))
    if pinned and pinned != "alloc":
        pin(out["ser"])
    return out


class DeviceBatch:
    """dense batch converted and uploaded once; run() is kernels only."""

    def __init__(self, dom, ctx, bignum=-1, **opts):
        L = lib()
        dom = np.ascontiguousarray(dom, dtype=np.int64)
        self.n, dr, dc = dom.shape
        if ctx is None:
            has, cr, cc, cp = 0, 0, 0, None
        else:
            ctx = np.ascontiguousarray(ctx, dtype=np.int64)
            has, cr, cc = 1, ctx.shape[1], ctx.shape[2]
            cp = ctx.ctypes.data_as(C.c_void_p)
        o = make_options(**opts)
        self.h = L.pip_device_batch_create(C.c_longlong(self.n), dr, dc, dom.ctypes.data_as(C.c_void_p),
                                           has, cr, cc, cp, int(bignum), C.byref(o))
        if not self.h:
            raise RuntimeError("pip_device_batch_create failed")

    def run(self, fetch_cells=False):
        ms = C.c_float(0)
        rc = lib().pip_device_batch_run(self.h, int(fetch_cells), C.byref(ms))
        if rc != 0:
            raise RuntimeError("pip_device_batch_run failed: %d" % rc)
        return float(ms.value)

    def results(self, want_hashes=False):
        status = np.zeros(self.n, dtype=np.int32)
        hashes = np.zeros(self.n, dtype=np.uint64) if want_hashes else None
        rc = lib().pip_device_batch_results(self.h, status.ctypes.data_as(C.c_void_p),
                                            hashes.ctypes.data_as(C.c_void_p) if want_hashes else None)
        if rc != 0:
            raise RuntimeError("pip_device_batch_results failed: %d" % rc)
        return status, hashes

    def close(self):
        if self.h:
            lib().pip_device_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class LargeProblem:
    """one large non-parametric tableau solved by the whole grid (pip_large_*_dp)."""

    def __init__(self, nvar, ni, nq, tab, cut_rows=1024, sol_size=0, maxcol=0):
        tab = np.ascontiguousarray(tab, dtype=np.int64).reshape(ni, nvar + 1)
        self.nvar, self.ni = nvar, ni
        self.cap = max(sol_size, 4096) + 8
        self.h = lib().pip_large_create_dp(nvar, ni, int(nq), tab.ctypes.data_as(C.c_void_p), cut_rows,
                                           sol_size, maxcol)
        if not self.h:
            raise RuntimeError("pip_large_create_dp failed")

    def run(self):
        ms = C.c_float(0)
        if lib().pip_large_run_dp(self.h, C.byref(ms)) != 0:
            raise RuntimeError("pip_large_run_dp failed")
        return float(ms.value)

    def fetch(self):
        st, nc = C.c_int(0), C.c_int(0)
        info = (C.c_longlong * 12)()
        cells = np.zeros(self.cap, dtype=CELL_DTYPE)
        if lib().pip_large_fetch_dp(self.h, C.byref(st), cells.ctypes.data_as(C.c_void_p), self.cap,
                                    C.byref(nc), info) != 0:
            raise RuntimeError("pip_large_fetch_dp failed")
        c = cells[:nc.value]
        return st.value, [[int(x["kind"]), int(x["p1"]), int(x["p2"])] for x in c], \
            dict(pivots=int(info[0]), cuts=int(info[1]), skipped_rows=int(info[2]), ni=int(info[3]),
                 cycles_choice=int(info[4]), cycles_update=int(info[5]),
                 sub=dict(zip(['swap', 'rowpick', 'column', 'det', 'active', 'spare'], [int(info[6 + i]) for i in range(6)])))

    def close(self):
        if self.h:
            lib().pip_large_destroy_dp(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
