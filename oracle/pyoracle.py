"""TEST INFRASTRUCTURE ONLY (never imported by piplib_b200/).

ctypes drivers for
  * oracle/_ref/libpipref.so  -- the unmodified reference + harness (oracle/ref_harness.c)
  * oracle/libpiporacle.so    -- our CPU restatement (oracle/pip_oracle.c)
plus python restatements of the reference's two text printers so that cell streams and
serialised quasts can be compared with the golden .ll files:
  * sol_edit_text      follows source/sol.c:291-422  (CLI output, test/*.ll)
  * quast_print_text   follows source/piplib.c:198-317 (library output, example/*.ll)
and parsers for the two fixture formats (.dat: doc/piplib.texi:570-659, .pip: example/example.c).
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SO = os.path.join(HERE, "_ref", "libpipref.so")
REF_BIG_SO = os.path.join(HERE, "_ref", "libpipref_big.so")     # same sources, SOL_SIZE / MAXCOL raised by -D
PORT_SO = os.path.join(HERE, "libpiporacle.so")

# solution cell kinds, source/sol.c:42-50
FREE, NIL, IF, LIST, FORM, NEW, DIV, VAL, ERROR = range(9)

OPT_NAMES = ["Nq", "Verbose", "Simplify", "Deepest_cut", "Maximize", "Urs_parms",
             "Urs_unknowns", "Compute_dual"]


def build(ref=True, port=True):
    """(re)build the checker libraries; building the checker is not using it."""
    targets = []
    if port:
        targets.append("libpiporacle.so")
    if ref and os.path.isdir("/root/reference/source"):
        targets += ["ref", "refbig"]
    if targets:
        subprocess.check_call(["make", "-s", "-C", HERE] + targets)


def opts_array(**kw):
    o = {"Nq": 1, "Verbose": -1, "Simplify": 0, "Deepest_cut": 0, "Maximize": 0, "Urs_parms": 0,
         "Urs_unknowns": 0, "Compute_dual": 0}
    o.update(kw)
    return (C.c_int * 8)(*[o[k] for k in OPT_NAMES])


def _i64(a):
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a, a.ctypes.data_as(C.POINTER(C.c_longlong))


class _Lib:
    def __init__(self, path):
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = C.CDLL(path)


class Ref(_Lib):
    """the real reference (oracle/_ref)."""

    def __init__(self, big=False):
        super().__init__(REF_BIG_SO if big else REF_SO)
        L = self.lib
        L.pipref_traiter.restype = C.c_int
        L.pipref_solve_ser.restype = C.c_int
        L.pipref_bench_dense.restype = C.c_double

    def traiter(self, nvar, nparm, ni, nc, bigparm, nq, tab, ctx, cap=4096):
        tab_a, tab_p = _i64(np.asarray(tab, dtype=np.int64).reshape(-1))
        ctx_a, ctx_p = _i64(np.asarray(ctx, dtype=np.int64).reshape(-1))
        fl = np.zeros(cap, dtype=np.int32)
        p1 = np.zeros(cap, dtype=np.int64)
        p2 = np.zeros(cap, dtype=np.int64)
        n = C.c_int(0)
        st = self.lib.pipref_traiter(nvar, nparm, ni, nc, bigparm, nq, tab_p, ctx_p,
                                     fl.ctypes.data_as(C.POINTER(C.c_int)),
                                     p1.ctypes.data_as(C.POINTER(C.c_longlong)),
                                     p2.ctypes.data_as(C.POINTER(C.c_longlong)), cap, C.byref(n))
        k = n.value
        cells = [(int(fl[i]), int(p1[i]), int(p2[i])) for i in range(k)]
        return st, cells

    def solve(self, dom, ctx, bg, want_text=False, ctx_cols=None, **opts):
        """dom: 2-D int array (PolyLib rows); ctx: 2-D int array or None."""
        dom = np.asarray(dom, dtype=np.int64)
        dom_a, dom_p = _i64(dom.reshape(-1))
        if ctx is None:
            has, cr, cc = 0, 0, 0
            ctx_a, ctx_p = _i64(np.zeros(0))
        else:
            ctx = np.asarray(ctx, dtype=np.int64)
            if ctx.ndim != 2:
                ctx = ctx.reshape(0, ctx_cols)
            has, cr, cc = 1, ctx.shape[0], ctx.shape[1]
            ctx_a, ctx_p = _i64(ctx.reshape(-1))
        cap = 1 << 20
        ser = np.zeros(cap, dtype=np.int64)
        n = C.c_long(0)
        tcap = 1 << 20
        text = C.create_string_buffer(tcap) if want_text else None
        st = self.lib.pipref_solve_ser(dom.shape[0], dom.shape[1], dom_p, has, cr, cc, ctx_p,
                                       int(bg), opts_array(**opts),
                                       ser.ctypes.data_as(C.POINTER(C.c_longlong)), C.c_long(cap),
                                       C.byref(n), text, C.c_long(tcap if want_text else 0))
        out = [int(x) for x in ser[:n.value]]
        if want_text:
            return st, out, text.value.decode()
        return st, out

    def bench_dense(self, first, count, dom, ctx, bg, **opts):
        """dom: [n, rows, cols] int64; ctx: [n, rows, cols] or None.  -> (seconds, status, hashes)"""
        dom = np.ascontiguousarray(dom, dtype=np.int64)
        n, dr, dc = dom.shape
        if ctx is None:
            has, cr, cc = 0, 0, 0
            ctx_p = None
        else:
            ctx = np.ascontiguousarray(ctx, dtype=np.int64)
            has, cr, cc = 1, ctx.shape[1], ctx.shape[2]
            ctx_p = ctx.ctypes.data_as(C.POINTER(C.c_longlong))
        status = np.zeros(count, dtype=np.int32)
        hashes = np.zeros(count, dtype=np.uint64)
        sec = self.lib.pipref_bench_dense(C.c_long(first), C.c_long(count), dr, dc,
                                          dom.ctypes.data_as(C.POINTER(C.c_longlong)), has, cr, cc,
                                          ctx_p, int(bg), opts_array(**opts),
                                          status.ctypes.data_as(C.POINTER(C.c_int)),
                                          hashes.ctypes.data_as(C.POINTER(C.c_ulonglong)))
        return sec, status, hashes


class PortStats(C.Structure):
    _fields_ = [("pivots", C.c_longlong), ("cuts_const", C.c_longlong), ("cuts_parm", C.c_longlong),
                ("traiter_calls", C.c_longlong), ("compa_rows", C.c_longlong),
                ("splits", C.c_longlong), ("max_rows", C.c_longlong), ("max_cols", C.c_longlong),
                ("max_depth", C.c_longlong), ("elem_updates", C.c_longlong),
                ("max_ctx_rows", C.c_longlong), ("wrapped", C.c_longlong)]


class Port(_Lib):
    """our CPU restatement (oracle/pip_oracle.c)."""

    def __init__(self):
        super().__init__(PORT_SO)
        L = self.lib
        L.piporacle_traiter.restype = C.c_int
        L.piporacle_solve_ser.restype = C.c_int
        L.piporacle_bench_dense.restype = C.c_double

    def traiter(self, nvar, nparm, ni, nc, bigparm, nq, tab, ctx, cap=4096, stats=None,
                sol_size=4096, maxcol=512):
        tab_a, tab_p = _i64(np.asarray(tab, dtype=np.int64).reshape(-1))
        ctx_a, ctx_p = _i64(np.asarray(ctx, dtype=np.int64).reshape(-1))
        cap = max(cap, sol_size)
        fl = np.zeros(cap, dtype=np.int32)
        p1 = np.zeros(cap, dtype=np.int64)
        p2 = np.zeros(cap, dtype=np.int64)
        n = C.c_int(0)
        st_obj = stats if stats is not None else PortStats()
        st = self.lib.piporacle_traiter(nvar, nparm, ni, nc, bigparm, nq, tab_p, ctx_p,
                                        fl.ctypes.data_as(C.POINTER(C.c_int)),
                                        p1.ctypes.data_as(C.POINTER(C.c_longlong)),
                                        p2.ctypes.data_as(C.POINTER(C.c_longlong)), cap,
                                        C.byref(n), C.byref(st_obj), sol_size, maxcol)
        k = n.value
        cells = [(int(fl[i]), int(p1[i]), int(p2[i])) for i in range(min(k, cap))]
        return st, cells

    def solve(self, dom, ctx, bg, stats=None, ctx_cols=None, **opts):
        dom = np.asarray(dom, dtype=np.int64)
        dom_a, dom_p = _i64(dom.reshape(-1))
        if ctx is None:
            has, cr, cc = 0, 0, 0
            ctx_a, ctx_p = _i64(np.zeros(0))
        else:
            ctx = np.asarray(ctx, dtype=np.int64)
            if ctx.ndim != 2:
                ctx = ctx.reshape(0, ctx_cols)
            has, cr, cc = 1, ctx.shape[0], ctx.shape[1]
            ctx_a, ctx_p = _i64(ctx.reshape(-1))
        cap = 1 << 20
        ser = np.zeros(cap, dtype=np.int64)
        n = C.c_long(0)
        st_obj = stats if stats is not None else PortStats()
        st = self.lib.piporacle_solve_ser(dom.shape[0], dom.shape[1], dom_p, has, cr, cc, ctx_p,
                                          int(bg), opts_array(**opts),
                                          ser.ctypes.data_as(C.POINTER(C.c_longlong)), C.c_long(cap),
                                          C.byref(n), C.byref(st_obj))
        return st, [int(x) for x in ser[:n.value]]

    def bench_dense(self, first, count, dom, ctx, bg, **opts):
        dom = np.ascontiguousarray(dom, dtype=np.int64)
        n, dr, dc = dom.shape
        if ctx is None:
            has, cr, cc = 0, 0, 0
            ctx_p = None
        else:
            ctx = np.ascontiguousarray(ctx, dtype=np.int64)
            has, cr, cc = 1, ctx.shape[1], ctx.shape[2]
            ctx_p = ctx.ctypes.data_as(C.POINTER(C.c_longlong))
        status = np.zeros(count, dtype=np.int32)
        hashes = np.zeros(count, dtype=np.uint64)
        stats = PortStats()
        sec = self.lib.piporacle_bench_dense(C.c_long(first), C.c_long(count), dr, dc,
                                             dom.ctypes.data_as(C.POINTER(C.c_longlong)), has, cr, cc,
                                             ctx_p, int(bg), opts_array(**opts),
                                             status.ctypes.data_as(C.POINTER(C.c_int)),
                                             hashes.ctypes.data_as(C.POINTER(C.c_ulonglong)),
                                             C.byref(stats))
        return sec, status, hashes, stats


# ---------------------------------------------------------------------------------------
# fixture parsers
# ---------------------------------------------------------------------------------------

def parse_dat(text):
    """One problem of the CLI format.  Returns dict(comment, nvar, nparm, ni, nc, bigparm, nq,
    tab [ni x ncol], ctx [nc x (nparm+1)]).  The comment is the text echoed by balance_xx
    (source/maind.c:49-61)."""
    i = text.index("(")
    # balance_xx: echo characters until the parenthesis level returns to zero
    level, j, echo = 0, i + 1, []
    while j < len(text):
        c = text[j]
        j += 1
        if c == "(":
            level += 1
        elif c == ")":
            level -= 1
            if level == 0:
                break
        echo.append(c)
    rest = text[j:]
    m = re.match(r"\s*(-?\d+)\s+(-?\d+)\s+(-?\d+)\s+(-?\d+)\s+(-?\d+)\s+(-?\d+)", rest)
    nvar, nparm, ni, nc, bigparm, nq = (int(x) for x in m.groups())
    rows = re.findall(r"\[([^\]]*)\]", rest[m.end():])
    vec = [[int(x) for x in r.split()] for r in rows]
    ncol = nvar + nparm + 1
    tab = vec[:ni]
    ctx = vec[ni:ni + nc]
    assert len(tab) == ni and all(len(r) == ncol for r in tab), "bad tableau rows"
    assert len(ctx) == nc and all(len(r) == nparm + 1 for r in ctx), "bad context rows"
    return dict(comment="".join(echo), nvar=nvar, nparm=nparm, ni=ni, nc=nc, bigparm=bigparm,
                nq=nq, tab=tab, ctx=ctx)


def _read_matrix(lines, pos):
    """pip_matrix_read_xx (source/piplib.c:576-619): skip '#' and blank lines."""
    while True:
        s = lines[pos]
        pos += 1
        st = s.strip()
        if not st or st.startswith("#"):
            continue
        parts = st.split()
        try:
            r, c = int(parts[0]), int(parts[1])
            break
        except (ValueError, IndexError):
            continue
    rows = []
    while len(rows) < r:
        s = lines[pos]
        pos += 1
        st = s.strip()
        if not st or st.startswith("#"):
            continue
        st = st.split("#")[0]
        rows.append([int(x) for x in st.split()[:c]])
    return (r, c, rows), pos


def parse_pip(text):
    """example/example.c input: context matrix, bignum, domain matrix, option keywords."""
    lines = text.split("\n")
    (cr, cc, crow), pos = _read_matrix(lines, 0)
    # fscanf(" %d") for the bignum
    while not lines[pos].strip():
        pos += 1
    bignum = int(lines[pos].split()[0])
    pos += 1
    (dr, dc, drow), pos = _read_matrix(lines, pos)
    opts = {"Nq": 1, "Maximize": 0, "Urs_parms": 0, "Urs_unknowns": 0, "Compute_dual": 0}
    for s in lines[pos:]:
        low = s.lower()
        if low.startswith("maximize"):
            opts["Maximize"] = 1
        if low.startswith("urs_parms"):
            opts["Urs_parms"] = 1
        if low.startswith("urs_unknowns"):
            opts["Urs_unknowns"] = 1
        if low.startswith("rational"):
            opts["Nq"] = 0
        if low.startswith("dual"):
            opts["Compute_dual"] = 1
    bg = bignum
    if bignum > 0:
        bg = bignum + dc - cc          # example/example.c:81-82
    return dict(ctx_shape=[cr, cc], ctx=crow, bignum_raw=bignum, bignum=bg, dom_shape=[dr, dc],
                dom=drow, opts=opts)


# ---------------------------------------------------------------------------------------
# printers
# ---------------------------------------------------------------------------------------

def _cgcd(a, b):
    """llabs(euclid) with C remainder semantics (source/integrer.c:43-50)."""
    import math
    return math.gcd(a, b)


def _val_text(n, d):
    g = _cgcd(n, d)
    if g == d:
        return " %d" % (_cdiv(n, g) if g else 0)
    return " %d/%d" % (_cdiv(n, g), _cdiv(d, g))


def _cdiv(a, b):
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b >= 0) else -q


def sol_edit_text(cells):
    """Text of `while((xq = sol_edit_xx(out, xq)) != q);` (source/maind.c:225) for a cell list."""
    out = []

    def edit(i):
        while True:
            k = cells[i][0]
            if k == FREE:
                i += 1
                continue
            if k == NEW:
                out.append("(newparm %d " % cells[i][1])
                i = edit(i + 1)
                out.append(")\n")
                continue
            break
        k, p1, p2 = cells[i]
        if k == NIL:
            out.append("()\n")
            i += 1
        elif k == ERROR:
            out.append("Error %d\n" % p1)
            i += 1
        elif k == IF:
            out.append("(if ")
            i = edit(i + 1)
            i = edit(i)
            i = edit(i)
            out.append(")\n")
        elif k == LIST:
            out.append("(list ")
            n = p1
            i += 1
            for _ in range(n):
                i = edit(i)
            out.append(")\n")
        elif k == FORM:
            out.append("#[")
            for _ in range(p1):
                i += 1
                out.append(_val_text(cells[i][1], cells[i][2]))
            out.append("]\n")
            i += 1
        elif k == DIV:
            out.append("(div ")
            i = edit(i + 1)
            i = edit(i)
            out.append(")\n")
        elif k == VAL:
            out.append(_val_text(p1, p2))
            i += 1
        else:
            out.append("Inconnu : sol\n")
        return i

    i = 0
    while i != len(cells):
        i = edit(i)
    return "".join(out)


def cli_output_text(comment, status, cells):
    """whole-problem CLI output, source/maind.c:152-231 (status 0 solved / 1 void)."""
    s = "(" + comment
    if status == 0:
        s += ")\n" + sol_edit_text(cells)
    else:
        s += "void\n"
    return s + ")\n"


def quast_print_text(ser):
    """pip_quast_print_xx(stdout, q, 0) (source/piplib.c:290-317) from the serialised stream."""
    out = []
    pos = [0]

    def get():
        v = ser[pos[0]]
        pos[0] += 1
        return v

    def vec():
        n = get()
        s = "#["
        for _ in range(n):
            a, d = get(), get()
            s += " %d" % a
            if d != 1:
                s += "/%d" % d
        return s + "]"

    def node(ind):
        nn = get()
        if nn == -1:
            out.append(" " * max(ind, 0) + "void\n")
            return
        for _ in range(nn):
            rank, deno = get(), get()
            out.append(" " * ind + "(newparm %d (div %s %d))\n" % (rank, vec(), deno))
        kind = get()
        if kind == 2:
            out.append(" " * ind + "(if " + vec() + "\n")
            node(ind + 1)
            node(ind + 1)
            out.append(" " * ind + ")\n")
        elif kind == 1:
            out.append(" " * ind + "(list\n")
            for _ in range(get()):
                if get():
                    out.append(" " * (ind + 1) + vec() + "\n")
            out.append(" " * ind + ")\n")
            if get():
                node(ind + 1)
        else:
            out.append(" " * ind + "()\n")

    node(0)
    assert pos[0] == len(ser), "trailing words in serialised quast"
    return "".join(out)


def example_output_text(p, ser):
    """full stdout of example/example.c (non-tty) for a parsed .pip and its solution."""
    def mat(shape, rows):
        s = "%d %d\n" % (shape[0], shape[1])
        for r in rows:
            s += "".join(" %d" % x for x in r) + "\n"
        return s
    s = "[PIP2-like future input] Please enter:\n- the context matrix,\n"
    s += mat(p["ctx_shape"], p["ctx"])
    s += "- the bignum column (start at 0, -1 if no bignum),\n%d\n" % p["bignum_raw"]
    s += "- the constraint matrix.\n" + mat(p["dom_shape"], p["dom"]) + "\n"
    return s + quast_print_text(ser)


def strip_ws_lines(text):
    """`diff -w` view: per line, all blanks removed; empty lines dropped."""
    return [re.sub(r"\s+", "", ln) for ln in text.split("\n") if re.sub(r"\s+", "", ln)]
