"""Per-problem solve reports of dense batches (pip_solve_dense_info_dp, PipProblemInfo_dp): the int64 overflow
flag and the pivot, cut and split counts of every problem, against the oracle's per-problem statistics and
across every route a dense batch can take through the library."""
import ctypes as C
import importlib.util
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("flags", "pivots", "cuts", "splits", "max_rows", "max_cols")


@pytest.fixture(scope="module")
def api():
    from piplib_b200 import api as a
    from piplib_b200 import build
    build.build()
    return a


@pytest.fixture(scope="module")
def port():
    from oracle import pyoracle as po
    po.build(ref=False, port=True)
    return po.Port()


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def overflow_family(n, seed=7, share=0.2, bits=20):
    """loopnest8x12p2 with dense random coefficients below 2^bits in a `share` of the problems: their pivot updates
    leave int64 (most then end in "Integer overflow"); the others are untouched"""
    from workloads import synth
    dom, ctx = synth.generate("loopnest8x12p2", n, seed=seed)
    rng = np.random.default_rng(seed)
    noise = rng.integers(-(1 << bits), 1 << bits, size=dom.shape)
    noise[:, :, 0] = 0
    sel = rng.random(n) < share
    dom = dom.copy()
    dom[sel] += noise[sel]
    return dom, ctx


def _family(name, n, seed):
    from workloads import synth
    if name == "overflow":
        return overflow_family(n, seed=seed) + (-1, {})
    dom, ctx = synth.generate(name, n, seed=seed)
    return dom, ctx, synth.bignum(name), synth.options(name)


def _oracle(port, dom, ctx, bg, **opts):
    """status and PortStats of every problem, from the oracle"""
    from oracle import pyoracle as po
    st, rec = [], []
    for i in range(dom.shape[0]):
        s = po.PortStats()
        st.append(port.solve(dom[i], ctx[i], bg, stats=s, ctx_cols=ctx.shape[2], **opts)[0])
        rec.append((int(s.wrapped > 0), s.pivots, s.cuts_const + s.cuts_parm, s.splits, s.max_rows, s.max_cols))
    return np.array(st), np.array(rec, dtype=np.int64)


def _records(info):
    """[n, 8] int64 of a report array: numpy INFO_DTYPE, or the int32 CUDA tensor of the torch route"""
    if hasattr(info, "cpu"):
        return info.cpu().numpy().view(np.uint32).astype(np.int64)
    return np.stack([info[f].astype(np.int64) for f in FIELDS] + [info["spare"][:, k].astype(np.int64) for k in (0, 1)], axis=1)


def _host(r):
    out = {}
    for k, v in r.items():
        a = v.cpu().numpy() if hasattr(v, "cpu") else v
        out[k] = a.view(np.uint64) if k == "hashes" and a is not None else a
    out["records"] = _records(r["info"])
    return out


def _words(r, i):
    return [int(x) for x in r["ser"][r["ser_off"][i]:r["ser_off"][i] + r["ser_len"][i]]]


def _same(a, b, hashes=True):
    """statuses, hashes and reports of every problem"""
    assert np.array_equal(a["status"], b["status"])
    if hashes:
        assert np.array_equal(a["hashes"], b["hashes"])
    bad = np.nonzero((a["records"] != b["records"]).any(axis=1))[0]
    assert bad.size == 0, [(int(i), a["records"][i].tolist(), b["records"][i].tolist()) for i in bad[:5]]


def _vs_oracle(r, st_o, rec_o):
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    mine = r["records"][:, :6]
    bad = np.nonzero((mine != rec_o).any(axis=1))[0]
    assert bad.size == 0, [(int(i), int(st_o[i]), mine[i].tolist(), rec_o[i].tolist()) for i in bad[:5]]
    assert (r["records"][:, 6:] == 0).all()


def _env(monkeypatch, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)


DEFAULT, STEAL, HANDOVER = {}, dict(PIPLIB_B200_STEAL="1"), dict(PIPLIB_B200_HEAVY_PIVOTS="64")


# ---- 1. counters against the oracle, problem for problem --------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("workload,n,env", [("loopnest16x24p3", 2000, DEFAULT), ("sor1d", 2000, DEFAULT),
                                            ("cg1", 1000, DEFAULT), ("fimmel", 600, DEFAULT), ("test10i", 1500, DEFAULT),
                                            ("boulet", 96, DEFAULT), ("overflow", 1500, DEFAULT),
                                            ("boulet", 96, STEAL), ("overflow", 1500, STEAL), ("fimmel", 600, STEAL),
                                            ("loopnest16x24p3", 2000, STEAL), ("loopnest16x24p3", 2000, HANDOVER),
                                            ("overflow", 1500, HANDOVER)],
                         ids=lambda x: str(x) if isinstance(x, (str, int)) else ("-".join(x) or "default"))
def test_counters_match_the_oracle_per_problem(api, port, workload, n, env, monkeypatch):
    """the flag, pivots, cuts, splits and the largest tableau of every problem equal the oracle's PortStats, fatal
    verdicts included, with the library's defaults (small batches: subtree donation; the tail of a call: the
    hand-over) and with donation or the hand-over forced; their sums equal pip_last_batch_stats_dp of the call"""
    _env(monkeypatch, env)
    dom, ctx, bg, opts = _family(workload, n, seed=31)
    r = _host(api.solve_dense(dom, ctx, bg, want_hashes=True, want_info=True, **opts))
    s = api.last_stats()
    st_o, rec_o = _oracle(port, dom, ctx, bg, **opts)
    _vs_oracle(r, st_o, rec_o)
    rec = r["records"]
    assert (int(s.pivots), int(s.cuts), int(s.splits), int(s.wrapped)) == \
        (int(rec[:, 1].sum()), int(rec[:, 2].sum()), int(rec[:, 3].sum()), int(rec[:, 0].sum()))
    assert (int(s.max_rows), int(s.max_cols)) == (int(rec[:, 4].max()), int(rec[:, 5].max()))
    if workload in ("boulet", "overflow"):
        assert (r["status"] >= 1000).any()                  # the fatal verdicts are really there


# ---- 2. the overflow flag -----------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_overflow_flag_equals_the_batch_flags(api, port, monkeypatch, capsys):
    """info.flags equals pip_last_batch_flags_dp after pip_solve_batch_dp on the same problems, its count
    PipBatchStats_dp.wrapped, and the oracle's wrapped > 0 on every problem"""
    n = 1500
    dom, ctx = overflow_family(n, seed=11)
    r = _host(api.solve_dense(dom, ctx, -1, want_hashes=True, want_info=True))
    flags = r["records"][:, 0]
    wrapped = int(api.last_stats().wrapped)
    assert 0.05 * n <= flags.sum() <= 0.5 * n, int(flags.sum())
    assert wrapped == int(flags.sum())
    api.solve_batch([dict(dom=dom[i], ctx=ctx[i], ctx_cols=ctx.shape[2], bignum=-1) for i in range(n)])
    assert np.array_equal(api.last_flags().astype(np.int64), flags)
    _, rec_o = _oracle(port, dom, ctx, -1)
    differ = np.nonzero(rec_o[:, 0] != flags)[0]
    with capsys.disabled():
        print("\noverflow flag: %d of %d problems flagged; the oracle's wrapped > 0 differs on %d: %s"
              % (int(flags.sum()), n, differ.size, differ[:20].tolist()))
    assert differ.size == 0


# ---- 3. every route gives the same reports --------------------------------------------------------------------------

@pytest.fixture(scope="module")
def loopnest(api):
    from workloads import synth
    n = 20000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=43)
    return dom, ctx


def _plain(api, dom, ctx, bg=-1, **opts):
    return _host(api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, want_info=True, **opts))


@pytest.mark.gpu
def test_host_pinned_and_device_routes(api, torch, loopnest, monkeypatch):
    """pageable host, page-locked host (DMA in and out) and CUDA tensors, and device inputs with host outputs"""
    dom, ctx = loopnest
    n = dom.shape[0]
    base = _plain(api, dom, ctx)
    out = api.alloc_result(n, pinned="alloc")
    pd, pc = api.pinned_copy(dom), api.pinned_copy(ctx)
    try:
        pinned = _host(api.solve_dense(pd, pc, -1, want_hashes=True, want_ser=True, want_info=True, out=out))
        _same(pinned, base)
    finally:
        api.pinned_free(out["ser"]); api.pinned_free(pd); api.pinned_free(pc)
    dd, dc = torch.from_numpy(dom).cuda(), torch.from_numpy(ctx).cuda()
    dev = api.solve_dense(dd, dc, -1, want_hashes=True, want_ser=True, want_info=True)
    assert dev["info"].is_cuda and dev["info"].dtype == torch.int32 and tuple(dev["info"].shape) == (n, 8)
    _same(_host(dev), base)
    again = api.solve_dense(dd, dc, -1, want_hashes=True, want_ser=True, want_info=True, out=dev)
    assert again["info"] is dev["info"]
    _same(_host(again), base)
    # device inputs, host outputs
    st = np.zeros(n, np.int32)
    hs = np.zeros(n, np.uint64)
    info = np.zeros(n, api.INFO_DTYPE)
    rc = api.lib().pip_solve_dense_info_dp(C.c_longlong(n), dom.shape[1], dom.shape[2], C.c_void_p(dd.data_ptr()), 1,
                                           ctx.shape[1], ctx.shape[2], C.c_void_p(dc.data_ptr()), -1,
                                           C.byref(api.make_options()), api._ptr(st), api._ptr(hs), None,
                                           C.c_longlong(0), None, None, api._ptr(info))
    assert rc == 0
    _same(dict(status=st, hashes=hs, records=_records(info)), base)


@pytest.mark.gpu
def test_host_decoder_and_cell_decoder_routes(api, port, loopnest, monkeypatch):
    """Simplify (host decoder on the cells) against the plain run; Maximize / Urs_unknowns / a big parameter (cells
    and the warp decoder) against the host decoder, the CUDA-tensor route and the oracle"""
    dom, ctx = loopnest
    dom, ctx = dom[:4000], ctx[:4000]
    base = _plain(api, dom, ctx)
    simp = _plain(api, dom, ctx, Simplify=1)
    _same(simp, base, hashes=False)
    from workloads import synth
    ex_dom, ex_ctx = synth.generate("expansion", 200, seed=5)
    for d, c, bg, opts in ((dom[:1500], ctx[:1500], -1, dict(Maximize=1)), (dom[:1500], ctx[:1500], -1, dict(Urs_unknowns=1)),
                           (ex_dom, ex_ctx, synth.bignum("expansion"), {})):
        cells = _plain(api, d, c, bg, **opts)
        monkeypatch.setenv("PIPLIB_B200_HOST_DECODE", "1")
        _same(_plain(api, d, c, bg, **opts), cells)
        monkeypatch.delenv("PIPLIB_B200_HOST_DECODE")
        monkeypatch.setenv("PIPLIB_B200_CELL_DECODE", "1")
        _same(_plain(api, d, c, bg, **opts), cells)
        monkeypatch.delenv("PIPLIB_B200_CELL_DECODE")
        st_o, rec_o = _oracle(port, d, c, bg, **opts)
        _vs_oracle(cells, st_o, rec_o)


@pytest.mark.gpu
@pytest.mark.parametrize("env", [dict(PIPLIB_B200_HEAVY_PIVOTS="64"), dict(PIPLIB_B200_STEAL="1"),
                                 dict(PIPLIB_B200_NO_WIDE_SLACK="1", PIPLIB_B200_LARGE_FROM="0")])
def test_handover_donation_and_escalation_routes(api, loopnest, env, monkeypatch):
    """forced hand-over, subtree donation, and size-class escalation with the whole-grid class moved down: the
    reports of the attempt that gave the verdict, as in the plain run"""
    dom, ctx = loopnest
    base = _plain(api, dom, ctx)
    _env(monkeypatch, env)
    _same(_plain(api, dom, ctx), base)


@pytest.mark.gpu
def test_whole_grid_class_reports(api, port, monkeypatch):
    """non-parametric problems that reach the whole-grid class (class L): their reports against the oracle"""
    monkeypatch.setenv("PIPLIB_B200_NO_WIDE_SLACK", "1")
    monkeypatch.setenv("PIPLIB_B200_LARGE_FROM", "0")
    dom, ctx, bg, opts = _family("vivien32", 4, seed=31)
    r = _host(api.solve_dense(dom, ctx, bg, want_hashes=True, want_info=True, **opts))
    st_o, rec_o = _oracle(port, dom, ctx, bg, **opts)
    _vs_oracle(r, st_o, rec_o)


@pytest.mark.gpu
def test_two_devices(api, torch, loopnest, monkeypatch):
    """the chunk queue over two GPUs: reports land by problem index"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    dom, ctx = loopnest
    base = _plain(api, dom, ctx)
    monkeypatch.setenv("PIPLIB_B200_CHUNK", "2048")
    api.set_devices([0, 1])
    try:
        _same(_plain(api, dom, ctx), base)
    finally:
        api.set_devices([])


@pytest.mark.gpu
def test_device_batch_in_three_parts(api):
    """DeviceBatch above 2^19 problems (three parts on lanes of their own): info() of the last run against the
    dense call on the same problems"""
    from workloads import synth
    n = (1 << 19) + 5000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=47)
    base = _host(api.solve_dense(dom, ctx, -1, want_hashes=True, want_info=True))
    db = api.DeviceBatch(dom, ctx, -1)
    try:
        db.run()
        with pytest.raises(RuntimeError):
            db.info()                                   # that run wrote no reports: they were not asked for
        db.keep_info()
        db.run()
        st, hs = db.results(want_hashes=True)
        info = db.info()
    finally:
        db.close()
    _same(dict(status=st, hashes=hs, records=_records(info)), base)


# ---- 4. no behaviour change -------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_info_does_not_change_the_answers(api, loopnest):
    """pip_solve_dense_dp and pip_solve_dense_info_dp on the same inputs: the same statuses, hashes and words"""
    dom, ctx = loopnest
    a = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    b = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True, want_info=True)
    assert np.array_equal(a["status"], b["status"]) and np.array_equal(a["hashes"], b["hashes"])
    assert np.array_equal(a["ser_len"], b["ser_len"]) and a["ser_off"][-1] == b["ser_off"][-1]
    for i in range(dom.shape[0]):
        assert _words(a, i) == _words(b, i)


@pytest.mark.gpu
def test_mixed_placement_is_refused(api, torch, loopnest):
    """a device-resident info beside host outputs, or a host info beside device outputs: -3, nothing written"""
    dom, ctx = loopnest
    dom, ctx = dom[:256], ctx[:256]
    n = dom.shape[0]
    L = api.lib()
    for dev_info in (True, False):
        st = torch.full((n,), -7, dtype=torch.int32, device="cuda") if not dev_info else np.full(n, -7, np.int32)
        info = torch.full((n, 8), -7, dtype=torch.int32, device="cuda") if dev_info else np.full((n, 8), -7, np.int32)
        rc = L.pip_solve_dense_info_dp(C.c_longlong(n), dom.shape[1], dom.shape[2], api._ptr(dom), 1, ctx.shape[1],
                                       ctx.shape[2], api._ptr(ctx), -1, C.byref(api.make_options()), api._ptr(st), None,
                                       None, C.c_longlong(0), None, None, api._ptr(info))
        assert rc == -3
        to_np = lambda a: a.cpu().numpy() if hasattr(a, "cpu") else a
        assert (to_np(st) == -7).all() and (to_np(info) == -7).all()


def _sass_tool():
    spec = importlib.util.spec_from_file_location("sass_digests", os.path.join(ROOT, "tools", "sass_digests.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_solver_kernels_unchanged():
    """no GPU: the solve kernels (every instantiation), the team kernel and the whole-grid kernel compile to the
    instructions recorded in tests/golden/sass_solver_kernels.json (tools/sass_digests.py), as they did before the
    reports existed -- the reports are built from records those kernels already write.  The fingerprints belong to
    one nvcc release: with another one installed the test says so and skips."""
    from piplib_b200 import build
    lib = build.build()
    T = _sass_tool()
    if not (os.path.exists(T.tool("cuobjdump")) and os.path.exists(T.tool("nvcc"))):
        pytest.skip("the CUDA toolkit's nvcc / cuobjdump are not installed")
    with open(T.GOLDEN) as f:
        golden = json.load(f)
    if T.nvcc_release() != golden["nvcc"]:
        pytest.skip("fingerprints recorded with nvcc %s, this is %s" % (golden["nvcc"], T.nvcc_release()))
    mine = T.digests(lib)
    assert len(golden["kernels"]) == 9 and set(mine) == set(golden["kernels"])
    assert {k for k in mine if mine[k] != golden["kernels"][k]} == set()
