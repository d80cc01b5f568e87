"""Parity of the CUDA path (through the C-ABI) with the reference: golden .ll files, live
reference answers recorded in tests/golden/, and the oracle on seeded synthetic batches."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

from conftest import load_golden
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

CLI = [c for c in load_golden("cli_suite.json") if "pipFile_1" not in c["name"]]
LIB = load_golden("lib_suite.json")
RLIB = load_golden("random_lib.json")
RCLI = load_golden("random_cli.json")
OPTS = load_golden("options_suite.json")


@pytest.fixture(scope="module")
def api():
    from piplib_b200 import api as a
    from piplib_b200 import build
    build.build()
    return a


def test_cli_suite(api):
    """test/*.dat (+challenges) in ONE batch: cells bit-exact, text token-exact vs the .ll"""
    out = api.traiter_batch(CLI)
    bad = []
    for c, (st, cells) in zip(CLI, out):
        if st != c["ref_status"] or cells != c["ref_cells"]:
            bad.append((c["name"], st, c["ref_status"], len(cells), len(c["ref_cells"])))
        elif c["golden_ll"] is not None:
            text = po.cli_output_text(c["comment"], st, [tuple(x) for x in cells])
            if po.strip_ws_lines(text) != po.strip_ws_lines(c["golden_ll"]):
                bad.append((c["name"], "text"))
    assert not bad, bad


def _norm(r):
    """pip_solve returns NULL for an empty context without any error: the reference harness
    reports that as status 0 + the one-word stream [-1]; our batch API says status 1 (VOID)."""
    st, ser = r
    return (0 if st == 1 else st, ser)


def _lib_problem(c):
    return dict(dom=c["dom"], ctx=c["ctx"], ctx_cols=c["ctx_shape"][1] if c["ctx_shape"] else None,
                bignum=c["bignum"])


def test_lib_suite(api):
    """example/*.pip and the option variants (Maximize, Urs_*, Rational, Simplify)"""
    bad = []
    for c in LIB:
        st, ser = _norm(api.solve_batch([_lib_problem(c)], **c["opts"])[0])
        if st != c["ref_status"] or ser != c["ref_ser"]:
            bad.append((c["name"], st))
        elif c["golden_ll"] is not None:
            text = po.example_output_text(c, ser)
            if po.strip_ws_lines(text) != po.strip_ws_lines(c["golden_ll"]):
                bad.append((c["name"], "text"))
    assert not bad, bad


def test_pip_solve_and_printer(api):
    """the reference call sequence of example/example.c:84-92 on example/max.pip"""
    c = [x for x in LIB if x["name"] == "max"][0]
    L = api.lib()
    libc = C.CDLL(None)
    libc.fopen.restype = C.c_void_p
    libc.fclose.argtypes = [C.c_void_p]
    dom = np.asarray(c["dom"], dtype=np.int64)
    d = api._matrix(dom.shape[0], dom.shape[1], dom)
    x = api._matrix(c["ctx_shape"][0], c["ctx_shape"][1], np.zeros(0))
    o = L.pip_options_init_dp()
    q = L.pip_solve_dp(d, x, c["bignum"], o)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "out.txt").encode()
        f = libc.fopen(path, b"w")
        L.pip_quast_print_dp(C.c_void_p(f), C.c_void_p(q), 0)
        libc.fclose(C.c_void_p(f))
        text = open(path).read()
    assert text == po.quast_print_text(c["ref_ser"])
    L.pip_quast_free_dp(q)
    L.pip_options_free_dp(o)
    L.pip_matrix_free_dp(d)
    L.pip_matrix_free_dp(x)


def test_random_lib(api):
    groups = {}
    for c in RLIB:
        groups.setdefault(tuple(sorted(c["opts"].items())), []).append(c)
    bad = []
    for opts, cases in groups.items():
        out = api.solve_batch([_lib_problem(c) for c in cases], **dict(opts))
        bad += [c["name"] for c, r in zip(cases, out) if _norm(r) != (c["ref_status"], c["ref_ser"])]
    assert not bad, bad


def test_options_suite(api):
    """Deepest_cut (device: Gondran's multiplier on constant cuts) and Compute_dual (device: row
    positions tracked through the entry sort, dual list at the leaf; host: equalities post-pass)
    against live answers of the reference; batch entry point and the dense entry point"""
    groups = {}
    for c in OPTS:
        groups.setdefault(tuple(sorted(c["opts"].items())), []).append(c)
    bad = []
    for opts, cases in groups.items():
        out = api.solve_batch([_lib_problem(c) for c in cases], **dict(opts))
        bad += [(c["name"], r[0]) for c, r in zip(cases, out) if _norm(r) != (c["ref_status"], c["ref_ser"])]
    assert not bad, bad
    # dense entry point: same shapes batched together, serialised stream word for word
    dense = {}
    for c in OPTS:
        if c["ctx"] is None or c["ctx_shape"] is None:
            dense.setdefault((tuple(c["dom_shape"]), tuple(sorted(c["opts"].items()))), []).append(c)
    checked = 0
    for (shape, opts), cases in dense.items():
        dom = np.asarray([c["dom"] for c in cases], dtype=np.int64).reshape(len(cases), *shape)
        r = api.solve_dense(dom, None, -1, want_hashes=True, want_ser=True, **dict(opts))
        for k, c in enumerate(cases):
            st = int(r["status"][k])
            mine = [int(x) for x in r["ser"][r["ser_off"][k]:r["ser_off"][k] + r["ser_len"][k]]]
            assert (0 if st == 1 else st) == c["ref_status"], c["name"]
            if c["ref_status"] == 0:
                assert mine == c["ref_ser"], c["name"]
            checked += 1
    assert checked > 50


def test_random_cli(api):
    out = api.traiter_batch(RCLI)
    bad = [(c["name"], st, c["ref_status"]) for c, (st, cells) in zip(RCLI, out)
           if st != c["ref_status"] or cells != c["ref_cells"]]
    assert not bad, bad


def test_batch_equals_singles(api):
    """pip_solve_batch must give the same trees as n sequential pip_solve calls"""
    cases = [c for c in LIB if c["opts"] == {"Nq": 1, "Maximize": 0, "Urs_parms": 0,
                                             "Urs_unknowns": 0, "Compute_dual": 0}]
    one = api.solve_batch([_lib_problem(c) for c in cases])
    for c, r in zip(cases, one):
        assert _norm(r) == _norm(api.solve_batch([_lib_problem(c)])[0]) == (c["ref_status"], c["ref_ser"])


@pytest.mark.parametrize("workload,n", [("loopnest16x24p3", 3000), ("loopnest8x12p2", 6000)])
def test_dense_batch_vs_oracle(api, port, workload, n):
    """seeded synthetic batch of the bench workload: status + quast hash per problem vs the oracle,
    and the serialised stream of a few problems word for word"""
    from workloads import synth
    dom, ctx = synth.generate(workload, n, seed=77)
    _, st_o, h_o, stats = port.bench_dense(0, n, dom, ctx, -1)
    r = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    ok = st_o == 0
    assert np.array_equal(r["hashes"][ok], h_o[ok])
    s = api.last_stats()
    if not (st_o >= 1000).any():                          # (a fatal verdict under donation leaves partial counters)
        assert int(s.pivots) == int(stats.pivots)        # same pivots, sub-solves included
    for i in range(0, n, max(1, n // 20)):
        st, ser = port.solve(dom[i], ctx[i], -1)
        mine = [int(x) for x in r["ser"][r["ser_off"][i]:r["ser_off"][i] + r["ser_len"][i]]]
        assert (st, ser) == (int(st_g[i]), mine) or st != 0


@pytest.mark.parametrize("workload,n", [("sor1d", 4000), ("cg1", 3000), ("fimmel", 1500), ("esced", 2000),
                                        ("expansion", 300), ("boulet", 48), ("test10i", 3000),
                                        ("test12i", 1500), ("vivien32", 24)])
def test_config3_and_5_families_vs_oracle(api, port, workload, n, monkeypatch):
    """BASELINE configs 3 (cut-heavy: test<N>i-shaped, vivien32-shaped) and 5 (dependence-analysis
    shapes with perturbed constants): status, quast hash and pivot count vs the oracle"""
    from workloads import synth
    # (pivot totals are compared: subtree donation -- tested on its own below -- leaves the counters of problems
    # that end in a fatal verdict partial, because the segments after the fatal point ran anyway or not at all)
    monkeypatch.setenv("PIPLIB_B200_STEAL", "0")
    monkeypatch.setenv("PIPLIB_B200_HEAVY_PIVOTS", "0")        # (the hand-over ends in a donation launch)
    dom, ctx = synth.generate(workload, n, seed=31)
    bg, opts = synth.bignum(workload), synth.options(workload)
    _, st_o, h_o, stats = port.bench_dense(0, n, dom, ctx, bg, **opts)
    r = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts)
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    ok = st_o == 0
    assert np.array_equal(r["hashes"][ok], h_o[ok])
    assert int(api.last_stats().pivots) >= int(stats.pivots)     # > only if a class was re-run
    for i in range(0, n, max(1, n // 8)):
        st, ser = port.solve(dom[i], ctx[i], bg, ctx_cols=ctx.shape[2], **opts)
        mine = [int(x) for x in r["ser"][r["ser_off"][i]:r["ser_off"][i] + r["ser_len"][i]]]
        assert (st, ser) == (int(st_g[i]), mine) or st != 0


def test_dense_batch_with_varying_equality_rows(api, port):
    """the dense path plans a chunk from its first problem (same shape assumed for all) and checks the
    assumption while converting: a batch where the number of equality rows varies from problem to
    problem must fall back to the exact plan and still match the oracle"""
    from workloads import synth
    n = 1500
    dom, ctx = synth.generate("loopnest8x12p2", n, seed=11)
    dom = dom.copy()
    rng = np.random.default_rng(5)
    for i in range(n):                       # turn 0..2 inequality rows of every second problem into equalities
        if i % 2:
            for r in rng.choice(dom.shape[1], size=int(rng.integers(0, 3)), replace=False):
                dom[i, r, 0] = 0
    _, st_o, h_o, stats = port.bench_dense(0, n, dom, ctx, -1)
    r = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    ok = st_o == 0
    assert ok.sum() > n // 8
    assert np.array_equal(r["hashes"][ok], h_o[ok])


def test_device_resident_batch(api, port):
    """kernel-only path (inputs resident in HBM) gives the same answers as the host-buffer path"""
    from workloads import synth
    dom, ctx = synth.generate("loopnest8x12p2", 4000, seed=5)
    db = api.DeviceBatch(dom, ctx, -1)
    ms = db.run(True)
    st, h = db.results(True)
    r = api.solve_dense(dom, ctx, -1)
    assert ms > 0 and np.array_equal(st, r["status"]) and np.array_equal(h, r["hashes"])
    db.close()


def test_device_job_in_parts(api, monkeypatch):
    """a device-resident job above 2^19 problems runs as parts of falling size on engine lanes of their own (the
    tail of a part is filled by the next one): statuses, hashes and counters equal to the one-launch job"""
    from workloads import synth
    n = 600000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=2026)
    db = api.DeviceBatch(dom, ctx, -1)
    monkeypatch.setenv("PIPLIB_B200_DEVICE_PARTS", "1")
    db.run(False)
    one = api.last_stats()
    st1, h1 = db.results(True)
    for parts in ("6", "3"):
        monkeypatch.setenv("PIPLIB_B200_DEVICE_PARTS", parts)
        for rep in range(2):
            ms = db.run(False)
            s = api.last_stats()
            st, h = db.results(True)
            assert ms > 0 and np.array_equal(st, st1) and np.array_equal(h, h1)
            assert s.launches >= 3 * int(parts) and abs(int(s.pivots) - int(one.pivots)) < int(one.pivots) // 1000
    db.close()
    r = api.solve_dense(dom[:50000], ctx[:50000], -1)
    assert np.array_equal(st1[:50000], r["status"]) and np.array_equal(h1[:50000], r["hashes"])


def test_large_tableau_kernel_fixtures(api):
    """grid-per-problem cooperative kernel on every non-parametric fixture (incl. 260 cuts)"""
    cases = [c for c in load_golden("cli_suite.json")
             if c["nparm"] == 0 and c["nc"] == 0 and "sysmo" not in c["name"]]
    cases += [c for c in RCLI if c["nparm"] == 0 and c["nc"] == 0][:40]
    bad = []
    for c in cases:
        p = api.LargeProblem(c["nvar"], c["ni"], c["nq"], c["tab"], cut_rows=400)
        p.run()
        st, cells, info = p.fetch()
        p.close()
        if st != c["ref_status"] or cells != c["ref_cells"]:
            bad.append((c["name"], st, c["ref_status"], len(cells), len(c["ref_cells"])))
    assert not bad, bad


@pytest.mark.parametrize("n", [256, 768])
def test_large_tableau_consecutive_ones(api, port, n):
    """config-4 shaped problem (totally unimodular rows) vs the oracle with raised limits"""
    from workloads import synth
    tab = synth.consecutive_ones(n, n, seed=11)
    st_o, cells_o = port.traiter(n, 0, n, 0, -1, 1, tab, [], sol_size=1 << 16, maxcol=1 << 14)
    p = api.LargeProblem(n, n, 1, tab, cut_rows=256, sol_size=1 << 16, maxcol=1 << 14)
    ms = p.run()
    st, cells, info = p.fetch()
    ms2 = p.run()                                   # the run is repeatable (tableau restored)
    st2, cells2, _ = p.fetch()
    p.close()
    assert ms > 0 and ms2 > 0
    assert st == st_o and [tuple(x) for x in cells] == cells_o
    assert (st2, cells2) == (st, cells) and info["pivots"] > 0


def test_int32_and_int64_instantiations_agree_at_scale(api, port, monkeypatch):
    """200 000 problems of the bench workload: the int32-storage kernel (class S32, widen-and-rerun)
    and the int64 kernel give the same status, quast hash and serialised stream for every problem;
    a 2000-problem sample is checked against the oracle; pivot totals agree"""
    from workloads import synth
    n = 200000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=2026)
    monkeypatch.setenv("PIPLIB_B200_HEAVY_PIVOTS", "0")     # pivot totals are compared: no donation launch
    a = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    piv_a = int(api.last_stats().pivots)
    monkeypatch.setenv("PIPLIB_B200_NO_INT32", "1")
    monkeypatch.setenv("PIPLIB_B200_HOST_DECODE", "1")       # also crosses device vs host decoder
    b = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    piv_b = int(api.last_stats().pivots)
    assert np.array_equal(a["status"], b["status"]) and np.array_equal(a["hashes"], b["hashes"])
    assert np.array_equal(a["ser_len"], b["ser_len"])
    assert piv_a >= piv_b          # the int32 pass re-runs the few widened problems
    for i in range(0, n, 997):
        x = a["ser"][a["ser_off"][i]:a["ser_off"][i] + a["ser_len"][i]]
        y = b["ser"][b["ser_off"][i]:b["ser_off"][i] + b["ser_len"][i]]
        assert np.array_equal(x, y)
    m = 2000
    _, st_o, h_o, _ = port.bench_dense(0, m, dom[:m], ctx[:m], -1)
    st_g = np.where(a["status"][:m] == 1, 0, a["status"][:m])
    assert np.array_equal(st_g, st_o) and np.array_equal(a["hashes"][:m][st_o == 0], h_o[st_o == 0])


def test_edge_cases(api, port):
    """empty batch, a problem without rows, no unknowns, a context without rows"""
    assert api.traiter_batch([]) == []
    r = api.solve_dense(np.zeros((0, 3, 4), dtype=np.int64), None, -1)
    assert r["status"].shape == (0,)
    # no constraints at all: every unknown is 0
    st, ser = api.solve(np.zeros((0, 4), dtype=np.int64).reshape(0, 4), None, -1)
    assert (st, ser) == port.solve(np.zeros((0, 4), dtype=np.int64), None, -1)
    # parameters but an empty context (0 x Np+2 matrix, doc/piplib.texi:2097-2102)
    st, ser = api.solve([[1, 1, -1, 0]], np.zeros((0, 3), dtype=np.int64), -1, ctx_cols=3)
    assert (st, ser) == port.solve([[1, 1, -1, 0]], np.zeros((0, 3), dtype=np.int64), -1, ctx_cols=3)


@pytest.mark.parametrize("knob", ["PIPLIB_B200_HOST_DECODE", "PIPLIB_B200_EXACT_PLAN",
                                  "PIPLIB_B200_NO_INT32", "PIPLIB_B200_NO_WIDE_SLACK", "PIPLIB_B200_NO_TMA"])
def test_alternative_paths_give_the_same_answers(api, port, monkeypatch, knob):
    """every run-time knob of INTEGRATION.md section 7 selects another route to the same answer: the
    host decoder, the exact planning pass, the int64 shared-memory class,
    the narrow capacity slack, the large kernel without shared-memory staging"""
    from workloads import synth
    monkeypatch.setenv(knob, "1")
    n = 1500
    dom, ctx = synth.generate("loopnest8x12p2", n, seed=23)
    _, st_o, h_o, stats = port.bench_dense(0, n, dom, ctx, -1)
    r = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    assert np.array_equal(r["hashes"][st_o == 0], h_o[st_o == 0])
    for i in range(0, n, n // 10):
        st, ser = port.solve(dom[i], ctx[i], -1)
        mine = [int(x) for x in r["ser"][r["ser_off"][i]:r["ser_off"][i] + r["ser_len"][i]]]
        assert (st, ser) == (int(st_g[i]), mine) or st != 0
    m = 160
    tab = synth.consecutive_ones(m, m, seed=9)
    st_l, cells_l = port.traiter(m, 0, m, 0, -1, 1, tab, [])
    lp = api.LargeProblem(m, m, 1, tab, cut_rows=64)
    lp.run()
    st, cells, info = lp.fetch()
    lp.close()
    assert st == st_l and [tuple(x) for x in cells] == cells_l


def test_ladder_hands_stragglers_to_the_grid_kernel(api, monkeypatch):
    """the last few non-parametric problems of a batch that reach the big global-memory classes are
    solved by the whole-grid kernel (class L) instead of one CTA each: same cells.  The hand-over
    point is moved down so that the heavy fixtures (vivien32: 260 cuts, the test<N>i chains) take it."""
    cases = [c for c in CLI if c["nparm"] == 0 and c["nc"] == 0 and c["ref_status"] == 0
             and len(c["tab"]) and "sysmo" not in c["name"]]
    heavy = [c for c in cases if "vivien" in c["name"]] + [c for c in cases if c["name"] in ("test12i", "test11i")]
    assert heavy
    monkeypatch.setenv("PIPLIB_B200_LARGE_FROM", "0")
    for c in heavy:
        (st, cells), = api.traiter_batch([c])
        stats = api.last_stats()
        assert (st, cells) == (c["ref_status"], c["ref_cells"]), c["name"]
    monkeypatch.setenv("PIPLIB_B200_LARGE_FROM", "-1")
    (st, cells), = api.traiter_batch([heavy[0]])
    assert (st, cells) == (heavy[0]["ref_status"], heavy[0]["ref_cells"])


# ---- parity at the sizes the bench quotes (VERDICT r1: "headline sizes are not parity-checked") ----

def test_full_bench_batch_vs_reference(api):
    """BASELINE config 2 at its full size: the WHOLE 10^6-problem loopnest16x24p3 batch of bench.py
    (seed 2026) through pip_solve_dense_dp against the unmodified reference (oracle/_ref, one process
    per host core): status and quast hash of every problem; total pivots against the oracle port."""
    from oracle import cpu_arm as ca
    from workloads import synth
    n = 1000000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=2026)
    r = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=False)
    piv_gpu = int(api.last_stats().pivots)
    ref = ca.cpu_arm(dom, ctx, n)
    assert ref["n"] == n
    assert ca.same_answers(r["status"], r["hashes"], ref), "GPU differs from the %s on the full batch" % ref["kind"]
    port = ca.cpu_arm(dom, ctx, n, kind="port")
    assert ca.same_answers(r["status"], r["hashes"], port)
    # the int32 class re-runs the few problems it hands to the int64 class: their pivots count twice
    assert piv_gpu >= port["pivots"] and piv_gpu - port["pivots"] < port["pivots"] // 1000


def test_c5_family_full_batch_vs_reference(api):
    """BASELINE config 5 family (sor1d-shaped, perturbed constants) at 10^6 problems, every problem
    against the unmodified reference"""
    from oracle import cpu_arm as ca
    from workloads import synth
    n = 1000000
    dom, ctx = synth.generate("sor1d", n, seed=2026)
    bg, opts = synth.bignum("sor1d"), synth.options("sor1d")
    r = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=False, **opts)
    ref = ca.cpu_arm(dom, ctx, n, bg=bg, opts=opts)
    assert ca.same_answers(r["status"], r["hashes"], ref)


def test_large_tableau_4096_vs_reference_golden(api):
    """BASELINE config 4 at its full size (4096 x 4097, the tableau bench.py times): cells and status
    identical to the unmodified reference built with raised limits (tests/golden/
    large_consecutive_ones_4096.json, tools/make_golden_large.py), pivot count identical to the oracle
    port's"""
    from workloads import synth
    g = load_golden("large_consecutive_ones_4096.json")
    n = g["n"]
    tab = synth.consecutive_ones(n, n, seed=g["seed"])
    p = api.LargeProblem(n, n, g["nq"], tab, cut_rows=1024, sol_size=1 << 20, maxcol=1 << 16)
    p.run()
    st, cells, info = p.fetch()
    p.close()
    assert st == g["status"] and info["pivots"] == g["pivots"] and info["cuts"] == g["cuts"]
    assert cells == g["cells"]


# ---- pinned caller buffers: DMA + device-side input conversion (SURVEY.md 8 f1) ----------------------

def _words(r, i):
    return [int(x) for x in r["ser"][r["ser_off"][i]:r["ser_off"][i] + r["ser_len"][i]]]


def _dense_equal(a, b, n):
    assert np.array_equal(a["status"], b["status"]) and np.array_equal(a["hashes"], b["hashes"])
    assert np.array_equal(a["ser_len"], b["ser_len"])
    for i in range(0, n, max(1, n // 200)):
        assert _words(a, i) == _words(b, i)


@pytest.mark.parametrize("workload,n", [("loopnest16x24p3", 40000), ("sor1d", 30000), ("fimmel", 2000)])
def test_pinned_buffers_dma_path_vs_oracle(api, port, workload, n, monkeypatch):
    """caller arrays in page-locked memory: raw PolyLib rows go up by DMA and tab_Matrix2Tableau runs as a
    kernel, the quasts come down straight into the caller's stream.  Against the oracle, and word for
    word against the pageable (host conversion, staged output) route and the two mixed routes."""
    from workloads import synth
    monkeypatch.setenv("PIPLIB_B200_CHUNK", "8192")          # several chunks, several lanes
    dom, ctx = synth.generate(workload, n, seed=41)
    bg, opts = synth.bignum(workload), synth.options(workload)
    base = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts)        # pageable
    api.pin(dom), api.pin(ctx)
    try:
        out = api.alloc_result(n, pinned=True)
        r = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, out=out, **opts)
        assert int(api.last_stats().h2d_bytes) >= dom.nbytes              # the raw rows really went up
        m = min(n, 6000)
        _, st_o, h_o, _ = port.bench_dense(0, m, dom[:m], ctx[:m], bg, **opts)
        st_g = np.where(r["status"][:m] == 1, 0, r["status"][:m])
        assert np.array_equal(st_g, st_o) and np.array_equal(r["hashes"][:m][st_o == 0], h_o[st_o == 0])
        for i in range(0, m, max(1, m // 10)):
            st, ser = port.solve(dom[i], ctx[i], bg, ctx_cols=ctx.shape[2], **opts)
            assert (st, ser) == (int(st_g[i]), _words(r, i)) or st != 0
        _dense_equal(r, base, n)
        monkeypatch.setenv("PIPLIB_B200_STAGED_OUT", "1")      # device conversion, staged output
        _dense_equal(api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts), base, n)
        monkeypatch.delenv("PIPLIB_B200_STAGED_OUT")
        monkeypatch.setenv("PIPLIB_B200_HOST_CONVERT", "1")    # host conversion, DMA output
        out2 = api.alloc_result(n, pinned=True)
        _dense_equal(api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, out=out2, **opts), base, n)
        api.unpin(out["ser"]), api.unpin(out2["ser"])
    finally:
        api.unpin(dom), api.unpin(ctx)


def test_device_conversion_column_surgery(api):
    """the option variants of every example (Maximize / Urs_parms / Urs_unknowns / big parameter: Shift,
    bignum and Urs column synthesis of tab_Matrix2Tableau, source/tab.c:292-393) through the device-side
    conversion: one-problem dense batches in pinned memory against the reference's serialised quasts"""
    checked = 0
    for c in LIB:
        if c["opts"].get("Simplify"):
            continue                              # host-only post-pass: takes the staged route anyway
        dom = np.ascontiguousarray(np.asarray(c["dom"], dtype=np.int64).reshape(1, *c["dom_shape"]))
        ctx = None
        if c["ctx_shape"] is not None:
            ctx = np.ascontiguousarray(np.asarray(c["ctx"], dtype=np.int64).reshape(1, *c["ctx_shape"]))
        if dom.size == 0:
            continue
        api.pin(dom)
        if ctx is not None and ctx.size:
            api.pin(ctx)
        try:
            r = api.solve_dense(dom, ctx, c["bignum"], want_hashes=True, want_ser=True, **c["opts"])
        finally:
            api.unpin(dom)
            if ctx is not None and ctx.size:
                api.unpin(ctx)
        st = int(r["status"][0])
        assert (0 if st == 1 else st) == c["ref_status"], c["name"]
        if c["ref_status"] == 0:
            assert _words(r, 0) == c["ref_ser"], c["name"]
        checked += 1
    assert checked > 60


def test_device_conversion_equalities_and_wide_inputs(api, port):
    """pinned route: a batch whose number of equality rows varies from problem to problem (the device
    counts them; the pool reserves the worst case), and inputs that leave int32 (the int32 pool flags
    them, the int64 pool is built on demand)"""
    from workloads import synth
    n = 3000
    dom, ctx = synth.generate("loopnest8x12p2", n, seed=13)
    dom = dom.copy()
    rng = np.random.default_rng(9)
    for i in range(n):
        if i % 2:
            for r in rng.choice(dom.shape[1], size=int(rng.integers(0, 3)), replace=False):
                dom[i, r, 0] = 0
        if i % 97 == 5:
            dom[i, int(rng.integers(0, dom.shape[1])), -1] += (1 << 40)      # a constant beyond int32
    dom = np.ascontiguousarray(dom)
    _, st_o, h_o, _ = port.bench_dense(0, n, dom, ctx, -1)
    api.pin(dom), api.pin(ctx)
    try:
        r = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    finally:
        api.unpin(dom), api.unpin(ctx)
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    ok = st_o == 0
    assert ok.sum() > n // 8 and np.array_equal(r["hashes"][ok], h_o[ok])


def test_one_call_over_several_gpus(api, port):
    """pip_set_devices_dp: one pip_solve_dense_dp call spreads its chunks over every visible GPU through
    a shared queue; the caller's arrays come back as from one device"""
    import torch
    ng = torch.cuda.device_count()
    if ng < 2:
        pytest.skip("needs at least two GPUs")
    from workloads import synth
    n = 60000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=19)
    one = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    api.set_devices(list(range(ng)))
    os.environ["PIPLIB_B200_CHUNK"] = "4096"
    try:
        for pinned in (False, True):
            if pinned:
                api.pin(dom), api.pin(ctx)
            out = api.alloc_result(n, pinned=pinned)
            r = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True, out=out)
            _dense_equal(r, one, n)
            if pinned:
                api.unpin(dom), api.unpin(ctx), api.unpin(out["ser"])
    finally:
        api.set_devices([])
        del os.environ["PIPLIB_B200_CHUNK"]


def test_reference_example_program_runs_on_our_library(api, tmp_path):
    """the reference's own caller (example/example.c: tests/fixtures/example.c compiled against include/ and
    linked with libpiplib_dp.so) replays every example/*.pip and its option variants: stdout must be the
    reference's .ll text (prompts, echoed matrices, pip_quast_print)"""
    import subprocess
    from test_cabi import build_example
    exe = build_example(api.LIB_PATH, tmp_path)
    flags = {"Maximize": "Maximize", "Urs_parms": "Urs_parms", "Urs_unknowns": "Urs_unknowns", "Compute_dual": "Dual"}

    def mat(shape, rows):
        return "%d %d\n" % tuple(shape) + "".join(" ".join(str(v) for v in r) + "\n" for r in rows)
    checked, bad = 0, []
    for c in LIB:
        if c["golden_ll"] is None or c["opts"].get("Simplify") or c["ref_status"] != 0:
            continue
        text = mat(c["ctx_shape"], c["ctx"]) + "%d\n" % c["bignum_raw"] + mat(c["dom_shape"], c["dom"]) + "\n"
        for k, word in flags.items():
            if c["opts"].get(k):
                text += word + "\n"
        if not c["opts"].get("Nq", 1):
            text += "Rational\n"
        r = subprocess.run([exe], input=text, capture_output=True, text=True, timeout=120)
        if r.returncode != 0 or po.strip_ws_lines(r.stdout) != po.strip_ws_lines(c["golden_ll"]):
            bad.append((c["name"], r.returncode, r.stderr[-200:]))
        checked += 1
    assert checked >= 15 and not bad, bad[:4]


@pytest.mark.parametrize("workload,n", [("boulet", 96), ("fimmel", 600), ("loopnest16x24p3", 3000), ("expansion", 200)])
def test_subtree_donation_on_the_device(api, port, workload, n, monkeypatch):
    """subtree donation (PipSteal): idle warps claim the ELSE branches other warps offer, solve them as separate
    segments, the copy kernel splices the segments in pre-order -- a small batch of heavy parametric trees, so
    that most warps are idle and claims really happen; status and quast hash of every problem against the
    oracle, serialised streams word for word against the undonated run"""
    from workloads import synth
    dom, ctx = synth.generate(workload, n, seed=37)
    bg, opts = synth.bignum(workload), synth.options(workload)
    monkeypatch.setenv("PIPLIB_B200_STEAL", "0")
    base = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts)
    monkeypatch.setenv("PIPLIB_B200_STEAL", "1")
    claims = 0
    for rep in range(3):                               # claims depend on timing: a few runs, all must agree
        r = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts)
        _dense_equal(r, base, n)
    _, st_o, h_o, _ = port.bench_dense(0, n, dom, ctx, bg, **opts)
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    ok = st_o == 0
    assert np.array_equal(r["hashes"][ok], h_o[ok])


@pytest.mark.parametrize("budget", ["8", "64", "1024"])
def test_heavy_problem_handover_on_the_device(api, port, budget, monkeypatch):
    """heavy-problem hand-over (PipLaunch::budget): problems past the pivot budget stop at their next split in
    the bulk launch and are solved from scratch by the donation launch that follows on the same stream.  With a
    tiny budget the list fills to its cap; streams word for word against the run without hand-over, statuses
    and hashes against the oracle.  (Pivot totals are not compared: for an exit(26) problem they count what ran
    before the verdict, which depends on who solved which subtree.)"""
    from workloads import synth
    n = 40000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=41)
    bg, opts = synth.bignum("loopnest16x24p3"), synth.options("loopnest16x24p3")
    monkeypatch.setenv("PIPLIB_B200_STEAL", "0")
    monkeypatch.setenv("PIPLIB_B200_HEAVY_PIVOTS", "0")
    base = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts)
    monkeypatch.delenv("PIPLIB_B200_STEAL")
    monkeypatch.setenv("PIPLIB_B200_HEAVY_PIVOTS", budget)
    for rep in range(2):
        r = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts)
        _dense_equal(r, base, n)
    _, st_o, h_o, _ = port.bench_dense(0, n, dom, ctx, bg, **opts)
    st_g = np.where(r["status"] == 1, 0, r["status"])
    assert np.array_equal(st_g, st_o)
    ok = st_o == 0
    assert np.array_equal(r["hashes"][ok], h_o[ok])


def test_big_parameter_column_outside_the_tableau_is_refused(api):
    """test/challenges/pipFile_1 names big-parameter column 12 in a 12-column tableau: the reference reads past
    the row end (source/traiter.c:111), so its answer depends on the heap layout.  The library refuses the
    problem with status 4002 (PIP_STATUS_UNSUPPORTED) -- every time -- instead of answering at random."""
    cs = [x for x in load_golden("cli_suite.json") if "pipFile_1" in x["name"]]
    assert cs and all(c["bigparm"] >= c["nvar"] + c["nparm"] + 1 for c in cs)
    for _ in range(3):
        for st, cells in api.traiter_batch(cs):
            assert st == 4002 and cells == []
