"""pip_solve_dense_dp on caller arrays in GPU memory (torch CUDA tensors): the PolyLib rows are converted where
they are and the results are written there.  Against the oracle, and word for word against the host routes
(pageable and page-locked buffers), for every combination of input and output placement."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    from piplib_b200 import api as a
    from piplib_b200 import build
    build.build()
    return a


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _cuda(torch, a, dev=0):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to("cuda:%d" % dev)


def _host(r):
    """the result dict of a call with CUDA outputs, as numpy (hashes back to their uint64 bits)"""
    out = {}
    for k, v in r.items():
        a = v.cpu().numpy() if hasattr(v, "cpu") else v
        out[k] = a.view(np.uint64) if k == "hashes" and a is not None else a
    return out


def _words(r, i):
    return [int(x) for x in r["ser"][r["ser_off"][i]:r["ser_off"][i] + r["ser_len"][i]]]


def _dense_equal(a, b, n):
    """statuses, hashes and lengths of every problem; the words of a sample of problems"""
    assert np.array_equal(a["status"], b["status"]) and np.array_equal(a["hashes"], b["hashes"])
    assert np.array_equal(a["ser_len"], b["ser_len"])
    for i in range(0, n, max(1, n // 200)):
        assert _words(a, i) == _words(b, i)


def _device_result(torch, n, cap, dev=0):
    """caller-owned CUDA result tensors for solve_dense(out=...)"""
    z = lambda k, dt: torch.zeros(k, dtype=dt, device="cuda:%d" % dev)
    return dict(status=z(n, torch.int32), hashes=z(n, torch.int64), ser=z(cap, torch.int64),
                ser_off=z(n + 1, torch.int64), ser_len=z(n, torch.int64))


def _call(api, dom, ctx, bg, status, hashes, ser, cap, ser_off, ser_len, dims, **opts):
    """pip_solve_dense_dp itself, on whatever mix of host arrays and CUDA tensors it is given"""
    n, dr, dc, cr, cc = dims
    p = lambda a: None if a is None else api._ptr(a)
    o = api.make_options(**opts)
    api._ready(dom, ctx, status, hashes, ser, ser_off, ser_len)
    return api.lib().pip_solve_dense_dp(C.c_longlong(n), dr, dc, p(dom), int(ctx is not None), cr, cc, p(ctx), bg,
                                        C.byref(o), p(status), p(hashes), p(ser), C.c_longlong(cap), p(ser_off),
                                        p(ser_len))


FAMILIES = [("loopnest16x24p3", 40000, {}), ("sor1d", 4000, {}), ("fimmel", 1500, {}), ("vivien32", 24, {}),
            ("expansion", 300, {}), ("loopnest8x12p2", 3000, {"Maximize": 1})]


@pytest.mark.parametrize("workload,n,extra", FAMILIES, ids=[f[0] + ("-max" if f[2] else "") for f in FAMILIES])
def test_device_in_device_out_vs_oracle_and_host_route(api, port, torch, workload, n, extra, monkeypatch):
    """loop nests (several chunks and lanes), equalities, cuts and class escalations, team classes, a big
    parameter (cells and the warp decoder), Maximize: status and hash against the oracle, every problem's
    status / hash / length and sampled words against the pageable host route; the rows never cross PCIe"""
    from workloads import synth
    monkeypatch.setenv("PIPLIB_B200_CHUNK", "8192")
    dom, ctx = synth.generate(workload, n, seed=41)
    bg, opts = synth.bignum(workload), synth.options(workload)
    opts.update(extra)
    base = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, **opts)
    d_dom, d_ctx = _cuda(torch, dom), _cuda(torch, ctx)
    rd = api.solve_dense(d_dom, d_ctx, bg, want_hashes=True, want_ser=True, **opts)
    assert int(api.last_stats().h2d_bytes) < dom.nbytes // 10
    assert all(v.is_cuda for v in rd.values())
    assert rd["status"].dtype == torch.int32 and rd["hashes"].dtype == torch.int64 and rd["ser"].dtype == torch.int64
    r = _host(rd)
    _dense_equal(r, base, n)
    m = min(n, 2000)
    _, st_o, h_o, _ = port.bench_dense(0, m, dom[:m], ctx[:m], bg, **opts)
    st_g = np.where(r["status"][:m] == 1, 0, r["status"][:m])
    assert np.array_equal(st_g, st_o) and np.array_equal(r["hashes"][:m][st_o == 0], h_o[st_o == 0])


def test_route_combinations(api, torch, monkeypatch):
    """device / pageable / pinned input x device / pageable / pinned output: the same answers"""
    from workloads import synth
    monkeypatch.setenv("PIPLIB_B200_CHUNK", "2048")
    n = 6000
    dom, ctx = synth.generate("loopnest8x12p2", n, seed=7)
    base = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    cap = int(base["ser_off"][n]) + 1024
    p_dom, p_ctx = api.pinned_copy(dom), api.pinned_copy(ctx)
    inputs = dict(device=(_cuda(torch, dom), _cuda(torch, ctx)), pageable=(dom, ctx), pinned=(p_dom, p_ctx))
    try:
        for iname, (d, c) in inputs.items():
            for oname in ("device", "pageable", "pinned"):
                if oname == "device":
                    out = _device_result(torch, n, cap)
                else:
                    out = api.alloc_result(n, pinned="alloc" if oname == "pinned" else False)
                r = api.solve_dense(d, c, -1, want_hashes=True, want_ser=True, out=out)
                assert r["ser"] is out["ser"], (iname, oname)
                _dense_equal(_host(r), base, n)
                if oname == "pinned":
                    api.pinned_free(out["ser"])
    finally:
        api.pinned_free(p_dom), api.pinned_free(p_ctx)


def test_inputs_beyond_int32(api, torch):
    """a few constants past 2^31 flag their problems in the int32 pool: the int64 pool is converted from the
    caller's device rows"""
    from workloads import synth
    n = 3000
    dom, ctx = synth.generate("loopnest8x12p2", n, seed=13)
    dom = dom.copy()
    rng = np.random.default_rng(9)
    for i in range(5, n, 97):
        dom[i, int(rng.integers(0, dom.shape[1])), -1] += (1 << 40)
    base = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    r = _host(api.solve_dense(_cuda(torch, dom), _cuda(torch, ctx), -1, want_hashes=True, want_ser=True))
    _dense_equal(r, base, n)


def test_edges(api, torch, monkeypatch):
    """no context, one problem, a batch that is not a multiple of the chunk, a stream too small: -2 with the
    words needed in the device ser_off[n], then a call with enough room"""
    from workloads import synth
    dom, _ = synth.generate("test10i", 500, seed=3)
    base = api.solve_dense(dom, None, -1, want_hashes=True, want_ser=True)
    _dense_equal(_host(api.solve_dense(_cuda(torch, dom), None, -1, want_hashes=True, want_ser=True)), base, 500)
    dom, ctx = synth.generate("loopnest16x24p3", 5003, seed=5)
    one = api.solve_dense(dom[:1], ctx[:1], -1, want_hashes=True, want_ser=True)
    _dense_equal(_host(api.solve_dense(_cuda(torch, dom[:1]), _cuda(torch, ctx[:1]), -1, want_hashes=True,
                                       want_ser=True)), one, 1)
    monkeypatch.setenv("PIPLIB_B200_CHUNK", "1024")
    n = 5003
    base = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    d_dom, d_ctx = _cuda(torch, dom), _cuda(torch, ctx)
    _dense_equal(_host(api.solve_dense(d_dom, d_ctx, -1, want_hashes=True, want_ser=True)), base, n)
    need = int(base["ser_off"][n])
    out = _device_result(torch, n, 64)
    rc = _call(api, d_dom, d_ctx, -1, out["status"], out["hashes"], out["ser"], 64, out["ser_off"], out["ser_len"],
               (n, dom.shape[1], dom.shape[2], ctx.shape[1], ctx.shape[2]))
    assert rc == -2 and int(out["ser_off"][n]) == need
    r = api.solve_dense(d_dom, d_ctx, -1, want_hashes=True, want_ser=True, out=out)
    assert r["ser"].shape[0] >= need
    _dense_equal(_host(r), base, n)


@pytest.mark.parametrize("two_gpus", [False, True], ids=["one-gpu", "two-gpus"])
def test_refusals(api, torch, two_gpus):
    """-3, with every output untouched: device rows with a host context, outputs partly on the host, Simplify
    (host decoder) with device arrays; arrays on two GPUs"""
    from workloads import synth
    n = 256
    dom, ctx = synth.generate("loopnest8x12p2", n, seed=17)
    dims = (n, dom.shape[1], dom.shape[2], ctx.shape[1], ctx.shape[2])
    d_dom, d_ctx = _cuda(torch, dom), _cuda(torch, ctx)

    def outputs(dev=0, host_hashes=False):
        o = _device_result(torch, n, 4096, dev)
        for v in o.values():
            v.fill_(-7)
        if host_hashes:
            o["hashes"] = np.full(n, -7, dtype=np.int64)
        return o

    def untouched(o):
        return all(bool(((v.cpu().numpy() if hasattr(v, "cpu") else v) == -7).all()) for v in o.values())

    cases = [("device rows, host context", d_dom, ctx, outputs(), {}),
             ("host and device outputs", d_dom, d_ctx, outputs(host_hashes=True), {}),
             ("Simplify", d_dom, d_ctx, outputs(), {"Simplify": 1})]
    if two_gpus:
        if torch.cuda.device_count() < 2:
            pytest.skip("needs at least two GPUs")
        cases = [("context on another GPU", d_dom, _cuda(torch, ctx, 1), outputs(), {}),
                 ("outputs on another GPU", d_dom, d_ctx, outputs(dev=1), {})]
    for name, dm, cx, o, opts in cases:
        rc = _call(api, dm, cx, -1, o["status"], o["hashes"], o["ser"], 4096, o["ser_off"], o["ser_len"], dims, **opts)
        torch.cuda.synchronize()
        assert rc == -3 and untouched(o), name
    if not two_gpus:
        with pytest.raises(RuntimeError, match="-3"):
            api.solve_dense(d_dom, d_ctx, -1, want_hashes=True, want_ser=True, Simplify=1)


def test_inputs_from_a_side_stream(api, torch):
    """inputs copied up by torch on a side stream just before the call: solve_dense synchronises the current
    stream first, so the call (made in that stream's context) reads the finished rows"""
    from workloads import synth
    n = 20000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=29)
    base = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    src_dom, src_ctx = torch.from_numpy(dom).pin_memory(), torch.from_numpy(ctx).pin_memory()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        d_dom = src_dom.to("cuda", non_blocking=True)
        d_ctx = src_ctx.to("cuda", non_blocking=True)
        r = api.solve_dense(d_dom, d_ctx, -1, want_hashes=True, want_ser=True)
    _dense_equal(_host(r), base, n)
    with torch.cuda.stream(side):                 # produced on the side stream, handed to the current one
        d_dom = (src_dom.to("cuda", non_blocking=True) * 3) - src_dom.to("cuda", non_blocking=True) * 2
    torch.cuda.current_stream().wait_stream(side)
    r = api.solve_dense(d_dom, d_ctx, -1, want_hashes=True, want_ser=True)
    _dense_equal(_host(r), base, n)


def test_runs_on_the_owning_device(api, torch):
    """with two devices configured for the dense path and the arrays on device 1, the call runs there: results
    on device 1, equal to a single-device run; the caller's current device is left as it was"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    from workloads import synth
    n = 20000
    dom, ctx = synth.generate("loopnest16x24p3", n, seed=19)
    one = api.solve_dense(dom, ctx, -1, want_hashes=True, want_ser=True)
    api.set_devices([0, 1])
    try:
        torch.cuda.set_device(0)
        r = api.solve_dense(_cuda(torch, dom, 1), _cuda(torch, ctx, 1), -1, want_hashes=True, want_ser=True)
        assert torch.cuda.current_device() == 0
        assert all(v.device == torch.device("cuda:1") for v in r.values())
        _dense_equal(_host(r), one, n)
    finally:
        api.set_devices([])
