"""What the per-problem solve reports cost, measured: one pip_solve_dense_dp batch with and without want_info, on
the page-locked host route (raw rows up by DMA, quasts and reports down by DMA) and on the CUDA-tensor route (every
result written in GPU memory).

The four runs are timed in one process and alternated, repetition after repetition, so that they share whatever
else the machine is doing.  Each timed call ends in a device synchronise; the time is the wall clock around it.
Statuses and hashes must be equal with and without the reports.  Prints one JSON line and, with --out, writes it.

    python tools/problem_info_bench.py [--n 1000000] [--reps 7] [--out profiles/problem_info_bench.json]

--tree DIR imports the library and its Python package from another checkout, built (e.g. the parent commit's): a
tree without the reports times the runs without them only, the same way.
"""
import argparse
import inspect
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info():
    """name and power limit of GPU 0 (a read-only query)"""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in q.split(",")[:2]]
        return name, limit
    except Exception as e:                       # the numbers are still measured; say what is missing
        return None, "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1000000)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--workload", default="loopnest16x24p3")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tree", default=ROOT)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sys.path.insert(0, os.path.abspath(a.tree))

    import torch
    from piplib_b200 import api
    from workloads import synth
    if not torch.cuda.is_available():
        raise SystemExit("problem_info_bench.py: no CUDA device")
    with_info = "want_info" in inspect.signature(api.solve_dense).parameters
    n = a.n
    dom, ctx = synth.generate(a.workload, n, seed=a.seed)
    bg, opts = synth.bignum(a.workload), synth.options(a.workload)

    def timed(f):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = f()
        torch.cuda.synchronize()
        return time.perf_counter() - t, r

    api.pin(dom), api.pin(ctx)
    host_out = api.alloc_result(n, pinned=True)
    host_info = api.alloc_result(n, pinned=True)
    d_dom, d_ctx = torch.from_numpy(dom).cuda(), torch.from_numpy(ctx).cuda()
    call = lambda d, c, out, info: api.solve_dense(d, c, bg, want_hashes=True, want_ser=True, out=out, **opts) if not info \
        else api.solve_dense(d, c, bg, want_hashes=True, want_ser=True, out=out, want_info=True, **opts)
    dev_out = call(d_dom, d_ctx, None, False)
    routes = dict(host_pinned=lambda: call(dom, ctx, host_out, False),
                  device_tensors=lambda: call(d_dom, d_ctx, dev_out, False))
    if with_info:
        host_info = call(dom, ctx, host_info, True)
        dev_info = call(d_dom, d_ctx, None, True)
        routes.update(host_pinned_info=lambda: call(dom, ctx, host_info, True),
                      device_tensors_info=lambda: call(d_dom, d_ctx, dev_info, True))
    for f in routes.values():                    # warm-up: modules, engine buffers, pinned staging
        f(), f()
    secs = {k: [] for k in routes}
    names = list(routes)
    for rep in range(a.reps):
        for k in names[rep % len(names):] + names[:rep % len(names)]:
            secs[k].append(timed(routes[k])[0])

    same = True
    if with_info:
        same = bool(np.array_equal(host_out["status"], host_info["status"]) and
                    np.array_equal(host_out["hashes"], host_info["hashes"]) and
                    np.array_equal(dev_out["status"].cpu().numpy(), dev_info["status"].cpu().numpy()) and
                    np.array_equal(dev_out["hashes"].cpu().numpy(), dev_info["hashes"].cpu().numpy()) and
                    np.array_equal(host_out["status"], dev_out["status"].cpu().numpy()))
    api.unpin(dom), api.unpin(ctx), api.unpin(host_out["ser"]), api.unpin(host_info["ser"])

    name, limit = gpu_info()
    tree = "in-tree" if os.path.abspath(a.tree) == ROOT else os.path.basename(os.path.abspath(a.tree))
    res = dict(tool="problem_info_bench", tree=tree, workload=a.workload, n=n, seed=a.seed, reps=a.reps,
               gpu=name or torch.cuda.get_device_name(0), power_limit=limit, same_answers=same)
    for k, v in secs.items():
        v = sorted(v)
        med = v[len(v) // 2]
        res[k] = dict(median_s=round(med, 4), problems_per_s=round(n / med), best_s=round(v[0], 4), worst_s=round(v[-1], 4),
                      spread=round((v[-1] - v[0]) / med, 4), seconds=[round(x, 4) for x in secs[k]])
    for route in ("host_pinned", "device_tensors"):
        if route + "_info" in res:
            res[route + "_info_cost"] = round(res[route + "_info"]["median_s"] / res[route]["median_s"] - 1, 4)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")
    if not same:
        raise SystemExit("problem_info_bench.py: the answers differ with the reports")


if __name__ == "__main__":
    main()
