"""Where the caller's buffers live, measured: one pip_solve_dense_dp batch with host buffers in page-locked memory,
the same batch with the caller's arrays already in GPU memory (torch CUDA tensors in, CUDA tensors out), and
the device job (DeviceBatch.run: converted and uploaded once, kernels only).

The three routes are timed in one process and alternated, repetition after repetition, so that they share
whatever else the machine is doing.  Each timed call ends in a device synchronise; the time is the wall clock
around it.  Statuses and hashes of the three routes must be equal.  Prints one JSON line.

    python tools/device_buffers_bench.py [--n 1000000] [--reps 5] [--sweep]

--sweep also times the device-resident route under a few PIPLIB_B200_CHUNK / PIPLIB_B200_LANES settings (the
default chunk schedule was tuned for overlapping PCIe copies with kernels).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sweep", action="store_true")
    a = ap.parse_args()

    import torch
    from piplib_b200 import api
    from workloads import synth
    if not torch.cuda.is_available():
        raise SystemExit("device_buffers_bench.py: no CUDA device")
    n = a.n
    dom, ctx = synth.generate(a.workload, n, seed=a.seed)
    bg, opts = synth.bignum(a.workload), synth.options(a.workload)

    def timed(f):
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = f()
        torch.cuda.synchronize()
        return time.perf_counter() - t, r

    # host route: caller buffers page-locked in place (raw rows up by DMA, quasts down by DMA)
    api.pin(dom), api.pin(ctx)
    host_out = api.alloc_result(n, pinned=True)

    def host():
        return api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, out=host_out, **opts)

    # device-resident route: the inputs are CUDA tensors before the clock starts, the results stay CUDA tensors
    d_dom, d_ctx = torch.from_numpy(dom).cuda(), torch.from_numpy(ctx).cuda()
    dev_out = api.solve_dense(d_dom, d_ctx, bg, want_hashes=True, want_ser=True, **opts)

    def device():
        return api.solve_dense(d_dom, d_ctx, bg, want_hashes=True, want_ser=True, out=dev_out, **opts)

    db = api.DeviceBatch(dom, ctx, bg, **opts)
    routes = dict(host_pinned=host, device_resident=device, device_job=lambda: db.run(False))
    for f in routes.values():                    # warm-up: modules, engine buffers, pinned staging
        f(), f()
    secs = {k: [] for k in routes}
    names = list(routes)
    for rep in range(a.reps):
        for k in names[rep % len(names):] + names[:rep % len(names)]:
            secs[k].append(timed(routes[k])[0])

    # the three routes answer alike
    st_h, h_h = host_out["status"], host_out["hashes"]
    st_d, h_d = dev_out["status"].cpu().numpy(), dev_out["hashes"].cpu().numpy().view(np.uint64)
    db.run(False)                                # (results are read from the engines' buffers: right after a run)
    st_j, h_j = db.results(True)
    same = bool(np.array_equal(st_h, st_d) and np.array_equal(st_h, st_j) and
                np.array_equal(h_h, h_d) and np.array_equal(h_h, h_j))
    device()
    s = api.last_stats()
    stats_dev = dict(h2d_bytes=int(s.h2d_bytes), d2h_bytes=int(s.d2h_bytes))
    host()
    s = api.last_stats()
    stats_host = dict(h2d_bytes=int(s.h2d_bytes), d2h_bytes=int(s.d2h_bytes))

    sweep = []
    if a.sweep:
        for chunk, lanes in [(1 << 17, 6), (1 << 18, 4), (1 << 19, 2), (1 << 16, 8), (1 << 17, 3)]:
            os.environ["PIPLIB_B200_CHUNK"], os.environ["PIPLIB_B200_LANES"] = str(chunk), str(lanes)
            device()
            t = sorted(timed(device)[0] for _ in range(3))
            sweep.append(dict(chunk=chunk, lanes=lanes, problems_per_s=round(n / t[1]), spread=round((t[-1] - t[0]) / t[1], 4)))
        for k in ("PIPLIB_B200_CHUNK", "PIPLIB_B200_LANES"):
            os.environ.pop(k, None)
    db.close()
    api.unpin(dom), api.unpin(ctx), api.unpin(host_out["ser"])

    name, limit = gpu_info()
    res = dict(tool="device_buffers_bench", workload=a.workload, n=n, seed=a.seed, reps=a.reps,
               gpu=name or torch.cuda.get_device_name(0), power_limit=limit, same_answers=same)
    for k, v in secs.items():
        v = sorted(v)
        med = v[len(v) // 2]
        res[k] = dict(problems_per_s=round(n / med), best=round(n / v[0]), worst=round(n / v[-1]),
                      spread=round((v[-1] - v[0]) / med, 4), seconds=[round(x, 4) for x in secs[k]])
    res["bytes_device_resident"], res["bytes_host_pinned"] = stats_dev, stats_host
    if sweep:
        res["device_resident_sweep"] = sweep
    print(json.dumps(res))
    if not same:
        raise SystemExit("device_buffers_bench.py: the routes disagree")


if __name__ == "__main__":
    main()
