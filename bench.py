#!/usr/bin/env python
"""bench.py -- the hot path of piplib-b200 on BASELINE.json's headline configuration.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--workload NAME] [--dump-outputs DIR]
  python bench.py --impl reference ...      (the reference's own CPU path, all host cores)

A "step" is one pass of the solver over one batch of B synthetic problems per GPU (weak
scaling: every rank solves its own B problems; no data-path collective exists, SURVEY.md 8e).
  value   problems/s, whole job, inputs already resident in HBM: the solve kernel AND the decode of
          its cells to serialised quasts (left in HBM), CUDA events around the kernels
  e2e     problems/s through the C-ABI call pip_solve_dense_dp with HOST buffers: PolyLib
          matrices in, serialised quasts + hashes out, host<->device copies inside the region
The workload is configs[1] of BASELINE.json: ~16 unknowns x 24 constraints, 3 parameters
(workloads/synth.py: loopnest16x24p3), data = synthetic.  Inputs (4 GB per 10^6 problems) are
far larger than L2, so no explicit L2 flush is needed between steps.

--dump-outputs DIR writes what the timed calls returned in their last step as DIR/<name>.npy (float64; a
64-bit integer array as <name>_hi = signed upper 32 bits and <name>_lo = lower 32 bits, both exact), so
that two builds can be compared output for output on the same seeded inputs:
  status, hash_*                 the device-resident job (the headline value): per-problem status, quast hash
  e2e_status, e2e_hash_*         pip_solve_dense_dp on page-locked caller buffers
  e2e_ser_index, e2e_ser_len,    the serialised quasts of a fixed seeded sample of problems (indices, words per
  e2e_ser_words_*                problem, the words one after the other)
  batch_api_status               pip_solve_batch_dp on the first problems of the batch
  config4_status, config4_cells_*  the large tableau (kind, p1, p2 per cell)
Above DUMP_PROBLEMS problems per-problem arrays hold a fixed seeded sample, listed in problem_index.
"""
import argparse
import atexit
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from piplib_b200 import dist as pdist  # noqa: E402
from workloads import synth  # noqa: E402

METRIC = "problems_per_sec"
UNIT = "problems/s"
# --dump-outputs budget, 64 MiB in all: 56 bytes per dumped problem (4 per-problem arrays, 48 bytes as float64
# halves, + problem_index) = 56 MB at DUMP_PROBLEMS, 4 MiB of serialised-quast words, ~0.8 MB batch API + config 4
DUMP_PROBLEMS = 1000000        # per-problem arrays up to this many problems are dumped whole
DUMP_SER_PROBLEMS = 512        # problems whose serialised quasts are dumped ...
DUMP_SER_WORDS = 1 << 18       # ... as long as their words fit in this many
DUMP_LIMIT = 64 << 20


def dump_outputs(path, arrays):
    """arrays: name -> integer array; writes float64 .npy files (64-bit integers split in exact halves)"""
    files = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype.itemsize == 8:
            v = a.view(np.int64)
            files[name + "_hi"] = (v >> 32).astype(np.float64)
            files[name + "_lo"] = (v & 0xffffffff).astype(np.float64)
        else:
            files[name] = a.astype(np.float64)
    total = sum(f.nbytes for f in files.values())
    if total > DUMP_LIMIT:
        raise SystemExit("bench.py: --dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for name, f in files.items():
        np.save(os.path.join(path, name + ".npy"), f)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu = gpu
        self.samples = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                if len(f) >= 9:
                    self.samples.append(f)
        except Exception:
            pass

    def stop(self):
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], [], set()
        for f in self.samples:
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU arms (the checker libraries; never the thing shipped): oracle/cpu_arm.py
# ------------------------------------------------------------------------------------------
from oracle.cpu_arm import cpu_arm, same_answers, usable_cores  # noqa: E402


def large_tableau_line(pk, pk_src, n=4096, reps=2, cpu=True, outputs=None):
    """BASELINE config 4 (the HBM-bound kernel of the path): one n x (n+1) int64 tableau solved by the
    whole grid, cooperative launch, CUDA events inside the library.  Algorithmic bytes per pivot =
    16*R*C + 8*C + 8*R (SURVEY.md 8d, dense figure).  Refuses to report unless the cells equal the ones
    the unmodified reference (raised limits) produced for this very tableau (tests/golden/)."""
    from piplib_b200 import api
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "large_consecutive_ones_%d.json" % n)))
    tab = synth.consecutive_ones(n, n, seed=g["seed"])
    p = api.LargeProblem(n, n, g["nq"], tab, cut_rows=1024, sol_size=1 << 20, maxcol=1 << 16)
    p.run()
    ms = min(p.run() for _ in range(reps))
    st, cells, info = p.fetch()
    p.close()
    if st != g["status"] or cells != g["cells"] or info["pivots"] != g["pivots"]:
        raise SystemExit("bench.py: config 4: the %d x %d tableau's answer differs from the reference's -- "
                         "refusing to report" % (n, n + 1))
    if outputs is not None:
        outputs["config4_status"] = np.asarray([st], dtype=np.int32)
        outputs["config4_cells"] = np.asarray(cells, dtype=np.int64).reshape(-1, 3)
    piv = max(1, info["pivots"])
    R, C = n - 1, n + 1
    alg = (16.0 * R * C + 8.0 * C + 8.0 * R) * piv
    ach = alg / (ms / 1e3) / 1e9
    rows_total = float(R) * piv
    out = {"workload": "consecutive-ones %d x %d int64, Nq=1, one problem over the whole grid" % (n, n + 1),
           "status": st, "pivots": info["pivots"], "kernel_ms": ms, "us_per_pivot": 1e3 * ms / piv,
           "pivots_per_sec": piv / (ms / 1e3),
           "parity": "cells, status and pivot count equal to the unmodified reference built with raised "
                     "limits (tests/golden/large_consecutive_ones_%d.json)" % n,
           "identity_rows_skipped_frac": info["skipped_rows"] / rows_total,
           "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                        "frac": ach / pk["hbm_gbs"], "peak_source": pk_src, "traffic": None,
                        "algorithmic_bytes": alg,
                        "note": "dense algorithmic figure 16*R*C+8*C+8*R per pivot (SURVEY.md 8d convention); rows "
                                "whose update is the identity are skipped (identity_rows_skipped_frac), so the "
                                "fraction can pass 1; frac_dram is the honest one: DRAM bytes of the ncu capture "
                                "per second of this run against the same peak"}}
    for name in sorted(os.listdir(os.path.join(ROOT, "profiles")), reverse=True):
        if name.endswith("large_kernel_traffic.json"):       # newest round first
            t = json.load(open(os.path.join(ROOT, "profiles", name)))
            if t.get("n") == n and t.get("pivots") == info["pivots"]:
                traffic = float(t["dram_bytes_read"] + t["dram_bytes_write"])
                out["roofline"]["traffic"] = traffic
                out["roofline"]["traffic_source"] = "profiles/" + name
                out["roofline"]["frac_dram"] = traffic / (ms / 1e3) / 1e9 / pk["hbm_gbs"]
                break
    if cpu:
        # the reference's CPU path on this very tableau: one core by construction (it cannot split a tableau)
        from oracle import pyoracle as po
        t0 = time.perf_counter()
        if os.path.exists(po.REF_BIG_SO):
            st_c, cells_c = po.Ref(big=True).traiter(n, 0, n, 0, -1, g["nq"], tab, [], cap=1 << 20)
            kind = "reference"
        else:
            po.build(ref=False, port=True)
            st_c, cells_c = po.Port().traiter(n, 0, n, 0, -1, g["nq"], tab, [], sol_size=1 << 20, maxcol=1 << 16)
            kind = "port"
        dt = time.perf_counter() - t0
        if st_c != st or [list(c) for c in cells_c] != cells:
            raise SystemExit("bench.py: config 4: CPU baseline and GPU disagree")
        out["cpu_baseline"] = {"value": piv / dt, "unit": "pivots/s", "cores": 1, "kind": kind, "seconds": dt,
                               "sample": "the whole problem (%d pivots), raised SOL_SIZE/MAXCOL" % piv}
    return out


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=int(os.environ.get("PIP_BENCH_BATCH", 1000000)))
    ap.add_argument("--workload", default="loopnest16x24p3")
    ap.add_argument("--total", type=int, default=0,
                    help="strong scaling (BASELINE config 5): this many problems in all, sharded over the ranks")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--cpu-sample", type=int, default=0, help="problems in the CPU baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-large", action="store_true", help="skip the config-4 large-tableau measurement")
    ap.add_argument("--check", type=int, default=65536,
                    help="problems of every rank's own range cross-checked against the reference before timing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed calls returned in their last step to DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")

    rank, world, local = pdist.env_rank()
    cores = len(usable_cores())
    bg, opts = synth.bignum(a.workload), synth.options(a.workload)
    W = max(a.warmup, 0)
    K = a.steps
    B = a.batch
    if a.total:
        B = (a.total + world - 1) // world
    # shape of the workload from one generated problem (PolyLib rows: flag, unknowns, parameters, constant)
    d1, c1 = synth.generate(a.workload, 1, seed=a.seed)
    nparm = max(c1.shape[2] - 2, 0)
    config = {"workload": "%s: %d problems/GPU/step, %d unknowns x %d constraints, %d parameters, "
                          "int64, pip_solve path (Nq=%d)" % (a.workload, B, d1.shape[2] - 2 - nparm, d1.shape[1], nparm,
                                                             synth.options(a.workload).get("Nq", 1)),
              "batch_per_gpu": B, "l2": "inputs (%.1f GB/step) exceed L2; no flush needed" %
              (B * (d1.shape[1] * d1.shape[2] + c1.shape[1] * c1.shape[2]) * 8 / 1e9), "seed": a.seed}

    # ---------------- reference arm: the reference's own CPU implementation ----------------
    if a.impl == "reference":
        if rank != 0:
            return
        sample = a.cpu_sample or min(B, cores * 16384)        # >= 0.5 s of work per core and step
        dom, ctx = synth.generate(a.workload, sample, seed=a.seed, first=0)
        for _ in range(W):
            cpu_arm(dom, ctx, min(sample, cores * 1024), cores, bg=bg, opts=opts)
        tot_s, r = 0.0, None
        for _ in range(K):
            r = cpu_arm(dom, ctx, sample, cores, bg=bg, opts=opts)
            tot_s += r["seconds"]
        value = sample * K / tot_s
        ppp = cpu_arm(dom, ctx, min(sample, cores * 1024), cores, bg=bg, opts=opts, kind="port")["pivots"] / \
            min(sample, cores * 1024)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
                "steps": K, "warmup": W, "ms_per_step": 1e3 * tot_s / K, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": config, "pivots_per_sec": value * ppp,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                 "sample": "first %d problems of the workload per step, one process "
                                           "per core" % sample},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ---------------- our arm ---------------------------------------------------------------
    import torch
    import torch.distributed as dist
    from piplib_b200 import api, build
    build.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- piplib-b200 has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL announces its version on stdout when the communicator comes up (NCCL_DEBUG=VERSION):
        # stdout carries exactly one JSON line, so fd 1 points at stderr until the first collective is done
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    api.set_device(local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    first, _ = pdist.problem_range(rank, world, B)
    dom, ctx = synth.generate(a.workload, B, seed=a.seed, first=first)

    # parity gate before any timing: the first `check` problems of THIS rank's range against the
    # unmodified reference (oracle/_ref; the oracle port where it is absent), on this rank's share of the cores
    ncheck = min(a.check, B)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    my_cores = usable_cores()
    share = max(1, len(my_cores) // max(1, local_world))
    my_cores = my_cores[(local % max(1, local_world)) * share:][:share] or my_cores[:1]
    if ncheck:
        gate = cpu_arm(dom, ctx, ncheck, my_cores, bg=bg, opts=opts)
        r = api.solve_dense(dom[:ncheck], None if ctx is None else ctx[:ncheck], bg, **opts)
        if not same_answers(r["status"], r["hashes"], gate):
            raise SystemExit("bench.py: GPU results differ from the %s on problems [%d, %d) -- refusing to time"
                             % (gate["kind"], first, first + ncheck))

    # kernel-only: inputs resident in HBM
    db = api.DeviceBatch(dom, ctx, bg, **opts)
    for _ in range(max(W, 3)):
        db.run(False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        atexit.register(sampler.stop)        # no nvidia-smi left running if the timed region raises
    barrier()
    t0 = time.perf_counter()
    dev_ms, launches = 0.0, 0
    stats = None
    for _ in range(K):
        dev_ms += db.run(False)
        stats = api.last_stats()
        launches += stats.launches
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    outputs = {} if a.dump_outputs and rank == 0 else None
    status, hashes = db.results(outputs is not None)
    if outputs is not None:
        outputs["status"], outputs["hash"] = status, hashes
    pivots_step = int(stats.pivots)
    elem_step = int(stats.elem_updates)
    cells_step = int(stats.cells)
    rounds = int(stats.rounds)
    db.close()

    # end to end through the C-ABI with HOST buffers.  Headline: caller buffers in page-locked memory
    # (pip_pin_buffer_dp), as the bench contract asks -- raw PolyLib rows go up by DMA, tab_Matrix2Tableau
    # runs on the device, the serialised quasts come down by DMA.  Beside it the same call on pageable
    # buffers (host-side conversion through pinned staging).
    e2e_s, e2e_pageable_s, h2d_b, d2h_b, res = None, None, 0, 0, None
    if not a.no_e2e:
        def run_e2e(out):
            for _ in range(max(W, 3)):
                out = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, out=out, **opts)
            barrier()
            t1 = time.perf_counter()
            for _ in range(K):
                out = api.solve_dense(dom, ctx, bg, want_hashes=True, want_ser=True, out=out, **opts)
            barrier()
            return time.perf_counter() - t1, out
        e2e_pageable_s, res_pg = run_e2e(None)
        del res_pg
        api.pin(dom), api.pin(ctx)
        res = api.alloc_result(B, words_per_problem=int(os.environ.get("PIP_BENCH_WORDS", 448)), pinned=True)
        e2e_s, res = run_e2e(res)
        s2 = api.last_stats()
        h2d_b, d2h_b = int(s2.h2d_bytes), int(s2.d2h_bytes)
        api.unpin(dom), api.unpin(ctx)
        if outputs is not None:
            outputs["e2e_status"], outputs["e2e_hash"] = res["status"], res["hashes"]
            idx = np.sort(np.random.default_rng(a.seed).choice(B, size=min(B, DUMP_SER_PROBLEMS), replace=False))
            idx = idx[np.cumsum(res["ser_len"][idx]) <= DUMP_SER_WORDS]
            outputs["e2e_ser_index"] = idx.astype(np.int32)
            outputs["e2e_ser_len"] = res["ser_len"][idx].astype(np.int32)
            outputs["e2e_ser_words"] = np.concatenate(
                [res["ser"][res["ser_off"][i]:res["ser_off"][i] + res["ser_len"][i]] for i in idx])
    if rank == 0:
        sampler.stop()

    # max over ranks
    (dev_ms, wall_ms, e2e_max, e2e_pg_max), (pivots_all, elem_all, cells_all) = pdist.reduce_stats(
        [dev_ms, wall_ms, e2e_s or 0.0, e2e_pageable_s or 0.0],
        [float(pivots_step), float(elem_step), float(cells_step)], device="cuda")

    if rank == 0:
        pk, pk_src = peaks()
        total_problems = B * world * K
        value = total_problems / (dev_ms / 1e3)
        ms_per_step = dev_ms / K
        # algorithmic HBM traffic of the solve kernel: every problem's input words are read once
        # and its solution cells written once (the working set itself lives in shared memory)
        mx = max(int(np.abs(dom).max()), int(np.abs(ctx).max()))
        elem = 1 if mx < 127 else 4 if mx < 2 ** 31 - 1 else 8       # the host ships the narrowest width
        in_bytes = (dom.shape[1] * (dom.shape[2] - 1) + ctx.shape[1] * (ctx.shape[2] - 1)) * elem + 32
        alg_bytes = float(B) * (in_bytes + 56) + 8.0 * cells_step
        achieved = alg_bytes / (ms_per_step / 1e3) / 1e9
        # per-problem DRAM traffic / warp instructions of the solve kernel from the newest committed ncu
        # capture OF THIS WORKLOAD (profiles/*solve_kernel_traffic.json); none for other workloads
        traffic, t = None, None
        for name in sorted(os.listdir(os.path.join(ROOT, "profiles")), reverse=True):
            if name.endswith("solve_kernel_traffic.json"):
                tt = json.load(open(os.path.join(ROOT, "profiles", name)))
                if tt.get("workload", "loopnest16x24p3") == a.workload:
                    t, t_src = tt, "profiles/" + name
                    traffic = (t["dram_bytes_read"] + t["dram_bytes_write"]) / t["problems"] * B
                    break
        uniq, counts = np.unique(status, return_counts=True)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if a.total else "weak",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": config,
            "pivots_per_sec": pivots_all * K / (dev_ms / 1e3),
            "elem_updates_per_sec": elem_all * K / (dev_ms / 1e3),
            "pivots_per_problem": pivots_all / (B * world),
            "wall_ms_per_step": wall_ms / K,
            "rounds_per_step": rounds,
            "status_counts": {str(int(u)): int(c) for u, c in zip(uniq, counts)},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "peak_source": pk_src,
                         "algorithmic_bytes": alg_bytes,
                         "note": "class-S kernel keeps the tableau in shared memory: HBM sees only "
                                 "inputs+cells; the binding resource is the INT pipe / issue slots "
                                 "(see elem_updates_per_sec and profiles/)"},
        }
        if traffic is not None and t.get("warp_instructions"):
            # the binding resource of the shared-memory-resident kernel: warp-instruction issue slots.
            # instructions per problem come from the committed ncu capture of this kernel and workload
            # (profiles/), the rate is this run's; peak = SMs x 4 schedulers x 1 instruction/cycle x clock
            ipp = t["warp_instructions"] / t["problems"]
            clk = (line["clocks"].get("sm_mhz") or pk.get("sm_max_mhz") or 1965.0) * 1e6
            peak_issue = 148 * 4 * clk
            line["issue_roofline"] = {"bound": "issue", "achieved": ipp * value / world, "peak": peak_issue,
                                      "unit": "warp-instructions/s per GPU", "frac": ipp * value / world / peak_issue,
                                      "warp_instructions_per_problem": ipp,
                                      "source": t_src + " (ncu smsp__inst_executed.sum, same workload)"}
        if e2e_max:
            line["e2e"] = {"value": B * world * K / e2e_max, "unit": UNIT,
                           "h2d_bytes_per_step": h2d_b, "d2h_bytes_per_step": d2h_b,
                           "api": "pip_solve_dense_dp (host PolyLib matrices in, serialised quasts + hashes out)",
                           "buffers": "caller arrays page-locked with pip_pin_buffer_dp: DMA both ways, "
                                      "tab_Matrix2Tableau on the device"}
            if e2e_pg_max:
                line["e2e_pageable"] = {"value": B * world * K / e2e_pg_max, "unit": UNIT,
                                        "buffers": "pageable caller arrays: host thread pool narrows into / widens "
                                                   "out of pinned staging"}
        if world == 1 and not a.no_large:
            line["config4_large_tableau"] = large_tableau_line(pk, pk_src, outputs=outputs)
        if world == 1 and not a.no_e2e:
            # the entry point north_star names: pip_solve_batch_dp (PipMatrix objects in, malloc'd PipQuast trees
            # out), on a bounded slice (building the matrices through ctypes is the slow part, outside the timing)
            nb = min(B, 50000)
            sec, st_b = api.time_solve_batch(dom[:nb], ctx[:nb], bg, **opts)
            if res is not None and not np.array_equal(np.where(st_b == 1, 0, st_b), np.where(res["status"][:nb] == 1, 0, res["status"][:nb])):
                raise SystemExit("bench.py: pip_solve_batch_dp and pip_solve_dense_dp disagree")
            if outputs is not None:
                outputs["batch_api_status"] = st_b
            line["batch_api"] = {"value": nb / sec, "unit": UNIT, "problems": nb,
                                 "api": "pip_solve_batch_dp: PipMatrix objects in, PipQuast trees out (host decode, malloc per node)"}
        if world == 1:
            # the reference's CPU path on the same inputs, >= 1 s of work per core; its statuses and
            # hashes are compared with what the timed e2e call returned for the same problems
            sample = a.cpu_sample or min(B, cores * 32768)
            r = cpu_arm(dom, ctx, sample, cores, bg=bg, opts=opts)
            if res is not None and not same_answers(res["status"], res["hashes"], r):
                raise SystemExit("bench.py: the timed e2e results differ from the %s on the first %d problems"
                                 % (r["kind"], sample))
            line["cpu_baseline"] = {"value": sample / r["seconds"], "unit": UNIT, "cores": r["cores"],
                                    "kind": r["kind"],
                                    "sample": "first %d problems of the batch, one process per core, "
                                              "pip_solve loop; statuses and quast hashes equal to the timed "
                                              "GPU run's" % sample}
        if outputs is not None:
            if B > DUMP_PROBLEMS:
                keep = np.sort(np.random.default_rng(a.seed + 1).choice(B, size=DUMP_PROBLEMS, replace=False))
                outputs["problem_index"] = keep.astype(np.int32)
                for k in ("status", "hash", "e2e_status", "e2e_hash"):
                    if k in outputs:
                        outputs[k] = outputs[k][keep]
        print(json.dumps(line))
        sys.stdout.flush()
        if outputs is not None:
            dump_outputs(a.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
