"""Cost of draw chunks (the reference's n.cores; scde_b200_diff_args.draw_chunks) at config-4 size: the synthetic 30 000
genes x 10 000 cells of bench.py's config 4, and config 5 (the same with a batch factor), at draw_chunks 1, 10 and 20.

For each config the arms (one per draw_chunks value) alternate within every round: a resident job step (run + download of
an uploaded job, after one warm-up run) and a one-shot call (scde_b200_expression_difference, counts in pinned host memory), each synchronised and
timed on the host clock.  Prints one JSON line per (config, draw_chunks) with the per-round times, their median, the
stage times and launch counts of the one-shot call, and the GPU's name and power limit read in the same run.

    python tools/bench_draw_chunks.py [--chunks 1,10,20] [--configs 4,5] [--rounds 5] [--n-boot 100] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunks", default="1,10,20")
    ap.add_argument("--configs", default="4,5")
    ap.add_argument("--genes", type=int, default=30000)
    ap.add_argument("--cells", type=int, default=10000)
    ap.add_argument("--n-boot", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import torch

    import bench
    from bench_contrasts import gpu_identity
    from scde_b200 import _lib, api

    ident = gpu_identity(0)
    ctx = _lib.default_context(0)
    chunks = [int(v) for v in args.chunks.split(",")]
    lines = []
    for config in [int(v) for v in args.configs.split(",")]:
        models, counts, prior, group, batch = bench.workload_host(config, args.genes, args.cells, torch.device("cuda:0"))
        mm, lt, sq = api.pack_models(models)
        x, y = prior["x"].to_numpy(), prior["y"].to_numpy()
        K = len(x)
        kw = dict(local_theta=lt, sqlogit=sq, zero_index=[K], chunked_draws=True)
        if batch is not None:
            kw.update(batch_codes=batch, n_batch_levels=2, zero_index_adjusted=[2 * K - 1])
        t_job = {n: [] for n in chunks}
        t_call = {n: [] for n in chunks}
        stats = {}

        def job_step(n):  # one job per context at a time: upload and a warm-up run, then one timed step
            job = api.DifferenceJob(ctx, counts, mm, x, y, group, args.n_boot, 1, n_cores=n, **kw)
            try:
                job.run()
                job.download()
                ctx.synchronize()
                t0 = time.perf_counter()
                job.run()
                job.download()
                return (time.perf_counter() - t0) * 1e3
            finally:
                job.close()

        def call(n):
            ctx.synchronize()
            t0 = time.perf_counter()
            res = api.expression_difference_call(ctx, counts, mm, x, y, group, args.n_boot, 1, n_cores=n, **kw)
            return (time.perf_counter() - t0) * 1e3, res["stats"]

        for n in chunks:  # warm-up: every shape of both arms
            job_step(n)
            call(n)
        for r in range(args.rounds):
            for n in chunks:
                t_job[n].append(job_step(n))
                ms, stats[n] = call(n)
                t_call[n].append(ms)
        for n in chunks:
            line = {"config": config, "draw_chunks": n, "genes": args.genes, "cells": args.cells, "n_boot": args.n_boot,
                    "resident_ms": [round(v, 2) for v in t_job[n]],
                    "resident_ms_median": round(float(np.median(t_job[n])), 2),
                    "one_shot_ms": [round(v, 2) for v in t_call[n]],
                    "one_shot_ms_median": round(float(np.median(t_call[n])), 2),
                    "stage_ms": {k: round(v, 3) for k, v in stats[n]["ms"].items()},
                    "launches": stats[n]["launches"], **ident}
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
