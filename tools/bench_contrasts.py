"""Many contrasts at config-4 size: a loop of one-shot calls (one per pair, on that pair's cells -- what a user does without
a session) against DifferenceSession (create + one call for every contrast), on the synthetic 30 000 genes x 10 000 cells
of bench.py's config 4, relabelled into k equal clusters of consecutive cells.

Prints one JSON line per k (and per contrast set) with the synchronised wall times after a warm-up (count matrices in
pinned host memory on both arms; the per-pair subsets are copied outside the timed calls), the session's stage
times and launch counts, the ratio stage's time per contrast next to a single-pair call's, the GPU's name and power limit
read in the same run, and, for a sample of contrasts, whether the grid indices of the two arms agree and the largest |dZ|
between them (the per-pair calls see fewer cells, so their "log 0" clamp -DBL_MAX / cells / 1.1 differs: the arms are not
expected to agree bit for bit).

    python tools/bench_contrasts.py [--ks 2,4,8,16] [--n-boot 100] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity(device: int) -> dict:
    import torch

    out = {"gpu": torch.cuda.get_device_name(device)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # the number is still reported, without its power limit
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="2,4,8,16")
    ap.add_argument("--genes", type=int, default=30000)
    ap.add_argument("--cells", type=int, default=10000)
    ap.add_argument("--n-boot", type=int, default=100)
    ap.add_argument("--sample", type=int, default=3, help="contrasts compared between the two arms")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import pandas as pd
    import torch

    import bench
    from scde_b200 import _lib, api

    dev = torch.device("cuda:0")
    models, counts, prior, _group, _batch = bench.workload_host(4, args.genes, args.cells, dev)
    mm, lt, sq = api.pack_models(models)
    x, y = prior["x"].to_numpy(), prior["y"].to_numpy()
    K = len(x)
    ctx = _lib.default_context(0)
    ident = gpu_identity(0)
    G, Cn = counts.shape

    # the per-pair count matrices are staged in pinned memory outside the timed call, as the session's matrix is
    staging = torch.empty((Cn, G), dtype=torch.int32, pin_memory=True).numpy()

    def pair_call(a_cells, b_cells):
        ids = np.concatenate([a_cells, b_cells])
        sub = staging[:len(ids)].T  # genes x cells, Fortran order
        sub[:] = counts[:, ids]
        g = np.concatenate([np.zeros(len(a_cells), np.int32), np.ones(len(b_cells), np.int32)])
        t0 = time.perf_counter()
        r = api.expression_difference_call(ctx, sub, np.asfortranarray(mm[ids]), x, y, g, args.n_boot, 1, local_theta=lt,
                                           sqlogit=sq)
        return r, (time.perf_counter() - t0) * 1e3

    lines = []
    for k in [int(v) for v in args.ks.split(",")]:
        lab = np.minimum(np.arange(Cn) * k // Cn, k - 1)
        levels = [f"c{i}" for i in range(k)]
        groups = pd.Categorical.from_codes(lab, categories=levels)
        sets = [("pairs", "pairs")] + ([("rest", "rest")] if k == 8 else [])
        for name, spec in sets:
            plan = api.expand_contrasts(levels, spec)
            sides = [(np.nonzero(np.isin(lab, [levels.index(v) for v in la]))[0],
                      np.nonzero(np.isin(lab, [levels.index(v) for v in lb]))[0]) for _l, la, lb, _a, _b in plan]

            def session():
                t0 = time.perf_counter()
                with api.DifferenceSession(models, counts, prior, context=ctx) as s:
                    t1 = time.perf_counter()
                    res = s.contrasts(groups, spec, n_randomizations=args.n_boot)
                    t2 = time.perf_counter()
                    return res, s.create_stats, s.last_stats, (t1 - t0) * 1e3, (t2 - t1) * 1e3

            session()  # warm-up
            pair_call(*sides[0])
            ctx.synchronize()
            res, cst, st, create_ms, call_ms = session()
            ctx.synchronize()
            loop_ms, loop = 0.0, []
            for a_cells, b_cells in sides:
                r, ms = pair_call(a_cells, b_cells)
                loop_ms += ms
                loop.append(r)
            diffv = api.fold_change_grid(x)
            sample = []
            for i in np.unique(np.linspace(0, len(plan) - 1, min(args.sample, len(plan))).astype(int)):
                label = plan[i][0]
                got = res[label]
                want = api._summary_frame(loop[i]["idx"], loop[i]["z"], diffv, got.index, cz=loop[i]["cz"])
                sample.append({"contrast": label,
                               "idx_equal": bool(np.array_equal(got[["lb", "mle", "ub"]].to_numpy(),
                                                                want[["lb", "mle", "ub"]].to_numpy())),
                               "max_abs_dZ": float(np.max(np.abs(got["Z"].to_numpy() - loop[i]["z"])))})
            one_ratio = [r["stats"]["ms"]["ratio"] for r in loop]
            line = {"k": k, "contrasts": name, "n_contrasts": len(plan), "genes": G, "cells": Cn, "n_boot": args.n_boot,
                    "grid": K,
                    "loop_ms": round(loop_ms, 2),
                    "session_ms": round(create_ms + call_ms, 2),
                    "session_create_ms": round(create_ms, 2), "session_call_ms": round(call_ms, 2),
                    "speedup": round(loop_ms / (create_ms + call_ms), 3),
                    "create_stage_ms": {k2: round(v, 3) for k2, v in cst["ms"].items()},
                    "call_stage_ms": {k2: round(v, 3) for k2, v in st["ms"].items()},
                    "call_launches": st["launches"],
                    "contract_launches": st["launches"]["contract"],
                    "ratio_ms_per_contrast_batched": round(st["ms"]["ratio"] / len(plan), 4),
                    "ratio_ms_single_pair_call_median": round(float(np.median(one_ratio)), 4),
                    "loop_contract_launches": int(sum(r["stats"]["launches"]["contract"] for r in loop)),
                    "sample": sample, **ident}
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
