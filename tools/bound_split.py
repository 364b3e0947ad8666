#!/usr/bin/env python
"""Per-kernel split of the pruning stage ("bound") of the device-resident job of bench.py, from torch.profiler with CUDA
activities.  The job of each config runs `--warmup` times unprofiled, then `--steps` times under the profiler; the
script prints the mean device time per step of every kernel of the bound stage, the bound stage's sum, and the other
kernels by name for reference.  Profile in a run of its own: tracing slows the host, not the kernels.

    tools/bound_split.py [--configs 4 5] [--steps 3] [--warmup 2] [--boot 100] [--opt NAME=VALUE ...]
"""
import argparse
import collections
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# the kernels the "bound" stage times (api.cu, contract_joint_i8): bound_i8_kernel, or in older trees the BOUND instance of
# contract_i8_kernel (told apart from the contraction by its template arguments) and prune_decide_kernel
BOUND_KERNELS = ("z_bounds_kernel", "bound_i8_kernel", "prune_decide_kernel", "prune_compact_kernel")


def short_name(name):
    n = name.replace("void ", "").replace("scde::", "").replace("(anonymous namespace)::", "")
    base = n.split("<")[0].split("(")[0]
    if base == "contract_i8_kernel" and n.split("<", 1)[-1].split(">")[0].replace(" ", "").endswith("true"):
        return "contract_i8_kernel<BOUND>"
    return base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[4, 5])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--boot", type=int, default=100)
    ap.add_argument("--opt", action="append", default=[])
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    from scde_b200 import _lib, api

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    props = torch.cuda.get_device_properties(0)
    print(f"# device: {props.name}, {props.multi_processor_count} SMs")
    ctx = _lib.Context(0)
    if args.opt:
        ctx.set_options(**{k: int(v) for k, v in (kv.split("=") for kv in args.opt)})
    for cfg in args.configs:
        genes, cells = bench.config_size(cfg)
        models, counts, prior, group, batch = bench.workload_host(cfg, genes, cells, dev)
        mm, lt, sq = api.pack_models(models)
        x = prior["x"].to_numpy()
        zi = api._zero_index(api.fold_change_grid(x), 0.0)
        job = api.DifferenceJob(ctx, counts, mm, x, prior["y"].to_numpy(), group, args.boot, 1, batch_codes=batch,
                                n_batch_levels=2 if batch is not None else 0, zero_index=zi, local_theta=lt, sqlogit=sq,
                                gene_range=(0, genes))
        for _ in range(args.warmup):
            job.run()
            job.download()
        stage = collections.defaultdict(float)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.steps):
                job.run()
                res = job.download()
                for k, v in res["stats"]["ms"].items():
                    stage[k] += v / args.steps
        job.close()
        per = collections.defaultdict(lambda: [0.0, 0])
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            k = short_name(ev.name)
            per[k][0] += ev.device_time / 1000.0 / args.steps  # us -> ms per step
            per[k][1] += 1
        print(f"\n## config {cfg}: {genes} genes x {cells} cells, {args.boot} randomizations, {args.steps} profiled steps")
        print("stage ms (CUDA events, profiled run): " + ", ".join(f"{k} {v:.2f}" for k, v in stage.items()))
        st = res["stats"]
        print("prune counters (last step): " + ", ".join(f"{k} {st[k]}" for k in
                                                         ("prune_items", "prune_live", "prune_work", "prune_live_work")))
        bsum = 0.0
        print("bound stage, ms per step (launches per step):")
        for k in sorted(per, key=lambda k: -per[k][0]):
            if k in BOUND_KERNELS or k == "contract_i8_kernel<BOUND>":
                bsum += per[k][0]
                print(f"  {k:32s} {per[k][0]:8.3f}  ({per[k][1] // args.steps})")
        print(f"  {'sum':32s} {bsum:8.3f}")
        print("other kernels, ms per step:")
        for k in sorted(per, key=lambda k: -per[k][0]):
            if not (k in BOUND_KERNELS or k == "contract_i8_kernel<BOUND>") and per[k][0] >= 0.05:
                print(f"  {k:32s} {per[k][0]:8.3f}  ({per[k][1] // args.steps})")
        sys.stdout.flush()


if __name__ == "__main__":
    main()
