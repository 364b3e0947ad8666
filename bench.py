#!/usr/bin/env python
"""bench.py -- genes/sec of scde.expression.difference (100 randomizations) on B200.

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own C++ on the host cores (oracle/_ref)
    python bench.py ... --dump-outputs DIR                   # also write each config's last timed outputs to DIR/*.npy

A "step" is one whole scde.expression.difference over one synthetic count matrix: device dedup of the counts,
log-posterior table, the bootstrap joint posteriors of both groups, the sliding-product ratio posterior and the
lb/mle/ub/Z summary.  Workload = BASELINE.json config 4: ONE 30 000-gene x 10 000-cell problem (two groups, B = 100),
the same matrix on every rank (rank-independent seed), GENES SHARDED over the N ranks in contiguous ranges
(R/functions.R:606-617) -- strong scaling, `genes_total` = 30 000 at every N.  No data-path exchange: per-shard Z / grid
indices are all-gathered over NCCL at the end of every step and rank 0 applies the Benjamini-Hochberg correction.

  value : genes/s with the counts, models, prior and draws already resident in HBM (device work only)
  e2e   : genes/s through the C ABI call with host (pinned) buffers -- H2D of the rank's count rows, D2H of results inside
  roofline : contraction kernel (the dominant one): HBM-bound gather -- algorithmic bytes = visited (gene, cell) pairs x
             (5 planes x 401 B of table + 8 B of list entry) against the measured copy bandwidth of MEASURED_PEAKS.json
  cpu_baseline : the reference's own C++ (src/jpmatLogBoot.cpp compiled unmodified against oracle/shim -> oracle/_ref),
             one worker process per host core on contiguous gene chunks as scde.posteriors(n.cores) does, bounded sample
  parity : (a) N > 1: the gathered idx / Z of the N shards == the unsharded one-device result, bit for bit;
           (b) idx / Z against the reference's C++ (cpu_baseline leg, Seed = 1) on a STRIDED gene sample
  weak  : (N > 1) every rank runs all 30 000 genes -- the weak-scaling number of round 1, as an extra key
  sub_records : configs 3 (20 000 x 2 000) and 5 (30 000 x 10 000, batch-corrected) measured the same way, each with parity
"""
from __future__ import annotations

import argparse
import ctypes as Cc
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K_GRID = 401
N_BOOT = 100
METRIC = "genes/sec scde.expression.difference (100 boot)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--genes", type=int, default=None, help="default: the config's size (3: 20000, 4 and 5: 30000)")
    ap.add_argument("--cells", type=int, default=None, help="default: the config's size (3: 2000, 4 and 5: 10000)")
    ap.add_argument("--config", type=int, default=4, choices=[3, 4, 5])
    ap.add_argument("--cpu-sample-genes-per-thread", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-sub-records", action="store_true", help="skip the config-3 / config-5 sub-records")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling extra key")
    ap.add_argument("--kernel", type=int, default=0,
                    help="contraction kernel: 0 auto (tcgen05 int8 fixed point), 1 generic FP64, 2 tiled FP64 (DMMA), 3 tcgen05")
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE",
                    help="scde_b200_options field (e.g. item_order=1, hot_rank=16); repeatable")
    ap.add_argument("--trace", action="store_true", help="host wall-clock of the one-shot call's phases on stderr")
    ap.add_argument("--boot", type=int, default=None, help="n.randomizations (default 100, BASELINE.json; R's default is 150)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step of each config returned (grid indices, "
                         "Z, BH-corrected cZ) as DIR/cfg<N>_<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.boot:
        global N_BOOT
        N_BOOT = args.boot
    return args


def config_size(config, genes=None, cells=None):
    g = genes if genes is not None else (20000 if config == 3 else 30000)  # BASELINE.json configs[2] / [3], [4]
    c = cells if cells is not None else (2000 if config == 3 else 10000)
    return g, c


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ workload
def workload_host(config, genes, cells, device, pinned=True):
    """Synthetic inputs of the named config; the SAME on every rank (the seed does not depend on the rank); counts in
    pinned host memory (genes x cells, Fortran order = R's layout)."""
    from scde_b200 import synth

    seed = synth.SEED_BASE + config
    rng = np.random.Generator(np.random.PCG64(seed))
    models = synth.make_models(rng, cells)
    counts = synth.make_counts_torch(models, genes, seed, device, pinned=pinned)
    prior = synth.make_prior(genes)
    group = np.where(np.arange(cells) < cells // 2, 0, 1).astype(np.int32)
    batch = (rng.uniform(size=cells) < 0.5).astype(np.int32) if config == 5 else None
    return models, counts, prior, group, batch


def spread_sample(n_genes, n):
    """n gene indices spread evenly over the whole matrix (so every rank's shard is sampled)"""
    return np.unique(np.linspace(0, n_genes - 1, min(n, n_genes)).astype(np.int64))


# ------------------------------------------------------------------------------------------------ CPU arm
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_leg(models, counts_sample, prior, group, batch, n_workers, n_boot=N_BOOT):
    """The reference's CPU implementation of the path on `counts_sample` (genes x cells): one worker PROCESS per host core
    on a contiguous gene chunk, as scde.posteriors chunks over n.cores (R/functions.R:606-617); every worker runs the
    reference's own logBootPosterior / logBootBatchPosterior (oracle/_ref, else the oracle port) with Seed = 1; then the
    ratio posterior (the reference's matSlideMult) and the summary (R-level code, oracle restatement) in this process.
    Returns (genes, seconds, detail): seconds = slowest worker's bootstrap time (table build measured and excluded, see
    oracle/ref_worker.py) + the ratio/summary time."""
    from oracle import oracle as O
    from oracle import ref as R

    impl = "reference" if os.path.exists(R._LIB_PATH) or R.can_build() else "port"
    if impl == "reference":
        R.lib()
    mm, lt, sq = O.pack_models(models)
    x, y = prior["x"].to_numpy(), prior["y"].to_numpy()
    mag = O.marginals_from_prior_x(x)
    G = counts_sample.shape[0]
    n_workers = max(1, min(n_workers, G))
    bounds = np.linspace(0, G, n_workers + 1).astype(int)
    tmp = tempfile.mkdtemp(prefix="scde_cpu_arm_")
    procs = []
    for w in range(n_workers):
        a, b = bounds[w], bounds[w + 1]
        inp, outp = os.path.join(tmp, f"in{w}.npz"), os.path.join(tmp, f"out{w}.npz")
        kw = dict(impl=impl, models=mm, counts=np.ascontiguousarray(counts_sample[a:b]), mag=mag, nboot=n_boot, seed=1,
                  localtheta=lt, sqlogit=sq, group=group)
        if batch is not None:
            kw["batch"] = batch
        np.savez(inp, **kw)
        procs.append((subprocess.Popen([sys.executable, "-m", "oracle.ref_worker", inp, outp], cwd=ROOT), outp))
    jps = {k: [] for k in ("jp0", "jp1", "bjp0", "bjp1")}
    t_full = t_table = 0.0
    for p, outp in procs:
        if p.wait() != 0:
            raise RuntimeError("CPU-arm worker failed")
        d = np.load(outp)
        for k in jps:
            if k in d.files:
                jps[k].append(d[k])
        t_full = max(t_full, float(d["t_full"]))
        t_table = max(t_table, float(d["t_table"]))
    for f in os.listdir(tmp):
        os.remove(os.path.join(tmp, f))
    os.rmdir(tmp)
    jp = {k: np.asfortranarray(np.concatenate(v, axis=0)) for k, v in jps.items() if v}
    t0 = time.perf_counter()
    slide = R.mat_slide_mult if impl == "reference" else O.mat_slide_mult

    def ratio(p1, p2, py):  # calculate.ratio.posterior, R/functions.R:3491-3510
        if py is not None:
            p1, p2 = p1 * py[None, :], p2 * py[None, :]
        rp = slide(p1, p2)
        rs = np.sum(rp.astype(np.longdouble), axis=1).astype(np.float64)  # rowSums: long double accumulation
        return np.asfortranarray(rp / rs[:, None])

    diffv = O.fold_change_grid(x)
    bd = ratio(jp["jp0"], jp["jp1"], y)
    res, idx = O.distribution_summary(bd, diffv, 0.0)
    out = {"results": res, "idx": idx}
    if batch is not None:
        bb = ratio(jp["bjp0"], jp["bjp1"], y)
        ab = ratio(bd, bb, None)
        ares, aidx = O.distribution_summary(ab, O.fold_change_grid(diffv), 0.0)
        out.update({"adjusted_results": ares, "adjusted_idx": aidx})
    t_ratio = time.perf_counter() - t0
    t_boot = max(t_full - t_table, 1e-9)
    out.update({"t_boot_s": t_boot, "t_table_s": t_table, "t_ratio_s": t_ratio, "impl": impl, "workers": n_workers})
    return G, t_boot + t_ratio, out


def cpu_baseline_record(g, s, det, C, how):
    return {"value": g / s, "unit": "genes/s", "cores": det["workers"], "kind": det["impl"],
            "sample": f"{how}: {g} genes x {C} cells, one worker process per core on contiguous gene chunks; "
                      f"bootstrap loops {det['t_boot_s']:.1f} s (slowest worker) + ratio posterior and summary "
                      f"{det['t_ratio_s']:.2f} s; per-chunk lp-table build ({det['t_table_s']:.1f} s, amortised over 1875 genes "
                      f"per chunk in a real run) measured and excluded, which favours the CPU arm",
            "extrapolated": True}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref; rank 0 only)."""
    if rank != 0:
        return
    from oracle import oracle as O
    from scde_b200 import synth

    O.build()
    G_all, C = config_size(args.config, args.genes, args.cells)
    n_workers = host_cores()
    seed = synth.SEED_BASE + args.config
    rng = np.random.Generator(np.random.PCG64(seed))
    models = synth.make_models(rng, C)
    gpt = max(1, args.cpu_sample_genes_per_thread)
    G = n_workers * gpt
    counts = synth.make_counts_torch(models, G, seed, "cpu", pinned=False)
    prior = synth.make_prior(G_all)
    group = np.where(np.arange(C) < C // 2, 0, 1).astype(np.int32)
    batch = (rng.uniform(size=C) < 0.5).astype(np.int32) if args.config == 5 else None
    det = None
    for _ in range(min(args.warmup, 1)):
        cpu_reference_leg(models, counts, prior, group, batch, n_workers)
    tot_g, tot_s = 0, 0.0
    for _ in range(args.steps):
        g, s, det = cpu_reference_leg(models, counts, prior, group, batch, n_workers)
        tot_g += g
        tot_s += s
    v = tot_g / tot_s
    cb = cpu_baseline_record(tot_g // max(1, args.steps), tot_s / max(1, args.steps), det, C, "per step")
    cb["value"] = v
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "genes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"cfg{args.config}: {G_all} genes x {C} cells, 2 groups, B={N_BOOT}"
                               + (", batch-corrected" if batch is not None else ""),
                   "sampled_genes_per_step": G,
                   "note": "cost is linear in genes: genes/s measured on a bounded gene sample of the same workload"},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "genes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa_node(index: int):
    """One process per GPU: run on the CPUs NVML names as local to the GPU, so that the pinned count matrix (first
    touch) and the host thread that feeds the copies sit on the GPU's NUMA node.  Returns the CPU list, or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1]
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return allowed
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------ GPU arm
class Bench:
    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.all_cpus = os.sched_getaffinity(0)
        self.numa = bind_to_gpu_numa_node(self.local_rank) if self.world > 1 and not os.environ.get("SCDE_B200_NO_AFFINITY") else None
        import torch
        import torch.distributed as dist

        from scde_b200 import _lib

        self.torch, self.dist, self._lib = torch, dist, _lib
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)
        self.ctx = _lib.Context(self.local_rank)
        opts = {}
        if args.kernel:
            opts["contract_kernel"] = args.kernel
        if args.trace or os.environ.get("SCDE_B200_TRACE"):
            opts["trace"] = 1
        for kv in args.opt:
            k, v = kv.split("=")
            opts[k] = int(v)
        if opts:
            self.ctx.set_options(**opts)
        self.opts = opts
        self.ext = torch.cuda.ExternalStream(self.ctx.stream, device=self.device)
        self.outputs = {}  # rank 0: "cfg<N>" -> what the last timed step of that config returned

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.device)
        self.ctx.synchronize()

    def gather(self, res, G_all, keys=("z", "idx")):
        """the one exchange of the path: per-shard Z and grid indices -> all ranks (NCCL all_gather on padded shards);
        returns full-length arrays in gene order"""
        from scde_b200.distributed import shard_range

        torch, dist = self.torch, self.dist
        if self.world == 1:
            return {k: res[k] for k in keys if k in res}
        sizes = [shard_range(G_all, r, self.world) for r in range(self.world)]
        longest = max(b - a for a, b in sizes)
        out = {}
        for k in keys:
            if k not in res:
                continue
            loc = np.ascontiguousarray(res[k])  # idx: (n, 3) row-major copy
            width = 1 if loc.ndim == 1 else loc.shape[1]
            t = torch.zeros((longest, width), dtype=torch.from_numpy(loc[:1]).dtype, device=self.device)
            t[: loc.shape[0]] = torch.from_numpy(loc.reshape(loc.shape[0], width)).to(self.device, non_blocking=True)
            bufs = [torch.empty_like(t) for _ in range(self.world)]
            dist.all_gather(bufs, t)
            full = torch.cat([bufs[r][: b - a] for r, (a, b) in enumerate(sizes)]).cpu().numpy()
            out[k] = full[:, 0] if loc.ndim == 1 else full
        return out

    def correct(self, z_all):
        """BH over all genes on rank 0 (host)"""
        if self.rank != 0:
            return None
        _lib = self._lib
        cz = np.empty_like(z_all)
        _lib.check(_lib.lib().scde_b200_bh_cz(_lib.p_f64(np.ascontiguousarray(z_all)), len(z_all), _lib.p_f64(cz)))
        return cz

    # --------------------------------------------------------------------------------------------
    def measure(self, config, genes, cells, steps, warmup, sharded=True, with_cpu=True, with_parity=True,
                sample_per_core=8, label=""):
        """One config: device-resident arm, end-to-end arm, parity, CPU baseline.  Returns the record (rank 0) or None."""
        torch = self.torch
        from scde_b200 import api
        from scde_b200.distributed import shard_range

        _lib, ctx, ext, world, rank = self._lib, self.ctx, self.ext, self.world, self.rank
        models, counts, prior, group, batch = workload_host(config, genes, cells, self.device)
        mm, lt, sq = api.pack_models(models)
        x, y = prior["x"].to_numpy(), prior["y"].to_numpy()
        diffv = api.fold_change_grid(x)
        zi = api._zero_index(diffv, 0.0)
        G_all, C = counts.shape
        g0, g1 = shard_range(G_all, rank, world) if sharded else (0, G_all)
        G = g1 - g0
        n_groups = [int((group == 0).sum()), int((group == 1).sum())]
        keys = ("z", "idx") + (("adjusted_z", "adjusted_idx") if batch is not None else ())
        # all ranks hold the same matrix: checksum of a strided sample of rows, compared across ranks
        chk = int(np.asarray(counts[:: max(1, G_all // 64)], dtype=np.int64).sum())
        same_matrix = True
        if world > 1:
            t = torch.tensor([chk], device=self.device, dtype=torch.int64)
            lst = [torch.empty_like(t) for _ in range(world)]
            self.dist.all_gather(lst, t)
            same_matrix = all(int(v) == chk for v in lst)

        def make_job(gr):
            return api.DifferenceJob(ctx, counts, mm, x, y, group, N_BOOT, 1, batch_codes=batch,
                                     n_batch_levels=2 if batch is not None else 0, zero_index=zi, local_theta=lt, sqlogit=sq,
                                     gene_range=gr)

        def finish(res, n_total):
            full = self.gather(res, n_total, keys)
            if rank == 0:
                full["cz"] = self.correct(full["z"])
                if batch is not None:
                    full["adjusted_cz"] = self.correct(full["adjusted_z"])
            return full

        def timed_resident(job, n_total, n_steps, n_warm):
            stats_acc = []
            for _ in range(n_warm):
                job.run()
                finish(job.download(), n_total)
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            # The library's work runs on its own stream (`ext`); the end-of-path exchange (all_gather of Z / indices over
            # NCCL, BH on rank 0) of step i runs on torch's stream and overlaps the device work of step i+1, as a
            # pipelined caller would do.  Both streams are drained before the closing event.
            prev, full = None, None
            e0.record(ext)
            for _ in range(n_steps):
                job.run()
                if prev is not None:
                    full = finish(prev, n_total)
                prev = job.download()
                stats_acc.append(prev["stats"])
            full = finish(prev, n_total)
            torch.cuda.current_stream(self.device).synchronize()
            e1.record(ext)
            self.barrier()
            return e0.elapsed_time(e1) / n_steps, stats_acc, full

        # ---------------- device-resident arm ----------------
        job = make_job((g0, g1))
        sampler = ClockSampler(self.local_rank)
        for _ in range(min(warmup, 1)):  # the sampler thread starts after the first warm-up (allocations done)
            job.run()
            finish(job.download(), G_all)
        sampler.start()
        ms_step, stats_acc, full = timed_resident(job, G_all, steps, max(0, warmup - 1))
        clocks = sampler.stop()
        job.close()
        if rank == 0:
            self.outputs[f"cfg{config}"] = full

        # ---------------- end-to-end arm: host buffers through the one-shot C-ABI call ----------------
        n_draw_sets = 4 if batch is not None else 2
        # whole job, summed over the ranks: every rank uploads its rows of the count matrix and the (small) shared inputs
        h2d = G_all * C * 4 + world * (mm.nbytes + x.nbytes + y.nbytes + group.nbytes + (batch.nbytes if batch is not None else 0)
                                       + n_draw_sets * N_BOOT * 4 * (n_groups[0] + n_groups[1]) // 2)
        d2h = G_all * (3 * 4 + 8) * (3 if batch is not None else 1)

        def e2e_step(gr, n_total):
            res = api.expression_difference_call(ctx, counts, mm, x, y, group, N_BOOT, 1, batch_codes=batch,
                                                 n_batch_levels=2 if batch is not None else 0, zero_index=zi,
                                                 local_theta=lt, sqlogit=sq, gene_range=gr)
            return finish(res, n_total), res["stats"]

        e2e_step((g0, g1), G_all)
        self.barrier()
        e2e_steps = steps
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e2.record(ext)  # the stream is idle here, so this timestamps the start of the host call
            for _ in range(e2e_steps):
                full_e2e, e2e_stats = e2e_step((g0, g1), G_all)
            e3.record(ext)
        self.barrier()
        e2e_ms = e2.elapsed_time(e3) / e2e_steps

        # ---------------- weak-scaling extra key: every rank processes all genes ----------------
        weak = None
        if world > 1 and sharded and not self.args.no_weak:
            wjob = make_job((0, G_all))
            wms, _, _ = timed_resident_local(self, wjob, steps, 1)
            wjob.close()
            weak = wms

        # ---------------- multi-rank parity: gathered shards == unsharded one-device result, bit for bit ----------------
        shard_parity = None
        if world > 1 and sharded and with_parity:
            if rank == 0:
                one = api.expression_difference_call(ctx, counts, mm, x, y, group, N_BOOT, 1, batch_codes=batch,
                                                     n_batch_levels=2 if batch is not None else 0, zero_index=zi,
                                                     local_theta=lt, sqlogit=sq)
                shard_parity = {"ranks": world,
                                "resident_equals_one_device": bool(all(np.array_equal(one[k], full[k]) for k in keys)),
                                "one_shot_equals_one_device": bool(all(np.array_equal(one[k], full_e2e[k]) for k in keys)),
                                "same_matrix_on_every_rank": bool(same_matrix), "compared": list(keys)}
            self.barrier()

        # ---------------- reduce timings over ranks (max) ----------------
        tt = torch.tensor([ms_step, e2e_ms, weak if weak is not None else 0.0], device=self.device, dtype=torch.float64)
        if world > 1:
            self.dist.all_reduce(tt, op=self.dist.ReduceOp.MAX)
        ms_step, e2e_ms, weak_ms = float(tt[0]), float(tt[1]), float(tt[2])
        # per-rank stage times (every rank's last-run stats) for the strong-scaling table
        stage_ms = {k: float(np.mean([s["ms"][k] for s in stats_acc])) for k in stats_acc[-1]["ms"]}
        names = list(stage_ms)
        st = torch.tensor([stage_ms[k] for k in names], device=self.device, dtype=torch.float64)
        st_all = [st]
        if world > 1:
            st_all = [torch.empty_like(st) for _ in range(world)]
            self.dist.all_gather(st_all, st)
        ent = torch.tensor([float(stats_acc[-1]["contract_cells"]), float(stats_acc[-1]["table_rows"])], device=self.device,
                           dtype=torch.float64)
        ent_all = [ent]
        if world > 1:
            ent_all = [torch.empty_like(ent) for _ in range(world)]
            self.dist.all_gather(ent_all, ent)
        if rank != 0:
            return None

        value = G_all / (ms_step * 1e-3)
        e2e_value = G_all / (e2e_ms * 1e-3)
        stage_by_rank = [{k: float(v) for k, v in zip(names, t.tolist())} for t in st_all]
        entries_by_rank = [float(t[0]) for t in ent_all]
        rows_by_rank = [int(t[1]) for t in ent_all]

        # ---------------- roofline of the contraction kernel (rank 0's launches) ----------------
        ms_c = stage_ms["contract"]
        n_c = int(stats_acc[-1]["launches"]["contract"])
        entries = float(stats_acc[-1]["contract_cells"])
        dense_entries = float(G) * (n_groups[0] + n_groups[1]) * (2 if batch is not None else 1)
        flops_exec = 2.0 * K_GRID * N_BOOT * entries
        peak, peak_src = 6650.0, "fallback 6650 GB/s (B200_PROFILING.md): MEASURED_PEAKS.json missing"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peak = float(json.load(f)["hbm_gbs"])
            peak_src = "MEASURED_PEAKS.json hbm_gbs (copy bandwidth, burst)"
        except Exception:
            pass
        if self.args.kernel in (0, 3):
            bytes_alg = entries * (5 * K_GRID + 8)
            achieved = bytes_alg / (ms_c * 1e-3) / 1e9
            traffic, traffic_src = None, None
            try:
                with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                    tj = json.load(f)["contract_i8_kernel"]
                if tj["genes"] == G and tj["cells"] == C and tj["config"] == config and tj.get("options", {}) == {
                        k: v for k, v in self.opts.items() if k in ("item_order", "hot_rank", "cold_evict_first")}:
                    traffic = float(tj["dram_bytes_per_launch"])
                    traffic_src = tj.get("source")
            except Exception:
                traffic = None
            roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "kernel": "contract_i8_kernel (tcgen05.mma kind::i8)",
                    "launches_per_step": n_c, "avg_launch_ms": ms_c / max(1, n_c),
                    "bytes_per_launch": bytes_alg / max(1, n_c),
                    "bytes_per_visited_pair": 5 * K_GRID + 8, "stored_bytes_per_visited_pair": 2048 + 8,
                    "dram_gbs": (traffic / (ms_c / max(1, n_c) * 1e-3) / 1e9) if traffic else None,
                    "dram_frac": (traffic / (ms_c / max(1, n_c) * 1e-3) / 1e9 / peak) if traffic else None,
                    "note": "achieved = algorithmic bytes (every visited pair's row once) / launch time on rank 0; rows of small "
                            "counts are shared by thousands of genes and hit the 126 MB L2, so the DRAM traffic of a launch "
                            "(`traffic`, from the ncu capture named in traffic_source) is smaller than the algorithmic bytes "
                            "and `frac` can exceed the DRAM fraction `dram_frac`",
                    "entries_visited_frac": entries / dense_entries, "peak_source": peak_src,
                    "int8_tops": 5.0 * flops_exec / (ms_c * 1e-3) / 1e12,
                    "fp64_equivalent_tflops": flops_exec / (ms_c * 1e-3) / 1e12,
                    "stage_ms": stage_ms}
        else:
            fp64_peak = ctx.measure_fp64_peak()
            achieved_tf = flops_exec / (ms_c * 1e-3) / 1e12
            roof = {"bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                    "frac": achieved_tf / fp64_peak if fp64_peak else None, "traffic": None,
                    "kernel": "contract_mma_kernel" if self.args.kernel != 1 else "contract_generic_kernel",
                    "launches_per_step": n_c, "avg_launch_ms": ms_c / max(1, n_c),
                    "flops_per_launch": flops_exec / max(1, n_c), "entries_visited_frac": entries / dense_entries,
                    "peak_source": "DFMA loop measured live on this device (scde_b200_measure_fp64_peak)",
                    "stage_ms": stage_ms}
        launches_per_step = int(sum(v for k, v in stats_acc[-1]["launches"].items() if k != "total"))

        rec = {
            "metric": METRIC, "value": value, "unit": "genes/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None,
            "dtype": "f64 + s8 fixed point (2^-29, exact int32 sums)" if self.args.kernel in (0, 3) else "f64",
            "data": "synthetic",
            "config": {"workload": f"cfg{config}: ONE {G_all} genes x {C} cells problem, 2 groups of {n_groups[0]}/{n_groups[1]}, "
                                   f"B={N_BOOT}, K={K_GRID}" + (", batch-corrected (4 joints)" if batch is not None else ""),
                       "genes_total": G_all, "genes_per_rank": [b - a for a, b in
                                                                [shard_range(G_all, r, world) for r in range(world)]] if sharded else [G_all] * world,
                       "sharding": "contiguous gene ranges, one per rank (R/functions.R:606), same matrix on every rank; "
                                   "NCCL all_gather of Z / grid indices at the end, BH on rank 0",
                       "host_affinity": ("GPU-local CPUs (NVML), %d" % len(self.numa)) if self.numa else "unchanged",
                       "options": self.opts,
                       "l2": "inputs larger than L2 (rank 0: counts %.2f GB, lp table %.1f GB)" % (
                           G * C * 4 / 1e9, stats_acc[-1]["table_rows"] * (2048 if self.args.kernel in (0, 3) else 416 * 8) / 1e9)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "genes/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms, "bytes_are": "whole job (sum over ranks)",
                    "stage_ms": e2e_stats["ms"]},
            "gpu_launches": launches_per_step * steps,
            "roofline": roof,
            "stage_ms_by_rank": stage_by_rank, "visited_pairs_by_rank": entries_by_rank, "table_rows_by_rank": rows_by_rank,
        }
        if weak_ms > 0:
            rec["weak"] = {"value": world * G_all / (weak_ms * 1e-3), "unit": "genes/s", "ms_per_step": weak_ms,
                           "workload": f"every rank processes all {G_all} genes (round 1's number); device-resident"}
        if shard_parity is not None:
            rec["shard_parity"] = shard_parity

        # ---------------- CPU baseline + parity on a strided gene sample (rank 0) ----------------
        if with_cpu:
            os.sched_setaffinity(0, self.all_cpus)  # the CPU arm gets every host core again
            n_workers = host_cores()
            sel = spread_sample(G_all, n_workers * max(1, sample_per_core))
            sample = np.ascontiguousarray(np.asarray(counts)[sel])
            g, s, det = cpu_reference_leg(models, sample, prior, group, batch, n_workers)
            rec["cpu_baseline"] = cpu_baseline_record(g, s, det, C, f"{g} genes spread over the whole matrix")
            if with_parity:
                def cmp(zc, zg, ic, ig):
                    reg = zc >= -6.0  # below -6 the reference's own tail formula makes one ulp worth 4e-5 in Z (DESIGN.md section 5)
                    return {"max_abs_dZ": float(np.max(np.abs(zc - zg))),
                            "max_abs_dZ_where_Z_ge_minus6": float(np.max(np.abs(zc - zg)[reg])) if reg.any() else 0.0,
                            "grid_indices_equal": bool(np.array_equal(ig, ic)),
                            "max_index_diff": int(np.max(np.abs(ig.astype(np.int64) - ic)))}
                par = {"genes": int(g), "sample": "strided over all genes (every rank's shard)", "against": det["impl"] +
                       (" (src/jpmatLogBoot.cpp + src/matSlideMult.cpp compiled unmodified, Seed = 1)" if det["impl"] == "reference" else ""),
                       "tolerance": "grid indices equal (<= 1 step allowed); |dZ| <= 1e-6 (2e-4 where Z < -6)"}
                par.update(cmp(det["results"][:, 4], full["z"][sel], det["idx"], full["idx"][sel]))
                par["e2e_path_equals_resident_path"] = bool(all(np.array_equal(full[k], full_e2e[k]) for k in keys))
                if batch is not None:
                    par["batch_adjusted"] = cmp(det["adjusted_results"][:, 4], full["adjusted_z"][sel], det["adjusted_idx"],
                                                full["adjusted_idx"][sel])
                rec["parity"] = par
        return rec


def timed_resident_local(b: Bench, job, n_steps, n_warm):
    """device-resident steps without the cross-rank gather (weak-scaling extra key)"""
    torch = b.torch
    for _ in range(n_warm):
        job.run()
        job.download()
    b.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(b.ext)
    for _ in range(n_steps):
        job.run()
        job.download()
    e1.record(b.ext)
    b.barrier()
    return e0.elapsed_time(e1) / n_steps, None, None


def dump_outputs(outputs, out_dir, max_bytes=60_000_000):
    """Writes every array of `outputs` ({"cfg<N>": {name: array}}) as out_dir/cfg<N>_<name>.npy in float64 (grid indices
    are small integers, exact in float64).  Where all of it would exceed max_bytes, every config keeps the same fixed,
    seeded sample of gene rows in each of its arrays, and the sampled rows are written as cfg<N>_genes.npy."""
    row_bytes = {cfg: 8 + sum(8 * np.asarray(v)[0].size for v in res.values()) for cfg, res in outputs.items()}
    total = sum(len(res["z"]) * row_bytes[cfg] for cfg, res in outputs.items())
    keep = min(1.0, max_bytes / max(1, total))
    os.makedirs(out_dir, exist_ok=True)
    for cfg, res in outputs.items():
        n_genes = len(res["z"])
        rows = slice(None)
        if keep < 1.0:
            rows = np.sort(np.random.default_rng(0).choice(n_genes, int(n_genes * keep), replace=False))
            np.save(os.path.join(out_dir, f"{cfg}_genes.npy"), rows.astype(np.float64))
        for name, v in res.items():
            np.save(os.path.join(out_dir, f"{cfg}_{name}.npy"), np.ascontiguousarray(np.asarray(v)[rows], dtype=np.float64))


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    b = Bench(args)
    G, C = config_size(args.config, args.genes, args.cells)
    line = b.measure(args.config, G, C, args.steps, args.warmup, with_cpu=not args.no_cpu_baseline,
                     with_parity=not args.no_parity, sample_per_core=args.cpu_sample_genes_per_thread)
    if args.config == 4 and not args.no_sub_records and args.genes is None and args.cells is None:
        subs = {}
        for cfg in (3, 5):
            g, c = config_size(cfg)
            sub = b.measure(cfg, g, c, args.steps, 2, with_cpu=not args.no_cpu_baseline,
                            with_parity=not args.no_parity, sample_per_core=2 if cfg == 5 else 8)
            if sub is not None:
                keep = ("value", "unit", "n_gpus", "ms_per_step", "scaling", "config", "e2e", "parity", "shard_parity",
                        "cpu_baseline", "stage_ms_by_rank", "weak")
                subs[f"cfg{cfg}"] = {k: sub[k] for k in keep if k in sub}
                subs[f"cfg{cfg}"]["roofline_frac"] = sub["roofline"]["frac"]
                subs[f"cfg{cfg}"]["stage_ms"] = sub["roofline"]["stage_ms"]
        if line is not None:
            line["sub_records"] = subs
    if args.dump_outputs and b.rank == 0:
        dump_outputs(b.outputs, args.dump_outputs)
    if line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        b.dist.destroy_process_group()


if __name__ == "__main__":
    main()
