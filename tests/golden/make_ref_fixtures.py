"""Writes tests/golden/ref_fixtures_*.npz: outputs of THE REFERENCE'S OWN C++ (src/jpmatLogBoot.cpp, src/matSlideMult.cpp
compiled unmodified against oracle/shim -> oracle/_ref/libscde_ref.so) on committed inputs.  Runs only where the
reference's sources are present (SCDE_REF_SRC); the tests use the committed fixtures.

    python tests/golden/make_ref_fixtures.py

Cases (inputs are re-derived by the tests from the committed es_mef_small / o_ifm / knn fixtures and scde_b200.synth):
  cfg1   es.mef.small + o.ifm (tests/tests.R filter), genes = 64 spread over the matrix + the vignette's six genes,
         ESC vs MEF, B = 100, Seed = 1: logBootPosterior(returnpost = 1) per group -> jp, modes; matSlideMult of the
         prior-weighted joints
  batch  synthetic 48 genes x 36 cells with a 2-level batch factor (scde_b200.synth config 5, seed 3), B = 100, Seed = 1:
         the two group joints and the two composition-sampled joints of logBootBatchPosterior
  knn    data/knn.rda models (local theta, conc.a2), 12 cells x 40 genes of seeded counts, B = 50: jp, modes
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, ".."))
import helpers  # noqa: E402
from oracle import oracle as O  # noqa: E402  (host prep only: unique(), pack; the numbers below come from oracle.ref)
from oracle import ref as R  # noqa: E402
from scde_b200 import synth  # noqa: E402

cfg1_inputs, knn_inputs, batch_inputs = helpers.ref_cfg1_inputs, helpers.ref_knn_inputs, helpers.ref_batch_inputs


def main():
    out = {}
    # ---- cfg1
    sub, ifm, prior, groups, sel = cfg1_inputs()
    mm, lt, sq = O.pack_models(ifm)
    mag = O.marginals_from_prior_x(prior["x"].to_numpy())
    codes = np.asarray(groups.codes)
    jps = []
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        flat, off, uci = O.unique_counts(np.asfortranarray(sub.to_numpy()[:, ii]))
        r = R.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1, returnpost=1)
        out[f"cfg1_jp{lev}"], out[f"cfg1_modes{lev}"] = r["jp"], r["modes"]
        jps.append(r["jp"])
    py = prior["y"].to_numpy()
    out["cfg1_slide"] = R.mat_slide_mult(jps[0] * py[None, :], jps[1] * py[None, :])
    out["cfg1_genes"] = sel
    # ---- batch
    w = batch_inputs()
    mm, lt, sq = O.pack_models(w.models)
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    codes, bc = np.asarray(w.groups.codes), np.asarray(w.batch.codes)
    pools = [np.nonzero(bc == l)[0].astype(np.int32) for l in range(2)]
    flat_all, off_all, uci_all = O.unique_counts(w.counts)
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        flat, off, uci = O.unique_counts(np.asfortranarray(w.counts[:, ii]))
        out[f"batch_jp{lev}"] = R.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1)["jp"]
        comp = np.bincount(bc[ii], minlength=2).astype(np.int32)
        out[f"batch_bjp{lev}"] = R.log_boot_batch_posterior(mm, flat_all, off_all, uci_all, mag, pools, comp, 100, seed=1)["jp"]
    # ---- knn (local theta, square logit)
    knn, counts = knn_inputs()
    mm, lt, sq = O.pack_models(knn)
    mag = O.marginals_from_prior_x(np.linspace(0, 4.8, 401))
    flat, off, uci = O.unique_counts(counts)
    r = R.log_boot_posterior(mm, flat, off, uci, mag, 50, seed=1, returnpost=1, localtheta=lt, sqlogit=sq)
    out["knn_jp"], out["knn_modes"] = r["jp"], r["modes"]
    for name, prefix in helpers.REF_FIXTURE_FILES.items():
        path = os.path.join(HERE, name)
        part = {k: v for k, v in out.items() if k.startswith(prefix)}
        np.savez_compressed(path, **part)
        print(path, os.path.getsize(path), {k: v.shape for k, v in part.items()})


if __name__ == "__main__":
    main()
