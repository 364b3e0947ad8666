"""The oracle's restatement (oracle/scde_oracle.c) against THE REFERENCE ITSELF: the reference's src/jpmatLogBoot.cpp and
src/matSlideMult.cpp compiled unmodified against the header shim oracle/shim/RcppArmadillo.h (oracle/_ref/libscde_ref.so,
`make -C oracle ref`).  Bit-exact on every entry point: the loop nests, the summation orders (Armadillo's two-accumulator
`accumulate`, column-wise `sum(.., 1)`), the libc `srand/rand` rejection loop, the snap rule, the clamp, the modes and
individual posteriors, the batch sampler, the ensemble and no-bootstrap forms.  What the shim cannot pin is R nmath's
`dnbinom` / `dpois` (R is absent): both sides use the oracle's restatement, which tests/test_oracle.py pins with mpmath.

Where the reference's sources (SCDE_REF_SRC) or a prebuilt oracle/_ref are present, every case calls the reference.
Elsewhere it compares the oracle's outputs with tests/golden/ref_digests.json: per case and output, the shape and the
SHA-256 of the float64 bytes of the reference's result.  The comparison stays bit for bit while the stored file stays
small (the individual posteriors of one case alone take megabytes).  The file's "source" says where its digests come
from; SCDE_RECORD_REF_DIGESTS=1 rewrites it from the reference library.
"""
import hashlib
import json
import os

import numpy as np
import pytest

import helpers
from oracle import oracle as O
from oracle import ref as R
from scde_b200 import synth

DIGESTS = os.path.join(helpers.GOLD, "ref_digests.json")
RECORD = os.environ.get("SCDE_RECORD_REF_DIGESTS") == "1"
_recorded = {}


def _digest(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return [list(a.shape), hashlib.sha256(a.tobytes()).hexdigest()]


def _stored():
    with open(DIGESTS) as f:
        return json.load(f)["cases"]


@pytest.fixture(scope="module", autouse=True)
def _record_digests():
    if RECORD and not R.available():
        pytest.fail("SCDE_RECORD_REF_DIGESTS=1 needs the reference library (SCDE_REF_SRC or oracle/_ref)")
    yield
    if RECORD:
        with open(DIGESTS, "w") as f:
            json.dump({"source": "oracle/_ref/libscde_ref.so (the reference's own C++), recorded by tests/test_ref.py",
                       "cases": _recorded}, f, indent=1, sort_keys=True)
            f.write("\n")


def _same_as_reference(key, got, ref_call):
    """got: {name: array} from the oracle; ref_call() -> the same names from the reference library.  Bit for bit."""
    if R.available():
        want = ref_call()
        assert set(got) == set(want), key
        for name in got:
            assert np.array_equal(got[name], want[name]), (key, name)
        if RECORD:
            _recorded[key] = {name: _digest(v) for name, v in want.items()}
    else:
        stored = _stored()[key]
        assert set(got) == set(stored), key
        for name, a in got.items():
            assert _digest(a) == stored[name], (key, name)


def _flat(out):
    """dict(jp[, modes][, post]) with post (a list of per-cell G x K matrices) stacked into one array"""
    return {k: (np.stack([np.asarray(p) for p in v]) if k == "post" else v) for k, v in out.items()}


def _prep(w):
    mm, lt, sq = O.pack_models(w.models)
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    flat, off, uci = O.unique_counts(w.counts)
    return mm, lt, sq, mag, flat, off, uci


@pytest.mark.parametrize("G,Cn,B,seed", [(97, 23, 100, 1), (5, 1, 7, 3), (33, 40, 150, 1), (1, 9, 100, 12143)])
@pytest.mark.parametrize("returnpost", [0, 1, 2, 3])
def test_log_boot_posterior_bit_exact(G, Cn, B, seed, returnpost):
    w = synth.make_workload(3, n_genes=G, n_cells=Cn, seed=5)
    mm, lt, sq, mag, flat, off, uci = _prep(w)
    a = O.log_boot_posterior(mm, flat, off, uci, mag, B, seed=seed, returnpost=returnpost)
    _same_as_reference(f"log_boot_posterior/{G}-{Cn}-{B}-{seed}/{returnpost}", _flat(a),
                       lambda: _flat(R.log_boot_posterior(mm, flat, off, uci, mag, B, seed=seed, returnpost=returnpost)))


def test_explicit_draws_equal_the_reference_rand_stream():
    """the oracle fed with the draws of orc_boot_indices (what the GPU path is fed with) == the reference drawing inside"""
    w = synth.make_workload(3, n_genes=40, n_cells=31, seed=2)
    mm, lt, sq, mag, flat, off, uci = _prep(w)
    for seed in (1, 7, 40):
        bi = O.boot_indices(seed, 31, 60)
        a = O.log_boot_posterior(mm, flat, off, uci, mag, 60, seed=999, boot_idx=bi)
        _same_as_reference(f"explicit_draws/{seed}", {"jp": a["jp"]},
                           lambda: {"jp": R.log_boot_posterior(mm, flat, off, uci, mag, 60, seed=seed)["jp"]})


def test_no_bootstrap_and_ensemble_bit_exact():
    w = synth.make_workload(3, n_genes=60, n_cells=17, seed=8)
    mm, lt, sq, mag, flat, off, uci = _prep(w)
    for kw in (dict(nboot=0), dict(nboot=10, ensemble=1), dict(nboot=0, ensemble=1)):
        a = O.log_boot_posterior(mm, flat, off, uci, mag, seed=1, **kw)
        _same_as_reference(f"no_bootstrap_ensemble/{kw['nboot']}-{kw.get('ensemble', 0)}", {"jp": a["jp"]},
                           lambda: {"jp": R.log_boot_posterior(mm, flat, off, uci, mag, seed=1, **kw)["jp"]})


@pytest.mark.parametrize("returnpost", [0, 1, 2])
def test_log_boot_batch_posterior_bit_exact(returnpost):
    w = synth.make_workload(5, n_genes=80, n_cells=36, seed=3, batch=True)
    mm, lt, sq, mag, flat, off, uci = _prep(w)
    bc = np.asarray(w.batch.codes)
    pools = [np.nonzero(bc == l)[0].astype(np.int32) for l in range(2)]
    codes = np.asarray(w.groups.codes)
    for lev in (0, 1):
        comp = np.bincount(bc[codes == lev], minlength=2).astype(np.int32)
        a = O.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 100, seed=1, returnpost=returnpost)
        _same_as_reference(f"log_boot_batch_posterior/{returnpost}/{lev}", _flat(a), lambda: _flat(
            R.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 100, seed=1, returnpost=returnpost)))
    # a level with zero composition is skipped by both (src/jpmatLogBoot.cpp:472)
    comp = np.array([0, 9], dtype=np.int32)
    a = O.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 30, seed=5)

    def ref():
        return {"jp": R.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 30, seed=5)["jp"]}

    _same_as_reference("log_boot_batch_posterior/zero_composition", {"jp": a["jp"]}, ref)
    bi = O.batch_boot_indices(5, pools, comp, 30)
    c = O.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 30, seed=77, boot_idx=bi)
    _same_as_reference("log_boot_batch_posterior/zero_composition", {"jp": c["jp"]}, ref)


def test_local_theta_and_square_logit_models_bit_exact():
    """knn.error.models output (data/knn.rda, 12 columns: corr.ltheta.*, conc.a2) -- src/jpmatLogBoot.cpp:136-138,148-176"""
    knn = helpers.knn_models().iloc[:12]
    rng = np.random.default_rng(3)
    counts = rng.negative_binomial(0.8, 0.02, size=(70, len(knn))).astype(np.int32)
    counts[rng.uniform(size=counts.shape) < 0.4] = 0
    mm, lt, sq = O.pack_models(knn)
    assert lt == 1 and sq == 1
    mag = O.marginals_from_prior_x(np.linspace(0, 4.8, 401))
    flat, off, uci = O.unique_counts(counts)
    a = O.log_boot_posterior(mm, flat, off, uci, mag, 50, seed=1, returnpost=3, localtheta=lt, sqlogit=sq)
    _same_as_reference("local_theta_square_logit", _flat(a), lambda: _flat(
        R.log_boot_posterior(mm, flat, off, uci, mag, 50, seed=1, returnpost=3, localtheta=lt, sqlogit=sq)))


def test_es_mef_small_slice_bit_exact():
    """config 1's data: the bundled es.mef.small counts + o.ifm models, a 300-gene slice, both groups"""
    cd, ifm, prior, groups = helpers.es_mef_inputs("tests")
    sub = cd.iloc[1000:1300]
    mm, lt, sq = O.pack_models(ifm)
    mag = O.marginals_from_prior_x(prior["x"].to_numpy())
    codes = np.asarray(groups.codes)
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        flat, off, uci = O.unique_counts(np.asfortranarray(sub.to_numpy()[:, ii]))
        a = O.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1, returnpost=1)
        _same_as_reference(f"es_mef_small_slice/{lev}", _flat(a), lambda: _flat(
            R.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, 100, seed=1, returnpost=1)))


def test_legacy_jpmat_forms_bit_exact():
    rng = np.random.default_rng(11)
    matl = [np.asfortranarray(-rng.gamma(2.0, 3.0, size=(13, 29))) for _ in range(9)]
    _same_as_reference("jpmat_log_boot", {"jp": O.jpmat_log_boot(matl, 40, seed=3)},
                       lambda: {"jp": R.jpmat_log_boot(matl, 40, seed=3)})
    matll = [matl[:4], matl[4:]]
    for comp in (np.array([3, 6], dtype=np.int32), np.array([0, 5], dtype=np.int32)):
        _same_as_reference(f"jpmat_log_batch_boot/{comp[0]}-{comp[1]}",
                           {"jp": O.jpmat_log_batch_boot(matll, comp, 25, seed=2)},
                           lambda: {"jp": R.jpmat_log_batch_boot(matll, comp, 25, seed=2)})


@pytest.mark.parametrize("n", [1, 2, 33, 401])
def test_mat_slide_mult_bit_exact(n):
    rng = np.random.default_rng(n)
    m1, m2 = rng.random((11, n)), rng.random((11, n))
    _same_as_reference(f"mat_slide_mult/{n}", {"out": O.mat_slide_mult(m1, m2)}, lambda: {"out": R.mat_slide_mult(m1, m2)})
