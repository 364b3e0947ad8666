"""Draw chunks (the reference's n.cores > 1): scde.posteriors splits the genes into n contiguous chunks and draws every
chunk's randomizations with Seed = its first gene (R/functions.R:606-617).  The library computes every chunk's draw set in
the same contraction launches (scde_b200_diff_args.draw_chunks); these tests pin it bit for bit to unchunked calls over
each chunk's genes with the chunk's seed, and within tolerance to the reference's own per-chunk loop restated on the
oracle.  Host-only tests are unmarked; the rest need a GPU."""
import ctypes as C
import os

import numpy as np
import pandas as pd
import pytest

import helpers
from oracle import oracle as O
from scde_b200 import _lib, api, synth

LOGP_RTOL = 1e-6


def chunked_reference(w, n_cores, nboot=100, seed=1, batch_codes=None, batch_models=None):
    """scde.expression.difference at n.cores = n_cores on the oracle: per gene chunk [b, e) the reference's own .Call
    sequence (unique counts of the chunk, logBootPosterior / logBootBatchPosterior with Seed = seed + b), joint posteriors
    stacked (rbind), then the ratio posteriors and summaries over all genes."""
    counts = np.asarray(w.counts, dtype=np.int32)
    codes = np.asarray(w.groups.codes)
    gidx = (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0])
    mm, lt, sq = O.pack_models(w.models)
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    chunks = api.draw_chunk_ranges(counts.shape[0], n_cores)
    jpl = []
    for ii in gidx:
        parts = []
        for b, e in chunks:
            flat, off, uci = O.unique_counts(np.asfortranarray(counts[b:e][:, ii]))
            parts.append(O.log_boot_posterior(np.asfortranarray(mm[ii]), flat, off, uci, mag, nboot, seed=seed + b,
                                              localtheta=lt, sqlogit=sq)["jp"])
        jpl.append(np.vstack(parts))
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    bdiffp = O.ratio_posterior(jpl[0], jpl[1], y)
    diffv = O.fold_change_grid(x)
    res, idx = O.distribution_summary(bdiffp, diffv, 0.0)
    out = {"results": res, "idx": idx, "joint.posteriors": jpl}
    if batch_codes is None:
        return out
    bcodes = np.asarray(batch_codes)
    L = int(bcodes.max()) + 1
    pools = [np.nonzero(bcodes == l)[0].astype(np.int32) for l in range(L)]
    bmm, blt, bsq = (mm, lt, sq) if batch_models is None else O.pack_models(batch_models)
    bjpl = []
    for ii in gidx:
        bc = bcodes[ii]
        comp = np.bincount(bc[bc >= 0], minlength=L).astype(np.int32)
        parts = []
        for b, e in chunks:
            flat, off, uci = O.unique_counts(np.asfortranarray(counts[b:e]))
            parts.append(O.log_boot_batch_posterior(bmm, flat, off, uci, mag, pools, comp, nboot, seed=seed + b,
                                                    localtheta=blt, sqlogit=bsq)["jp"])
        bjpl.append(np.vstack(parts))
    bb = O.ratio_posterior(bjpl[0], bjpl[1], y)
    bres, bidx = O.distribution_summary(bb, diffv, 0.0)
    ab = O.ratio_posterior(bdiffp, bb, None)
    ares, aidx = O.distribution_summary(ab, O.fold_change_grid(diffv), 0.0)
    out.update({"batch.idx": bidx, "batch.results": bres, "adjusted.idx": aidx, "adjusted.results": ares,
                "batch.joint.posteriors": bjpl})
    return out


def _logp_close(a, b, rtol=LOGP_RTOL, floor=1e-290):
    a, b = np.asarray(a), np.asarray(b)
    big = (a > floor) & (b > floor)
    la, lb = np.log(a[big]), np.log(b[big])
    return bool(np.all(np.abs(la - lb) <= rtol * np.maximum(np.abs(lb), 1.0)) and
                np.all(np.abs(a[~big] - b[~big]) <= 1e-280))


def _z_close(got, want):
    tol = np.where(want < -6.0, 2e-4, 1e-6 * np.maximum(1.0, np.abs(want)) + 1e-9)
    assert not (np.abs(got - want) > tol).any(), float(np.max(np.abs(got - want)))


# ------------------------------------------------------------------------------------------------ host only
@pytest.mark.parametrize("G,n", [(20, 5), (203, 7), (6, 5), (5, 5), (3, 5), (20, 1), (20, 0)])
def test_chunk_ranges_equal_r_expression(G, n):
    got = api.draw_chunk_ranges(G, n)
    if n > 1 and G > n:
        lab = np.sort(np.resize(np.arange(1, n + 1), G))  # sort(rep_len(1:n, G))
        want = [(int(np.nonzero(lab == i)[0][0]), int(np.nonzero(lab == i)[0][-1]) + 1) for i in range(1, n + 1)]
    else:
        want = [(0, G)]  # one draw set with `seed`
    assert got == want


def test_chunked_reference_equals_unchunked_on_first_chunk():
    w = synth.make_workload(3, n_genes=60, n_cells=30, seed=17)
    codes = np.asarray(w.groups.codes)
    one = O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                  (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=50, seed=1)
    five = chunked_reference(w, 5, nboot=50)
    b, e = api.draw_chunk_ranges(60, 5)[0]
    for i in range(2):
        np.testing.assert_allclose(five["joint.posteriors"][i][b:e], one["joint.posteriors"][i][b:e], rtol=1e-13, atol=0)
        assert not np.allclose(five["joint.posteriors"][i][e:], one["joint.posteriors"][i][e:], rtol=1e-6, atol=0)
    assert np.array_equal(five["idx"][b:e], one["idx"][b:e])


def test_chunked_draws_with_explicit_draws_is_refused_before_the_library():
    w = synth.make_workload(3, n_genes=20, n_cells=12, seed=2)
    bi = np.zeros((10, 6), dtype=np.int32)
    with pytest.raises(ValueError, match="boot_idx"):
        api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, n_randomizations=10, n_cores=4,
                                       chunked_draws=True, boot_idx=(bi, None, None, None))
    with pytest.raises(ValueError, match="boot_idx"):
        api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=10, n_cores=4, chunked_draws=True,
                            boot_idx=np.zeros((10, 12), dtype=np.int32))
    with pytest.raises(ValueError, match="boot_idx"):
        api.expression_difference_call(None, w.counts, np.zeros((12, 12)), w.prior["x"], w.prior["y"],
                                       np.zeros(12, np.int32), 10, n_cores=4, chunked_draws=True,
                                       boot_idx=(bi, None, None, None))


# ------------------------------------------------------------------------------------------------ GPU
def _problem(mode, G=203, Cn=64, seed=23):
    batch = mode != "plain"
    w = synth.make_workload(5 if batch else 3, n_genes=G, n_cells=Cn, seed=seed, batch=batch)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    kw = dict(local_theta=lt, sqlogit=sq, zero_index=[len(x)], joint_posteriors=True)
    bmodels = None
    if batch:
        kw.update(batch_codes=np.asarray(w.batch.codes, dtype=np.int32), n_batch_levels=2,
                  zero_index_adjusted=[2 * len(x) - 1])
    if mode == "batch_models":
        bmodels = w.models.copy()
        bmodels["fail.r"] = bmodels["fail.r"] + 0.25
        kw.update(batch_mm=api.pack_models(bmodels)[0], batch_local_theta=lt, batch_sqlogit=sq)
    return w, mm, x, y, np.asarray(w.groups.codes, dtype=np.int32), kw, bmodels


SUMMARY_KEYS = ["idx", "z", "batch_idx", "batch_z", "adjusted_idx", "adjusted_z"]


@pytest.mark.gpu
@pytest.mark.parametrize("n,mode,n_boot,kernel",
                         [(n, m, 100, 0) for n in (2, 7, 20) for m in ("plain", "batch", "batch_models")] +
                         [(7, "plain", 150, 0), (7, "batch", 150, 0)] +  # 150: two passes (paired passes, twin joints)
                         # the FP64 kernels with sets: DMMA (the fallback of a flagged joint) and generic
                         [(7, m, nb, k) for k in (1, 2) for m in ("plain", "batch") for nb in (100, 150)])
def test_chunked_call_equals_unchunked_calls_per_chunk(ctx, n, mode, n_boot, kernel):
    w, mm, x, y, codes, kw, _ = _problem(mode)
    G = w.counts.shape[0]
    ctx.set_contract_kernel(kernel)
    try:
        _compare_chunks(ctx, w, mm, x, y, codes, kw, n, n_boot, api.draw_chunk_ranges(G, n))
    finally:
        ctx.set_contract_kernel(0)


@pytest.mark.gpu
def test_chunks_at_the_cap(ctx):
    """256 draw sets (the cap) on 300 genes: chunks of one and two genes, every contraction launch over all sets"""
    w, mm, x, y, codes, kw, _ = _problem("batch", G=300, Cn=40, seed=61)
    ranges = api.draw_chunk_ranges(300, 256)
    assert len(ranges) == 256
    _compare_chunks(ctx, w, mm, x, y, codes, kw, 256, 100, [ranges[i] for i in (0, 1, 43, 44, 127, 200, 255)])


def _compare_chunks(ctx, w, mm, x, y, codes, kw, n, n_boot, ranges):
    """rows [b, e) of the chunked call == an unchunked call over [b, e) with seed 1 + b, for every (b, e) of ranges;
    cZ == BH of the gathered Z"""
    G = w.counts.shape[0]
    got = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, n_boot, 1, n_cores=n, chunked_draws=True, **kw)
    keys = [k for k in SUMMARY_KEYS if k in got]
    jkeys = [k for k in ("joint_posteriors", "batch_joint_posteriors") if k in got]
    for b, e in ranges:
        want = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, n_boot, 1 + b, gene_range=(b, e), **kw)
        for k in keys:
            assert np.array_equal(got[k][b:e], want[k]), (k, b, e)
        for k in jkeys:
            for i in range(2):
                assert np.array_equal(got[k][i][b:e], want[k][i]), (k, i, b, e)
    for k in ("", "batch_", "adjusted_"):
        if k + "z" in got:
            cz = np.empty(G)
            _lib.check(_lib.lib().scde_b200_bh_cz(_lib.p_f64(np.ascontiguousarray(got[k + "z"])), G, _lib.p_f64(cz)))
            assert np.array_equal(got[k + "cz"], cz), k


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 2])
@pytest.mark.parametrize("mode", ["plain", "batch"])
def test_chunked_call_against_chunked_reference(ctx, kernel, mode):
    w, mm, x, y, codes, kw, _ = _problem(mode, G=157, Cn=48, seed=31)
    want = chunked_reference(w, 7, batch_codes=kw.get("batch_codes"))
    ctx.set_contract_kernel(kernel)
    try:
        got = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, 100, 1, n_cores=7, chunked_draws=True, **kw)
    finally:
        ctx.set_contract_kernel(0)
    for i in range(2):
        assert _logp_close(got["joint_posteriors"][i], want["joint.posteriors"][i]), i
    assert np.array_equal(got["idx"], want["idx"])
    _z_close(got["z"], want["results"][:, 4])
    if mode == "batch":
        for i in range(2):
            assert _logp_close(got["batch_joint_posteriors"][i], want["batch.joint.posteriors"][i]), i
        assert np.array_equal(got["batch_idx"], want["batch.idx"])
        assert np.array_equal(got["adjusted_idx"], want["adjusted.idx"])
        _z_close(got["batch_z"], want["batch.results"][:, 4])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["plain", "batch"])
def test_resident_job_and_two_devices_equal_one_shot(ctx, mode):
    w, mm, x, y, codes, kw, _ = _problem(mode, G=211, Cn=56, seed=37)
    one = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, 100, 1, n_cores=10, chunked_draws=True, **kw)
    jkw = {k: v for k, v in kw.items() if k != "joint_posteriors"}
    job = api.DifferenceJob(ctx, w.counts, mm, x, y, codes, 100, 1, n_cores=10, chunked_draws=True, **jkw)
    try:
        for _ in range(2):
            job.run()
            res = job.download(joint_posteriors=True)
            for k in [k for k in SUMMARY_KEYS if k in one]:
                assert np.array_equal(res[k], one[k]), k
            for i in range(2):
                assert np.array_equal(res["joint_posteriors"][i], one["joint_posteriors"][i])
    finally:
        job.close()
    # a gene range holds the draw sets of the chunks it meets, with their global seeds
    sub = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, 100, 1, n_cores=10, chunked_draws=True,
                                         gene_range=(30, 140), **kw)
    assert np.array_equal(sub["z"], one["z"][30:140]) and np.array_equal(sub["idx"], one["idx"][30:140])
    if _lib.lib().scde_b200_device_count() < 2:
        pytest.skip("the two-device half needs 2 CUDA devices")
    mctx = _lib.Context(devices=[0, 1])
    try:
        two = api.expression_difference_call(mctx, w.counts, mm, x, y, codes, 100, 1, n_cores=10, chunked_draws=True, **kw)
    finally:
        mctx.close()
    for k in [k for k in SUMMARY_KEYS + ["cz"] if k in one]:
        assert np.array_equal(two[k], one[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("contrasts", ["pairs", "rest"])
def test_contrasts_equal_one_shot_calls(ctx, contrasts):
    w = synth.make_workload(5, n_genes=190, n_cells=72, seed=43, batch=True)
    rng = np.random.default_rng(43)
    groups = pd.Categorical.from_codes(rng.permutation(np.arange(72) % 3), categories=["A", "B", "C"])
    with api.DifferenceSession(w.models, w.counts, w.prior, context=ctx) as s:
        got = s.contrasts(groups, contrasts=contrasts, batch=w.batch, n_randomizations=100, n_cores=20,
                          chunked_draws=True)
    for label, la, lb, na, nb in api.expand_contrasts(["A", "B", "C"], contrasts):
        g = np.asarray(groups.astype(object))
        two = pd.Categorical.from_codes(np.where(np.isin(g, la), 0, np.where(np.isin(g, lb), 1, -1)), categories=[na, nb])
        want = api.scde_expression_difference(w.models, w.counts, w.prior, groups=two, batch=w.batch,
                                              n_randomizations=100, n_cores=20, chunked_draws=True, context=ctx)
        for key in ("results", "batch.adjusted", "batch.effect"):
            pd.testing.assert_frame_equal(got[label][key], want[key], check_exact=True)


@pytest.mark.gpu
def test_one_contraction_launch_whatever_the_chunks(ctx):
    w, mm, x, y, codes, kw, _ = _problem("batch", G=400, Cn=64, seed=47)
    launches = {}
    for n in (1, 20):
        res = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, 150, 1, n_cores=n, chunked_draws=True, **kw)
        launches[n] = res["stats"]["launches"]
    assert launches[20]["contract"] == launches[1]["contract"], launches
    assert launches[20]["softmax"] == launches[1]["softmax"], launches


@pytest.mark.gpu
def test_argument_errors_leave_the_context_usable(ctx):
    w, mm, x, y, codes, kw, _ = _problem("plain", G=40, Cn=24, seed=5)
    base = dict(kw)
    cases = [
        (dict(draw_chunks=-1), -1, "draw_chunks -1 < 0"),
        (dict(draw_chunks=3, boot_idx=True), -1, "cannot be combined with explicit boot_idx"),
        (dict(draw_chunks=257), -5, "above SCDE_B200_MAX_DRAW_CHUNKS"),
    ]
    n0 = int(np.sum(codes == 0))
    for extra, code, msg in cases:
        boot = (np.zeros((10, n0), np.int32), None, None, None) if extra.get("boot_idx") else (None,) * 4
        a, keep, G, K, hb = api._diff_args(w.counts, mm, x, y, codes, 10, 1, None, 0, base["zero_index"], None,
                                           base["local_theta"], base["sqlogit"], boot, (0, 0),
                                           draw_chunks=extra["draw_chunks"])
        o, res = api._diff_out(G, K, hb, False, False)
        rc = _lib.lib().scde_b200_expression_difference(ctx.handle, C.byref(a), C.byref(o), None)
        assert rc == code, (extra, rc)
        assert msg in _lib.lib().scde_b200_last_error().decode()
        del keep
    ok = api.expression_difference_call(ctx, w.counts, mm, x, y, codes, 10, 1, n_cores=256, chunked_draws=True, **kw)
    assert np.isfinite(ok["z"]).all()


@pytest.mark.gpu
def test_python_api_and_r_shim_against_reference(ctx):
    w = synth.make_workload(3, n_genes=173, n_cells=40, seed=53)
    want = chunked_reference(w, 10)
    got = api.scde_expression_difference(w.models, w.counts, w.prior, groups=w.groups, n_randomizations=100,
                                         n_cores=10, chunked_draws=True, return_posteriors=True, context=ctx)
    lev = list(w.groups.categories)
    for i in range(2):
        assert _logp_close(got["joint.posteriors"][lev[i]].to_numpy(), want["joint.posteriors"][i])
    _z_close(got["results"]["Z"].to_numpy(), want["results"][:, 4])
    # scde.posteriors: one library call per chunk, as the reference
    codes = np.asarray(w.groups.codes)
    cells = w.models.index[codes == 0]
    cdf = pd.DataFrame(np.asarray(w.counts), index=[f"g{i}" for i in range(w.counts.shape[0])], columns=w.models.index)
    jp = api.scde_posteriors(w.models.loc[cells], cdf, w.prior, n_randomizations=100, n_cores=5, chunked_draws=True,
                             context=ctx)
    mm, lt, sq = O.pack_models(w.models.loc[cells])
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    counts = np.asarray(w.counts, dtype=np.int32)[:, codes == 0]
    parts = []
    for b, e in api.draw_chunk_ranges(counts.shape[0], 5):
        flat, off, uci = O.unique_counts(np.asfortranarray(counts[b:e]))
        parts.append(O.log_boot_posterior(np.asfortranarray(mm), flat, off, uci, mag, 100, seed=1 + b, localtheta=lt,
                                          sqlogit=sq)["jp"])
    assert _logp_close(jp.to_numpy(), np.vstack(parts))
    # the R shim's fused entry with DrawChunks
    path = os.path.abspath(os.path.join(helpers.GOLD, "..", "..", "integration", "_build", "libscde_shim.so"))
    if not os.path.exists(path):
        pytest.fail("integration/_build/libscde_shim.so is missing: __graft_entry__.build() builds it (make -C integration)")
    shim = C.CDLL(path)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    K, G, Cn = len(x), 173, 40
    cnt = np.asfortranarray(w.counts, dtype=np.int32)
    g = codes.astype(np.int32)
    idx, z, cz = np.zeros(3 * G), np.zeros(G), np.zeros(G)
    err = C.create_string_buffer(256)
    dev = np.zeros(1, dtype=np.int32)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    rc = shim.shim_diff_chunked(cnt.ctypes.data_as(ip), G, Cn, np.asfortranarray(mm).ctypes.data_as(dp),
                                x.ctypes.data_as(dp), y.ctypes.data_as(dp), K, g.ctypes.data_as(ip), None, 0, 100, K,
                                2 * K - 1, dev.ctypes.data_as(ip), 1, 10, idx.ctypes.data_as(dp), z.ctypes.data_as(dp),
                                cz.ctypes.data_as(dp), err)
    assert rc == 0, err.value
    assert np.array_equal(idx.reshape(3, G).T, want["idx"])
    _z_close(z, want["results"][:, 4])
    np.testing.assert_array_equal(z, got["results"]["Z"].to_numpy())
