"""Pruned tcgen05 contraction (scde_b200_options.prune_pieces, DESIGN.md 4.3): the (gene, piece) items whose grid points
bounds computed before the gather prove more than 746 nats below every boot's row maximum are not contracted, and the
soft-max skips their points.  Such points add exactly 0.0 to the soft-max, so pruning on and pruning off must agree bit
for bit -- for every call shape that reaches the contraction -- while removing a good share of the gathered items at
realistic group sizes."""
import ctypes as C

import numpy as np
import pandas as pd
import pytest

from scde_b200 import _lib, api, synth

pytestmark = pytest.mark.gpu

KEYS = ["idx", "z", "cz", "batch_idx", "batch_z", "batch_cz", "adjusted_idx", "adjusted_z", "adjusted_cz"]


def _problem(config, G, Cn, seed, batch=False):
    w = synth.make_workload(config, n_genes=G, n_cells=Cn, seed=seed, batch=batch)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    kw = dict(local_theta=lt, sqlogit=sq, zero_index=[len(x)])
    if batch:
        kw.update(batch_codes=np.asarray(w.batch.codes, dtype=np.int32), n_batch_levels=2,
                  zero_index_adjusted=[2 * len(x) - 1])
    return w, (w.counts, mm, x, y, np.asarray(w.groups.codes, dtype=np.int32)), kw


def _both(ctx, run):
    """run() with pruning on and off"""
    out = {}
    for prune in (1, 0):
        keep = ctx.set_options(prune_pieces=prune)
        try:
            out[prune] = run()
        finally:
            ctx.restore_options(keep)
    return out[1], out[0]


def _same(a, b):
    for k in KEYS:
        if k in a:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
    for jk in ("joint_posteriors", "batch_joint_posteriors"):
        for i in range(len(a.get(jk, []))):
            assert np.array_equal(a[jk][i], b[jk][i]), (jk, i)


def _call(ctx, args, kw, n_boot=100, **extra):
    return api.expression_difference_call(ctx, *args, n_boot, 1, joint_posteriors=True, **kw, **extra)


def test_one_shot_equals_unpruned_and_prunes(ctx):
    """2 x 2600 cells: peaked joints -- items are pruned, and nothing changes"""
    _, args, kw = _problem(4, 300, 5200, 11)
    on, off = _both(ctx, lambda: _call(ctx, args, kw))
    _same(on, off)
    st = on["stats"]
    assert st["prune_items"] > 0 and st["prune_live"] < st["prune_items"]
    assert off["stats"]["prune_items"] == 0
    assert st["launches"]["bound"] > 0 and off["stats"]["launches"]["bound"] == 0


def test_resident_job_equals_unpruned(ctx):
    _, args, kw = _problem(4, 200, 5200, 12)

    def job():
        j = api.DifferenceJob(ctx, *args, 100, 1, **kw)
        try:
            res = []
            for _ in range(2):  # repeated runs: the live counts stay on the device
                j.run()
                res.append(j.download(joint_posteriors=True))
            return res
        finally:
            j.close()

    on, off = _both(ctx, job)
    for a, b in zip(on + off[:1], off + on[:1]):
        _same(a, b)


def test_gene_range_draw_chunks_two_passes(ctx):
    """150 randomizations (two passes, paired in one launch) with 10 draw sets, over a gene range"""
    _, args, kw = _problem(4, 220, 5200, 13)
    on, off = _both(ctx, lambda: _call(ctx, args, kw, n_boot=150, n_cores=10, chunked_draws=True, gene_range=(17, 201)))
    _same(on, off)
    assert on["stats"]["prune_live"] < on["stats"]["prune_items"]


def test_batch_factor_twin_launch(ctx):
    """a batch-corrected call: the two composition-sampled joints share the launches (an item is live for both when it is
    live for either)"""
    _, args, kw = _problem(5, 200, 5200, 14, batch=True)
    on, off = _both(ctx, lambda: _call(ctx, args, kw))
    _same(on, off)
    assert on["stats"]["prune_live"] < on["stats"]["prune_items"]


def test_config2_sized_inputs(ctx):
    """40 cells: below the size where pruning pays (PRUNE_MIN_CELLS), so the call does not prune"""
    _, args, kw = _problem(3, 500, 40, 15)
    on, off = _both(ctx, lambda: _call(ctx, args, kw))
    _same(on, off)
    assert on["stats"]["prune_items"] == 0 and on["stats"]["launches"]["bound"] == 0


def test_contrasts_dataset(ctx):
    w = synth.make_workload(5, n_genes=150, n_cells=7800, seed=16, batch=True)
    rng = np.random.default_rng(16)
    groups = pd.Categorical.from_codes(rng.permutation(np.arange(7800) % 3), categories=["A", "B", "C"])

    def run():
        with api.DifferenceSession(w.models, w.counts, w.prior, context=ctx) as s:
            return s.contrasts(groups, contrasts="pairs", batch=w.batch, n_randomizations=100)

    on, off = _both(ctx, run)
    assert on.keys() == off.keys()
    for label in on:
        for key in ("results", "batch.adjusted", "batch.effect"):
            pd.testing.assert_frame_equal(on[label][key], off[label][key], check_exact=True)


def test_two_devices(ctx):
    if _lib.lib().scde_b200_device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    _, args, kw = _problem(4, 200, 5200, 17)
    mctx = _lib.Context(devices=[0, 1])
    try:
        on, off = _both(mctx, lambda: _call(mctx, args, kw))
    finally:
        mctx.close()
    _same(on, off)


def test_prune_rate_at_config4_cells(ctx):
    """config 4's data (10 000 cells, two groups of 5000, B = 100) on 600 genes: at least 30 % of the visited-pair work
    (every (gene, piece) item weighted by its gene's list length) is not gathered"""
    _, args, kw = _problem(4, 600, 10000, None)
    res = _call(ctx, args, kw)
    st = res["stats"]
    share = 1.0 - st["prune_live_work"] / st["prune_work"]
    print(f"pruned share of the gather at config-4 cells: {share:.3f} (items: {1 - st['prune_live'] / st['prune_items']:.3f})")
    assert share >= 0.30


# ---- the bounds themselves ---------------------------------------------------------------------------------------------
Q_PW, Q_PIECE, UB_PTS, UB_N, LB_STEP, LB_OFF, LB_N = 102, 512, 16, 26, 12, 6, 35
WP, KP = 104, 416


def _table(ctx, n_genes, n_cells, seed, K=None, inputs=None, **options):
    """the fused table of a config-4-like workload -- or of inputs = (models, counts) -- on the prior's grid or on one of K
    points, with its bound rows (scde_b200_probe_table_bounds), under the given scde_b200_options fields"""
    if inputs is None:
        w = synth.make_workload(4, n_genes=n_genes, n_cells=n_cells, seed=seed)
        inputs = w.models, w.counts
    counts = np.asarray(inputs[1], dtype=np.int32)
    n_cells = counts.shape[1]
    mm, lt, sq = api.pack_models(inputs[0])
    mm = np.asfortranarray(mm, dtype=np.float64)
    x = synth.make_prior(n_genes, length_out=(K or 401) - 1)["x"].to_numpy()
    K = len(x)
    with np.errstate(divide="ignore"):
        mag = np.log(np.maximum(10.0 ** x - 1.0, 0.0))
    flat, off, uci = api._unique_index(counts)
    n_rows = int(off[-1])
    out = dict(q=np.zeros((n_rows, -(-K // Q_PW) * Q_PIECE), np.int8), rr=np.zeros(n_rows, np.uint32),
               zero_row=np.empty(n_cells, np.int32), based=np.empty(n_cells, np.int32), zero_rows=np.empty((n_cells, K)),
               qb=np.full((n_rows, 128), 0x55, np.int8))  # (not a bound row: a row the probe leaves unwritten shows)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    keep = ctx.set_options(**options)
    try:
        _lib.check(_lib.lib().scde_b200_probe_table_bounds(
            ctx.handle, _lib.p_f64(mm), n_cells, _lib.p_i32(np.ascontiguousarray(flat, np.int32)), _lib.p_i32(off),
            _lib.p_f64(np.ascontiguousarray(mag)), K, lt, sq, n_cells, vp(out["q"]), vp(out["rr"]),
            _lib.p_i32(out["zero_row"]), _lib.p_i32(out["based"]), _lib.p_f64(out["zero_rows"]), vp(out["qb"])))
    finally:
        ctx.restore_options(keep)
    out.update(counts=counts, off=off, uci=uci, K=K)
    return out


def _values(q, K):
    """x = 2^29 D of every row and grid point, from the planes"""
    k = np.arange(K)
    pc, i = k // Q_PW, k % Q_PW
    x = np.zeros((q.shape[0], K), np.int64)
    for pl in range(4, -1, -1):
        x = x * 256 + q[:, pc * Q_PIECE + pl * Q_PW + i].astype(np.int64)
    return x


def test_bound_rows_are_directed_bounds_of_the_planes(ctx):
    """every bound row the row kernels wrote equals the one recomputed on the host from its planes: ceil(max x / 2^24)
    over the admissible points of each block (so >= every admissible value), floor(x / 2^24) at each sample"""
    t = _table(ctx, 120, 2000, 31)
    K, q, rr = t["K"], t["q"], t["rr"]
    regular = rr != 0xFFFFFFFF
    assert regular.mean() > 0.99
    x = _values(q[regular], K)
    klo, khi = (rr[regular] & 0xFFFF).astype(np.int64), (rr[regular] >> 16).astype(np.int64)
    k = np.arange(K)
    adm = (k[None, :] >= klo[:, None]) & (k[None, :] <= khi[:, None])
    qb = t["qb"][regular].astype(np.int64)
    got = qb[:, :64] + 256 * qb[:, 64:]
    big = np.iinfo(np.int64).min
    for u in range(UB_N):
        blk = slice(u * UB_PTS, min((u + 1) * UB_PTS, K))
        m = np.where(adm[:, blk], x[:, blk], big).max(axis=1)
        want = np.where(m == big, 0, -((-m) // (1 << 24)))
        assert np.array_equal(got[:, u], want), u
        has = m != big
        assert np.all(got[has, u] * (1 << 24) >= m[has])
    for c in range(LB_N):
        kc = LB_STEP * c + LB_OFF
        want = x[:, kc] // (1 << 24) if kc < K else np.zeros(len(x), np.int64)
        assert np.array_equal(got[:, UB_N + c], want), c
    assert not got[:, UB_N + LB_N:].any()


def test_pruned_items_are_invisible_to_the_softmax(ctx):
    """2000 cells, 104 boots: the unpruned T (scde_b200_probe_prune_i8) against the decision's own bounds -- every LB is at
    most its boot's row maximum, every UB at least its piece's admissible maximum, and every admissible value of a pruned
    piece lies more than 746 nats below the maximum for every boot; exp_nonpos is exactly 0 from -746 on"""
    n_cells, G = 2000, 120
    t = _table(ctx, G, n_cells, 32)
    K = t["K"]
    rng = np.random.default_rng(32)
    drawable = np.flatnonzero((t["based"] != 0) & (t["zero_row"] >= 0))
    draws = rng.choice(drawable, size=(WP, n_cells), replace=True)
    W = np.zeros((n_cells, WP), np.int64)
    for b in range(WP):
        np.add.at(W[:, b], draws[b], 1)
    assert W.max() <= 127
    n_w_rows = (n_cells + 1 + 15) // 16 * 16
    w8 = np.zeros((n_w_rows, 128), np.int8)
    w8[:n_cells, :WP] = W
    Z = np.zeros((WP, KP))
    Z[:, :K] = W[drawable].T.astype(np.float64) @ t["zero_rows"][drawable]
    lists = []
    for g in range(G):
        cells = drawable[t["counts"][g, drawable] > 0]
        lists.append((t["off"][cells] + t["uci"][g, cells], cells))
    ld = max(32, (max(len(c) for _, c in lists) + 31) // 32 * 32)
    lst_row = np.zeros((G, ld), np.int32)
    lst_cell = np.full((G, ld), n_cells, np.int32)  # padding: the all-zero W row
    lst_len = np.zeros(G, np.int32)
    for g, (rows, cells) in enumerate(lists):
        lst_row[g, :len(rows)], lst_cell[g, :len(cells)], lst_len[g] = rows, cells, len(rows)
    T = np.zeros((G, WP, KP))
    lb, ub = np.zeros((G, WP)), np.zeros((G, WP, 4))
    live, ex, flags = np.zeros(G, np.uint8), np.zeros(3), np.zeros(1, np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(_lib.lib().scde_b200_probe_prune_i8(
        ctx.handle, vp(t["q"]), t["q"].shape[0], K, vp(t["rr"]), vp(t["qb"]), vp(Z), vp(w8), n_w_rows, vp(lst_row),
        vp(lst_cell), vp(lst_len), G, ld, vp(T), vp(lb), vp(ub), vp(live), vp(ex), vp(flags)))
    assert ex[0] > 0.0 and ex[1] == 0.0 and ex[2] == 0.0
    assert flags[0] == 0
    adm = T[:, :, :K] > -1e299
    full = np.where(adm, T[:, :, :K] + Z[None, :, :K], -np.inf)
    m = full.max(axis=2)
    assert np.all(np.isfinite(m))
    assert np.all(lb <= m + 1e-6 * np.abs(m))
    n_dead = 0
    for p in range(4):
        sl = slice(p * Q_PW, min((p + 1) * Q_PW, K))
        pm = full[:, :, sl].max(axis=2)
        has = np.isfinite(pm)
        assert np.all(ub[:, :, p][has] >= pm[has] - 1e-6 * np.abs(pm[has])), p
        dead = ((live >> p) & 1) == 0
        n_dead += int(dead.sum())
        assert np.all(pm[dead] < m[dead] - 746.0), p
    assert n_dead > 0  # the check above bites
