"""Piece pruning (DESIGN.md 4.3 "Pruned pieces") against references that do not share its code.

Pruning leaves a result unchanged only if every bound row is a directed bound of the planes the contraction sums and the
bound pass decides on those sums as documented.  The tests here check, for every producer of the table:

1. each bound row element by element against the layout of common.cuh recomputed on the host from the decoded planes
   and the row's range, and against the oracle's table values (the planes' own tolerance);
2. the bound pass's LB, UB and live pieces against the numpy restatement of the decision, on grids of one to four pieces
   and on tables whose lists hold the zero-count rows of unbased cells, and that a dead piece is invisible to the soft-max;
3. pruned calls at pruning sizes (2600 - 3000 cells per joint) against the CPU oracle and the FP64 DMMA kernel, which
   never prunes, as well as against the same call without pruning.
"""
import functools

import ctypes as C
import numpy as np
import pandas as pd
import pytest

import helpers
from oracle import oracle as O
from scde_b200 import _lib, api, synth
from test_bound_pass import _decision
from test_gpu_parity import _logp_close, _z_close
from test_prune_pieces import KP, LB_N, LB_OFF, LB_STEP, Q_PW, UB_N, UB_PTS, WP, _same, _table
from test_table_rows import (GRID_IDS, GRIDS, LOCAL_GRIDS, LONG_COUNTS, PRODUCERS, Q_RANGE_IRREGULAR, SCALE,
                             SENTINEL_ZERO_MODEL, Case, _extreme_models, _frame, fast_case, local_case, probe,
                             row_reference)

pytestmark = pytest.mark.gpu

BSLOTS = 64
UNIT = 1 << 24  # a bound is x / 2^24 (units of 2^-5 nat) with x = 2^29 D


# ---- 1. bound rows --------------------------------------------------------------------------------------------------------
def host_bound_rows(X, rr, K):
    """the bound rows of rows X [n][K] (x = 2^29 D) with regular ranges rr, as common.cuh lays them out: slot u < 26 is
    ceil(max x / 2^24) over the admissible points of block [16 u, 16 u + 16) (0 when it has none), slot 26 + c is
    floor(x / 2^24) at 12 c + 6 (0 at a sentinel or at k >= K), every other slot 0"""
    k = np.arange(K)
    adm = (k[None, :] >= (rr & 0xFFFF).astype(np.int64)[:, None]) & (k[None, :] <= (rr >> 16).astype(np.int64)[:, None])
    out = np.zeros((len(X), BSLOTS), np.int64)
    for u in range(UB_N):
        if u * UB_PTS >= K:
            continue
        blk = slice(u * UB_PTS, min((u + 1) * UB_PTS, K))
        has = adm[:, blk].any(axis=1)
        m = np.where(adm[:, blk], X[:, blk], np.iinfo(np.int64).min).max(axis=1)
        out[:, u] = np.where(has, -((-np.where(has, m, 0)) // UNIT), 0)
    for c in range(LB_N):
        kc = LB_STEP * c + LB_OFF
        if kc < K:
            out[:, UB_N + c] = np.where(adm[:, kc], X[:, kc] // UNIT, 0)
    return out


def slots(qb):
    """the bound slots of bound rows qb [n][128]: two signed radix-256 digits, bytes i and 64 + i"""
    qb = np.asarray(qb).view(np.int8).astype(np.int64)
    return qb[:, :BSLOTS] + 256 * qb[:, BSLOTS:]


def check_bound_rows(case, out):
    """every bound row of a regular row: exactly the host's, directed over the planes, and bounds of the oracle's values
    within the planes' tolerance (one unit of 2^-29 where the element is normal, 0.7 below); returns coverage counters"""
    K = case.K
    k = np.arange(K)
    X, rr = out["X"], out["range"]
    got = slots(out["qb"])
    regular = rr != Q_RANGE_IRREGULAR
    klo, khi = (rr & 0xFFFF).astype(np.int64), (rr >> 16).astype(np.int64)
    want = host_bound_rows(X[regular], rr[regular], K)
    bad = np.nonzero((got[regular] != want).any(axis=1))[0]
    if len(bad):
        r = np.nonzero(regular)[0][bad[0]]
        s = np.nonzero(got[r] != want[bad[0]])[0]
        pytest.fail(f"{len(bad)} bound rows differ from the host's; row {r} (range {klo[r]}..{khi[r]}), slots {s.tolist()}: "
                    f"got {got[r, s].tolist()}, want {want[bad[0], s].tolist()}")
    # directed over the planes (implied by the above; stated on its own so that a failure names the broken promise)
    adm = (k[None, :] >= klo[:, None]) & (k[None, :] <= khi[:, None]) & regular[:, None]
    ub_k = got[:, k // UB_PTS] * UNIT
    assert np.all(np.where(adm, X <= ub_k, True)), "a UB below an admissible plane value of its block"
    for c in range(LB_N):
        kc = LB_STEP * c + LB_OFF
        if kc < K:
            assert np.all(np.where(adm[:, kc], got[:, UB_N + c] * UNIT <= X[:, kc], True)), f"LB sample {c} above its value"
    # bounds of the reference
    seen = {"rows": int(regular.sum()), "irregular": int((~regular).sum()), "partial_range": 0, "rows_at_K": 0,
            "checked_points": 0}
    for c in range(case.n_cells):
        for j, x in enumerate(case.lists[c]):
            r = case.off[c] + j
            if not regular[r]:
                continue
            seen["partial_range"] += int(klo[r] > 0 or khi[r] < K - 1)
            seen["rows_at_K"] += int(K % UB_PTS != 0 and khi[r] >= (K - 1) // UB_PTS * UB_PTS)
            wv, normal, both, c_row = row_reference(case, out, c, j)
            v = wv + c_row
            with np.errstate(over="ignore", invalid="ignore"):  # ("log 0" elements, outside `both`)
                t = np.rint(v * SCALE)
            ub = got[r, k // UB_PTS]
            lb_at = np.full(K, np.iinfo(np.int64).min)
            ks = LB_STEP * np.arange(LB_N) + LB_OFF
            ks_in = ks < K
            lb_at[ks[ks_in]] = got[r, UB_N + np.arange(LB_N)[ks_in]]
            is_lb = lb_at != np.iinfo(np.int64).min
            where = f"cell {c} count {x} (row {r}, range {klo[r]}..{khi[r]}, constant {c_row:.6f})"
            nm, low = both & normal, both & ~normal
            assert np.all(t[nm] <= ub[nm] * UNIT + 1), f"{where}: the oracle lies above UB at k = {k[nm][t[nm] > ub[nm] * UNIT + 1]}"
            assert np.all(v[low] <= ub[low] / 32.0 + 0.7), f"{where}: the oracle lies above UB (low elements)"
            s = nm & is_lb
            assert np.all(lb_at[s] * UNIT <= t[s] + 1), f"{where}: LB above the oracle at k = {k[s][lb_at[s] * UNIT > t[s] + 1]}"
            s = low & is_lb
            assert np.all(lb_at[s] / 32.0 <= v[s] + 0.7), f"{where}: LB above the oracle (low elements)"
            seen["checked_points"] += int(both.sum())
    return seen


def _bound_case(ctx, case, what, **options):
    out = probe(ctx, case, bounds=True, **options)
    seen = check_bound_rows(case, out)
    print(what, f"K={case.K}", seen)
    assert seen["partial_range"] > 0, "no row with a partial range: the range clipping is not exercised"
    if case.K % UB_PTS:
        assert seen["rows_at_K"] > 0, "no row reaches the block that crosses K"
    return seen


@pytest.mark.parametrize("gi", range(len(GRIDS)), ids=GRID_IDS)
@pytest.mark.parametrize("producer", list(PRODUCERS))
def test_bound_rows_every_producer(ctx, producer, gi):
    """lp_rows_q_kernel (both instances), q_bound_row in lp_rows_fast_kernel (staged planes, and the zero-count rows of
    every compact table) and in quantize_rows_kernel, over the eight grids of test_table_rows"""
    _bound_case(ctx, fast_case(gi), producer, **PRODUCERS[producer])


@pytest.mark.parametrize("gi", LOCAL_GRIDS, ids=[GRID_IDS[g] for g in LOCAL_GRIDS])
def test_bound_rows_local_theta(ctx, gi):
    """local-theta, square-logit models (knn fit): FP64 rows of the general kernel, bound rows from the quantize pass"""
    _bound_case(ctx, local_case(gi), "local_theta")


@functools.lru_cache(maxsize=None)
def extreme_case(gi):
    """the high-theta, steep drop-out and unbased models of test_table_rows, every decade of counts, and a cell of the
    unbased model without a zero count"""
    K, x0, clamp = GRIDS[gi]
    models = _extreme_models() + [SENTINEL_ZERO_MODEL]
    lists = [LONG_COUNTS] * (len(models) - 1) + [LONG_COUNTS[1:]]
    return Case(models, lists, K, x0, clamp)


@pytest.mark.parametrize("gi", [1, 3, 5], ids=[GRID_IDS[g] for g in (1, 3, 5)])
@pytest.mark.parametrize("producer", list(PRODUCERS))
def test_bound_rows_extreme_models(ctx, producer, gi):
    _bound_case(ctx, extreme_case(gi), "extreme " + producer, **PRODUCERS[producer])


# ---- 2. the decision on those tables ---------------------------------------------------------------------------------------
DECISION_K = [102, 204, 306, 383, 401, 408]
DECISION_TABLES = ["q_kernel", "quantize_pass", "local_theta", "unbased"]


@functools.lru_cache(maxsize=None)
def decision_inputs(kind, n_genes=60, n_cells=1500, seed=41):
    """(models, counts) of a decision case: config-4 cells, knn models tiled to n_cells, or config-4 cells mixed with cells
    of the unbased model (a third of the genes zero in those)"""
    if kind == "local_theta":
        knn = helpers.knn_models()
        reps = -(-n_cells // len(knn))
        models = pd.concat([knn] * reps)
        models.index = [f"cell{i}" for i in range(len(models))]
        counts = synth.make_counts(np.random.default_rng(seed), models, n_genes)
        return models, counts
    w = synth.make_workload(4, n_genes=n_genes, n_cells=n_cells, seed=seed)
    if kind != "unbased":
        return w.models, w.counts
    n_un = 100
    rows = [r for r in api.pack_models(w.models)[0]] + [SENTINEL_ZERO_MODEL] * n_un
    models = _frame(rows)
    counts = np.zeros((n_genes, n_cells + n_un), np.int32, order="F")
    counts[:, :n_cells] = w.counts
    counts[:, n_cells:] = synth.make_counts(np.random.default_rng(seed + 1), models.iloc[n_cells:], n_genes)
    counts[::3, n_cells:] = 0
    return models, counts


def _probe_decision(ctx, t, seed):
    """draws of every cell (104 boots), the lists build_lists_kernel makes (cells that are not based, or whose count is not
    zero), Z over the based cells; scde_b200_probe_prune_i8 -> (T, lb, ub, live, flags, W, Z, lists)"""
    K = t["K"]
    n_cells = t["counts"].shape[1]
    based = t["based"] != 0
    rng = np.random.default_rng(seed)
    draws = rng.integers(0, n_cells, size=(WP, n_cells))
    W = np.zeros((n_cells + 1, WP), np.int64)
    for b in range(WP):
        np.add.at(W[:, b], draws[b], 1)
    assert W.max() <= 127
    n_w_rows = (n_cells + 1 + 15) // 16 * 16
    w8 = np.zeros((n_w_rows, 128), np.int8)
    w8[:n_cells, :WP] = W[:n_cells]
    Z = np.zeros((WP, KP))
    Z[:, :K] = W[:n_cells][based].T.astype(np.float64) @ t["zero_rows"][based]
    G = t["counts"].shape[0]
    lists = []
    for g in range(G):
        cells = np.flatnonzero(~based | (t["counts"][g] > 0))
        lists.append(((t["off"][cells] + t["uci"][g, cells]).astype(np.int64), cells))
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
    return T, lb, ub, live, int(flags[0]), W, Z, lists


@pytest.mark.parametrize("K", DECISION_K)
@pytest.mark.parametrize("kind", DECISION_TABLES)
def test_decision_on_every_table(ctx, kind, K):
    """the bound pass on tables of every producer (lp_rows_q_kernel <false> below K = 384 and <true> from there, the
    quantize pass over constant-theta and over local-theta rows, a table with unbased cells whose zero-count rows are
    listed), on one to four pieces: LB, UB and the live mask equal the numpy decision exactly, every admissible value of a
    dead piece lies more than 746 nats below its boot's maximum of the unpruned T + Z, and something is dead -- except on
    a grid of one piece, where nothing can be: that piece holds the boot's maximum, and UB >= maximum >= LB."""
    options = {"fused_fixed_point": 0} if kind == "quantize_pass" else {}
    models, counts = decision_inputs(kind)
    t = _table(ctx, counts.shape[0], counts.shape[1], None, K=K, inputs=(models, counts), **options)
    if kind == "unbased":
        n_un = int((t["based"] == 0).sum())
        assert n_un >= 100, n_un
    T, lb, ub, live, flags, W, Z, lists = _probe_decision(ctx, t, 41 + K)
    assert flags & 2 == 0
    want_lb, want_ub, want_live = _decision(t["qb"], t["rr"].astype(np.int64), W, Z[:, :K], lists, K)
    assert np.array_equal(lb, want_lb)
    assert np.array_equal(ub, want_ub)
    assert np.array_equal(live, want_live)
    n_pieces = (K + Q_PW - 1) // Q_PW
    adm = T[:, :, :K] > -1e299
    full = np.where(adm, T[:, :, :K] + Z[None, :, :K], -np.inf)
    m = full.max(axis=2)
    fin = np.isfinite(m)
    assert fin.mean() > 0.99
    assert np.all(lb[fin] <= m[fin] + 1e-6 * np.abs(m[fin]))
    n_dead = 0
    for p in range(n_pieces):
        pm = full[:, :, p * Q_PW:min((p + 1) * Q_PW, K)].max(axis=2)
        has = np.isfinite(pm)
        assert np.all(ub[:, :, p][has] >= pm[has] - 1e-6 * np.abs(pm[has])), p
        dead = ((live >> p) & 1) == 0
        n_dead += int(dead.sum())
        assert np.all(pm[dead] < m[dead] - 746.0), p
    print(kind, f"K={K}", f"pieces {n_pieces}", f"dead pieces {n_dead} of {len(live) * n_pieces}", f"flags {flags}")
    if n_pieces == 1:
        assert np.all(live == 1)
    else:
        assert n_dead > 0


# ---- 3. pruned calls against independent references ----------------------------------------------------------------------
G3 = 14


def _on_off_fp64(ctx, run):
    """run() with pruning on, with it off, and on the FP64 DMMA kernel"""
    out = {}
    for prune in (1, 0):
        keep = ctx.set_options(prune_pieces=prune)
        try:
            out[prune] = run()
        finally:
            ctx.restore_options(keep)
    ctx.set_contract_kernel(2)
    try:
        fp64 = run()
    finally:
        ctx.set_contract_kernel(0)
    return out[1], out[0], fp64


def _prunes_one_shot(ctx, models, counts, prior, n_boot):
    """the cells and models of a posterior call, twice over as the two groups of the one-shot call: its stats"""
    mm, lt, sq = api.pack_models(models)
    x, y = prior["x"].to_numpy(), prior["y"].to_numpy()
    C2 = counts.shape[1]
    both = np.asfortranarray(np.hstack([counts, counts]).astype(np.int32))
    codes = np.array([0] * C2 + [1] * C2, np.int32)
    res = api.expression_difference_call(ctx, both, np.vstack([mm, mm]), x, y, codes, n_boot, 1, local_theta=lt,
                                         sqlogit=sq, zero_index=api._zero_index(api.fold_change_grid(x), 0.0))
    st = res["stats"]
    print(f"one-shot call on the same cells: prune_live / prune_items = {st['prune_live']} / {st['prune_items']}")
    assert 0 < st["prune_live"] < st["prune_items"]


def _posterior_inputs(kind, n_cells=2800, seed=61):
    if kind == "knn":
        knn = helpers.knn_models()
        models = pd.concat([knn] * (-(-n_cells // len(knn))))
        models.index = [f"cell{i}" for i in range(len(models))]
        counts = synth.make_counts(np.random.default_rng(seed), models, G3)
        return models, counts, synth.make_prior(G3)
    w = synth.make_workload(4, n_genes=G3, n_cells=n_cells, seed=seed)
    return w.models, w.counts, w.prior


POSTERIOR_CASES = {"B100": ("synth", 100, False), "B150": ("synth", 150, False), "B0": ("synth", 0, False),
                   "knn_B100": ("knn", 100, False), "modes_B100": ("synth", 100, True)}


@pytest.mark.parametrize("case", list(POSTERIOR_CASES))
def test_pruned_posteriors_match_references(ctx, case):
    """scde.posteriors of 2800 cells (paired passes at B = 150, the plain product at B = 0, local theta + conc.a2 knn
    models, per-cell modes): pruning on equals pruning off bit for bit, matches the oracle on the same draws (modes
    exactly) and the FP64 DMMA kernel; the same cells prune in the one-shot call"""
    kind, B, modes = POSTERIOR_CASES[case]
    models, counts, prior = _posterior_inputs(kind)
    Cn = counts.shape[1]
    mm, lt, sq = O.pack_models(models)
    mag = O.marginals_from_prior_x(prior["x"].to_numpy())
    flat, off, uci = O.unique_counts(counts)
    want = O.log_boot_posterior(mm, flat, off, uci, mag, B, boot_idx=O.boot_indices(1, Cn, B) if B else None,
                                returnpost=1 if modes else 0, localtheta=lt, sqlogit=sq)

    def run():
        r = api.scde_posteriors(models, counts, prior, n_randomizations=B, return_individual_posterior_modes=modes,
                                context=ctx)
        return {"jp": r["jp"].to_numpy(), "modes": r["modes"].to_numpy()} if modes else {"jp": r.to_numpy()}

    on, off_, fp64 = _on_off_fp64(ctx, run)
    for key in on:
        assert np.array_equal(on[key], off_[key]), key
    ok, worst = _logp_close(on["jp"], want["jp"])
    assert ok, ("oracle", worst)
    ok, worst = _logp_close(on["jp"], fp64["jp"])
    assert ok, ("fp64", worst)
    if modes:
        assert np.array_equal(on["modes"], want["modes"])
    _prunes_one_shot(ctx, models, counts, prior, B if B else 100)


def test_pruned_batch_posterior_matches_references(ctx):
    """scde_b200_log_boot_batch_posterior with 2800 cells drawn per boot"""
    w = synth.make_workload(5, n_genes=G3, n_cells=2800, seed=62, batch=True)
    mm, lt, sq = O.pack_models(w.models)
    mag = O.marginals_from_prior_x(w.prior["x"].to_numpy())
    flat, off, uci = O.unique_counts(w.counts)
    bcodes = np.asarray(w.batch.codes)
    pools = [np.nonzero(bcodes == l)[0].astype(np.int32) for l in range(2)]
    comp = np.array([len(p) for p in pools], np.int32)
    want = O.log_boot_batch_posterior(mm, flat, off, uci, mag, pools, comp, 100, seed=1)["jp"]

    def run():
        return api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=100, batch=w.batch, composition=comp,
                                   context=ctx).to_numpy()

    on, off_, fp64 = _on_off_fp64(ctx, run)
    assert np.array_equal(on, off_)
    ok, worst = _logp_close(on, want)
    assert ok, ("oracle", worst)
    ok, worst = _logp_close(on, fp64)
    assert ok, ("fp64", worst)
    _prunes_one_shot(ctx, w.models, w.counts, w.prior, 100)


@functools.lru_cache(maxsize=None)
def one_shot_inputs(kind):
    """(models, counts, prior, group codes) of a one-shot case"""
    if kind == "unbased":
        w = synth.make_workload(4, n_genes=G3, n_cells=5400, seed=71)
        n_un = 200
        rows = [r for r in api.pack_models(w.models)[0]] + [SENTINEL_ZERO_MODEL] * n_un
        models = _frame(rows)
        counts = np.zeros((G3, 5400 + n_un), np.int32, order="F")
        counts[:, :5400] = w.counts
        counts[:, 5400:] = synth.make_counts(np.random.default_rng(72), models.iloc[5400:], G3)
        counts[::3, 5400:] = 0
        codes = np.array([i // 2700 for i in range(5400)] + [i % 2 for i in range(n_un)], np.int32)
        return models, counts, w.prior, codes
    if kind == "uneven":
        w = synth.make_workload(4, n_genes=G3, n_cells=4200, seed=73)
        return w.models, w.counts, w.prior, (np.arange(4200) >= 3000).astype(np.int32)
    K = int(kind[1:]) if kind.startswith("K") else 401
    w = synth.make_workload(4, n_genes=G3, n_cells=5600, seed=74)
    return w.models, w.counts, synth.make_prior(G3, length_out=K - 1), np.asarray(w.groups.codes, np.int32)


@functools.lru_cache(maxsize=None)
def one_shot_oracle(kind):
    models, counts, prior, codes = one_shot_inputs(kind)
    return O.expression_difference(models, counts, prior["x"].to_numpy(), prior["y"].to_numpy(),
                                   (np.nonzero(codes == 0)[0], np.nonzero(codes == 1)[0]), nboot=100, seed=1)


ONE_SHOT_CASES = {"lp_rows_kernel": ("K401", {"lp_rows_kernel": 1}), "fused_fixed_point0": ("K401", {"fused_fixed_point": 0}),
                  "K103": ("K103", {}), "K204": ("K204", {}), "K306": ("K306", {}), "K408": ("K408", {}),
                  "unbased": ("unbased", {}), "uneven": ("uneven", {})}


@pytest.mark.parametrize("case", list(ONE_SHOT_CASES))
def test_pruned_one_shot_call_matches_references(ctx, case):
    """the one-shot call with the FastPlanes rows, with FP64 rows and the quantize pass, on priors of 103 to 408 points,
    with unbased cells in both groups, and with uneven groups (3000 against 1200 cells: only the large joint prunes):
    pruning on equals off bit for bit; joint posteriors, idx and Z match the oracle; joint posteriors match the FP64
    DMMA kernel; the call pruned"""
    kind, options = ONE_SHOT_CASES[case]
    models, counts, prior, codes = one_shot_inputs(kind)
    mm, lt, sq = api.pack_models(models)
    x, y = prior["x"].to_numpy(), prior["y"].to_numpy()
    want = one_shot_oracle(kind)

    def run():
        keep = ctx.set_options(**options)
        try:
            return api.expression_difference_call(ctx, counts, mm, x, y, codes, 100, 1, local_theta=lt, sqlogit=sq,
                                                  zero_index=api._zero_index(api.fold_change_grid(x), 0.0),
                                                  joint_posteriors=True)
        finally:
            ctx.restore_options(keep)

    on, off_, fp64 = _on_off_fp64(ctx, run)
    _same(on, off_)
    for i in range(2):
        ok, worst = _logp_close(on["joint_posteriors"][i], want["joint.posteriors"][i])
        assert ok, ("oracle", i, worst)
        ok, worst = _logp_close(on["joint_posteriors"][i], fp64["joint_posteriors"][i])
        assert ok, ("fp64", i, worst)
    assert np.array_equal(on["idx"], want["idx"])
    _z_close(on["z"], want["results"][:, 4])
    st = on["stats"]
    print(case, f"K={len(x)}", f"prune_live / prune_items = {st['prune_live']} / {st['prune_items']}")
    assert 0 < st["prune_live"] < st["prune_items"]
    if kind == "uneven":  # one joint's items: 14 genes x 4 pieces
        assert st["prune_items"] == G3 * ((len(x) + Q_PW - 1) // Q_PW)
