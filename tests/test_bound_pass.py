"""The bound pass of the pruned tcgen05 contraction (bound_i8_kernel, DESIGN.md 4.3): the sums of the drawn rows' bound
rows stay in tensor memory and the kernel's epilogue takes the pruning decision itself.  Its LB, UB and live pieces must
equal a numpy restatement of the decision exactly, and pruning on must equal pruning off bit for bit for every mix of
list lengths (empty lists, lists shorter than a stage, lists of thousands of entries) that walks its accumulator ring."""
import ctypes as C

import numpy as np
import pytest

from scde_b200 import _lib, api, synth
from test_prune_pieces import KP, LB_N, LB_OFF, LB_STEP, Q_PW, UB_N, UB_PTS, WP, _both, _call, _same, _table

pytestmark = pytest.mark.gpu


def _decision(qb, rr, W, Z, lists, K):
    """LB [G][104], UB [G][104][4] and live [G] as the bound pass decides them (DESIGN.md 4.3): sums of the drawn bound
    rows (two radix-256 digits per slot), Z extrema, the (gene, boot) sentinel ranges"""
    G = len(lists)
    zb = np.full((WP, 64), -np.inf)
    for u in range(UB_N):
        if u * UB_PTS < K:  # (blocks past the grid keep -inf, as z_bounds_kernel writes them)
            zb[:, u] = Z[:, u * UB_PTS:min((u + 1) * UB_PTS, K)].max(axis=1)
    for c in range(LB_N):
        if LB_STEP * c + LB_OFF < K:
            zb[:, UB_N + c] = Z[:, LB_STEP * c + LB_OFF]
    lb, ub = np.full((G, WP), -np.inf), np.full((G, WP, 4), -np.inf)
    live = np.zeros(G, np.uint8)
    n_pieces = (K + Q_PW - 1) // Q_PW
    for g, (rows, cells) in enumerate(lists):
        w = W[cells].astype(np.int64)  # [entries][104]
        S = w.T @ qb[rows].astype(np.int64)  # [104][128]: exact digit sums
        val = zb + (S[:, :64].astype(np.float64) + 256.0 * S[:, 64:].astype(np.float64)) * (1.0 / 32.0)
        klo, khi = np.zeros(WP, np.int64), np.full(WP, K - 1, np.int64)
        for b in range(WP):
            drawn = rr[rows[w[:, b] > 0]]
            if len(drawn):
                klo[b] = max(0, int((drawn & 0xFFFF).max()))
                khi[b] = min(K - 1, int((drawn >> 16).min()))
        dead = (1 << n_pieces) - 1
        for b in range(WP):
            for c in range(LB_N):
                k = LB_STEP * c + LB_OFF
                if klo[b] <= k <= khi[b]:
                    lb[g, b] = max(lb[g, b], val[b, UB_N + c])
            for u in range(UB_N):
                lo, hi = max(u * UB_PTS, klo[b]), min(u * UB_PTS + UB_PTS - 1, khi[b])
                if lo > hi:
                    continue
                for p in range(4):
                    if max(lo, p * Q_PW) <= min(hi, p * Q_PW + Q_PW - 1):
                        ub[g, b, p] = max(ub[g, b, p], val[b, u])
            d = sum(1 << p for p in range(4) if ub[g, b, p] < lb[g, b] - 747.0)
            dead &= d
        live[g] = ~dead & ((1 << n_pieces) - 1)
    return lb, ub, live


def test_bounds_and_decision_equal_numpy(ctx):
    """1500 cells, 104 boots, 60 genes: the probe's LB, UB and live mask against the numpy restatement, exactly"""
    n_cells, G = 1500, 60
    t = _table(ctx, G, n_cells, 41)
    K = t["K"]
    rng = np.random.default_rng(41)
    drawable = np.flatnonzero((t["based"] != 0) & (t["zero_row"] >= 0))
    draws = rng.choice(drawable, size=(WP, n_cells), replace=True)
    W = np.zeros((n_cells + 1, WP), np.int64)
    for b in range(WP):
        np.add.at(W[:, b], draws[b], 1)
    n_w_rows = (n_cells + 1 + 15) // 16 * 16
    w8 = np.zeros((n_w_rows, 128), np.int8)
    w8[:n_cells, :WP] = W[:n_cells]
    Z = np.zeros((WP, KP))
    Z[:, :K] = W[drawable].T.astype(np.float64) @ t["zero_rows"][drawable]
    lists = []
    for g in range(G):
        cells = drawable[t["counts"][g, drawable] > 0]
        lists.append(((t["off"][cells] + t["uci"][g, cells]).astype(np.int64), cells))
    ld = max(32, (max(len(c) for _, c in lists) + 31) // 32 * 32)
    lst_row = np.zeros((G, ld), np.int32)
    lst_cell = np.full((G, ld), n_cells, np.int32)
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
    assert flags[0] == 0
    want_lb, want_ub, want_live = _decision(t["qb"], t["rr"].astype(np.int64), W, Z[:, :K], lists, K)
    assert np.array_equal(lb, want_lb)
    assert np.array_equal(ub, want_ub)
    assert np.array_equal(live, want_live)
    assert (live != (1 << ((K + Q_PW - 1) // Q_PW)) - 1).any()  # something is pruned: the comparison bites


LENGTHS = [0, 1, 31, 33, 4000, 32, 0, 2600, 1, 64, 33, 5000, 31]


def _mixed_lengths(config, G, n_cells, seed, batch=False):
    """a workload whose genes have 0, 1, 31, 33 ... thousands of non-zero counts (list entries per joint), in mixed order"""
    w = synth.make_workload(config, n_genes=G, n_cells=n_cells, seed=seed, batch=batch)
    counts = np.array(w.counts, copy=True)
    rng = np.random.default_rng(seed)
    for g in range(G):
        n = min(LENGTHS[g % len(LENGTHS)], n_cells)
        keep = np.zeros(n_cells, bool)
        keep[rng.choice(n_cells, size=n, replace=False)] = True
        counts[g, ~keep] = 0
        counts[g, keep] = np.maximum(counts[g, keep], 1)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    kw = dict(local_theta=lt, sqlogit=sq, zero_index=[len(x)])
    if batch:
        kw.update(batch_codes=np.asarray(w.batch.codes, dtype=np.int32), n_batch_levels=2,
                  zero_index_adjusted=[2 * len(x) - 1])
    return (counts, mm, x, y, np.asarray(w.groups.codes, dtype=np.int32)), kw


def test_mixed_list_lengths_one_side(ctx):
    """1300 genes (about nine per SM: every accumulator buffer is reused with both parities), one side per launch"""
    args, kw = _mixed_lengths(4, 1300, 5200, 42)
    on, off = _both(ctx, lambda: _call(ctx, args, kw))
    _same(on, off)
    assert on["stats"]["prune_live"] < on["stats"]["prune_items"]


def test_mixed_list_lengths_two_sides(ctx):
    """the same mix through two-sided launches: 150 randomizations (paired passes, the second ragged) and a batch factor
    (two joints per launch)"""
    args, kw = _mixed_lengths(4, 700, 5200, 43)
    on, off = _both(ctx, lambda: _call(ctx, args, kw, n_boot=150))
    _same(on, off)
    args, kw = _mixed_lengths(5, 700, 5200, 44, batch=True)
    on, off = _both(ctx, lambda: _call(ctx, args, kw))
    _same(on, off)
    assert on["stats"]["prune_live"] < on["stats"]["prune_items"]
