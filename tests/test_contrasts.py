"""Many contrasts on one resident dataset (scde_b200_dataset_*, api.DifferenceSession): every contrast equals the one-shot
call on the full matrix with codes 0 / 1 / -1, the joints are shared, and bad input is refused.  Host-only tests (contrast
expansion, argument errors) are unmarked; the rest need a GPU."""
import ctypes as C
import os

import numpy as np
import pandas as pd
import pytest

import helpers
from oracle import oracle as O
from scde_b200 import _lib, api, synth


# ------------------------------------------------------------------------------------------------ host only
def test_expand_pairs_and_rest():
    pairs = api.expand_contrasts(["a", "b", "c"], "pairs")
    assert [p[0] for p in pairs] == ["a vs b", "a vs c", "b vs c"]
    assert [(p[1], p[2]) for p in pairs] == [(["a"], ["b"]), (["a"], ["c"]), (["b"], ["c"])]
    rest = api.expand_contrasts(["a", "b", "c"], "rest")
    assert [p[0] for p in rest] == ["a vs rest", "b vs rest", "c vs rest"]
    assert rest[1][1:] == (["b"], ["a", "c"], "b", "rest")


def test_expand_level_lists():
    got = api.expand_contrasts(["a", "b", "c", "d"], [("c", "a"), (["a", "b"], ["c", "d"]), ("d", ["b"])])
    assert [g[0] for g in got] == ["c vs a", "a+b vs c+d", "d vs b"]
    assert got[1][1:] == (["a", "b"], ["c", "d"], "a+b", "c+d")


@pytest.mark.parametrize("levels,contrasts,msg", [
    (["a", "b"], [("a", "x")], "unknown level x"),
    (["a", "b"], [("a", "a")], "share level"),
    (["a", "b", "c"], [(["a", "b"], ["b", "c"])], "share level"),
    (["a", "b"], [("a", [])], "names no level"),
    (["a", "b"], "all", "contrasts must be"),
    (["a"], "pairs", "at least two levels"),
    (["a", "b"], [("a", "b"), ("a", "b")], "listed twice"),
    (["a", "b"], [], "no contrasts"),
])
def test_expand_errors(levels, contrasts, msg):
    with pytest.raises(ValueError, match="^ERROR: .*" + msg):
        api.expand_contrasts(levels, contrasts)


# ------------------------------------------------------------------------------------------------ GPU
def _four_groups(n_genes=200, n_cells=120, seed=13, batch=False):
    w = synth.make_workload(5 if batch else 3, n_genes=n_genes, n_cells=n_cells, seed=seed, batch=batch)
    rng = np.random.default_rng(seed)
    codes = rng.permutation(np.arange(n_cells) % 4)  # interleaved, unequal order of the cells
    groups = pd.Categorical.from_codes(codes, categories=["A", "B", "C", "D"])
    return w, groups


def _two_level(groups, la, lb, na, nb):
    g = np.asarray(groups.astype(object))
    codes = np.where(np.isin(g, la), 0, np.where(np.isin(g, lb), 1, -1))
    return pd.Categorical.from_codes(codes, categories=[na, nb])


def _assert_same(got, want):
    if isinstance(want, pd.DataFrame):
        pd.testing.assert_frame_equal(got, want, check_exact=True)
        return
    assert set(got) == set(want)
    for k in want:
        if k == "stats":
            continue
        if k == "joint.posteriors":
            assert list(got[k]) == list(want[k])
            for name in want[k]:
                pd.testing.assert_frame_equal(got[k][name], want[k][name], check_exact=True)
        else:
            pd.testing.assert_frame_equal(got[k], want[k], check_exact=True, obj=k)


def _check_against_fused(ctx, w, groups, res, contrasts, **kw):
    plan = api.expand_contrasts(list(groups.categories), contrasts)
    assert list(res) == [p[0] for p in plan]
    for label, la, lb, na, nb in plan:
        want = api.scde_expression_difference(w.models, w.counts, w.prior, groups=_two_level(groups, la, lb, na, nb),
                                              context=ctx, **kw)
        _assert_same(res[label], want)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [0, 2])  # default (tcgen05 fixed point), FP64 DMMA
def test_contrasts_equal_fused_call(ctx, kernel):
    w, groups = _four_groups()
    ctx.set_contract_kernel(kernel)
    try:
        with api.DifferenceSession(w.models, w.counts, w.prior, context=ctx) as s:
            pairs = s.contrasts(groups, "pairs", n_randomizations=100, return_posteriors=True)
            rest = s.contrasts(groups, "rest", n_randomizations=100, return_posteriors=True)
        _check_against_fused(ctx, w, groups, pairs, "pairs", n_randomizations=100, return_posteriors=True)
        _check_against_fused(ctx, w, groups, rest, "rest", n_randomizations=100, return_posteriors=True)
    finally:
        ctx.set_contract_kernel(0)


@pytest.mark.gpu
def test_contrasts_batch_models_na_batch_and_shared_batch_joint(ctx):
    w = synth.make_workload(5, n_genes=90, n_cells=60, seed=17, batch=True)
    rng = np.random.default_rng(3)
    bm = w.models.copy()
    bm["corr.b"] = bm["corr.b"] + rng.uniform(-0.3, 0.3, len(bm))
    bm["conc.b"] = bm["conc.b"] - 0.5
    bcodes = np.asarray(w.batch.codes).copy()
    bcodes[[3, 17, 44]] = -1
    batch = pd.Categorical.from_codes(bcodes, categories=list(w.batch.categories))
    # X and Y: six batch1 and six batch2 cells each (equal composition: one batch joint for both); Z: every other cell
    b1, b2 = np.nonzero(bcodes == 0)[0], np.nonzero(bcodes == 1)[0]
    lab = np.full(60, "Z", dtype=object)
    lab[b1[:6]] = lab[b2[:6]] = "X"
    lab[b1[6:12]] = lab[b2[6:12]] = "Y"
    groups = pd.Categorical(lab, categories=["X", "Y", "Z"])
    kw = dict(batch=batch, batch_models=bm, n_randomizations=100, return_posteriors=True)
    with api.DifferenceSession(w.models, w.counts, w.prior, context=ctx) as s:
        res = s.contrasts(groups, "pairs", **kw)
        st = s.last_stats
        # batch.models = models afterwards: the table is rebuilt from the models first
        plain = s.contrasts(groups, "pairs", batch=batch, n_randomizations=100)
    _check_against_fused(ctx, w, groups, res, "pairs", **kw)
    _check_against_fused(ctx, w, groups, plain, "pairs", batch=batch, n_randomizations=100)
    # three group joints + one launch for the two distinct compositions (X = Y, Z), 100 randomizations = one pass
    assert st["launches"]["contract"] == 4, st


@pytest.mark.gpu
def test_joints_are_shared_and_table_is_reused(ctx):
    w, groups = _four_groups(seed=19)
    codes = np.asarray(groups.codes, dtype=np.int32)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    fused_cells = 0
    for a in range(4):
        for b in range(a + 1, 4):
            g = np.where(codes == a, 0, np.where(codes == b, 1, -1)).astype(np.int32)
            fused_cells += api.expression_difference_call(ctx, w.counts, mm, x, y, g, 100, 1, local_theta=lt,
                                                          sqlogit=sq)["stats"]["contract_cells"]
    other = pd.Categorical.from_codes(np.arange(120) % 3, categories=["p", "q", "r"])
    with api.DifferenceSession(w.models, w.counts, w.prior, context=ctx) as s:
        assert s.create_stats["launches"]["dedup"] > 0 and s.create_stats["launches"]["lp_table"] > 0
        s.contrasts(groups, "pairs", n_randomizations=100)
        st = s.last_stats
        again = s.contrasts(other, "rest", n_randomizations=60)
    assert st["launches"]["contract"] == 4, st
    assert st["launches"]["dedup"] == 0 and st["launches"]["lp_table"] == 0, st
    assert st["contract_cells"] * 3 == fused_cells
    with api.DifferenceSession(w.models, w.counts, w.prior, context=ctx) as s:
        fresh = s.contrasts(other, "rest", n_randomizations=60)
    for k in fresh:
        _assert_same(again[k], fresh[k])


@pytest.mark.gpu
def test_one_contrast_against_oracle(ctx):
    w = synth.make_workload(3, n_genes=150, n_cells=90, seed=7)
    lab = np.array(["u", "v", "t"] * 30, dtype=object)
    groups = pd.Categorical(lab, categories=["u", "v", "t"])
    res = api.scde_expression_difference_contrasts(w.models, w.counts, w.prior, groups, [("t", "u")],
                                                   n_randomizations=100, context=ctx)["t vs u"]
    want = O.expression_difference(w.models, w.counts, w.prior["x"].to_numpy(), w.prior["y"].to_numpy(),
                                   (np.nonzero(lab == "t")[0], np.nonzero(lab == "u")[0]), nboot=100, seed=1)
    diffv = api.fold_change_grid(w.prior["x"].to_numpy())
    assert np.array_equal(res[["lb", "mle", "ub"]].to_numpy(), diffv[want["idx"]] / np.log10(2.0))
    from test_gpu_parity import _z_close

    _z_close(res["Z"].to_numpy(), want["results"][:, 4])


def _raw_contrasts(ctx, ds, groups, pairs, K, n_zero=1):
    off = np.zeros(len(groups) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(g) for g in groups])
    cells = np.concatenate([np.asarray(g, dtype=np.int32) for g in groups]) if groups else np.zeros(1, np.int32)
    pr = np.asarray(pairs, dtype=np.int32).ravel()
    zi = np.array([K], dtype=np.int32)
    a = _lib.ContrastArgs()
    a.n_groups, a.group_offsets, a.group_cells = len(groups), _lib.p_i32(off), _lib.p_i32(cells)
    a.n_contrasts, a.pairs = len(pr) // 2, _lib.p_i32(pr)
    a.n_boot, a.seed, a.zero_index, a.n_zero = 20, 1, _lib.p_i32(zi), n_zero
    G = 30
    idx, z = np.empty(3 * G * max(1, len(pr) // 2), np.int32), np.empty(G * max(1, len(pr) // 2))
    o = _lib.ContrastOut()
    o.idx, o.z = _lib.p_i32(idx), _lib.p_f64(z)
    rc = _lib.lib().scde_b200_dataset_contrasts(ctx.handle, ds, C.byref(a), C.byref(o), None)
    return rc, _lib.lib().scde_b200_last_error().decode()


@pytest.mark.gpu
def test_errors_leave_the_context_usable(ctx):
    w = synth.make_workload(3, n_genes=30, n_cells=24, seed=3)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    K = len(x)
    counts = _lib.i32(w.counts)
    d = _lib.DatasetArgs()
    d.n_genes, d.n_cells, d.n_grid = 30, 24, K
    d.counts, d.models, d.prior_x, d.prior_y = _lib.p_i32(counts), _lib.p_f64(mm), _lib.p_f64(_lib.f64(x)), _lib.p_f64(_lib.f64(y))
    ds = C.c_void_p()
    L = _lib.lib()
    assert L.scde_b200_dataset_create(ctx.handle, C.byref(d), C.byref(ds), None) == 0
    try:
        cases = [
            ([[0, 1, 2], [2, 3]], [[0, 1]], "share cell 2"),
            ([[0, 1, 2], []], [[0, 1]], "group 1 is empty"),
            ([[0, 1, 2], [3, 4]], [[1, 1]], "with itself"),
            ([[0, 1, 2], [3, 4]], [[0, 2]], "outside"),
            ([[0, 2, 1], [3, 4]], [[0, 1]], "not ascending"),
            ([[0, 1, 24], [3, 4]], [[0, 1]], "cell 24 outside"),
        ]
        for groups, pairs, msg in cases:
            rc, err = _raw_contrasts(ctx, ds, groups, pairs, K)
            assert rc == -1, (msg, rc, err)  # SCDE_B200_EINVAL
            assert msg in err, (msg, err)
        # groups may overlap across contrasts
        rc, err = _raw_contrasts(ctx, ds, [[0, 1, 2], [3, 4], [2, 5, 6]], [[0, 1], [1, 2]], K)
        assert rc == 0, err
        # the one-shot call is refused while the dataset holds the workspace
        g = np.where(np.arange(24) < 12, 0, 1).astype(np.int32)
        with pytest.raises(_lib.ScdeB200Error, match="another expression_difference job is alive") as e:
            api.expression_difference_call(ctx, w.counts, mm, x, y, g, 20, 1, local_theta=lt, sqlogit=sq)
        assert e.value.code == -1
    finally:
        L.scde_b200_dataset_free(ctx.handle, ds)
    api.expression_difference_call(ctx, w.counts, mm, x, y, g, 20, 1, local_theta=lt, sqlogit=sq)
    groups = pd.Categorical(np.where(np.arange(24) < 12, "a", "b"))
    with pytest.raises(ValueError, match="unknown level zz"):
        api.scde_expression_difference_contrasts(w.models, w.counts, w.prior, groups, [("a", "zz")], context=ctx)
    with pytest.raises(ValueError, match="no cells in c"):
        api.scde_expression_difference_contrasts(w.models, w.counts, w.prior,
                                                 pd.Categorical(groups.astype(object), categories=["a", "b", "c"]),
                                                 [("a", "c")], context=ctx)
    api.expression_difference_call(ctx, w.counts, mm, x, y, g, 20, 1, local_theta=lt, sqlogit=sq)


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [False, True])
def test_two_devices_equal_one_device(ctx, batch):
    if _lib.lib().scde_b200_device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    mctx = _lib.Context(devices=[0, 1])
    w, groups = _four_groups(n_genes=301, n_cells=128, seed=41, batch=batch)
    kw = dict(batch=w.batch if batch else None, n_randomizations=100, return_posteriors=True)
    one = api.scde_expression_difference_contrasts(w.models, w.counts, w.prior, groups, "pairs", context=ctx, **kw)
    two = api.scde_expression_difference_contrasts(w.models, w.counts, w.prior, groups, "pairs", context=mctx, **kw)
    for k in one:
        _assert_same(two[k], one[k])
    mctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [False, True])
def test_r_shim_contrasts_entry(ctx, batch):
    path = os.path.abspath(os.path.join(helpers.GOLD, "..", "..", "integration", "_build", "libscde_shim.so"))
    if not os.path.exists(path):
        pytest.fail("integration/_build/libscde_shim.so is missing: __graft_entry__.build() builds it (make -C integration)")
    shim = C.CDLL(path)
    w, groups = _four_groups(n_genes=120, n_cells=40, seed=29, batch=batch)
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    K, G, Cn = len(x), 120, 40
    counts = np.asfortranarray(w.counts, dtype=np.int32)
    codes = np.asarray(groups.codes)
    sides = [np.nonzero(codes == g)[0].astype(np.int32) for g in range(4)]
    off = np.zeros(5, dtype=np.int32)
    off[1:] = np.cumsum([len(s) for s in sides])
    cells = np.concatenate(sides)
    pairs = np.array([[a, b] for a in range(4) for b in range(a + 1, 4)], dtype=np.int32).ravel()
    nc = len(pairs) // 2
    bc = np.asarray(w.batch.codes, dtype=np.int32) if batch else None
    n_sets = 3 if batch else 1
    idx, z, cz = np.zeros(n_sets * nc * 3 * G), np.zeros(n_sets * nc * G), np.zeros(n_sets * nc * G)
    err = C.create_string_buffer(256)
    dev = np.zeros(1, dtype=np.int32)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    rc = shim.shim_diff_contrasts(counts.ctypes.data_as(ip), G, Cn, np.asfortranarray(mm).ctypes.data_as(dp),
                                  x.ctypes.data_as(dp), y.ctypes.data_as(dp), K, off.ctypes.data_as(ip), 4,
                                  cells.ctypes.data_as(ip), pairs.ctypes.data_as(ip), nc,
                                  bc.ctypes.data_as(ip) if batch else None, 2 if batch else 0, 100, K, 2 * K - 1,
                                  dev.ctypes.data_as(ip), 1, idx.ctypes.data_as(dp), z.ctypes.data_as(dp),
                                  cz.ctypes.data_as(dp), err)
    assert rc == 0, err.value
    names = [("idx", "z", "cz")] + ([("batch_idx", "batch_z", "batch_cz"), ("adjusted_idx", "adjusted_z", "adjusted_cz")] if batch else [])
    for c in range(nc):
        a, b = pairs[2 * c], pairs[2 * c + 1]
        g = np.where(codes == a, 0, np.where(codes == b, 1, -1)).astype(np.int32)
        want = api.expression_difference_call(ctx, counts, mm, x, y, g, 100, 1, batch_codes=bc,
                                              n_batch_levels=2 if batch else 0, zero_index=[K],
                                              zero_index_adjusted=[2 * K - 1], local_theta=lt, sqlogit=sq)
        for s, (ki, kz, kc) in enumerate(names):
            i0 = (s * nc + c) * 3 * G
            assert np.array_equal(idx[i0:i0 + 3 * G].reshape(3, G).T, want[ki]), (c, ki)
            z0 = (s * nc + c) * G
            assert np.array_equal(z[z0:z0 + G], want[kz]), (c, kz)
            assert np.array_equal(cz[z0:z0 + G], want[kc]), (c, kc)
