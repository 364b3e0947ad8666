"""The fixed-point log-posterior table, element by element, against the oracle (DESIGN.md section 5: table rows 1e-9).

The tcgen05 contraction reads every table row of a non-zero count as five signed radix-256 digit planes plus the row's
admissible range.  A joint posterior is a soft-max over the grid, so an element error away from its peak never reaches
it: these tests decode the rows that `scde_b200_probe_table` returns -- the table exactly as the fused
differential-expression path builds it -- and compare every element with the oracle's `cell_table` (the reference's C++
bit for bit), at the model and count extremes where the hand-written arithmetic of the row kernels lives:

* CPU: a numpy decoder of the planes, and a numpy classifier of every element (easy, cross-over, one-term gradual
  underflow, cross-over inside the underflow band, "log 0", and the 1e-9 margins of the class boundaries) checked
  against the oracle's values; the chosen inputs must reach every class and every snap position the row kernel treats
  apart, so that narrowing them fails instead of silently testing less;
* GPU: every row of every producer of the planes (the register-resident row kernel, the per-element kernel, the
  quantize pass over FP64 rows, local-theta models), the zero-count rows, `based` and the ranges;
* GPU: posteriors of high-theta and steep drop-out models, and the one-shot call and the contrasts of a session with a
  cell whose zero-count row holds "log 0" points.
"""
import functools
import itertools

import ctypes as C
import numpy as np
import pandas as pd
import pytest

import helpers
from oracle import oracle as O
from scde_b200 import _lib, api, synth

Q_FRAC, Q_NV, Q_PW, Q_PIECE, Q_MAX_K = 29, 5, 102, 512, 408  # scde_b200/csrc/common.cuh
Q_RANGE_IRREGULAR = 0xFFFFFFFF
SCALE = float(2 ** Q_FRAC)
LOG0 = -1e300  # at or below: the reference's "log 0" clamp -DBL_MAX/n/1.1

# counts of every row kind: the smallest, every decade up to the largest the count type holds
COUNTS = [0, 1, 2, 3, 5, 10, 20, 30, 50, 70, 100, 150, 200, 300, 500, 700, 1000, 5000, 65535, 65536, 10 ** 6,
          2 ** 31 - 1]
# cells with more than 64 rows (two 32-row header batches and more than one 64-row work chunk of lp_rows_q_kernel)
LONG_COUNTS = sorted(set(COUNTS) | set(np.unique(np.round(np.geomspace(4, 2.0e9, 110))).astype(np.int64).tolist()))
# (grid points, first grid value, n_cells_for_clamp): one piece, piece boundaries (102, 204, 306), the FULL template of
# the row kernel from 384 on, the largest fixed-point grid; grid point 0 at magnitude -Inf (x = 0) or finite
GRIDS = [(16, 0.0, 1), (102, 0.3, 10000), (200, 0.0, 10000), (383, 0.1, 1), (384, 0.0, 10000), (401, 0.0, 10000),
         (401, 0.25, 1), (408, 0.0, 1)]
GRID_IDS = [f"K{k}-x{x0}-n{n}" for k, x0, n in GRIDS]


def _model(conc_b, conc_a, corr_b, corr_a, theta, fail_r=synth.FAIL_R):
    m = np.full(12, np.nan)
    m[:6] = [conc_b, conc_a, fail_r, corr_b, corr_a, theta]
    return m


# steep drop-out, low dispersion: its zero-count row keeps six "log 0" points, so its cell is not based
SENTINEL_ZERO_MODEL = _model(-6.0, 70.0, 2.4, 1.5, 50.0)


def _mag(K, x0):
    return O.marginals_from_prior_x(np.linspace(x0, 4.8, K))


# ---- decoder and packing --------------------------------------------------------------------------------------------
def q_row_bytes(K):
    return -(-K // Q_PW) * Q_PIECE


def _plane_index(K):
    k = np.arange(K)
    return (k // Q_PW) * Q_PIECE + k % Q_PW  # plane 0 of grid point k; plane p is Q_PW bytes further


def decode(q, K):
    """X[r, k] = sum_p 256^p d_p with the signed digits d_p of rows q[n_rows][q_row_bytes(K)]; the value is X 2^-29"""
    q = np.asarray(q).view(np.int8).reshape(len(q), -1)
    col = _plane_index(K)
    X = np.zeros((q.shape[0], K), np.int64)
    for p in reversed(range(Q_NV)):
        X = X * 256 + q[:, col + p * Q_PW].astype(np.int64)
    return X


def encode(v, K):
    """The packing of DESIGN.md section 4.2 / 4.3 restated: rint(v 2^29) is held, biased by 0x8080808080, in the low 40
    bits of the mantissa of v 2^29 + 1.5 2^52 + 0x8080808080; the top bit of every byte flipped gives the signed digits;
    values at or below the "log 0" clamp get zero digits.  v[n_rows][K] -> planes [n_rows][q_row_bytes(K)]."""
    v = np.asarray(v, dtype=np.float64)
    alive = v > LOG0
    y = np.where(alive, v, 0.0) * SCALE + (6755399441055744.0 + 551911719040.0)
    bits = y.view(np.uint64) & np.uint64((1 << 40) - 1)
    out = np.zeros((v.shape[0], q_row_bytes(K)), np.uint8)
    col = _plane_index(K)
    for p in range(Q_NV):
        byte = ((bits >> np.uint64(8 * p)) & np.uint64(0xFF)).astype(np.uint8) ^ np.uint8(0x80)
        out[:, col + p * Q_PW] = np.where(alive, byte, 0)
    return out.view(np.int8)


# ---- classifier ---------------------------------------------------------------------------------------------------
_dnbinom = np.frompyfunc(O.lib().orc_dnbinom_log, 3, 1)
CLASSES = ("easy", "cross-over", "one-term underflow", "cross-over in underflow", "log 0")


def grid_vectors(m, mag, lt=0, sq=0):
    """mu, log d, log(1 - d) and theta of the grid, as the reference computes them (src/jpmatLogBoot.cpp:133-162)"""
    with np.errstate(all="ignore"):
        mu = np.exp(mag * m[4] + m[3])
        c = ((m[1] + mag * m[11]) * mag if sq else mag * m[1]) + m[0]
        cf = 1 / (np.exp(c) + 1)
        lcfp, lcfpr = np.log(cf), np.log(1 - cf)
        if lt:
            t = np.power(np.power(10.0, (-mag + m[8]) * m[9]) + 1, m[10])
            th = np.exp(-((m[7] - m[6]) / t + m[6]))
            th = np.minimum(np.where(~np.isfinite(th) | (th < 1e-2), 1e-2, th), 1e3)
        else:
            th = np.full(len(mag), m[5])
    return mu, lcfp, lcfpr, th


def snap_point(mu, x):
    """the grid point where the reference replaces mu_k by the count (:173,182), or -1"""
    hit = np.zeros(len(mu), bool)
    hit[:-1] = (x > mu[:-1]) & (x < mu[1:])
    hit[-1] = x > mu[-1]
    k = np.nonzero(hit)[0]
    return int(k[0]) if len(k) else -1


def nb_terms(x, vecs):
    """a_k = log NB(x; theta_k, mu~_k) + log(1 - d_k) with the snap rule, and the snap point"""
    mu, lcfp, lcfpr, th = vecs
    ks = snap_point(mu, x)
    muv = mu.copy()
    if ks >= 0:
        muv[ks] = x
    with np.errstate(all="ignore"):
        return _dnbinom(float(x), th, th / (th + muv)).astype(np.float64) + lcfpr, ks


def row_terms(m, mag, x, lt=0, sq=0, vecs=None):
    """a_k = log NB + log(1 - d_k), e_k = log d_k + f of one row, both relative to the row maximum M, the snap point and
    log S (S = sum_k exp(a_k) + exp(e_k) relative to M)"""
    vecs = vecs if vecs is not None else grid_vectors(m, mag, lt, sq)
    lcfp = vecs[1]
    a, ks = nb_terms(x, vecs)
    with np.errstate(all="ignore"):
        f = O.dpois_log(x, np.exp(m[2]))
        e = lcfp + f
        M = max(np.max(a), np.max(lcfp) + f)
        A, E = a - M, e - M
        log_s = np.log(np.sum(np.exp(A) + np.exp(E)))
    return A, E, ks, log_s


def classify(A, E):
    """class index per element (CLASSES) and the margin flags (within 1e-9 of hi = -746, hi = -708, |a - e| = 37.5)"""
    with np.errstate(invalid="ignore"):
        d = np.abs(A - E)
        hi = np.maximum(A, E)
        band = d <= 37.5
        cls = np.where(hi < -746.0, 4, np.where(hi < -708.0, np.where(band, 3, 2), np.where(band, 1, 0)))
        margin = np.stack([np.abs(hi + 746.0) <= 1e-9, np.abs(hi + 708.0) <= 1e-9, np.abs(d - 37.5) <= 1e-9])
    return cls, margin


def _tune_margins(mag):
    """models (fail.r tuned by bisection) that put one element of their count-300 row within 1e-10 of each class
    boundary: hi = -746, hi = -708, |a - e| = 37.5.  Only the Poisson term f depends on fail.r."""
    out = []
    x = 300
    for base, target in ((_model(-3.0, 5.0, 1.3, 0.7, 50.0), -746.0), (_model(-3.0, 5.0, 1.3, 0.7, 50.0), -708.0),
                         (_model(-1.0, 0.8, 1.3, 0.5, 1.0), 37.5), (_model(-3.0, 5.0, 1.3, 0.7, 50.0), 37.5)):
        vecs = grid_vectors(base, mag)
        a, _ = nb_terms(x, vecs)
        lcfp = vecs[1]

        def q(fr):
            f = O.dpois_log(x, np.exp(fr))
            with np.errstate(all="ignore"):
                M = max(np.max(a), np.max(lcfp) + f)
                A, E = a - M, lcfp + f - M
                return np.abs(A - E) - target if target > 0 else np.maximum(A, E) - target

        lo, hi = -12.0, np.log(x)
        ql, qh = q(lo), q(hi)
        with np.errstate(invalid="ignore"):
            cand = np.nonzero(np.isfinite(ql) & np.isfinite(qh) & (np.sign(ql) != np.sign(qh)))[0]
        for k in cand[len(cand) // 2:][:8]:
            u, w = lo, hi
            for _ in range(200):
                mid = 0.5 * (u + w)
                if np.sign(q(mid)[k]) == np.sign(q(u)[k]):
                    u = mid
                else:
                    w = mid
            best = min((u, w), key=lambda fr: abs(q(fr)[k]))
            if abs(q(best)[k]) <= 1e-10:
                m = base.copy()
                m[2] = best
                out.append(m)
                break
    return out


# ---- inputs -----------------------------------------------------------------------------------------------------------
class Case:
    """one table: models (column-major n x 12), each cell's distinct counts, the grid, the oracle's rows"""

    def __init__(self, models, lists, K, x0, clamp, lt=0, sq=0):
        self.mm = np.asfortranarray(np.asarray(models, dtype=np.float64))
        self.lists = [np.asarray(u, dtype=np.int32) for u in lists]
        self.off = np.concatenate([[0], np.cumsum([len(u) for u in self.lists])]).astype(np.int32)
        self.flat = np.concatenate(self.lists).astype(np.int32)
        self.K, self.x0, self.clamp, self.lt, self.sq = K, x0, clamp, lt, sq
        self.mag = _mag(K, x0)
        self.ref = [O.cell_table(self.mm[c], self.lists[c], self.mag, localtheta=lt, sqlogit=sq,
                                 ncells_for_clamp=clamp)[0] for c in range(len(self.lists))]

    @property
    def n_cells(self):
        return len(self.lists)


def _fast_models():
    """(model, long list?) pairs: corners of the synthetic ranges, high theta x steep drop-out, the sentinel zero-row
    model, o.ifm rows"""
    out = []
    keys = ["conc.b", "conc.a", "corr.b", "corr.a", "corr.theta"]
    for i, corner in enumerate(itertools.product(*[synth.OIFM_RANGES[k] for k in keys])):
        out.append((_model(*corner), i in (0, 11, 22, 31)))
    for th, ca in itertools.product((0.01, 50.0, 1e3, 1e4), (5.0, 70.0)):
        out.append((_model(-3.0, ca, 1.3, 0.7, th), True))
    out.append((SENTINEL_ZERO_MODEL, True))
    ifm = helpers.o_ifm()
    ifm = ifm[ifm["corr.a"] > 0]
    mm, _, _ = api.pack_models(ifm)
    for i in range(0, len(mm), 4):
        out.append((mm[i], i in (0, 16)))
    return out


@functools.lru_cache(maxsize=None)
def fast_case(gi):
    K, x0, clamp = GRIDS[gi]
    rng = np.random.default_rng(100 + gi)
    models, lists = [], []
    for m, long_list in _fast_models():
        models.append(m)
        if long_list:
            lists.append(LONG_COUNTS)
        else:  # 1-3 rows: cells change inside a 32-row header batch of lp_rows_q_kernel
            lists.append(sorted(rng.choice(COUNTS, size=int(rng.integers(1, 4)), replace=False)))
    lists[32 + 7] = LONG_COUNTS[1:]  # theta 1e4, conc.a 70 without a zero count: zero_row = -1
    for m in _tune_margins(_mag(K, x0)):
        models.append(m)
        lists.append([0, 300])
    order = rng.permutation(len(models))
    return Case([models[i] for i in order], [lists[i] for i in order], K, x0, clamp)


LOCAL_GRIDS = [0, 5, 7]


@functools.lru_cache(maxsize=None)
def local_case(gi):
    K, x0, clamp = GRIDS[gi]
    mm, lt, sq = api.pack_models(helpers.knn_models())
    assert lt == 1 and sq == 1
    rng = np.random.default_rng(200 + gi)
    lists = [LONG_COUNTS if c % 16 == 0 else sorted(rng.choice(COUNTS, size=int(rng.integers(1, 4)), replace=False))
             for c in range(len(mm))]
    return Case(mm, lists, K, x0, clamp, lt=1, sq=1)


@functools.lru_cache(maxsize=None)
def classified(gi, local=False):
    """per row of the case: (count, class per element, margin flags, snap point, A, E, log S)"""
    case = local_case(gi) if local else fast_case(gi)
    rows = []
    for c in range(case.n_cells):
        vecs = grid_vectors(case.mm[c], case.mag, case.lt, case.sq)
        for x in case.lists[c]:
            A, E, ks, log_s = row_terms(case.mm[c], case.mag, int(x), vecs=vecs)
            cls, margin = classify(A, E)
            rows.append((int(x), cls, margin, ks, A, E, log_s))
    return rows


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_decoder_round_trip():
    """the numpy packing and decoder are inverse: X = rint(v 2^29) for |v| <= 752 (ties to even, as the addition of the
    magic constant rounds), the "log 0" element is five zero digits, and the digits are those quantize_rows_kernel
    writes"""
    rng = np.random.default_rng(1)
    for K in (1, 16, 101, 102, 103, 401, 408):
        v = rng.uniform(-752.0, 752.0, size=(7, K))
        v[0, :4] = [752.0, -752.0, 0.0, -0.0][: min(4, K)]
        v[1, 0] = -1.7e307  # the clamp
        v[2, :] = rng.normal(0.0, 1e-6, K)
        if K > 3:  # exact ties
            v[3, 1:3] = [3 * 2.0 ** -30, -3 * 2.0 ** -30]
        q = encode(v, K)
        assert q.shape == (7, q_row_bytes(K))
        X = decode(q, K)
        want = np.rint(np.where(v > LOG0, v, 0.0) * SCALE).astype(np.int64)
        assert np.array_equal(X, want)
        assert np.all(q[1, _plane_index(K)[0] + Q_PW * np.arange(Q_NV)] == 0)
        # the two spare bytes of every piece and the pieces beyond the grid stay zero
        used = np.zeros(q_row_bytes(K), bool)
        used[(_plane_index(K)[:, None] + Q_PW * np.arange(Q_NV)[None, :]).ravel()] = True
        assert np.all(q[:, ~used] == 0)
    # the digits of quantize_rows_kernel: d = (int8)(x & 0xFF), x = (x - d) >> 8
    x = np.array([0, 1, -1, 127, 128, -128, -129, 752 * 2 ** 29, -752 * 2 ** 29,
                  0x7F7F7F7F7F, -0x8080808080], np.int64)  # the last two: the extremes of five digits
    q = np.zeros((len(x), q_row_bytes(1)), np.int8)
    r = x.copy()
    for p in range(Q_NV):
        d = ((r + 128) & 0xFF) - 128
        q[:, p * Q_PW] = d
        r = (r - d) >> 8
    assert np.all(r == 0)
    assert np.array_equal(decode(q, 1)[:, 0], x)
    assert np.array_equal(q, encode(x[:, None] / SCALE, 1))


@pytest.mark.parametrize("gi", range(len(GRIDS)), ids=GRID_IDS)
def test_classifier_agrees_with_oracle(gi):
    """every element's class predicts the oracle's value: hi - log S (easy), hi + log1p(exp(-|a - e|)) - log S
    (cross-over), within 0.7 or "log 0" below -735 in the gradual-underflow band (the reference's exp() is a denormal
    there), exactly "log 0" when both exponentials underflow"""
    case = fast_case(gi)
    rows = iter(classified(gi))
    for c in range(case.n_cells):
        for j, x in enumerate(case.lists[c]):
            x_, cls, margin, ks, A, E, log_s = next(rows)
            ref = case.ref[c][:, j]
            with np.errstate(all="ignore"):
                hi = np.maximum(A, E)
                cross = hi + np.log1p(np.exp(-np.abs(A - E))) - log_s
            where = f"cell {c} count {x}"
            e = cls == 0
            np.testing.assert_allclose(ref[e], (hi - log_s)[e], rtol=0, atol=1e-9, err_msg=where)
            e = cls == 1
            np.testing.assert_allclose(ref[e], cross[e], rtol=0, atol=1e-9, err_msg=where)
            e = (cls == 2) | (cls == 3)
            flip = e & (ref < LOG0)
            assert np.all((hi - log_s)[flip] < -735.0), where
            e &= ref > -735.0  # below: the smallest denormals, two roundings apart from the exact value
            assert np.all(np.abs(ref[e] - np.where(cls == 2, hi - log_s, cross)[e]) <= 0.7), where
            assert np.all(ref[cls == 4] < LOG0), where


def _coverage(gis, local=False):
    n_cls = np.zeros(len(CLASSES), np.int64)
    n_margin = np.zeros(3, np.int64)
    snaps = set()
    for gi in gis:
        K = GRIDS[gi][0]
        for x, cls, margin, ks, *_ in classified(gi, local):
            if x == 0:
                continue
            n_cls += np.bincount(cls, minlength=len(CLASSES))
            n_margin += margin.sum(axis=1)
            if ks < 0:
                snaps.add("none")
                continue
            if ks == K - 1:
                snaps.add("last")
            snaps.add("single" if ks >= 384 else (ks // 128, ks % 4))
    return n_cls, n_margin, snaps


def test_inputs_reach_every_class_and_snap_position():
    """the rows of non-zero counts the GPU tests build hit every element class, every class boundary to within 1e-9, and
    the snap point in every position lp_rows_q_kernel treats apart: none, each of the three 128-point rounds x each
    position in a quad, the single points from 384 on, the last grid point"""
    n_cls, n_margin, snaps = _coverage(range(len(GRIDS)))
    print("classes", dict(zip(CLASSES, n_cls.tolist())), "margins (-746, -708, 37.5)", n_margin.tolist())
    assert np.all(n_cls >= 20), dict(zip(CLASSES, n_cls.tolist()))
    assert np.all(n_margin >= 3), n_margin.tolist()
    want = {"none", "last", "single"} | {(j, e) for j in range(3) for e in range(4)}
    assert want <= snaps, sorted(want - snaps, key=str)
    n_cls, _, _ = _coverage(LOCAL_GRIDS, local=True)
    assert np.all(n_cls[[0, 1, 4]] >= 20), dict(zip(CLASSES, n_cls.tolist()))


def test_sentinel_zero_row_model_is_not_based():
    """the steep drop-out, low-dispersion model keeps "log 0" points in its zero-count row (based = 0 on the device)"""
    for gi in (0, 5, 7):
        ref = O.cell_table(SENTINEL_ZERO_MODEL, np.array([0], np.int32), _mag(*GRIDS[gi][:2]),
                           ncells_for_clamp=GRIDS[gi][2])[0][:, 0]
        assert np.any(ref < LOG0), GRIDS[gi]


# ---- GPU: the probe against the oracle -----------------------------------------------------------------------------------
def probe(ctx, case, **options):
    """scde_b200_probe_table under the given scde_b200_options fields"""
    n_rows, K = int(case.off[-1]), case.K
    out = {"q": np.zeros((n_rows, q_row_bytes(K)), np.int8), "range": np.zeros(n_rows, np.uint32),
           "zero_row": np.empty(case.n_cells, np.int32), "based": np.empty(case.n_cells, np.int32),
           "zero_rows": np.empty((case.n_cells, K))}
    keep = ctx.set_options(**options)
    try:
        _lib.check(_lib.lib().scde_b200_probe_table(
            ctx.handle, _lib.p_f64(case.mm), case.n_cells, _lib.p_i32(case.flat), _lib.p_i32(case.off),
            _lib.p_f64(_lib.f64(case.mag)), K, case.lt, case.sq, case.clamp, out["q"].ctypes.data_as(C.c_void_p),
            out["range"].ctypes.data_as(C.c_void_p), _lib.p_i32(out["zero_row"]), _lib.p_i32(out["based"]),
            _lib.p_f64(out["zero_rows"])))
    finally:
        ctx.restore_options(keep)
    out["X"] = decode(out["q"], K)
    return out


def check_probe(case, out):
    """every row of the probe against the oracle; returns counts of what was checked"""
    from test_gpu_parity import _rows_close

    K = case.K
    k = np.arange(K)
    seen = {"rows": 0, "normal": 0, "low": 0, "log0": 0, "flips": 0, "irregular": 0, "not_based": 0}
    for c in range(case.n_cells):
        ucl, ref = case.lists[c], case.ref[c]
        j0 = int(np.nonzero(ucl == 0)[0][0]) if np.any(ucl == 0) else -1
        assert out["zero_row"][c] == (case.off[c] + j0 if j0 >= 0 else -1), c
        z_dev = out["zero_rows"][c]
        if j0 >= 0:
            _rows_close(z_dev, ref[:, j0])
            assert out["based"][c] == int(np.all(z_dev > LOG0)), c  # (_rows_close: "log 0" as the reference's)
        else:
            assert out["based"][c] == 0, c
        based = bool(out["based"][c])
        seen["not_based"] += not based
        for j, x in enumerate(ucl):
            r = case.off[c] + j
            lp = ref[:, j]
            sub = based and x != 0
            Z = z_dev if sub else np.zeros(K)
            want = lp - Z
            normal = (lp > -700.0) & ((z_dev > -700.0) if sub else True)
            X, rr = out["X"][r], int(out["range"][r])
            where = f"cell {c} count {x} (row {r}, based {based})"
            ref_ok = lp > LOG0
            seen["rows"] += 1
            if rr == Q_RANGE_IRREGULAR:
                seen["irregular"] += 1
                idx = np.nonzero(ref_ok)[0]
                interval = len(idx) > 0 and idx[-1] - idx[0] + 1 == len(idx)
                assert not interval or np.all(lp[ref_ok] < -735.0), where
                continue
            lo, hi = rr & 0xFFFF, rr >> 16
            assert lo <= hi < K, where
            dev_ok = (k >= lo) & (k <= hi)
            assert np.all(X[~dev_ok] == 0), f"{where}: digits of a \"log 0\" element"
            seen["log0"] += int(np.sum(~dev_ok))
            both = ref_ok & dev_ok
            v = X / SCALE
            sel = both & normal if np.any(both & normal) else both
            c_row = float(np.median(v[sel] - want[sel])) if np.any(sel) else 0.0
            flip = ref_ok != dev_ok
            if flip.any():
                seen["flips"] += int(flip.sum())
                assert np.all(lp[flip & ref_ok] < -735.0), f"{where}: range differs above the denormal edge"
                assert np.all((v - c_row + Z)[flip & dev_ok] < -735.0), f"{where}: range differs above the denormal edge"
            if x == 0 and np.any(both & normal):  # FP64-normalised rows carry no row constant
                assert abs(c_row) <= 1e-8, f"{where}: zero-count row not normalised ({c_row})"
            nm = both & normal
            dX = np.abs(X[nm] - np.rint((want[nm] + c_row) * SCALE))
            assert np.all(dX <= 1), f"{where}: |dX| = {dX.max():.0f} at k = {k[nm][np.argmax(dX)]}"
            low = both & ~normal
            assert np.all(np.abs(v[low] - (want[low] + c_row)) <= 0.7), where
            seen["normal"] += int(nm.sum())
            seen["low"] += int(low.sum())
    return seen


PRODUCERS = {"q_kernel": {}, "per_element_kernel": {"lp_rows_kernel": 1}, "quantize_pass": {"fused_fixed_point": 0}}


@pytest.mark.gpu
@pytest.mark.parametrize("gi", range(len(GRIDS)), ids=GRID_IDS)
@pytest.mark.parametrize("producer", list(PRODUCERS))
def test_table_rows_match_oracle(ctx, producer, gi):
    """every element of every row: normal elements to one unit of 2^-29 after the row constant (fused rows omit log S),
    lower ones within 0.7, "log 0" elements all-zero digits and outside the row's range, zero-count rows in FP64 within
    1e-9, `based` exactly "the zero-count row has no log 0"."""
    case = fast_case(gi)
    seen = check_probe(case, probe(ctx, case, **PRODUCERS[producer]))
    print(producer, GRID_IDS[gi], seen)
    assert seen["not_based"] >= 2 and seen["log0"] > 0 and seen["low"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("gi", LOCAL_GRIDS, ids=[GRID_IDS[g] for g in LOCAL_GRIDS])
def test_table_rows_local_theta(ctx, gi):
    """local-theta, square-logit models (knn fit): the general row kernel and the quantize pass"""
    case = local_case(gi)
    seen = check_probe(case, probe(ctx, case))
    print("local_theta", GRID_IDS[gi], seen)


@pytest.mark.gpu
@pytest.mark.parametrize("gi", range(len(GRIDS)), ids=GRID_IDS)
def test_q_kernel_equals_per_element_kernel(ctx, gi):
    """lp_rows_q_kernel against lp_rows_fast_kernel on the same rows: one unit of 2^-29 on normal elements, 0.7 below,
    the same zero-count rows and flags, the same ranges except at grid points below -735 (where the reference's own
    exp() is one of the smallest denormals or zero, so either side of "log 0" is the reference's value to rounding)"""
    case = fast_case(gi)
    a, b = probe(ctx, case), probe(ctx, case, lp_rows_kernel=1)
    for key in ("zero_row", "based"):
        assert np.array_equal(a[key], b[key]), key
    assert np.array_equal(a["zero_rows"], b["zero_rows"], equal_nan=True)
    k = np.arange(case.K)
    n_diff = 0
    for c in range(case.n_cells):
        for j in range(len(case.lists[c])):
            r, lp = case.off[c] + j, case.ref[c][:, j]
            ok = []
            for out in (a, b):
                rr = int(out["range"][r])
                ok.append(np.zeros(case.K, bool) if rr == Q_RANGE_IRREGULAR else (k >= (rr & 0xFFFF)) & (k <= rr >> 16))
            if a["range"][r] != b["range"][r]:
                n_diff += 1
                assert np.all(lp[ok[0] != ok[1]] < -735.0), (c, int(case.lists[c][j]))
            both = ok[0] & ok[1]
            dX = np.abs(a["X"][r] - b["X"][r])
            assert np.all(dX[both & (lp > -700.0)] <= 1), (c, int(case.lists[c][j]))
            assert np.all(dX[both] <= 0.7 * SCALE), (c, int(case.lists[c][j]))
    print("q vs per-element", GRID_IDS[gi], "rows with different ranges:", n_diff)


@pytest.mark.gpu
def test_probe_rejects_grids_without_fixed_point_form(ctx):
    case = fast_case(0)
    big = Case(case.mm[:2], case.lists[:2], Q_MAX_K + 1, 0.0, 1)
    with pytest.raises(_lib.ScdeB200Error, match="fixed-point"):
        probe(ctx, big)


# ---- GPU: the new model regions end to end ---------------------------------------------------------------------------
def _extreme_models():
    rows = [_model(-3.0, ca, 1.3, 0.7, th) for th in (50.0, 1e3, 1e4) for ca in (5.0, 70.0)]
    rows += [_model(-1.5, 0.8, 1.0, 0.5, 1.0), SENTINEL_ZERO_MODEL]
    return rows


def _frame(rows, prefix="cell"):
    cols = ["conc.b", "conc.a", "fail.r", "corr.b", "corr.a", "corr.theta"]
    return pd.DataFrame(np.array(rows)[:, :6], columns=cols, index=[f"{prefix}{i}" for i in range(len(rows))])


@pytest.mark.gpu
def test_posteriors_high_theta_and_steep_dropout(ctx):
    """counts drawn from high-theta and steep drop-out models: the tcgen05 path against the oracle (1e-6) on the same
    draws and against the FP64 kernel"""
    from test_gpu_parity import _logp_close

    rng = np.random.default_rng(8)
    models = _frame([r for r in _extreme_models() for _ in range(4)])
    counts = synth.make_counts(rng, models, 150)
    prior = synth.make_prior(150)
    mm, lt, sq = api.pack_models(models)
    mag = api.marginals_from_prior(prior)
    flat, off, uci = O.unique_counts(counts)
    want = O.log_boot_posterior(mm, flat, off, uci, mag, 100, boot_idx=O.boot_indices(1, counts.shape[1], 100))["jp"]
    got = {}
    for kernel in (3, 2):
        ctx.set_contract_kernel(kernel)
        try:
            got[kernel] = api.scde_posteriors(models, counts, prior, n_randomizations=100, context=ctx).to_numpy()
        finally:
            ctx.set_contract_kernel(0)
        ok, worst = _logp_close(got[kernel], want)
        assert ok, (kernel, worst)
    ok, worst = _logp_close(got[3], got[2])
    assert ok, worst


def _mixed_based_workload():
    """ordinary cells and two cells of the sentinel zero-row model in each group; a third of the genes zero in those"""
    w = synth.make_workload(3, n_genes=120, n_cells=20, seed=41)
    rows = [r for r in api.pack_models(w.models)[0]] + [SENTINEL_ZERO_MODEL] * 4
    models = _frame(rows)
    counts = np.zeros((120, 24), np.int32, order="F")
    counts[:, :20] = w.counts
    counts[:, 20:] = synth.make_counts(np.random.default_rng(4), models.iloc[20:], 120)
    counts[::3, 20:] = 0
    codes = np.array([i % 2 for i in range(20)] + [0, 1, 0, 1], dtype=np.int32)
    return models, counts, w.prior, codes


@pytest.mark.gpu
def test_one_shot_call_with_unbased_cells(ctx):
    """a cell whose zero-count row holds "log 0" (based = 0) next to ordinary cells in both groups of the one-shot call:
    its zero-count entries are listed for the contraction, its zero-count row's planes come from the FP64 row launch,
    the base sums skip it.  Each group's joint posterior against the oracle."""
    from test_gpu_parity import _logp_close

    models, counts, prior, codes = _mixed_based_workload()
    mm, lt, sq = api.pack_models(models)
    mag = api.marginals_from_prior(prior)
    # the path is reached: the device marks those cells as not based
    lists = [np.unique(counts[:, c]) for c in range(counts.shape[1])]
    out = probe(ctx, Case(mm, lists, len(mag), 0.0, counts.shape[1]))
    assert out["based"][20:].tolist() == [0] * 4 and np.all(out["based"][:20] == 1)
    x, y = prior["x"].to_numpy(), prior["y"].to_numpy()
    zi = api._zero_index(api.fold_change_grid(x), 0.0)
    res = api.expression_difference_call(ctx, counts, mm, x, y, codes, 100, 1, zero_index=zi, local_theta=lt, sqlogit=sq,
                                         joint_posteriors=True)
    for lev in (0, 1):
        ii = np.nonzero(codes == lev)[0]
        fl, of, uc = O.unique_counts(counts[:, ii])
        wj = O.log_boot_posterior(np.asfortranarray(mm[ii]), fl, of, uc, mag, 100,
                                  boot_idx=O.boot_indices(1, len(ii), 100))["jp"]
        ok, worst = _logp_close(res["joint_posteriors"][lev], wj)
        assert ok, (lev, worst)


@pytest.mark.gpu
def test_contrasts_with_unbased_cells_equal_one_shot_call(ctx):
    """DifferenceSession.contrasts over the same data equals the one-shot call bit for bit"""
    from test_contrasts import _assert_same

    models, counts, prior, codes = _mixed_based_workload()
    groups = pd.Categorical.from_codes(codes, categories=["a", "b"])
    kw = dict(n_randomizations=100, return_posteriors=True)
    with api.DifferenceSession(models, counts, prior, context=ctx) as s:
        res = s.contrasts(groups, "pairs", **kw)
    want = api.scde_expression_difference(models, counts, prior, groups=groups, context=ctx, **kw)
    _assert_same(res["a vs b"], want)
