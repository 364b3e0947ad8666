"""The FP64 rerun of a call whose tcgen05 status word asks for it: the caller's options stay as they were set, and the
result is that of the same call on the FP64 DMMA kernel (scde_b200_set_contract_kernel(ctx, 2)), bit for bit."""
import numpy as np
import pytest

from scde_b200 import api, synth

pytestmark = pytest.mark.gpu

N_BOOT = 10


def _diff_args(w, bi):
    """the two-group call on w with group 0 = the first 150 cells, whose draws are bi"""
    mm, lt, sq = api.pack_models(w.models)
    x, y = w.prior["x"].to_numpy(), w.prior["y"].to_numpy()
    codes = np.where(np.arange(w.counts.shape[1]) < bi.shape[1], 0, 1).astype(np.int32)
    args = (np.asarray(w.counts, dtype=np.int32, order="F"), mm, x, y, codes, N_BOOT, 1)
    kw = {"zero_index": api._zero_index(api.fold_change_grid(x), 0.0), "local_theta": lt, "sqlogit": sq,
          "boot_idx": (bi, None, None, None)}
    return args, kw


def _one_shot(ctx, w, bi):
    args, kw = _diff_args(w, bi)
    return api.expression_difference_call(ctx, *args, joint_posteriors=True, **kw)


def _resident_job(ctx, w, bi):
    args, kw = _diff_args(w, bi)
    job = api.DifferenceJob(ctx, *args, **kw)
    try:
        job.run()
        return job.download(joint_posteriors=True)
    finally:
        job.close()


def _log_boot(ctx, w, bi):
    return {"jp": api.scde_posteriors(w.models, w.counts, w.prior, n_randomizations=N_BOOT, boot_idx=bi,
                                      context=ctx).to_numpy()}


@pytest.mark.parametrize("call", [_one_shot, _resident_job, _log_boot], ids=["one_shot", "resident_job", "log_boot"])
def test_multiplicity_fallback_keeps_options_and_equals_fp64_kernel(ctx, call):
    """every draw of a group of 150 cells hits its first cell: a multiplicity of 150 does not fit the int8 operand, so
    the whole call (log_boot) or the whole run (two-group job) is repeated on the FP64 DMMA kernel"""
    w = synth.make_workload(3, n_genes=150, n_cells=150 if call is _log_boot else 640, seed=2)
    bi = np.zeros((N_BOOT, 150), dtype=np.int32)
    res = {}
    for kernel in (0, 2):
        ctx.set_contract_kernel(kernel)
        try:
            before = bytes(ctx.options())
            res[kernel] = call(ctx, w, bi)
            assert bytes(ctx.options()) == before
        finally:
            ctx.set_contract_kernel(0)
    for k in ("jp", "idx", "z", "cz"):
        if k in res[0]:
            assert np.array_equal(res[0][k], res[2][k]), k
    for i in range(len(res[0].get("joint_posteriors", []))):
        assert np.array_equal(res[0]["joint_posteriors"][i], res[2]["joint_posteriors"][i])
