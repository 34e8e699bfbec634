"""CPU tests: the oracle restatement against golden vectors produced by the REFERENCE'S OWN CODE.

``tests/golden/golden_ref_v1.npz`` was written by ``tests/golden/make_golden_ref.py``, which imports
/root/reference/src/model.py and eval.py unmodified (absent third-party packages replaced by stand-ins, see
that script's header) and runs ``Generator`` / ``Discriminator`` / ``bSSFPToDWITensorModel._gen_step /
_discr_step / training_step`` and ``do_calc_diff_maps / do_calc_error_avg / do_calc_scalar_maps /
do_invert_dwi_tensor_norm``. These tests pin ``oracle/`` to those outputs; the GPU tests then compare the
sm_100a path with both the oracle and the same goldens (tests/test_reference_golden_gpu.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import eval_oracle as E
from oracle import model_oracle as O
from tests.golden.make_golden_ref import GOLDEN_THREADS, state_checksum, synth_batch, zero_dropout

REF = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_ref_v1.npz"))


@pytest.fixture(autouse=True)
def _reference_thread_count():
    """Run on the reference's thread count: the training-step goldens keep the rounding of its reductions."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def _same_init(mod):
    torch.manual_seed(0)
    g, d = O.Generator(mod), O.Discriminator(mod)
    ok = abs(state_checksum(g) - float(REF[f"{mod}_g_checksum"])) <= 1e-9 * float(REF[f"{mod}_g_checksum"])
    return g, d, ok


@pytest.mark.parametrize("mod", ["bssfp", "t1w"])
def test_module_tree_is_the_references(mod):
    g, d, ok = _same_init(mod)
    assert list(g.state_dict().keys()) == list(REF[f"{mod}_g_keys"])
    assert list(d.state_dict().keys()) == list(REF[f"{mod}_d_keys"])
    assert [str(tuple(v.shape)) for v in g.state_dict().values()] == list(REF[f"{mod}_g_shapes"])
    assert [str(tuple(v.shape)) for v in d.state_dict().values()] == list(REF[f"{mod}_d_shapes"])
    assert sum(p.numel() for p in g.parameters()) == int(REF[f"{mod}_g_nparams"]) == 22646182
    assert sum(p.numel() for p in d.parameters()) == int(REF[f"{mod}_d_nparams"]) == 11230593
    if not ok:
        pytest.skip("default torch init differs from the torch version that generated the goldens")
    # same construction order => the same draws from the init RNG stream
    assert abs(state_checksum(d) - float(REF[f"{mod}_d_checksum"])) <= 1e-9 * float(REF[f"{mod}_d_checksum"])


@pytest.mark.parametrize("mod", ["bssfp", "t1w"])
def test_forward_values_and_losses(mod):
    g, d, ok = _same_init(mod)
    if not ok:
        pytest.skip("default torch init differs from the torch version that generated the goldens")
    xb, yb = synth_batch(O.in_channels_of(mod))
    g.eval()
    with torch.no_grad():
        np.testing.assert_allclose(g(xb[:1]).numpy(), REF[f"{mod}_g_eval_32"], rtol=1e-4, atol=2e-5)
    d.train()
    with torch.no_grad():
        np.testing.assert_allclose(d(xb, yb).numpy(), REF[f"{mod}_d_train_32_b2"], rtol=1e-3, atol=1e-4)
    d.eval()
    with torch.no_grad():
        np.testing.assert_allclose(d(xb, yb).numpy(), REF[f"{mod}_d_eval_32_b2"], rtol=1e-3, atol=1e-4)
    # _gen_step / _discr_step of the reference's LightningModule (train mode, dropout 0) on fresh weights
    g, d, _ = _same_init(mod)
    zero_dropout(g)
    g.train(); d.train()
    with torch.no_grad():
        gl, y_hat = O.gen_loss(g, d, xb, yb)
        dl = O.discr_loss(g, d, xb, yb)
        l1 = torch.nn.functional.l1_loss(y_hat, yb)
    assert abs(gl.item() - float(REF[f"{mod}_gen_loss"])) < 1e-4 * abs(float(REF[f"{mod}_gen_loss"]))
    assert abs(dl.item() - float(REF[f"{mod}_discr_loss"])) < 1e-4
    assert abs(l1.item() - float(REF[f"{mod}_gen_loss_recon_L1"])) < 1e-5
    # recon = (L1 + Perceptual[=0]) / 2 * 1e2   (ref:src/model.py:201-213)
    assert abs(O.recon_loss(y_hat, yb).item() - float(REF[f"{mod}_gen_loss_recon"])) < 1e-3
    assert abs(float(REF[f"{mod}_gen_loss_recon"]) - float(REF[f"{mod}_gen_loss_recon_L1"]) * 50.0) < 1e-4


def test_phase_gradients_and_freezing():
    """G phase: D receives no gradient (toggle_optimizer), G's gradients equal the reference's; D phase likewise."""
    mod = "bssfp"
    g, d, ok = _same_init(mod)
    if not ok:
        pytest.skip("default torch init differs from the torch version that generated the goldens")
    assert int(REF["bssfp_discr_grads_in_gen_phase"]) == 0 and int(REF["bssfp_gen_grads_in_discr_phase"]) == 0
    zero_dropout(g)
    g.train(); d.train()
    xb, yb = synth_batch(24)
    O._set_requires_grad(d, False)
    gl, _ = O.gen_loss(g, d, xb, yb)
    gl.backward()
    O._set_requires_grad(d, True)
    assert all(p.grad is None for p in d.parameters())
    gp = dict(g.named_parameters(remove_duplicate=False))
    for k in [k for k in REF.files if k.startswith("bssfp_ggrad::")]:
        ref = torch.from_numpy(REF[k])
        got = gp[k.split("::")[1]].grad
        assert ((got - ref).norm() / ref.norm()).item() < 2e-3, k
    g.zero_grad(set_to_none=True)
    O._set_requires_grad(g, False)
    dl = O.discr_loss(g, d, xb, yb)
    dl.backward()
    O._set_requires_grad(g, True)
    assert all(p.grad is None for p in g.parameters())
    dp = dict(d.named_parameters(remove_duplicate=False))
    for k in [k for k in REF.files if k.startswith("bssfp_dgrad::")]:
        ref = torch.from_numpy(REF[k])
        got = dp[k.split("::")[1]].grad
        assert ((got - ref).norm() / ref.norm()).item() < 2e-3, k


def test_three_training_steps_follow_the_reference():
    """oracle.gan_step x 3 == the reference's training_step x 3 (same losses, same weights afterwards)."""
    mod = "bssfp"
    g, d, ok = _same_init(mod)
    if not ok:
        pytest.skip("default torch init differs from the torch version that generated the goldens")
    zero_dropout(g)
    g.train(); d.train()
    opt_g, opt_d = O.make_optimizers(g, d)
    xb, yb = synth_batch(24)
    gls, dls = [], []
    for _ in range(3):
        gl, dl = O.gan_step(g, d, opt_g, opt_d, xb, yb)
        gls.append(float(gl)); dls.append(float(dl))
    np.testing.assert_allclose(gls, REF["bssfp_train3_gen_loss"], rtol=2e-3)
    np.testing.assert_allclose(dls, REF["bssfp_train3_discr_loss"], rtol=2e-3, atol=1e-4)
    assert abs(state_checksum(g) / float(REF["bssfp_train3_gen_checksum"]) - 1) < 1e-4
    assert abs(state_checksum(d) / float(REF["bssfp_train3_discr_checksum"]) - 1) < 1e-4
    assert int(d.d2.bn.num_batches_tracked) == int(REF["bssfp_train3_num_batches_tracked_d2"]) == 9
    np.testing.assert_allclose(d.d2.bn.running_mean.numpy(), REF["bssfp_train3_bn_running_mean_d2"], rtol=5e-2, atol=1e-3)
    np.testing.assert_allclose(g.blocks["bssfp"].bn.running_var.numpy(), REF["bssfp_train3_head_running_var"], rtol=1e-3)


def test_lightning_shell_restatement_is_pinned_by_the_reference_run():
    """oracle/lightning_shell.py (the LightningModule statements with injectable classes) driven with the oracle's
    classes reproduces what the REAL ``bSSFPToDWITensorModel.training_step`` x 3 logged and left behind; the GPU test
    then injects the sm_100a drop-in classes into this same shell."""
    from oracle.lightning_shell import LightningShell, OracleClasses
    torch.manual_seed(0)
    lm = LightningShell("bssfp", OracleClasses)
    if abs(state_checksum(lm.gen) - float(REF["bssfp_lm_gen_checksum0"])) > 1e-9 * float(REF["bssfp_lm_gen_checksum0"]):
        pytest.skip("default torch init differs from the torch version that generated the goldens")
    assert abs(state_checksum(lm.discr) - float(REF["bssfp_lm_discr_checksum0"])) <= 1e-9 * float(REF["bssfp_lm_discr_checksum0"])
    zero_dropout(lm)
    lm.train()
    xb, yb = synth_batch(24)
    gls, dls = [], []
    for it in range(3):
        lm.training_step({"bssfp": {"data": xb}, "dwi-tensor_orig": {"data": yb}}, it)
        gls.append(lm.logged["train_gen_loss"]); dls.append(lm.logged["train_discr_loss"])
    np.testing.assert_allclose(gls, REF["bssfp_train3_gen_loss"], rtol=2e-3)
    np.testing.assert_allclose(dls, REF["bssfp_train3_discr_loss"], rtol=2e-3, atol=1e-4)
    assert abs(state_checksum(lm.gen) / float(REF["bssfp_train3_gen_checksum"]) - 1) < 1e-4
    assert abs(state_checksum(lm.discr) / float(REF["bssfp_train3_discr_checksum"]) - 1) < 1e-4
    assert all(p.requires_grad for p in lm.parameters())            # untoggled again
    lm.eval()
    with torch.no_grad():
        np.testing.assert_allclose(lm(xb[:1]).numpy(), REF["bssfp_train3_g_eval_32"], rtol=5e-2, atol=5e-3)


def test_eval_arithmetic_is_the_references():
    pred, tgt, mask, probseg = REF["eval_pred"], REF["eval_target"], REF["eval_mask"], REF["eval_probseg"]
    diff = E.rel_error_map(pred, tgt)
    np.testing.assert_array_equal(diff, REF["eval_diff_rel"])                  # bit-exact, NaN == NaN
    errs, cleaned = E.roi_error_avg(diff, mask, probseg)
    np.testing.assert_allclose(errs, REF["eval_errs_rel"], rtol=1e-12, equal_nan=True)
    np.testing.assert_array_equal(cleaned, REF["eval_diff_rel_cleaned"])
    assert np.isnan(REF["eval_errs_rel"][:, 0]).all() and np.isfinite(REF["eval_errs_rel"][:, 1:]).all()
    da = E.rel_error_map(REF["eval_ang_pred"], REF["eval_ang_target"], kind="azimuth")
    np.testing.assert_array_equal(da, REF["eval_diff_ang"])
    errs_a, _ = E.roi_error_avg(da, mask, probseg)
    np.testing.assert_allclose(errs_a, REF["eval_errs_ang"], rtol=1e-12)
    lo, hi = REF["denorm_minmax"]
    np.testing.assert_array_equal(E.invert_dwi_tensor_norm(pred, lo, hi), REF["denorm_out"])


def test_dti_scalar_maps_are_the_references():
    """The batched oracle equals the reference's per-voxel LAPACK loop, eigenvector signs included."""
    maps = E.dti_scalar_maps(REF["dti_tensor6"])
    for k in ("fa", "md", "ad", "rd", "azimuth", "inclination", "rgb"):
        np.testing.assert_allclose(maps[k], REF[f"dti_{k}"], rtol=1e-9, atol=1e-9, err_msg=k)


def test_golden_eval_inputs_regenerate_from_the_script():
    """The evaluation inputs stored beside the reference's outputs are the ones ``make_golden_ref.py`` draws from its
    seeds, so the fixture cannot drift from the script that claims to have produced it."""
    from tests.golden import make_golden_ref as M
    pred, tgt, mask, probseg = M.synth_eval_volumes()
    for k, v in (("eval_pred", pred), ("eval_target", tgt), ("eval_mask", mask), ("eval_probseg", probseg),
                 ("eval_ang_pred", (pred[..., 0] * 720.0 - 180.0).astype(np.float32)),
                 ("eval_ang_target", (tgt[..., 0] * 360.0).astype(np.float32))):
        np.testing.assert_array_equal(REF[k], v, err_msg=k)
    np.testing.assert_allclose(REF["dti_tensor6"], M.synth_dti(), rtol=1e-6, atol=0)    # QR: LAPACK-dependent last bits


def test_config1_full_size_matches_the_reference():
    """BASELINE config 1 exactly (G fwd + bwd, one 64^3 bSSFP patch, batch 1, fp32 CPU) against the reference's run."""
    g, _, ok = _same_init("bssfp")
    if not ok:
        pytest.skip("default torch init differs from the torch version that generated the goldens")
    zero_dropout(g)
    g.train()
    x, y = synth_batch(24, b=1, s=64, seed=4321)
    y_hat = g(x)
    loss = torch.nn.functional.l1_loss(y_hat, y)
    loss.backward()
    assert abs(loss.item() - float(REF["cfg1_loss"])) < 1e-6
    np.testing.assert_allclose(y_hat.detach()[0, :, ::21, ::21, ::21].numpy(), REF["cfg1_out_probe"], rtol=1e-4, atol=1e-5)
    names = [k for k, p in g.named_parameters() if p.grad is not None]
    assert names == list(REF["cfg1_grad_names"])
    norms = np.array([p.grad.double().norm().item() for k, p in g.named_parameters() if p.grad is not None])
    # conv biases in front of a batch-statistics norm: analytically zero gradients, rounding noise on both sides
    big = np.array([not (k.endswith("conv.bias") and "final_conv" not in k and "deconv" not in k) for k in names])
    np.testing.assert_allclose(norms[big], REF["cfg1_grad_norms"][big], rtol=2e-3)
    np.testing.assert_allclose(g.blocks["unet"].final_conv.weight.grad.numpy(), REF["cfg1_grad_final_conv_weight"],
                               rtol=1e-3, atol=1e-7)
