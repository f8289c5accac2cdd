"""The oracle restatement (oracle/restatement.py) against the golden fixtures generated from the REAL reference
modules by oracle/make_golden.py.  CPU only.  (In the authoring container make_golden.py additionally asserts
bit-equality with the imported reference; this test is what re-checks the pin wherever the suite runs.)"""
import pytest
import torch

from oracle import restatement as R
from oracle.make_golden import GOLDEN_THREADS
from tests import helpers as H

CASES = ["model_ad_h4", "model_ad_h8", "model_cnn_ad", "model_single", "model_transformer", "model_transformer_res",
         "model_cnn", "model_ad_dim64",
         "model_ad_full_b2",         # BASELINE configs[0]: model_ad, batch 2, 91x109x91, fwd+bwd on CPU
         "mnet_b4"]                  # BASELINE configs[4]: the MiSePyNet baseline
TOL = 2e-4      # other host CPUs may pick different oneDNN/MKL kernels than the container that wrote the fixtures


@pytest.fixture
def golden_threads():
    """Sum in the order the fixtures were written with: the thread count splits the fp32 reductions, and the near-zero
    conv-bias gradients (and the batch-2 full-size gradients) are that rounding noise."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name, golden_threads):
    gold = H.load_golden(name)
    mri, pet, label = H.case_inputs(gold)
    inputs = (mri,) if gold["kind"] == "model_single" else (mri, pet)
    sd = R.clone_state(H.case_state(gold))
    outs = H.oracle_forward(gold["kind"], sd, inputs, gold["kwargs"], True, 0.0)
    ce, ad, total = H.losses(outs, label)
    total.backward()
    for o, g in zip(outs, gold["train_outs"]):
        assert torch.allclose(o, g, atol=TOL, rtol=TOL)
    assert abs(float(total) - gold["train_losses"][2]) < TOL
    for k, gs in gold["grad_sample"].items():
        g = sd[k].grad
        assert g is not None, k
        scale = max(gold["grad_norm"][k], 1e-6)
        assert float((H.sample(g) - gs).abs().max()) <= 5e-3 * scale + 1e-6, k
        assert abs(float(g.norm()) - gold["grad_norm"][k]) <= 2e-3 * scale + 1e-6, k
    for k, v in gold["buffers_after"].items():
        assert torch.allclose(sd[k].to(v.dtype), v, atol=TOL, rtol=TOL), k
    # eval path with the updated running statistics
    sd_eval = R.clone_state(sd, requires_grad=False)
    with torch.no_grad():
        e_outs = H.oracle_forward(gold["kind"], sd_eval, inputs, gold["kwargs"], False)
    for o, g in zip(e_outs, gold["eval_outs"]):
        assert torch.allclose(o, g, atol=TOL, rtol=TOL)
    assert torch.equal(e_outs[0].argmax(1), gold["eval_argmax"])


def test_bf16_rounding_oracle_is_close_to_fp32_oracle():
    """Oracle-A (bf16 rounding at the CUDA path's rounding points) stays near Oracle-B on a small case."""
    gold = H.load_golden("model_single")
    mri, pet, label = H.case_inputs(gold)
    sd_a = R.clone_state(H.case_state(gold))
    sd_b = R.clone_state(H.case_state(gold))
    la = R.model_single_forward(sd_a, mri, True, R.bf16_round)
    lb = R.model_single_forward(sd_b, mri, True, None)
    assert float((la - lb).abs().max()) < 5e-2


def test_gradient_reversal_sign_and_scale():
    x = torch.randn(4, 8, requires_grad=True)
    R.revgrad(x, 2.0).sum().backward()
    assert torch.equal(x.grad, torch.full_like(x, -2.0))
