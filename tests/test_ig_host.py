"""Host-side rules of interpret.integrated_gradients (no GPU, no kernel launch): the path tables, the argument refusals,
and the block-1 factorisation itself restated in float64 on a tiny random block 1 (DESIGN section 3.10)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from transmf_ad_b200 import _lib as L
from transmf_ad_b200.interpret import integrated_gradients, ig_path
from transmf_ad_b200.models import mymodel as M
from transmf_ad_b200.models.MiSePyNet import Mnet


@pytest.mark.parametrize("n", [1, 2, 7, 50])
def test_path_tables_against_numpy(n):
    a, w = ig_path(n, "gausslegendre")
    t, wt = np.polynomial.legendre.leggauss(n)
    assert np.array_equal(a, (1 + t) / 2) and np.array_equal(w, wt / 2)
    a2, w2 = ig_path(n, "riemann_middle")
    assert np.allclose(a2, (np.arange(n) + 0.5) / n, rtol=0, atol=1e-15) and np.allclose(w2, 1.0 / n, rtol=0, atol=0)
    for alpha, weight in ((a, w), (a2, w2)):
        assert alpha.shape == weight.shape == (n,)
        assert abs(weight.sum() - 1.0) < 1e-13
        assert (alpha > 0).all() and (alpha < 1).all() and (np.diff(alpha) > 0).all()


@pytest.fixture
def no_launch(monkeypatch):
    def refuse(name, *args, **kw):
        raise AssertionError(f"{name} launched before the arguments were checked")
    monkeypatch.setattr(L, "call", refuse)


def _model():
    return M.model_CNN_ad(128).eval()


def _inputs(B=2):
    return torch.zeros(B, 1, 8, 8, 8), torch.zeros(B, 1, 8, 8, 8)


@pytest.mark.parametrize("method", ["riemann_left", "riemann_trapezoid", "riemann_right", "", None, "GaussLegendre"])
def test_unknown_and_alpha_zero_methods_are_refused(method, no_launch):
    with pytest.raises(ValueError, match="method"):
        integrated_gradients(_model(), _inputs(), 0, method=method)


@pytest.mark.parametrize("n", [0, -3, 2.0, True, None, "50"])
def test_bad_step_counts_are_refused(n, no_launch):
    with pytest.raises(ValueError, match="n_steps"):
        integrated_gradients(_model(), _inputs(), 0, n_steps=n)


@pytest.mark.parametrize("ibs", [0, -8, 8.0, False, "64"])
def test_bad_internal_batch_sizes_are_refused(ibs, no_launch):
    with pytest.raises(ValueError, match="internal_batch_size"):
        integrated_gradients(_model(), _inputs(), 0, internal_batch_size=ibs)


def test_training_mode_is_refused(no_launch):
    with pytest.raises(ValueError, match="eval"):
        integrated_gradients(_model().train(), _inputs(), 0)
    model = _model()
    model.fc_cls.train()
    with pytest.raises(ValueError, match="eval"):
        integrated_gradients(model, _inputs(), 0)


def test_a_model_without_towers_is_refused(no_launch):
    with pytest.raises(ValueError, match="sNet"):
        integrated_gradients(Mnet().eval(), _inputs(), 0)


@pytest.mark.parametrize("inputs", [torch.zeros(2, 1, 8, 8), (torch.zeros(2, 2, 8, 8, 8),) * 2, (), ("mri", "pet"),
                                    (torch.zeros(2, 1, 8, 8, 8),), (torch.zeros(2, 1, 8, 8, 8), torch.zeros(2, 1, 8, 8, 9))])
def test_bad_inputs_are_refused(inputs, no_launch):
    with pytest.raises(ValueError, match="inputs"):
        integrated_gradients(_model(), inputs, 0)


def test_cpu_inputs_are_refused(no_launch):
    with pytest.raises(ValueError, match="CUDA"):
        integrated_gradients(_model(), _inputs(), 0)


@pytest.mark.parametrize("where", ["tower", "tower_pre", "conv1", "conv1_pre"])
def test_hooks_on_a_tower_or_block_1_are_refused(where, no_launch):
    model = _model()
    mod = model.mri_cnn if where.startswith("tower") else model.pet_cnn.conv1
    if where.endswith("_pre"):
        mod.register_forward_pre_hook(lambda m, a: None)
    else:
        mod.register_forward_hook(lambda m, a, o: None)
    with pytest.raises(ValueError, match="hook"):
        integrated_gradients(model, _inputs(), 0)


def test_a_negative_block1_slope_is_refused(no_launch):
    model = _model()
    model.pet_cnn.conv1[2].negative_slope = -0.1
    with pytest.raises(ValueError, match="slope"):
        integrated_gradients(model, _inputs(), 0)


def test_refusals_leave_the_model_as_found(no_launch):
    model = _model()
    model.fc_cls[0].weight.requires_grad_(False)
    flags = [p.requires_grad for p in model.parameters()]
    for kw in ({"n_steps": 0}, {"method": "riemann_left"}):
        with pytest.raises(ValueError):
            integrated_gradients(model, _inputs(), 0, **kw)
    assert flags == [p.requires_grad for p in model.parameters()]
    assert all(t._ig_src is None for t in model.modules() if isinstance(t, M.sNet))
    assert not model.training


# ---------------------------------------------------------------------------------------------------------------
# the factorisation in float64 (no kernels): block 1 = Conv3d(1,C,3,p1) + BatchNorm3d(eval) + LeakyReLU + MaxPool3d(2)
# ---------------------------------------------------------------------------------------------------------------
def _block1(x, p, slope):
    y = F.conv3d(x, p["w"], p["b"], padding=1)
    z = F.batch_norm(y, p["mean"], p["var"], p["gamma"], p["beta"], training=False, eps=1e-5)
    return F.max_pool3d(F.leaky_relu(z, slope), 2)


def _fold(p):
    scale = p["gamma"] / torch.sqrt(p["var"] + 1e-5)
    return p["w"] * scale.view(-1, 1, 1, 1, 1), (p["b"] - p["mean"]) * scale + p["beta"]


def _params(C, seed):
    g = torch.Generator().manual_seed(seed)
    p = {"w": torch.randn(C, 1, 3, 3, 3, generator=g), "b": torch.randn(C, generator=g) * 0.3,
         "gamma": torch.randn(C, generator=g), "beta": torch.randn(C, generator=g) * 0.3,
         "mean": torch.randn(C, generator=g) * 0.2, "var": torch.rand(C, generator=g) + 0.5}
    p["gamma"][:C // 2] = -p["gamma"][:C // 2].abs()                # negative BatchNorm scales fold a sign into W'
    return {k: v.double() for k, v in p.items()}


@pytest.mark.parametrize("slope", [0.0, 0.01])
@pytest.mark.parametrize("method", ["gausslegendre", "riemann_middle"])
def test_block1_factorisation_in_float64(slope, method):
    C, B, D, H, W = 8, 2, 7, 8, 6                                     # odd extent: the last plane lies outside every window
    p = _params(C, seed=3)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, 1, D, H, W, generator=g).double()
    R1 = torch.randn(B, C, D // 2, H // 2, W // 2, generator=g).double()
    R2 = torch.randn(B, C, D // 2, H // 2, W // 2, generator=g).double()
    head = lambda a: (torch.tanh(a * R1) * R2).sum()                  # any downstream objective: g_k changes with alpha
    Wf, bf = _fold(p)
    u = F.conv3d(x, Wf, padding=1)                                    # u' = W' * x, no bias
    umax, win = F.max_pool3d(u, 2, return_indices=True)
    alpha, w = ig_path(5, method)
    G = torch.zeros_like(umax)
    plain = torch.zeros_like(x)
    for a, wk in zip(alpha.tolist(), w.tolist()):
        xa = (a * x).requires_grad_(True)
        a1 = _block1(xa, p, slope)
        z = a * umax + bf.view(1, -1, 1, 1, 1)
        assert torch.allclose(a1, F.leaky_relu(z, slope), rtol=1e-12, atol=1e-12)      # forward: winners fixed
        plain += wk * torch.autograd.grad(head(a1), xa)[0]
        a1f = F.leaky_relu(z, slope).requires_grad_(True)
        gk = torch.autograd.grad(head(a1f), a1f)[0]
        G += wk * gk * torch.where(z > 0, torch.ones_like(z), torch.full_like(z, slope))
    routed = F.max_unpool3d(G, win, 2, output_size=u.shape[2:])
    factored = F.conv_transpose3d(routed, Wf, padding=1)
    assert torch.allclose(factored, plain, rtol=1e-10, atol=1e-12 * float(plain.abs().max()))
    assert float((x * factored).abs().sum()) > 0
