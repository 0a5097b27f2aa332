"""CPU: pins oracle/ddm_oracle.py against the golden vectors recorded from the unmodified reference
(tests/golden/make_golden.py)."""
import json
import os

import pytest
import torch

from oracle import ddm_oracle as O
from tests.golden.make_golden import TINY, CIFAR, inputs, checksum


def _load(golden_dir, name):
    return json.load(open(os.path.join(golden_dir, name)))


def _close(a, b, rel=1e-5):
    assert abs(a - b) <= rel * max(1.0, abs(b)), (a, b)


def test_state_dict_layout_matches_reference(golden_dir):
    for name, cfg in (("unet_tiny.json", TINY), ("unet_cifar.json", CIFAR)):
        g = _load(golden_dir, name)
        shapes, _ = O.unet_layout(cfg)
        assert {k: list(v) for k, v in shapes.items()} == g["state_dict_shapes"]
    assert len(_load(golden_dir, "unet_cifar.json")["state_dict_shapes"]) == 829  # SURVEY §8 a-7


def test_tiny_step_matches_reference(golden_dir):
    g = _load(golden_dir, "unet_tiny.json")
    sd = {k: v.requires_grad_(not k.endswith("resample_filter")) for k, v in O.make_state_dict(TINY, 0).items()}
    x, t, noise, aug = inputs(TINY, g["batch"], 1)
    fn = lambda xx, tt, **kw: O.edm_precond_forward(sd, TINY, xx, tt, **kw)
    xn = O.q_sample(x, noise, t)
    c_pred, e_pred = fn(xn, t, augment_labels=aug)
    loss, ls = O.ddm_loss(c_pred, e_pred, x, noise, t)
    _close(loss.item(), g["loss"])
    for got, ref in ((checksum(c_pred), g["c_pred"]), (checksum(e_pred), g["eps_pred"])):
        _close(got["sum"], ref["sum"], 1e-4)
        _close(got["abssum"], ref["abssum"])
        for a, b in zip(got["probes"], ref["probes"]):
            _close(a, b, 1e-4)
    loss.backward()
    for name, ref in g["grad_norms"].items():
        _close(sd[name].grad.double().norm().item(), ref, 1e-4)


def test_tiny_sampler_matches_reference(golden_dir):
    g = _load(golden_dir, "unet_tiny.json")
    ref = torch.load(os.path.join(golden_dir, "sample_tiny.pt"))
    sd = O.make_state_dict(TINY, 0)
    gen = torch.Generator().manual_seed(7)
    x_T = torch.randn(g["batch"], 3, 16, 16, generator=gen, dtype=torch.float64)
    with torch.no_grad():
        img = O.sample_fn_d(lambda xx, tt: O.edm_precond_forward(sd, TINY, xx, tt), x_T, g["sample_steps"])
    assert img.dtype == torch.float64 and img.min() >= 0 and img.max() <= 1
    assert (img - ref).abs().max().item() < 1e-5


def test_cifar_forward_matches_reference(golden_dir):
    g = _load(golden_dir, "unet_cifar.json")
    sd = O.make_state_dict(CIFAR, 0)
    x, t, noise, aug = inputs(CIFAR, g["batch"], 1)
    with torch.no_grad():
        c_pred, e_pred = O.edm_precond_forward(sd, CIFAR, O.q_sample(x, noise, t), t, augment_labels=aug)
        loss, _ = O.ddm_loss(c_pred, e_pred, x, noise, t)
    _close(loss.item(), g["loss"])
    _close(checksum(c_pred)["abssum"], g["c_pred"]["abssum"])
    _close(checksum(e_pred)["abssum"], g["eps_pred"]["abssum"])


# ---------------------------------------------------------------- DDM-const math pinned DIRECTLY to the reference
def _ddm_math(golden_dir):
    return torch.load(os.path.join(golden_dir, "ddm_math.pt"))


def _same(a, b, tol=1e-6):
    a, b = a.double(), b.double()
    assert a.shape == b.shape
    assert (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item()), (a - b).abs().max().item()


def test_oracle_elementwise_math_vs_reference_functions(golden_dir):
    """oracle.q_sample / pred_x0_from_xt / pred_xtms_from_xt vs the unmodified ddm/ddm_const.py:284-303."""
    g = _ddm_math(golden_dir)
    x, t, noise, s = g["x"], g["t"], g["noise"], g["s"]
    xt = O.q_sample(x, noise, t)
    _same(xt, g["q_sample"], 0)  # same torch expression -> bit-exact
    _same(O.pred_x0_from_xt(xt, noise, -x, t), g["pred_x0_from_xt"], 0)
    _same(O.pred_xtms_from_xt(xt, noise, -x, t, s, g["pred_xtms_z"]), g["pred_xtms_from_xt"], 0)


@pytest.mark.parametrize("weighting", [True, False])
@pytest.mark.parametrize("use_l1", [False, True])
def test_oracle_p_losses_vs_reference_p_losses(golden_dir, weighting, use_l1):
    """oracle.p_losses vs DDPM.p_losses (ddm_const.py:305-364) on the noise the reference itself drew."""
    from tests.golden.make_golden_ddm import toy_model
    g = _ddm_math(golden_dir)
    ref = g[f"p_losses_w{int(weighting)}_l1{int(use_l1)}"]
    loss, ld = O.p_losses(toy_model, g["x"], g["t"], ref["noise"], weighting=weighting, use_l1=use_l1)
    _close(loss.item(), ref["loss"].item(), 1e-6)
    for k in ("train/loss_simple", "train/loss_vlb", "train/loss"):
        _close(float(ld[k]), float(ref[k]), 1e-6)


@pytest.mark.parametrize("n", [2, 5, 10])
def test_oracle_samplers_vs_reference_samplers(golden_dir, n):
    """oracle.sample_fn_d / sample_fn_s vs ddm_const.py:425-476 / :381-422 with the reference's own random draws."""
    from tests.golden.make_golden_ddm import toy_model
    g = _ddm_math(golden_dir)
    d = g[f"sample_fn_d_{n}"]
    img = O.sample_fn_d(toy_model, d["x_T"], n)
    assert img.dtype == torch.float64
    _same(img, d["img"], 1e-12)
    s = g[f"sample_fn_s_{n}"]
    img = O.sample_fn_s(toy_model, s["x_T"], list(s["z"]), n)
    _same(img, s["img"], 1e-5)


@pytest.mark.parametrize("use_l1", [False, True])
def test_oracle_latent_loss_const2_variant_vs_reference(golden_dir, use_l1):
    """oracle.p_losses_latent(variant='const_2') vs the sibling LatentDiffusion.p_losses (ddm_const_2.py:527-588)."""
    from tests.golden.make_golden_ddm import toy_model
    g = _ddm_math(golden_dir)
    ref = g[f"latent2_p_losses_l1{int(use_l1)}"]
    loss, ld = O.p_losses_latent(toy_model, g["x"], g["t"], ref["noise"], use_l1=use_l1, variant="const_2")
    _close(loss.item(), ref["loss"].item(), 1e-6)
    _close(float(ld["train/loss_vlb"]), float(ref["train/loss_vlb"]), 1e-6)


def test_const2_plumbing_crosscheck(golden_dir):
    """The importable sibling class reproduced the restated step exactly when given its three formulas."""
    g = _load(golden_dir, "const2_step.json")
    _close(g["loss_restated"], g["loss_ref"], 1e-6)
    _close(g["loss_dict"]["train/loss"], g["loss_ref"] / (4 * 3 * 16 * 16), 1e-5)


def test_t_steps():
    ts = O.t_steps_deterministic(10)
    assert ts.shape == (11,) and ts[0] == 1.0 and ts[-1] == 0.0
    assert abs(ts[-2].item() - 1e-4) < 1e-12  # sigma_min ** 2 (ddm_const.py:429)
    assert abs(ts[1].item() - (1 + (1e-4 - 1) / 9)) < 1e-12
    assert O.t_steps_deterministic(1).tolist() == [1.0, 0.0]  # documented deviation from the reference's NaN


@pytest.mark.parametrize("name", ["ddpmpp", "ncsnpp"])
def test_oracle_song_unet_vs_reference_golden(golden_dir, name):
    """oracle.song_precond_forward (EDMPrecond + SongUNet, uncond_unet.py:253-441) against D_x / D_y and parameter
    gradients recorded from the unmodified reference (make_golden_song.py), DDPM++ and NCSN++ flavours, CPU fp32."""
    from tests.golden.make_golden_song import CONFIGS, inputs, state_dict_for
    g = torch.load(os.path.join(golden_dir, "song_unet.pt"))[name]
    cfg = O.song_config(**CONFIGS[name])
    sd = {k: v.requires_grad_(True) for k, v in state_dict_for(g["keys"]).items()}
    x, t, aug, g1, g2 = inputs()
    d_x, d_y = O.song_precond_forward(sd, cfg, x, t, aug if cfg["augment_dim"] else None)
    assert torch.allclose(d_x, g["d_x"], rtol=1e-4, atol=1e-4) and torch.allclose(d_y, g["d_y"], rtol=1e-4, atol=1e-4)
    ((d_x * g1).sum() + (d_y * g2).sum()).backward()
    for k, ref in g["grads"].items():
        assert torch.allclose(sd[k].grad, ref, rtol=1e-3, atol=1e-4 * float(ref.abs().max()) + 1e-6), k
    for k, n in g["grad_norms"].items():
        assert abs(float(sd[k].grad.norm()) - n) <= 1e-3 * n + 1e-6, k


# ---------------------------------------------------------------- relation layer of the conditional UNet (row f-3)
from oracle import relation_oracle as R  # noqa: E402


def _relation_golden(golden_dir):
    from tests.golden.make_golden_relation import load
    return load(golden_dir)


@pytest.mark.parametrize("commute", [False, True])
def test_relation_layer_oracle_matches_reference(golden_dir, commute):
    """oracle.relation_layer (cond_unet.py:192-252) against the unmodified reference module's output and gradients
    (tests/golden/make_golden_relation.py) — in the reference's op order, and with out_conv applied to the pooled tokens
    before the bilinear resize (the order the fused sm_100a path uses): the same linear map."""
    for name, g in _relation_golden(golden_dir).items():
        spec = g["spec"]
        x1, x2 = g["x1"].clone().requires_grad_(True), g["x2"].clone().requires_grad_(True)
        sd = {k: v.clone().requires_grad_(True) for k, v in g["state_dict"].items()}
        out = R.relation_layer(sd, x1, x2, spec["nhead"], spec["window_size1"], spec["window_size2"],
                               commute_out_conv=commute)
        assert torch.allclose(out, g["out"], rtol=1e-4, atol=2e-5), (name, (out - g["out"]).abs().max())
        (out * g["probe"]).sum().backward()
        for key, got, ref in ([("x1", x1.grad, g["dx1"]), ("x2", x2.grad, g["dx2"])]
                              + [(k, sd[k].grad, g["grads"][k]) for k in g["grads"]]):
            # k_lin.bias shifts every logit of a query by the same amount, so its gradient is exactly zero in real
            # arithmetic and rounding noise (1e-5) in both implementations: hence the absolute floor
            assert (got - ref).norm() <= 2e-4 * ref.norm() + 2e-4, (name, key, (got - ref).norm(), ref.norm())


def test_relation_kernel_algorithms_match_autograd():
    """The algorithms of csrc/relation_ops.cu restated on the CPU (fp64) against torch: separable transposed resize,
    zero-padded window pool, and the closed-form backward of GroupNorm(x + y) + resize(z)."""
    import torch.nn.functional as F
    torch.manual_seed(4)
    for (h, w, ho, wo) in [(4, 4, 16, 16), (3, 5, 24, 40), (16, 16, 16, 16), (20, 12, 7, 5), (1, 1, 9, 9)]:
        x = torch.randn(2, h, w, 8, dtype=torch.float64, requires_grad=True)
        ref = F.interpolate(x.permute(0, 3, 1, 2), size=(ho, wo), mode="bilinear", align_corners=True).permute(0, 2, 3, 1)
        assert torch.allclose(R.bilinear_fwd(x.detach(), (ho, wo)), ref, atol=1e-5)  # fp32 coordinates, as ATen
        dy = torch.randn_like(ref)
        ref.backward(dy)
        assert torch.allclose(R.bilinear_bwd_separable(dy, (h, w)), x.grad, atol=1e-4)
    for (h, w, win) in [(32, 32, (8, 8)), (10, 7, (4, 4)), (9, 9, (2, 4))]:
        x = torch.randn(2, h, w, 8, dtype=torch.float64)
        ph, pw = (-h) % win[0], (-w) % win[1]
        ref = F.avg_pool2d(F.pad(x.permute(0, 3, 1, 2), (0, pw, 0, ph)), win).permute(0, 2, 3, 1)
        assert torch.allclose(R.window_pool(x, win), ref, atol=1e-12)
    b, h, w, c, G = 2, 12, 10, 32, 8
    x, y = (torch.randn(b, h, w, c, dtype=torch.float64, requires_grad=True) for _ in range(2))
    z = torch.randn(b, 3, 5, c, dtype=torch.float64)
    gamma = (torch.rand(c, dtype=torch.float64) + 0.5).requires_grad_(True)
    beta = torch.randn(c, dtype=torch.float64, requires_grad=True)
    ref = (F.group_norm((x + y).permute(0, 3, 1, 2), G, gamma, beta, 1e-5)
           + F.interpolate(z.permute(0, 3, 1, 2), size=(h, w), mode="bilinear", align_corners=True)).permute(0, 2, 3, 1)
    out, _, _ = R.relation_tail(x.detach(), y.detach(), z, gamma.detach(), beta.detach(), G)
    assert torch.allclose(out, ref, atol=1e-5)
    dout = torch.randn_like(ref)
    ref.backward(dout)
    dpre, dgamma, dbeta = R.relation_tail_bwd(dout, x.detach(), y.detach(), gamma.detach(), G)
    assert torch.allclose(dpre, x.grad, atol=1e-9) and torch.allclose(dpre, y.grad, atol=1e-9)
    assert torch.allclose(dgamma, gamma.grad, atol=1e-9) and torch.allclose(dbeta, beta.grad, atol=1e-9)
