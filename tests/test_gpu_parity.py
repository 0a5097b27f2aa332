"""GPU (B200): parity of the CUDA path, called through the C-ABI, against the oracle / golden vectors.

Tolerances (north_star): bf16 mode — loss within 1e-2 relative, per-parameter gradient cosine >= 0.999, fixed-seed
samples PSNR >= 40 dB against the reference trajectory.  Elementwise fp32/fp64 kernels: 1e-5 relative or bit-exact.
GEMM-engine results with fp32 output: 1e-5 relative against an fp32 matmul of the same bf16-rounded inputs.
"""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module", autouse=True)
def _need_gpu_and_lib():
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from adm_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "libadm_b200.so missing: the CUDA path must be built (no fallback)"
    yield
    assert _lib.load().adm_device_error() == 0
    assert _lib.load().adm_launch_count() > 0, "no adm_b200 kernel was launched"


# ---------------------------------------------------------------- kernels vs torch on the same inputs
from tests.gpu_checks import check_kernels as CK  # noqa: E402
from tests.gpu_checks import check_unet as CU  # noqa: E402


@pytest.mark.parametrize("case", ["gemm_nt_basic", "gemm_nn_tn", "conv_fprop_3x3", "conv_fprop_concat_1x1",
                                  "conv_dgrad_wgrad", "conv_dgrad_shadow", "conv_large_kernels", "row_maps",
                                  "elementwise"])
def test_gemm_engine_and_ddm_kernels(case):
    assert CK.CASES[case]()


def test_ddm_kernels_vs_reference_functions():
    """K1/K2/K3 (both samplers) against outputs of the unmodified ddm/ddm_const.py functions (tests/golden/ddm_math.pt)."""
    assert CK.CASES["ddm_math_vs_reference"]()


def test_stochastic_sampler_vs_oracle():
    assert CU.CASES["stochastic_sampler"]()


def test_benchmark_configuration_b128_step_vs_oracle():
    assert CU.CASES["unet_cifar_b128"]()


def test_training_mode_dropout_masks_vs_oracle():
    assert CU.CASES["unet_dropout_on"]()


@pytest.mark.parametrize("case", ["groupnorm", "conv_splitk", "small_ops", "attention", "spatial_att"])
def test_norm_attention_kernels(case):
    assert CU.CASES[case]()


# ---------------------------------------------------------------- whole hot path vs oracle / golden
def test_unet_tiny_step_and_sampler_vs_oracle_and_golden():
    assert CU.CASES["unet_tiny"]()


def test_unet_cifar_config_step_vs_oracle():
    assert CU.CASES["unet_cifar"]()


def test_cifar_forward_matches_reference_golden(golden_dir):
    """Same seeded inputs as tests/golden/make_golden.py (recorded from the unmodified reference UNet)."""
    from oracle import ddm_oracle as O
    from tests.golden.make_golden import CIFAR, inputs
    from adm_b200.ddm.ddm_const import DDPM
    g = json.load(open(os.path.join(golden_dir, "unet_cifar.json")))
    net = CU_build(CIFAR)
    cfg = dict(image_size=[32, 32], sampling_timesteps=10, eps=1e-4, sigma_max=1, sigma_min=0.01, weighting_loss=True)
    dpm = DDPM(model=net, cfg=cfg, **cfg).cuda()
    x, t, noise, aug = (a.cuda() for a in inputs(CIFAR, g["batch"], 1))
    with torch.no_grad():
        loss, ld = dpm.p_losses(x, t, noise=noise, augment_labels=aug)
    assert abs(loss.item() - g["loss"]) / g["loss"] < 1e-2
    assert abs(ld["train/loss"].item() - g["loss"] / (g["batch"] * 3 * 32 * 32)) / (g["loss"] / 6144) < 1e-2


def CU_build(cfg, seed=0):
    from oracle import ddm_oracle as O
    from adm_b200.unet.uncond_unet import EDMPrecond
    kw = {k: v for k, v in cfg.items() if k not in ("img_resolution", "img_channels", "label_dim")}
    net = EDMPrecond(img_resolution=cfg["img_resolution"], img_channels=3, sigma_data=1.0, model_type="DhariwalUNet", **kw)
    net.load_state_dict(O.make_state_dict(cfg, seed), strict=True)
    return net.cuda().eval()


# ---------------------------------------------------------------- size-independent properties at larger sizes
def test_gradient_is_linear_over_the_batch():
    """DP semantics: the gradient of a batch equals the mean of its shards' gradients (what the all-reduce computes)."""
    from tests.golden.make_golden import TINY, inputs
    from adm_b200.ddm.ddm_const import DDPM
    cfg = dict(image_size=[16, 16], sampling_timesteps=3, eps=1e-4, weighting_loss=True)
    x, t, noise, aug = (a.cuda() for a in inputs(TINY, 32, 5))

    def grads(sl):
        net = CU_build(TINY)
        dpm = DDPM(model=net, cfg=cfg, **cfg).cuda()
        loss, _ = dpm.p_losses(x[sl], t[sl], noise=noise[sl], augment_labels=aug[sl])
        loss.backward()
        return torch.cat([p.grad.flatten() for p in net.parameters()]), loss.item()

    g_all, l_all = grads(slice(0, 32))
    g_a, l_a = grads(slice(0, 16))
    g_b, l_b = grads(slice(16, 32))
    g_mean = 0.5 * (g_a + g_b)
    cos = torch.dot(g_all, g_mean) / (g_all.norm() * g_mean.norm())
    # bf16 compute: the batch of 32 and its halves run different tilings (tile width, K split), i.e. different fp32
    # summation orders before each bf16 rounding; 1e-3 is a tenth of the north-star loss tolerance for bf16 (1e-2)
    assert abs(l_all - 0.5 * (l_a + l_b)) / l_all < 1e-3
    assert cos.item() > 0.9995 and abs(g_all.norm().item() / g_mean.norm().item() - 1) < 2e-2


def test_step_is_repeatable_and_dropout_changes_it():
    from tests.golden.make_golden import TINY, inputs
    from adm_b200.ddm.ddm_const import DDPM
    cfg = dict(image_size=[16, 16], sampling_timesteps=3, eps=1e-4, weighting_loss=True)
    x, t, noise, aug = (a.cuda() for a in inputs(TINY, 8, 2))
    net = CU_build(TINY)
    dpm = DDPM(model=net, cfg=cfg, **cfg).cuda()
    with torch.no_grad():
        l1, _ = dpm.p_losses(x, t, noise=noise)
        l2, _ = dpm.p_losses(x, t, noise=noise)
    assert abs(l1.item() - l2.item()) / l1.item() < 1e-3  # fp32 atomics in the GroupNorm statistics reorder sums
    for m in net.modules():
        if hasattr(m, "dropout"):
            m.dropout = 0.5
    net.train()
    with torch.no_grad():
        l3, _ = dpm.p_losses(x, t, noise=noise)
        c3, e3 = net(x, t)
        c4, e4 = net(x, t)
    net.eval()
    with torch.no_grad():
        c1, e1 = net(x, t)
        c2, e2 = net(x, t)
    rel = lambda a, b: abs(a.item() - b.item()) / abs(b.item())
    dist = lambda a, b: ((a.float() - b.float()).norm() / b.float().norm()).item()
    assert rel(l3, l1) > 5e-3  # dropout active
    # fresh masks per call: two training-mode forwards differ element-wise by far more than two evaluation-mode forwards
    # (a scalar loss averages ~10^5 independent mask elements and hides the difference)
    noise = max(dist(c1, c2), dist(e1, e2))  # small batches: fp32 atomics reorder the GroupNorm sums, bf16 roundings flip
    assert noise < 2e-2
    assert min(dist(c3, c4), dist(e3, e4)) > max(10 * noise, 5e-2)


def test_sampler_full_size_properties():
    """CIFAR config, batch 64, 10 steps: output is a valid image batch, deterministic in x_T, and sharding the batch
    (the multi-GPU sampling scheme) reproduces the unsharded result."""
    from tests.golden.make_golden import CIFAR
    from adm_b200.ddm.ddm_const import DDPM
    net = CU_build(CIFAR)
    cfg = dict(image_size=[32, 32], sampling_timesteps=10, eps=1e-4, sigma_max=1, sigma_min=0.01)
    dpm = DDPM(model=net, cfg=cfg, **cfg).cuda()
    g = torch.Generator().manual_seed(3)
    x_T = torch.randn(64, 3, 32, 32, generator=g, dtype=torch.float64).cuda()
    img = dpm.sample(batch_size=64, x_T=x_T)
    assert img.shape == (64, 3, 32, 32) and img.dtype == torch.float64
    assert float(img.min()) >= 0.0 and float(img.max()) <= 1.0 and torch.isfinite(img).all()
    shard = torch.cat([dpm.sample(batch_size=32, x_T=x_T[:32]), dpm.sample(batch_size=32, x_T=x_T[32:])])
    mse = ((img - shard) ** 2).mean().item()
    assert mse < 1e-4  # PSNR >= 40 dB between sharded and unsharded sampling


def test_fused_optimizer_step_matches_torch_adamw():
    from tests.golden.make_golden import TINY, inputs
    from adm_b200.ddm.ddm_const import DDPM
    from adm_b200.train import TrainStep
    cfg = dict(image_size=[16, 16], sampling_timesteps=3, eps=1e-4, weighting_loss=True)
    x, t, noise, aug = (a.cuda() for a in inputs(TINY, 8, 4))
    net = CU_build(TINY)
    dpm = DDPM(model=net, cfg=cfg, **cfg).cuda()
    ref = {k: v.clone() for k, v in net.state_dict().items()}
    step = TrainStep(dpm, lr=1e-3, weight_decay=1e-2, max_grad_norm=1.0)
    step.micro_step(x, t, noise)
    grads = {n: p.grad.clone() for n, p in net.named_parameters()}
    step.optimizer_step()
    # torch reference update on the same gradients
    ps = {n: torch.nn.Parameter(ref[n].clone()) for n, _ in net.named_parameters()}
    for n, p in ps.items():
        p.grad = grads[n].clone()
    torch.nn.utils.clip_grad_norm_(list(ps.values()), 1.0)
    torch.optim.AdamW(list(ps.values()), lr=1e-3, weight_decay=1e-2).step()
    for n, p in net.named_parameters():
        assert torch.allclose(p.detach(), ps[n].detach(), rtol=1e-5, atol=1e-7), n
    assert float(step.arena.grads.abs().max()) == 0.0  # gradients are cleared for the next step


def test_arena_fast_path_matches_plain_backward():
    """TrainStep stores conv weights channels-last with a bf16 shadow and lets wgrad / the grouped affine GEMM write
    straight into the gradient arena; the gradients must equal those of the plain (re-pack / un-pack) path, and after
    an optimizer step the shadow must equal the bf16 rounding of the fp32 masters."""
    from tests.golden.make_golden import TINY, inputs
    from adm_b200.ddm.ddm_const import DDPM
    from adm_b200.train import TrainStep
    cfg = dict(image_size=[16, 16], sampling_timesteps=3, eps=1e-4, weighting_loss=True)
    x, t, noise, aug = (a.cuda() for a in inputs(TINY, 16, 7))
    net_a = CU_build(TINY)
    dpm_a = DDPM(model=net_a, cfg=cfg, **cfg).cuda()
    loss_a, _ = dpm_a.p_losses(x, t, noise=noise, augment_labels=aug)
    loss_a.backward()
    ga = {n: p.grad.clone() for n, p in net_a.named_parameters()}
    net_b = CU_build(TINY)
    dpm_b = DDPM(model=net_b, cfg=cfg, **cfg).cuda()
    step = TrainStep(dpm_b, lr=1e-3)
    packed = [n for n, p in net_b.named_parameters() if getattr(p, "_adm_pack", None) is not None]
    assert len(packed) > 10 and step.engine.affine_pack is not None
    assert not net_b.state_dict()[packed[0]].is_contiguous()  # channels-last storage behind the reference shape
    loss_b = step.micro_step(x, t, noise, augment_labels=aug)
    assert abs(loss_a.item() - loss_b.item()) / abs(loss_a.item()) < 1e-5
    # The two paths share every kernel except the data gradient (the arena path runs it through the fprop kernels on the
    # transposed weight shadow: another summation order, so bf16 roundings flip here and there).  Single-element tensors
    # (the SpatialAtt 1->1 convs behind a rank-1 softmax at the bottleneck) are noise-limited under such flips and a
    # cosine of two scalars is only a sign: they are judged with the rest of their module, as in check_unet.
    scalars = {}
    for n, p in net_b.named_parameters():
        a, b = ga[n].flatten().double(), p.grad.flatten().double()
        if a.norm().item() < 1e-6:  # mathematically zero gradients (softmax shift invariance of k_conv.bias): noise
            assert b.norm().item() < 1e-6, n
            continue
        if a.numel() == 1:
            scalars.setdefault(n.rsplit(".", 2)[0], []).append(n)
            continue
        cos = torch.dot(a, b) / (a.norm() * b.norm() + 1e-30)
        assert cos.item() > 0.9999 and abs(a.norm().item() / (b.norm().item() + 1e-30) - 1) < 1e-2, n
    grads_b = {n: p.grad for n, p in net_b.named_parameters()}
    for mod in scalars:
        members = [n for n in ga if n.startswith(mod + ".")]
        a = torch.cat([ga[n].flatten().double() for n in members])
        b = torch.cat([grads_b[n].flatten().double() for n in members])
        cos = torch.dot(a, b) / (a.norm() * b.norm() + 1e-30)
        assert cos.item() > 0.999 and abs(a.norm().item() / (b.norm().item() + 1e-30) - 1) < 2e-2, mod
    step.optimizer_step()
    torch.cuda.synchronize()
    assert torch.equal(step.arena.shadow, step.arena.flat.bfloat16())
    # state_dict round trip through the reference layout
    sd = {k: v.clone() for k, v in net_b.state_dict().items()}
    net_c = CU_build(TINY, seed=3)
    net_c.load_state_dict(sd)
    for k, v in net_c.state_dict().items():
        assert torch.equal(v, sd[k]), k
    # out-of-band writes are picked up: load into the arena-resident model, shadow follows via the version check
    net_b.load_state_dict(CU_build(TINY, seed=3).state_dict())
    with torch.no_grad():
        l1, _ = dpm_b.p_losses(x, t, noise=noise, augment_labels=aug)
        l2, _ = DDPM(model=CU_build(TINY, seed=3), cfg=cfg, **cfg).cuda().p_losses(x, t, noise=noise, augment_labels=aug)
    assert abs(l1.item() - l2.item()) / abs(l2.item()) < 1e-4


# ---------------------------------------------------------------- conditional UNet / LatentDiffusion (SURVEY §8 a-15..a-19)
from tests.gpu_checks import check_cond as CC  # noqa: E402


@pytest.mark.parametrize("case", ["ws_pack", "channel_layernorm", "linear_attention", "attention_padded_heads",
                                  "resnet_block", "relation_tail", "resize_and_pool", "relation_layer_golden"])
def test_cond_unet_kernels(case):
    """K11 weight-standardise+pack, K12 fused LinearAttention, padded-head Attention, ResnetBlock fwd/bwd vs torch."""
    assert CC.CASES[case]()


def test_cond_unet_and_latent_diffusion_vs_reference_golden():
    """Whole cond Unet (outputs, latent DDM loss, per-parameter gradients, 3-step latent sampler) against vectors recorded
    from the unmodified reference unet.cond_unet.Unet (tests/golden/make_golden_cond.py)."""
    assert CC.CASES["cond_unet_golden"]()


def test_segmented_graph_step_matches_eager_step():
    """The multi-rank launch structure (a chain of CUDA graphs cut at the gradient-bucket boundaries, all-reduces
    launched between replays) on one GPU: three replayed steps must produce the parameters of three eager steps
    (same x, t, noise; dropout is 0 in this config, so only the fp32 atomics' summation order differs)."""
    from tests.golden.make_golden import TINY, inputs
    from adm_b200.ddm.ddm_const import DDPM
    from adm_b200.train import TrainStep
    cfg = dict(image_size=[16, 16], sampling_timesteps=3, eps=1e-4, weighting_loss=True)
    x, t, noise, _ = (a.cuda() for a in inputs(TINY, 16, 8))

    def run(mode):
        net = CU_build(TINY)
        net.train()
        dpm = DDPM(model=net, cfg=cfg, **cfg).cuda()
        step = TrainStep(dpm, lr=1e-3, bucket_mb=2)
        start = step.arena.flat.clone()
        if mode == "segments":
            segs = step.capture_dp(x, warmup=1, t=t, noise=noise)  # one eager warm-up step, then capture
            assert len(segs) >= 4  # several bucket cuts + the optimizer graph
            for _ in range(3):
                loss = step.replay(x)
        else:
            for _ in range(4):
                loss = step.micro_step(x, t, noise)
                step.optimizer_step()
        assert step.step_count == 4
        torch.cuda.synchronize()
        return start, step.arena.flat.clone(), float(loss)

    s0, p_eager, l_eager = run("eager")
    _, p_seg, l_seg = run("segments")
    assert abs(l_seg - l_eager) / l_eager < 1e-3
    upd_e, upd_s = p_eager - s0, p_seg - s0
    cos = torch.dot(upd_e, upd_s) / (upd_e.norm() * upd_s.norm())
    assert cos.item() > 0.999 and abs(upd_s.norm().item() / upd_e.norm().item() - 1) < 1e-2


@pytest.mark.parametrize("steps", [1, 50])
def test_sampler_step_count_sweep_vs_oracle(steps):
    """BASELINE config 3 sweeps sampling_timesteps over 1 / 10 / 50.  N = 1 is NaN in the reference (0/0 in t_steps,
    SURVEY §7-8); both the product and the oracle define it as t_steps = [sigma_max, 0].  PSNR >= 40 dB against the
    oracle's fp64 trajectory on the same weights and x_T; the whole N-step loop replays as one CUDA graph."""
    from oracle import ddm_oracle as O
    from tests.golden.make_golden import TINY
    from adm_b200.ddm.ddm_const import DDPM
    net = CU_build(TINY)
    cfg = dict(image_size=[16, 16], sampling_timesteps=steps, eps=1e-4, sigma_max=1, sigma_min=0.01)
    dpm = DDPM(model=net, cfg=cfg, **cfg).cuda()
    g = torch.Generator().manual_seed(21)
    x_T = torch.randn(4, 3, 16, 16, generator=g, dtype=torch.float64)
    img = dpm.sample(batch_size=4, x_T=x_T.cuda())
    img2 = dpm.sample(batch_size=4, x_T=x_T.cuda())  # second call replays the captured graph
    # not bit-equal: at batch 4 the multi-block GroupNorm statistics use fp32 atomics (summation order varies)
    # (a random-weight net amplifies that over 50 steps; both replays stay within the PSNR bar of each other)
    assert ((img - img2) ** 2).mean().item() < 1e-4 and img.dtype == torch.float64
    assert float(img.min()) >= 0.0 and float(img.max()) <= 1.0
    sd = O.make_state_dict(TINY, 0)
    ref = O.sample_fn_d(lambda xx, tt: O.edm_precond_forward(sd, TINY, xx, tt), x_T, steps)
    mse = ((img.cpu() - ref) ** 2).mean().item()
    assert 10 * torch.log10(torch.tensor(1.0 / max(mse, 1e-20))).item() >= 40.0


# ---------------------------------------------------------------- CelebAHQ-latent family (BASELINE config 4)
def test_unet_celebahq_family_vs_oracle():
    """model_channels 96, mult 1-2-3 (channels 96 / 192 / 288: not multiples of 64; heads of width 64 and 72) against
    the oracle: loss 1e-2, every parameter's gradient cosine >= 0.999."""
    assert CU.CASES["unet_celeb_small"]()


def test_unet_celebahq_full_config_runs():
    """configs/celebahq/celeb_uncond_ddm_const_uncond_unet_ldm.yaml UNet at full size (64x64 latent, 121 M parameters,
    attention over 1024 and 256 pixels): one latent training step and a 2-step latent sample, finite and in range."""
    from adm_b200.ddm.ddm_const import LatentDiffusion
    from adm_b200.unet.uncond_unet import EDMPrecond

    class AE(torch.nn.Module):
        down_ratio = 4

        def encode(self, x):
            return torch.nn.functional.avg_pool2d(x, 4)

        def decode(self, z):
            return torch.nn.functional.interpolate(z, scale_factor=4)

    torch.manual_seed(0)
    net = EDMPrecond(img_resolution=64, img_channels=3, sigma_data=1.0, model_type="DhariwalUNet", model_channels=96,
                     channel_mult=[1, 2, 3, 4], channel_mult_emb=4, num_blocks=3, attn_resolutions=[32, 16], dropout=0.1,
                     label_dropout=0, augment_dim=0).cuda()
    assert sum(p.numel() for p in net.parameters()) == 121_053_232  # SURVEY section 8a
    cfg = dict(image_size=[256, 256], sampling_timesteps=2, eps=1e-4, sigma_max=1, sigma_min=0.01, weighting_loss=False,
               use_l1=True, scale_factor=0.165, scale_by_std=True, default_scale=True)
    ldm = LatentDiffusion(auto_encoder=AE(), model=net, cfg=cfg, **cfg).cuda()
    x = 2 * torch.rand(2, 3, 256, 256, device="cuda") - 1
    loss, ld = ldm.training_step({"image": x})
    loss.backward()
    assert torch.isfinite(loss) and all(torch.isfinite(p.grad).all() for p in net.parameters() if p.grad is not None)
    img = ldm.sample(batch_size=2)
    assert img.shape == (2, 3, 256, 256) and float(img.min()) >= 0 and float(img.max()) <= 1


# ---------------------------------------------------------------- SongUNet (SURVEY section 8 row f-4)
def test_song_unet_ddm_step_vs_oracle():
    assert CU.CASES["song_unet_ddm_step"]()


@pytest.mark.parametrize("case", ["song_unet_ddpmpp", "song_unet_ncsnpp"])
def test_song_unet_vs_reference_golden(case):
    """EDMPrecond(model_type='SongUNet') — DDPM++ and NCSN++ flavours — forward and backward against vectors recorded from
    the unmodified reference (tests/golden/make_golden_song.py)."""
    assert CU.CASES[case]()


# ---------------------------------------------------------------- AugmentPipe as one kernel (SURVEY section 8 row f-4)
def test_fused_augment_pipe_vs_reference_golden(golden_dir):
    """adm_augment_warp (flips + reflect pad + sym6 upsample + affine bilinear sample + sym6 decimate + crop in ONE kernel,
    one CTA per sample) against the batches recorded from the unmodified reference AugmentPipe (make_golden_augment.py:
    the DDM configuration at p = 0.15 and the same with p = 1 so that every transform fires on every sample), and against
    the in-tree torch-op sequence on the same draws; labels exact, images to float32 round-off."""
    from adm_b200 import _lib
    from adm_b200.ddm.augment import AugmentPipe
    from tests.golden.make_golden_augment import KW, KW_HOT, SEEDS, inputs
    g = torch.load(os.path.join(golden_dir, "augment.pt"))
    for name, kw in (("cfg", KW), ("hot", KW_HOT)):
        for seed in SEEDS:
            pipe = AugmentPipe(**kw)
            x = inputs(seed).cuda()
            assert pipe.fused and pipe.fused_ok(x)
            l0 = _lib.load().adm_launch_count()
            torch.manual_seed(seed)
            y, lab = pipe(x)
            assert _lib.load().adm_launch_count() == l0 + 1  # the whole pipe was one kernel of ours
            ref = g[f"{name}_{seed}"]
            assert torch.equal(lab.cpu(), ref["labels"])
            assert (y.cpu() - ref["images"]).abs().max().item() < 1e-4, (name, seed)
            pipe.fused = False
            torch.manual_seed(seed)
            y2, _ = pipe(x)
            assert (y - y2).abs().max().item() < 1e-4


# ---------------------------------------------------------------- frozen first stage (SURVEY section 8 row f-1)
def test_autoencoder_kl_vs_reference_golden(golden_dir):
    """AutoencoderKL.encode / decode against vectors recorded from the unmodified reference (make_golden_ae.py):
    posterior mean / logvar and the decoded image, plus the encoder.* / decoder.* / quant conv key layout."""
    from tests.golden.make_golden_ae import build_ours, inputs
    g = torch.load(os.path.join(golden_dir, "ae_small.pt"))
    ae = build_ours().cuda()
    assert {k: list(v.shape) for k, v in ae.state_dict().items()} == g["keys"] and ae.down_ratio == 4
    post = ae.encode(inputs().cuda())
    rel = lambda a, b: ((a.float().cpu() - b).norm() / b.norm()).item()
    assert rel(post.mean, g["mean"]) < 2e-2 and rel(post.logvar, g["logvar"]) < 2e-2
    dec = ae.decode(g["mean"].cuda())
    mse = ((dec.float().cpu() - g["dec"]) ** 2).mean().item()
    psnr = 10 * torch.log10(torch.tensor(4.0 / mse)).item()  # images live in [-1, 1]
    assert rel(dec, g["dec"]) < 4e-2 and psnr >= 40.0, (rel(dec, g["dec"]), psnr)
    # plugs into LatentDiffusion as the frozen first stage
    assert post.sample().shape == (2, 3, 16, 16) and not any(p.requires_grad for p in [])


# ---------------------------------------------------------------- Trainer / Sampler shells + EMA (SURVEY section 8 row f-2)
def test_trainer_checkpoint_resume_and_ema_sampling(tmp_path):
    from tests.golden.make_golden import TINY
    from adm_b200.ddm.ddm_const import DDPM
    from adm_b200.trainer import Sampler, Trainer
    cfg = dict(image_size=[16, 16], sampling_timesteps=3, eps=1e-4, weighting_loss=True)
    tcfg = {"trainer": {"warmup_iter": 4, "min_lr": 1e-6, "ema_update_after_step": 2, "ema_update_every": 2}}

    def loader():
        g = torch.Generator().manual_seed(0)
        while True:
            yield {"image": 2 * torch.rand(8, 3, 16, 16, generator=g) - 1}

    def make(resume=0):
        dpm = DDPM(model=CU_build(TINY), cfg=cfg, **cfg).cuda()
        return Trainer(dpm, loader(), train_batch_size=8, gradient_accumulate_every=2, train_lr=1e-3,
                       train_num_steps=6, save_and_sample_every=3, num_samples=4, results_folder=str(tmp_path),
                       log_freq=100, resume_milestone=resume, cfg=tcfg)

    tr = make()
    tr.train()
    assert tr.step == 6 and torch.isfinite(tr.last_loss) and (tmp_path / "model-2.pt").exists()
    ck = torch.load(tmp_path / "model-2.pt", map_location="cpu", weights_only=False)
    assert set(ck) == {"step", "model", "opt", "lr_scheduler", "ema", "scaler"} and ck["step"] == 6
    assert any(k.startswith("ema_model.model.") for k in ck["ema"]) and "model.model.map_layer0.weight" in ck["model"]
    # resume: parameters, step and optimizer moments come back
    tr2 = make(resume=2)
    assert tr2.step == 6 and tr2.step_fn.step_count == tr.step_fn.step_count
    for (n, a), (_, b) in zip(tr.model.named_parameters(), tr2.model.named_parameters()):
        assert torch.equal(a, b), n
    assert torch.equal(tr.step_fn.m, tr2.step_fn.m)
    # the EMA copy differs from the online weights and samples through its own engine caches
    d = sum(float((a - b).abs().sum()) for a, b in zip(tr.ema.ema_model.parameters(), tr.model.parameters()))
    assert d > 0
    img = Sampler(DDPM(model=CU_build(TINY), cfg=cfg, **cfg).cuda(), batch_size=4, sample_num=6,
                  ckpt_path=str(tmp_path / "model-2.pt"), use_ema=True).sample()
    assert img.shape == (6, 3, 16, 16) and float(img.min()) >= 0 and float(img.max()) <= 1
