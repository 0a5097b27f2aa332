"""CPU: host-side logic of the drop-in mirror — state_dict layout, config -> object resolution, samplers' time grid,
parameter arena / gradient-completion order."""
import json
import os

import pytest
import torch

from oracle import ddm_oracle as O
from tests.golden.make_golden import CIFAR, TINY

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _net(cfg):
    from adm_b200.unet.uncond_unet import EDMPrecond
    kw = {k: v for k, v in cfg.items() if k not in ("img_resolution", "img_channels", "label_dim")}
    return EDMPrecond(img_resolution=cfg["img_resolution"], img_channels=3, sigma_data=1.0, model_type="DhariwalUNet", **kw)


@pytest.mark.parametrize("name,cfg", [("unet_tiny.json", TINY), ("unet_cifar.json", CIFAR)])
def test_state_dict_layout_equals_reference(golden_dir, name, cfg):
    ref = json.load(open(os.path.join(golden_dir, name)))["state_dict_shapes"]
    ours = {k: list(v.shape) for k, v in _net(cfg).state_dict().items()}
    assert ours == ref
    assert list(ours) == list(ref)  # same key ORDER as the reference module (checkpoint round trips)


def test_load_reference_style_state_dict_and_attributes():
    net = _net(TINY)
    sd = O.make_state_dict(TINY, 3)
    missing, unexpected = net.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    assert torch.equal(net.model.enc["16x16_conv"].weight, sd["model.enc.16x16_conv.weight"])
    assert net.channels == 3 and net.self_condition is None and net.img_resolution == 16


def test_construct_by_reference_class_names():
    from adm_b200.ddm.utils import construct_class_by_name
    from adm_b200.unet.uncond_unet import EDMPrecond
    from adm_b200.ddm.ddm_const import DDPM
    unet_cfg = dict(class_name="unet.uncond_unet.EDMPrecond", img_resolution=16, img_channels=3, sigma_data=1.0,
                    model_type="DhariwalUNet", model_channels=64, channel_mult=[1, 2], channel_mult_emb=4, num_blocks=1,
                    attn_resolutions=[8], dropout=0.1, label_dropout=0, augment_dim=9)
    unet = construct_class_by_name(**unet_cfg)
    assert isinstance(unet, EDMPrecond)
    model_cfg = dict(class_name="ddm.ddm_const.DDPM", image_size=[16, 16], ckpt_path=None, ignore_keys=[],
                     only_model=False, sampling_timesteps=10, loss_type="l2", start_dist="normal", perceptual_weight=1.0,
                     eps=1e-4, sigma_max=1, sigma_min=0.01, ldm=False, weighting_loss=True, use_l1=False,
                     use_augment=False, unet=unet_cfg)
    dpm = construct_class_by_name(model=unet, cfg=model_cfg, **model_cfg)  # train_uncond_dpm.py:44-46
    assert isinstance(dpm, DDPM)
    assert dpm.image_size == [16, 16] and dpm.sampling_timesteps == 10 and dpm.weighting_loss
    assert "eps" in dpm.state_dict() and len(dpm.state_dict()) == 1 + len(unet.state_dict())
    with pytest.raises(AssertionError):
        construct_class_by_name(model=unet, cfg=model_cfg, **{**model_cfg, "start_dist": "laplace"})


def test_reference_yaml_builds_our_classes():
    """The CIFAR-10 model section (configs/cifar10/... keeps the reference's hyper-parameters) under the reference's own
    dotted class names builds this package's classes at the reference's size."""
    import yaml
    from adm_b200.ddm.utils import construct_class_by_name
    cfg = yaml.load(open(os.path.join(ROOT, "configs/cifar10/ddm_uncond_const_uncond_unet.yaml")), Loader=yaml.FullLoader)
    model_cfg = cfg["model"]
    model_cfg["class_name"] = "ddm.ddm_const.DDPM"
    model_cfg["unet"]["class_name"] = "unet.uncond_unet.EDMPrecond"
    model_cfg["use_augment"] = False  # AugmentPipe is host-side data glue (SURVEY 8 f-4)
    unet = construct_class_by_name(**model_cfg["unet"])
    dpm = construct_class_by_name(model=unet, cfg=model_cfg, **model_cfg)
    assert sum(p.numel() for p in unet.parameters()) == 216_141_136  # SURVEY 8 a-7
    assert len(unet.state_dict()) == 829
    assert dpm.sigma_min == 0.01 and dpm.sampling_timesteps == 10


def test_t_steps_match_oracle():
    from adm_b200.ddm.ddm_const import DDPM
    net = _net(TINY)
    for n in (1, 2, 10, 50):
        cfg = dict(image_size=[16, 16], sampling_timesteps=n, sigma_min=0.01, sigma_max=1)
        dpm = DDPM(model=net, cfg=cfg, **cfg)
        ours = torch.tensor(dpm.t_steps(), dtype=torch.float64)
        assert torch.allclose(ours, O.t_steps_deterministic(n), rtol=0, atol=1e-15)


def test_completion_order_and_arena():
    from adm_b200.train import ParamArena, completion_order
    net = _net(TINY)
    order = completion_order(net)
    assert len(order) == len(list(net.parameters())) == len({id(p) for p in order})
    before = {k: v.clone() for k, v in net.state_dict().items()}
    arena = ParamArena(net, order)
    assert arena.numel >= sum(p.numel() for p in order)
    for k, v in net.state_dict().items():
        assert torch.equal(v, before[k])  # re-homing keeps values and the state_dict layout
    p0 = order[0]
    assert p0.data_ptr() == arena.flat.data_ptr() and p0.grad.data_ptr() == arena.grads.data_ptr()
    p0.grad = None
    arena.rebind_grads()
    assert p0.grad.data_ptr() == arena.grads.data_ptr()
    # out_conv2 finishes first, the batched affine + mapping layers last
    names = {id(p): n for n, p in net.named_parameters()}
    assert names[id(order[0])].startswith("model.out_conv2")
    assert names[id(order[-1])].startswith("model.map_augment")


def test_lr_schedule():
    from adm_b200.train import lr_lambda
    assert lr_lambda(0, 800000, 1e-4, 5e-6) == pytest.approx(1 / 5000)
    assert lr_lambda(4999, 800000, 1e-4, 5e-6) == pytest.approx(1.0)
    assert lr_lambda(800000, 800000, 1e-4, 5e-6) == pytest.approx(0.05)


def test_cond_unet_state_dict_layout_matches_reference(golden_dir):
    """1158 keys; every non-Swin key and shape equals the layout recorded from the reference (the Swin part was checked
    by the strict load_state_dict into the reference module when the golden file was generated)."""
    import json
    import os
    from tests.golden.make_golden_cond import CFG
    from adm_b200.unet.cond_unet import Unet
    g = json.load(open(os.path.join(golden_dir, "cond_unet_small.json")))
    sd = Unet(**CFG).state_dict()
    assert len(sd) == g["n_keys"] == 1158
    ours = {k: list(v.shape) for k, v in sd.items() if not k.startswith("init_conv_mask.")}
    assert ours == g["keys"]
    assert sum(k.startswith("init_conv_mask.") for k in sd) == g["n_swin_keys"]


def test_latent_diffusion_constructor_and_errors():
    import pytest
    import torch
    from adm_b200.ddm.ddm_const import LatentDiffusion

    class AE(torch.nn.Module):
        down_ratio = 4

        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.ones(1))

        def encode(self, x):
            return x[..., ::4, ::4]

        def decode(self, z):
            return z.repeat_interleave(4, -1).repeat_interleave(4, -2)

    class Net(torch.nn.Module):
        channels, self_condition = 3, None

    cfg = dict(image_size=[64, 64], sampling_timesteps=5, eps=1e-4, sigma_min=0.01, sigma_max=1, weighting_loss=True,
               use_l1=True, scale_factor=0.195, scale_by_std=True, default_scale=True)
    ldm = LatentDiffusion(auto_encoder=AE(), model=Net(), cfg=cfg, **cfg)
    assert float(ldm.scale_factor) == pytest.approx(0.195) and not any(p.requires_grad for p in ldm.first_stage_model.parameters())
    assert ldm.t_steps()[0] == 1 and ldm.t_steps()[-1] == 0.0 and len(ldm.t_steps()) == 6
    z, c, x = ldm.get_input({"image": torch.zeros(2, 3, 64, 64), "cond": torch.ones(2, 3, 16, 16)})
    assert z.shape == (2, 3, 16, 16) and c.shape == (2, 3, 16, 16)
    with pytest.raises(RuntimeError):  # no CPU fallback
        ldm.training_step({"image": torch.zeros(2, 3, 64, 64)})
    with pytest.raises(NotImplementedError):
        LatentDiffusion(auto_encoder=AE(), model=Net(), cfg=dict(cfg, use_disloss=True), **cfg)


def test_autoencoder_kl_layout_and_errors(golden_dir):
    import os
    import pytest
    import torch
    from tests.golden.make_golden_ae import DDCONFIG
    from adm_b200.ddm.encoder_decoder import AutoencoderKL
    g = torch.load(os.path.join(golden_dir, "ae_small.pt"))
    ae = AutoencoderKL(ddconfig=DDCONFIG, lossconfig={"disc_start": 1}, embed_dim=3)
    assert {k: list(v.shape) for k, v in ae.state_dict().items()} == g["keys"]
    assert ae.down_ratio == 4
    with pytest.raises(RuntimeError):  # no CPU fallback
        ae.encode(torch.zeros(1, 3, 64, 64))


def test_augment_pipe_reproduces_the_reference(golden_dir):
    """adm_b200.ddm.augment.AugmentPipe vs the batch recorded from the unmodified reference AugmentPipe
    (tests/golden/make_golden_augment.py; ddm/augment.py:115-328 with the arguments of ddm_const.py:179-180) under the
    same global seed: labels exact, images to float32 round-off; p = 1 makes every transform fire on every sample."""
    import torch
    from adm_b200.ddm.augment import AugmentPipe
    from tests.golden.make_golden_augment import KW, KW_HOT, SEEDS, inputs
    g = torch.load(os.path.join(golden_dir, "augment.pt"))
    for name, kw in (("cfg", KW), ("hot", KW_HOT)):
        for seed in SEEDS:
            torch.manual_seed(seed)
            y, lab = AugmentPipe(**kw)(inputs(seed))
            ref = g[f"{name}_{seed}"]
            assert lab.shape == (16, 9) and torch.equal(lab, ref["labels"])
            assert (y - ref["images"]).abs().max().item() < 1e-4
    with pytest.raises(NotImplementedError):
        AugmentPipe(brightness=1)


def test_ema_schedule_and_state_dict_match_reference_semantics():
    """ddm/ema.py:132-156: copy until update_after_step, then lerp with decay 1 - (1 + epoch)^-power clamped to beta,
    every update_every calls; state_dict keys online_model.* / ema_model.* / initted / step."""
    import torch
    from adm_b200.ddm.ema import EMA
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.BatchNorm1d(3))
    ema = EMA(net, beta=0.99, update_after_step=4, update_every=2, power=2 / 3)
    assert set(k.split(".")[0] for k in ema.state_dict()) == {"online_model", "ema_model", "initted", "step"}
    ref = {n: p.detach().clone() for n, p in net.named_parameters()}
    initted = False
    for step in range(20):
        with torch.no_grad():
            for p in net.parameters():
                p.add_(0.1 * torch.randn_like(p))
        # expected (restating the reference's update())
        if step % 2 == 0:
            if step <= 4:
                ref = {n: p.detach().clone() for n, p in net.named_parameters()}
            else:
                if not initted:
                    ref = {n: p.detach().clone() for n, p in net.named_parameters()}
                    initted = True
                epoch = max(step + 1 - 4 - 1, 0.)
                decay = 0. if epoch <= 0 else min(max(1 - (1 + epoch) ** -(2 / 3), 0.), 0.99)
                for n, p in net.named_parameters():
                    ref[n].lerp_(p.detach(), 1. - decay)
        ema.update()
        for n, p in ema.ema_model.named_parameters():
            assert torch.allclose(p, ref[n], atol=1e-6), (step, n)
    assert int(ema.step) == 20 and bool(ema.initted)
    assert not any(p.requires_grad for p in ema.ema_model.parameters())


def test_yaml_config_builds_the_reference_surface():
    """configs/cifar10/...yaml (reference schema) -> EDMPrecond + DDPM through construct_class_by_name, and the reference's
    own dotted names resolve to this package (LatentDiffusion, cond Unet, AutoencoderKL, EMA included)."""
    import os
    import yaml
    from adm_b200.ddm.utils import get_obj_by_name
    from scripts.train_uncond_dpm import build_model
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfg = yaml.safe_load(open(os.path.join(root, "configs", "cifar10", "ddm_uncond_const_uncond_unet.yaml")))
    cfg["model"]["unet"].update(model_channels=32, channel_mult=[1, 2], num_blocks=1, attn_resolutions=[8])  # small
    model = build_model(cfg, "cpu")
    assert type(model).__name__ == "DDPM" and model.sampling_timesteps == 10 and model.image_size == [32, 32]
    assert "model.model.map_layer0.weight" in model.state_dict() and "eps" in model.state_dict()
    for ref_name, ours in [("ddm.ddm_const.LatentDiffusion", "adm_b200.ddm.ddm_const"),
                           ("unet.cond_unet.Unet", "adm_b200.unet.cond_unet"),
                           ("ddm.encoder_decoder.AutoencoderKL", "adm_b200.ddm.encoder_decoder"),
                           ("ddm.ema.EMA", "adm_b200.ddm.ema"), ("unet.uncond_unet.EDMPrecond", "adm_b200.unet.uncond_unet")]:
        assert get_obj_by_name(ref_name).__module__ == ours


def test_use_augment_builds_the_in_tree_pipe():
    """use_augment: True (the reference CIFAR YAML, line 17) builds adm_b200.ddm.augment.AugmentPipe with the reference's
    arguments (ddm_const.py:179-180); without the flag there is no pipe."""
    import torch
    from adm_b200.ddm.augment import AugmentPipe
    from adm_b200.ddm.ddm_const import DDPM

    class Net(torch.nn.Module):
        channels, self_condition = 3, None

    cfg = dict(image_size=[32, 32], use_augment=True)
    d = DDPM(model=Net(), cfg=cfg, **cfg)
    assert isinstance(d.augment, AugmentPipe) and d.augment.p == 0.15 and d.augment.xflip == 1e8
    d = DDPM(model=Net(), cfg=dict(image_size=[32, 32]), image_size=[32, 32])
    assert d.augment is None and d.use_augment is False


@pytest.mark.parametrize("name", ["ddpmpp", "ncsnpp"])
def test_song_unet_state_dict_layout_matches_reference(golden_dir, name):
    """EDMPrecond(model_type='SongUNet') builds the reference's key -> shape map (recorded by make_golden_song.py from the
    unmodified reference) for the DDPM++ and the NCSN++ flavour, and loads a reference-style state_dict."""
    import torch
    from adm_b200.unet.uncond_unet import EDMPrecond
    from tests.golden.make_golden_song import CONFIGS, state_dict_for
    g = torch.load(os.path.join(golden_dir, "song_unet.pt"))[name]
    net = EDMPrecond(**CONFIGS[name])
    assert {k: list(v.shape) for k, v in net.state_dict().items()} == g["keys"]
    assert list(net.state_dict().keys()) == list(g["keys"].keys())
    missing, unexpected = net.load_state_dict(state_dict_for(g["keys"]), strict=False)
    assert not unexpected and all(k.endswith("resample_filter") for k in missing)
    with pytest.raises(RuntimeError):  # no CPU fallback
        net(torch.zeros(1, 3, 16, 16), torch.ones(1))


def test_latent_loader_scales_and_cycles():
    """scripts/train_uncond_ldm.py: the loader wrapper applies the frozen first stage + scale factor
    (ddm_const_2.py:494-524) and can be iterated again when a finite loader is exhausted."""
    import importlib.util
    import os

    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("train_uncond_ldm", os.path.join(root, "scripts", "train_uncond_ldm.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    class FakeLDM:
        scale_by_softsign, scale_by_std, scale_factor = False, True, 0.5
        started = 0

        def on_train_batch_start(self, batch):
            self.started += 1

        def get_input(self, batch):
            return [batch["image"] * 2.0, None, batch["image"]]

    ldm = FakeLDM()
    data = [{"image": torch.full((2, 3, 4, 4), float(i))} for i in (1, 2)]
    loader = mod.LatentLoader(ldm, data, torch.device("cpu"))
    for _ in range(2):  # a second pass over the exhausted loader yields the same batches
        out = [b["image"] for b in loader]
        assert len(out) == 2 and torch.equal(out[0], torch.full((2, 3, 4, 4), 1.0)) and torch.equal(out[1], torch.full((2, 3, 4, 4), 2.0))
    assert ldm.started == 1  # std-rescaling hook runs on the first batch only


def test_cond_trainer_loop_schedule_and_resume(tmp_path):
    """scripts/train_cond_ldm.py CondTrainer (train_cond_ldm.py:96-330): accumulation, warm-up schedule through the device
    learning-rate scalar, checkpoint keys and resume — on a stand-in module (the real one needs the GPU)."""
    import importlib.util
    import os

    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("train_cond_ldm", os.path.join(root, "scripts", "train_cond_ldm.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    class Toy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = torch.nn.Linear(4, 4)

        def training_step(self, batch):
            loss = ((self.lin(batch["cond"]) - batch["image"]) ** 2).mean()
            return loss, {"train/loss": loss.detach()}

    def loader():
        g = torch.Generator().manual_seed(0)
        while True:
            yield {"image": torch.randn(8, 4, generator=g), "cond": torch.randn(8, 4, generator=g)}

    cfg = {"trainer": {"warmup_iter": 4, "min_lr": 1e-6, "ema_update_after_step": 1, "ema_update_every": 1}}
    torch.manual_seed(0)
    tr = mod.CondTrainer(Toy(), loader(), gradient_accumulate_every=2, train_lr=1e-2, train_num_steps=6,
                         save_and_sample_every=3, results_folder=str(tmp_path), log_freq=100, cfg=cfg)
    w0 = tr.model.lin.weight.detach().clone()
    tr.train()
    assert tr.step == 6 and not torch.equal(w0, tr.model.lin.weight)
    assert abs(tr.lr_t.item() - 1e-2 * tr.lr_lambda(5)) < 1e-9  # the value the last step ran with
    ck = torch.load(str(tmp_path / "model-2.pt"), weights_only=False)
    assert set(ck) == {"step", "model", "opt", "lr_scheduler", "ema", "scaler"} and ck["step"] == 6
    assert any(k.startswith("ema_model.") for k in ck["ema"]) and any(k.startswith("online_model.") for k in ck["ema"])
    torch.manual_seed(1)
    tr2 = mod.CondTrainer(Toy(), loader(), gradient_accumulate_every=2, train_lr=1e-2, train_num_steps=8,
                          save_and_sample_every=100, results_folder=str(tmp_path), log_freq=100, resume_milestone=2, cfg=cfg)
    assert tr2.step == 6 and torch.equal(tr2.model.lin.weight, tr.model.lin.weight)
    assert tr2.opt.param_groups[0]["lr"] is tr2.lr_t
    tr2.train()
    assert tr2.step == 8


def test_sample_cond_script_shards_batches_and_picks_ema_weights(tmp_path):
    """scripts/sample_cond_ldm.py: round-robin sharding of the condition batches over ranks (no communication) and the
    checkpoint weight selection of sample_cond_ldm.py:140-154 — on a stand-in model."""
    import importlib.util
    import os

    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("sample_cond_ldm", os.path.join(root, "scripts", "sample_cond_ldm.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    class Toy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.zeros(1))

        def sample(self, batch_size, cond=None, mask=None):
            return cond + self.w

    cfg = {"data": {"class_name": "synthetic", "image_size": [16, 16], "batch_size": 2}}
    batches = list(mod.condition_batches(cfg, 2, 5, 4, seed=7))
    assert [b["cond"].shape[0] for b in batches] == [2, 2, 1] and batches[0]["cond"].shape[1:] == (3, 4, 4)
    m = Toy()
    full = mod.sample_all(m, batches, torch.device("cpu"))
    parts = [mod.sample_all(m, batches, torch.device("cpu"), rank=r, world=2) for r in range(2)]
    assert full.shape[0] == 5 and parts[0].shape[0] == 3 and parts[1].shape[0] == 2
    assert torch.equal(torch.cat([parts[0][:2], parts[1], parts[0][2:]]), full)
    torch.save({"model": {"w": torch.ones(1)}, "ema": {"ema_model.w": torch.full((1,), 2.0), "online_model.w": torch.ones(1),
                                                       "step": torch.tensor(3)}}, str(tmp_path / "model-1.pt"))
    mod.load_weights(m, str(tmp_path / "model-1.pt"), use_ema=True)
    assert m.w.item() == 2.0
    mod.load_weights(m, str(tmp_path / "model-1.pt"), use_ema=False)
    assert m.w.item() == 1.0
