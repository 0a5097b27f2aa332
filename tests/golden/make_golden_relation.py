"""Generates tests/golden/relation_layer.pt by running the UNMODIFIED reference ``unet.cond_unet.BasicAttetnionLayer``
(/root/reference/unet/cond_unet.py:153-252; build container only; CPU fp32, eval mode) on seeded inputs:

    python tests/golden/make_golden_relation.py

Recorded: the output and the gradients of sum(output * probe) with respect to both inputs and every parameter.  The
inputs themselves are not stored: ``draw`` makes them from the recorded seed (the layer's state_dict, drawn by the
layer's own init, with the GroupNorm affine and the conv biases perturbed so that they are exercised; then x1 (condition
features), x2 (trunk features) and the probe), and ``load`` redraws them through the in-tree layer, whose init follows
the reference's draw for draw, and checks them against the SHA-256 recorded with the reference's draw.  Two cases: a
low-resolution condition map (4x4 -> 16x16, the DIV2K config's geometry: Swin features are resized up to the trunk
resolution) and equal resolutions with ragged windows (the zero padding of F.pad + AvgPool2d).
"""
import hashlib
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tests.golden.make_golden_cond import import_reference_cond  # noqa: E402

CASES = {
    "lowres_cond": dict(embed_dim=64, nhead=8, ffn_dim=128, window_size1=[2, 2], window_size2=[4, 4], b=2,
                        hw1=(4, 4), hw2=(16, 16)),
    "ragged_windows": dict(embed_dim=64, nhead=8, ffn_dim=128, window_size1=[4, 4], window_size2=[3, 3], b=1,
                           hw1=(10, 10), hw2=(10, 10)),
}


def draw(layer_cls, spec, seed):
    """The layer (CPU, fp32) and the inputs x1, x2, probe (NCHW) of one case, from the global RNG seeded with `seed`."""
    torch.manual_seed(seed)
    layer = layer_cls(embed_dim=spec["embed_dim"], nhead=spec["nhead"], ffn_dim=spec["ffn_dim"],
                      window_size1=spec["window_size1"], window_size2=spec["window_size2"])
    with torch.no_grad():
        layer.gn.weight.add_(0.3 * torch.randn_like(layer.gn.weight))
        layer.gn.bias.add_(0.2 * torch.randn_like(layer.gn.bias))
        for m in (layer.concat_conv, layer.out_conv, layer.mlp.fc1, layer.mlp.fc2, layer.q_lin, layer.k_lin, layer.v_lin):
            m.bias.add_(0.1 * torch.randn_like(m.bias))
    c, b = spec["embed_dim"], spec["b"]
    x1 = torch.randn(b, c, *spec["hw1"])
    x2 = torch.randn(b, c, *spec["hw2"]) * 1.3 + 0.2
    probe = torch.randn(b, c, *spec["hw2"])
    return layer, x1, x2, probe


def digest(state_dict, *tensors):
    h = hashlib.sha256()
    for t in list(state_dict.values()) + list(tensors):
        h.update(t.detach().contiguous().numpy().tobytes())
    return h.hexdigest()


def make(cu, spec, seed):
    layer, x1, x2, probe = draw(cu.BasicAttetnionLayer, spec, seed)
    layer.eval()
    sd = layer.state_dict()
    sha = digest(sd, x1, x2, probe)
    x1, x2 = x1.requires_grad_(True), x2.requires_grad_(True)
    out = layer(x1, x2)
    (out * probe).sum().backward()
    return dict(spec=spec, seed=seed, inputs_sha256=sha, out=out.detach(), dx1=x1.grad.clone(), dx2=x2.grad.clone(),
                grads={k: p.grad.clone() for k, p in layer.named_parameters()})


def load(golden_dir):
    """The recorded cases, each completed with its redrawn state_dict, x1, x2 and probe."""
    from adm_b200.unet.cond_unet import BasicAttetnionLayer
    rec = torch.load(os.path.join(golden_dir, "relation_layer.pt"))
    with torch.random.fork_rng(devices=[]):
        for name, r in rec.items():
            layer, x1, x2, probe = draw(BasicAttetnionLayer, r["spec"], r["seed"])
            sd = {k: v.detach().clone() for k, v in layer.state_dict().items()}
            assert digest(sd, x1, x2, probe) == r["inputs_sha256"], \
                f"{name}: the redrawn inputs differ from the ones the reference ran on (layer init or draw order changed)"
            r.update(state_dict=sd, x1=x1, x2=x2, probe=probe)
    return rec


def main():
    cu = import_reference_cond()
    rec = {name: make(cu, spec, 100 + i) for i, (name, spec) in enumerate(CASES.items())}
    path = os.path.join(HERE, "relation_layer.pt")
    torch.save(rec, path)
    print("wrote", path, {k: tuple(v["out"].shape) for k, v in rec.items()}, f"{os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
