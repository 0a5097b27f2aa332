"""Data-parallel training of the conditional latent model (adm_b200.train.AutogradDataParallel inside
scripts/train_cond_ldm.py's CondTrainer), two ranks in two processes.

CPU, gloo: replica synchronisation, the summed gradient buffer and the mean the optimizer step applies, one reduction
per accumulation window, a rank-0 checkpoint load reaching every rank, per-rank data.  The helper does not depend on the
module type, so a small torch module stands in for the UNet.
GPU (one B200, gloo on CUDA tensors: NCCL refuses two ranks on one device): the reduced gradient of the small
conditional UNet against one process that accumulates the same two halves as two micro-batches, and the graphed
step of several ranks (two CUDA graphs around the eager all-reduce) keeping the replicas identical."""
import os
import socket
import time

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

WORLD = 2
TIMEOUT_S = 900


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(fn, *args):
    """fn(rank, world, port, *args) in WORLD spawned processes, joined with a timeout; none outlives the call."""
    ctx = mp.start_processes(fn, args=(WORLD, _free_port(), *args), nprocs=WORLD, join=False, start_method="spawn")
    deadline = time.monotonic() + TIMEOUT_S
    try:
        while not ctx.join(timeout=5):
            if time.monotonic() > deadline:
                pytest.fail(f"workers did not finish within {TIMEOUT_S} s")
    finally:
        for p in ctx.processes:
            if p.is_alive():
                p.kill()
            p.join()


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _gathered(t):
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t.contiguous())
    return out


def _same_on_all_ranks(t):
    return all(torch.equal(x, t) for x in _gathered(t))


class Toy(torch.nn.Module):
    """Stand-in for LatentDiffusion: trainable layers, a frozen one and a buffer, ``training_step(batch)``."""

    def __init__(self):
        super().__init__()
        self.frozen = torch.nn.Linear(6, 6)
        self.frozen.requires_grad_(False)
        self.net = torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.Tanh(), torch.nn.Linear(16, 6))
        self.register_buffer("scale", torch.rand(()) + 0.5)
        self.forwards = 0

    def training_step(self, batch):
        self.forwards += 1
        loss = ((self.net(self.frozen(batch["cond"])) * self.scale - batch["image"]) ** 2).mean() * 50
        return loss, {"train/loss": loss.detach()}


def _batches(seed, n=4, b=8):
    g = torch.Generator().manual_seed(seed)
    return [{"image": torch.randn(b, 6, generator=g), "cond": torch.randn(b, 6, generator=g)} for _ in range(n)]


CFG = {"trainer": {"warmup_iter": 2, "min_lr": 1e-6, "ema_update_after_step": 0, "ema_update_every": 1}}


def _trainer(model, batches, folder, accum=1, resume=0):
    from scripts.train_cond_ldm import CondTrainer
    return CondTrainer(model, iter(batches), gradient_accumulate_every=accum, train_lr=1e-2, train_num_steps=100,
                       save_and_sample_every=2, results_folder=str(folder), log_freq=1000, resume_milestone=resume,
                       cfg=CFG)


# ------------------------------------------------------------------------------------------------ CPU, gloo
def _w_replicas(rank, world, port):
    _init(rank, world, port)
    from adm_b200.train import AutogradDataParallel
    torch.manual_seed(100 + rank)  # replicas start from different weights, frozen layer and buffer included
    m = Toy()
    before = torch.cat([t.detach().flatten() for t in m.state_dict().values()])
    assert not _same_on_all_ranks(before)
    dp = AutogradDataParallel(m, [p for p in m.parameters() if p.requires_grad])
    assert dp.world == world
    for k, t in m.state_dict().items():
        assert _same_on_all_ranks(t), k
    # every trainable .grad is a view of the one flat buffer; the frozen layer has none
    a = dp.arena
    for p, o in zip(a.params, a.offsets):
        assert p.grad.data_ptr() == a.grads.data_ptr() + 4 * o
    assert m.frozen.weight.grad is None and len(a.params) == 4
    dist.destroy_process_group()


def test_replicas_identical_after_construction():
    _run(_w_replicas)


def _w_sum_and_mean(rank, world, port, out_dir):
    _init(rank, world, port)
    from adm_b200.train import AutogradDataParallel
    torch.manual_seed(rank)
    m = Toy()
    params = [p for p in m.parameters() if p.requires_grad]
    dp = AutogradDataParallel(m, params)
    init = {k: v.clone() for k, v in m.state_dict().items()}
    data = _batches(7)
    mine = data[rank]
    dp.zero_grad()
    loss, _ = m.training_step(mine)
    loss.backward()
    local = [p.grad.clone() for p in params]
    dp.all_reduce()
    for p, g in zip(params, local):
        assert torch.equal(p.grad, sum(_gathered(g))), "each .grad view holds the sum over the ranks"
    norm = dp.clip_mean_(1.0)
    # reference: one process, both ranks' batches as two micro-batches, clip_grad_norm_ on the mean
    ref = Toy()
    ref.load_state_dict(init)
    rp = [p for p in ref.parameters() if p.requires_grad]
    for b in data[:world]:
        (ref.training_step(b)[0] / world).backward()
    ref_norm = torch.nn.utils.clip_grad_norm_(rp, 1.0)
    assert float(ref_norm) > 1.0, "the test must exercise the clip"
    assert torch.allclose(norm, ref_norm, rtol=1e-5)
    for p, r in zip(params, rp):
        assert torch.allclose(p.grad, r.grad, rtol=1e-5, atol=1e-7)
    # a whole CondTrainer step applies the same update on both ranks: the mean, clipped, through AdamW
    torch.manual_seed(50 + rank)
    m2 = Toy()
    tr = _trainer(m2, [data[rank]], os.path.join(out_dir, f"r{rank}"))
    start = {k: v.clone() for k, v in m2.state_dict().items()}
    tr.train_one_step()
    ref2 = Toy()
    ref2.load_state_dict(start)
    rp2 = [p for p in ref2.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(rp2, lr=1e-2 * tr.lr_lambda(0), weight_decay=1e-4)
    for b in data[:world]:
        (ref2.training_step(b)[0] / world).backward()
    torch.nn.utils.clip_grad_norm_(rp2, 1.0)
    opt.step()
    for (k, v), r in zip(m2.state_dict().items(), ref2.state_dict().values()):
        assert _same_on_all_ranks(v), k
        assert torch.allclose(v, r, rtol=1e-5, atol=1e-6), k
    dist.destroy_process_group()


def test_reduced_gradient_is_the_sum_and_the_step_applies_the_mean(tmp_path):
    _run(_w_sum_and_mean, str(tmp_path))


def _w_accumulation(rank, world, port, out_dir):
    _init(rank, world, port)
    torch.manual_seed(rank)
    m = Toy()
    tr = _trainer(m, _batches(20 + rank, n=4), os.path.join(out_dir, f"r{rank}"), accum=2)
    grads = tr.dp.arena.grads
    calls = []
    real = dist.all_reduce

    def counting(t, *a, **kw):
        if t.data_ptr() == grads.data_ptr():
            calls.append(m.forwards)  # micro-batches run when the reduction is issued
        return real(t, *a, **kw)
    dist.all_reduce = counting
    try:
        tr.train_one_step()
        tr.train_one_step()
    finally:
        dist.all_reduce = real
    assert calls == [2, 4], calls  # one reduction per optimizer step, after its second (last) micro-batch
    for v in m.state_dict().values():
        assert _same_on_all_ranks(v)
    dist.destroy_process_group()


def test_accumulation_reduces_once_after_the_last_micro_batch(tmp_path):
    _run(_w_accumulation, str(tmp_path))


def _w_load(rank, world, port, out_dir):
    _init(rank, world, port)
    folder = os.path.join(out_dir, f"r{rank}")  # only rank 0's folder will hold the checkpoint
    torch.manual_seed(rank)
    tr = _trainer(Toy(), _batches(30 + rank, n=3), folder)
    for _ in range(2):
        tr.train_one_step()
    tr.save(1)
    assert os.path.isfile(os.path.join(folder, "model-1.pt")) == (rank == 0)
    saved = torch.load(os.path.join(out_dir, "r0", "model-1.pt"), weights_only=False) if rank == 0 else None
    dist.barrier()
    torch.manual_seed(200 + rank)  # fresh replicas with different weights and no optimizer state
    tr2 = _trainer(Toy(), _batches(40 + rank, n=3), folder, resume=1)
    assert tr2.step == 2
    assert tr2.opt.param_groups[0]["lr"] is tr2.lr_t
    for k, v in tr2.model.state_dict().items():
        assert _same_on_all_ranks(v), k
        if rank == 0:
            assert torch.equal(v, saved["model"][k]), k
    for i, p in enumerate(tr2.params):
        st = tr2.opt.state[p]
        assert set(st) == {"step", "exp_avg", "exp_avg_sq"}
        for k in ("step", "exp_avg", "exp_avg_sq"):
            assert _same_on_all_ranks(st[k].reshape(-1)), (i, k)
            if rank == 0:
                assert torch.equal(st[k], saved["opt"]["state"][i][k])
    assert (tr2.ema is not None) == (rank == 0)
    tr2.train_one_step()  # and training goes on in step on both ranks
    for v in tr2.model.state_dict().values():
        assert _same_on_all_ranks(v)
    dist.destroy_process_group()


def test_rank0_load_reaches_every_rank(tmp_path):
    _run(_w_load, str(tmp_path))


class TinyPairs(torch.utils.data.Dataset):
    """Ten numbered super-resolution pairs (for the sharded-dataset loader)."""

    def __init__(self, **_):
        pass

    def __len__(self):
        return 10

    def __getitem__(self, i):
        return {"image": torch.full((3, 4, 4), float(i)), "cond": torch.full((3, 2, 2), float(i))}


def _w_loaders(rank, world, port):
    _init(rank, world, port)
    from scripts.train_cond_ldm import make_loader
    d = {"class_name": "synthetic", "image_size": [8, 8], "batch_size": 2}
    first = [next(make_loader(d, 2, 2, rank, world)) for _ in range(2)]
    for k in ("image", "cond"):
        assert torch.equal(first[0][k], first[1][k])  # deterministic per rank
        mine = _gathered(first[0][k])
        assert not torch.equal(mine[0], mine[1])  # different data on each rank
    dl = make_loader({"class_name": "tests.test_dp_cond.TinyPairs", "batch_size": 2}, 2, 2, rank, world)
    epoch0 = torch.cat([next(dl)["image"][:, 0, 0, 0] for _ in range(2)])  # 10 items / 2 ranks / batch 2: 2 batches
    assert len(set(torch.cat(_gathered(epoch0)).tolist())) == 8  # the ranks' shards are disjoint
    dist.destroy_process_group()


def test_per_rank_loaders():
    _run(_w_loaders)


# ------------------------------------------------------------------------------------------------ GPU
def _small_cond_ldm(dropout):
    """LatentDiffusion around the small conditional UNet of tests/golden/make_golden_cond.py (identity first stage)."""
    import torchvision
    from adm_b200.ddm.ddm_const import LatentDiffusion
    from tests.golden.make_golden_cond import LAT, build_ours

    class _AE(torch.nn.Module):
        down_ratio = 1

        def encode(self, x):
            return x

        def decode(self, z):
            return z

    net = build_ours().cuda().train()
    if not dropout:
        for mod in net.modules():
            if isinstance(mod, (torch.nn.Dropout, torchvision.ops.StochasticDepth)):
                mod.p = 0.0
    cfg = dict(image_size=[LAT, LAT], sampling_timesteps=3, eps=1e-4, sigma_max=1, sigma_min=0.01, weighting_loss=True,
               use_l1=True)
    return LatentDiffusion(auto_encoder=_AE(), model=net, scale_by_std=False, cfg=cfg, **cfg).cuda().train()


N_REF = 5  # runs of the one-process reference that calibrate the gradient bound


def _angle(a, b):
    return float(torch.arccos(torch.nn.functional.cosine_similarity(a.flatten(), b.flatten(), dim=0).clamp(-1, 1)))


def _gpu_grad_worker(rank, world, port, out_path):
    _init(rank, world, port)
    torch.cuda.set_device(0)
    from adm_b200.train import AutogradDataParallel
    from tests.golden.make_golden_cond import BATCH, COND, LAT
    ldm = _small_cond_ldm(dropout=False)  # the two processes and the reference must draw nothing
    g = torch.Generator().manual_seed(3)
    n = 2 * BATCH
    x = (2 * torch.rand(n, 3, LAT, LAT, generator=g) - 1).cuda()
    t = (torch.rand(n, generator=g) * 0.8 + 0.1).cuda()
    noise = torch.randn(n, 3, LAT, LAT, generator=g).cuda()
    cond = (2 * torch.rand(n, 3, COND, COND, generator=g) - 1).cuda()
    halves = [slice(0, BATCH), slice(BATCH, n)]
    params = [p for p in ldm.parameters() if p.requires_grad]
    names = [k for k, p in ldm.named_parameters() if p.requires_grad]
    dp = AutogradDataParallel(ldm, params)
    dp.zero_grad()
    h = halves[rank]
    loss, _ = ldm.p_losses(x[h], t[h], cond[h], noise=noise[h])
    loss.backward()
    dp.all_reduce()
    dp_mean = [p.grad.double() / world for p in params]
    if rank == 0:
        def reference():  # one process, the two halves as two micro-batches
            dp.zero_grad()
            for s in halves:
                (ldm.p_losses(x[s], t[s], cond[s], noise=noise[s])[0] / len(halves)).backward()
            return [p.grad.double() for p in params]
        refs = [reference() for _ in range(N_REF)]
        pairs = [(a, b) for a in range(N_REF) for b in range(a + 1, N_REF)]
        rows = []
        for i, k in enumerate(names):
            spread = max(_angle(refs[a][i], refs[b][i]) for a, b in pairs)
            nearest = min(_angle(dp_mean[i], r[i]) for r in refs)
            rows.append((k, nearest, spread, float(dp_mean[i].norm()), float(refs[0][i].norm())))
        torch.save(rows, out_path)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_reduced_gradient_matches_two_micro_batches_on_gpu(tmp_path):
    """Small conditional config of tests/golden/make_golden_cond.py, dropout 0, explicit latents / condition / t /
    noise per rank.  Split-K weight gradients (and some norm-parameter reductions) accumulate with fp32 atomics, so
    gradients are not bit-reproducible, and a tensor whose true gradient is nearly zero (the key bias of an attention)
    is mostly that noise.  The bound is calibrated in the test from N_REF runs of the one-process reference: per
    tensor, the angle between the reduced mean and the nearest reference run must be at most twice the widest angle
    between two reference runs (the angle obeys the triangle inequality; 1 - cosine, its square, does not).  One
    reference run alone estimates the scatter too noisily for the low-signal tensors."""
    out = str(tmp_path / "rows.pt")
    _run(_gpu_grad_worker, out)
    rows = torch.load(out)
    assert len(rows) > 100
    bad = []
    for k, a_dp, spread, n_dp, n_ref in rows:
        if n_ref == 0.0:
            assert n_dp == 0.0, k
            continue
        # 1e-6 rad: the float64 rounding of the angle itself when the runs agree bit for bit
        if a_dp > 2.0 * spread + 1e-6:
            bad.append((k, a_dp, spread))
    assert not bad, bad[:10]


def _gpu_graph_worker(rank, world, port, out_dir):
    _init(rank, world, port)
    torch.cuda.set_device(0)
    from tests.golden.make_golden_cond import COND, LAT
    side = torch.cuda.Stream()  # autograd's AccumulateGrad nodes must not be bound to the default stream
    side.wait_stream(torch.cuda.current_stream())
    torch.cuda.set_stream(side)
    torch.manual_seed(100 + rank)  # different initial weights, t, noise and dropout on each rank
    ldm = _small_cond_ldm(dropout=True)
    g = torch.Generator().manual_seed(rank)
    data = [{"image": 2 * torch.rand(2, 3, LAT, LAT, generator=g) - 1,
             "cond": 2 * torch.rand(2, 3, COND, COND, generator=g) - 1} for _ in range(7)]
    from scripts.train_cond_ldm import CondTrainer
    tr = CondTrainer(ldm, iter(data), train_lr=1e-4, train_num_steps=100, save_and_sample_every=100,
                     results_folder=os.path.join(out_dir, f"r{rank}"), log_freq=1000, cfg=CFG, use_graph=True)

    def weights():  # every parameter, trainable and frozen (BatchNorm running statistics stay per rank)
        return torch.cat([p.detach().float().flatten() for p in ldm.parameters()]).cpu()
    w0 = weights()
    assert _same_on_all_ranks(w0)
    losses = [float(tr.train_one_step()) for _ in range(7)]  # 3 eager steps, then capture and 4 replays
    torch.cuda.synchronize()
    assert tr.graph is not None and tr.graph_update is not None
    w = weights()
    assert _same_on_all_ranks(w), "replicas diverged under the graphed data-parallel step"
    assert not torch.equal(w, w0) and all(map(lambda v: v == v and abs(v) < float("inf"), losses)), losses
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_graphed_dp_step_keeps_replicas_identical_on_gpu(tmp_path):
    """--graph with several ranks: forward + backward graph, eager all-reduce, clip + AdamW graph.  Two processes on
    one GPU over gloo, the small conditional config with dropout on: after the replays both replicas are identical."""
    _run(_gpu_graph_worker, str(tmp_path))
