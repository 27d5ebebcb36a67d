"""GPU tests of the training path (SURVEY.md section 8 row e2, BASELINE config 5): model-level backward
parity against fp64 autograd of the CPU oracle, the bf16 (autocast) step, the PWC-Net `npost` branch, and --
when the box has two GPUs -- DistributedDataParallel over NCCL: gradients after the all-reduce equal the
single-process gradients on the concatenated batch within 1e-5 (relative to the gradient's magnitude)."""
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from eavsr_b200 import train as T
from eavsr_b200.model import EAVSRP
from eavsr_b200.synthetic import clip_inputs, seeded_parameters
from oracle import eavsrp_cpu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _no_tf32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _crops(n, t, size, seed):
    lr = torch.cat([clip_inputs(1, t, size, size, seed=seed + i) for i in range(n)])
    hr = F.interpolate(lr.view(n * t, 3, size, size), scale_factor=4, mode="bicubic", align_corners=False)
    return lr, hr.clamp(0, 1).view(n, t, 3, 4 * size, 4 * size)


def _net(nb, device, fmt=True):
    net = EAVSRP(4, n_resblock=nb)
    seeded_parameters(net)
    net = net.to(device)
    return net.to(memory_format=torch.channels_last) if fmt else net


def test_model_backward_matches_fp64_oracle_autograd(cuda):
    """fp32 training forward + backward of the whole network (T=3, 64x64, 1 residual block per stack) against
    autograd through the fp64 CPU restatement on the same weights: loss and every parameter gradient."""
    nb, t = 1, 3
    net = _net(nb, cuda)
    lr, hr = _crops(1, t, 64, seed=40)
    tr = T.Trainer(net, dtype=torch.float32)
    sr = tr.forward(lr.to(cuda))
    loss = tr.compute_loss(sr, hr.to(cuda))
    loss.backward()
    got = {n: p.grad.detach().double().cpu() for n, p in net.named_parameters() if p.grad is not None}

    sd = {k: v.detach().double().cpu() for k, v in net.state_dict().items()}
    leaves = {k: v.requires_grad_() for k, v in sd.items() if not k.startswith("spynet.") and v.dtype == torch.float64
              and k in dict(net.named_parameters())}
    ref_sr = eavsrp_cpu.eavsrp_forward(sd, lr.double(), 4, "restatement", nb=nb)
    ref_loss = (ref_sr - hr.double()).abs().mean()
    grads = torch.autograd.grad(ref_loss, list(leaves.values()), allow_unused=True)
    assert abs(loss.item() - ref_loss.item()) < 1e-5
    assert (sr.detach().double().cpu() - ref_sr.detach()).abs().max().item() < 1e-3
    trainable = {n for n, p in net.named_parameters() if p.requires_grad}
    assert set(got) == trainable and not any(n.startswith("spynet.") for n in got)
    worst = {}
    for (name, _), g in zip(leaves.items(), grads):
        assert g is not None and name in got, name
        denom = g.norm().item()
        if denom < 1e-10:
            continue
        worst[name] = (got[name] - g).norm().item() / denom
    bad = {k: v for k, v in worst.items() if v > 2e-3}
    assert len(worst) > 250 and not bad, sorted(bad.items(), key=lambda kv: -kv[1])[:8]


def test_bf16_autocast_step_tracks_fp32(cuda):
    nb, t = 2, 4
    lr, hr = _crops(2, t, 64, seed=50)
    lr, hr = lr.to(cuda), hr.to(cuda)
    n32, n16 = _net(nb, cuda), _net(nb, cuda)
    t32, t16 = T.Trainer(n32, dtype=torch.float32), T.Trainer(n16, dtype=torch.bfloat16)
    l32, l16 = t32.step(lr, hr), t16.step(lr, hr)
    assert torch.isfinite(l16) and abs(l16.item() - l32.item()) < 2e-3
    g32, g16 = t32.gradients(), t16.gradients()
    assert set(g32) == set(g16)
    a = torch.cat([g.flatten().float() for _, g in sorted(g32.items())])
    b = torch.cat([g.flatten().float() for _, g in sorted(g16.items())])
    assert all(g.dtype == torch.float32 for g in g16.values())          # fp32 master weights and gradients
    assert F.cosine_similarity(a, b, dim=0).item() > 0.98
    for p in n16.parameters():
        assert p.dtype == torch.float32 and torch.isfinite(p).all()


def test_npost_branch_masks_sr_with_pwc_validity(cuda):
    """models/eavsrp_model.py:85-97: for epoch >= npost the SR is multiplied by the get_backwarp validity mask
    of the frozen PWC-Net (which runs the cost volume and backwarp kernels); the PWC-Net gets no gradient."""
    from eavsr_b200 import _lib
    from eavsr_b200.pwc import PWCNET
    net = _net(1, cuda)
    pwc = PWCNET()
    seeded_parameters(pwc)
    pwc = pwc.to(cuda)
    lr, hr = _crops(1, 3, 64, seed=60)
    tr = T.Trainer(net, pwcnet=pwc, npost=5)
    sr0 = tr.forward(lr.to(cuda), hr.to(cuda), epoch=0)
    before = _lib.launch_count()
    sr1 = tr.forward(lr.to(cuda), hr.to(cuda), epoch=5)
    assert _lib.launch_count() - before >= 3 * (5 + 4 + 1)      # per frame: 5 cost volumes, 4 + 1 backwarps
    ratio = sr1.detach() / sr0.detach().clamp_min(1e-6)
    assert ((ratio - 1).abs() < 1e-4).logical_or(sr1.detach() == 0).all()
    loss = tr.step(lr.to(cuda), hr.to(cuda), epoch=5)
    assert torch.isfinite(loss) and all(p.grad is None for p in pwc.parameters())


# ---------------------------------------------------------------------------------------------
# two GPUs, NCCL
# ---------------------------------------------------------------------------------------------
def _ddp_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        net = _net(1, dev)
        tr = T.Trainer(net, ddp=True, device_ids=[rank])
        lr, hr = _crops(2 * world, 3, 64, seed=70)
        mine = slice(2 * rank, 2 * rank + 2)
        loss = tr.step(lr[mine].to(dev), hr[mine].to(dev))
        ret[rank] = ({n: g.detach().float().cpu() for n, g in tr.gradients().items()}, loss.item())
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_ddp_gradients_equal_single_process(cuda):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ret = mp.Manager().dict()
    mp.spawn(_ddp_worker, args=(2, port, ret), nprocs=2, join=True)
    net = _net(1, cuda)
    tr = T.Trainer(net)
    lr, hr = _crops(4, 3, 64, seed=70)
    loss = tr.step(lr.to(cuda), hr.to(cuda))
    single = {n: g.detach().float().cpu() for n, g in tr.gradients().items()}
    assert abs(0.5 * (ret[0][1] + ret[1][1]) - loss.item()) < 1e-5
    for r in (0, 1):
        grads = ret[r][0]
        assert sorted(grads) == sorted(single)
        for n, g in single.items():
            # scatter-add gradients (warp / DCN d(x)) are summed with floating-point atomics: 1e-5 relative to
            # the tensor's largest gradient (SURVEY.md section 4, distributed row)
            assert (grads[n] - g).abs().max().item() <= 1e-5 * max(g.abs().max().item(), 1e-3) + 1e-7, n
    for n in single:
        assert torch.equal(ret[0][0][n], ret[1][0][n]), n           # both ranks hold the same reduced gradient


def test_graph_captured_step_equals_eager_step(cuda):
    """Trainer.capture: forward + L1 + backward + Adam as ONE CUDA graph; a replayed step changes the parameters
    exactly as an eager step from the same state does (up to the atomics' summation order)."""
    import copy
    lr, hr = _crops(2, 3, 64, seed=80)
    lr, hr = lr.to(cuda), hr.to(cuda)
    net_g = _net(1, cuda)
    tg = T.Trainer(net_g, dtype=torch.bfloat16, capturable=True)
    tg.capture(lr, hr, warmup=2)                       # two real steps, then the recording (which does not execute)
    net_e = copy.deepcopy(net_g)
    te = T.Trainer(net_e, dtype=torch.bfloat16, capturable=True)
    te.optimizer.load_state_dict(copy.deepcopy(tg.optimizer.state_dict()))
    lr2, hr2 = _crops(2, 3, 64, seed=81)
    lg = tg.step_graphed(lr2.to(cuda), hr2.to(cuda))
    le = te.step(lr2.to(cuda), hr2.to(cuda))
    assert torch.isfinite(lg) and abs(lg.item() - le.item()) < 1e-5
    worst = 0.0
    for (n, a), (_, b) in zip(net_g.named_parameters(), net_e.named_parameters()):
        worst = max(worst, (a - b).abs().max().item())
    assert worst < 5e-5, worst                         # one Adam step moves a weight by <= lr = 1e-4
