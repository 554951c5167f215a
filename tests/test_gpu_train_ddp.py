"""-m gpu, needs TWO devices (skipped on a machine with one GPU): the data-parallel fine-tune step
over NCCL - two ranks x B/2 images with SyncBatchNorm and the bucketed gradient all-reduce must equal one process x B images (reference semantics:
DistributedDataParallel + SyncBatchNorm, trainer/trainer.py:334, utils/distributed/dist.py:138-157)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1200)]
SIZE, B = 192, 4


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _setup(dev, rank=None, world=1):
    from focoos_b200 import DETRConfig, FAIDetr
    from focoos_b200.criterion import DETRTargets
    from focoos_b200.train_step import FlatAdamW, GradBucketReducer, TrainStep, get_optimizer_params
    from focoos_b200.utils.seeded_weights import desaturate_classifiers
    from oracle.gen_golden import synth_images
    from oracle.gen_golden_train import synth_targets
    from tests.parity_utils import seeded_sd

    m = FAIDetr(DETRConfig(), precision="fp32")
    m.load_state_dict(desaturate_classifiers(seeded_sd(0)), strict=True)
    m.to(dev).train()
    m.sync_bn = world > 1
    opt = FlatAdamW(get_optimizer_params(m, base_lr=5e-4, weight_decay=0.02, weight_decay_norm=0.0, backbone_multiplier=0.1), clip_gradients=0.1, amp=True, world_size=world)
    opt.track_unused_parameters()
    red = GradBucketReducer(opt, model=m)
    red.attach_hooks()
    x = torch.from_numpy(np.stack(synth_images(5, [(SIZE, SIZE)] * B))).permute(0, 3, 1, 2).float()
    t = synth_targets(6, B, m.config.num_classes)
    sl = slice(None) if rank is None else slice(rank * B // world, (rank + 1) * B // world)
    targets = [DETRTargets(labels=a.to(dev), boxes=b.to(dev)) for a, b in t[sl]]
    return m, opt, TrainStep(m, opt, red), x[sl].to(dev), targets


def _summary(m, opt, losses):
    bn = m.pixel_decoder.backbone.conv1.conv1_1.norm
    return {"loss": float(sum(v.detach() for v in losses.values())), "params": opt.flat_params.detach().cpu().numpy(), "grad_norm": opt.stats()["grad_norm"],
            "rm": bn.running_mean.cpu().numpy(), "rv": bn.running_var.cpu().numpy(), "match": m.criterion().last_match.cpu().numpy()}


def _worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    m, opt, step, x, targets = _setup(dev, rank, world)
    p0 = opt.flat_params.detach().cpu().numpy().copy()
    losses = step(x, targets)
    torch.cuda.synchronize()
    s = _summary(m, opt, losses)
    s["p0"] = p0
    q.put((rank, s))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpus_equal_one_gpu_on_the_full_batch():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    dev = torch.device("cuda", 0)
    m, opt, step, x, targets = _setup(dev)
    p0 = opt.flat_params.detach().cpu().numpy().copy()
    ref = _summary(m, opt, step(x, targets))
    del m, opt, step
    torch.cuda.empty_cache()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=900) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
    a, b = out[0], out[1]
    assert np.array_equal(a["params"], b["params"]), "replicas stay bit-identical after an exchanged step"
    d_ref, d_ddp = ref["params"] - p0, a["params"] - a["p0"]
    assert np.array_equal(a["p0"], p0)
    # the per-rank losses are normalised by the GLOBAL box count (all-reduced), so their sum over ranks / world is the full-batch loss
    assert abs(0.5 * (a["loss"] + b["loss"]) - ref["loss"]) <= 2e-3 * abs(ref["loss"]), (a["loss"], b["loss"], ref["loss"])
    assert abs(a["grad_norm"] - ref["grad_norm"]) <= 5e-3 * ref["grad_norm"], (a["grad_norm"], ref["grad_norm"])
    assert np.abs(a["rm"] - ref["rm"]).max() < 1e-4 and np.abs(a["rv"] - ref["rv"]).max() < 1e-3, "SyncBatchNorm: running statistics of the FULL batch on every rank"
    nz = np.abs(d_ref) > 0
    rel = np.linalg.norm(d_ddp - d_ref) / np.linalg.norm(d_ref)
    assert rel < 2e-2, f"AdamW update of the two-rank step differs from the full-batch step by {rel:.3e} (relative, whole model)"
    print(f"[ddp] loss {ref['loss']:.5f} vs {(a['loss'] + b['loss']) / 2:.5f}; update rel. diff {rel:.2e}; {int(nz.sum())} parameters moved")
