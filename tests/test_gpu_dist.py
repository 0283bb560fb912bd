"""2-GPU parity of the data-parallel step (SURVEY 8e; the reference's nn.DataParallel / DDP wrappers, trainer.py:165-171,
191-196): one process per GPU over NCCL, per-replica BatchNorm and class-aware loss, one all-reduce (mean) per gradient
bucket slice issued while backward is still running.

Checked against a SINGLE-PROCESS emulation of the same step: the fused trainer's `all_reduce` hook is replaced by one
that records / substitutes gradient slices, so that
    phase 1: each shard's step yields its discriminator gradients (they only depend on the shared initial weights),
    phase 2: each shard's step, with the AVERAGED discriminator gradients substituted, yields its generator gradients
             (the G step runs through the discriminators as updated by the averaged gradients),
    phase 3: shard 0's step with every averaged gradient substituted is what rank 0 must hold after the real 2-rank step.
Same kernels, reproducible reductions, fp32 on the wire: parameters, Adam moments, EMA weights and rank 0's (per-replica)
BatchNorm buffers must agree to 1e-6 relative (NCCL's mean of two fp32 values is exact). Needs 2 GPUs (skipped otherwise;
log of a 2-GPU run in profiles/r02_two_gpu_parity.txt)."""
import os
import socket
import tempfile

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
BRANCHES, B, SEED = 3, 8, 0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _build(dev, all_reduce=None):
    from oracle.stackgan_oracle import Cfg, init_d_state, init_g_state
    from sg2b200 import model, trainer
    from tests.parity_util import set_cfg
    ocfg = Cfg(BRANCH_NUM=BRANCHES)
    cfg = set_cfg(ocfg)
    torch.manual_seed(SEED)                         # identical initial weights on every rank / in the emulation
    netG = model.G_NET()
    netG.load_state_dict(init_g_state(ocfg))
    netsD = []
    for i, cls in enumerate((model.D_NET64, model.D_NET128, model.D_NET256)[:BRANCHES]):
        d = cls()
        d.load_state_dict(init_d_state(ocfg, i))
        netsD.append(d.to(dev))
    tr = trainer.FusedTrainer(netG.to(dev), netsD, cfg, all_reduce=all_reduce)
    return cfg, tr


def _shard(cfg, rank, dev):
    from tests.parity_util import train_batch
    b = train_batch(cfg, B, 800 + rank)
    return {k: ([t.to(dev) for t in v] if isinstance(v, list) else v.to(dev)) for k, v in b.items()}


def _rank_main(rank, world, port, out_path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from sg2b200 import dist as sdist
    sdist.init_from_env(backend="nccl")
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    cfg, tr = _build(dev, all_reduce=sdist.GradAllReducer(channels=4))
    b = _shard(cfg, rank, dev)
    losses = tr.step(b["z"], b["emb"], b["real"], b["wrong"], b["labels"], eps=b["eps"]).clone()
    torch.cuda.synchronize()
    if rank == 0:
        snap = tr.snapshot()
        torch.save({"snap": {"buckets": [{k: v.cpu() for k, v in bk.items()} for bk in snap["buckets"]],
                             "buffers": [[t.cpu() for t in l] for l in snap["buffers"]]}, "losses": losses.cpu()}, out_path)
    dist.barrier()
    dist.destroy_process_group()


class _Hook:
    """Stands in for the NCCL all-reduce in the single-process emulation (see module docstring)."""

    def __init__(self, tr):
        self.tr, self.mode, self.rec, self.sub = tr, "off", {}, {}

    def __call__(self, g, chan):
        nD = len(self.tr.bD)
        bucket = self.tr.bD[chan] if chan < nD else self.tr.bG
        key = (chan, (g.data_ptr() - bucket.grad.data_ptr()) // 4, g.numel())
        if key in self.sub:
            g.copy_(self.sub[key])
        elif self.mode == "record":
            self.rec[key] = g.clone()
        return g


def test_two_rank_step_equals_mean_gradient_emulation():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    port = _free_port()
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "rank0.pt")
        procs = [ctx.Process(target=_rank_main, args=(r, 2, port, out)) for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(600)
            assert p.exitcode == 0, p.exitcode
        real = torch.load(out)
    dev = torch.device("cuda", 0)
    cfg, tr = _build(dev)
    # the rank processes run their persistent kernels on the data-parallel grid (SMs reserved for NCCL): the emulation must
    # use the same grid, because the tile -> CTA assignment fixes the summation order of the BatchNorm / wgrad partials
    # (a different order changes them by 1e-7, which bf16 storage and small-batch BatchNorm amplify chaotically)
    from sg2b200 import _lib
    _lib.call("sg2_set_sm_reserve", int(os.environ.get("SG2_SM_RESERVE", "8")))
    try:
        _emulate_and_compare(cfg, tr, dev, real)
    finally:
        _lib.call("sg2_set_sm_reserve", 0)


def _emulate_and_compare(cfg, tr, dev, real):
    from tests.parity_util import rel, snapshot_diff
    hook = _Hook(tr)
    tr.all_reduce = hook
    nD = len(tr.bD)
    shards = [_shard(cfg, r, dev) for r in range(2)]
    snap0 = tr.snapshot()

    def run(b):
        tr.restore(snap0)
        out_ = tr.step(b["z"], b["emb"], b["real"], b["wrong"], b["labels"], eps=b["eps"]).clone()
        torch.cuda.synchronize()
        return out_

    per = []
    for b in shards:                                   # phase 1: D gradients of each shard
        hook.mode, hook.rec, hook.sub = "record", {}, {}
        run(b)
        per.append({k: v for k, v in hook.rec.items() if k[0] < nD})
    avg_d = {k: (per[0][k] + per[1][k]) * 0.5 for k in per[0]}
    per = []
    for b in shards:                                   # phase 2: G gradients given the averaged D update
        hook.mode, hook.rec, hook.sub = "record", {}, dict(avg_d)
        run(b)
        per.append({k: v for k, v in hook.rec.items() if k[0] == nD})
    avg_g = {k: (per[0][k] + per[1][k]) * 0.5 for k in per[0]}
    hook.mode, hook.rec, hook.sub = "off", {}, {**avg_d, **avg_g}
    losses = run(shards[0])                            # phase 3: what rank 0 must end up with
    emu = tr.snapshot()
    ref = {"buckets": [{k: v.to(dev) for k, v in bk.items()} for bk in real["snap"]["buckets"]],
           "buffers": [[t.to(dev) for t in l] for l in real["snap"]["buffers"]]}
    d, bitwise = snapshot_diff(emu, ref)
    assert d <= 1e-6, (d, bitwise)
    assert rel(losses, real["losses"].to(dev)) <= 1e-6
    # the emulation really exchanged something: rank 0 alone (no averaging) ends elsewhere
    hook.sub = {}
    run(shards[0])
    d_alone, _ = snapshot_diff(tr.snapshot(), ref)
    assert d_alone > 1e-4, d_alone
    print(f"2-rank step vs mean-gradient emulation: max rel diff {d:.3e} (bitwise {bitwise}); without averaging {d_alone:.3e}")
