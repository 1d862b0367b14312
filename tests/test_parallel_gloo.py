"""Multi-rank host logic on CPU (gloo, world_size 2): per-flow gradient buckets are reduced as soon
as each flow's backward finishes, gradients end up as the cross-rank mean, utterance sharding has no
overlap.  The CUDA kernels are not involved (tiny stand-in flows built from nn.Linear)."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from torch import nn

from constant_memory_waveglow_b200.parallel import FlowGradSync, flow_buckets, shard_utterances


class ToyFlowModel(nn.Module):
    def __init__(self, flows=3, width=5):
        super().__init__()
        self.upsampler = nn.Linear(width, width)
        self.invconv1x1 = nn.ModuleList(nn.Linear(width, width, bias=False) for _ in range(flows))
        self.WNs = nn.ModuleList(nn.Sequential(nn.Linear(width, width), nn.Tanh(), nn.Linear(width, width))
                                 for _ in range(flows))

    def forward(self, x):
        y = self.upsampler(x)
        for c, w in zip(self.invconv1x1, self.WNs):
            x = c(x)
            x = x + w(x) * y
        return x.pow(2).mean()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out, mode="overlap"):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        model = ToyFlowModel()
        ref = ToyFlowModel()
        ref.load_state_dict(model.state_dict())
        xs = [torch.randn(4, 5, generator=torch.Generator().manual_seed(100 + r)) for r in range(world)]
        # expected: mean over ranks of the local gradients
        expect = None
        for r in range(world):
            ref.zero_grad()
            ref(xs[r]).backward()
            g = [p.grad.clone() for p in ref.parameters()]
            expect = g if expect is None else [a + b for a, b in zip(expect, g)]
        expect = [g / world for g in expect]

        buckets = flow_buckets(model)
        assert len(buckets) == 4 and len(buckets[0]) == 5       # flow 2 first, upsampler last
        sync = FlowGradSync(buckets, mode=mode)
        assert sync.whole is not None and all(f.data_ptr() >= sync.whole.data_ptr() for f in sync.flat)
        for step in range(2):
            sync.zero_grad()
            model(xs[rank]).backward()
            sync.finish()
            # buckets are launched in backward-completion order: last flow first, upsampler last
            assert sync.launch_order == [0, 1, 2, 3], sync.launch_order
            for p, e in zip(model.parameters(), expect):
                assert torch.allclose(p.grad, e, atol=1e-6), (step, rank)
        # gradients are views of the flat communication buffers (no copies)
        p0 = buckets[0][0]
        assert p0.grad.data_ptr() == sync.flat[0].data_ptr()
        out[rank] = 1
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["overlap", "deferred"])   # per-flow all-reduces during the backward / one at its end
def test_flow_grad_sync_two_ranks_gloo(mode):
    world = 2
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, out, mode), nprocs=world, join=True)
    assert dict(out) == {0: 1, 1: 1}


def test_single_process_buckets_and_sharding():
    model = ToyFlowModel(flows=2)
    sync = FlowGradSync(flow_buckets(model))
    sync.zero_grad()
    model(torch.randn(3, 5)).backward()
    sync.finish()
    assert sync.launch_order == [0, 1, 2]
    assert all(p.grad is not None and p.grad.abs().sum() > 0 for p in model.parameters())
    shards = [shard_utterances(10, r, 4) for r in range(4)]
    assert sorted(sum(shards, [])) == list(range(10))
    assert shards[0] == [0, 4, 8] and shards[3] == [3, 7]


# ---- the Lightning-free Trainer under two ranks (train.py:51-53,73-78 gets this from Lightning's DDPPlugin) ----
class _ToyLit:
    """A LightningModule over the toy flow: what Trainer.fit needs from LightModel, without CUDA kernels."""

    @staticmethod
    def build(n_items):
        from constant_memory_waveglow_b200 import trainer as TR
        from torch.utils.data import DataLoader, TensorDataset

        class Lit(TR.LightningModule):
            def __init__(self):
                super().__init__()
                self.model = ToyFlowModel()
                self.seen = []

            def configure_optimizers(self):
                return torch.optim.SGD(self.parameters(), lr=0.05)

            def train_dataloader(self):
                data = torch.arange(n_items, dtype=torch.float32).unsqueeze(1).repeat(1, 5) / n_items
                return DataLoader([row for row in data], batch_size=2, shuffle=False)

            def training_step(self, batch, batch_idx):
                self.seen.extend(int(round(v * n_items)) for v in batch[:, 0].tolist())
                loss = self.model(batch)
                self.log("loss", loss.detach(), sync_dist=True)
                return loss

        return Lit()


def _trainer_worker(rank, world, port, root, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank),
                      LOCAL_RANK=str(rank))
    from constant_memory_waveglow_b200 import trainer as TR
    try:
        torch.manual_seed(0)
        lit = _ToyLit.build(12)
        tr = TR.Trainer(max_epochs=2, default_root_dir=root, log_every_n_steps=1)
        tr.fit(lit)
        assert dist.is_initialized() and dist.get_world_size() == world
        # every rank saw its own half of the data set each epoch (DistributedSampler), 3 steps of 2 items per epoch
        assert tr.global_step == 6 and len(lit.seen) == 12
        assert sorted(set(lit.seen)) == list(range(rank, 12, world))
        flat = torch.cat([p.detach().flatten() for p in lit.parameters()])
        gathered = [torch.zeros_like(flat) for _ in range(world)]
        dist.all_gather(gathered, flat)
        assert torch.equal(gathered[0], gathered[1])          # averaged gradients: replicas stay identical
        if rank == 0:
            assert tr.last_checkpoint and os.path.exists(tr.last_checkpoint)
            assert os.path.exists(os.path.join(tr.logger.log_dir, "metrics.csv"))
        else:
            assert tr.logger is None
        out[rank] = 1
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def test_trainer_two_ranks_gloo(tmp_path, monkeypatch):
    # the ranks are CPU processes on any machine: with a GPU visible Trainer.fit would give each rank a device of its own
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    world = 2
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_trainer_worker, args=(world, port, str(tmp_path), out), nprocs=world, join=True)
    assert dict(out) == {0: 1, 1: 1}
