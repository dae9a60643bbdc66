"""Worker of tests/test_training_u8_gpu.py::test_ddp_u8_gradient_allreduce_two_gpus (one process per GPU, torchrun):
the stage-1 model under DistributedDataParallel fed with the loader's raw uint8 frames through forward(u8=...), the
path on which DDP prepares its gradient all-reduce."""
import os
import random
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
import torch.nn.functional as F

from sbl_for_multilingual_lip_reading_b200 import ops, stage1, synth
from sbl_for_multilingual_lip_reading_b200.video_frontend import random_crop_offsets

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
dist.init_process_group("nccl", device_id=dev)
ops.init()
n, t_in, t = 4, 29, 31
torch.manual_seed(7)
model = stage1.Stage1Classifier(n_layers_enc=3, dropout=0.0).to(dev).train()
model.load_synthetic(1, 3)
u8 = synth.synthetic_u8_clips(n, t_in, seed=500 + rank).to(dev)
crop = random_crop_offsets(n, t_in, rng=random.Random(rank))
flip = torch.tensor([(i + rank) % 2 == 0 for i in range(n)])
y = torch.randint(0, 1500, (n,), generator=torch.Generator().manual_seed(rank)).to(dev)
lang = torch.randint(0, 2, (n,), generator=torch.Generator().manual_seed(10 + rank)).to(dev)


def loss_of(m):
    torch.manual_seed(99)                       # same always-on dropout mask in both passes
    v_t, v_l = m(u8=u8, frames=t, crop=crop, flip=flip)
    return F.cross_entropy(v_t, y) + 0.1 * F.cross_entropy(v_l, lang)


# this shard's gradients without DDP
model.zero_grad()
loss_of(model).backward()
local = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
# the same step under DDP
ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[dev.index], broadcast_buffers=False)
model.zero_grad()
loss_of(ddp).backward()
ok = True
bad = []
for k, p in model.named_parameters():
    want = local[k].clone()
    dist.all_reduce(want)
    want /= world
    same = torch.equal(p.grad, want)
    g0 = p.grad.clone()
    dist.broadcast(g0, 0)
    same_ranks = torch.equal(g0, p.grad)       # every rank holds the same reduced gradient
    if not (same and same_ranks):
        bad.append((k, same, same_ranks, ((p.grad - want).norm() / (want.norm() + 1e-20)).item()))
    ok = ok and same and same_ranks
print(f"rank {rank}: ddp u8 gradient all-reduce {'OK' if ok else 'MISMATCH'} {bad[:4]}", flush=True)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
