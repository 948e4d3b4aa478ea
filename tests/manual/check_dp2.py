"""2-GPU check (torchrun --nproc-per-node 2): the all-reduced gradient equals the mean of the two ranks' single-GPU
gradients, and both ranks hold identical parameters after a data-parallel optimiser step."""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import motifs_jl_b200 as mb
from motifs_jl_b200 import model as mdl, parallel, synth

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
ctx = mb.Context(local)
hp = mdl.Hyperparam()
a = synth.planted_gapped(240, 100, 3)
seqs = ctx.seqs_from_ascii(a)
cdl = mdl.ucdl(hp, np.random.default_rng(5))
m = mb._lib.CscModel(ctx, hp, 100)
m.set_params(cdl.flat)
idx_all = np.random.default_rng(7).permutation(240)[:12]
_, g_own = m.loss_grad(seqs, idx_all[6 * rank: 6 * rank + 6])
# data-parallel step through the same calls train_ucdl makes
side = torch.cuda.Stream(device=dev)
ctx.set_stream(side.cuda_stream)
with torch.cuda.stream(side):
    _, gptr = m.device_ptrs()
    gview = torch.as_tensor(mdl._DevArray(gptr, m.n_total), device=dev)
    m.step_begin(seqs, idx_all[6 * rank: 6 * rank + 6])
    parallel.all_reduce_mean_(gview)
    g_avg = gview.cpu().numpy()[: m.n_trainable].copy()
    loss, l1 = m.adabelief_step()
torch.cuda.synchronize()
ctx.set_stream(None)
both = [torch.zeros(m.n_trainable, device=dev) for _ in range(world)]
dist.all_gather(both, torch.from_numpy(g_own).to(dev))
mean = torch.stack(both).mean(0).cpu().numpy()
p = torch.from_numpy(m.get_params()).to(dev)
ps = [torch.zeros_like(p) for _ in range(world)]
dist.all_gather(ps, p)
if rank == 0:
    err = np.abs(g_avg - mean).max() / np.abs(mean).max()
    same = bool(torch.equal(ps[0], ps[1]))
    print(f"dp2: max |allreduced - mean of single-GPU grads| / max|grad| = {err:.2e}; parameters identical on both ranks: {same}")
    assert err < 1e-6 and same
dist.destroy_process_group()
