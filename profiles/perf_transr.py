"""TransR training step: the group kernel (loss_step_corrupt) vs the generic kernels (rank_loss + backward)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "joint-kg-recommender_b200")]
import torch
import bench
import kgrec_b200 as K
dev = torch.device("cuda:0")
gen = torch.Generator().manual_seed(1)
def t(fn, reps=5):
    fn(); fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps
for nb, n_rel in ((32, 500), (32, 20), (1, 500), (1, 20)):
    ix = [x.to(dev) for x in bench.make_indices(torch, gen, nb)]
    pos, corrupt = (ix[0], ix[1], ix[2] % n_rel), ix[3]
    rep = lambda x: x.view(-1, 1).expand(-1, 10).reshape(-1)
    neg = (torch.where(corrupt < 0, ~corrupt, rep(pos[0])), torch.where(corrupt >= 0, corrupt, rep(pos[1])), rep(pos[2]).contiguous())
    n_tri = pos[0].numel() * 11
    m = K.TransRModel(False, 100, 100_000, n_rel)
    m.grad_mode = "sparse"
    def step():
        m.zero_grad(set_to_none=True)
        m.loss_step_corrupt(pos, corrupt, margin=1.0, batch_pos=1024)
    def generic():
        m.zero_grad(set_to_none=True)
        l, _, _ = m.rank_loss(pos, neg, margin=1.0, batch_pos=1024)
        l.sum().backward()
    a = t(step)
    b = t(generic) if nb == 32 and n_rel == 500 else float("nan")
    print(f"batches {nb:3d} relations {n_rel:4d}: group step {a:.3f} ms ({n_tri / a * 1e3:.3g} triples/s)   generic fwd+bwd: {b:.3f} ms")
# the whole training step through the optimizer (clip + sparse-row Adagrad; the d x d matrices are swept in segments)
from kgrec_b200.optim import SparseRowOptimizer
ix = [x.to(dev) for x in bench.make_indices(torch, gen, 32)]
m = K.TransRModel(False, 100, 100_000, 500)
opt = SparseRowOptimizer(m, optimizer_type="Adagrad", lr=0.01, clip=5.0)
a = t(lambda: opt.step_corrupt(tuple(ix[:3]), ix[3], margin=1.0, batch_pos=1024))
print(f"optimizer step, batches 32 relations 500: {a:.3f} ms")
