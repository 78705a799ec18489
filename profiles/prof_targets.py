"""One small workload per kernel, for `ncu -k regex:<kernel>` captures (round 2).
    python profiles/prof_targets.py <target> [reps]
targets: transr_step step_e100k step_e500k step_e5m eval_d128 eval_h_d128 opt transr_eval tup_step gumbel_eval soft_eval_d128"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "joint-kg-recommender_b200")]
import torch
import kgrec_b200 as K
from kgrec_b200.models.base import device_init
target = sys.argv[1]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 4
dev = torch.device("cuda:0")
g = torch.Generator().manual_seed(3)
D, NB, B, KN = 100, 256, 1024, 10


def kg_ids(E, R=500, kn=KN):
    n = NB * B
    ph, pt = (torch.randint(0, E, (n,), generator=g, dtype=torch.int32).to(dev) for _ in range(2))
    pr = torch.randint(0, R, (n,), generator=g, dtype=torch.int32).to(dev)
    c = torch.randint(0, E, (n * kn,), generator=g, dtype=torch.int32)
    c = torch.where(torch.rand(n * kn, generator=g) < 0.5, ~c, c).to(dev)
    return (ph, pt, pr), c


if target.startswith("step_"):
    E = {"step_e100k": 100_000, "step_e500k": 500_000, "step_e5m": 5_000_000}[target]
    with device_init(dev):
        m = K.TransEModel(False, D, E, 500)
    m.grad_mode = "sparse"
    sets = [kg_ids(E) for _ in range(2)]
    for i in range(reps):
        m.zero_grad(set_to_none=True)
        m.loss_step_corrupt(sets[i % 2][0], sets[i % 2][1], margin=1.0, batch_pos=B)
elif target == "transr_step":
    with device_init(dev):
        m = K.TransRModel(False, D, 100_000, 500)
    m.grad_mode = "sparse"
    NB = 32
    pos, c = kg_ids(100_000)
    for i in range(reps):
        m.zero_grad(set_to_none=True)
        m.loss_step_corrupt(pos, c, margin=1.0, batch_pos=B)
elif target in ("eval_d128", "eval_h_d128"):
    with device_init(dev):
        m = (K.TransEModel if target == "eval_d128" else K.TransHModel)(False, 128, 5_000_000, 500)
    q = torch.randint(0, 5_000_000, (2048,), generator=g).to(dev)
    r = torch.randint(0, 500, (2048,), generator=g).to(dev)
    for i in range(reps):
        m.topk("tail", q, r, k=10)
elif target == "opt":
    from kgrec_b200.optim import SparseRowOptimizer
    m = K.TransEModel(False, D, 100_000, 500)
    opt = SparseRowOptimizer(m, "Adagrad", lr=0.01, clip=5.0)
    sets = [kg_ids(100_000) for _ in range(2)]
    for i in range(reps):
        opt.step_corrupt(sets[i % 2][0], sets[i % 2][1], margin=1.0, batch_pos=B)
elif target == "transr_eval":
    with device_init(dev):
        m = K.TransRModel(False, D, 1_000_000, 500)
    q = torch.randint(0, 1_000_000, (1024,), generator=g).to(dev)
    r = torch.randint(0, 8, (1024,), generator=g).to(dev)
    for i in range(reps):
        m.topk("tail", q, r, k=10)
elif target == "tup_step":
    with device_init(dev):
        m = K.TransUPModel(False, D, 50_000, 50_000, 20, True)
    m.grad_mode = "sparse"
    n = NB * B
    u, pi, ni = (torch.randint(0, 50_000, (n,), generator=g, dtype=torch.int32).to(dev) for _ in range(3))
    for i in range(reps):
        m.zero_grad(set_to_none=True)
        m.loss_step((u, pi), (u, ni), target=-1.0, batch_pos=B)
elif target in ("tup_soft_opt", "ktup_soft_opt", "tup_gumbel_opt"):
    from kgrec_b200.optim import SparseRowOptimizer
    import numpy as np
    n = NB * B
    if target in ("tup_soft_opt", "tup_gumbel_opt"):
        with device_init(dev):
            m = K.TransUPModel(False, D, 50_000, 50_000, 20, target == "tup_gumbel_opt")
        nu_, ni_ = 50_000, 50_000
    else:
        nu_, ni_, ne_ = 6040, 3706, 500_000
        ents = np.random.RandomState(0).permutation(ne_)[:ni_]
        new_map = {i: (int(ents[i]) if i % 10 < 7 else -1, i) for i in range(ni_)}
        with device_init(dev):
            m = K.jTransUPModel(False, D, nu_, ni_, ne_, 20, {i: i for i in range(ni_)}, new_map, False, False)
    opt = SparseRowOptimizer(m, "Adagrad", lr=0.005, clip=5.0)
    u = torch.randint(0, nu_, (n,), generator=g, dtype=torch.int32).to(dev)
    pi, ni = (torch.randint(0, ni_, (n,), generator=g, dtype=torch.int32).to(dev) for _ in range(2))
    for i in range(reps):
        opt.step_pairs((u, pi), (u, ni), target=-1.0, batch_pos=B, reg=True)
elif target in ("gumbel_eval", "soft_eval_d128"):
    gum = target == "gumbel_eval"
    d = 100 if gum else 128
    n_it = 50_000 if gum else 1_000_000
    with device_init(dev):
        m = K.TransUPModel(False, d, 50_000, n_it, 20, gum)
    qu = torch.arange(1024 if gum else 4096, device=dev) % 50_000
    cat = None if gum else m.soft_catalog()
    for i in range(reps):
        m.topk_items(qu, k=10) if gum else m.topk_items(qu, k=10, soft_catalog=cat)
torch.cuda.synchronize()
print("done", target)
