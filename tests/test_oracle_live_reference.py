"""Pin the numpy oracle against the reference ITSELF at shapes the other goldens do not reach.

The goldens of test_oracle_golden.py are d=20 / 37 entities / 9 triples plus one BASELINE configs[1] shape.
Here the unmodified reference classes were instantiated on the CPU at a grid of embedding sizes --
including the BASELINE ones, d=100 and d=128, and an odd size -- with the reference drivers' call pattern
(positives repeated per negative, utils/data.py:12-56 -> knowledge_representation.py:187-205), and what
their forward / autograd / evaluate* / ranking helpers produced is stored in ``tests/golden/live_*.npz``
(recorded by ``tests/golden/make_golden_live.py``).  Every quantity the GPU parity tests take from the
oracle is compared with it:

    scores, margin / BPR loss, dense table gradients, full-catalog score matrices (head and tail),
    ST-Gumbel with the reference's own uniform draw captured by re-seeding, the regularisers,
    getRecPerformance / getKGPerformance with and without filters.

The inputs are regenerated here from their seeds; the tables come from this package's constructors, which
draw exactly what the reference constructors draw for the same seed, and each table is checked against a
fingerprint of the reference's before it is used.  Arrays too large to store whole are kept as a fixed,
seeded sample of entries plus their L2 norm and largest magnitude (``summarize``).

CPU only.  Test infrastructure: nothing under ``oracle/`` is imported by the product.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import kg_oracle as O

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

pytestmark = pytest.mark.filterwarnings("ignore")

FULL_MAX = 256          # arrays up to this many entries are stored whole
N_SAMPLE = 64           # entries kept of a larger array


def npy(t):
    return t.detach().cpu().numpy().copy()


def close(a, b, rtol=3e-5, atol=3e-6):
    np.testing.assert_allclose(np.asarray(a, np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol)


# ---------------------------------------------------------------------------------------------
# shared with tests/golden/make_golden_live.py: inputs, table perturbation and the stored summary
# ---------------------------------------------------------------------------------------------
def perturb_noise(shapes, seed, scale=0.05):
    """Noise that moves the tables off their initial unit rows (trained tables are not normalised),
    drawn table by table in sorted name order."""
    g = torch.Generator().manual_seed(seed)
    return {k: scale * torch.randn(shapes[k], generator=g) for k in sorted(shapes)}


def summarize(prefix, x):
    """What is stored of the reference array `x` under `prefix`: the whole array when small, else a seeded
    sample of entries (half of them among the non-zeros, so that sparse gradients are sampled where they
    carry information) with the array's L2 norm and largest magnitude."""
    x = np.asarray(x, np.float32)
    out = {prefix + "#shape": np.asarray(x.shape, np.int64)}
    if x.size <= FULL_MAX:
        out[prefix] = x
        return out
    flat = x.reshape(-1)
    rng = np.random.RandomState(x.size % 100_003)
    nz = np.flatnonzero(flat)
    pick = rng.choice(nz, min(N_SAMPLE // 2, nz.size), replace=False) if nz.size else np.zeros(0, np.int64)
    rest = rng.choice(flat.size, N_SAMPLE - pick.size, replace=False)
    idx = np.unique(np.concatenate([pick, rest])).astype(np.int64)
    out.update({prefix + "#idx": idx, prefix + "#val": flat[idx],
                prefix + "#l2": np.float64(np.linalg.norm(flat.astype(np.float64))),
                prefix + "#amax": np.float64(np.abs(flat).max())})
    return out


def fingerprint(prefix, w):
    """A table as stored for the check that the regenerated one is the reference's: the first entries of
    three rows, and the sum and sum of squares of the whole table."""
    w = np.asarray(w, np.float32)
    rows = np.unique([0, w.shape[0] // 2, w.shape[0] - 1])
    w64 = w.astype(np.float64)
    return {prefix + "_rows": w[rows, :16], prefix + "_sums": np.asarray([w64.sum(), (w64 * w64).sum()])}


def pack(d):
    """{key: array} as a few flat buffers and a JSON index (one zip member per key would cost more than the data)."""
    bufs, index = {"f4": [], "f8": [], "i8": []}, {}
    size = {"f4": 0, "f8": 0, "i8": 0}
    for k in sorted(d):
        a = np.asarray(d[k])
        kind = "f4" if a.dtype == np.float32 else "f8" if a.dtype.kind == "f" else "i8"
        flat = a.reshape(-1).astype(kind)
        index[k] = [kind, size[kind], list(a.shape)]
        bufs[kind].append(flat)
        size[kind] += flat.size
    out = {kind: (np.concatenate(v) if v else np.zeros(0, kind)) for kind, v in bufs.items()}
    out["index"] = np.asarray(json.dumps(index, sort_keys=True))
    return out


def unpack(z):
    index = json.loads(str(z["index"]))
    return {k: z[kind][off:off + int(np.prod(shape, dtype=np.int64))].reshape(shape) for k, (kind, off, shape) in index.items()}


def kg_key(model, d, n_ent, n_rel, n_pos, k_neg, l1):
    return "%s_d%d_e%d_r%d_p%d_k%d_%s" % (model, d, n_ent, n_rel, n_pos, k_neg, "l1" if l1 else "l2")


def kg_inputs(d, n_ent, n_rel, n_pos, k_neg):
    rng = np.random.RandomState(d * 7 + n_pos)
    ph, pt, pr = rng.randint(0, n_ent, n_pos), rng.randint(0, n_ent, n_pos), rng.randint(0, n_rel, n_pos)
    # the drivers' batch: every positive repeated k_neg times against head- or tail-corrupted negatives
    rh, rt, rr = np.repeat(ph, k_neg), np.repeat(pt, k_neg), np.repeat(pr, k_neg)
    head = rng.rand(n_pos * k_neg) < 0.5
    cor = rng.randint(0, n_ent, n_pos * k_neg)
    nh, nt = np.where(head, cor, rh), np.where(head, rt, cor)
    q, qr = rng.randint(0, n_ent, 5), rng.randint(0, n_rel, 5)
    return rh, rt, rr, nh, nt, q, qr


def tup_key(d, n_user, n_item, n_pref, n_pos, gumbel, l1):
    return "tup_d%d_u%d_i%d_p%d_n%d_%s_%s" % (d, n_user, n_item, n_pref, n_pos, "gumbel" if gumbel else "soft", "l1" if l1 else "l2")


def tup_inputs(d, n_user, n_item, n_pos):
    rng = np.random.RandomState(d + n_pos)
    u, pi, ni = rng.randint(0, n_user, n_pos), rng.randint(0, n_item, n_pos), rng.randint(0, n_item, n_pos)
    qu = rng.randint(0, n_user, 3)
    return u, pi, ni, qu


def ktup_key(d, n_user, n_item, n_ent, n_rel, n_pos, gumbel, l1):
    return "ktup_d%d_u%d_i%d_e%d_r%d_n%d_%s_%s" % (d, n_user, n_item, n_ent, n_rel, n_pos, "gumbel" if gumbel else "soft",
                                                  "l1" if l1 else "l2")


def ktup_inputs(d, n_user, n_item, n_ent, n_rel, n_pos):
    rng = np.random.RandomState(d + n_rel)
    aligned = rng.rand(n_item) < 0.7
    ents = rng.permutation(n_ent)[:n_item]
    i_map = {i: i for i in range(n_item)}
    new_map = {i: ((int(ents[i]) if aligned[i] else -1), i) for i in range(n_item)}
    u, pi, ni = rng.randint(0, n_user, n_pos), rng.randint(0, n_item, n_pos), rng.randint(0, n_item, n_pos)
    ph, pt, nt = rng.randint(0, n_ent, n_pos), rng.randint(0, n_ent, n_pos), rng.randint(0, n_ent, n_pos)
    pr = rng.randint(0, n_rel, n_pos)
    qu = rng.randint(0, n_user, 3)
    q, qr = rng.randint(0, n_ent, 4), rng.randint(0, n_rel, 4)
    return dict(i_map=i_map, new_map=new_map, u=u, pi=pi, ni=ni, ph=ph, pt=pt, nt=nt, pr=pr, qu=qu, q=q, qr=qr)


def regulariser_inputs():
    """utils/loss.py:18-23 inputs: rows on both sides of the unit sphere."""
    g = torch.Generator().manual_seed(3)
    out = []
    for d, n in ((100, 64), (128, 33), (10, 7)):
        rows = torch.randn(n, d, generator=g) * torch.linspace(0.5, 1.6, n).view(-1, 1) / d ** 0.5
        rel = torch.randn(n, d, generator=g) * 0.2
        nrm = torch.randn(n, d, generator=g) * 0.2
        out.append((d, rows, rel, nrm))
    return out


def ranking_inputs():
    """getRecPerformance / getKGPerformance (utils/misc.py:125-146, 213-248) inputs: random tie-free rows."""
    rng = np.random.RandomState(12)
    out = []
    for c in range(40):
        n = int(rng.randint(15, 400))
        topn = int(rng.choice([1, 5, 10, 20]))
        scores = (rng.permutation(n).astype(np.float32) + 1.0) / 3.0
        gold = set(int(x) for x in rng.choice(n, int(rng.randint(1, 6)), replace=False))
        filt = (set(int(x) for x in rng.choice(n, int(rng.randint(0, n // 3 + 1)), replace=False)) - gold) if c % 3 else None
        out.append((scores, gold, filt, topn))
    return out


# ---------------------------------------------------------------------------------------------
# checks against the stored reference values
# ---------------------------------------------------------------------------------------------
_cache = {}


def golden(name):
    if name not in _cache:
        with np.load(os.path.join(GOLDEN, name + ".npz")) as z:
            _cache[name] = unpack(z)
    return _cache[name]


def check(g, prefix, got, rtol, atol):
    """`got` (the oracle's full array) against what summarize() stored of the reference's."""
    got = np.asarray(got, np.float64)
    assert tuple(got.shape) == tuple(g[prefix + "#shape"]), (prefix, got.shape, g[prefix + "#shape"])
    if prefix in g:
        close(got, g[prefix], rtol=rtol, atol=atol)
        return
    flat = got.reshape(-1)
    close(flat[g[prefix + "#idx"]], g[prefix + "#val"], rtol=rtol, atol=atol)
    close(np.linalg.norm(flat), g[prefix + "#l2"], rtol=max(rtol, 1e-5), atol=atol)
    close(np.abs(flat).max(), g[prefix + "#amax"], rtol=rtol, atol=atol)


def grad_atol(g, prefix, factor):
    """The tolerance of a gradient table: factor x max(1, largest magnitude of the reference's)."""
    amax = g[prefix + "#amax"] if prefix + "#amax" in g else np.abs(g[prefix]).max(initial=0.0)
    return factor * max(1.0, float(amax))


def regenerated_tables(m, seed, g, zero_last_ent=False):
    """The package model's initial tables (same draws as the reference constructor), moved by the same noise
    as the recorded reference model, checked against the reference's fingerprint."""
    W = {k.replace("_embeddings.weight", ""): v.detach().cpu().clone() for k, v in m.state_dict().items()}
    noise = perturb_noise({k: tuple(v.shape) for k, v in W.items()}, seed)
    W = {k: (v + noise[k]).numpy() for k, v in W.items()}
    if zero_last_ent:
        W["ent"][-1] = 0.0                     # the padding row stays zero (jTransUP.py:83-94)
    for k, w in W.items():
        want = fingerprint("w_" + k, w)
        for part in ("_rows", "_sums"):
            assert np.array_equal(want["w_" + k + part], g["w_" + k + part]), "table %s differs from the reference's" % k
    return W


KG_ORACLE = {
    "transe": (("ent", "rel"), O.transe_score, O.transe_eval, O.transe_grads, "TransEModel"),
    "transh": (("ent", "rel", "norm"), O.transh_score, O.transh_eval, O.transh_grads, "TransHModel"),
    "transr": (("ent", "rel", "proj"), O.transr_score, O.transr_eval, O.transr_grads, "TransRModel"),
}

KG_CASES = [
    ("transe", 100, 3000, 50, 64, 10),      # BASELINE configs[1] row width and negatives per positive
    ("transe", 128, 500, 7, 33, 3),         # configs[4] row width
    ("transe", 50, 211, 5, 17, 1),          # d % 4 != 0: the kernels' scalar path is checked against the same oracle
    ("transh", 100, 2000, 40, 48, 10),
    ("transh", 64, 300, 9, 21, 4),
    ("transr", 100, 600, 12, 24, 10),
    ("transr", 32, 150, 4, 19, 2),
]
TUP_CASES = [(100, 300, 400, 20, 40), (128, 90, 70, 7, 23), (36, 50, 60, 3, 11)]
KTUP_CASES = [(100, 120, 200, 500, 20, 32), (24, 40, 55, 90, 4, 13)]


@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("model,d,n_ent,n_rel,n_pos,k_neg", KG_CASES)
def test_kg_models_live(model, d, n_ent, n_rel, n_pos, k_neg, l1):
    import kgrec_b200 as K
    g = golden("live_kg")
    key = kg_key(model, d, n_ent, n_rel, n_pos, k_neg, l1)
    g = {k[len(key) + 1:]: v for k, v in g.items() if k.startswith(key + "/")}
    names, score, evalf, grads, cls = KG_ORACLE[model]
    torch.manual_seed(1000 + d + n_pos)
    W = regenerated_tables(getattr(K, cls)(L1_flag=l1, embedding_size=d, ent_total=n_ent, rel_total=n_rel), 5, g)
    T = tuple(W[k] for k in names)
    rh, rt, rr, nh, nt, q, qr = kg_inputs(d, n_ent, n_rel, n_pos, k_neg)
    op, on = score(*T, rh, rt, rr, l1), score(*T, nh, nt, rr, l1)
    check(g, "pos", op, 3e-5, 3e-6)
    check(g, "neg", on, 3e-5, 3e-6)
    close(O.margin_loss(op, on, 1.0), g["loss"], rtol=1e-5)
    gp, gn = O.margin_loss_grads(op, on, 1.0)
    a, b = grads(*T, rh, rt, rr, l1, gp), grads(*T, nh, nt, rr, l1, gn)
    assert set(a) == set(names)
    for k in a:
        check(g, "grad_" + k, a[k] + b[k], 2e-4, grad_atol(g, "grad_" + k, 2e-5))
    check(g, "eval_head", evalf(*T, q, qr, l1, "head"), 1e-4, 1e-5)
    check(g, "eval_tail", evalf(*T, q, qr, l1, "tail"), 1e-4, 1e-5)


def _draw(seed, shape):
    """What `logits.data.new(*logits.size()).uniform_()` (transUP.py:84-102) returns after this re-seed."""
    torch.manual_seed(seed)
    return npy(torch.empty(*shape).uniform_())


@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("gumbel", [False, True])
@pytest.mark.parametrize("d,n_user,n_item,n_pref,n_pos", TUP_CASES)
def test_tup_live(d, n_user, n_item, n_pref, n_pos, gumbel, l1):
    import kgrec_b200 as K
    key = tup_key(d, n_user, n_item, n_pref, n_pos, gumbel, l1)
    g = {k[len(key) + 1:]: v for k, v in golden("live_tup").items() if k.startswith(key + "/")}
    torch.manual_seed(77 + d)
    m = K.TransUPModel(L1_flag=l1, embedding_size=d, user_total=n_user, item_total=n_item, preference_total=n_pref,
                       use_st_gumbel=gumbel)
    W = regenerated_tables(m, 6, g)
    T = (W["user"], W["item"], W["pref"], W["pref_norm"])
    u, pi, ni, qu = tup_inputs(d, n_user, n_item, n_pos)
    s1, s2, s3 = 901, 902, 903
    n1 = _draw(s1, (n_pos, n_pref)) if gumbel else None
    n2 = _draw(s2, (n_pos, n_pref)) if gumbel else None
    op, on = O.tup_score(*T, u, pi, l1, n1), O.tup_score(*T, u, ni, l1, n2)
    check(g, "pos", op, 1e-4, 1e-5)
    check(g, "neg", on, 1e-4, 1e-5)
    close(O.bpr_loss(op, on, -1.0), g["loss"], rtol=1e-4)
    gp, gn = O.bpr_loss_grads(op, on, -1.0)
    a, b = O.tup_grads(*T, u, pi, l1, gp, n1), O.tup_grads(*T, u, ni, l1, gn, n2)
    assert set(a) == {"user", "item", "pref", "pref_norm"}
    for k in a:
        check(g, "grad_" + k, a[k] + b[k], 5e-4, grad_atol(g, "grad_" + k, 5e-5))
    n3 = _draw(s3, (3, n_item, n_pref)) if gumbel else None
    check(g, "eval", O.tup_eval(*T, qu, l1, n3), 2e-4, 2e-5)


@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("gumbel", [False, True])
@pytest.mark.parametrize("d,n_user,n_item,n_ent,n_rel,n_pos", KTUP_CASES)
def test_ktup_live(d, n_user, n_item, n_ent, n_rel, n_pos, gumbel, l1):
    import kgrec_b200 as K
    key = ktup_key(d, n_user, n_item, n_ent, n_rel, n_pos, gumbel, l1)
    g = {k[len(key) + 1:]: v for k, v in golden("live_ktup").items() if k.startswith(key + "/")}
    x = ktup_inputs(d, n_user, n_item, n_ent, n_rel, n_pos)
    torch.manual_seed(31 + d)
    m = K.jTransUPModel(l1, d, n_user, n_item, n_ent, n_rel, x["i_map"], x["new_map"], False, gumbel)
    W = regenerated_tables(m, 8, g, zero_last_ent=True)
    item2ent = O.ktup_item2ent(x["i_map"], x["new_map"], n_item, n_ent)
    T = (W["user"], W["item"], W["ent"], W["rel"], W["norm"], W["pref"], W["pref_norm"], item2ent)
    u, pi, ni = x["u"], x["pi"], x["ni"]
    s1, s2, s3 = 41, 42, 43
    n1 = _draw(s1, (n_pos, n_rel)) if gumbel else None
    n2 = _draw(s2, (n_pos, n_rel)) if gumbel else None
    op, on = O.ktup_rec_score(*T, u, pi, l1, n1), O.ktup_rec_score(*T, u, ni, l1, n2)
    check(g, "pos", op, 1e-4, 1e-5)
    check(g, "neg", on, 1e-4, 1e-5)
    gp, gn = O.bpr_loss_grads(op, on, -1.0)
    a, b = O.ktup_rec_grads(*T, u, pi, l1, gp, n1), O.ktup_rec_grads(*T, u, ni, l1, gn, n2)
    for k in a:
        check(g, "grad_" + k, a[k] + b[k], 5e-4, grad_atol(g, "grad_" + k, 5e-5))
    # KG branch of the joint model == TransH on its ent / rel / norm tables (jTransUP.py:144-157)
    ph, pt, nt, pr = x["ph"], x["pt"], x["nt"], x["pr"]
    H = (W["ent"], W["rel"], W["norm"])
    okp, okn = O.transh_score(*H, ph, pt, pr, l1), O.transh_score(*H, ph, nt, pr, l1)
    check(g, "kg_pos", okp, 3e-5, 3e-6)
    check(g, "kg_neg", okn, 3e-5, 3e-6)
    gp, gn = O.margin_loss_grads(okp, okn, 1.0)
    a, b = O.transh_grads(*H, ph, pt, pr, l1, gp), O.transh_grads(*H, ph, nt, pr, l1, gn)
    for k in a:
        check(g, "kg_grad_" + k, a[k] + b[k], 2e-4, 2e-5)
    n3 = _draw(s3, (3, n_item, n_rel)) if gumbel else None
    check(g, "eval_rec", O.ktup_rec_eval(*T, x["qu"], l1, n3), 2e-4, 2e-5)
    check(g, "eval_head", O.transh_eval(*H, x["q"], x["qr"], l1, "head"), 1e-4, 1e-5)
    check(g, "eval_tail", O.transh_eval(*H, x["q"], x["qr"], l1, "tail"), 1e-4, 1e-5)


def test_regularisers_live():
    """utils/loss.py:18-23 on rows on both sides of the unit sphere, values and autograd gradients."""
    g = golden("live_misc")
    for d, rows, rel, nrm in regulariser_inputs():
        p = "reg_d%d/" % d
        close(O.norm_loss(npy(rows)), g[p + "norm_loss"], rtol=1e-5)
        close(O.orthogonal_loss(npy(rel), npy(nrm)), g[p + "orth_loss"], rtol=1e-5)
        check({k[len(p):]: v for k, v in g.items() if k.startswith(p)}, "grad_rows", O.norm_loss_grads(npy(rows)), 1e-5, 1e-7)
        gr, gn = O.orthogonal_loss_grads(npy(rel), npy(nrm))
        check({k[len(p):]: v for k, v in g.items() if k.startswith(p)}, "grad_rel", gr, 1e-4, 1e-7)
        check({k[len(p):]: v for k, v in g.items() if k.startswith(p)}, "grad_norm", gn, 1e-4, 1e-7)


def test_ranking_live():
    """getRecPerformance / getKGPerformance (utils/misc.py:125-146, 213-248) on random tie-free rows."""
    g = golden("live_misc")
    for c, (scores, gold, filt, topn) in enumerate(ranking_inputs()):
        p = "rank_%d/" % c
        mine = O.rec_topk(scores, filt, topn)
        assert [int(x) for x in mine] == g[p + "top_ids"].tolist()
        close(O.rec_metrics(mine, gold), g[p + "rec_metrics"], rtol=1e-9, atol=1e-12)
        mine_kg = O.kg_ranks(scores, gold, filt, topn)       # {gold id: (hit, rank)}
        ids = g[p + "gold_ids"].tolist()
        assert sorted(mine_kg) == sorted(ids)
        assert [mine_kg[i][1] for i in ids] == g[p + "ranks"].tolist()
        assert [mine_kg[i][0] for i in ids] == g[p + "hits"].tolist()
