"""GPU parity: the CUDA path (through the C ABI, via the drop-in modules) against
 (1) the golden vectors recorded from the reference classes, and
 (2) the numpy oracle on seeded random inputs at larger sizes.
Tolerance: 1e-4 relative in fp32 (BASELINE.json north_star); index sets exact."""
import numpy as np
import pytest
import torch

from oracle import kg_oracle as O

pytestmark = pytest.mark.gpu

RTOL = 1e-4


def dev():
    return torch.device("cuda:0")


def close(a, b, rtol=RTOL, atol=1e-5, max_outliers=0):
    """max_outliers: elements allowed outside the tolerance -- L1 gradients are sign(e) and a residual
    component within rounding of 0 may take either sign on the two sides."""
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    a, b = a.astype(np.float64), np.asarray(b, np.float64)
    if max_outliers:
        bad = np.abs(a - b) > atol + rtol * np.abs(b)
        if 0 < bad.sum() <= max_outliers:
            return
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def lt(x):
    return torch.as_tensor(np.asarray(x), dtype=torch.long, device=dev())


def load_weights(model, g):
    sd = {k[2:] + ".weight": torch.from_numpy(v) for k, v in g.items() if k.startswith("w_")}
    model.load_state_dict(sd)
    return model.cuda()


def dense(gr):
    return gr.to_dense() if gr.is_sparse else gr


@pytest.fixture(params=["auto", "force"])
def rec_engine(request, monkeypatch):
    """TUP / KTUP training calls run twice: size-based engine choice (small batches -> one warp
    per pair) and every call forced through the tile engine (csrc/train_rec_tile.cu)."""
    if request.param == "force":
        monkeypatch.setenv("KGREC_REC_TILE", "force")
    else:
        monkeypatch.delenv("KGREC_REC_TILE", raising=False)
    return request.param


def grads_by_name(model):
    return {n.replace(".weight", ""): dense(p.grad) for n, p in model.named_parameters() if p.grad is not None}


# ------------------------------------------------------------------------------------------
# (1) golden vectors from the reference classes
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["transe", "transh", "transr"])
@pytest.mark.parametrize("tag", ["l2", "l1"])
@pytest.mark.parametrize("grad_mode", ["dense", "sparse"])
def test_golden_kg(golden, name, tag, grad_mode):
    import kgrec_b200 as K
    g = golden(f"{name}_{tag}")
    cls = {"transe": K.TransEModel, "transh": K.TransHModel, "transr": K.TransRModel}[name]
    E, D = g["w_ent_embeddings"].shape
    m = load_weights(cls(bool(g["l1"]), D, E, g["w_rel_embeddings"].shape[0]), g)
    m.grad_mode = grad_mode
    pos = m(lt(g["ph"]), lt(g["pt"]), lt(g["pr"]))
    neg = m(lt(g["nh"]), lt(g["nt"]), lt(g["nr"]))
    close(pos, g["pos"])
    close(neg, g["neg"])
    # the reference's marginLoss written with stock ops, as the unchanged driver does
    loss = torch.clamp(pos - neg + float(g["margin"]), min=0).sum()
    close(loss, g["loss"])
    loss.backward()
    for k, v in grads_by_name(m).items():
        close(v, g["grad_" + k], rtol=2e-4, atol=2e-5)
    m.zero_grad()
    # fused ranking loss: same numbers from one launch
    fl, fp, fn = m.rank_loss((lt(g["ph"]), lt(g["pt"]), lt(g["pr"])), (lt(g["nh"]), lt(g["nt"]), lt(g["nr"])),
                             margin=float(g["margin"]))
    close(fp, g["pos"])
    close(fn, g["neg"])
    close(fl.sum(), g["loss"])
    fl.sum().backward()
    for k, v in grads_by_name(m).items():
        close(v, g["grad_" + k], rtol=2e-4, atol=2e-5)
    close(m.evaluateHead(lt(g["q"]), lt(g["qr"])), g["eval_head"])
    close(m.evaluateTail(lt(g["q"]), lt(g["qr"])), g["eval_tail"])
    m.check_indices()


@pytest.mark.parametrize("tag", ["l2", "l1"])
@pytest.mark.parametrize("mode", ["soft", "gumbel"])
@pytest.mark.parametrize("grad_mode", ["dense", "sparse"])
def test_golden_transup(golden, tag, mode, grad_mode, rec_engine):
    import kgrec_b200 as K
    g = golden(f"transup_{tag}_{mode}")
    U, D = g["w_user_embeddings"].shape
    m = load_weights(K.TransUPModel(bool(g["l1"]), D, U, g["w_item_embeddings"].shape[0],
                                    g["w_pref_embeddings"].shape[0], bool(g["gumbel"])), g)
    m.grad_mode = grad_mode
    npos = torch.from_numpy(g["noise_pos"]) if "noise_pos" in g else None
    nneg = torch.from_numpy(g["noise_neg"]) if "noise_neg" in g else None
    pos = m(lt(g["u"]), lt(g["pi"]), gumbel_u=npos)
    neg = m(lt(g["u"]), lt(g["ni"]), gumbel_u=nneg)
    close(pos, g["pos"])
    close(neg, g["neg"])
    loss = -torch.nn.functional.logsigmoid(float(g["target"]) * (pos - neg)).mean()
    close(loss, g["loss"])
    loss.backward()
    for k, v in grads_by_name(m).items():
        close(v, g["grad_" + k], rtol=5e-4, atol=2e-6)
    m.zero_grad()
    noise = torch.cat([npos, nneg]) if npos is not None else None
    fl, fp, fn = m.rank_loss((lt(g["u"]), lt(g["pi"])), (lt(g["u"]), lt(g["ni"])), target=float(g["target"]),
                             gumbel_u=noise)
    close(fp, g["pos"])
    close(fn, g["neg"])
    close(fl.sum(), g["loss"])
    fl.sum().backward()
    for k, v in grads_by_name(m).items():
        close(v, g["grad_" + k], rtol=5e-4, atol=2e-6)
    nev = torch.from_numpy(g["noise_eval"]) if "noise_eval" in g else None
    close(m.evaluate(lt(g["qu"]), gumbel_u=nev), g["eval"], rtol=2e-4)


@pytest.mark.parametrize("tag", ["l2", "l1"])
@pytest.mark.parametrize("mode", ["soft", "gumbel"])
def test_golden_jtransup(golden, tag, mode, rec_engine):
    import kgrec_b200 as K
    g = golden(f"jtransup_{tag}_{mode}")
    U, D = g["w_user_embeddings"].shape
    I = g["w_item_embeddings"].shape[0]
    E = g["w_ent_embeddings"].shape[0] - 1
    R = g["w_rel_embeddings"].shape[0]
    i_map = {i: i for i in range(I)}
    new_map = {i: ((int(g["item2ent"][i]) if g["item2ent"][i] != E else -1), i) for i in range(I)}
    m = load_weights(K.jTransUPModel(bool(g["l1"]), D, U, I, E, R, i_map, new_map, False, bool(g["gumbel"])), g)
    assert m.item2ent.cpu().tolist() == [int(x) for x in g["item2ent"]]
    npos = torch.from_numpy(g["noise_pos"]) if "noise_pos" in g else None
    nneg = torch.from_numpy(g["noise_neg"]) if "noise_neg" in g else None
    pos = m((lt(g["u"]), lt(g["pi"])), None, is_rec=True, gumbel_u=npos)
    neg = m((lt(g["u"]), lt(g["ni"])), None, is_rec=True, gumbel_u=nneg)
    close(pos, g["pos"])
    close(neg, g["neg"])
    loss = -torch.nn.functional.logsigmoid(float(g["target"]) * (pos - neg)).mean()
    close(loss, g["loss"])
    loss.backward()
    got = grads_by_name(m)
    for k in ("user_embeddings", "item_embeddings", "ent_embeddings", "rel_embeddings", "norm_embeddings",
              "pref_embeddings", "pref_norm_embeddings"):
        close(got[k], g["grad_" + k], rtol=5e-4, atol=2e-6)
    m.zero_grad()
    # KG branch
    kpos = m(None, (lt(g["ph"]), lt(g["pt"]), lt(g["pr"])), is_rec=False)
    kneg = m(None, (lt(g["nh"]), lt(g["nt"]), lt(g["pr"])), is_rec=False)
    close(kpos, g["kg_pos"])
    close(kneg, g["kg_neg"])
    kl = torch.clamp(kpos - kneg + float(g["margin"]), min=0).sum()
    close(kl, g["kg_loss"])
    kl.backward()
    got = grads_by_name(m)
    for k in ("ent_embeddings", "rel_embeddings", "norm_embeddings"):
        close(got[k], g["kggrad_" + k], rtol=2e-4, atol=2e-5)
    nev = torch.from_numpy(g["noise_eval"]) if "noise_eval" in g else None
    close(m.evaluateRec(lt(g["qu"]), gumbel_u=nev), g["eval_rec"], rtol=2e-4)
    close(m.evaluateHead(lt(g["q"]), lt(g["qr"])), g["eval_head"])
    close(m.evaluateTail(lt(g["q"]), lt(g["qr"])), g["eval_tail"])
    with pytest.raises(NotImplementedError):
        m(None, None, is_rec=True)


# ------------------------------------------------------------------------------------------
# (2) numpy oracle on seeded inputs, sizes the oracle finishes in seconds
# ------------------------------------------------------------------------------------------
def np_tables(model):
    return {k.replace("_embeddings.weight", ""): v.detach().cpu().numpy() for k, v in model.state_dict().items()}


@pytest.mark.parametrize("d", [100, 64, 128, 200, 50])
@pytest.mark.parametrize("l1", [False, True])
def test_oracle_transe_transh(d, l1):
    import kgrec_b200 as K
    torch.manual_seed(d + int(l1))
    rng = np.random.RandomState(d)
    E, R, B, KN = 3000, 17, 257, 3
    for cls, score, grads in ((K.TransEModel, O.transe_score, O.transe_grads),
                              (K.TransHModel, O.transh_score, O.transh_grads)):
        m = cls(l1, d, E, R)
        W = np_tables(m)
        T = (W["ent"], W["rel"]) + ((W["norm"],) if "norm" in W else ())
        h, t, r = rng.randint(0, E, B), rng.randint(0, E, B), rng.randint(0, R, B)
        nh = np.repeat(h, KN)
        nt = rng.randint(0, E, B * KN)
        nr = np.repeat(r, KN)
        swap = rng.rand(B * KN) < 0.5                      # corrupt head or tail (utils/data.py:13-14)
        nh2 = np.where(swap, rng.randint(0, E, B * KN), nh)
        nt2 = np.where(swap, np.repeat(t, KN), nt)
        s = m(lt(h), lt(t), lt(r))
        close(s, score(*T, h, t, r, l1))
        for gm in ("dense", "sparse"):
            m.grad_mode = gm
            m.zero_grad()
            fl, fp, fn = m.rank_loss((lt(h), lt(t), lt(r)), (lt(nh2), lt(nt2), lt(nr)), margin=1.0, batch_pos=100)
            op, on = score(*T, h, t, r, l1), score(*T, nh2, nt2, nr, l1)
            close(fp, op)
            close(fn, on)
            want = [O.margin_loss(np.repeat(op[b:b + 100], KN), on[b * KN:(b + 100) * KN], 1.0) for b in range(0, B, 100)]
            close(fl, want, rtol=2e-4)
            fl.sum().backward()
            gp, gn = O.margin_loss_grads(np.repeat(op, KN), on, 1.0)
            a = grads(*T, np.repeat(h, KN), np.repeat(t, KN), np.repeat(r, KN), l1, gp)
            b = grads(*T, nh2, nt2, nr, l1, gn)
            got = grads_by_name(m)
            for k in a:
                close(got[k + "_embeddings"], a[k] + b[k], rtol=1e-3, atol=1e-4)
        m.check_indices()


@pytest.mark.parametrize("l1", [False, True])
def test_oracle_transr(l1):
    import kgrec_b200 as K
    torch.manual_seed(5)
    rng = np.random.RandomState(5)
    d, E, R, B = 100, 500, 7, 65
    m = K.TransRModel(l1, d, E, R)
    W = np_tables(m)
    h, t, r = rng.randint(0, E, B), rng.randint(0, E, B), rng.randint(0, R, B)
    s = m(lt(h), lt(t), lt(r))
    close(s, O.transr_score(W["ent"], W["rel"], W["proj"], h, t, r, l1), rtol=2e-4)
    gup = rng.randn(B).astype(np.float32)
    s.backward(torch.from_numpy(gup).cuda())
    want = O.transr_grads(W["ent"], W["rel"], W["proj"], h, t, r, l1, gup)
    got = grads_by_name(m)
    for k in want:
        close(got[k + "_embeddings"], want[k], rtol=2e-3, atol=2e-4)
    q, qr = rng.randint(0, E, 9), rng.randint(0, R, 9)
    close(m.evaluateTail(lt(q), lt(qr)), O.transr_eval(W["ent"], W["rel"], W["proj"], q, qr, l1, "tail"), rtol=5e-4, atol=1e-4)
    close(m.evaluateHead(lt(q), lt(qr)), O.transr_eval(W["ent"], W["rel"], W["proj"], q, qr, l1, "head"), rtol=5e-4, atol=1e-4)


@pytest.mark.parametrize("d,l1", [(100, False), (32, True), (128, False), (64, False)])
def test_transr_native_eval(d, l1):
    """SURVEY 8a row a6: TransR full-catalog evaluation without a library GEMM -- per distinct relation the
    catalog is projected by k_transr_project, then the distance kernels run on the projected rows.  Score
    matrices vs the oracle (transR.py:80-128), filtered top-K and rank counts vs the ranking walk on the
    kernel's own scores, and a row-sharded catalog giving the same keys."""
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(d)
    rng = np.random.RandomState(d + 1)
    E, R, B, topn = 1500, 9, 37, 7
    m = K.TransRModel(l1, d, E, R)
    W = np_tables(m)
    q, r = rng.randint(0, E, B), rng.randint(0, R, B)       # unsorted relations, several queries per relation
    for side, fn in (("tail", m.evaluateTail), ("head", m.evaluateHead)):
        full = fn(lt(q), lt(r))
        close(full, O.transr_eval(W["ent"], W["rel"], W["proj"], q, r, l1, side), rtol=5e-4, atol=1e-4)
        fullh = full.cpu().numpy()
        filt = [set(int(x) for x in rng.choice(E, rng.randint(0, 30), replace=False)) for _ in range(B)]
        csr = KE.build_filter_csr(list(range(B)), [{i: filt[i] for i in range(B)}], dev())
        ids, sc = KE.keys_to_ids_scores(m.topk(side, lt(q), lt(r), k=topn, filter_csr=csr))
        for b in range(B):
            assert ids[b].tolist() == O.rec_topk(fullh[b], filt[b], topn), (side, b)
            np.testing.assert_array_equal(sc[b].cpu().numpy(), fullh[b][ids[b].cpu().numpy()])     # bit-identical scores
        gold = rng.randint(0, E, B)
        cnt = m.rank_counts(side, lt(q), lt(r), lt(gold)).cpu().numpy()
        for b in range(B):
            key = (fullh[b], np.arange(E))
            want = int(np.sum((key[0] < fullh[b][gold[b]]) | ((key[0] == fullh[b][gold[b]]) & (key[1] < gold[b]))))
            assert cnt[b] == want, (side, b, cnt[b], want)
        # two row shards, merged: the same keys as the whole table
        parts = []
        for lo, hi in (KE.shard_bounds(E, 2, 0), KE.shard_bounds(E, 2, 1)):
            parts.append(m.topk(side, lt(q), lt(r), k=topn, catalog=m.ent_embeddings.weight.detach()[lo:hi], id_base=lo))
        merged = KE.merge_topk(torch.stack(parts))
        assert torch.equal(merged, m.topk(side, lt(q), lt(r), k=topn))
    assert m.evaluateTail(lt([]), lt([])).shape == (0, E)
    m.check_indices()


@pytest.mark.parametrize("d", [20, 32, 64])
@pytest.mark.parametrize("l1", [False, True])
def test_oracle_transr_driver_shapes(d, l1):
    """TransR at the drivers' shapes: few relations, so every relation's matrix collects the gradient of
    many triples of the batch (dense accumulation), through forward + autograd backward twice (positives,
    negatives) as knowledge_representation.py:189-207 calls it."""
    import kgrec_b200 as K
    torch.manual_seed(d)
    rng = np.random.RandomState(d)
    E, R, B = 600, 8, 256
    m = K.TransRModel(l1, d, E, R)
    m.grad_mode = "dense"
    W = np_tables(m)
    h, t, r = rng.randint(0, E, B), rng.randint(0, E, B), rng.randint(0, R, B)
    nh, nt = h.copy(), t.copy()
    flip = rng.rand(B) < 0.5
    nh[flip] = rng.randint(0, E, flip.sum())
    nt[~flip] = rng.randint(0, E, (~flip).sum())
    sp, sn = m(lt(h), lt(t), lt(r)), m(lt(nh), lt(nt), lt(r))
    op = O.transr_score(W["ent"], W["rel"], W["proj"], h, t, r, l1)
    on = O.transr_score(W["ent"], W["rel"], W["proj"], nh, nt, r, l1)
    close(sp, op, rtol=2e-4)
    close(sn, on, rtol=2e-4)
    loss = torch.clamp(sp - sn + 1.0, min=0).sum()
    loss.backward()
    gp, gn = O.margin_loss_grads(op, on, 1.0)
    a = O.transr_grads(W["ent"], W["rel"], W["proj"], h, t, r, l1, gp)
    b = O.transr_grads(W["ent"], W["rel"], W["proj"], nh, nt, r, l1, gn)
    got = grads_by_name(m)
    for k in a:
        close(got[k + "_embeddings"], a[k] + b[k], rtol=2e-3, atol=2e-4)


@pytest.mark.parametrize("d,P", [(100, 20), (64, 13), (128, 50), (52, 4)])
@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("gumbel", [False, True])
def test_oracle_tup(d, P, l1, gumbel, rec_engine):
    import kgrec_b200 as K
    torch.manual_seed(P)
    rng = np.random.RandomState(P)
    U, I, B = 400, 700, 131
    m = K.TransUPModel(l1, d, U, I, P, gumbel)
    W = np_tables(m)
    T = (W["user"], W["item"], W["pref"], W["pref_norm"])
    u, i = rng.randint(0, U, B), rng.randint(0, I, B)
    noise = rng.rand(B, P).astype(np.float32) if gumbel else None
    tn = torch.from_numpy(noise) if gumbel else None
    s = m(lt(u), lt(i), gumbel_u=tn)
    close(s, O.tup_score(*T, u, i, l1, noise), rtol=2e-4)
    gup = rng.randn(B).astype(np.float32)
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad()
        m(lt(u), lt(i), gumbel_u=tn).backward(torch.from_numpy(gup).cuda())
        want = O.tup_grads(*T, u, i, l1, gup, noise)
        got = grads_by_name(m)
        for k in want:
            close(got[k + "_embeddings"], want[k], rtol=2e-3, atol=2e-4)
    qu = rng.randint(0, U, 5)
    nev = rng.rand(5, I, P).astype(np.float32) if gumbel else None
    ev = m.evaluate(lt(qu), gumbel_u=torch.from_numpy(nev) if gumbel else None)
    close(ev, O.tup_eval(*T, qu, l1, nev), rtol=5e-4, atol=1e-4)
    # in-kernel noise: repeatable per seed, and a valid score of SOME preference per pair
    if gumbel:
        torch.manual_seed(3)
        m._seed_counter = 0
        a = m(lt(u), lt(i))
        torch.manual_seed(3)
        m._seed_counter = 0
        b = m(lt(u), lt(i))
        assert torch.equal(a, b)


def test_oracle_ktup_gumbel_l1(rec_engine):
    import kgrec_b200 as K
    torch.manual_seed(11)
    rng = np.random.RandomState(11)
    d, U, I, E, R, B = 100, 300, 200, 900, 24, 97
    aligned = rng.rand(I) < 0.7
    ents = rng.permutation(E)[:I]
    i_map = {i: i for i in range(I)}
    new_map = {i: ((int(ents[i]) if aligned[i] else -1), i) for i in range(I)}
    m = K.jTransUPModel(True, d, U, I, E, R, i_map, new_map, False, True)
    W = np_tables(m)
    i2e = m.item2ent.cpu().numpy().astype(np.int64)
    T = (W["user"], W["item"], W["ent"], W["rel"], W["norm"], W["pref"], W["pref_norm"], i2e)
    u, i = rng.randint(0, U, B), rng.randint(0, I, B)
    noise = rng.rand(B, R).astype(np.float32)
    s = m((lt(u), lt(i)), None, is_rec=True, gumbel_u=torch.from_numpy(noise))
    close(s, O.ktup_rec_score(*T, u, i, True, noise), rtol=2e-4)
    gup = rng.randn(B).astype(np.float32)
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad()
        m((lt(u), lt(i)), None, is_rec=True, gumbel_u=torch.from_numpy(noise)).backward(torch.from_numpy(gup).cuda())
        want = O.ktup_rec_grads(*T, u, i, True, gup, noise)
        got = grads_by_name(m)
        for k in want:
            close(got[k + "_embeddings"], want[k], rtol=2e-3, atol=2e-4)
    qu = rng.randint(0, U, 4)
    nev = rng.rand(4, I, R).astype(np.float32)
    close(m.evaluateRec(lt(qu), gumbel_u=torch.from_numpy(nev)), O.ktup_rec_eval(*T, qu, True, nev), rtol=5e-4, atol=1e-4)


@pytest.mark.parametrize("d,P,gumbel,l1,ktup", [(100, 20, False, False, False), (100, 20, True, True, False),
                                                 (100, 20, False, False, True), (64, 13, False, True, True),
                                                 (128, 32, True, False, True), (16, 8, False, False, False)])
def test_rec_tile_engine_large(d, P, gumbel, l1, ktup):
    """Batches large enough for the tile engine's own size rule (ragged last tile, several tiles
    per CTA): flat forward / backward and the fused ranking loss against the oracle."""
    import kgrec_b200 as K
    torch.manual_seed(d + P)
    rng = np.random.RandomState(d * P)
    U, I, E = 3000, 2500, 4000
    if ktup:
        aligned = rng.rand(I) < 0.7
        ents = rng.permutation(E)[:I]
        i_map = {i: i for i in range(I)}
        new_map = {i: ((int(ents[i]) if aligned[i] else -1), i) for i in range(I)}
        m = K.jTransUPModel(l1, d, U, I, E, P, i_map, new_map, False, gumbel)
        W = np_tables(m)
        T = (W["user"], W["item"], W["ent"], W["rel"], W["norm"], W["pref"], W["pref_norm"],
             m.item2ent.cpu().numpy().astype(np.int64))
        fscore, fgrads = O.ktup_rec_score, O.ktup_rec_grads
        call = lambda u, i, nz: m((lt(u), lt(i)), None, is_rec=True, gumbel_u=nz)
    else:
        m = K.TransUPModel(l1, d, U, I, P, gumbel)
        W = np_tables(m)
        T = (W["user"], W["item"], W["pref"], W["pref_norm"])
        fscore, fgrads = O.tup_score, O.tup_grads
        call = lambda u, i, nz: m(lt(u), lt(i), gumbel_u=nz)

    def check_grads(want, scale):
        got = grads_by_name(m)
        for k in want:
            w = np.asarray(want[k], np.float64)
            close(got[k + "_embeddings"], w, rtol=2e-3, atol=2e-4 * max(1.0, scale * float(np.abs(w).max())),
                  max_outliers=3 if l1 else 0)

    # flat calls (the unchanged drivers' shape, one big batch)
    B = 21013
    u, i = rng.randint(0, U, B), rng.randint(0, I, B)
    noise = rng.rand(B, P).astype(np.float32) if gumbel else None
    tn = torch.from_numpy(noise) if gumbel else None
    close(call(u, i, tn), fscore(*T, u, i, l1, noise), rtol=2e-4)
    gup = (rng.randn(B) / 8).astype(np.float32)
    want = fgrads(*T, u, i, l1, gup, noise)
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad()
        call(u, i, tn).backward(torch.from_numpy(gup).cuda())
        check_grads(want, 1.0)

    # fused ranking loss: n_pos positives x K negatives, BPR mean per batch of 1024
    n_pos, Kn, target, bp = 7001, 2, -1.0, 1024
    u, pi = rng.randint(0, U, n_pos), rng.randint(0, I, n_pos)
    un, ni = np.repeat(u, Kn), rng.randint(0, I, n_pos * Kn)
    noise = rng.rand(n_pos * (1 + Kn), P).astype(np.float32) if gumbel else None
    tn = torch.from_numpy(noise) if gumbel else None
    sp = fscore(*T, u, pi, l1, None if noise is None else noise[:n_pos])
    sn = fscore(*T, un, ni, l1, None if noise is None else noise[n_pos:])
    m.grad_mode = "sparse"
    m.zero_grad()
    fl, fp, fn = m.rank_loss((lt(u), lt(pi)), (lt(un), lt(ni)), target=target, batch_pos=bp, gumbel_u=tn)
    close(fp, sp, rtol=2e-4)
    close(fn, sn, rtol=2e-4)
    spr = np.repeat(sp, Kn)
    nb = (n_pos + bp - 1) // bp
    want_l = [O.bpr_loss(spr[b * bp * Kn:(b + 1) * bp * Kn], sn[b * bp * Kn:(b + 1) * bp * Kn], target) for b in range(nb)]
    close(fl, np.asarray(want_l), rtol=2e-4)
    fl.sum().backward()
    gp_all, gn_all = np.zeros(n_pos * Kn, np.float32), np.zeros(n_pos * Kn, np.float32)
    for b in range(nb):
        sl = slice(b * bp * Kn, (b + 1) * bp * Kn)
        gp_all[sl], gn_all[sl] = O.bpr_loss_grads(spr[sl], sn[sl], target)
    g_all = np.concatenate([gp_all.reshape(n_pos, Kn).sum(1), gn_all]).astype(np.float32)
    want = fgrads(*T, np.concatenate([u, un]), np.concatenate([pi, ni]), l1, g_all, noise)
    check_grads(want, 1.0)

    # the same step as ONE kernel pass (kgrec_rank_loss_step): forward + loss + backward
    two_pass = {k: v.clone() for k, v in grads_by_name(m).items()}
    for gm in ("sparse", "dense"):
        m.grad_mode = gm
        m.zero_grad()
        sl, sp1, sn1 = m.loss_step((lt(u), lt(pi)), (lt(un), lt(ni)), target=target, batch_pos=bp, gumbel_u=tn)
        assert torch.allclose(sp1, fp, rtol=1e-6, atol=1e-6) and torch.allclose(sn1, fn, rtol=1e-6, atol=1e-6)
        assert torch.allclose(sl, fl, rtol=1e-5, atol=1e-6)
        check_grads(want, 1.0)
        got = grads_by_name(m)
        for k in two_pass:
            assert torch.allclose(got[k], two_pass[k], rtol=2e-3, atol=1e-4 * max(1.0, float(two_pass[k].abs().max())))


@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel"])
@pytest.mark.parametrize("l1", [False, True])
def test_step_with_fused_regularisers(cls_name, l1):
    """loss_step_corrupt(reg=True) == the loss of knowledge_representation.py:189-204 built from the
    autograd ranking loss plus torch normLoss / orthogonalLoss on the rows the driver gathers."""
    import kgrec_b200 as K
    torch.manual_seed(21)
    rng = np.random.RandomState(21)
    d, E, R, n_pos, Kn, bp = 100, 900, 7, 1531, 3, 512
    m = getattr(K, cls_name)(l1, d, E, R)
    with torch.no_grad():          # off the kink of max(|x|^2 - 1, 0): half of the rows above 1, half below
        scale = torch.where(torch.arange(E, device=dev()) % 2 == 0, 1.05, 0.95).view(-1, 1)
        m.ent_embeddings.weight.mul_(scale)
        m.rel_embeddings.weight.mul_(torch.where(torch.arange(R, device=dev()) % 2 == 0, 1.07, 0.9).view(-1, 1))
    h, t, r = rng.randint(0, E, n_pos), rng.randint(0, E, n_pos), rng.randint(0, R, n_pos)
    ce = rng.randint(0, E, n_pos * Kn)
    head = rng.rand(n_pos * Kn) < 0.4
    corrupt = torch.as_tensor(np.where(head, ~ce, ce).astype(np.int32), device=dev())
    nh = np.where(head, ce, np.repeat(h, Kn))
    nt = np.where(head, np.repeat(t, Kn), ce)
    nr = np.repeat(r, Kn)
    pos = (lt(h), lt(t), lt(r))
    m.grad_mode = "dense"
    m.zero_grad()
    l, _, _ = m.rank_loss_corrupt(pos, corrupt, margin=1.0, batch_pos=bp)

    def norm_loss(x):
        return torch.clamp((x ** 2).sum(1) - 1.0, min=0).sum()
    nb = (n_pos + bp - 1) // bp
    regs = []
    for b in range(nb):
        ps, ns = slice(b * bp, (b + 1) * bp), slice(b * bp * Kn, (b + 1) * bp * Kn)
        er = m.ent_embeddings(lt(np.concatenate([h[ps], t[ps], nh[ns], nt[ns]])))
        rr_ids = lt(np.concatenate([r[ps], nr[ns]]))
        rr = m.rel_embeddings(rr_ids)
        reg = norm_loss(er) + norm_loss(rr)
        if cls_name == "TransHModel":
            w = m.norm_embeddings(rr_ids)
            reg = reg + (((w * rr).sum(1) ** 2) / (rr ** 2).sum(1)).sum()
        regs.append(reg)
    regs = torch.stack(regs)
    (l + regs).sum().backward()
    want = {k: v.clone() for k, v in grads_by_name(m).items()}
    want_loss = (l + regs).detach()
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad()
        sl, _, _ = m.loss_step_corrupt(pos, corrupt, margin=1.0, batch_pos=bp, reg=True)
        assert torch.allclose(sl, want_loss, rtol=2e-4), (sl, want_loss)
        got = grads_by_name(m)
        for k in want:
            assert torch.allclose(got[k], want[k], rtol=2e-3, atol=2e-4 * max(1.0, float(want[k].abs().max()))), k


@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel"])
@pytest.mark.parametrize("Kn", [1, 2, 31, 32, 40])
def test_step_kernel_negative_counts(cls_name, Kn):
    """The step kernels hold a group's corrupted ids one per lane: 1 and 2 negatives (the reference's own 1 per
    positive), the lane-count edges 31 / 32, and 40 (falls back to the general kernel) against the two-kernel
    autograd path on the same inputs; the slot row ids are checked through the sparse gradients."""
    import kgrec_b200 as K
    torch.manual_seed(Kn)
    rng = np.random.RandomState(Kn)
    d, E, R, n_pos, bp = 64, 700, 5, 517, 128
    m = getattr(K, cls_name)(Kn % 2 == 0, d, E, R)
    h, t, r = rng.randint(0, E, n_pos), rng.randint(0, E, n_pos), rng.randint(0, R, n_pos)
    ce = rng.randint(0, E, n_pos * Kn)
    corrupt = torch.as_tensor(np.where(rng.rand(n_pos * Kn) < 0.5, ~ce, ce).astype(np.int32), device=dev())
    pos = (lt(h), lt(t), lt(r))
    for loss, param in (("margin", 1.0), ("bpr", -1.0)):
        m.grad_mode = "dense"
        m.zero_grad()
        l, ps, ns = m.rank_loss_corrupt(pos, corrupt, margin=param, loss=loss, batch_pos=bp)
        l.sum().backward()
        want = {k: v.clone() for k, v in grads_by_name(m).items()}
        for gm in ("dense", "sparse"):
            m.grad_mode = gm
            m.zero_grad()
            sl, sp, sn = m.loss_step_corrupt(pos, corrupt, margin=param, loss=loss, batch_pos=bp)
            assert torch.allclose(sp, ps, rtol=1e-5, atol=1e-6) and torch.allclose(sn, ns, rtol=1e-5, atol=1e-6)
            assert torch.allclose(sl, l, rtol=1e-4, atol=1e-5)
            got = grads_by_name(m)
            for k in want:
                assert torch.allclose(got[k], want[k], rtol=2e-3, atol=2e-4 * max(1.0, float(want[k].abs().max()))), (k, gm, loss)


@pytest.mark.parametrize("Kn,l1,loss,param", [(10, False, "margin", 1.0), (1, True, "margin", 2.0), (13, False, "bpr", -1.0)])
def test_transr_group_step(Kn, l1, loss, param):
    """TransR single-pass group kernel (one pass over the relation's matrix per group, its gradient added once
    per group) against the generic kernels on the expanded triples."""
    import kgrec_b200 as K
    torch.manual_seed(Kn)
    rng = np.random.RandomState(Kn)
    d, E, R, n_pos, bp = 100, 600, 7, 403, 128
    m = K.TransRModel(l1, d, E, R)
    h, t, r = rng.randint(0, E, n_pos), rng.randint(0, E, n_pos), rng.randint(0, R, n_pos)
    ce = rng.randint(0, E, n_pos * Kn)
    head = rng.rand(n_pos * Kn) < 0.5
    corrupt = torch.as_tensor(np.where(head, ~ce, ce).astype(np.int32), device=dev())
    nh = np.where(head, ce, np.repeat(h, Kn))
    nt = np.where(head, np.repeat(t, Kn), ce)
    nr = np.repeat(r, Kn)
    pos, neg = (lt(h), lt(t), lt(r)), (lt(nh), lt(nt), lt(nr))
    m.grad_mode = "dense"
    m.zero_grad()
    l, ps, ns = m.rank_loss(pos, neg, margin=param, loss=loss, batch_pos=bp)
    l.sum().backward()
    want = {k: v.clone() for k, v in grads_by_name(m).items()}
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad()
        sl, sp, sn = m.loss_step_corrupt(pos, corrupt, margin=param, loss=loss, batch_pos=bp)
        assert torch.allclose(sp, ps, rtol=2e-4, atol=1e-5) and torch.allclose(sn, ns, rtol=2e-4, atol=1e-5)
        assert torch.allclose(sl, l, rtol=2e-4, atol=1e-4)
        got = grads_by_name(m)
        for k in want:
            assert torch.allclose(got[k], want[k], rtol=3e-3, atol=3e-4 * max(1.0, float(want[k].abs().max()))), (k, gm)


@pytest.mark.parametrize("d,R,n_pos", [(32, 5, 300), (36, 5, 300), (64, 3, 257), (68, 5, 300), (96, 4, 300), (108, 5, 211),
                                       (112, 5, 300), (128, 6, 403), (100, 1, 97), (100, 200, 403), (20, 4, 300)])
def test_transr_run_kernel_shapes(d, R, n_pos):
    """The relation-run TransR step (k_run_step_r) over its tile configurations -- d < 64 / d <= 108 / d <= 128 dM tiles,
    d % 32 != 0 remainder rows, 64- and 128-row tiles, a single relation, runs cut by the chunk ends -- and the shapes that
    keep the warp kernel (fewer than 4 groups per relation; d < 32), against the generic kernels on the expanded triples."""
    import kgrec_b200 as K
    torch.manual_seed(d)
    rng = np.random.RandomState(d + R)
    E, Kn, bp = 500, 3, 100
    m = K.TransRModel(False, d, E, R)
    h, t, r = rng.randint(0, E, n_pos), rng.randint(0, E, n_pos), rng.randint(0, R, n_pos)
    ce = rng.randint(0, E, n_pos * Kn)
    head = rng.rand(n_pos * Kn) < 0.5
    corrupt = torch.as_tensor(np.where(head, ~ce, ce).astype(np.int32), device=dev())
    nh = np.where(head, ce, np.repeat(h, Kn))
    nt = np.where(head, np.repeat(t, Kn), ce)
    pos, neg = (lt(h), lt(t), lt(r)), (lt(nh), lt(nt), lt(np.repeat(r, Kn)))
    m.grad_mode = "dense"
    m.zero_grad()
    l, ps, ns = m.rank_loss(pos, neg, margin=1.0, batch_pos=bp)
    l.sum().backward()
    want = {k: v.clone() for k, v in grads_by_name(m).items()}
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad()
        sl, sp, sn = m.loss_step_corrupt(pos, corrupt, margin=1.0, batch_pos=bp)
        assert torch.allclose(sp, ps, rtol=2e-4, atol=1e-5) and torch.allclose(sn, ns, rtol=2e-4, atol=1e-5)
        assert torch.allclose(sl, l, rtol=2e-4, atol=1e-4)
        got = grads_by_name(m)
        for k in want:
            assert torch.allclose(got[k], want[k], rtol=3e-3, atol=3e-4 * max(1.0, float(want[k].abs().max()))), (k, gm)
    m.check_indices()


def test_transr_run_kernel_reports_bad_ids():
    """An out-of-range relation or entity id in the relation-run step is clamped to row 0 and reported
    through the status word (check_indices raises), like in the other kernels."""
    import kgrec_b200 as K
    rng = np.random.RandomState(1)
    E, R, n_pos, Kn = 300, 4, 128, 2
    for what in ("rel", "ent", "corrupt"):
        m = K.TransRModel(False, 64, E, R)
        m.grad_mode = "dense"
        h, t, r = rng.randint(0, E, n_pos), rng.randint(0, E, n_pos), rng.randint(0, R, n_pos)
        ce = rng.randint(0, E, n_pos * Kn).astype(np.int32)
        if what == "rel": r[17] = R + 3
        elif what == "ent": t[5] = E
        else: ce[9] = E + 11
        m.loss_step_corrupt((lt(h), lt(t), lt(r)), torch.as_tensor(ce, device=dev()), margin=1.0, batch_pos=n_pos)
        with pytest.raises(IndexError):
            m.check_indices()


def test_rank_loss_step_other_shapes():
    """kgrec_rank_loss_step outside the single-pass kernel's shapes (KG model; many negatives) falls
    back to forward + backward kernels behind the same call."""
    import kgrec_b200 as K
    from kgrec_b200 import functional as KF, _lib
    torch.manual_seed(5)
    rng = np.random.RandomState(5)
    m = K.TransUPModel(False, 64, 500, 400, 11, False)
    m.grad_mode = "sparse"
    n_pos, Kn = 5003, 17          # 17 negatives per positive do not fit one warp's rows
    u, pi = rng.randint(0, 500, n_pos), rng.randint(0, 400, n_pos)
    un, ni = np.repeat(u, Kn), rng.randint(0, 400, n_pos * Kn)
    fl, fp, fn = m.rank_loss((lt(u), lt(pi)), (lt(un), lt(ni)), target=-1.0, batch_pos=1000)
    fl.sum().backward()
    ref = {k: v.clone() for k, v in grads_by_name(m).items()}
    m.zero_grad()
    sl, sp, sn = m.loss_step((lt(u), lt(pi)), (lt(un), lt(ni)), target=-1.0, batch_pos=1000)
    assert torch.equal(sp, fp) and torch.equal(sn, fn) and torch.allclose(sl, fl)
    got = grads_by_name(m)
    for k in ref:
        assert torch.allclose(got[k], ref[k], rtol=1e-3, atol=1e-5)
    # KG model through the same C entry point
    e = K.TransEModel(True, 100, 2000, 13)
    e.grad_mode = "sparse"
    B, Kn = 999, 3
    h, t, r = rng.randint(0, 2000, B), rng.randint(0, 2000, B), rng.randint(0, 13, B)
    nh, nt, nr = rng.randint(0, 2000, B * Kn), np.repeat(t, Kn), np.repeat(r, Kn)
    fl, fp, fn = e.rank_loss((lt(h), lt(t), lt(r)), (lt(nh), lt(nt), lt(nr)), margin=1.0, batch_pos=100)
    fl.sum().backward()
    ref = {k: v.clone() for k, v in grads_by_name(e).items()}
    e.zero_grad()
    sl, sp, sn = e._loss_step(_lib.TRANSE, (lt(h), lt(t), lt(r)), (lt(nh), lt(nt), lt(nr)), "margin", 1.0, 100)
    assert torch.equal(sp, fp) and torch.equal(sn, fn) and torch.allclose(sl, fl)
    got = grads_by_name(e)
    for k in ref:
        assert torch.allclose(got[k], ref[k], rtol=1e-4, atol=1e-6)


# ------------------------------------------------------------------------------------------
# evaluation: full matrix vs oracle, top-K / rank vs the oracle's ranking walk
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel"])
@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("d", [100, 128, 200])
def test_eval_kg_vs_oracle(cls_name, l1, d):
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(1)
    rng = np.random.RandomState(d)
    E, R, Q, topn = 5003, 11, 37, 10
    m = getattr(K, cls_name)(l1, d, E, R)
    W = np_tables(m)
    q, r = rng.randint(0, E, Q), rng.randint(0, R, Q)
    for side in ("head", "tail"):
        if cls_name == "TransEModel":
            want = O.transe_eval(W["ent"], W["rel"], q, r, l1, side)
        else:
            want = O.transh_eval(W["ent"], W["rel"], W["norm"], q, r, l1, side)
        full = m.evaluateHead(lt(q), lt(r)) if side == "head" else m.evaluateTail(lt(q), lt(r))
        close(full, want, rtol=2e-4, atol=1e-5)
        # top-K with filters: index sets must equal the ranking walk over the KERNEL's own scores
        # (bit-exact: same arithmetic), and the oracle's wherever the K-th gap exceeds fp32 noise
        filt = [set(int(x) for x in rng.choice(E, 30, replace=False)) for _ in range(Q)]
        csr = KE.build_filter_csr(list(range(Q)), [dict(enumerate(filt))], dev())
        keys = m.topk(side, lt(q), lt(r), k=topn, filter_csr=csr)
        ids, scores = KE.keys_to_ids_scores(keys)
        fnp = full.cpu().numpy()
        for b in range(Q):
            assert ids[b].tolist() == O.rec_topk(fnp[b], filt[b], topn)
            np.testing.assert_array_equal(scores[b].cpu().numpy(), fnp[b][ids[b].cpu().numpy()])
            wo = O.rec_topk(want[b], filt[b], topn + 1)
            srt = np.sort(want[b])
            if want[b][wo[topn]] - want[b][wo[topn - 1]] > 1e-4 * srt[topn]:
                assert set(ids[b].tolist()) == set(wo[:topn])
        # rank of a gold id = #entities strictly before it
        gold = rng.randint(0, E, Q)
        cnt = m.rank_counts(side, lt(q), lt(r), lt(gold)).cpu().numpy()
        for b in range(Q):
            order = O.sort_order(fnp[b]).tolist()
            assert cnt[b] == order.index(int(gold[b]))


def test_eval_properties_full_size():
    """Size-independent properties at BASELINE config sizes (d=100, |E|=100k)."""
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(0)
    d, E, R, Q = 100, 100_000, 500, 64
    g = torch.Generator().manual_seed(1)
    h, t, r = (torch.randint(0, n, (Q,), generator=g).cuda() for n in (E, E, R))
    for cls in (K.TransEModel, K.TransHModel):
        m = cls(False, d, E, R)
        s = m(h, t, r)
        tail = m.evaluateTail(h, r)
        head = m.evaluateHead(t, r)
        ar = torch.arange(Q, device="cuda")
        close(tail[ar, t], s.detach().cpu().numpy(), rtol=1e-4)       # SURVEY 4, invariant 1
        close(head[ar, h], s.detach().cpu().numpy(), rtol=1e-4)
        keys = m.topk("tail", h, r, k=10)
        ids, sc = KE.keys_to_ids_scores(keys)
        ref = torch.sort(tail, dim=1, stable=True)
        assert torch.equal(ids, ref.indices[:, :10])                   # bit-exact sets and order
        assert torch.equal(sc, ref.values[:, :10])
        # catalog sharding: per-shard top-K merged == unsharded
        parts = []
        for g_ in range(4):
            lo, hi = KE.shard_bounds(E, 4, g_)
            parts.append(m.topk("tail", h, r, k=10, catalog=m.ent_embeddings.weight.detach()[lo:hi], id_base=lo))
        assert torch.equal(KE.merge_topk(torch.stack(parts)), keys)
    # TransH with zero normals == TransE (invariant 3)
    mh = K.TransHModel(False, d, 1000, 5)
    me = K.TransEModel(False, d, 1000, 5)
    with torch.no_grad():
        mh.norm_embeddings.weight.zero_()
        me.ent_embeddings.weight.copy_(mh.ent_embeddings.weight)
        me.rel_embeddings.weight.copy_(mh.rel_embeddings.weight)
    hh, tt, rr = h % 1000, t % 1000, r % 5
    assert torch.allclose(mh(hh, tt, rr), me(hh, tt, rr), rtol=1e-6, atol=1e-7)


def test_eval_rec_topk_and_eval_matches_forward():
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(2)
    d, U, I, P = 100, 500, 50_000, 20
    m = K.TransUPModel(False, d, U, I, P, False)
    u = torch.arange(0, 70, device="cuda")
    full = m.evaluate(u)
    items = torch.randint(0, I, (70,), device="cuda")
    close(full[torch.arange(70), items], m(u, items).detach().cpu().numpy(), rtol=2e-4)   # invariant 2
    keys = m.topk_items(u, k=10)
    ids, sc = KE.keys_to_ids_scores(keys)
    ref = torch.sort(full, dim=1, stable=True)
    assert torch.equal(ids, ref.indices[:, :10])
    assert torch.equal(sc, ref.values[:, :10])


def test_errors_are_loud():
    import kgrec_b200 as K
    m = K.TransEModel(False, 100, 50, 5)
    m(lt([0, 1]), lt([2, 3]), lt([0, 9]))          # relation 9 out of range
    with pytest.raises(IndexError):
        m.check_indices()
    cpu = K.TransEModel(False, 100, 50, 5).cpu()
    with pytest.raises(RuntimeError, match="no CPU"):
        cpu(torch.tensor([0]), torch.tensor([1]), torch.tensor([0]))
    big = K.TransEModel(False, 600, 10, 2)
    with pytest.raises(RuntimeError, match="512"):
        big(lt([0]), lt([1]), lt([0]))


@pytest.mark.parametrize("d", [128, 64])
def test_eval_scores_independent_of_row_position(d):
    """A (query, row) score is bit-identical whatever tile / lane / shard the row sits in, also
    for rows of an even number of 16-byte units (the skewed dimension walk is keyed by row id)."""
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(4)
    E, R, Q = 20_011, 7, 200
    for cls in (K.TransEModel, K.TransHModel):
        m = cls(False, d, E, R)
        g = torch.Generator().manual_seed(2)
        h, r = torch.randint(0, E, (Q,), generator=g).cuda(), torch.randint(0, R, (Q,), generator=g).cuda()
        full = m.evaluateTail(h, r)
        keys = m.topk("tail", h, r, k=10)
        parts = []
        for s in range(3):
            lo, hi = KE.shard_bounds(E, 3, s)
            parts.append(m.topk("tail", h, r, k=10, catalog=m.ent_embeddings.weight.detach()[lo:hi], id_base=lo))
        assert torch.equal(KE.merge_topk(torch.stack(parts)), keys)
        gold = torch.randint(0, E, (Q,), generator=g).cuda()
        gs = m.gold_scores("tail", h, r, gold)
        assert torch.equal(gs, full[torch.arange(Q, device="cuda"), gold])
        cnt = m.rank_counts("tail", h, r, gold, gold_scores=gs).cpu().numpy()
        fnp = full.cpu().numpy()
        for b in range(0, Q, 17):
            assert cnt[b] == O.sort_order(fnp[b]).tolist().index(int(gold[b]))


@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel"])
@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("loss,param", [("margin", 1.0), ("bpr", -1.0)])
@pytest.mark.parametrize("d", [100, 200])
def test_corrupt_format_matches_expanded_triples(cls_name, l1, loss, param, d):
    """The group-compact negative format gives the same scores, losses and gradients as the
    expanded (nh, nt, nr) triples, and both match the oracle."""
    import kgrec_b200 as K
    from kgrec_b200 import functional as KF
    torch.manual_seed(3)
    rng = np.random.RandomState(d + int(l1))
    E, R, B, KN = 4000, 9, 203, 5
    m = getattr(K, cls_name)(l1, d, E, R)
    W = np_tables(m)
    T = (W["ent"], W["rel"]) + ((W["norm"],) if "norm" in W else ())
    score, grads = (O.transe_score, O.transe_grads) if cls_name == "TransEModel" else (O.transh_score, O.transh_grads)
    h, t, r = rng.randint(0, E, B), rng.randint(0, E, B), rng.randint(0, R, B)
    cid = rng.randint(0, E, B * KN)
    head = rng.rand(B * KN) < 0.5
    corrupt = np.where(head, ~cid, cid).astype(np.int32)
    nh = np.where(head, cid, np.repeat(h, KN))
    nt = np.where(head, np.repeat(t, KN), cid)
    nr = np.repeat(r, KN)
    pos, neg = (lt(h), lt(t), lt(r)), (lt(nh), lt(nt), lt(nr))
    tc = torch.from_numpy(corrupt).cuda()
    enc = KF.encode_corrupt(pos, neg)
    same = (nh == np.repeat(h, KN)) & (nt == np.repeat(t, KN))          # corrupted id happened to equal the original
    assert torch.equal(enc[torch.from_numpy(~same).cuda()], tc[torch.from_numpy(~same).cuda()])
    op, on = score(*T, h, t, r, l1), score(*T, nh, nt, nr, l1)
    if loss == "margin":
        want_loss = [O.margin_loss(np.repeat(op[b:b + 64], KN), on[b * KN:(b + 64) * KN], param) for b in range(0, B, 64)]
        gp, gn = O.margin_loss_grads(np.repeat(op, KN), on, param)
    else:
        want_loss = [O.bpr_loss(np.repeat(op[b:b + 64], KN), on[b * KN:(b + 64) * KN], param) for b in range(0, B, 64)]
        gp = np.concatenate([O.bpr_loss_grads(np.repeat(op[b:b + 64], KN), on[b * KN:(b + 64) * KN], param)[0] for b in range(0, B, 64)])
        gn = -gp
    a = grads(*T, np.repeat(h, KN), np.repeat(t, KN), np.repeat(r, KN), l1, gp)
    b2 = grads(*T, nh, nt, nr, l1, gn)
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad()
        cl, cp, cn = m.rank_loss_corrupt(pos, tc, margin=param, loss=loss, batch_pos=64)
        close(cp, op)
        close(cn, on)
        close(cl, want_loss, rtol=2e-4)
        cl.sum().backward()
        got = grads_by_name(m)
        for k in a:
            close(got[k + "_embeddings"], a[k] + b2[k], rtol=2e-3, atol=2e-4)
        m.zero_grad()
        fl, fp, fn = m.rank_loss(pos, neg, margin=param, loss=loss, batch_pos=64)
        close(fl, cl.detach().cpu().numpy(), rtol=1e-5)
        close(fn, cn.detach().cpu().numpy(), rtol=1e-5)
    m.check_indices()


@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel"])
@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("loss,param", [("margin", 1.0), ("bpr", -1.0)])
def test_single_pass_step_equals_forward_plus_backward(cls_name, l1, loss, param):
    """kgrec_corrupt_loss_step == kgrec_corrupt_loss_fwd + autograd backward of loss.sum()."""
    import kgrec_b200 as K
    torch.manual_seed(9)
    d, E, R, B, KN = 100, 5000, 11, 300, 10
    m = getattr(K, cls_name)(l1, d, E, R)
    g = torch.Generator().manual_seed(5)
    pos = tuple(torch.randint(0, n, (B,), generator=g).cuda() for n in (E, E, R))
    cid = torch.randint(0, E, (B * KN,), generator=g, dtype=torch.int32)
    corrupt = torch.where(torch.rand(B * KN, generator=g) < 0.5, ~cid, cid).cuda()
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad(set_to_none=True)
        l1_, p1, n1 = m.rank_loss_corrupt(pos, corrupt, margin=param, loss=loss, batch_pos=128)
        (2.0 * l1_.sum()).backward()
        want = {k: v.clone() for k, v in grads_by_name(m).items()}
        m.zero_grad(set_to_none=True)
        l2_, p2, n2 = m.loss_step_corrupt(pos, corrupt, margin=param, loss=loss, batch_pos=128, grad_loss=2.0)
        close(p2, p1.cpu().numpy(), rtol=2e-6, atol=0)      # same arithmetic, different kernels: <= a few ulp
        close(n2, n1.cpu().numpy(), rtol=2e-6, atol=0)
        close(l2_, l1_.detach().cpu().numpy(), rtol=1e-5)
        got = grads_by_name(m)
        assert set(got) == set(want)
        for k in want:
            close(got[k], want[k].cpu().numpy(), rtol=1e-4, atol=2e-5)
        # accumulates like autograd
        m.loss_step_corrupt(pos, corrupt, margin=param, loss=loss, batch_pos=128, grad_loss=2.0)
        for k in want:
            close(grads_by_name(m)[k], 2 * want[k].cpu().numpy(), rtol=1e-4, atol=4e-5)
    m.check_indices()


def _big_table(rows, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    w = torch.randn(rows, d, device="cuda", generator=g)
    return torch.nn.Parameter(torch.nn.functional.normalize(w, dim=1))


def test_full_scale_configs():
    """BASELINE.json configs[3] / configs[4] sizes: 500k-entity training tables, 5M-entity d=128
    catalog, 1M x 1M rec tables.  Checked through size-independent properties against plain
    torch arithmetic on a few rows (the oracle cannot run at these sizes)."""
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(0)
    # ---- configs[4]: d=128, 5M entities, top-10 + rank counts, catalog in 3 shards
    d, E, R, Q = 128, 5_000_000, 50, 300
    m = K.TransHModel(False, d, 8, R)
    m.ent_embeddings.weight = _big_table(E, d, 1)
    m.ent_total = E
    g = torch.Generator().manual_seed(3)
    h = torch.randint(0, E, (Q,), generator=g).cuda()
    r = torch.randint(0, R, (Q,), generator=g).cuda()
    keys = m.topk("tail", h, r, k=10)
    ids, sc = KE.keys_to_ids_scores(keys)
    ent, rel, nrm = m.ent_embeddings.weight.detach(), m.rel_embeddings.weight.detach(), m.norm_embeddings.weight.detach()
    for b in range(0, Q, 97):
        w = nrm[r[b]]
        c = ent[h[b]] - (ent[h[b]] @ w) * w + rel[r[b]]
        pe = ent - (ent @ w)[:, None] * w
        ref = ((c - pe) ** 2).sum(1)
        top = torch.topk(ref, 10, largest=False)
        assert set(ids[b].tolist()) == set(top.indices.tolist())
        close(sc[b], top.values.sort().values.cpu().numpy(), rtol=1e-4)
    parts = []
    for s in range(3):
        lo, hi = KE.shard_bounds(E, 3, s)
        parts.append(m.topk("tail", h, r, k=10, catalog=ent[lo:hi], id_base=lo))
    assert torch.equal(KE.merge_topk(torch.stack(parts)), keys)
    gold = ids[:, 3].contiguous()                                  # the 4th best of each query ...
    assert m.rank_counts("tail", h, r, gold).tolist() == [3] * Q   # ... has exactly 3 entities before it
    del m, ent, parts
    torch.cuda.empty_cache()
    # ---- configs[3]: 500k entities d=100, fused single-pass step, dense == sparse gradients
    d, E, R, B, KN = 100, 500_000, 30, 8192, 10
    m = K.TransHModel(True, d, 8, R)
    m.ent_embeddings.weight = _big_table(E + 1, d, 2)
    m.ent_total = E + 1
    pos = tuple(torch.randint(0, n, (B,), generator=g).cuda() for n in (E, E, R))
    cid = torch.randint(0, E, (B * KN,), generator=g, dtype=torch.int32)
    corrupt = torch.where(torch.rand(B * KN, generator=g) < 0.5, ~cid, cid).cuda()
    out = {}
    for gm in ("dense", "sparse"):
        m.grad_mode = gm
        m.zero_grad(set_to_none=True)
        loss, ps, ns = m.loss_step_corrupt(pos, corrupt, margin=1.0, batch_pos=1024)
        out[gm] = (loss.clone(), {k: v.clone() for k, v in grads_by_name(m).items()})
    assert torch.equal(out["dense"][0], out["sparse"][0]) and out["dense"][0].numel() == 8
    for k in out["dense"][1]:     # dense mode accumulates with atomics: summation order varies run to run
        assert torch.allclose(out["dense"][1][k], out["sparse"][1][k], rtol=1e-3, atol=1e-4)
    # loss of batch 0 against plain torch arithmetic
    ent, rel, nrm = m.ent_embeddings.weight.detach(), m.rel_embeddings.weight.detach(), m.norm_embeddings.weight.detach()
    hb, tb, rb = (x[:1024] for x in pos)
    c0 = corrupt[:10240].view(1024, 10)
    nh = torch.where(c0 < 0, (~c0).long(), hb[:, None].expand(-1, 10))
    nt = torch.where(c0 < 0, tb[:, None].expand(-1, 10), c0.long())

    def score(hh, tt, rr):
        w = nrm[rr]
        ph = ent[hh] - (ent[hh] * w).sum(-1, keepdim=True) * w
        pt = ent[tt] - (ent[tt] * w).sum(-1, keepdim=True) * w
        return (ph + rel[rr] - pt).abs().sum(-1)
    sp = score(hb, tb, rb)
    sn = score(nh, nt, rb[:, None].expand(-1, 10))
    close(loss[0], torch.clamp(sp[:, None] - sn + 1.0, min=0).sum().item(), rtol=1e-4)
    m.check_indices()
    del m
    torch.cuda.empty_cache()
    # ---- rec side at 1M x 1M, d=128, P=20, soft preferences: eval scores == forward scores of the same pairs
    mu = K.TransUPModel(False, 128, 8, 8, 20, False)
    mu.user_embeddings.weight = _big_table(1_000_000, 128, 4)
    mu.item_embeddings.weight = _big_table(1_000_000, 128, 5)
    mu.user_total = mu.item_total = 1_000_000
    u = torch.arange(0, 64, device="cuda") * 15_000
    k1 = mu.topk_items(u, k=10)
    ids1, sc1 = KE.keys_to_ids_scores(k1)
    for b in (0, 63):
        close(mu(u[b].expand(10), ids1[b]), sc1[b].cpu().numpy(), rtol=2e-4)      # eval score == forward score
    assert (sc1[:, 1:] >= sc1[:, :-1]).all()


@pytest.mark.parametrize("ktup", [False, True])
@pytest.mark.parametrize("l1", [False, True])
def test_st_gumbel_eval_large_catalog_vs_oracle(ktup, l1):
    """ST-Gumbel full-catalog evaluation at a BASELINE-sized catalog (50k items, d=100, P=20; configs[2]) with
    explicit noise on a query slice, against the oracle's per-pair statement of transUP.py:84-102 / jTransUP.py:163-191:
    the squared-L2 case runs the tiled kernel on augmented rows (its arg-max must pick the oracle's preference for
    every one of the 200k pairs), L1 the one-warp-per-row kernel; plus top-K == ranking walk on the kernel's scores."""
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(77)
    rng = np.random.RandomState(77)
    d, U, I, E, P, Q = 100, 300, 50_000, 60_000, 20, 4
    if ktup:
        ents = rng.permutation(E)[:I]
        new_map = {i: ((int(ents[i]) if i % 10 < 7 else -1), i) for i in range(I)}
        m = K.jTransUPModel(l1, d, U, I, E, P, {i: i for i in range(I)}, new_map, False, True)
    else:
        m = K.TransUPModel(l1, d, U, I, P, True)
    W = np_tables(m)
    qu = rng.randint(0, U, Q)
    noise = rng.rand(Q, I, P).astype(np.float32)
    tn = torch.from_numpy(noise)
    if ktup:
        want = O.ktup_rec_eval(W["user"], W["item"], W["ent"], W["rel"], W["norm"], W["pref"], W["pref_norm"],
                               m.item2ent.cpu().numpy().astype(np.int64), qu, l1, noise)
        got = m.evaluateRec(lt(qu), gumbel_u=tn)
    else:
        want = O.tup_eval(W["user"], W["item"], W["pref"], W["pref_norm"], qu, l1, noise)
        got = m.evaluate(lt(qu), gumbel_u=tn)
    close(got, want, rtol=5e-4, atol=1e-4)
    goth = got.cpu().numpy()
    ids, sc = KE.keys_to_ids_scores(m.topk_items(lt(qu), k=10, gumbel_u=tn))
    for b in range(Q):
        assert ids[b].tolist() == O.rec_topk(goth[b], None, 10)
        np.testing.assert_array_equal(sc[b].cpu().numpy(), goth[b][ids[b].cpu().numpy()])
    # in-kernel noise: a different draw, same distribution -- scores stay in the support of the explicit-noise run
    free = m.topk_items(lt(qu), k=10)
    assert free.shape == (Q, 10) and (KE.keys_to_ids_scores(free)[0] >= 0).all()
    m.check_indices()


def test_edge_cases():
    """Empty and single-element inputs, K larger than the catalog, everything filtered, duplicate
    rows in one batch (gradient accumulation), ragged last loss batch."""
    import kgrec_b200 as K
    from kgrec_b200 import evaluation as KE
    torch.manual_seed(0)
    m = K.TransEModel(False, 100, 50, 3)
    W = np_tables(m)
    empty = lt([])
    assert m(empty, empty, empty).shape == (0,)
    assert m.evaluateTail(empty, empty).shape == (0, 50)
    assert m.topk("tail", empty, empty, k=5).shape == (0, 5)
    one = m(lt([7]), lt([8]), lt([2]))
    close(one, O.transe_score(W["ent"], W["rel"], np.array([7]), np.array([8]), np.array([2]), False))
    # K > catalog: the tail of the list is empty (id -1, score +inf)
    keys = m.topk("tail", lt([1, 2]), lt([0, 1]), k=64)
    ids, sc = KE.keys_to_ids_scores(keys)
    assert (ids[:, :50] >= 0).all() and (ids[:, 50:] == -1).all() and torch.isinf(sc[:, 50:]).all()
    assert sorted(ids[0, :50].tolist()) == list(range(50))
    # everything filtered for query 0, nothing for query 1
    csr = KE.build_filter_csr([0, 1], [{0: set(range(50))}], dev())
    ids, _ = KE.keys_to_ids_scores(m.topk("tail", lt([1, 2]), lt([0, 1]), k=5, filter_csr=csr))
    assert (ids[0] == -1).all() and (ids[1] >= 0).all()
    # the same row many times in one batch: dense accumulation == oracle scatter-add
    m.grad_mode = "dense"
    h, t, r = np.array([4] * 40), np.array([5] * 40), np.array([1] * 40)
    m.zero_grad()
    m(lt(h), lt(t), lt(r)).sum().backward()
    want = O.transe_grads(W["ent"], W["rel"], h, t, r, False, np.ones(40, np.float32))
    close(m.ent_embeddings.weight.grad, want["ent"], rtol=1e-4, atol=1e-5)
    # one positive, one negative, loss batches of 1; ragged: 5 positives in batches of 2
    l, p, n = m.rank_loss_corrupt((lt([1]), lt([2]), lt([0])), torch.tensor([~3], dtype=torch.int32).cuda(), margin=1.0)
    close(n, O.transe_score(W["ent"], W["rel"], np.array([3]), np.array([2]), np.array([0]), False))
    l5, _, _ = m.rank_loss_corrupt((lt([1, 2, 3, 4, 5]), lt([6, 7, 8, 9, 10]), lt([0, 1, 2, 0, 1])),
                                   torch.arange(20, 30, dtype=torch.int32).cuda(), margin=1.0, batch_pos=2)
    assert l5.shape == (3,)
    with pytest.raises(ValueError):
        m.rank_loss_corrupt((lt([1, 2]), lt([2, 3]), lt([0, 0])), torch.tensor([1, 2, 3], dtype=torch.int32).cuda())
    m.check_indices()


def _assert_optimizer_clean(opt):
    for k in opt.acc:                                  # accumulators are all-zero again after a step
        assert not opt.acc[k].any(), k


@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel", "TransRModel"])
@pytest.mark.parametrize("opt_name,steps", [("SGD", 3), ("Adagrad", 3), ("Adam", 1)])
@pytest.mark.parametrize("clip", [None, 0.7])
def test_sparse_row_optimizer_matches_torch(cls_name, opt_name, steps, clip):
    """SURVEY 8f row 1: the sparse-row optimizer (fused step + clip + update of touched rows)
    leaves the tables where torch's dense optimizer + clip_grad_norm_ leaves them.  (Adam is
    compared after one step: dense Adam keeps moving untouched rows afterwards, SURVEY 7.3-3.)"""
    import copy
    import kgrec_b200 as K
    from kgrec_b200.optim import SparseRowOptimizer
    torch.manual_seed(21)
    d, E, R, B, KN, lr = 100, 3000, 7, 500, 4, 0.05
    if cls_name == "TransRModel":
        d, lr = 32, 0.01
    m1 = getattr(K, cls_name)(False, d, E, R)
    m2 = copy.deepcopy(m1)
    m2.grad_mode = "dense"
    ref = getattr(torch.optim, opt_name)(m2.parameters(), lr=lr)
    opt = SparseRowOptimizer(m1, optimizer_type=opt_name, lr=lr, clip=clip)
    g = torch.Generator().manual_seed(8)
    for _ in range(steps):
        pos = tuple(torch.randint(0, n, (B,), generator=g).cuda() for n in (E, E, R))
        cid = torch.randint(0, E, (B * KN,), generator=g, dtype=torch.int32)
        corrupt = torch.where(torch.rand(B * KN, generator=g) < 0.5, ~cid, cid).cuda()
        ref.zero_grad()
        if cls_name == "TransRModel":      # no autograd pair for the TransR group kernel: the step entry point in dense mode
            l2_, _, _ = m2.loss_step_corrupt(pos, corrupt, margin=1.0, batch_pos=128)
        else:
            l2_, _, _ = m2.rank_loss_corrupt(pos, corrupt, margin=1.0, batch_pos=128)
            l2_.sum().backward()
        if clip is not None:
            torch.nn.utils.clip_grad_norm_(m2.parameters(), clip)
        ref.step()
        l1_ = opt.step_corrupt(pos, corrupt, margin=1.0, batch_pos=128)
        close(l1_, l2_.detach().cpu().numpy(), rtol=2e-4)
    for (n1, p1), (n2, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        assert n1 == n2
        close(p1, p2.detach().cpu().numpy(), rtol=2e-4, atol=5e-5)   # atomic accumulation order differs between the runs
    _assert_optimizer_clean(opt)
    m1.check_indices()


@pytest.mark.parametrize("ktup,gumbel,rows_path", [(False, False, False), (False, True, False), (True, False, False),
                                                   (False, False, True), (True, False, True), (False, True, True), (True, True, True)])
@pytest.mark.parametrize("opt_name,steps", [("SGD", 2), ("Adagrad", 3), ("Adam", 1)])
def test_sparse_row_optimizer_rec_models(ktup, gumbel, rows_path, opt_name, steps, monkeypatch):
    """The same for TUP / the rec branch of KTUP (tile kernel in dense-accumulate mode, KTUP's aligned
    entity rows marked through item2ent, rel / norm moved by the pref / pref_norm gradient), with the
    drivers' regularisers (item_recommendation.py:177-180, knowledgable_recommendation.py:343-344)
    against torch autograd of the reference's loss.py formulas on the module's own tables."""
    import copy
    import kgrec_b200 as K
    from kgrec_b200.optim import SparseRowOptimizer
    # rows_path: the row-factored soft step (csrc/train_rec_rows.cu: [P x d] work per distinct row) instead of the pair kernel
    monkeypatch.setenv("KGREC_REC_ROWS", "force" if rows_path else "0")
    torch.manual_seed(31)
    rng = np.random.RandomState(31)
    d, U, I, E, P, B, lr, clip = 64, 900, 700, 1100, 9, 600, 0.05, 1.5
    if rows_path:
        U, I, B = 90, 70, 2500          # heavy row re-use: every user / item many times per step
    if ktup:
        ents = rng.permutation(E)[:I]
        new_map = {i: ((int(ents[i]) if i % 10 < 7 else -1), i) for i in range(I)}
        m1 = K.jTransUPModel(False, d, U, I, E, P, {i: i for i in range(I)}, new_map, False, gumbel)
    else:
        m1 = K.TransUPModel(False, d, U, I, P, gumbel)
    with torch.no_grad():                      # push rows off the unit sphere so normLoss is active on about half of them
        for p in m1.parameters():
            p.mul_(0.9 + 0.2 * torch.rand(p.shape[0], 1, device=p.device))
    m2 = copy.deepcopy(m1)
    m2.grad_mode = "dense"
    ref = getattr(torch.optim, opt_name)(m2.parameters(), lr=lr)
    opt = SparseRowOptimizer(m1, optimizer_type=opt_name, lr=lr, clip=clip)
    g = torch.Generator().manual_seed(9)
    if gumbel:
        steps = 1      # after a step the two copies differ by rounding (atomic order): a near-tie arg-max of the
                       # ST-Gumbel preference may then pick a different row on the two sides -- a property of the test

    def orth(rel, nrm):                        # utils/loss.py:18-19
        return torch.sum(torch.sum(nrm * rel, dim=1, keepdim=True) ** 2 / torch.sum(rel ** 2, dim=1, keepdim=True))

    def nloss(rows):                           # utils/loss.py:21-23
        return torch.sum(torch.clamp(torch.sum(rows ** 2, dim=1, keepdim=True) - 1.0, min=0.0))
    for _ in range(steps):
        u = torch.randint(0, U, (B,), generator=g).cuda()
        pi = torch.randint(0, I, (B,), generator=g).cuda()
        ni = torch.randint(0, I, (B,), generator=g).cuda()
        noise = torch.rand(2 * B, P, generator=g).cuda() if gumbel else None
        ref.zero_grad()
        l2_, _, _ = m2.rank_loss((u, pi), (u, ni), target=-1.0, gumbel_u=noise)
        reg = orth(m2.pref_embeddings.weight, m2.pref_norm_embeddings.weight)
        if not ktup:
            reg = reg + nloss(m2.user_embeddings(u)) + nloss(m2.item_embeddings(torch.cat([pi, ni]))) \
                + nloss(m2.pref_embeddings.weight)
        (l2_.sum() + reg).backward()
        torch.nn.utils.clip_grad_norm_(m2.parameters(), clip)
        ref.step()
        l1_, reg1 = opt.step_pairs((u, pi), (u, ni), target=-1.0, gumbel_u=noise, reg=True)
        close(l1_, l2_.detach().cpu().numpy(), rtol=2e-4)
        close(reg1, np.array([reg.item()]), rtol=2e-4)
    p2 = dict(m2.named_parameters())
    for n1, p1 in m1.named_parameters():
        touched = p2[n1].grad is not None
        assert touched or ktup
        close(p1, p2[n1].detach().cpu().numpy(), rtol=3e-4, atol=5e-5)
    _assert_optimizer_clean(opt)
    m1.check_indices()


@pytest.mark.parametrize("ktup", [False, True])
@pytest.mark.parametrize("l1,gumbel", [(False, False), (True, False), (False, True)])
@pytest.mark.parametrize("loss,n_neg", [("bpr", 1), ("margin", 3)])
def test_rec_rows_step_matches_pair_kernel(ktup, l1, gumbel, loss, n_neg, monkeypatch):
    """The row-factored step (soft preferences, L1 and L2; ST-Gumbel with the L2 score, explicit noise) against the pair
    (tile) kernel on the same step: scores, per-batch losses and every table after one SGD step (i.e. every
    accumulated gradient), BPR and margin, 1 and 3 negatives."""
    import copy
    import kgrec_b200 as K
    from kgrec_b200.optim import SparseRowOptimizer
    torch.manual_seed(51)
    rng = np.random.RandomState(51)
    d, U, I, E, P, B = 100, 120, 150, 400, 20, 3000
    if ktup:
        ents = rng.permutation(E)[:I]
        new_map = {i: ((int(ents[i]) if i % 10 < 7 else -1), i) for i in range(I)}
        m1 = K.jTransUPModel(l1, d, U, I, E, P, {i: i for i in range(I)}, new_map, False, gumbel)
    else:
        m1 = K.TransUPModel(l1, d, U, I, P, gumbel)
    m2 = copy.deepcopy(m1)
    g = torch.Generator().manual_seed(4)
    u = torch.randint(0, U, (B,), generator=g).cuda()
    pi = torch.randint(0, I, (B,), generator=g).cuda()
    ni = torch.randint(0, I, (B * n_neg,), generator=g).cuda()
    un = u.repeat_interleave(n_neg)
    noise = torch.rand(B * (1 + n_neg), P, generator=g).cuda() if gumbel else None
    res = []
    for m, env in ((m1, "force"), (m2, "0")):
        monkeypatch.setenv("KGREC_REC_ROWS", env)
        opt = SparseRowOptimizer(m, optimizer_type="SGD", lr=0.01, clip=None)
        res.append(opt.step_pairs((u, pi), (un, ni), target=-1.0 if loss == "bpr" else 1.0, loss=loss, batch_pos=512,
                                  gumbel_u=noise))
        _assert_optimizer_clean(opt)
        if env == "force":
            assert opt._rows_ws is not None
    close(res[0][0], res[1][0].cpu().numpy(), rtol=2e-4)
    for (n1, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        close(p1, p2.detach().cpu().numpy(), rtol=3e-4, atol=3e-6, max_outliers=12 if l1 else 0)
    m1.check_indices()


def test_sparse_row_optimizer_ktup_kg_branch_and_sparse_touch():
    """KTUP's KG branch through the same optimizer object (joint training alternates the two,
    knowledgable_recommendation.py:320-383), kg_lambda as grad_loss, fused KG regularisers; and
    rows no batch touched do not move."""
    import copy
    import kgrec_b200 as K
    from kgrec_b200.optim import SparseRowOptimizer
    torch.manual_seed(41)
    d, U, I, E, P, B, KN = 100, 50, 60, 5000, 6, 300, 2
    m1 = K.jTransUPModel(True, d, U, I, E, P, {i: i for i in range(I)}, {i: (i, i) for i in range(I)}, False, False)
    m2 = copy.deepcopy(m1)
    m2.grad_mode = "dense"
    before = m1.ent_embeddings.weight.detach().clone()
    opt = SparseRowOptimizer(m1, optimizer_type="Adagrad", lr=0.1, clip=5.0)
    ref = torch.optim.Adagrad(m2.parameters(), lr=0.1)
    g = torch.Generator().manual_seed(3)
    pos = tuple(torch.randint(0, n, (B,), generator=g).cuda() for n in (E, E, P))
    cid = torch.randint(0, E, (B * KN,), generator=g, dtype=torch.int32)
    corrupt = torch.where(torch.rand(B * KN, generator=g) < 0.5, ~cid, cid).cuda()
    ref.zero_grad()
    l2_, _, _ = m2.kg_loss_step_corrupt(pos, corrupt, margin=1.0, grad_loss=0.5, reg=True)
    torch.nn.utils.clip_grad_norm_(m2.parameters(), 5.0)
    ref.step()
    l1_ = opt.step_corrupt(pos, corrupt, margin=1.0, grad_loss=0.5, reg=True)
    close(l1_, l2_.detach().cpu().numpy(), rtol=2e-4)
    for (n1, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        close(p1, p2.detach().cpu().numpy(), rtol=3e-4, atol=5e-5)
    ids = torch.cat([pos[0], pos[1], torch.where(corrupt < 0, ~corrupt, corrupt).long()]).unique()
    moved = (m1.ent_embeddings.weight.detach() != before).any(dim=1).nonzero().view(-1)
    assert set(moved.tolist()) <= set(ids.tolist()) and moved.numel() > 0
    _assert_optimizer_clean(opt)


@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel", "jTransUPModel"])
def test_driver_level_eval_matches_ranking_walk(cls_name):
    """SURVEY 8f row 3: metrics from on-chip top-K / rank counts == the reference's argsort walk
    (oracle restatement) over the full score matrix, with filters and multi-gold queries."""
    import kgrec_b200 as K
    from kgrec_b200 import metrics as KM
    torch.manual_seed(12)
    rng = np.random.RandomState(12)
    d, E, R, U, I, topn = 100, 2500, 6, 300, 900, 10
    if cls_name == "jTransUPModel":
        i_map = {i: i for i in range(I)}
        new_map = {i: ((int(rng.randint(0, E)) if rng.rand() < 0.7 else -1), i) for i in range(I)}
        m = K.jTransUPModel(False, d, U, I, E, R, i_map, new_map, False, False)
        n_ent = E + 1
    else:
        m = getattr(K, cls_name)(True, d, E, R)
        n_ent = E
    # ---- KG side
    def rand_dict(n_keys, key_hi, lo, hi):
        out = {}
        while len(out) < n_keys:
            key = (int(rng.randint(0, key_hi)), int(rng.randint(0, R)))
            out[key] = set(int(x) for x in rng.choice(E, rng.randint(lo, hi), replace=False))
        return out
    head_eval, tail_eval = rand_dict(90, E, 1, 4), rand_dict(110, E, 1, 4)
    head_all = [{k: set(int(x) for x in rng.choice(E, 15, replace=False)) for k in list(head_eval)[::2]}]
    tail_all = [{k: set(int(x) for x in rng.choice(E, 25, replace=False)) for k in list(tail_eval)[::3]}, {}]
    got = KM.evaluate_kg(m, head_eval, tail_eval, head_all, tail_all, topn=topn, batch=64)
    want = {}
    for side, ev, alld in (("head", head_eval, head_all), ("tail", tail_eval, tail_all)):
        keys = list(ev)
        q, r = lt([k[0] for k in keys]), lt([k[1] for k in keys])
        full = (m.evaluateHead(q, r) if side == "head" else m.evaluateTail(q, r)).cpu().numpy()
        assert full.shape[1] == n_ent
        res = []
        for b, key in enumerate(keys):
            filt = set()
            for dct in alld:
                if key in dct:
                    filt.update(dct[key])
            res.extend(O.kg_ranks(full[b], ev[key], filt, topn).values())
        want[side] = np.asarray(res, dtype=np.float64)
    for side, g_ in (("head", got[2]), ("tail", got[3])):
        np.testing.assert_allclose(g_, want[side].mean(axis=0), rtol=1e-12)
    tot = len(want["head"]) + len(want["tail"])
    np.testing.assert_allclose(got[0], (want["head"][:, 0].sum() + want["tail"][:, 0].sum()) / tot, rtol=1e-12)
    np.testing.assert_allclose(got[1], (want["head"][:, 1].sum() + want["tail"][:, 1].sum()) / tot, rtol=1e-12)
    # ---- rec side
    if cls_name == "jTransUPModel":
        eval_dict = {int(u): set(int(x) for x in rng.choice(I, rng.randint(0, 5), replace=False)) for u in rng.choice(U, 120, replace=False)}
        train = {u: set(int(x) for x in rng.choice(I, 40, replace=False)) - eval_dict[u] for u in eval_dict}
        got_r = KM.evaluate_rec(m, eval_dict, [train], topn=topn, batch=50)
        users = [u for u in eval_dict if eval_dict[u]]
        full = m.evaluateRec(lt(users)).cpu().numpy()
        rows = [O.rec_metrics(O.rec_topk(full[b], train[u], topn), eval_dict[u]) for b, u in enumerate(users)]
        np.testing.assert_allclose(got_r, np.asarray(rows, dtype=np.float64).mean(axis=0), rtol=1e-12)


def test_device_negative_sampling():
    """SURVEY 8f row 2: the device samplers honour the reference's rules (utils/data.py:12-85):
    a negative never equals its positive's original id, never is a known triple / rating, the
    head/tail coin is fair, entities are uniform, and a seed reproduces the batch."""
    from kgrec_b200.sampling import TripleNegativeSampler, RatingNegativeSampler
    rng = np.random.RandomState(3)
    E, R, B, KN = 500, 4, 4000, 8
    # a dense known set so that rejection actually happens: ~30 % of all (h, r, *) tails are known
    known = np.stack([rng.randint(0, 40, 60000), rng.randint(0, E, 60000), rng.randint(0, R, 60000)], axis=1)
    known = np.unique(known, axis=0)
    kset = set(map(tuple, known.tolist()))
    s = TripleNegativeSampler(E, R, torch.from_numpy(known))
    pos = known[rng.choice(len(known), B, replace=False)]
    h, t, r = (lt(pos[:, i]) for i in range(3))
    c = s.sample((h, t, r), KN, seed=11)
    assert torch.equal(c, s.sample((h, t, r), KN, seed=11))
    assert not torch.equal(c, s.sample((h, t, r), KN, seed=12))
    cn = c.cpu().numpy().reshape(B, KN)
    head = cn < 0
    ent = np.where(head, ~cn, cn)
    assert ent.min() >= 0 and ent.max() < E
    nh = np.where(head, ent, pos[:, :1])
    nt = np.where(head, pos[:, 1:2], ent)
    assert not (head & (ent == pos[:, :1])).any() and not (~head & (ent == pos[:, 1:2])).any()
    bad = sum((int(a), int(b), int(pos[j, 2])) in kset for j in range(B) for a, b in zip(nh[j], nt[j]))
    assert bad == 0
    assert abs(head.mean() - 0.5) < 0.02                                   # fair coin (32k draws)
    # tails of h < 40 are filtered heavily; unfiltered draws are uniform over the entities
    free = TripleNegativeSampler(E, R, None).sample((h, t, r), KN, seed=5).cpu().numpy()
    e2 = np.where(free < 0, ~free, free)
    cnt = np.bincount(e2, minlength=E)
    assert cnt.min() > 0 and abs(cnt.std() / cnt.mean() - 1 / np.sqrt(cnt.mean())) < 0.05   # Poisson-like spread
    # ratings
    U, I = 50, 300
    kr = np.unique(np.stack([rng.randint(0, U, 6000), rng.randint(0, I, 6000)], axis=1), axis=0)
    rs = RatingNegativeSampler(I, torch.from_numpy(kr))
    pr = kr[rng.choice(len(kr), 2000, replace=False)]
    ni = rs.sample(lt(pr[:, 0]), lt(pr[:, 1]), 3, seed=4).cpu().numpy().reshape(-1, 3)
    rset = set(map(tuple, kr.tolist()))
    assert ni.min() >= 0 and ni.max() < I
    assert not any((int(pr[j, 0]), int(x)) in rset for j in range(len(pr)) for x in ni[j])
    # the sampler's output drives the fused step directly
    import kgrec_b200 as K
    m = K.TransEModel(False, 100, E, R)
    loss, _, _ = m.loss_step_corrupt((h, t, r), c, margin=1.0, batch_pos=1000)
    assert loss.shape == (4,) and torch.isfinite(loss).all()
    m.check_indices()


@pytest.mark.parametrize("with_norm", [False, True])
def test_unchanged_driver_call_pattern_trajectory(with_norm):
    """The reference's KG train_loop body (knowledge_representation.py:179-216) written against
    the drop-in module, step for step: LongTensor ids, pos/neg forward calls, marginLoss, the
    regulariser gathers through model.ent_embeddings / rel_embeddings / norm_embeddings
    (loss.py:18-23), backward with dense grads, clip_grad_norm, Adam with weight decay.  Five
    steps must follow the same trajectory as the reference's op sequence on the CPU
    (oracle/torch_port.py, itself pinned to the golden vectors)."""
    import kgrec_b200 as K
    from oracle import torch_port as TP
    torch.manual_seed(31)
    d, E, R, B = 100, 400, 6, 128
    gpu = (K.TransHModel if with_norm else K.TransEModel)(False, d, E, R)      # L2: smooth gradients
    with torch.no_grad():
        # rows start exactly L2-normalised, i.e. ON the kink of the reference's normLoss
        # (max(|x|^2 - 1, 0), loss.py:21-23) where CPU and GPU rounding decide differently;
        # move them off it so the trajectory is well defined
        gpu.ent_embeddings.weight.mul_(1.04)
        gpu.rel_embeddings.weight.mul_(0.95)
    cpu = TP.TransPort(False, d, E, R, with_norm)
    cpu.load_state_dict({k: v.detach().cpu().clone() for k, v in gpu.state_dict().items()})

    def norm_loss(emb):
        return torch.clamp((emb ** 2).sum(1) - 1.0, min=0).sum()

    def orth_loss(rel, nrm):
        return (((nrm * rel).sum(1) ** 2) / (rel ** 2).sum(1)).sum()

    opts = [torch.optim.Adam([p for _, p in m.named_parameters()], lr=0.01, weight_decay=1e-5) for m in (gpu, cpu)]
    g = torch.Generator().manual_seed(7)
    for step in range(5):
        ids = [torch.randint(0, n, (B,), generator=g) for n in (E, E, R, E, E)]
        losses = []
        for m, opt, dev_ in ((gpu, opts[0], "cuda"), (cpu, opts[1], "cpu")):
            ph, pt, pr, nh, nt = (x.to(dev_) for x in ids)
            nr = pr
            opt.zero_grad()
            pos = m(ph, pt, pr)
            neg = m(nh, nt, nr)
            loss = torch.sum(torch.max(pos - neg + 1.0, torch.zeros_like(pos)))            # marginLoss
            ent = m.ent_embeddings(torch.cat([ph, pt, nh, nt]))
            rel = m.rel_embeddings(torch.cat([pr, nr]))
            if with_norm:
                loss = loss + orth_loss(rel, m.norm_embeddings(torch.cat([pr, nr])))
            loss = loss + norm_loss(ent) + norm_loss(rel)
            loss.backward()
            torch.nn.utils.clip_grad_norm_([p for _, p in m.named_parameters()], 5.0)
            opt.step()
            losses.append(float(loss))
        assert abs(losses[0] - losses[1]) <= 2e-4 * abs(losses[1]), (step, losses)
    for (n1, p1), (n2, p2) in zip(gpu.named_parameters(), cpu.named_parameters()):
        assert n1 == n2
        close(p1, p2.detach().numpy(), rtol=1e-3, atol=2e-4)
    # and the evaluation the driver runs afterwards: scores.data.cpu().numpy() per batch
    q, r = torch.randint(0, E, (16,), generator=g), torch.randint(0, R, (16,), generator=g)
    close(gpu.evaluateTail(q.cuda(), r.cuda()).data.cpu().numpy(), cpu.evaluate_side(q, r, False).detach().numpy(), rtol=1e-3, atol=1e-4)


@pytest.mark.parametrize("cls_name,grad_mode", [("TransEModel", "sparse"), ("TransHModel", "dense")])
def test_graphed_loss_step_matches_module_call(cls_name, grad_mode):
    """The single-batch latency path: the step kernels replayed from a CUDA graph over static id buffers give
    what loss_step_corrupt gives, batch after batch."""
    import kgrec_b200 as K
    torch.manual_seed(17)
    d, E, R, B, KN = 100, 3000, 11, 256, 10
    m = getattr(K, cls_name)(False, d, E, R)
    m.grad_mode = grad_mode
    gs = m.graphed_loss_step(B, KN, margin=1.0)
    g = torch.Generator().manual_seed(2)
    for _ in range(3):
        h, t = (torch.randint(0, E, (B,), generator=g, dtype=torch.int32).cuda() for _ in range(2))
        r = torch.randint(0, R, (B,), generator=g, dtype=torch.int32).cuda()
        c = torch.randint(0, E, (B * KN,), generator=g, dtype=torch.int32)
        c = torch.where(torch.rand(B * KN, generator=g) < 0.5, ~c, c).cuda()
        for buf, src in ((gs.h, h), (gs.t, t), (gs.r, r), (gs.corrupt, c)):
            buf.copy_(src)
        loss = gs.replay()
        m.zero_grad()
        want_l, want_p, want_n = m.loss_step_corrupt((h, t, r), c, margin=1.0)
        assert torch.equal(loss, want_l) and torch.equal(gs.pos_scores, want_p) and torch.equal(gs.neg_scores, want_n)
        got = gs.grads["ent"]
        got = got.to_dense() if got.is_sparse else got
        want = m.ent_embeddings.weight.grad
        want = want.to_dense() if want.is_sparse else want
        close(got, want.cpu().numpy(), rtol=1e-5, atol=1e-6)
    m.check_indices()


@pytest.mark.parametrize("name", ["transe_l2", "transe_l1", "transh_l2"])
@pytest.mark.parametrize("path", ["step", "autograd"])
def test_golden_config_shape_cfg2(golden, name, path):
    """BASELINE configs[1] shape (d=100, |E|=100k, |R|=500, 1024 positives x 10 negatives) against vectors recorded
    from the unmodified reference classes with the reference's own call pattern for K negatives per positive
    (model(pos.repeat_interleave(10)), model(neg), marginLoss, backward): tests/golden/make_golden_cfg2.py.
    The tables are rebuilt from the seed (same generator consumption as the reference constructors)."""
    import kgrec_b200 as K
    g = golden("cfg2_" + name)
    l1 = name.endswith("l1")
    torch.manual_seed(int(g["seed"]))
    m = (K.TransHModel if name.startswith("transh") else K.TransEModel)(l1, 100, 100_000, 500)
    np.testing.assert_array_equal(m.ent_embeddings.weight.detach()[:4].cpu().numpy(), g["ent_rows_check"])
    np.testing.assert_array_equal(m.rel_embeddings.weight.detach()[-4:].cpu().numpy(), g["rel_rows_check"])
    m.grad_mode = "dense"
    pos = (lt(g["ph"]), lt(g["pt"]), lt(g["pr"]))
    corrupt = torch.from_numpy(g["corrupt"]).cuda()
    if path == "step":          # one kernel: forward + margin loss + backward
        loss, ps, ns = m.loss_step_corrupt(pos, corrupt, margin=1.0)
    else:                       # fused forward, autograd backward
        loss, ps, ns = m.rank_loss_corrupt(pos, corrupt, margin=1.0)
        loss.sum().backward()
    close(ps, g["pos_scores"], rtol=1e-4)
    close(ns, g["neg_scores"], rtol=1e-4)
    close(loss.sum(), g["loss"], rtol=1e-4)
    eg = m.ent_embeddings.weight.grad
    close(eg[torch.from_numpy(g["ent_grad_ids"]).cuda()], g["ent_grad_rows"], rtol=1e-3, atol=2e-5, max_outliers=8 if l1 else 0)
    close((eg.double() ** 2).sum(), g["ent_grad_sqnorm"], rtol=1e-3)
    close(m.rel_embeddings.weight.grad, g["rel_grad"], rtol=1e-3, atol=5e-5, max_outliers=8 if l1 else 0)
    if "norm_grad" in g:
        close(m.norm_embeddings.weight.grad, g["norm_grad"], rtol=1e-3, atol=5e-5)
    m.check_indices()


@pytest.mark.parametrize("cls_name", ["TransEModel", "TransHModel"])
@pytest.mark.parametrize("l1", [False, True])
@pytest.mark.parametrize("mode", ["sparse", "dense"])
def test_step_kernels_vs_oracle_k10_d100(cls_name, l1, mode):
    """The step kernels (k_group_step_e / _h) at the benchmark's group shape (10 negatives per positive, d=100)
    directly against the numpy oracle: scores, per-batch margin losses and the gradient of every table."""
    import kgrec_b200 as K
    torch.manual_seed(23)
    rng = np.random.RandomState(23)
    d, E, R, B, KN, bp = 100, 4000, 17, 700, 10, 256
    m = getattr(K, cls_name)(l1, d, E, R)
    m.grad_mode = mode
    W = np_tables(m)
    h, t, r = rng.randint(0, E, B), rng.randint(0, E, B), rng.randint(0, R, B)
    cid = rng.randint(0, E, B * KN)
    head = rng.rand(B * KN) < 0.5
    nh = np.where(head, cid, np.repeat(h, KN))
    nt = np.where(head, np.repeat(t, KN), cid)
    nr = np.repeat(r, KN)
    corrupt = torch.from_numpy(np.where(head, ~cid, cid).astype(np.int32)).cuda()
    loss, ps, ns = m.loss_step_corrupt((lt(h), lt(t), lt(r)), corrupt, margin=1.0, batch_pos=bp)
    if cls_name == "TransEModel":
        score = lambda a, b, c: O.transe_score(W["ent"], W["rel"], a, b, c, l1)                       # noqa: E731
        grads = lambda a, b, c, g: O.transe_grads(W["ent"], W["rel"], a, b, c, l1, g)                  # noqa: E731
    else:
        score = lambda a, b, c: O.transh_score(W["ent"], W["rel"], W["norm"], a, b, c, l1)            # noqa: E731
        grads = lambda a, b, c, g: O.transh_grads(W["ent"], W["rel"], W["norm"], a, b, c, l1, g)       # noqa: E731
    op, on = score(h, t, r), score(nh, nt, nr)
    close(ps, op, rtol=1e-4)
    close(ns, on, rtol=1e-4)
    opr = np.repeat(op, KN)
    nb = (B + bp - 1) // bp
    close(loss, np.array([O.margin_loss(opr[b * bp * KN:(b + 1) * bp * KN], on[b * bp * KN:(b + 1) * bp * KN], 1.0) for b in range(nb)]), rtol=1e-4)
    gp, gn = O.margin_loss_grads(opr, on, 1.0)
    a = grads(np.repeat(h, KN), np.repeat(t, KN), nr, gp)
    b = grads(nh, nt, nr, gn)
    got = grads_by_name(m)
    for k in a:
        w = a[k] + b[k]                      # relation rows collect hundreds of +- terms: absolute tolerance scales with them
        close(got[k + "_embeddings"], w, rtol=2e-3, atol=2e-4 * max(1.0, float(np.abs(w).max())), max_outliers=6 if l1 else 0)
    m.check_indices()


def test_device_prefetcher_ring_reuse():
    """Host batches staged through the fixed device ring arrive intact, in order, including a ragged last batch,
    while the consumer's (slow) kernels on slot s are ordered before the copy that refills it."""
    from kgrec_b200.data import DevicePrefetcher
    g = torch.Generator().manual_seed(1)
    host = [[torch.randint(0, 1 << 30, (50_000 if i < 6 else 777,), generator=g, dtype=torch.int32).pin_memory(),
             torch.randint(0, 1 << 30, (123,), generator=g, dtype=torch.int64).pin_memory()] for i in range(7)]
    sink = torch.zeros(4096, 4096, device="cuda")
    sums = []
    for dev_batch in DevicePrefetcher(iter(host), "cuda", depth=2):
        sink = sink @ sink                                   # keep the compute stream busy past the next copies
        sums.append((dev_batch[0].long().sum() + dev_batch[1].sum()))
    want = [int(a.long().sum() + b.sum()) for a, b in host]
    assert [int(s) for s in sums] == want
    for a, b in zip(DevicePrefetcher(iter(host[:3]), "cuda"), host[:3]):     # a second pass reuses the ring
        assert torch.equal(a[0].cpu(), b[0]) and torch.equal(a[1].cpu(), b[1])


def test_bench_dump_outputs_are_repeatable(tmp_path):
    """`bench.py --dump-outputs DIR`: the last timed launch's losses, scores and a seeded sample of its gradient rows,
    float32 / float64, under 64 MB, the same from run to run with the same arguments (the inputs are seeded)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    nb = 2
    runs = []
    for i in range(2):
        out = tmp_path / ("run%d" % i)
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1", "--batches-per-step", str(nb),
               "--launches-per-step", "2", "--headline-only", "--no-eval", "--no-cpu-baseline", "--dump-outputs", str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        runs.append({f[:-4]: np.load(str(out / f)) for f in sorted(os.listdir(str(out)))})
    a, b = runs
    assert set(a) == {"loss_per_batch", "pos_scores", "neg_scores", "ent_grad_slots", "ent_grad_rows", "ent_grad_values",
                      "rel_grad_slots", "rel_grad_rows", "rel_grad_values"}
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["loss_per_batch"].shape == (nb,) and a["pos_scores"].shape == (nb * 1024,)
    assert a["neg_scores"].shape == (nb * 1024 * 10,) and a["ent_grad_values"].shape[1] == 100
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        if k.endswith(("_slots", "_rows")):
            assert np.array_equal(a[k], b[k]), k
        else:                                   # a reduction may add in another order from run to run
            np.testing.assert_allclose(a[k], b[k], rtol=1e-5, atol=1e-6, err_msg=k)
