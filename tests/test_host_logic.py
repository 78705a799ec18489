"""CPU-only checks: the C-ABI library loads and exports every symbol the header declares,
the host-side mirror keeps the reference's surface, and the multi-GPU host logic (shard
bounds, key merge, all-gather of per-shard top-K) is right on a world_size-2 gloo group."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import kg_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from kgrec_b200 import _lib
    header = open(os.path.join(ROOT, "include", "kgrec_b200.h")).read()
    declared = set(re.findall(r"\b(kgrec_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.EXPORTS), (declared ^ set(_lib.EXPORTS))
    lib = _lib.load()                       # dlopen + resolve each symbol; no GPU needed
    for name in declared:
        assert hasattr(lib, name)
    assert lib.kgrec_abi_version() == _lib.ABI_VERSION
    assert lib.kgrec_rank_loss_workspace_bytes(1024) >= 4096


def test_struct_layouts_match_header():
    import ctypes as C
    from kgrec_b200 import _lib
    # natural alignment of the header's struct: 4 x int32, 4 x int64, 2 x int32, 9 pointers
    assert C.sizeof(_lib.Tables) == 16 + 32 + 8 + 9 * 8
    assert C.sizeof(_lib.Grads) == 8 + 8 * 8
    assert _lib.Tables.ent.offset == 56 and _lib.Tables.item2ent.offset == 56 + 64
    # kgrec_opt_table: 5 pointers, int64, 4 x int32; kgrec_mark_seg: pointer, int64, 2 x int32, pointer, int64, pointer, int64
    assert C.sizeof(_lib.OptTable) == 5 * 8 + 8 + 4 * 4 and _lib.OptTable.rows.offset == 40 and _lib.OptTable.keep_acc.offset == 52
    assert C.sizeof(_lib.MarkSeg) == 56 and _lib.MarkSeg.remap.offset == 24 and _lib.MarkSeg.marks.offset == 40


def test_module_surface_matches_reference_protocol():
    """Constructors, attribute modules and state_dict keys of SURVEY 8b."""
    import kgrec_b200 as K
    e = K.TransEModel(L1_flag=True, embedding_size=8, ent_total=5, rel_total=2)
    h = K.TransHModel(L1_flag=False, embedding_size=8, ent_total=5, rel_total=2)
    r = K.TransRModel(L1_flag=False, embedding_size=8, ent_total=5, rel_total=2)
    u = K.TransUPModel(L1_flag=False, embedding_size=8, user_total=4, item_total=6, preference_total=3,
                       use_st_gumbel=True)
    j = K.jTransUPModel(L1_flag=False, embedding_size=8, user_total=4, item_total=6, entity_total=9,
                        relation_total=3, i_map={i: i for i in range(6)},
                        new_map={i: (i if i % 2 else -1, i) for i in range(6)}, isShare=False, use_st_gumbel=False)
    assert set(e.state_dict()) == {"ent_embeddings.weight", "rel_embeddings.weight"}
    assert set(h.state_dict()) == set(e.state_dict()) | {"norm_embeddings.weight"}
    assert set(r.state_dict()) == set(e.state_dict()) | {"proj_embeddings.weight"}
    assert r.proj_embeddings.weight.shape == (2, 64)
    assert set(u.state_dict()) == {"user_embeddings.weight", "item_embeddings.weight", "pref_embeddings.weight",
                                   "pref_norm_embeddings.weight"}
    assert set(j.state_dict()) == set(u.state_dict()) | set(h.state_dict())
    assert j.ent_embeddings.weight.shape == (10, 8) and not j.ent_embeddings.weight[-1].any()
    assert j.item2ent.tolist() == [9, 1, 9, 3, 9, 5]
    for m in (e, h, r, u, j):
        assert m.is_pretrained is False
        m.disable_grad()
        assert not any(p.requires_grad for p in m.parameters())
        m.enable_grad()
        assert all(p.requires_grad for p in m.parameters())
        for name, p in m.named_parameters():
            if name.startswith(("proj", )) or (m is j and name.startswith("ent")):
                continue
            np.testing.assert_allclose(p.detach().norm(dim=1).cpu().numpy(), 1.0, rtol=1e-5)   # rows L2-normalised
        assert hasattr(m, "forward") and callable(getattr(m, "evaluateHead", getattr(m, "evaluate", None)))
    # the attribute modules stay nn.Embedding-compatible: drivers call model.ent_embeddings(ids)
    assert e.ent_embeddings(torch.tensor([0, 1], device=e.ent_embeddings.weight.device)).shape == (2, 8)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    import kgrec_b200 as K
    m = K.TransEModel(False, 8, 5, 2)
    with pytest.raises(RuntimeError, match="no CPU"):
        m(torch.tensor([0]), torch.tensor([1]), torch.tensor([0]))
    with pytest.raises(RuntimeError, match="no CPU"):
        m.evaluateTail(torch.tensor([0]), torch.tensor([0]))


def test_dropin_overlay_resolves_reference_module_names():
    from kgrec_b200 import dropin
    import kgrec_b200 as K
    mods = dropin.install()
    try:
        import importlib
        for ref_name, cls in (("transE", "TransEModel"), ("transH", "TransHModel"), ("transR", "TransRModel"),
                              ("transUP", "TransUPModel"), ("jTransUP", "jTransUPModel")):
            mod = importlib.import_module("jTransUP.models." + ref_name)
            assert getattr(mod, cls) is getattr(K, cls)
            assert callable(mod.build_model)

        class F:      # the flags build_model reads (jTransUP/models/base.py:22-98)
            L1_flag, embedding_size, num_preferences, use_st_gumbel, share_embeddings = False, 8, 3, True, False
        import jTransUP.models.transUP as tup
        m = tup.build_model(F, 4, 6, 9, 3)
        assert isinstance(m, K.TransUPModel) and m.preference_total == 3
    finally:
        dropin.uninstall(mods)


def test_shard_bounds_and_key_merge():
    from kgrec_b200 import evaluation as KE
    for n, w in ((10, 4), (100_000, 8), (7, 8), (5_000_000, 3)):
        spans = [KE.shard_bounds(n, w, r) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
    rng = np.random.RandomState(0)
    scores = rng.rand(6, 400).astype(np.float32)
    k = 10
    lists = []
    for lo, hi in ((0, 150), (150, 400)):
        part = []
        for row in scores:
            ids = O.rec_topk(row[lo:hi], None, k)
            part.append([(int(row[lo + i].view(np.uint32)) << 32) | (lo + i) for i in ids])
        lists.append(part)
    keys = torch.from_numpy(np.array(lists, dtype=np.uint64).view(np.int64))
    merged = KE.merge_topk_host(keys)
    ids, sc = KE.keys_to_ids_scores(merged)
    for b in range(6):
        assert ids[b].tolist() == O.rec_topk(scores[b], None, k)
        np.testing.assert_array_equal(sc[b].numpy(), scores[b][ids[b].numpy()])
    # empty places (UINT64_MAX) sort last and decode to id -1
    pad = torch.full((1, 6, k), -1, dtype=torch.int64)
    merged2 = KE.merge_topk_host(torch.cat([keys[:1], pad]))
    assert torch.equal(merged2, keys[0])
    assert KE.keys_to_ids_scores(pad[0])[0].eq(-1).all()


def test_filter_csr_and_metrics():
    from kgrec_b200 import evaluation as KE
    train = {0: {1, 5}, 2: {7}}
    valid = {0: {9}, 1: {3}}
    ptr, ids = KE.build_filter_csr([0, 1, 2, 3], [train, valid], torch.device("cpu"))
    assert ptr.tolist() == [0, 3, 4, 5, 5] and ids.tolist() == [1, 5, 9, 3, 7]
    ptr, ids = KE.build_filter_csr([0], [train, valid], torch.device("cpu"), id_lo=4, id_hi=9)
    assert ids.tolist() == [5]
    tops = [[4, 2, 9, 7], [1, 2, 3, 4]]
    golds = [{2, 7, 30}, {99}]
    got = KE.rec_metrics_from_topk(tops, golds)
    for g, t, gold in zip(got, tops, golds):
        np.testing.assert_allclose(g, O.rec_metrics(t, gold), rtol=1e-12)


GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "joint-kg-recommender_b200"))
import numpy as np, torch, torch.distributed as dist
from kgrec_b200 import evaluation as KE
from oracle import kg_oracle as O
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
rank = dist.get_rank()
rng = np.random.RandomState(0)
scores = rng.rand(5, 301).astype(np.float32)           # every rank holds the same oracle view
lo, hi = KE.shard_bounds(301, 2, rank)
k = 7
local = []
for row in scores:                                      # this rank's shard top-K, as the kernel would emit it
    ids = O.rec_topk(row[lo:hi], None, k)
    local.append([(int(row[lo + i].view(np.uint32)) << 32) | (lo + i) for i in ids])
keys = torch.from_numpy(np.array(local, dtype=np.uint64).view(np.int64))
merged = KE.sharded_topk(keys)                          # the one collective: all-gather + merge
ids, _ = KE.keys_to_ids_scores(merged)
for b in range(5):
    assert ids[b].tolist() == O.rec_topk(scores[b], None, k), (rank, b)
cnt = torch.tensor([int((scores[b, lo:hi] < 0.5).sum()) for b in range(5)], dtype=torch.int32)
tot = KE.sharded_rank_counts(cnt.clone())
assert tot.tolist() == [int((scores[b] < 0.5).sum()) for b in range(5)]
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_sharded_topk_world2_gloo(tmp_path):
    port = 29000 + (os.getpid() % 2000)
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    outs = [p.communicate(timeout=240)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_dataio_round_trip(tmp_path):
    """SURVEY 8f row 4: the reference's TSV layouts parse to the same lists / dicts its loaders
    build (load_triple_data.py:5-30, load_rating_data.py:19-38), cache round-trips, CSR filter
    lists match the dict walk, and checkpoints keep the reference's layout."""
    from kgrec_b200 import dataio, evaluation as KE
    import kgrec_b200 as K
    rng = np.random.RandomState(0)
    trip = np.stack([rng.randint(0, 50, 400), rng.randint(0, 50, 400), rng.randint(0, 5, 400)], axis=1)
    kg = tmp_path / "train.dat"
    kg.write_text("".join("%d\t%d\t%d\n" % tuple(r) for r in trip) + "malformed line\n\n7\t8\n")
    f = dataio.TripleFile(str(kg))
    assert f.total == 400 and f.as_list() == [tuple(int(v) for v in r) for r in trip]
    hd, td = f.head_dict(), f.tail_dict()
    for h, t, r in trip.tolist():
        assert h in hd[(t, r)] and t in td[(h, r)]
    assert sum(len(v) for v in hd.values()) == len({tuple(r) for r in trip.tolist()})
    assert os.path.exists(str(kg) + ".kgrec.npz")
    assert np.array_equal(dataio.TripleFile(str(kg)).rows, f.rows)           # from the cache
    rat = tmp_path / "ratings.dat"
    rat.write_text("".join("%d\t%d\t%d\n" % (u, i, 5) for u, i in zip(rng.randint(0, 9, 100), rng.randint(0, 30, 100))))
    rf = dataio.RatingFile(str(rat), use_cache=False)
    rd = rf.rating_dict()
    assert rf.total == 100 and all(i in rd[u] for u, i in rf.as_list())
    keys = list(td)[:20]
    p1, i1 = dataio.csr_from_dicts(keys, [td, {keys[0]: {1, 2, 3}}])
    p2, i2 = KE.build_filter_csr(keys, [td, {keys[0]: {1, 2, 3}}], torch.device("cpu"))
    assert torch.equal(p1, p2) and torch.equal(i1, i2)
    m = K.TransHModel(False, 8, 50, 5)
    opt = torch.optim.Adagrad(m.parameters(), lr=0.1)
    ck = tmp_path / "exp.ckpt"
    dataio.save_checkpoint(str(ck), m, opt, step=12, best_step=10, best_dev_performance=0.5)
    raw = torch.load(str(ck), map_location="cpu")
    assert set(raw) == {"step", "best_step", "best_dev_performance", "model_state_dict", "optimizer_state_dict"}
    assert set(raw["model_state_dict"]) == {"ent_embeddings.weight", "rel_embeddings.weight", "norm_embeddings.weight"}
    m2 = K.TransHModel(False, 8, 50, 5)
    assert dataio.load_checkpoint(str(ck), m2) == (12, 10, 0.5)
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    # a TransE checkpoint warm-starts a TransH model (strict=False), as trainer.loadEmbedding-style reuse does
    e = K.TransEModel(False, 8, 50, 5)
    dataio.save_checkpoint(str(ck), e)
    dataio.load_checkpoint(str(ck), m2)
    assert torch.equal(m2.ent_embeddings.weight, e.ent_embeddings.weight)
    # a checkpoint as the REFERENCE trainer writes it (utils/trainer.py:115-122): best_dev_performance is whatever
    # np.mean returned -- a numpy scalar, which torch >= 2.6's weights-only unpickler refuses
    torch.save({"step": 7, "best_step": 5, "best_dev_performance": np.float64(0.25),
                "model_state_dict": {k: v.detach().cpu() for k, v in m.state_dict().items()}, "optimizer_state_dict": {}}, str(ck))
    m3 = K.TransHModel(False, 8, 50, 5)
    assert dataio.load_checkpoint(str(ck), m3) == (7, 5, 0.25)
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m3.state_dict().values()))
    with pytest.raises(Exception):
        dataio.load_checkpoint(str(ck), m3, trusted=False)


def test_corrupt_format_encoding_round_trip():
    """functional.encode_corrupt: (nh, nt) triples of the reference sampler -> one int32 per negative
    (>= 0 tail replaced, < 0 head replaced by ~id) and back; pure host logic, runs on CPU tensors."""
    import numpy as np
    import torch
    from kgrec_b200 import functional as KF
    rng = np.random.RandomState(3)
    n_pos, K, E = 57, 4, 1000
    h, t, r = (torch.from_numpy(rng.randint(0, E, n_pos)) for _ in range(3))
    ce = torch.from_numpy(rng.randint(0, E, n_pos * K))
    head = torch.from_numpy(rng.rand(n_pos * K) < 0.5)
    # make every corrupted id differ from the row it replaces (the sampler's own guarantee, data.py:23-56)
    ce = torch.where(head & (ce == h.repeat_interleave(K)), (ce + 1) % E, ce)
    ce = torch.where(~head & (ce == t.repeat_interleave(K)), (ce + 1) % E, ce)
    nh = torch.where(head, ce, h.repeat_interleave(K))
    nt = torch.where(head, t.repeat_interleave(K), ce)
    c = KF.encode_corrupt((h, t, r), (nh, nt, r.repeat_interleave(K)))
    assert c.dtype == torch.int32 and c.shape == (n_pos * K,)
    assert torch.equal(c < 0, head)
    assert torch.equal(torch.where(c < 0, ~c, c).long(), ce)
    # the slot row ids the step kernels emit are [h, t, corrupted_1..K] per group
    want = torch.cat([h.view(-1, 1), t.view(-1, 1), ce.view(n_pos, K)], dim=1).reshape(-1)
    assert want.numel() == n_pos * (2 + K)


LOADER_DATASET = dict(users=40, items=90, ratings=900, entities=70, relations=5, triples=800, aligned_frac=0.6)


def canon(x):
    """A loader output in a form JSON keeps and == compares like the original: dicts and sets as sorted
    lists, tuples as lists, numpy scalars as Python numbers."""
    if isinstance(x, dict):
        return sorted(([canon(k), canon(v)] for k, v in x.items()), key=json.dumps)
    if isinstance(x, (set, frozenset)):
        return sorted((canon(v) for v in x), key=json.dumps)
    if isinstance(x, (list, tuple)):
        return [canon(v) for v in x]
    if isinstance(x, np.generic):
        return x.item()
    return x


def test_vocab_and_alignment_loaders_match_the_reference(tmp_path):
    """SURVEY 8f row 4: loadVocab / loadR2KgMap / rebuildEntityItemVocab (load_rating_data.py:6-16,
    load_kg_rating_data.py:5-48) and the item -> entity table against what the reference's own loaders
    returned on a synthetic dataset in its on-disk layout (tests/golden/loaders.json.gz, recorded by
    tests/golden/make_golden_live.py)."""
    import gzip
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import synth_dataset
    from kgrec_b200 import dataio
    from kgrec_b200.models.jTransUP import build_item2ent
    with gzip.open(os.path.join(ROOT, "tests", "golden", "loaders.json.gz"), "rt") as f:
        ref = json.load(f)
    info = synth_dataset.write_dataset(str(tmp_path), **LOADER_DATASET)
    base = info["path"]
    ds = dataio.JointDataset(base, ["valid.dat"], ["valid.dat"], use_cache=False)
    assert canon(ds.u_map) == ref["u_map"]
    assert canon(ds.e_map) == ref["e_map"]
    assert [canon(ds.i2kg), canon(ds.kg2i)] == [ref["i2kg"], ref["kg2i"]]
    assert canon((ds.ikg_map, ds.e_remap, ds.i_remap, ds.aligned)) == ref["rebuilt"]
    assert ref["load_data_i_remap"] == canon(ds.i_remap) and ref["load_data_e_remap"] == canon(ds.e_remap)
    assert ref["load_data_ikg_map"] == canon(ds.ikg_map)
    assert ref["rating_train_list"] == canon(ds.rating_train.as_list())
    assert ref["triple_train_list"] == canon(ds.triple_train.as_list())
    assert ref["rating_train_dict"] == canon(ds.rating_train.rating_dict())
    assert ref["triple_train_tail_dict"] == canon(ds.triple_train.tail_dict())
    # the item -> entity table == the reference's per-call paddingItems over every item
    _, item_total, entity_total, rel_total = ds.totals()
    pad = entity_total
    got = build_item2ent(item_total, pad, ds.i_remap, ds.ikg_map).tolist()
    assert got == ref["pad_table"]
    assert sum(1 for e in got if e != pad) == ds.aligned == info["aligned"] == ref["aligned"]


def test_device_gumbel_uniform_stays_inside_the_unit_interval():
    """common.cuh gumbel_fast: u = (float(bits >> 9) + 0.5) * 2^-23 in fp32.  With 24 bits (bits >> 8) the top value
    16777215.5 is not representable, rounds to 2^24 and gives u = 1.0 -> noise +inf -> NaN gradients about once per
    2^24 draws (a few per configs[2] training step).  The fp32 arithmetic restated in numpy for the edge inputs."""
    f = np.float32
    for bits in (0, 1, 0x1ff, 0x200, 0x7fffffff, 0xfffffdff, 0xfffffe00, 0xffffffff):
        u = (f(bits >> 9) + f(0.5)) * f(1.0 / 8388608.0)
        assert f(0.0) < u < f(1.0), (bits, u)
        g = -np.log(-np.log(u.astype(np.float64)))
        assert np.isfinite(g)
    assert (f(0xffffffff >> 8) + f(0.5)) * f(1.0 / 16777216.0) == f(1.0)       # the 24-bit form that was shipped before


class _FakeKGEngine:
    """Stands in for a model's evaluation kernels in the host-logic test of kgrec_b200.metrics: the same entry points
    `_kg_side` calls (`_eval` for TransE / TransH / KTUP, `_scores` + `rank_counts` for TransR), answered on the CPU
    from one fixed [n_query_keys, n_ent] score table looked up by (q, r) -- every (query, row) score is the same number
    wherever the row sits, which is the property the real kernels guarantee (bit-identical scores on gathered rows)."""

    def __init__(self, model_const, scores_by_key, n_ent, n_rel):
        import types
        self.MODEL = model_const
        self.table = scores_by_key                        # {(q, r): float32 [n_ent]}
        self.ent_embeddings = types.SimpleNamespace(weight=torch.arange(n_ent, dtype=torch.float32).view(-1, 1))
        self.calls = {"_eval": 0, "_scores": 0, "rank_counts": 0}

    def _require_cuda(self):
        return torch.device("cpu")

    def _rows(self, q, r, cols):
        return torch.from_numpy(np.stack([self.table[(int(a), int(b))][cols] for a, b in zip(q.tolist(), r.tolist())]))

    def _eval(self, kg, sd, q, r, mode, catalog=None, cat_ids=None, gold_scores=None, gold_ids=None):
        self.calls["_eval"] += 1
        if mode == "scores":                               # gathered sub-catalog: its first column carries the row ids
            assert torch.equal(catalog[:, 0].long(), cat_ids.long())
            return self._rows(q, r, cat_ids.numpy())
        assert mode == "rank" and catalog.shape[0] == self.ent_embeddings.weight.shape[0]
        return self._count(q, r, gold_scores, gold_ids)

    def _scores(self, sd, q, r, catalog=None, id_base=0, cat_ids=None):
        self.calls["_scores"] += 1
        assert torch.equal(catalog[:, 0].long(), cat_ids.long())
        return self._rows(q, r, cat_ids.numpy())

    def rank_counts(self, side, q, r, gold_ids, gold_scores=None):
        self.calls["rank_counts"] += 1
        assert side in ("head", "tail")
        return self._count(q, r, gold_scores, gold_ids)

    def _count(self, q, r, gs, gi):
        full = self._rows(q, r, slice(None)).numpy()
        ids = np.arange(full.shape[1])
        g, i = gs.numpy()[:, None], gi.numpy()[:, None]
        return torch.from_numpy(((full < g) | ((full == g) & (ids[None, :] < i))).sum(1).astype(np.int32))


@pytest.mark.parametrize("family", ["TRANSE", "TRANSR"])
def test_driver_level_kg_metrics_host_logic(family):
    """kgrec_b200.metrics.evaluate_kg: rank = on-chip count of everything sorting before the gold, minus the filtered
    ids and the other gold ids among them; gold ids inside the filter set are skipped; ties by (score, id).  Host
    arithmetic only, against the reference's walk (oracle restatement of utils/misc.py:125-146) on scores WITH ties;
    the TransR branch goes through TransRModel's own entry points (native per-relation projection on the GPU)."""
    from kgrec_b200 import _lib, metrics as KM
    rng = np.random.RandomState(4)
    E, R, topn = 120, 3, 5

    def rand_dict(n_keys):
        out = {}
        while len(out) < n_keys:
            out[(int(rng.randint(0, E)), int(rng.randint(0, R)))] = set(int(x) for x in rng.choice(E, rng.randint(1, 4), replace=False))
        return out
    head_eval, tail_eval = rand_dict(20), rand_dict(25)
    head_eval[(E + 5, 0)] = set()                                   # empty gold set: skipped (misc.py:169)
    # few distinct values -> many exact ties
    table = {k: (rng.randint(0, 12, E) / 4).astype(np.float32) for k in list(head_eval) + list(tail_eval)}
    head_all = [{k: set(int(x) for x in rng.choice(E, 10, replace=False)) for k in list(head_eval)[::2]}]
    tail_all = [{k: set(int(x) for x in rng.choice(E, 20, replace=False)) for k in list(tail_eval)[::3]}, {}]
    k0 = next(iter(tail_eval))
    tail_all[1][k0] = {next(iter(tail_eval[k0]))}                   # a gold id that is itself filtered
    eng = _FakeKGEngine(getattr(_lib, family), table, E, R)
    got = KM.evaluate_kg(eng, head_eval, tail_eval, head_all, tail_all, topn=topn, batch=7)
    want = {}
    for side, ev, alld in (("head", head_eval, head_all), ("tail", tail_eval, tail_all)):
        res = []
        for key, gold in ev.items():
            if not gold:
                continue
            filt = set()
            for dct in alld:
                filt |= dct.get(key, set())
            res.extend(O.kg_ranks(table[key], gold, filt, topn).values())
        want[side] = np.asarray(res, dtype=np.float64)
    np.testing.assert_allclose(got[2], want["head"].mean(axis=0), rtol=1e-12)
    np.testing.assert_allclose(got[3], want["tail"].mean(axis=0), rtol=1e-12)
    tot = len(want["head"]) + len(want["tail"])
    np.testing.assert_allclose(got[0], (want["head"][:, 0].sum() + want["tail"][:, 0].sum()) / tot, rtol=1e-12)
    np.testing.assert_allclose(got[1], (want["head"][:, 1].sum() + want["tail"][:, 1].sum()) / tot, rtol=1e-12)
    if family == "TRANSR":
        assert eng.calls["_eval"] == 0 and eng.calls["_scores"] > 0 and eng.calls["rank_counts"] > 0
    else:
        assert eng.calls["_scores"] == 0 and eng.calls["rank_counts"] == 0 and eng.calls["_eval"] > 0


def test_bench_reference_arm_contract():
    """`bench.py --impl reference`: one JSON line with the contract's keys, timed on the host cores through the
    reference's own classes when baseline/_ref exists (kind "reference"), else the torch-CPU port (kind "port");
    ranks other than 0 print nothing and exit 0 (the driver launches the arm under torchrun at N > 1)."""
    import json
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
           "--ref-batches-per-step", "1", "--no-regions", "--gpus", "2"]
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "triples/s" and d["n_gpus"] == 2
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("configs[1]") and d["dtype"] == "f32" and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    r1 = subprocess.run(cmd, capture_output=True, text=True, timeout=120, env=dict(env, RANK="1"), cwd=ROOT)
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_bench_region_bookkeeping():
    """bench.add_region_aliases: the configs[3] / configs[4] GPU numbers of the `joint_train_cfg4` and `eval` legs listed
    under `regions` beside the configs[1..2] keys; bookkeeping on measured values only, tolerant of missing legs."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("kgrec_bench", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    out = {"regions": {"cfg2_transe_forward": 1.0},
           "joint_train_cfg4": {"rec_pairs_per_s": 2.0, "kg_triples_per_s": 3.0},
           "eval": {"kg_top10": {"queries": 8, "catalog_rows": 50, "pairs_per_s": 4.0},
                    "rec_top10": {"users_scored": 6, "items": 70, "pairs_per_s": 5.0}, "sharding": "x"}}
    reg = b.add_region_aliases(out)["regions"]
    assert reg["cfg2_transe_forward"] == 1.0
    assert reg["cfg4_ktup_rec_step_forward_backward_regularisers_clip_update"] == 2.0
    assert reg["cfg4_ktup_kg_step_forward_backward_regularisers_clip_update"] == 3.0
    assert reg["cfg5_transe_evaluateTail_top10_8q_x_50_d128"] == 4.0
    assert reg["cfg5_tup_soft_evaluate_top10_6u_x_70_d128"] == 5.0
    assert b.add_region_aliases({"value": 1}) == {"value": 1}                       # N > 1 lines carry no regions
    assert b.add_region_aliases({"regions": {}, "eval": {"kg_top10": {}}}) == {"regions": {}, "eval": {"kg_top10": {}}}


def test_c_abi_argument_validation_without_a_gpu():
    """Error behaviour of the C ABI (include/kgrec_b200.h: "return value: KGREC_OK or an error code; kgrec_last_error() has
    the text"): every rejection below happens on the host BEFORE any kernel launch, so it is checked here without a GPU;
    so are the size / layout queries the bindings allocate from.  Pointers are fake but well-formed (16-byte aligned,
    never dereferenced on the host)."""
    import ctypes as C
    from kgrec_b200 import _lib
    lib = _lib.load()
    FAKE = 0x7000_0000_1000

    def err():
        return lib.kgrec_last_error().decode()

    def tables(**kw):
        t = _lib.Tables(dim=100, ld=100, n_ent=50, n_rel=7, ent=FAKE, rel=FAKE + 0x100000)
        for k, v in kw.items():
            setattr(t, k, v)
        return t

    def score(t, model=_lib.TRANSE, idx_bytes=8, n=4, a=FAKE, scores=FAKE):
        return lib.kgrec_score_fwd(C.byref(t) if t is not None else None, model, a, FAKE, FAKE, idx_bytes, n, None, 0, scores, None, None)
    assert score(None) != 0 and "tables is NULL" in err()
    assert score(tables(dim=0)) != 0 and "bad dim/ld" in err()
    assert score(tables(dim=100, ld=96)) != 0 and "bad dim/ld" in err()
    assert score(tables(dim=600, ld=600)) != 0 and "> 512" in err()
    assert score(tables(), model=99) != 0 and "unknown model" in err()
    assert score(tables(ent=None)) != 0 and "needs table 'ent'" in err()
    assert score(tables(), model=_lib.TRANSH) != 0 and "needs table 'norm'" in err()
    assert score(tables(), model=_lib.TRANSR) != 0 and "needs table 'proj'" in err()
    assert score(tables(), idx_bytes=3) != 0 and "idx_bytes must be 4 or 8" in err()
    assert score(tables(), a=None) != 0 and "index array is NULL" in err()
    assert score(tables(), n=-1) != 0 and score(tables(), scores=None) != 0
    assert score(tables(), n=0) == 0                                       # empty batch: accepted, nothing launched
    # TUP / KTUP table requirements (transUP.py:46-60, jTransUP.py:64-103)
    rec = dict(user=FAKE, item=FAKE, pref=FAKE, pref_norm=FAKE, n_user=10, n_item=10)
    assert score(tables(**rec, n_pref=0), model=_lib.TUP) != 0 and "preference_total" in err()
    assert score(tables(**rec, n_pref=4, norm=FAKE), model=_lib.KTUP) != 0 and "item2ent" in err()
    assert score(tables(**rec, n_pref=4, norm=FAKE, item2ent=FAKE), model=_lib.KTUP) != 0 and "n_pref == n_rel" in err()
    # fused ranking loss: loss kind and shape checks (loss.py:8-16, 29-31)
    t = tables()

    def rank_loss(loss_kind=_lib.LOSS_MARGIN, n_pos=4, n_neg=2, batch_pos=4, ws=FAKE):
        return lib.kgrec_rank_loss_fwd(C.byref(t), _lib.TRANSE, FAKE, FAKE, FAKE, FAKE, FAKE, FAKE, 8, n_pos, n_neg, batch_pos,
                                       loss_kind, 1.0, None, 0, FAKE, FAKE, FAKE, ws, None, None)
    assert rank_loss(loss_kind=7) != 0 and "unknown loss" in err()
    assert rank_loss(n_neg=0) != 0 and rank_loss(batch_pos=0) != 0 and rank_loss(n_pos=-1) != 0
    assert rank_loss(ws=None) != 0 and "NULL" in err()
    assert rank_loss(n_pos=0) == 0
    g = _lib.Grads(mode=0, ent=FAKE)                                       # rel gradient buffer missing
    assert lib.kgrec_score_bwd(C.byref(t), _lib.TRANSE, FAKE, FAKE, FAKE, 8, 4, None, 0, FAKE, C.byref(g), None) != 0
    assert "gradient buffer" in err()
    g = _lib.Grads(mode=5, ent=FAKE, rel=FAKE)
    assert lib.kgrec_score_bwd(C.byref(t), _lib.TRANSE, FAKE, FAKE, FAKE, 8, 4, None, 0, FAKE, C.byref(g), None) != 0
    # negative samplers (utils/data.py:12-85)
    assert lib.kgrec_hashset_capacity(0) == 1024 and lib.kgrec_hashset_capacity(1000) == 2048
    assert lib.kgrec_hashset_capacity(1 << 20) == 1 << 21
    assert lib.kgrec_hashset_build(FAKE, 10, FAKE, 1000, None) != 0 and "power of two" in err()
    assert lib.kgrec_hashset_build(FAKE, 600, FAKE, 1024, None) != 0                     # load factor > 1/2
    assert lib.kgrec_sample_corrupt(FAKE, FAKE, FAKE, 8, 4, 1, 1, 3, None, 0, 0, FAKE, None, None) != 0      # one entity: no negative exists
    assert lib.kgrec_sample_corrupt(FAKE, FAKE, None, 8, 4, 1, 50, 3, None, 0, 0, FAKE, None, None) != 0 and "relations" in err()
    assert lib.kgrec_sample_corrupt(FAKE, FAKE, FAKE, 8, 0, 1, 50, 3, None, 0, 0, FAKE, None, None) == 0
    assert lib.kgrec_sample_neg_items(FAKE, FAKE, 8, 4, 0, 50, None, 0, 0, FAKE, None, None) != 0
    assert lib.kgrec_sample_neg_items(FAKE, FAKE, 8, 4, 1, 50, FAKE, 1000, 0, FAKE, None, None) != 0 and "capacity" in err()
    # layout / size queries the bindings allocate from
    assert lib.kgrec_rank_loss_workspace_bytes(0) == 4 and lib.kgrec_rank_loss_workspace_bytes(1000) == 4000
    assert lib.kgrec_pref_aug_ld(100) == 308 and lib.kgrec_pref_aug_ld(128) == 388        # 3 d + pad, (ld / 4) odd
    for d in (4, 20, 64, 100, 128, 200, 256):
        ld = lib.kgrec_pref_aug_ld(d)
        assert ld > 3 * d and ld % 4 == 0 and (ld // 4) % 2 == 1
    assert lib.kgrec_gumbel_aug_ld(100, 20) == 140 and lib.kgrec_gumbel_aug_ld(128, 7) == 144
    assert lib.kgrec_eval_workspace_bytes(4096, 10) >= 4096 * 10 * 8
    assert lib.kgrec_eval_workspace_bytes(8192, 10) > lib.kgrec_eval_workspace_bytes(4096, 10)
    assert lib.kgrec_transr_workspace_floats(64, 1000, 100) >= 1000 * 100
    assert lib.kgrec_abi_version() == _lib.ABI_VERSION and lib.kgrec_sm_count() > 0


def test_c_abi_eval_argument_validation_without_a_gpu():
    """The evaluation entry points' host-side rejections (eval.cu: eval_plan and the three callers), no GPU involved."""
    import ctypes as C
    from kgrec_b200 import _lib
    lib = _lib.load()
    FAKE = 0x7000_0000_1000

    def err():
        return lib.kgrec_last_error().decode()

    def tables(**kw):
        t = _lib.Tables(dim=100, ld=100, n_ent=5000, n_rel=7, ent=FAKE, rel=FAKE, norm=FAKE)
        for k, v in kw.items():
            setattr(t, k, v)
        return t

    def scores(t=None, model=_lib.TRANSE, side=_lib.SIDE_TAIL, q=FAKE, r=FAKE, idx_bytes=8, qvec=None, nq=16, cat=FAKE,
               cat_ld=100, n_cat=5000, out=FAKE, ld_out=5000, cat_ids=None):
        t = tables() if t is None else t
        return lib.kgrec_eval_scores(C.byref(t), model, side, q, r, idx_bytes, qvec, nq, cat, cat_ld, n_cat, 0, cat_ids, None, 0,
                                     out, ld_out, None)
    assert lib.kgrec_eval_scores(None, 0, 1, FAKE, FAKE, 8, None, 16, FAKE, 100, 5000, 0, None, None, 0, FAKE, 5000, None) != 0
    assert "tables is NULL" in err()
    assert scores(nq=0) != 0 and "empty catalog / query set" in err()
    assert scores(n_cat=0) != 0 and scores(cat=None) != 0
    assert scores(t=tables(dim=300, ld=300), cat_ld=300) != 0 and "outside [1, 256]" in err()
    assert scores(t=tables(dim=50, ld=50), cat_ld=50) != 0 and "multiples of 4" in err()            # evaluate* needs d % 4 == 0
    assert scores(cat=FAKE + 4) != 0 and "16-byte aligned" in err()
    assert scores(cat_ld=96) != 0                                                                     # leading dimension < d
    assert scores(model=42) != 0 and "unknown model" in err()
    assert scores(model=_lib.TRANSR) != 0 and "explicit query vectors" in err()                        # transR.py:80-128 via kgrec_transr_eval_*
    assert scores(side=_lib.SIDE_REC) != 0 and "does not fit model" in err()                           # a KG model has no rec side
    assert scores(t=tables(ent=None)) != 0 and "NULL or not 16-byte aligned" in err()
    assert scores(model=_lib.TRANSH, t=tables(norm=None)) != 0
    assert scores(out=None) != 0 and "bad out / ld_out" in err()
    assert scores(ld_out=100) != 0
    assert scores(q=None) != 0 and "query ids are NULL" in err()
    assert scores(r=None) != 0
    assert scores(idx_bytes=2) != 0 and "idx_bytes must be 4 or 8" in err()

    def topk(k=10, id_base=0, n_cat=5000, out=FAKE, ws=FAKE, ws_bytes=1 << 40, idx_bytes=4):
        t = tables()
        return lib.kgrec_eval_topk(C.byref(t), _lib.TRANSE, _lib.SIDE_HEAD, FAKE, FAKE, idx_bytes, None, 16, FAKE, 100, n_cat, id_base, k,
                                   None, None, None, 0, out, ws, ws_bytes, None)
    assert topk(k=0) != 0 and "topn" in err()
    assert topk(k=129) != 0 and "[1, 128]" in err()
    assert topk(out=None) != 0 and "out_keys is NULL" in err()
    assert topk(id_base=-1) != 0 and "fit 32 bits" in err()
    assert topk(id_base=(1 << 32) - 10) != 0 and "fit 32 bits" in err()                                # ids are the low half of the keys
    assert topk(ws_bytes=64) != 0 and "workspace too small" in err()
    assert topk(ws=None) != 0
    assert topk(idx_bytes=16) != 0 and "idx_bytes" in err()

    def rank(gold_scores=FAKE, gold_ids=FAKE, counts=FAKE, id_base=0):
        t = tables()
        return lib.kgrec_eval_rank_count(C.byref(t), _lib.TRANSH, _lib.SIDE_TAIL, FAKE, FAKE, 8, None, 16, FAKE, 100, 5000, id_base,
                                         gold_scores, gold_ids, counts, None)
    assert rank(gold_scores=None) != 0 and "NULL argument" in err()
    assert rank(counts=None) != 0 and rank(gold_ids=None) != 0
    assert rank(id_base=1 << 32) != 0 and "fit 32 bits" in err()
    # merge of per-shard lists; augmented-row builders; KTUP catalog
    assert lib.kgrec_merge_topk(None, 2, 16, 10, FAKE, None) != 0 and "merge_topk" in err()
    assert lib.kgrec_merge_topk(FAKE, 0, 16, 10, FAKE, None) != 0 and lib.kgrec_merge_topk(FAKE, 2, 16, 200, FAKE, None) != 0
    assert lib.kgrec_merge_topk(FAKE, 2, 0, 10, FAKE, None) == 0                                        # no queries: nothing to do
    rt = tables(user=FAKE, item=FAKE, pref=FAKE, pref_norm=FAKE, n_pref=20)
    assert lib.kgrec_pref_aug_rows(C.byref(rt), _lib.TRANSE, 0, None, 8, FAKE, 100, 10, FAKE, 308, None) != 0
    assert lib.kgrec_pref_aug_rows(C.byref(rt), _lib.TUP, 0, None, 8, FAKE, 100, 10, FAKE, 300, None) != 0 and "ld_out = 308" in err()
    assert lib.kgrec_pref_aug_rows(C.byref(tables(user=FAKE, item=FAKE, n_pref=20)), _lib.TUP, 0, None, 8, FAKE, 100, 10, FAKE, 308, None) != 0
    assert lib.kgrec_pref_aug_rows(C.byref(rt), _lib.TUP, 0, None, 8, FAKE, 100, 0, FAKE, 308, None) == 0
    assert lib.kgrec_gumbel_aug_rows(C.byref(rt), _lib.TUP, None, 8, FAKE, 100, 10, FAKE, 128, None, None) != 0 and "ld_out = 140" in err()
    assert lib.kgrec_gumbel_aug_rows(C.byref(rt), _lib.TUP, FAKE, 3, FAKE, 100, 10, FAKE, 140, None, None) != 0 and "idx_bytes" in err()
    assert lib.kgrec_gumbel_aug_supported(100, 20, 10) == 1 and lib.kgrec_gumbel_aug_supported(100, 20, 0) == 1
    assert lib.kgrec_gumbel_aug_supported(50, 20, 10) == 0 and lib.kgrec_gumbel_aug_supported(100, 65, 10) == 0
    assert lib.kgrec_ktup_item_table(C.byref(tables(item=FAKE)), 0, 10, FAKE, 100, None) != 0 and "ktup_item_table" in err()
    assert lib.kgrec_ktup_item_table(C.byref(tables(item=FAKE, item2ent=FAKE)), 0, 0, FAKE, 100, None) == 0


def test_c_abi_optimizer_argument_validation_without_a_gpu():
    """Host-side rejections of the sparse-row optimizer / regulariser entry points (optim.cu, reg.cu): segment and table
    counts, missing state for Adagrad / Adam (utils/trainer.py:63-81 builds exactly one of SGD / Adagrad / Adam)."""
    import ctypes as C
    from kgrec_b200 import _lib
    lib = _lib.load()
    FAKE = 0x7000_0000_1000

    def err():
        return lib.kgrec_last_error().decode()
    seg = _lib.MarkSeg(ids=FAKE, n=10, idx_bytes=4, compact=0, remap=None, n_remap=0, marks=FAKE, rows=100)
    arr = (_lib.MarkSeg * 9)(*([seg] * 9))
    assert lib.kgrec_rows_mark(arr, 0, 1, None, None) != 0 and "id segments per call" in err()
    assert lib.kgrec_rows_mark(arr, 9, 1, None, None) != 0
    assert lib.kgrec_rows_mark(None, 1, 1, None, None) != 0
    bad = (_lib.MarkSeg * 1)(_lib.MarkSeg(ids=FAKE, n=10, idx_bytes=2, marks=FAKE, rows=100))
    assert lib.kgrec_rows_mark(bad, 1, 1, None, None) != 0 and "bad segment 0" in err()
    bad = (_lib.MarkSeg * 1)(_lib.MarkSeg(ids=None, n=10, idx_bytes=4, marks=FAKE, rows=100))
    assert lib.kgrec_rows_mark(bad, 1, 1, None, None) != 0
    empty = (_lib.MarkSeg * 1)(_lib.MarkSeg(ids=None, n=0, idx_bytes=8, marks=None, rows=100))
    assert lib.kgrec_rows_mark(empty, 1, 1, None, None) == 0                   # an empty step marks nothing

    def tab(**kw):
        t = _lib.OptTable(table=FAKE, acc=FAKE, state1=FAKE, state2=FAKE, marks=FAKE, rows=100, dim=100, keep_acc=0)
        for k, v in kw.items():
            setattr(t, k, v)
        return t
    one = (_lib.OptTable * 1)(tab())
    nine = (_lib.OptTable * 9)(*([tab()] * 9))
    assert lib.kgrec_rows_sqnorm(nine, 9, 1, FAKE, None) != 0 and "tables per call" in err()
    assert lib.kgrec_rows_sqnorm(one, 0, 1, FAKE, None) != 0
    assert lib.kgrec_rows_sqnorm(one, 1, 1, None, None) != 0 and "sqnorm is NULL" in err()
    noacc = (_lib.OptTable * 1)(tab(acc=None))
    assert lib.kgrec_rows_sqnorm(noacc, 1, 1, FAKE, None) != 0 and "no accumulator" in err()

    def update(tabs, kind):
        return lib.kgrec_rows_update(tabs, 1, 1, kind, 0.01, 1e-10, 0.9, 0.999, 1, 0.0, None, 0.0, None)
    assert update(one, 3) != 0 and "unknown kind" in err()
    assert update(one, -1) != 0
    assert update((_lib.OptTable * 1)(tab(state1=None)), 1) != 0 and "state missing" in err()      # Adagrad needs its sum
    assert update((_lib.OptTable * 1)(tab(state2=None)), 2) != 0 and "state missing" in err()      # Adam needs m and v
    assert update((_lib.OptTable * 1)(tab(table=None)), 0) != 0
    assert update((_lib.OptTable * 1)(tab(rows=0)), 0) != 0
    # regularisers (utils/loss.py:18-23)
    assert lib.kgrec_reg_norm_rows(None, 10, 100, None, 8, 10, 1.0, None, None, None, None) != 0
    assert lib.kgrec_reg_norm_rows(FAKE, 10, 100, None, 8, 11, 1.0, None, None, None, None) != 0 and "n > rows" in err()
    assert lib.kgrec_reg_norm_rows(FAKE, 10, 100, FAKE, 5, 10, 1.0, None, None, None, None) != 0
    assert lib.kgrec_reg_norm_rows(FAKE, 10, 100, FAKE, 8, 0, 1.0, None, None, None, None) == 0
    assert lib.kgrec_reg_orth_tables(FAKE, None, 10, 100, 1.0, None, None, None, None) != 0 and "reg_orth" in err()
    assert lib.kgrec_reg_orth_tables(FAKE, FAKE, 0, 100, 1.0, None, None, None, None) != 0


def test_c_abi_group_format_argument_validation_without_a_gpu():
    """Host-side rejections of the group-compact (corrupted-id) ranking-loss entry points (train_group.cu: group_check):
    the format the reference's sampler produces -- head OR tail of the positive replaced, utils/data.py:12-56 -- exists
    for the KG families only and holds entity ids in 31 bits."""
    import ctypes as C
    from kgrec_b200 import _lib
    lib = _lib.load()
    FAKE = 0x7000_0000_1000

    def err():
        return lib.kgrec_last_error().decode()

    def tables(**kw):
        t = _lib.Tables(dim=100, ld=100, n_ent=50, n_rel=7, ent=FAKE, rel=FAKE, norm=FAKE)
        for k, v in kw.items():
            setattr(t, k, v)
        return t

    def fwd(t=None, model=_lib.TRANSE, idx_bytes=4, n_pos=4, corrupt=FAKE, n_neg=2, batch_pos=4, loss_kind=_lib.LOSS_MARGIN, ws=FAKE):
        t = tables() if t is None else t
        return lib.kgrec_corrupt_loss_fwd(C.byref(t), model, FAKE, FAKE, FAKE, idx_bytes, n_pos, corrupt, n_neg, batch_pos, loss_kind,
                                          1.0, FAKE, FAKE, FAKE, ws, None, None)
    rec = dict(user=FAKE, item=FAKE, pref=FAKE, pref_norm=FAKE, n_pref=4, n_user=9, n_item=9)
    assert fwd(t=tables(**rec), model=_lib.TUP) != 0 and "TransE / TransH" in err()
    assert fwd(t=tables(proj=FAKE), model=_lib.TRANSR) != 0 and "TransE / TransH" in err()        # TransR: the step entry point only
    assert fwd(t=tables(dim=50, ld=50)) != 0 and "embedding_size % 4 == 0" in err()
    assert fwd(t=tables(ent=FAKE + 4)) != 0 and "16-byte aligned" in err()
    assert fwd(idx_bytes=1) != 0 and "idx_bytes" in err()
    assert fwd(corrupt=None) != 0 and "index array is NULL" in err()
    assert fwd(loss_kind=9) != 0 and "unknown loss" in err()
    assert fwd(n_neg=0) != 0 and fwd(batch_pos=0) != 0 and fwd(n_pos=1 << 31) != 0
    assert fwd(t=tables(n_ent=1 << 31)) != 0 and "31 bits" in err()
    assert fwd(ws=None) != 0
    assert fwd(n_pos=0) == 0
    # the single-pass step: the same checks + gradient descriptor; workspace sizes the bindings allocate
    g = _lib.Grads(mode=1, ent=FAKE, rel=FAKE)

    def step(t=None, model=_lib.TRANSE, grads=g, n_neg=2, reg=0):
        t = tables() if t is None else t
        return lib.kgrec_corrupt_loss_step(C.byref(t), model, FAKE, FAKE, FAKE, 4, 4, FAKE, n_neg, 4, _lib.LOSS_MARGIN, 1.0, 1.0, reg,
                                           FAKE, FAKE, FAKE, C.byref(grads) if grads is not None else None, None, None, FAKE, None, None)
    assert step(model=_lib.TUP, t=tables(**rec)) != 0
    assert step(grads=None) != 0
    assert step(model=_lib.TRANSH, grads=_lib.Grads(mode=1, ent=FAKE, rel=FAKE)) != 0            # TransH needs the norm gradient too
    t = tables(n_rel=500)
    assert lib.kgrec_corrupt_loss_step_workspace_bytes(C.byref(t), _lib.TRANSE, 1024) == 4096
    assert lib.kgrec_corrupt_loss_step_workspace_bytes(C.byref(t), _lib.TRANSR, 1024) == 4 * (2 * 1024 + 501)
    assert lib.kgrec_corrupt_loss_step_workspace_bytes(C.byref(t), _lib.TRANSE, 0) == 4


def test_device_train_iterator_follows_the_reference_epoch_rule():
    """kgrec_b200.data.DeviceTrainIterator vs MakeTrainIterator (utils/data.py:87-110): same batch size, same number
    of batches per epoch (the reference restarts as soon as start > n - batch_size, whatever -negtive_samples is), every
    batch made of rows of the data, no row twice within an epoch when negtive_samples = 1, a fresh order every epoch,
    reproducible per seed.  Plumbing only (torch index ops on the data's device): runs on the CPU here."""
    from kgrec_b200.data import DeviceTrainIterator
    rng = np.random.RandomState(0)
    n, bs = 103, 10
    data = np.stack([np.arange(n), rng.randint(0, 50, n), rng.randint(0, 5, n)], axis=1)      # column 0 identifies the row
    it = DeviceTrainIterator(data, bs, device="cpu", seed=5)
    assert it.batches_per_epoch == (n - bs) // bs + 1 == 10
    epochs = []
    for _ in range(3):
        seen = []
        for _ in range(it.batches_per_epoch):
            h, t, r = next(it)
            assert h.shape == t.shape == r.shape == (bs,) and h.dtype == torch.int32 and h.is_contiguous()
            assert np.array_equal(data[h.numpy(), 1], t.numpy()) and np.array_equal(data[h.numpy(), 2], r.numpy())
            seen.extend(h.tolist())
        assert len(set(seen)) == len(seen) == 100                      # a permutation prefix: no row twice in an epoch
        epochs.append(seen)
    assert it.epoch == 2 and epochs[0] != epochs[1] != epochs[2]
    # the reference's own iterator yields the same count before it reshuffles: compare with its arithmetic on a python list
    start, count = -bs, 0
    while True:
        start += bs
        if start > n - bs:
            break
        count += 1
    assert count == it.batches_per_epoch
    again = DeviceTrainIterator(data, bs, device="cpu", seed=5)
    assert [next(again)[0].tolist() for _ in range(10)] == [epochs[0][i * bs:(i + 1) * bs] for i in range(10)]
    # -negtive_samples k: the order is range(n) * k shuffled; rows may repeat inside an epoch, all ids stay in range
    it3 = DeviceTrainIterator(data[:, :2], 25, negtive_samples=3, device="cpu", seed=1)
    assert it3.order.numel() == 3 * n and int(it3.order.max()) < n and it3.batches_per_epoch == (n - 25) // 25 + 1
    assert torch.equal(torch.bincount(it3.order, minlength=n), torch.full((n,), 3))
    u, i = next(it3)
    assert u.shape == (25,) and np.array_equal(data[u.numpy(), 1], i.numpy())
    # a batch larger than the data set: the reference yields the whole (short) shuffled prefix every time
    small = DeviceTrainIterator(data[:7], 10, device="cpu")
    assert small.batches_per_epoch == 1 and next(small)[0].numel() == 7 and next(small)[0].numel() == 7
    with pytest.raises(ValueError):
        DeviceTrainIterator(np.zeros((0, 3), np.int64), 4, device="cpu")


def test_sharding_host_logic_properties():
    """Property tests (hypothesis) of the multi-GPU host logic around the one collective: contiguous row shards tile the
    catalog for any (rows, world); per-shard top-K lists merged by the host statement of kgrec_merge_topk equal the
    top-K of the whole catalog, ties included ((score, id) order == integer order of the 64-bit keys); the filter CSR
    restricted to the shards partitions the unrestricted one."""
    from hypothesis import given, settings, strategies as st
    from kgrec_b200 import evaluation as KE

    @settings(max_examples=200, deadline=None)
    @given(st.integers(0, 5000), st.integers(1, 16))
    def shards_tile(n, world):
        bounds = [KE.shard_bounds(n, world, r) for r in range(world)]
        assert bounds[0][0] == 0 and bounds[-1][1] == n
        for (lo, hi), (lo2, _) in zip(bounds, bounds[1:]):
            assert lo <= hi == lo2
        per = (n + world - 1) // world
        assert all(hi - lo <= per for lo, hi in bounds)
    shards_tile()

    def keys_of(scores, ids):
        bits = np.asarray(scores, np.float32).view(np.uint32).astype(np.uint64)
        return (bits << np.uint64(32)) | np.asarray(ids, np.uint64)

    @settings(max_examples=60, deadline=None)
    @given(st.integers(1, 300), st.integers(1, 6), st.integers(1, 12), st.integers(0, 2 ** 31 - 1))
    def merged_equals_global(n, world, k, seed):
        rng = np.random.RandomState(seed)
        nq = 3
        scores = (rng.randint(0, 7, (nq, n)) / 4).astype(np.float32)            # few distinct values: many ties
        lists = np.full((world, nq, k), np.iinfo(np.uint64).max, dtype=np.uint64)
        for g in range(world):
            lo, hi = KE.shard_bounds(n, world, g)
            for q in range(nq):
                ks = np.sort(keys_of(scores[q, lo:hi], np.arange(lo, hi)))[:k]
                lists[g, q, :len(ks)] = ks
        merged = KE.merge_topk_host(torch.from_numpy(lists.view(np.int64)))
        ids, sc = KE.keys_to_ids_scores(merged)
        for q in range(nq):
            want = O.rec_topk(scores[q], None, k)                                   # stable argsort: (score, id)
            got = [int(x) for x in ids[q] if x >= 0]
            assert got == want
            assert np.array_equal(sc[q].numpy()[:len(want)], scores[q][want])
            assert (ids[q][len(want):] == -1).all()
    merged_equals_global()

    @settings(max_examples=60, deadline=None)
    @given(st.integers(1, 200), st.integers(1, 5), st.integers(0, 2 ** 31 - 1))
    def filter_partitions(n, world, seed):
        rng = np.random.RandomState(seed)
        keys = list(range(6))
        dicts = [{q: set(int(x) for x in rng.choice(n, rng.randint(0, min(n, 9) + 1), replace=False)) for q in keys[::2]},
                 {q: set(int(x) for x in rng.choice(n, rng.randint(0, min(n, 5) + 1), replace=False)) for q in keys}]
        ptr, ids = KE.build_filter_csr(keys, dicts, torch.device("cpu"))
        whole = [sorted(ids[int(ptr[i]):int(ptr[i + 1])].tolist()) for i in range(len(keys))]
        parts = [[] for _ in keys]
        for g in range(world):
            lo, hi = KE.shard_bounds(n, world, g)
            p, i_ = KE.build_filter_csr(keys, dicts, torch.device("cpu"), lo, hi)
            for q in range(len(keys)):
                row = i_[int(p[q]):int(p[q + 1])].tolist() if int(p[q + 1]) > int(p[q]) else []
                assert all(lo <= x < hi for x in row) and row == sorted(row)
                parts[q].extend(row)
        assert parts == whole
    filter_partitions()
