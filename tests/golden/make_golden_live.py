"""Record what the unmodified reference computes for the inputs of
tests/test_oracle_live_reference.py, test_drivers.py::test_dropin_constructors_start_from_the_reference_tables
and test_host_logic.py::test_vocab_and_alignment_loaders_match_the_reference:

    python tests/golden/make_golden_live.py --reference <checkout of TaoMiner/joint-kg-recommender>

It builds ``baseline/_ref`` from the checkout (baseline/make_ref.py: a patched copy, git-ignored; nothing of
it is written under tests/), runs the reference classes and loaders there on the CPU with the inputs the
tests regenerate from their seeds, and writes

    live_kg.npz live_tup.npz live_ktup.npz live_misc.npz   (test_oracle_live_reference.summarize / .pack)
    dropin_init.npz                                         (initial tables and the generator state after them)
    loaders.json.gz                                         (loader outputs on the synthetic dataset, canonical JSON)
"""
import argparse
import gzip
import json
import os
import sys
import tempfile
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, os.path.join(ROOT, "baseline"), TESTS):
    sys.path.insert(0, p)
import make_ref                          # noqa: E402
import synth_dataset                     # noqa: E402
import test_oracle_live_reference as L   # noqa: E402
from test_host_logic import LOADER_DATASET, canon   # noqa: E402
from test_drivers import DROPIN_INIT_CASES          # noqa: E402

LT = torch.LongTensor


def load_reference(src):
    make_ref.make(src, force=True)
    for p in reversed(make_ref.env_paths()):
        sys.path.insert(0, p)
    import gflags  # noqa: F401  (the shim; restores numpy.asfarray)
    warnings.filterwarnings("ignore")
    import importlib
    return {n: importlib.import_module("jTransUP.models." + n) for n in ("transE", "transH", "transR", "transUP", "jTransUP")}


def perturb(m, seed):
    sd = {k.replace("_embeddings.weight", ""): p for k, p in m.named_parameters()}
    noise = L.perturb_noise({k: tuple(p.shape) for k, p in sd.items()}, seed)
    with torch.no_grad():
        for k, p in sd.items():
            p.add_(noise[k])


def tables_out(m):
    out = {}
    for k, v in m.state_dict().items():
        out.update(L.fingerprint("w_" + k.replace("_embeddings.weight", ""), L.npy(v)))
    return out


def grads_out(m, prefix="grad_"):
    out = {}
    for k, p in m.named_parameters():
        g = L.npy(p.grad) if p.grad is not None else np.zeros(tuple(p.shape), np.float32)
        out.update(L.summarize(prefix + k.replace("_embeddings.weight", ""), g))
    return out


def record_kg(R, loss):
    cls = {"transe": R["transE"].TransEModel, "transh": R["transH"].TransHModel, "transr": R["transR"].TransRModel}
    out = {}
    for model, d, n_ent, n_rel, n_pos, k_neg in L.KG_CASES:
        for l1 in (False, True):
            torch.manual_seed(1000 + d + n_pos)
            m = cls[model](L1_flag=l1, embedding_size=d, ent_total=n_ent, rel_total=n_rel)
            perturb(m, 5)
            o = tables_out(m)
            rh, rt, rr, nh, nt, q, qr = L.kg_inputs(d, n_ent, n_rel, n_pos, k_neg)
            pos, neg = m(LT(rh), LT(rt), LT(rr)), m(LT(nh), LT(nt), LT(rr))
            ls = loss.marginLoss()(pos, neg, 1.0)
            ls.backward()
            o.update(L.summarize("pos", L.npy(pos)), **L.summarize("neg", L.npy(neg)), loss=L.npy(ls), **grads_out(m))
            with torch.no_grad():
                o.update(L.summarize("eval_head", L.npy(m.evaluateHead(LT(q), LT(qr)))))
                o.update(L.summarize("eval_tail", L.npy(m.evaluateTail(LT(q), LT(qr)))))
            key = L.kg_key(model, d, n_ent, n_rel, n_pos, k_neg, l1)
            out.update({key + "/" + k: v for k, v in o.items()})
    return out


def record_tup(R, loss):
    out = {}
    for d, n_user, n_item, n_pref, n_pos in L.TUP_CASES:
        for gumbel in (False, True):
            for l1 in (False, True):
                torch.manual_seed(77 + d)
                m = R["transUP"].TransUPModel(L1_flag=l1, embedding_size=d, user_total=n_user, item_total=n_item,
                                              preference_total=n_pref, use_st_gumbel=gumbel)
                perturb(m, 6)
                o = tables_out(m)
                u, pi, ni, qu = L.tup_inputs(d, n_user, n_item, n_pos)
                torch.manual_seed(901)
                pos = m(LT(u), LT(pi))
                torch.manual_seed(902)
                neg = m(LT(u), LT(ni))
                ls = loss.bprLoss(pos, neg, target=-1.0)
                ls.backward()
                o.update(L.summarize("pos", L.npy(pos)), **L.summarize("neg", L.npy(neg)), loss=L.npy(ls), **grads_out(m))
                torch.manual_seed(903)
                with torch.no_grad():
                    o.update(L.summarize("eval", L.npy(m.evaluate(LT(qu)))))
                key = L.tup_key(d, n_user, n_item, n_pref, n_pos, gumbel, l1)
                out.update({key + "/" + k: v for k, v in o.items()})
    return out


def record_ktup(R, loss):
    out = {}
    for d, n_user, n_item, n_ent, n_rel, n_pos in L.KTUP_CASES:
        for gumbel in (False, True):
            for l1 in (False, True):
                x = L.ktup_inputs(d, n_user, n_item, n_ent, n_rel, n_pos)
                torch.manual_seed(31 + d)
                m = R["jTransUP"].jTransUPModel(L1_flag=l1, embedding_size=d, user_total=n_user, item_total=n_item,
                                                entity_total=n_ent, relation_total=n_rel, i_map=x["i_map"],
                                                new_map=x["new_map"], isShare=False, use_st_gumbel=gumbel)
                perturb(m, 8)
                with torch.no_grad():
                    m.ent_embeddings.weight[-1].zero_()
                o = tables_out(m)
                torch.manual_seed(41)
                pos = m((LT(x["u"]), LT(x["pi"])), None, is_rec=True)
                torch.manual_seed(42)
                neg = m((LT(x["u"]), LT(x["ni"])), None, is_rec=True)
                loss.bprLoss(pos, neg, target=-1.0).backward()
                o.update(L.summarize("pos", L.npy(pos)), **L.summarize("neg", L.npy(neg)), **grads_out(m))
                m.zero_grad()
                kpos = m(None, (LT(x["ph"]), LT(x["pt"]), LT(x["pr"])), is_rec=False)
                kneg = m(None, (LT(x["ph"]), LT(x["nt"]), LT(x["pr"])), is_rec=False)
                loss.marginLoss()(kpos, kneg, 1.0).backward()
                o.update(L.summarize("kg_pos", L.npy(kpos)), **L.summarize("kg_neg", L.npy(kneg)))
                o.update({k: v for k, v in grads_out(m, "kg_grad_").items()
                          if k.startswith(("kg_grad_ent", "kg_grad_rel", "kg_grad_norm"))})
                torch.manual_seed(43)
                with torch.no_grad():
                    o.update(L.summarize("eval_rec", L.npy(m.evaluateRec(LT(x["qu"])))))
                    o.update(L.summarize("eval_head", L.npy(m.evaluateHead(LT(x["q"]), LT(x["qr"])))))
                    o.update(L.summarize("eval_tail", L.npy(m.evaluateTail(LT(x["q"]), LT(x["qr"])))))
                key = L.ktup_key(d, n_user, n_item, n_ent, n_rel, n_pos, gumbel, l1)
                out.update({key + "/" + k: v for k, v in o.items()})
    return out


def record_misc(loss, misc):
    out = {}
    for d, rows, rel, nrm in L.regulariser_inputs():
        for t in (rows, rel, nrm):
            t.requires_grad_(True)
        nl, ol = loss.normLoss(rows), loss.orthogonalLoss(rel, nrm)
        (nl + ol).backward()
        p = "reg_d%d/" % d
        out[p + "norm_loss"], out[p + "orth_loss"] = L.npy(nl), L.npy(ol)
        for name, t in (("grad_rows", rows), ("grad_rel", rel), ("grad_norm", nrm)):
            out.update({p + k: v for k, v in L.summarize(name, L.npy(t.grad)).items()})
    for c, (scores, gold, filt, topn) in enumerate(L.ranking_inputs()):
        p = "rank_%d/" % c
        f1, prec, rec, hit, ndcg, top_ids = misc.getRecPerformance(scores, gold, fliter_samples=filt, topn=topn)
        hits, ranks, gold_ids = misc.getKGPerformance(scores, gold, fliter_samples=filt, topn=topn)
        out[p + "top_ids"] = np.asarray([int(x) for x in top_ids], np.int64)
        out[p + "rec_metrics"] = np.asarray([f1, prec, rec, hit, ndcg], np.float64)
        out[p + "gold_ids"] = np.asarray([int(x) for x in gold_ids], np.int64)
        out[p + "ranks"] = np.asarray([int(x) for x in ranks], np.int64)
        out[p + "hits"] = np.asarray([int(x) for x in hits], np.int64)
    return out


def record_dropin_init(R):
    out = {}
    cls = {"transE": R["transE"].TransEModel, "transH": R["transH"].TransHModel, "transR": R["transR"].TransRModel,
           "transUP": R["transUP"].TransUPModel, "jTransUP": R["jTransUP"].jTransUPModel}
    for name, args in DROPIN_INIT_CASES:
        torch.manual_seed(11)
        m = cls[name](*args)
        out[name + "/rand"] = L.npy(torch.rand(3))
        for k, v in m.state_dict().items():
            out[name + "/" + k] = L.npy(v)
    return out


def record_loaders():
    from jTransUP.data import load_kg_rating_data as ref_joint, load_rating_data as ref_rec, load_triple_data as ref_kg
    from jTransUP.models.jTransUP import jTransUPModel
    with tempfile.TemporaryDirectory() as tmp:
        info = synth_dataset.write_dataset(tmp, **LOADER_DATASET)
        base = info["path"]
        u_map = ref_rec.loadVocab(os.path.join(base, "u_map.dat"))
        i_map = ref_rec.loadVocab(os.path.join(base, "i_map.dat"))
        e_map = ref_kg.loadVocab(os.path.join(base, "kg", "e_map.dat"))
        i2kg, kg2i = ref_joint.loadR2KgMap(os.path.join(base, "i2kg_map.tsv"))
        rebuilt = ref_joint.rebuildEntityItemVocab(e_map, i_map, kg2i)
        out = ref_joint.load_data(base, ["valid.dat"], ["valid.dat"], 32)
        ikg_map, e_remap, i_remap, _ = rebuilt
        item_total, entity_total, rel_total = len(i_remap), len(e_remap), len(out[7])
        ref_model = jTransUPModel(False, 4, 3, item_total, entity_total, rel_total, i_remap, ikg_map, False, False)
        pad_table = ref_model.paddingItems(list(range(item_total)), entity_total)
    return {"u_map": canon(u_map), "e_map": canon(e_map), "i2kg": canon(i2kg), "kg2i": canon(kg2i), "rebuilt": canon(rebuilt),
            "load_data_i_remap": canon(out[3]), "load_data_e_remap": canon(out[6]), "load_data_ikg_map": canon(out[8]),
            "rating_train_list": canon(out[0][2]), "triple_train_list": canon(out[4][2]),
            "rating_train_dict": canon(out[0][3]), "triple_train_tail_dict": canon(out[4][4]),
            "pad_table": canon(pad_table), "aligned": int(info["aligned"])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of TaoMiner/joint-kg-recommender")
    args = ap.parse_args()
    R = load_reference(os.path.abspath(args.reference))
    from jTransUP.utils import loss, misc
    torch.set_num_threads(2)
    np.savez_compressed(os.path.join(HERE, "live_kg.npz"), **L.pack(record_kg(R, loss)))
    np.savez_compressed(os.path.join(HERE, "live_tup.npz"), **L.pack(record_tup(R, loss)))
    np.savez_compressed(os.path.join(HERE, "live_ktup.npz"), **L.pack(record_ktup(R, loss)))
    np.savez_compressed(os.path.join(HERE, "live_misc.npz"), **L.pack(record_misc(loss, misc)))
    np.savez_compressed(os.path.join(HERE, "dropin_init.npz"), **record_dropin_init(R))
    with gzip.GzipFile(os.path.join(HERE, "loaders.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(record_loaders(), sort_keys=True).encode())
    print("wrote", sorted(f for f in os.listdir(HERE) if f.startswith(("live_", "dropin_init", "loaders"))))


if __name__ == "__main__":
    main()
