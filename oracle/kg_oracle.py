"""CPU oracle for the joint KG + recommendation scoring hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product:
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline
legs may import it, and only as the checker (or as the timed CPU baseline),
never as the thing shipped.  The product path is the CUDA library behind
``include/kgrec_b200.h``.

This file is a plain-numpy restatement of the arithmetic the reference
(TaoMiner/joint-kg-recommender, pure Python on PyTorch) performs on its hot
path.  Every function cites the reference ``file:line`` it follows (paths are
relative to the reference checkout).  The reference holds no tests or golden
vectors for this path (SURVEY.md section 4), so the oracle is pinned against
vectors produced by importing the unmodified reference classes in the build
container: ``tests/golden/make_golden.py`` writes them, ``tests/golden/*.npz``
holds them, ``tests/test_oracle_golden.py`` checks this file against them.
It is also checked at the BASELINE row widths (d = 100, 128): ``tests/golden/make_golden_live.py`` records
what the unmodified classes return, ``tests/test_oracle_live_reference.py`` compares every function below
with that forward / autograd / evaluate* / ranking output.

Conventions
-----------
* tables are ``[rows, d]`` float arrays; ``dtype`` of the tables decides the
  arithmetic precision (float32 reproduces the reference, float64 is used as
  ground truth when judging which of two fp32 results is closer);
* ``l1`` selects ``sum(abs(e))`` else ``sum(e*e)`` -- no square root anywhere;
* index arrays are integer numpy arrays;
* gradients are returned dense (``[rows, d]``), the layout the reference's
  autograd produces, so they compare 1:1 with ``param.grad``.
"""
from __future__ import annotations

import numpy as np

EPS_GUMBEL = 1e-20  # transUP.py:159, jTransUP.py:304


# --------------------------------------------------------------------------
# small helpers
# --------------------------------------------------------------------------
def dist(e, l1):
    """L(e): transE.py:56-61 (and every other model's last two lines)."""
    if l1:
        return np.abs(e).sum(axis=-1)
    return (e * e).sum(axis=-1)


def ddist(e, l1):
    """d L(e) / d e, as torch autograd defines it (sign(0) == 0)."""
    if l1:
        return np.sign(e).astype(e.dtype)
    return (2 * e).astype(e.dtype)


def proj_hyperplane(x, w):
    """projection_transH_pytorch: utils/misc.py:18-19.  w is NOT normalised."""
    return x - (x * w).sum(axis=-1, keepdims=True) * w


def proj_matrix(x, m_flat):
    """projection_transR_pytorch: utils/misc.py:21-26.

    ``m_flat`` is ``[B, d*d]`` holding a row-major ``[d_rel, d_ent]`` matrix;
    the result is ``M @ x`` per row.
    """
    d = x.shape[-1]
    m = m_flat.reshape(-1, m_flat.shape[-1] // d, d)
    return np.einsum("bij,bj->bi", m, x).astype(x.dtype)


def _scatter_add(rows, d, idx, vals, dtype):
    out = np.zeros((rows, d), dtype=dtype)
    np.add.at(out, np.asarray(idx).reshape(-1), vals.reshape(-1, d))
    return out


# --------------------------------------------------------------------------
# TransE  (models/transE.py)
# --------------------------------------------------------------------------
def transe_score(ent, rel, h, t, r, l1):
    """TransEModel.forward: transE.py:51-63."""
    return dist(ent[h] + rel[r] - ent[t], l1)


def transe_eval(ent, rel, q, r, l1, side, catalog=None):
    """TransEModel.evaluateHead / evaluateTail: transE.py:65-84 / 86-105.

    side == "head": q holds tail ids, c = E[t] - R[r]
    side == "tail": q holds head ids, c = E[h] + R[r]
    returns ``[B, N]`` scores against every row of ``catalog`` (default ent).
    """
    cat = ent if catalog is None else catalog
    c = ent[q] - rel[r] if side == "head" else ent[q] + rel[r]
    out = np.empty((len(q), cat.shape[0]), dtype=ent.dtype)
    for b in range(len(q)):  # one query at a time keeps [N, d] temporaries
        out[b] = dist(c[b][None, :] - cat, l1)
    return out


def transe_grads(ent, rel, h, t, r, l1, g):
    """Autograd of transE.py:51-63 given upstream ``g = dLoss/dscore [B]``."""
    e = ent[h] + rel[r] - ent[t]
    ge = g[:, None].astype(ent.dtype) * ddist(e, l1)
    d = ent.shape[1]
    g_ent = _scatter_add(ent.shape[0], d, np.concatenate([h, t]),
                         np.concatenate([ge, -ge]), ent.dtype)
    g_rel = _scatter_add(rel.shape[0], d, r, ge, ent.dtype)
    return {"ent": g_ent, "rel": g_rel}


# --------------------------------------------------------------------------
# TransH  (models/transH.py)
# --------------------------------------------------------------------------
def transh_score(ent, rel, norm, h, t, r, l1):
    """TransHModel.forward: transH.py:58-71."""
    w = norm[r]
    return dist(proj_hyperplane(ent[h], w) + rel[r] - proj_hyperplane(ent[t], w), l1)


def transh_eval(ent, rel, norm, q, r, l1, side, catalog=None):
    """TransHModel.evaluateHead / evaluateTail: transH.py:73-96 / 98-121.

    Every catalog entity is projected with the query's own hyperplane normal.
    """
    cat = ent if catalog is None else catalog
    w = norm[r]
    pq = proj_hyperplane(ent[q], w)
    c = pq - rel[r] if side == "head" else pq + rel[r]
    out = np.empty((len(q), cat.shape[0]), dtype=ent.dtype)
    for b in range(len(q)):
        pe = proj_hyperplane(cat, w[b][None, :])
        out[b] = dist(c[b][None, :] - pe, l1)
    return out


def transh_grads(ent, rel, norm, h, t, r, l1, g):
    """Autograd of transH.py:58-71 (projection misc.py:19)."""
    w = norm[r]
    x = ent[h] - ent[t]
    e = proj_hyperplane(ent[h], w) + rel[r] - proj_hyperplane(ent[t], w)
    eps = g[:, None].astype(ent.dtype) * ddist(e, l1)
    ew = (eps * w).sum(-1, keepdims=True)
    xw = (x * w).sum(-1, keepdims=True)
    gx = eps - ew * w              # d/dh ; d/dt is the negative
    gw = -(ew * x + xw * eps)
    d = ent.shape[1]
    return {
        "ent": _scatter_add(ent.shape[0], d, np.concatenate([h, t]),
                            np.concatenate([gx, -gx]), ent.dtype),
        "rel": _scatter_add(rel.shape[0], d, r, eps, ent.dtype),
        "norm": _scatter_add(norm.shape[0], d, r, gw, ent.dtype),
    }


# --------------------------------------------------------------------------
# TransR  (models/transR.py)
# --------------------------------------------------------------------------
def transr_score(ent, rel, proj, h, t, r, l1):
    """TransRModel.forward: transR.py:65-78; projection misc.py:21-26."""
    m = proj[r]
    return dist(proj_matrix(ent[h], m) + rel[r] - proj_matrix(ent[t], m), l1)


def transr_eval(ent, rel, proj, q, r, l1, side, catalog=None):
    """TransRModel.evaluateHead / evaluateTail: transR.py:80-103 / 105-128.

    The whole catalog is projected by each query's matrix (misc.py:29-33).
    """
    cat = ent if catalog is None else catalog
    d = ent.shape[1]
    m = proj[r]
    pq = proj_matrix(ent[q], m)
    c = pq - rel[r] if side == "head" else pq + rel[r]
    out = np.empty((len(q), cat.shape[0]), dtype=ent.dtype)
    for b in range(len(q)):
        mb = m[b].reshape(-1, d)
        pe = (cat @ mb.T).astype(ent.dtype)
        out[b] = dist(c[b][None, :] - pe, l1)
    return out


def transr_grads(ent, rel, proj, h, t, r, l1, g):
    """Autograd of transR.py:65-78."""
    d = ent.shape[1]
    m = proj[r].reshape(len(r), -1, d)
    x = ent[h] - ent[t]
    e = proj_matrix(ent[h], proj[r]) + rel[r] - proj_matrix(ent[t], proj[r])
    eps = g[:, None].astype(ent.dtype) * ddist(e, l1)
    gx = np.einsum("bij,bi->bj", m, eps).astype(ent.dtype)   # M^T eps
    gm = np.einsum("bi,bj->bij", eps, x).reshape(len(r), -1).astype(ent.dtype)
    return {
        "ent": _scatter_add(ent.shape[0], d, np.concatenate([h, t]),
                            np.concatenate([gx, -gx]), ent.dtype),
        "rel": _scatter_add(rel.shape[0], d, r, eps, ent.dtype),
        "proj": _scatter_add(proj.shape[0], proj.shape[1], r, gm, ent.dtype),
    }


# --------------------------------------------------------------------------
# TUP preference induction  (models/transUP.py:105-170, jTransUP.py:250-315)
# --------------------------------------------------------------------------
def softmax_last(x):
    """masked_softmax (no masking, eps unused): transUP.py:138-141."""
    m = x.max(axis=-1, keepdims=True)
    ex = np.exp(x - m)
    return (ex / ex.sum(axis=-1, keepdims=True)).astype(x.dtype)


def st_gumbel_softmax(logits, u):
    """st_gumbel_softmax: transUP.py:143-170 with the uniform draw ``u`` given.

    Returns (p_forward, y, k_star).  ``p_forward = (onehot - y) + y`` evaluated
    in the table dtype exactly as the reference's ``(y_hard - y).detach() + y``.
    """
    dt = logits.dtype
    eps = dt.type(EPS_GUMBEL)
    noise = -np.log(-np.log(u.astype(dt) + eps) + eps)     # :160-161
    y = softmax_last((logits + noise).astype(dt))             # :162-163, T=1
    k = y.argmax(axis=-1)                                     # :164
    hard = np.zeros_like(y)
    np.put_along_axis(hard, k[..., None], 1, axis=-1)         # :165-167
    p = ((hard - y) + y).astype(dt)                           # :168
    return p, y, k


def tup_preferences(s, pref, pref_norm, gumbel_u=None, half=False):
    """getPreferences: transUP.py:105-115 (half=False), jTransUP.py:250-260 (half=True).

    ``s`` = u_e + i_e ``[..., d]``; ``pref``/``pref_norm`` the (possibly summed)
    preference tables.  Non-Gumbel mode mixes with the RAW logits (no softmax).
    Returns (p, r_e, w, y) with y None in non-Gumbel mode.
    """
    dt = s.dtype
    z = (s @ pref.T).astype(dt) / dt.type(2)
    y = None
    if gumbel_u is not None:
        p, y, _ = st_gumbel_softmax(z, gumbel_u)
    else:
        p = z
    r_e = (p @ pref).astype(dt)
    w = (p @ pref_norm).astype(dt)
    if half:
        r_e = r_e / dt.type(2)
        w = w / dt.type(2)
    return p, r_e, w, y


def _tup_pair_score(u_e, i_e, pref, pref_norm, l1, gumbel_u, half):
    _, r_e, w, _ = tup_preferences(u_e + i_e, pref, pref_norm, gumbel_u, half)
    return dist(proj_hyperplane(u_e, w) + r_e - proj_hyperplane(i_e, w), l1)


def tup_score(user, item, pref, pref_norm, u, i, l1, gumbel_u=None):
    """TransUPModel.forward: transUP.py:69-82.  gumbel_u: ``[B, P]`` or None."""
    return _tup_pair_score(user[u], item[i], pref, pref_norm, l1, gumbel_u, False)


def tup_eval(user, item, pref, pref_norm, u, l1, gumbel_u=None):
    """TransUPModel.evaluate: transUP.py:84-102.  gumbel_u: ``[B, I, P]`` or None."""
    out = np.empty((len(u), item.shape[0]), dtype=user.dtype)
    for b in range(len(u)):
        ue = np.broadcast_to(user[u[b]], item.shape)
        gu = None if gumbel_u is None else gumbel_u[b]
        out[b] = _tup_pair_score(ue, item, pref, pref_norm, l1, gu, False)
    return out


def _tup_pair_grads(u_e, i_e, pref, pref_norm, l1, g, gumbel_u, half):
    """Shared backward of the TUP / KTUP-rec pair score.

    Returns (g_u_e, g_i_e, g_pref, g_pref_norm) with the table grads dense.
    """
    dt = u_e.dtype
    hf = dt.type(0.5) if half else dt.type(1)
    s = u_e + i_e
    p, r_e, w, y = tup_preferences(s, pref, pref_norm, gumbel_u, half)
    x = u_e - i_e
    e = proj_hyperplane(u_e, w) + r_e - proj_hyperplane(i_e, w)
    eps = g[:, None].astype(dt) * ddist(e, l1)
    ew = (eps * w).sum(-1, keepdims=True)
    xw = (x * w).sum(-1, keepdims=True)
    gx = eps - ew * w
    gw = -(ew * x + xw * eps)
    # r = hf * p @ pref ; w = hf * p @ pref_norm
    gp = hf * ((eps @ pref.T) + (gw @ pref_norm.T))
    g_pref = hf * (p.T @ eps)
    g_pnorm = hf * (p.T @ gw)
    if y is not None:   # straight-through: backward through y = softmax(z + noise)
        gz = y * (gp - (y * gp).sum(-1, keepdims=True))
    else:
        gz = gp
    gs = (gz @ pref) / dt.type(2)
    g_pref = g_pref + (gz.T @ s) / dt.type(2)
    return ((gx + gs).astype(dt), (-gx + gs).astype(dt),
            g_pref.astype(dt), g_pnorm.astype(dt))


def tup_grads(user, item, pref, pref_norm, u, i, l1, g, gumbel_u=None):
    """Autograd of transUP.py:69-82 (+105-115, 143-170)."""
    gu, gi, gp, gn = _tup_pair_grads(user[u], item[i], pref, pref_norm, l1, g, gumbel_u, False)
    d = user.shape[1]
    return {
        "user": _scatter_add(user.shape[0], d, u, gu, user.dtype),
        "item": _scatter_add(item.shape[0], d, i, gi, user.dtype),
        "pref": gp, "pref_norm": gn,
    }


# --------------------------------------------------------------------------
# KTUP / jTransUP  (models/jTransUP.py)
# --------------------------------------------------------------------------
def ktup_item2ent(i_map, new_map, item_total, pad_index):
    """paddingItems: jTransUP.py:114-120 as a lookup table built once.

    ``i_map[item] -> joint index``; ``new_map[joint][0] -> entity id or -1``.
    """
    out = np.empty(item_total, dtype=np.int64)
    for it in range(item_total):
        ent_id = new_map[i_map[it]][0]
        out[it] = ent_id if ent_id != -1 else pad_index
    return out


def ktup_rec_score(user, item, ent, rel, norm, pref, pref_norm, item2ent, u, i, l1, gumbel_u=None):
    """jTransUPModel.forward(is_rec=True): jTransUP.py:124-143 (+250-260)."""
    ie = item[i] + ent[item2ent[i]]
    return _tup_pair_score(user[u], ie, pref + rel, pref_norm + norm, l1, gumbel_u, True)


def ktup_rec_eval(user, item, ent, rel, norm, pref, pref_norm, item2ent, u, l1, gumbel_u=None):
    """jTransUPModel.evaluateRec: jTransUP.py:163-191 (all items, not shared)."""
    ie = item + ent[item2ent]
    p2, n2 = pref + rel, pref_norm + norm
    out = np.empty((len(u), item.shape[0]), dtype=user.dtype)
    for b in range(len(u)):
        ue = np.broadcast_to(user[u[b]], ie.shape)
        gu = None if gumbel_u is None else gumbel_u[b]
        out[b] = _tup_pair_score(ue, ie, p2, n2, l1, gu, True)
    return out


def ktup_rec_grads(user, item, ent, rel, norm, pref, pref_norm, item2ent, u, i, l1, g, gumbel_u=None):
    """Autograd of jTransUP.py:124-143.  The padding entity row gets no gradient
    (``padding_idx`` of ent_embeddings, jTransUP.py:96)."""
    a = item2ent[i]
    ie = item[i] + ent[a]
    gu, gie, gp, gn = _tup_pair_grads(user[u], ie, pref + rel, pref_norm + norm, l1, g, gumbel_u, True)
    d = user.shape[1]
    g_ent = _scatter_add(ent.shape[0], d, a, gie, user.dtype)
    g_ent[ent.shape[0] - 1] = 0
    return {
        "user": _scatter_add(user.shape[0], d, u, gu, user.dtype),
        "item": _scatter_add(item.shape[0], d, i, gie, user.dtype),
        "ent": g_ent,
        "pref": gp, "rel": gp.copy(),
        "pref_norm": gn, "norm": gn.copy(),
    }


# KTUP's KG branch (jTransUP.py:144-157) and evaluateHead/Tail (193-247) are
# TransH on (ent [E+1 rows incl. the zero padding row], rel, norm): use
# transh_score / transh_eval / transh_grads with those tables.


# --------------------------------------------------------------------------
# ranking losses  (utils/loss.py)
# --------------------------------------------------------------------------
def margin_loss(pos, neg, margin):
    """marginLoss.forward: loss.py:12-16 -- a SUM over the batch."""
    return np.maximum(pos - neg + pos.dtype.type(margin), 0).sum(dtype=pos.dtype)


def margin_loss_grads(pos, neg, margin):
    act = ((pos - neg + pos.dtype.type(margin)) > 0).astype(pos.dtype)
    return act, -act


def bpr_loss(pos, neg, target):
    """bprLoss: loss.py:29-31 -- mean of -logsigmoid(target * (pos - neg))."""
    x = pos.dtype.type(target) * (pos - neg)
    # -logsigmoid(x) = softplus(-x), evaluated stably
    sp = np.maximum(-x, 0) + np.log1p(np.exp(-np.abs(x)))
    return sp.mean(dtype=pos.dtype)


def bpr_loss_grads(pos, neg, target):
    x = pos.dtype.type(target) * (pos - neg)
    sig_neg = 1 / (1 + np.exp(x))               # sigmoid(-x)
    gp = (-pos.dtype.type(target) * sig_neg / pos.dtype.type(pos.size)).astype(pos.dtype)
    return gp, -gp


def orthogonal_loss(rel_rows, norm_rows):
    """orthogonalLoss: loss.py:18-19."""
    return (((norm_rows * rel_rows).sum(1) ** 2) / (rel_rows ** 2).sum(1)).sum()


def norm_loss(rows):
    """normLoss: loss.py:21-23."""
    return np.maximum((rows ** 2).sum(1) - 1, 0).sum()


def norm_loss_grads(rows):
    """d normLoss / d rows: 2 x on the rows outside the unit sphere (torch's max(., 0) passes the
    gradient where the first argument is the larger one)."""
    return (2 * rows * ((rows ** 2).sum(1, keepdims=True) > 1)).astype(rows.dtype)


def orthogonal_loss_grads(rel_rows, norm_rows):
    """(d/d rel, d/d norm) of orthogonalLoss = sum (w.r)^2 / |r|^2."""
    wr = (norm_rows * rel_rows).sum(1, keepdims=True)
    n2 = (rel_rows ** 2).sum(1, keepdims=True)
    q = wr / n2
    return (2 * q * norm_rows - 2 * q * q * rel_rows).astype(rel_rows.dtype), (2 * q * rel_rows).astype(rel_rows.dtype)


# --------------------------------------------------------------------------
# full-catalog ranking  (utils/misc.py:125-146, 213-248; utils/evaluation.py)
# --------------------------------------------------------------------------
def sort_order(scores):
    """Ascending order with ties broken by id (``(score, id)`` lexicographic).

    The reference uses ``np.argsort`` (misc.py:127, 215) whose tie order is
    unspecified; this is the tie rule the CUDA path implements.
    """
    return np.argsort(scores, kind="stable")


def rec_topk(scores, filt, topn):
    """Top-n unfiltered ids of one user: the walk in getRecPerformance, misc.py:213-229."""
    out = []
    for rid in sort_order(scores):
        if filt is not None and int(rid) in filt:
            continue
        out.append(int(rid))
        if len(out) >= topn:
            break
    return out


def dcg_at_k(r, k, method=0):
    """dcg_at_k: utils/evaluation.py:41-78 (np.asfarray spelled out)."""
    r = np.asarray(r, dtype=float)[:k]
    if r.size:
        if method == 0:
            return r[0] + np.sum(r[1:] / np.log2(np.arange(2, r.size + 1)))
        if method == 1:
            return np.sum(r / np.log2(np.arange(2, r.size + 2)))
        raise ValueError("method must be 0 or 1.")
    return 0.0


def ndcg_at_k(r, k, method=0):
    """ndcg_at_k: utils/evaluation.py:80-110."""
    dcg_max = dcg_at_k(sorted(r, reverse=True), k, method)
    if not dcg_max:
        return 0.0
    return dcg_at_k(r, k, method) / dcg_max


def rec_metrics(top_ids, gold):
    """f1, p, r, hit, ndcg from the top list: misc.py:231-248."""
    hits = [1 if i in gold else 0 for i in top_ids]
    n_hit = sum(hits)
    if n_hit == 0:
        return 0.0, 0.0, 0.0, 0, 0.0
    k = len(hits)
    p = n_hit / k
    r = n_hit / len(gold)
    return 2 * p * r / (p + r), p, r, 1, ndcg_at_k(hits, k)


def kg_ranks(scores, gold, filt, topn):
    """getKGPerformance: misc.py:125-146.

    rank(g) = number of unfiltered, non-gold ids sorted before g; hit = rank < topn.
    Returns {gold id: (hit, rank)} (a filtered gold id is never reached, as in
    the reference).
    """
    out = {}
    cur = 0
    for rid in sort_order(scores):
        rid = int(rid)
        if filt is not None and rid in filt:
            continue
        if rid in gold:
            out[rid] = (1 if cur < topn else 0, cur)
            if len(out) == len(gold):
                break
        else:
            cur += 1
    return out
