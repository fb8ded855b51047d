"""Negative sampling and sampled-candidate evaluation restated plainly (RecBole 1.0.1: recbole/sampler/sampler.py,
trainer/trainer.py _neg_sample_batch_eval, evaluator/collector.py eval_batch_collect) -- the oracle the device sampler
(acsr_neg_sample) and ranking (acsr_candidate_rank) are checked against, beside acsr_oracle.py."""
import numpy as np
import torch


def used_ids(splits, n_users, phase):
    """sampler.py get_used_ids: for phase p (0 train, 1 valid, 2 test) the set of target item ids of every row of user u in the
    splits 0..p.  splits: [(user_id array, item_id array)] of train / valid / test."""
    used = [set() for _ in range(n_users)]
    for uid, iid in splits[:phase + 1]:
        for u, i in zip(np.asarray(uid).tolist(), np.asarray(iid).tolist()):
            used[u].add(i)
    return used


def popularity_probs(splits, n_items):
    """the popularity distribution: each item's count among the targets of all rows of all splits, normalised"""
    counts = np.zeros(n_items, dtype=np.float64)
    for _, iid in splits:
        np.add.at(counts, np.asarray(iid), 1.0)
    return counts / counts.sum()


def alias_probs(prob, alias):
    """the distribution an alias table (prob[i], alias[i]) draws from: column i uniform, then i with probability prob[i]"""
    prob = np.asarray(prob, dtype=np.float64)
    n = len(prob)
    p = prob.copy()
    np.add.at(p, np.asarray(alias), 1.0 - prob)
    return p / n


def sampled_topk(scores, cand, n_items, kmax):
    """RecBole's way: scatter the candidate scores (column 0 the positive) into a -inf [B, n_items] matrix (duplicate candidates
    collapse onto one entry), torch.topk, hit flags of the positive -> (flags [B, kmax] int32, topk_idx, the scattered matrix)"""
    B = scores.shape[0]
    full = torch.full((B, n_items), -float('inf'), dtype=torch.float64)
    full.scatter_(1, cand.long(), scores.double())
    _, idx = torch.topk(full, kmax, dim=-1)
    return (idx == cand[:, :1].long()).to(torch.int32), idx, full


def sampled_rank_bounds(full, pos, tol=0.0):
    """per row the interval [lo, hi] of ranks of the positive that are right up to ties within tol: lo = number of other
    candidates scoring more than s_pos + tol, hi = number scoring at least s_pos - tol"""
    s0 = full.gather(1, pos.view(-1, 1).long())
    other = torch.isfinite(full)
    other.scatter_(1, pos.view(-1, 1).long(), False)
    lo = ((full > s0 + tol) & other).sum(1)
    hi = ((full >= s0 - tol) & other).sum(1)
    return lo, hi


def flags_rank(flags, kmax):
    """rank of the positive encoded by hit flags (the first kmax columns of [B, kmax] or [B, kmax+1]); kmax when it is absent"""
    hit = torch.as_tensor(flags)[:, :kmax].to(torch.int64)
    return torch.where(hit.sum(1) > 0, hit.argmax(1), torch.full_like(hit[:, 0], kmax))
