"""Literal restatement of RecBole 1.0.1's GAUC and item-distribution metrics (evaluator/metrics.py GAUC, ItemCoverage,
AveragePopularity, GiniIndex, ShannonEntropy, TailPercentage; evaluator/collector.py rec.meanrank and _average_rank), written as
loops over users and items the way the reference code is, so the vectorised evaluator can be checked against it.

GAUC goes through the reference's own route: the [B, n_items] score matrix (-inf where an item is not a candidate) is sorted
descending, _average_rank gives tied items their average 1-based rank, the positive's entry is picked out, and user_len is the
argmin of the sorted row (the first -inf).  The meanrank tensor is float32, as the collector's is."""
from collections import Counter

import numpy as np
import torch


def average_rank(scores):
    """collector.py _average_rank: 1-based average rank of every entry of rows sorted descending"""
    length, width = scores.shape
    true_tensor = torch.full((length, 1), True, dtype=torch.bool)
    obs = torch.cat([true_tensor, scores[:, 1:] != scores[:, :-1]], dim=1)
    bias = torch.arange(0, length).repeat(width).reshape(width, -1).transpose(1, 0).reshape(-1)
    dense = obs.view(-1).cumsum(0) + bias
    count = torch.where(torch.cat([obs, true_tensor], dim=1))[1]
    return .5 * (count[dense] + count[dense - 1] + 1).view(length, -1)


def mean_rank(scores, positive):
    """collector.py eval_batch_collect 'rec.meanrank': scores [B, n_items] (non-candidates -inf), one positive item per row ->
    [B, 3] float32 (pos_rank_sum, user_len, pos_len)"""
    scores = torch.as_tensor(scores)
    desc_scores, desc_index = torch.sort(scores, dim=-1, descending=True)
    pos_matrix = torch.zeros_like(scores)
    pos_matrix[torch.arange(scores.shape[0]), torch.as_tensor(positive)] = 1
    pos_index = torch.gather(pos_matrix, dim=1, index=desc_index)
    avg_rank = average_rank(desc_scores)
    pos_rank_sum = torch.where(pos_index == 1, avg_rank, torch.zeros_like(avg_rank)).sum(dim=-1, keepdim=True)
    pos_len_list = torch.sum(pos_matrix, dim=1, keepdim=True)
    user_len_list = desc_scores.argmin(dim=1, keepdim=True)
    return torch.cat((pos_rank_sum, user_len_list, pos_len_list), dim=1)


def gauc(meanrank):
    """metrics.py GAUC.metric_info"""
    meanrank = np.asarray(meanrank)
    pos_rank_sum, user_len_list, pos_len_list = (a.squeeze(-1) for a in np.split(meanrank, 3, axis=1))
    neg_len_list = user_len_list - pos_len_list
    non_zero_idx = np.full(len(user_len_list), True, dtype=bool)
    non_zero_idx *= (pos_len_list != 0)
    non_zero_idx *= (neg_len_list != 0)
    user_len_list, neg_len_list, pos_len_list, pos_rank_sum = (x[non_zero_idx] for x in (user_len_list, neg_len_list, pos_len_list,
                                                                                          pos_rank_sum))
    pair_num = (user_len_list + 1) * pos_len_list - pos_len_list * (pos_len_list + 1) / 2 - np.squeeze(pos_rank_sum)
    user_auc = pair_num / (neg_len_list * pos_len_list)
    return (user_auc * pos_len_list).sum() / pos_len_list.sum()


def item_coverage(item_matrix, num_items):
    return np.unique(item_matrix).shape[0] / num_items


def _topk_mean(values, k):
    result = values.cumsum(axis=1) / np.arange(1, values.shape[1] + 1)
    return result.mean(axis=0)[k - 1]


def average_popularity(item_matrix, item_count, k):
    """item_count: dict item id -> training rows (data.count_items; ids absent count 0)"""
    value = np.zeros_like(item_matrix)
    for i in range(item_matrix.shape[0]):
        row = item_matrix[i, :]
        for j in range(row.shape[0]):
            value[i][j] = item_count.get(row[j], 0)
    return _topk_mean(value, k)


def gini_index(item_matrix, num_items):
    item_count = dict(Counter(item_matrix.flatten()))
    sorted_count = np.array(sorted(item_count.values()))
    num_recommended_items = sorted_count.shape[0]
    total_num = item_matrix.shape[0] * item_matrix.shape[1]
    idx = np.arange(num_items - num_recommended_items + 1, num_items + 1)
    gini = np.sum((2 * idx - num_items - 1) * sorted_count) / total_num
    return gini / num_items


def shannon_entropy(item_matrix):
    item_count = dict(Counter(item_matrix.flatten()))
    total_num = item_matrix.shape[0] * item_matrix.shape[1]
    result = 0.0
    for cnt in item_count.values():
        p = cnt / total_num
        result += -p * np.log(p)
    return result / len(item_count)


def tail_percentage(item_matrix, count_items, k, tail_ratio):
    tail = tail_ratio
    if tail is None or tail <= 0:
        tail = 0.1
    if tail > 1:
        tail_items = [item for item, cnt in count_items.items() if cnt <= tail]
    else:
        count_items = sorted(count_items.items(), key=lambda kv: (kv[1], kv[0]))
        cut = max(int(len(count_items) * tail), 1)
        tail_items = [item for item, cnt in count_items[:cut]]
    value = np.zeros_like(item_matrix)
    for i in range(item_matrix.shape[0]):
        row = item_matrix[i, :]
        for j in range(row.shape[0]):
            value[i][j] = 1 if row[j] in tail_items else 0
    return _topk_mean(value, k)


def evaluate(metrics, topk, scores, positive, item_matrix, num_items, item_count, tail_ratio=None, decimal_place=4):
    """the six metrics above for `metrics` (lower-case RecBole names) -> {key: rounded value}.  scores [B, n_items] with -inf on
    non-candidates (for GAUC), item_matrix [B, kmax] the top-k ids, item_count {id: training rows}"""
    out = {}
    for m in metrics:
        if m == 'gauc':
            out['gauc'] = round(float(gauc(mean_rank(scores, positive).numpy())), decimal_place)
            continue
        for k in topk:
            rk = item_matrix[:, :k]
            if m == 'itemcoverage':
                v = item_coverage(rk, num_items)
            elif m == 'averagepopularity':
                v = average_popularity(item_matrix, item_count, k)
            elif m == 'giniindex':
                v = gini_index(rk, num_items)
            elif m == 'shannonentropy':
                v = shannon_entropy(rk)
            elif m == 'tailpercentage':
                v = tail_percentage(item_matrix, item_count, k, tail_ratio)
            else:
                raise KeyError(m)
            out['%s@%d' % (m, k)] = round(float(v), decimal_place)
    return out
