"""Sampled-candidate evaluation cost at the C2 shape (V = 12 102, 2 layers, 2 heads, d 64, inner 256, L 50, B 256, N 100).

    python scripts/sampled_eval_micro.py [--users 8192] [--neg 100] [--out DIR]

Prints one JSON line:
  - eval users/s of the trainer's graphed full-sort batch and of its graphed sampled batch (sampler + encoder + rank), each
    timed over whole passes with CUDA events after a warm-up pass;
  - the per-launch device time of acsr_neg_sample and acsr_candidate_rank, each captured `reps` times back to back in one CUDA
    graph and replayed (as bench.py times kernels), with their algorithmic bytes and the implied bandwidth;
  - the GPU's name and power limit, which every number here depends on.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import ac_tsr_b200 as A  # noqa: E402
from oracle import acsr_oracle as O  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
        return r.stdout.strip().splitlines()[0]
    except Exception:
        return torch.cuda.get_device_name(0)


def time_pass(fn, batches, reps):
    fn_all = lambda: [fn(b) for b in batches]      # noqa: E731
    fn_all()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn_all()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def kernel_us(launch, reps=50):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        launch()
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(reps):
                launch()
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            g.replay()
        e1.record()
        side.synchronize()
    torch.cuda.current_stream().wait_stream(side)
    return e0.elapsed_time(e1) * 1e3 / (4 * reps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--users', type=int, default=8192)
    ap.add_argument('--neg', type=int, default=100)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('sampled_eval_micro.py measures on the GPU; no CUDA device found')
    A.LIB.load()
    V, B, N, n = 12102, a.batch, a.neg, a.users
    d = dict(O.default_cfg(), USER_ID_FIELD='user_id', ITEM_ID_FIELD='item_id', LIST_SUFFIX='_list', ITEM_LIST_LENGTH_FIELD='item_length',
             NEG_PREFIX='neg_', device=torch.device('cuda'), seed=42, learning_rate=1e-3, epochs=1, eval_batch_size=B,
             train_batch_size=B, topk=[1, 5, 10, 20, 50], metrics=['Hit', 'MRR', 'NDCG', 'Recall'], valid_metric='Hit@10',
             checkpoint_dir='/tmp/acsr_micro_ckpt')
    config = A.Config(model='ACSASRec', config_dict=d)
    ds = A.data.SyntheticSequentialDataset(config, n, V, seed=3)
    f = ds.inter_feat
    off, items = A.ops.used_item_csr(f['user_id'].numpy(), f['item_id'].numpy(), n + 1, V)
    torch.manual_seed(0)
    model = A.ACSASRec(config, ds).cuda()
    trainer = A.ACSASRecTrainer(config, model)
    model.eval()
    res = {'gpu': gpu_info(), 'shape': dict(V=V, B=B, N=N, users=n, d=64, L=50, layers=2, heads=2)}
    full_batches = list(A.data.FullSortEvalDataLoader(config, ds))
    with torch.no_grad():
        t_full = time_pass(lambda b: trainer.eval_batch(b), full_batches, a.reps)
    res['full_sort_users_per_s'] = round(n / t_full, 1)
    for dist in ('uniform', 'popularity'):
        s = A.ops.NegSampler(dist, off, items, V, seed=42, phase=1, counts=np.bincount(f['item_id'].numpy(), minlength=V))
        loader = A.data.NegSampleEvalDataLoader(config, ds, s, N)
        batches = list(loader)
        with torch.no_grad():
            t = time_pass(lambda b: trainer.eval_batch(b, neg_sampler=s, neg_num=N), batches, a.reps)
        res['sampled_%s_users_per_s' % dist] = round(n / t, 1)
    # per-launch kernel times at one batch
    s = A.ops.NegSampler('uniform', off, items, V, seed=42).to_device('cuda')
    sp = A.ops.NegSampler('popularity', off, items, V, seed=42, counts=np.bincount(f['item_id'].numpy(), minlength=V)).to_device('cuda')
    users = f['user_id'][:B].cuda()
    pos = f['item_id'][:B].cuda()
    cand = torch.empty((B, N + 1), dtype=torch.int64, device='cuda')
    cand[:, 0] = pos
    out = torch.randn(B, 64, device='cuda') * 0.3
    table = model.item_embedding.weight.detach()
    kmax = max(config['topk'])
    for name, smp in (('neg_sample_uniform', s), ('neg_sample_popularity', sp)):
        us = kernel_us(lambda: smp.draw(users, N, positives=pos, out=cand[:, 1:], ld=N + 1, advance=False))
        ab = A._lib.ALGO_BYTES['acsr_neg_sample']((None,) * 5 + (B, N))
        res[name] = dict(us=round(us, 2), algo_bytes=ab, gb_per_s=round(ab / us / 1e3, 1))
    rec = torch.empty((B, kmax + 1), dtype=torch.int32, device='cuda')

    def rank():
        A.LIB.call('acsr_candidate_rank', out.data_ptr(), table.data_ptr(), V, 64, cand.data_ptr(), B, N + 1, kmax, rec.data_ptr(),
                   None, torch.cuda.current_stream().cuda_stream)
    us = kernel_us(rank)
    ab = A._lib.ALGO_BYTES['acsr_candidate_rank']((None, None, V, 64, None, B, N + 1, kmax, None, None, None))
    res['candidate_rank'] = dict(us=round(us, 2), algo_bytes=ab, gb_per_s=round(ab / us / 1e3, 1))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'sampled_eval_micro.json'), 'w') as fh:
            fh.write(line + '\n')


if __name__ == '__main__':
    main()
