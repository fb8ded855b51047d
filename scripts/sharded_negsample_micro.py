"""Cost of sampled evaluation and BPR training over a vocab-sharded item table, at 1M items (B 256, N 100, d 64, L 50, the
default 2-layer encoder).  Run with one process per GPU:

    torchrun --standalone --nproc_per_node=2 scripts/sharded_negsample_micro.py [--out DIR]

Prints one JSON line on rank 0 (and writes it to DIR/sharded_negsample_micro.json):
  - the per-launch device time of each shard kernel at the shapes rank 0 runs (each captured `reps` times back to back in one
    CUDA graph and replayed, as bench.py times kernels), with its algorithmic bytes;
  - sampled-evaluation users/s of the trainer's graphed batch on the sharded table (all ranks' users over the wall time),
    next to the same trainer on one GPU with the replicated table;
  - the graphed BPR step in ms of vocab-parallel training on the sharded table, next to batch data-parallel training with a
    replicated table (dense all-reduce of the table gradient, full-size Adam moments on every rank);
  - every GPU's name and power limit, which every number here depends on.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

import ac_tsr_b200 as A  # noqa: E402
from oracle import acsr_oracle as O  # noqa: E402
from sampled_eval_micro import kernel_us  # noqa: E402


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--items', type=int, default=1000000)
    ap.add_argument('--users', type=int, default=4096, help='evaluation users per rank')
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    A.LIB.load()
    V, B, N, d, L, n = a.items, 256, 100, 64, 50, a.users
    cfg = dict(O.default_cfg(loss_type='BPR'), USER_ID_FIELD='user_id', ITEM_ID_FIELD='item_id', LIST_SUFFIX='_list',
               ITEM_LIST_LENGTH_FIELD='item_length', NEG_PREFIX='neg_', device=dev, seed=42, learning_rate=1e-3, epochs=1,
               eval_batch_size=B, train_batch_size=B, topk=[1, 5, 10, 20, 50], metrics=['Hit', 'MRR', 'NDCG', 'Recall'],
               valid_metric='Hit@10', checkpoint_dir='/tmp/acsr_micro_ckpt_%d' % rank, MAX_ITEM_LIST_LENGTH=L)
    config = A.Config(model='ACSASRec', config_dict=cfg)
    ds = A.data.SyntheticSequentialDataset(config, n, V, seed=3 + rank)
    f = ds.inter_feat
    off, items = A.ops.used_item_csr(f['user_id'].numpy(), f['item_id'].numpy(), n + 1, V)
    res = {'gpus': gpu_info(), 'world': world, 'shape': dict(V=V, B=B, N=N, d=d, L=L, eval_users_per_rank=n, layers=2, heads=2)}
    g = torch.Generator().manual_seed(7 + rank)
    seq = torch.randint(1, V, (B, L), generator=g)
    inter = A.Interaction({'item_id_list': seq.to(dev), 'item_length': torch.full((B,), L).to(dev),
                           'item_id': torch.randint(1, V, (B,), generator=g).to(dev),
                           'neg_item_id': torch.randint(1, V, (B,), generator=g).to(dev)})

    def build(mode):
        torch.manual_seed(0)
        model = A.ACSASRec(config, ds).to(dev)
        trainer = A.ACSASRecTrainer(config, model)
        if mode == 'dp':
            trainer.enable_data_parallel()
        elif mode == 'vp_sharded':
            trainer.enable_data_parallel(vocab_parallel=True, shard_table=True)
        return model, trainer

    def eval_users_per_s(model, trainer, users):
        s = A.ops.NegSampler('uniform', off, items, V, seed=42 + rank, phase=1)
        batches = list(A.data.NegSampleEvalDataLoader(config, ds, s, N))
        model.eval()
        with torch.no_grad():
            ms = timed(lambda: [trainer.eval_batch(b, neg_sampler=s, neg_num=N) for b in batches], 3)
        return round(users / (ms / 1e3), 1)

    # ---- BPR step: data-parallel with a replicated table vs vocab-parallel on the sharded table ----
    for mode in ('dp', 'vp_sharded'):
        model, trainer = build(mode)
        model.train()
        res['bpr_step_ms_' + mode] = round(timed(lambda: trainer.graphed_step(inter), a.steps), 3)
        if mode == 'vp_sharded':
            res['sampled_eval_users_per_s_sharded'] = eval_users_per_s(model, trainer, world * n)
            vp = trainer.vp
        del trainer, model
        torch.cuda.empty_cache()
        dist.barrier()
    # ---- one GPU, replicated table: the single-GPU sampled-evaluation figure ----
    if rank == 0:
        model, trainer = build('single')
        s = A.ops.NegSampler('uniform', off, items, V, seed=42, phase=1)
        batches = list(A.data.NegSampleEvalDataLoader(config, ds, s, N))
        model.eval()
        with torch.no_grad():
            for b in batches:
                trainer.eval_batch(b, neg_sampler=s, neg_num=N)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                for b in batches:
                    trainer.eval_batch(b, neg_sampler=s, neg_num=N)
            e1.record()
            torch.cuda.synchronize()
        res['sampled_eval_users_per_s_single_gpu_replicated'] = round(n / (e0.elapsed_time(e1) / 3 / 1e3), 1)
        # ---- per-launch kernel times at rank 0's shapes ----
        W = world
        ab = A._lib.ALGO_BYTES
        shard = torch.randn(vp.per, d, device=dev) * 0.1
        lo, hi = vp.lo, vp.hi
        out_all = torch.randn(W * B, d, device=dev)
        cand_all = torch.randint(0, V, (W * B, N + 1), device=dev)
        scores = torch.empty((W * B, N + 1), device=dev)
        kmax = 50
        rec = torch.empty((B, kmax + 1), dtype=torch.int32, device=dev)
        cnt = torch.empty((B, 3), dtype=torch.int32, device=dev)
        o2 = torch.randn(2 * W * B, d, device=dev)
        pos2 = torch.randint(1, V, (2 * W * B,), device=dev)
        neg2 = torch.randint(1, V, (2 * W * B,), device=dev)
        dots = torch.empty((2 * W * B, 2), device=dev)
        rx, rl, loss = torch.zeros(2 * B, device=dev), torch.empty(2 * B, device=dev), torch.empty(2, device=dev)
        rx2, rs2 = torch.zeros(2 * W * B, device=dev), torch.full((2 * W * B,), 1.0 / B, device=dev)
        d_out = torch.empty_like(o2)
        sg = torch.zeros_like(shard)
        st = lambda: torch.cuda.current_stream().cuda_stream      # noqa: E731
        calls = {
            'acsr_candidate_scores_shard': (out_all.data_ptr(), shard.data_ptr(), lo, hi, V, d, cand_all.data_ptr(),
                                            W * B, N + 1, scores.data_ptr()),
            'acsr_candidate_rank_scores': (scores.data_ptr(), cand_all.data_ptr(), V, B, N + 1, kmax, rec.data_ptr(), cnt.data_ptr()),
            'acsr_bpr_dots_shard': (o2.data_ptr(), shard.data_ptr(), lo, hi, V, pos2.data_ptr(), neg2.data_ptr(), 2 * W * B, d,
                                    dots.data_ptr()),
            'acsr_bpr_loss_from_dots': (dots.data_ptr(), 2 * B, 2, 1e-10, rx.data_ptr(), rl.data_ptr(), loss.data_ptr()),
            'acsr_bpr_loss_bwd_shard': (o2.data_ptr(), shard.data_ptr(), lo, hi, V, pos2.data_ptr(), neg2.data_ptr(), rx2.data_ptr(),
                                        rs2.data_ptr(), 2 * W * B, d, 1e-10, 0, W * B, d_out.data_ptr(), sg.data_ptr()),
        }
        kern = {}
        for name, args in calls.items():
            us = kernel_us(lambda: A.LIB.call(name, *args, st()))
            b = ab[name](args + (None,))
            kern[name] = dict(us=round(us, 2), algo_bytes=b, gb_per_s=round(b / us / 1e3, 1))
        res['kernels'] = kern
        line = json.dumps(res)
        print(line)
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            with open(os.path.join(a.out, 'sharded_negsample_micro.json'), 'w') as fh:
                fh.write(line + '\n')
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
