"""Run under torchrun with 2+ GPUs (one rank per GPU: NCCL cannot put two ranks on one device).  loss_type BPR and sampled
evaluation in the three multi-GPU modes of the trainer, on the same synthetic data:
  (a) batch data-parallel, replicated item table (dense all-reduce of the flat gradient)          -- the reference point
  (b) vocab-parallel over a replicated table (each table row scored by its owner, reduce-scatter of the dots and of d_out)
  (c) vocab-parallel with SHARDED table storage (rows, gradient and Adam moments on the owner only)
Checked: both losses, every gradient (the sharded table gradient gathered back to the reference layout), the parameters after
two optimisation steps through the CUDA-graph path, sampled ranking of the same explicit candidates (rec and counts identical
in all three modes), and trainer.evaluate on a uni100 loader graphed and eager on the sharded table.  Prints one 'ok' line
on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def main():
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    import ac_tsr_b200 as A
    from oracle import acsr_oracle as O
    from test_gpu_negsample import make_config
    cfg = O.default_cfg(loss_type='BPR', hidden_dropout_prob=0.0, attn_dropout_prob=0.0)
    V, B, L, k, N, n_users = 5003, 64, 50, 50, 100, 512
    params = O.init_params(cfg, V, seed=11)
    seq, ln, pos = O.synth_batch(B * world, L, V, seed=12)
    gen = torch.Generator().manual_seed(13)
    neg = torch.randint(1, V, (B * world,), generator=gen)
    cand = torch.randint(0, V, (B * world, N + 1), generator=gen)
    cand[:, 0] = pos
    cand[::3, 5] = cand[::3, 0]                                        # the positive again among the negatives
    cand[:, 7:9] = cand[:, 6:7]                                        # duplicates
    sl = slice(rank * B, (rank + 1) * B)
    g = torch.Generator().manual_seed(100 + rank)
    noise = {(l, 'noise'): torch.randn(B, cfg['n_heads'], L, L, generator=g).to(dev) for l in range(cfg['n_layers'])}
    modes = [('dp', False, False), ('vocab-parallel', True, False), ('vocab-parallel + sharded table', True, True)]
    res = {}
    for name, vocab_parallel, shard in modes:
        config = make_config(A, cfg, device=dev, checkpoint_dir='/tmp/acsr_mgpu_neg_%d' % rank, train_batch_size=B)
        ds = A.data.SyntheticSequentialDataset(config, n_users, V, seed=30 + rank)         # different users on every rank
        model = A.ACSASRec(config, ds).to(dev)
        model.load_state_dict({kk: v.to(dev) for kk, v in params.items()})
        model._debug_rand = noise
        trainer = A.ACSASRecTrainer(config, model)
        trainer.enable_data_parallel(vocab_parallel=vocab_parallel, shard_table=shard)
        assert (trainer.vp is not None and trainer.vp.sharded) == shard
        model.train()
        inter = A.Interaction({'item_id_list': seq[sl].to(dev), 'item_length': ln[sl].to(dev), 'item_id': pos[sl].to(dev),
                               'neg_item_id': neg[sl].to(dev)})
        la, lc = trainer.fused(inter)
        trainer._allreduce_grads()
        grads = {}
        for n, p in model.named_parameters():
            gr = p.grad.detach()
            if n == 'item_embedding.weight' and shard:
                gr = trainer.vp.gather_full(gr)
            grads[n] = gr.clone()
        trainer.optimizer.zero_grad()
        for _ in range(2):                  # the trainer's own CUDA-graph path, NCCL collectives captured
            trainer.graphed_step(inter)
        sd = trainer._full_state_dict()
        entry = dict(la=float(la), lc=float(lc), grads=grads, sd=sd)
        model.eval()
        with torch.no_grad():
            _, rec, counts = model.sampled_topk(inter, cand[sl].to(dev), k, counts=True)
        entry.update(rec=rec.cpu(), counts=counts.cpu())
        if shard:
            # sampled evaluation on the sharded table: every rank draws its own users' negatives; graphed == eager
            uid, iid = ds.inter_feat['user_id'].numpy(), ds.inter_feat['item_id'].numpy()
            off, items = A.ops.used_item_csr(uid, iid, n_users + 1, V)
            s = A.ops.NegSampler('uniform', off, items, V, seed=42 + rank, phase=1)
            loader = A.data.NegSampleEvalDataLoader(config, ds, s, N)
            s.to_device(dev)
            st = s.rng.state.clone()
            got = trainer.evaluate(loader, load_best_model=False)
            assert any(key[0] == 'sampled' for key in trainer._eval_graphs)
            s.rng.state.copy_(st)
            trainer.use_graph = False
            want = trainer.evaluate(loader, load_best_model=False)
            trainer.use_graph = True
            assert got == want, (got, want)
            assert all(np.isfinite(v) for v in got.values())
        res[name] = entry
        del trainer, model
        torch.cuda.synchronize()
        dist.barrier()
    ref = res['dp']
    worst = 0.0
    for name in ('vocab-parallel', 'vocab-parallel + sharded table'):
        e = res[name]
        assert abs(e['la'] - ref['la']) < 1e-5 * abs(ref['la']) and abs(e['lc'] - ref['lc']) < 1e-5 * abs(ref['lc']), (name, e['la'], ref['la'])
        for n, gr in ref['grads'].items():
            scale = float(gr.abs().max())
            err = float((e['grads'][n] - gr).abs().max())
            assert err <= 2e-4 * scale + 1e-9, (name, n, err, scale)
            if scale > 1e-6:
                worst = max(worst, err / scale)
        for n, v in ref['sd'].items():
            upd_ref, upd = v - params[n], e['sd'][n] - params[n]
            big = ref['grads'][n].cpu().abs() > 1e-2 * ref['grads'][n].abs().max().cpu()      # Adam moves by ~lr * sign(g)
            if bool(big.any()):
                assert float((upd_ref - upd)[big].abs().max()) < 1e-4, (name, n)
        assert torch.equal(e['rec'], ref['rec']) and torch.equal(e['counts'], ref['counts']), name
    dist.barrier()
    if rank == 0:
        print('multi-gpu BPR / sampled-eval check ok: world %d, 3 modes, worst grad rel err %.2e' % (world, worst))
    torch.cuda.synchronize()
    os._exit(0)


if __name__ == '__main__':
    main()
