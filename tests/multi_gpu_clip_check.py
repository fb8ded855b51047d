"""Run under torchrun with 2+ GPUs: gradient clipping by global norm (`clip_grad_norm`) in the three multi-GPU modes of the trainer
  (a) batch data-parallel, replicated item table                       -- the reference point
  (b) vocab-parallel logits / CE over a replicated table
  (c) vocab-parallel with SHARDED table storage: the norm combines the replicated parameters' partial with every rank's shard
      partial (one 8-byte all-gather per rank, captured in the step's graph)
Checked for norm_type 2 and inf: both losses, the norm, every clipped gradient (the sharded table gradient gathered back to the
reference layout), the parameters after two more steps through the CUDA-graph path, and that the replicated parameters are
bit-identical on every rank.  Prints 'multi-gpu clip check ok' on rank 0."""
import os
import sys

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
    from test_gpu_model import make_config, DS
    cfg = O.default_cfg(hidden_dropout_prob=0.0, attn_dropout_prob=0.0)
    V, B, L = 5003, 64, 50
    max_norm = 1e-3                                  # far below the gradient norm: every step is clipped
    params = O.init_params(cfg, V, seed=11)
    seq, ln, pos = O.synth_batch(B * world, L, V, seed=12)
    sl = slice(rank * B, (rank + 1) * B)
    g = torch.Generator().manual_seed(100 + rank)
    noise = {(l, 'noise'): torch.randn(B, cfg['n_heads'], L, L, generator=g).to(dev) for l in range(cfg['n_layers'])}
    modes = [('dp', False, False), ('vocab-parallel', True, False), ('vocab-parallel + sharded table', True, True)]
    worst = 0.0
    for norm_type in (2, 'inf'):
        res = {}
        for name, vocab_parallel, shard in modes:
            config = make_config(A, cfg, cuda_graph=True, device=dev, checkpoint_dir='/tmp/acsr_mgpu_clip_%d' % rank,
                                 clip_grad_norm={'max_norm': max_norm, 'norm_type': norm_type})
            model = A.ACSASRec(config, DS(V)).to(dev)
            model.load_state_dict({kk: v.to(dev) for kk, v in params.items()})
            model._debug_rand = noise
            trainer = A.ACSASRecTrainer(config, model)
            trainer.enable_data_parallel(vocab_parallel=vocab_parallel, shard_table=shard)
            assert trainer.fused is not None and not trainer.torch_clip
            model.train()
            inter = A.Interaction({'item_id_list': seq[sl].to(dev), 'item_length': ln[sl].to(dev), 'item_id': pos[sl].to(dev)})
            # one eager step; after it every .grad holds the clipped gradient
            la, lc = trainer.train_step(inter)
            norm = float(trainer.optimizer.grad_norm)
            assert norm > 10 * max_norm, (name, norm)
            grads = {}
            for n, p in model.named_parameters():
                gr = p.grad.detach()
                if n == 'item_embedding.weight' and shard:
                    gr = trainer.vp.gather_full(gr)
                grads[n] = gr.clone()
            # two more steps through the trainer's CUDA-graph path, the collectives (and the norm all-gather) captured
            for _ in range(2):
                trainer.graphed_step(inter)
            assert trainer._graph is not None
            torch.cuda.synchronize()
            # replicated parameters are bit-identical on every rank (the sharded table's slot excepted)
            flat = trainer.optimizer.flat_param
            if shard:
                a, b = trainer.optimizer.slot(model.item_embedding.weight)
                flat = torch.cat((flat[:a], flat[b:]))
            gathered = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(gathered, flat)
            for r in range(1, world):
                assert torch.equal(gathered[0], gathered[r]), (norm_type, name, 'rank %d diverged' % r)
            res[name] = dict(la=float(la), lc=float(lc), norm=norm, grads=grads, sd=trainer._full_state_dict())
            del trainer, model
            torch.cuda.synchronize()
            dist.barrier()
        ref = res['dp']
        for name in ('vocab-parallel', 'vocab-parallel + sharded table'):
            e = res[name]
            assert abs(e['la'] - ref['la']) < 1e-5 * abs(ref['la']) and abs(e['lc'] - ref['lc']) < 1e-5 * abs(ref['lc']), (name, e['la'], ref['la'])
            assert abs(e['norm'] - ref['norm']) <= 2e-4 * ref['norm'], (norm_type, name, e['norm'], ref['norm'])
            for n, gr in ref['grads'].items():
                scale = float(gr.abs().max())
                err = float((e['grads'][n] - gr).abs().max())
                assert err <= 2e-4 * scale + 1e-12, (norm_type, name, n, err, scale)
                if scale > 1e-9:
                    worst = max(worst, err / scale)
            for n, v in ref['sd'].items():
                upd_ref, upd = v - params[n], e['sd'][n] - params[n]
                big = ref['grads'][n].cpu().abs() > 1e-2 * ref['grads'][n].abs().max().cpu()
                if bool(big.any()):
                    assert float((upd_ref - upd)[big].abs().max()) < 1e-4, (norm_type, name, n)
        dist.barrier()
    if rank == 0:
        print('multi-gpu clip check ok: world %d, 3 modes x norm_type 2 / inf, worst clipped-grad rel err %.2e' % (world, worst))
    torch.cuda.synchronize()
    os._exit(0)


if __name__ == '__main__':
    main()
