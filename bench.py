"""bench.py -- AC-SASRec training seq/s (+ full-sort eval users/s) on B200, BASELINE.json config #2:
synthetic Amazon-Beauty shape (22,363 users, 12,101 items + pad -> V=12,102, L=50, d=64, 2 layers,
2 heads, inner 256, B=256, top-k 50).

    python bench.py --gpus N --steps K --warmup W            # this implementation
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm (oracle port of the reference)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also writes the last timed step's outputs as DIR/*.npy

A "step" is one pass of the training hot path over one batch of 256 sequences: both losses, both
routed backward passes, Adam (trainer.py:660-687).  `value` times it with the batch already resident
in HBM; `e2e` times the trainer's public step with the batch in pinned host memory (H2D inside the
timed region) and the two losses read back every step.  Each timed step is bracketed by CUDA events
on the launching stream; L2 is flushed (256 MiB write) between timed steps, outside the brackets.
One JSON line is printed by rank 0.
"""
import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch

WORKLOADS = {
    # BASELINE.json configs[1]: the configuration the metric is quoted on (default; the driver's bench line)
    'c2': dict(name='C2 synthetic Amazon-Beauty shape', users=22363, V=12102, L=50, d=64, n_layers=2, n_heads=2, inner=256, B=256, topk=50),
    # the other configs are parity-test cases (tests/); `--workload` times them with the same harness for DESIGN.md's table
    'c1': dict(name='C1 ml-100k shape', users=943, V=1683, L=50, d=64, n_layers=2, n_heads=2, inner=256, B=256, topk=50),
    'c3': dict(name='C3 synthetic Yelp shape', users=30431, V=20034, L=50, d=64, n_layers=2, n_heads=2, inner=256, B=256, topk=50),
    'c3v': dict(name='C3 synthetic Yelp shape, repo variant (config/yelp.yaml)', users=30431, V=20034, L=50, d=128, n_layers=3, n_heads=8,
                inner=64, B=256, topk=50),
    'c4': dict(name='C4 1M-item catalogue', users=22363, V=1000001, L=50, d=64, n_layers=2, n_heads=2, inner=256, B=256, topk=50),
    'c5': dict(name='C5 long-sequence stress', users=22363, V=12102, L=200, d=256, n_layers=4, n_heads=4, inner=1024, B=2048, topk=50),
}
WORKLOAD = dict(WORKLOADS['c2'])


def workload_string(full_len=False):
    """names the workload; IDENTICAL in both arms (`--impl ours` / `--impl reference`)"""
    w = WORKLOAD
    return ('%s: V=%d, users=%d, L=%d, d=%d, layers=%d, heads=%d, inner=%d, train/eval batch %d per GPU, top-%d; lengths %s, items Zipf(1)'
            % (w['name'], w['V'], w['users'], w['L'], w['d'], w['n_layers'], w['n_heads'], w['inner'], w['B'], w['topk'],
               'all = L' if full_len else 'LogNormal(ln7,0.8)'))


def model_cfg():
    return dict(n_layers=WORKLOAD['n_layers'], n_heads=WORKLOAD['n_heads'], hidden_size=WORKLOAD['d'],
                inner_size=WORKLOAD['inner'], hidden_dropout_prob=0.5, attn_dropout_prob=0.5, hidden_act='gelu',
                layer_norm_eps=1e-12, initializer_range=0.02, loss_type='CE', combine_option='gate',
                rich_calibrated_combine='none', two_level=True, use_position_embedding=False, use_order=True,
                use_distance=True, trainable_mask_loss_weight=False, mask_loss_weight=0.03, MAX_ITEM_LIST_LENGTH=WORKLOAD['L'])


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """polls SM clock + throttle reasons of one GPU while the timed regions run (NVML)."""
    REASONS = {0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown', 0x2: 'applications_clocks_setting'}

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = int(vis.split(',')[index]) if vis and vis.split(',')[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {'sm_mhz': (s[len(s) // 2] if s else None), 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


def timed_steps(fn, n, flush):
    """run fn() n times, each bracketed by CUDA events on the current stream; flush L2 in between.  -> total ms"""
    evs = []
    for _ in range(n):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs)


def dump_outputs(out_dir, arrays):
    """write each host tensor as out_dir/<name>.npy: floating point as float32, integers as float64 (exact)"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.numpy().astype(np.float32 if t.is_floating_point() else np.float64))


# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(name, per_step_calls, cfg, B, V):
    """ALGORITHMIC HBM bytes of all launches of one kernel in one training step (DESIGN.md §kernels)."""
    L, d, N, I = cfg['MAX_ITEM_LIST_LENGTH'], cfg['hidden_size'], cfg['n_layers'], cfg['inner_size']
    T = B * L
    if name == 'acsr_attn_calib_fwd':       # 5 inputs + gate logits + ids, n_out contexts; attacked only on the last layer
        return sum(B * ((5 + (2 if l == N - 1 else 1)) * L * d * 4 + L * L * 4 + 8 * L) for l in range(N))
    if name in ('acsr_attn_calib_bwd', 'acsr_attn_calib_bwd2'):       # both cotangent streams x N layers: 5 inputs + gate + ids + n_cot cotangents in, 5 grads + dgate out
        tot = 0
        for l in range(N):
            for n_cot in ((1, 1) if l < N - 1 else (1, 1)):
                tot += B * ((5 + n_cot + 5) * L * d * 4 + 2 * L * L * 4 + 8 * L)
        return tot
    if name == 'acsr_bias_dropout_res_ln_fwd':
        return per_step_calls * T * d * 4 * 3
    if name in ('acsr_bias_dropout_res_ln_bwd', 'acsr_bias_act_bwd', 'acsr_bias_act_fwd'):
        return None                                # row counts differ per call since the last layer runs on compact rows
    if name == 'acsr_bias_dropout_res_ln_bwd':
        return per_step_calls * T * d * 4 * 5
    if name == 'acsr_bias_act_fwd':
        return per_step_calls * T * I * 4 * 2
    if name == 'acsr_bias_act_bwd':
        return per_step_calls * T * I * 4 * 3
    if name == 'acsr_embed_ln_dropout_fwd':
        return T * (8 + 4 * d + 4 * d)
    if name == 'acsr_embed_ln_dropout_bwd':
        return per_step_calls * T * (8 + 4 * d + 4 * d + 8 * d)
    if name == 'acsr_logits_ce_partial':
        return V * d * 4 + 2 * B * d * 4
    if name == 'acsr_logits_ce_grad':
        return per_step_calls * (V * d * 4 + 2 * B * d * 4 + 2 * B * V * 4)
    if name == 'acsr_ce_bwd_dout':                  # table + out in, d_out read-modify-write (2B rows)
        return per_step_calls * (V * d * 4 + 2 * B * d * 4 + 2 * (2 * B * d * 4))
    if name == 'acsr_ce_bwd_dtable':                # table + the calibrated rows of out in, d_table read-modify-write
        return per_step_calls * (V * d * 4 + B * d * 4 + 2 * V * d * 4)
    if name == 'acsr_adam_step':
        return None                                # filled by caller (28 B / parameter)
    return None


def build(dev, rank, world, cuda_graph=True, B=None):
    import ac_tsr_b200 as A
    cfg = model_cfg()
    d = dict(cfg)
    B = WORKLOAD['B'] if B is None else B
    d.update(USER_ID_FIELD='user_id', ITEM_ID_FIELD='item_id', LIST_SUFFIX='_list', ITEM_LIST_LENGTH_FIELD='item_length',
             NEG_PREFIX='neg_', device=dev, seed=42, learning_rate=1e-4, epochs=1, train_batch_size=B,
             eval_batch_size=B, topk=[1, 3, 5, 10, 20, 50], metrics=['Hit', 'MRR', 'NDCG'], valid_metric='Hit@10',
             checkpoint_dir='/tmp/acsr_bench_ckpt', cuda_graph=cuda_graph, logits_passes=3,
             step_branches=int(os.environ.get('ACSR_STEP_BRANCHES', 1)))
    config = A.Config(model='ACSASRec', config_dict=d)

    class DS:
        item_num = WORKLOAD['V']

        def num(self, f):
            return WORKLOAD['V']
    torch.manual_seed(42)
    model = A.ACSASRec(config, DS()).to(dev)
    trainer = A.ACSASRecTrainer(config, model)
    return A, cfg, config, model, trainer


TRAFFIC_PROFILE = os.path.join(ROOT, 'profiles', 'r02_traffic.json')     # ncu dram__bytes_{read,write}.sum per launch
NCU_NAMES = {'acsr_linear_tok': 'void acsr::linear_tok_kernel<0>', 'acsr_linear_tok_ragged': 'void acsr::linear_tok_kernel<0>', 'acsr_linear_tok_bdrl': 'void acsr::linear_tok_kernel<2>',
             'acsr_attn_calib_bwd2': 'void acsr::attn_bwd_kernel<32, 2>', 'acsr_attn_calib_fwd': 'void acsr::attn_fwd_kernel<32>',
             'acsr_linear_wgrad': 'void acsr::linear_wgrad_kernel<2>'}


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture of this same workload (profiles/), or None."""
    try:
        prof = json.load(open(TRAFFIC_PROFILE))
        e = prof[NCU_NAMES[kernel]]
        return int(e['dram_read_bytes_per_launch'] + e['dram_write_bytes_per_launch'])
    except Exception:
        return None


class StdoutGuard:
    """Everything any library prints on fd 1 (NCCL's version banner, ...) goes to stderr; the JSON line alone reaches stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + '\n').encode())


def kernel_breakdown(A, trainer, devb, nb, cfg, B, V, K):
    """per-kernel device time of the training step: eager (non-graph) steps with every C-ABI launch bracketed by events on the
    launching stream.  -> (kernels dict sorted by time, launches per step, eager ms per step)"""
    kt_steps = min(K, 10)
    # (1) one eager step with the arguments of every launch kept, then every launch replayed inside its own CUDA graph:
    # the per-launch device time the graph-replayed step pays (see _lib.replay_in_graph)
    ingraph = None
    if trainer.fused is not None and os.environ.get('ACSR_BENCH_INGRAPH', '1') == '1':
        rec = A._lib.KernelTimer(keep_calls=True)
        A.LIB.timer = rec
        saved = trainer.fused.overlap_wgrad
        trainer.fused.overlap_wgrad = False
        trainer.train_step(devb[0])
        torch.cuda.synchronize()
        A.LIB.timer = None
        trainer.fused.overlap_wgrad = saved
        per_call = [] if os.environ.get('ACSR_BENCH_CALLS') else None
        ingraph = A._lib.replay_in_graph(A.LIB, rec.calls, per_call=per_call)
        if per_call:
            for name, ints, us, ab in per_call:
                sys.stderr.write('CALL %-30s %8.2f us  %7.1f GB/s  %s\n' % (name, us, (ab or 0) / us / 1e3, ints))
        trainer.optimizer.zero_grad()
    # (2) eager steps with an event pair around every launch (includes the event-record overhead: kept for the shares / as a cross-check)
    timer = A._lib.KernelTimer()
    A.LIB.timer = timer
    saved_branches = None
    if trainer.fused is not None:
        trainer.fused.overlap_wgrad = False       # per-kernel events are recorded on the launching (main) stream
        saved_branches, trainer.fused.n_branches = trainer.fused.n_branches, 1
    torch.cuda.synchronize()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    # the host needs ~15 us per eager launch, most kernels take less: park the GPU behind a spin kernel so the launches
    # queue up and the event pairs bracket device time only (kernel + its launch gap), not host submission time
    torch.cuda._sleep(int(0.25 * 1.9e9))
    t0.record()
    for i in range(kt_steps):
        trainer.train_step(devb[i % nb])
    t1.record()
    ksum = timer.summary()
    A.LIB.timer = None
    if trainer.fused is not None:
        trainer.fused.overlap_wgrad = True
        trainer.fused.n_branches = saved_branches
    eager_ms = t0.elapsed_time(t1) / kt_steps
    launches_per_step = timer.launches / kt_steps + 1                   # adam_step enqueues two kernels
    n_param = trainer.optimizer.flat_param.numel()
    kernels = {}
    total_k = sum(t for _, t in ksum.values())
    for name, (n, t) in sorted(ksum.items(), key=lambda x: -x[1][1]):
        per_step_calls = n / kt_steps
        ab = algorithmic_bytes(name, per_step_calls, cfg, B, V)
        if name in timer.bytes:
            ab = timer.bytes[name] / kt_steps
        if name == 'acsr_adam_step':
            ab = 28 * n_param
        ms = t / kt_steps
        kernels[name] = {'calls_per_step': per_step_calls, 'ms_per_step': round(ms, 5), 'share': round(t / total_k, 4),
                         'algo_bytes_per_step': ab, 'gbs': (round(ab / ms / 1e6, 1) if ab else None)}
        if ingraph is not None and name in ingraph:
            n_g, us_g, _ = ingraph[name]
            kernels[name]['graph_us_per_launch'] = round(us_g / n_g, 2)
            kernels[name]['graph_ms_per_step'] = round(us_g / 1e3, 5)
            kernels[name]['graph_gbs'] = round(ab / us_g / 1e3, 1) if ab else None
    if ingraph is not None:
        tot_g = sum(v.get('graph_ms_per_step', 0.0) for v in kernels.values())
        for v in kernels.values():
            if 'graph_ms_per_step' in v:
                v['graph_share'] = round(v['graph_ms_per_step'] / tot_g, 4)
    return kernels, launches_per_step, eager_ms


def roofline_of(kernels, workload_is_c2):
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak, peak_src = (peaks.get('hbm_gbs'), 'measured (MEASURED_PEAKS.json hbm_gbs)') if peaks.get('hbm_gbs') else (6650.0, 'fallback 6.65 TB/s')
    have_graph = any('graph_ms_per_step' in v for v in kernels.values())
    if have_graph:                         # dominant kernel by in-graph device time (what the graph-replayed step pays)
        top = max((k for k in kernels if 'graph_ms_per_step' in kernels[k]), key=lambda k: kernels[k]['graph_ms_per_step'])
    else:
        top = next(iter(kernels))
    tk = kernels[top]
    calls = max(1.0, tk['calls_per_step'])
    gbs = tk.get('graph_gbs') if have_graph else tk['gbs']
    r = {'kernel': top, 'bound': 'hbm', 'achieved': gbs, 'peak': peak, 'unit': 'GB/s',
         'frac': (round(gbs / peak, 4) if gbs else None), 'traffic': measured_traffic(top) if workload_is_c2 else None,
         'traffic_source': os.path.relpath(TRAFFIC_PROFILE, ROOT) + ' (ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, same workload)',
         'peak_source': peak_src,
         'avg_launch_us': tk.get('graph_us_per_launch') if have_graph else round(tk['ms_per_step'] / calls * 1e3, 2),
         'algo_bytes_per_launch': (int(tk['algo_bytes_per_step'] / calls) if tk['algo_bytes_per_step'] else None),
         'share_of_kernel_time': tk.get('graph_share') if have_graph else tk['share']}
    if have_graph:
        r['timing'] = ('CUDA events around a CUDA-graph replay of 16 back-to-back copies of each recorded launch of one step (same arguments '
                       'and buffers; _lib.replay_in_graph), per launch')
        r['eager_event_pair_us'] = round(tk['ms_per_step'] / calls * 1e3, 2)      # the same launch timed eagerly with its own event pair
        r['eager_event_pair_frac'] = round(tk['gbs'] / peak, 4) if tk['gbs'] else None
    return r


def parity_check(A, dev, cfg, B, L, V):
    """BASELINE.md section 4.6: parity asserted inside the bench run.  One fused training step of the headline shape on the
    first synthetic batch, every dropout mask and the attack noise injected, against the CPU oracle: both losses and every
    routed gradient.  Raises when out of tolerance (losses 1e-3 relative = north_star; gradients 1e-3 of max |g|)."""
    from oracle import acsr_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    params = O.init_params(cfg, V, seed=42)
    seq, ln, pos = O.synth_batch(B, L, V, seed=42)
    rnd = O.draw_rand(cfg, B, L, seed=43, train=True)
    la_o, lc_o, grads = O.train_grads(params, cfg, seq, ln, pos, rnd)
    _, _, config, model, trainer = build(dev, 0, 1, cuda_graph=False, B=B)
    model.load_state_dict({k: v.to(dev) for k, v in params.items()}, strict=True)
    model._debug_rand = {k: v.to(dev) for k, v in rnd.d.items()}
    model.train()
    inter = A.Interaction({'item_id_list': seq.to(dev), 'item_length': ln.to(dev), 'item_id': pos.to(dev)})
    la, lc = trainer.fused(inter)
    ra = abs(float(la) - float(la_o)) / abs(float(la_o))
    rc = abs(float(lc) - float(lc_o)) / abs(float(lc_o))
    worst, worst_name, grads_ok = 0.0, '', True
    for n, p in model.named_parameters():
        ref = grads[n]
        scale = float(ref.abs().max())
        err = float((p.grad.cpu() - ref).abs().max())
        # same criterion as tests/: 1e-3 of max |g| plus an absolute floor (a key-side bias has an exactly-zero true gradient --
        # softmax is shift invariant -- so both sides hold rounding noise only)
        grads_ok = grads_ok and err <= 1e-3 * scale + 1e-8
        if scale > 1e-6 and err / scale > worst:
            worst, worst_name = err / scale, n
    ok = ra < 1e-3 and rc < 1e-3 and grads_ok
    out = {'checked': 'fused train step vs CPU oracle, B=%d V=%d, injected masks/noise' % (B, V), 'loss_attacked_rel_err': float('%.3g' % ra),
           'loss_calibrated_rel_err': float('%.3g' % rc), 'max_grad_rel_err': float('%.3g' % worst), 'worst_grad': worst_name,
           'tolerance': 1e-3, 'ok': bool(ok)}
    if not ok:
        raise AssertionError('bench parity check failed: %s' % json.dumps(out))
    del model, trainer
    return out


def eager_cuda_baseline(cfg, B, L, V, dev, steps=10):
    """Reference-SEMANTICS step in eager PyTorch on the same B200 (proxy for running /root/reference with device='cuda',
    trainer.py:660-687; the reference itself cannot travel to the GPU box): the oracle restatement -- stock ATen / cuBLAS
    kernels, autograd, two routed backward passes, Adam -- with the masks / noise drawn once and reused (the reference draws its
    attack noise on the CPU every step, layers.py:917, so this proxy is faster than the real thing)."""
    from oracle import acsr_oracle as O
    params = {k: v.to(dev) for k, v in O.init_params(cfg, V, seed=42).items()}
    state = {k: (torch.zeros_like(v), torch.zeros_like(v)) for k, v in params.items()}
    seq, ln, pos = (t.to(dev) for t in O.synth_batch(B, L, V, seed=42))
    rnd = O.draw_rand(cfg, B, L, seed=1, train=True)
    rnd = O.Rand({k: v.to(dev) for k, v in rnd.d.items()})
    cnt = [0]

    def step():
        cnt[0] += 1
        la, lc, grads = O.train_grads(params, cfg, seq, ln, pos, rnd)
        for k in params:
            params[k], m, v = O.adam_step(params[k], grads[k], state[k][0], state[k][1], cnt[0], 1e-4)
            state[k] = (m, v)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {'value': round(B / (ms / 1e3), 1), 'unit': 'seq/s', 'ms_per_step': round(ms, 3), 'kind': 'port',
            'sample': '%d eager-CUDA steps of B=%d: oracle restatement of the reference step on cuda:0 (stock ATen/cuBLAS kernels, autograd, '
                      'Adam; masks and noise drawn once)' % (steps, B)}


def run_ours(args):
    guard = StdoutGuard()
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    use_graph = (world == 1 or bool(args.dp_graph)) and WORKLOAD['L'] <= 64
    A, cfg, config, model, trainer = build(dev, rank, world, cuda_graph=use_graph)
    vocab_parallel = world > 1 and WORKLOAD['V'] >= 500000     # C4: logits / CE / top-k sharded by catalogue rows over the ranks
    if world > 1:
        trainer.enable_data_parallel(vocab_parallel=vocab_parallel)
    B, L, V, K, W = WORKLOAD['B'], WORKLOAD['L'], WORKLOAD['V'], args.steps, args.warmup
    parity = None
    if rank == 0 and world == 1 and not args.no_parity and WORKLOAD['L'] <= 64 and V <= 100000:
        parity = parity_check(A, dev, cfg, min(B, 256), L, V)
    nb = 8                                                             # distinct synthetic batches cycled through
    seq, ln, tgt = A.data.synth_sequences(nb * B, L, V, seed=42 + rank, full_len=bool(args.full_len))
    # host batches in pinned memory, the three fields of a batch back to back (what TrainDataLoader yields): one H2D copy per step
    host = [A.Interaction({'item_id_list': seq[i * B:(i + 1) * B], 'item_length': ln[i * B:(i + 1) * B],
                           'item_id': tgt[i * B:(i + 1) * B]}).pack(['item_id_list', 'item_length', 'item_id']) for i in range(nb)]
    devb = [h.to(dev) for h in host]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    model.train()
    step = trainer.graphed_step if use_graph else trainer.train_step
    it = [0]
    last = {}                                                          # what the latest timed train step / eval batch returned

    def dev_step():
        last['train'] = step(devb[it[0] % nb])
        it[0] += 1
    loss_pin = torch.empty(3, dtype=torch.float32).pin_memory()

    def e2e_step():
        b = host[it[0] % nb]
        la, lc = step(b if use_graph else b.to(dev))
        last = getattr(trainer.fused, 'last_losses', None) if trainer.fused is not None else None
        if last is not None:                                           # [CE_cal, CE_att, attacked loss] live in one buffer
            loss_pin.copy_(last, non_blocking=True)
        else:
            loss_pin[0:1].copy_(la.reshape(1), non_blocking=True)
            loss_pin[1:2].copy_(lc.reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()                      # the losses are read on the host every step
        it[0] += 1

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(W, 3)):
        dev_step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    ms_dev = timed_steps(dev_step, K, flush)
    barrier()
    outputs = {}
    if args.dump_outputs and rank == 0:
        # what the caller of the step receives: the two losses.  The graphed step returns them in its static buffers, so they are
        # copied before the next step.  The parameters are not written: the step accumulates gradients with float atomics, whose
        # order varies from run to run, and Adam turns that rounding into visible noise in parameters whose true gradient is zero.
        la, lc = last['train']
        outputs['train_loss_attacked'], outputs['train_loss_calibrated'] = la.detach().cpu(), lc.detach().cpu()
    for _ in range(3):
        e2e_step()
    barrier()
    ms_e2e = timed_steps(e2e_step, K, flush)
    barrier()
    # ---- epoch mode: training data resident in HBM, on-device shuffle, the batch gathered inside the captured step (f-2):
    # nothing crosses PCIe on the way in; the three losses are still read back every step ----
    ms_e2e_dev = None
    if use_graph and world == 1 and trainer.fused is not None:
        ds = A.data.SyntheticSequentialDataset(config, 512 * B, V, seed=4242)       # ~131k training sequences, the size of the Beauty split
        dloader = A.data.DeviceTrainDataLoader(config, ds, shuffle=True)
        dloader.new_epoch()
        dstate = [0]

        def epoch_step():
            if dstate[0] == dloader.full_batches:                      # next epoch: new permutation drawn on the device
                dloader.new_epoch()
                dstate[0] = 0
            trainer.device_loader_step(dloader)
            dstate[0] += 1
            loss_pin.copy_(trainer.fused.last_losses, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for _ in range(3):
            epoch_step()
        barrier()
        ms_e2e_dev = timed_steps(epoch_step, K, flush)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        dloader.new_epoch()                                            # the per-epoch on-device shuffle, timed on its own
        ev1.record()
        torch.cuda.synchronize()
        ms_shuffle = ev0.elapsed_time(ev1)
    # ---- full-sort eval (fused logits + top-k), same batch size ----
    model.eval()
    kmax = WORKLOAD['topk']
    rec_pin = torch.empty((B, kmax + 1), dtype=torch.int32).pin_memory()

    def eval_dev():
        b = devb[it[0] % nb]
        with torch.no_grad():
            last['eval'] = trainer.eval_batch((b, None, None, b['item_id']))
        it[0] += 1

    def eval_e2e():
        b = host[it[0] % nb]
        with torch.no_grad():
            trainer.eval_batch((b, None, None, b['item_id']), rec_out=rec_pin)      # D2H of the hit flags straight from the graph's output
        torch.cuda.current_stream().synchronize()
        it[0] += 1
    for _ in range(3):
        eval_dev()
    barrier()
    ms_eval = timed_steps(eval_dev, K, flush)
    if args.dump_outputs and rank == 0:
        outputs['eval_rec_topk'] = last['eval'].cpu()
    for _ in range(3):
        eval_e2e()
    barrier()
    ms_eval_e2e = timed_steps(eval_e2e, K, flush)
    barrier()
    clocks = sampler.stop()
    if outputs:
        dump_outputs(args.dump_outputs, outputs)

    model.train()
    kernels, launches_per_step, eager_ms = kernel_breakdown(A, trainer, devb, nb, cfg, B, V, K)
    roof = roofline_of(kernels, args.workload == 'c2')

    # max over ranks
    t = torch.tensor([ms_dev, ms_e2e, ms_eval, ms_eval_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_eval, ms_eval_e2e = [float(x) for x in t.tolist()]

    def shutdown():
        """release the captured graph (it pins NCCL resources) before tearing the process group down; never hang at exit"""
        if world == 1:
            return
        import gc
        trainer._graph = None
        gc.collect()
        torch.cuda.synchronize()
        sys.stdout.flush()
        threading.Timer(20.0, lambda: os._exit(0)).start()
        try:
            dist.barrier()
            dist.destroy_process_group()
        except Exception:
            pass
        os._exit(0)
    # ---- the 1M-item catalogue (BASELINE config #4) at this N: item table / logits / CE / top-k vocab-sharded over the ranks
    # (N = 1: the same model on one GPU, the base of the curve).  All ranks take part.
    sharded = None
    if args.workload == 'c2' and args.batch == 0 and not args.no_vocab_sharded:
        sharded = vocab_sharded_record(A, dev, rank, world, max(10, min(K, 30)), flush)
    # ---- the long-sequence stress configuration (BASELINE config #5: L=200, d=256, 4 layers, B=2048 per GPU) at this N, batch
    # data-parallel: eager launches (the long-sequence attention backward walks the batch in workspace-sized chunks) ----
    longseq = None
    if args.workload == 'c2' and args.batch == 0 and not args.no_long_seq:
        try:
            longseq = long_sequence_record(A, dev, rank, world, 3)
        except Exception as e:                                          # a sub-record must never sink the bench line
            longseq = {'error': str(e)[:300]}
            torch.cuda.empty_cache()
    if rank != 0:
        shutdown()
        return
    # ---- large-batch record (SURVEY section 7: "report throughput at B=256 and at large B"): B = 2048, the RecBole default the
    # reference's dataset YAMLs inherit; same model, own per-kernel roofline ----
    large = None
    if world == 1 and not args.no_large_batch and args.workload == 'c2' and args.batch == 0:
        large = large_batch_record(A, dev, cfg, 2048, L, V, max(10, K // 4), flush)
    siblings = None
    if world == 1 and not args.no_siblings and args.workload == 'c2' and args.batch == 0:
        siblings = sibling_models_record(A, dev, B, L, V, max(10, K // 5))
    cpu = eager = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(cfg, B if args.workload == 'c2' else min(B, 32), L, V, budget_s=20.0)
        if WORKLOAD['L'] <= 64 and V <= 100000:
            try:
                eager = eager_cuda_baseline(cfg, B, L, V, dev)
            except Exception as e:                                      # a proxy measurement must never sink the bench line
                eager = {'error': str(e)[:200]}
    h2d = sum(host[0][k].numel() * host[0][k].element_size() for k in host[0].columns)
    line = {
        'metric': 'AC-SASRec train seq/s', 'value': round(world * B * K / (ms_dev / 1e3), 1), 'unit': 'seq/s',
        'n_gpus': world, 'steps': K, 'warmup': max(W, 3), 'ms_per_step': round(ms_dev / K, 4), 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_string(bool(args.full_len))},
        'notes': {'timing': 'CUDA events around every step on the launching stream; L2 flushed (256 MiB write) between timed steps',
                  'parallelism': ('dp%d (batch-parallel, NCCL all-reduce of the flat gradient%s)'
                                  % (world, '; logits/CE/top-k vocab-sharded: all-gather of out and of the (max, sum-exp) partials, '
                                     'reduce-scatter of d_out' if vocab_parallel else ', replicated item table')) if world > 1 else 'single GPU',
                  'launch': ('CUDA graph replay of the whole step' + (' (NCCL all-reduce captured)' if world > 1 else '')) if use_graph else 'eager launches + NCCL',
                  'gemm': '3xTF32 tcgen05 (fp32-level accuracy), no library GEMM on the step'},
        'e2e': {'value': round(world * B * K / (ms_e2e / 1e3), 1), 'unit': 'seq/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 12},
        'e2e_device_resident': ({'value': round(B * K / (ms_e2e_dev / 1e3), 1), 'unit': 'seq/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 12,
                                 'how': 'data.DeviceTrainDataLoader: training rows resident in HBM, per-epoch permutation drawn on the device, '
                                        'batch gathered by the first kernel of the captured step; losses read back every step',
                                 'epoch_shuffle_ms': round(ms_shuffle, 3), 'rows': 512 * B}
                                if ms_e2e_dev is not None else None),
        'gpu_launches': int(round(launches_per_step * K)),
        'clocks': clocks,
        'eval': {'metric': 'AC-SASRec full-sort eval users/s', 'value': round(world * B * K / (ms_eval / 1e3), 1), 'unit': 'users/s',
                 'ms_per_batch': round(ms_eval / K, 4),
                 'e2e': {'value': round(world * B * K / (ms_eval_e2e / 1e3), 1), 'unit': 'users/s', 'h2d_bytes_per_step': h2d,
                         'd2h_bytes_per_step': B * (kmax + 1) * 4}},
        'roofline': roof,
        'kernels': kernels,
        'eager_ms_per_step': round(eager_ms, 4),
    }
    if parity is not None:
        line['parity'] = parity
    if large is not None:
        line['large_batch'] = large
    if siblings is not None:
        line['sibling_models'] = siblings
    if sharded is not None:
        line['vocab_sharded'] = sharded
    if longseq is not None:
        line['long_sequence'] = longseq
    if cpu is not None:
        line['cpu_baseline'] = cpu
        line['cpu_baseline_eval'] = cpu_baseline_eval(cfg, B if args.workload == 'c2' else min(B, 32), L, V, kmax, budget_s=8.0)
    if eager is not None:
        line['eager_cuda_baseline'] = eager
    guard.emit(json.dumps(line))
    shutdown()


def vocab_sharded_record(A, dev, rank, world, K, flush):
    """BASELINE config #4 (V = 1,000,001, B = 256 per GPU) at `world` GPUs: batch data-parallel encoder, the item table
    (rows, gradient, Adam moments), the logits / CE and the top-k sharded by item rows (dist.py); weak scaling."""
    import torch.distributed as dist
    saved = dict(WORKLOAD)
    WORKLOAD.clear()
    WORKLOAD.update(WORKLOADS['c4'])
    try:
        B, L, V, kmax = WORKLOAD['B'], WORKLOAD['L'], WORKLOAD['V'], WORKLOAD['topk']
        _, cfg, config, model, trainer = build(dev, rank, world, cuda_graph=True)
        if world > 1:
            trainer.enable_data_parallel(vocab_parallel=True)
        nb = 4
        seq, ln, tgt = A.data.synth_sequences(nb * B, L, V, seed=142 + rank)
        devb = [A.Interaction({'item_id_list': seq[i * B:(i + 1) * B], 'item_length': ln[i * B:(i + 1) * B],
                               'item_id': tgt[i * B:(i + 1) * B]}).pack(['item_id_list', 'item_length', 'item_id']).to(dev) for i in range(nb)]
        it = [0]

        def sync():
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize()

        def dev_step():
            trainer.graphed_step(devb[it[0] % nb])
            it[0] += 1

        def eval_dev():
            b = devb[it[0] % nb]
            with torch.no_grad():
                trainer.eval_batch((b, None, None, b['item_id']))
            it[0] += 1
        model.train()
        for _ in range(3):
            dev_step()
        sync()
        ms = timed_steps(dev_step, K, flush)
        sync()
        model.eval()
        for _ in range(3):
            eval_dev()
        sync()
        ms_eval = timed_steps(eval_dev, K, flush)
        sync()
        t = torch.tensor([ms, ms_eval], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_eval = [float(x) for x in t.tolist()]
        vp = getattr(trainer, 'vp', None)
        rec = {'workload': workload_string(False), 'n_gpus': world, 'steps': K, 'scaling': 'weak',
               'value': round(world * B * K / (ms / 1e3), 1), 'unit': 'seq/s', 'ms_per_step': round(ms / K, 4),
               'eval': {'value': round(world * B * K / (ms_eval / 1e3), 1), 'unit': 'users/s', 'ms_per_batch': round(ms_eval / K, 4)},
               'storage': ('item table sharded by rows: %d rows (+ gradient + Adam moments) per rank' % vp.per) if (vp is not None and vp.sharded)
               else ('replicated table' if world > 1 else 'single GPU'),
               'collectives_per_step': ([] if world == 1 else [
                   'all-gather item ids [B*L] + reduce-scatter embedding rows [W*B*L, d]', 'all-gather out [2B, d]',
                   'all-gather (max, sum-exp, target logit) partials', 'reduce-scatter d_out [W*2B, d]',
                   'all-gather gradient rows [B*L, d]', 'all-reduce encoder gradients (%d floats)' % (trainer.optimizer.flat_grad.numel() - model.item_embedding.weight.numel())]),
               'launch': 'CUDA graph replay (NCCL collectives captured)'}
        trainer._graph, trainer._eval_graphs = None, {}
        del trainer, model
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        return rec
    finally:
        WORKLOAD.clear()
        WORKLOAD.update(saved)


def long_sequence_record(A, dev, rank, world, K):
    """BASELINE config #5 (L = 200, d = 256, 4 layers, 4 heads, inner 1024, B = 2048 per GPU; calibrators forward + backward) at
    `world` GPUs, batch data-parallel, weak scaling: train step and full-sort eval batch, device-timed, max over ranks."""
    import torch.distributed as dist
    saved = dict(WORKLOAD)
    WORKLOAD.clear()
    WORKLOAD.update(WORKLOADS['c5'])
    try:
        B, L, V = WORKLOAD['B'], WORKLOAD['L'], WORKLOAD['V']
        _, cfg, config, model, trainer = build(dev, rank, world, cuda_graph=False)
        if world > 1:
            trainer.enable_data_parallel()
        nb = 2
        seq, ln, tgt = A.data.synth_sequences(nb * B, L, V, seed=542 + rank)
        devb = [A.Interaction({'item_id_list': seq[i * B:(i + 1) * B], 'item_length': ln[i * B:(i + 1) * B],
                               'item_id': tgt[i * B:(i + 1) * B]}).pack(['item_id_list', 'item_length', 'item_id']).to(dev) for i in range(nb)]
        it = [0]

        def sync():
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
                torch.cuda.synchronize()

        def timed(fn, n):
            sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            sync()
            return e0.elapsed_time(e1) / n

        def dev_step():
            trainer.train_step(devb[it[0] % nb])
            it[0] += 1

        def eval_dev():
            b = devb[it[0] % nb]
            with torch.no_grad():
                trainer.eval_batch((b, None, None, b['item_id']))
            it[0] += 1
        model.train()
        for _ in range(2):
            dev_step()
        ms = timed(dev_step, K)
        model.eval()
        eval_dev()
        ms_eval = timed(eval_dev, K)
        t = torch.tensor([ms, ms_eval], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_eval = [float(x) for x in t.tolist()]
        rec = {'workload': workload_string(False), 'n_gpus': world, 'steps': K, 'scaling': 'weak',
               'value': round(world * B / (ms / 1e3), 1), 'unit': 'seq/s', 'ms_per_step': round(ms, 3),
               'eval': {'value': round(world * B / (ms_eval / 1e3), 1), 'unit': 'users/s', 'ms_per_batch': round(ms_eval, 3)},
               'parallelism': 'single GPU' if world == 1 else 'dp%d: NCCL all-reduce of the flat gradient (%d floats)' % (world, trainer.optimizer.flat_grad.numel()),
               'launch': 'eager launches; inputs larger than L2 (no flush needed: the step touches ~80 GB)'}
        del trainer, model
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        return rec
    finally:
        WORKLOAD.clear()
        WORKLOAD.update(saved)


def large_batch_record(A, dev, cfg, B, L, V, K, flush):
    """the training step at a large batch (B sequences, CUDA-graph replay, batch resident in HBM) + its per-kernel roofline"""
    _, _, config, model, trainer = build(dev, 0, 1, cuda_graph=True, B=B)
    nb = 4
    seq, ln, tgt = A.data.synth_sequences(nb * B, L, V, seed=7)
    devb = [A.Interaction({'item_id_list': seq[i * B:(i + 1) * B], 'item_length': ln[i * B:(i + 1) * B],
                           'item_id': tgt[i * B:(i + 1) * B]}).pack(['item_id_list', 'item_length', 'item_id']).to(dev) for i in range(nb)]
    model.train()
    it = [0]

    def dev_step():
        trainer.graphed_step(devb[it[0] % nb])
        it[0] += 1
    for _ in range(3):
        dev_step()
    torch.cuda.synchronize()
    ms = timed_steps(dev_step, K, flush)
    kernels, launches, eager_ms = kernel_breakdown(A, trainer, devb, nb, cfg, B, V, K)
    roof = roofline_of(kernels, False)
    top3 = {k: kernels[k] for k in list(kernels)[:3]}
    return {'batch': B, 'value': round(B * K / (ms / 1e3), 1), 'unit': 'seq/s', 'ms_per_step': round(ms / K, 4), 'steps': K,
            'launches_per_step': launches, 'roofline': roof, 'top_kernels': top3}


def run_profile(args):
    """Same kernels as the timed step, launched eagerly so ncu lists them one by one (never a bench value)."""
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(0)
    import __graft_entry__ as ge
    ge.build()
    A, cfg, config, model, trainer = build(dev, 0, 1, cuda_graph=False)
    B, L, V = WORKLOAD['B'], WORKLOAD['L'], WORKLOAD['V']
    seq, ln, tgt = A.data.synth_sequences(B, L, V, seed=42)
    b = A.Interaction({'item_id_list': seq, 'item_length': ln, 'item_id': tgt}).to(dev)
    model.train()
    for _ in range(args.warmup + args.steps):
        trainer.train_step(b)
    model.eval()
    with torch.no_grad():
        for _ in range(args.steps):
            model.full_sort_topk(b, WORKLOAD['topk'], b['item_id'])
    torch.cuda.synchronize()
    print('profile run done')


# ------------------------------------------------------------------------------------------------
def oracle_step_fn(cfg, B, L, V, seed=42):
    """one reference-semantics training step on the CPU (oracle port): losses, two routed backward passes, Adam."""
    from oracle import acsr_oracle as O
    params = O.init_params(cfg, V, seed=seed)
    state = {k: (torch.zeros_like(v), torch.zeros_like(v)) for k, v in params.items()}
    seq, ln, pos = O.synth_batch(B, L, V, seed=seed)
    cnt = [0]

    def step():
        cnt[0] += 1
        rnd = O.draw_rand(cfg, B, L, seed=cnt[0], train=True)
        la, lc, grads = O.train_grads(params, cfg, seq, ln, pos, rnd)
        for k in params:
            params[k], m, v = O.adam_step(params[k], grads[k], state[k][0], state[k][1], cnt[0], 1e-4)
            state[k] = (m, v)
        return float(la), float(lc)
    return step


def oracle_eval_fn(cfg, B, L, V, k, seed=42):
    """one reference-semantics full-sort eval batch on the CPU (oracle port): forward, scores, scores[:,0] = -inf, top-k, hit flags
    (acsasrec.py:157-164, trainer.py:941-942, collector.py:145-153)."""
    from oracle import acsr_oracle as O
    params = O.init_params(cfg, V, seed=seed)
    seq, ln, pos = O.synth_batch(B, L, V, seed=seed)

    def step():
        with torch.no_grad():
            scores = O.full_sort_scores(params, cfg, seq, ln)
            _, idx = O.full_sort_topk(scores, k)
            return O.hit_flags(idx, pos)
    return step


def _timed_cpu(step, budget_s, max_n):
    step()                                       # warm-up
    t0 = time.time()
    n = 0
    while True:
        step()
        n += 1
        if time.time() - t0 > budget_s or n >= max_n:
            break
    return n, time.time() - t0


def sibling_models_record(A, dev, B, L, V, K):
    """SURVEY section 8 f-4: the sibling AC models on the same kernels, at the headline shape (C2: V, B, L of the workload, d = 64,
    2 layers, 2 heads).  Train step = calculate_loss + the two routed backward passes + fused Adam through the autograd Functions
    (eager launches; the fused one-pass step is AC-SASRec's), eval = the trainer's graphed full-sort batch.  Device-timed.  Next
    to each: the oracle port of the reference's CPU step on a bounded batch, all host threads."""
    from oracle import acsr_oracle as O
    out = {}
    base = model_cfg()
    base.update(n_layers=2, n_heads=2, hidden_size=64, inner_size=256, MAX_ITEM_LIST_LENGTH=L)
    common = dict(USER_ID_FIELD='user_id', ITEM_ID_FIELD='item_id', LIST_SUFFIX='_list', ITEM_LIST_LENGTH_FIELD='item_length',
                  NEG_PREFIX='neg_', TIME_FIELD='timestamp', device=dev, seed=42, learning_rate=1e-4, epochs=1, train_batch_size=B,
                  eval_batch_size=B, topk=[1, 3, 5, 10, 20, 50], metrics=['Hit', 'MRR', 'NDCG'], valid_metric='Hit@10',
                  checkpoint_dir='/tmp/acsr_bench_ckpt', cuda_graph=True, logits_passes=3)
    specs = [
        ('AcBERT4Rec', dict(combine_option='fixed', mask_ratio=0.2, MAX_ITEM_LIST_LENGTH=L - 1), A.AcBERT4Rec, A.AcBERT4RecTrainer),
        ('ACSSEPT', dict(user_hidden_size=32, item_hidden_size=32), A.ACSSEPT, A.ACSSEPTTrainer),
        ('ACTiSASRec', dict(time_span=256), A.ACTiSASRec, A.ACTiSASRecTrainer),
    ]
    Bc = 32                                    # rows of the CPU sample
    for name, extra, Model, Trainer in specs:
        try:
            d = dict(base)
            d.update(common)
            d.update(extra)
            config = A.Config(model=name, config_dict=d)
            config['model'] = name
            Lm = d['MAX_ITEM_LIST_LENGTH']
            ds = A.data.SyntheticSequentialDataset(config, 2 * B, V, seed=77, pin=False)
            torch.manual_seed(42)
            model = Model(config, ds).to(dev)
            trainer = Trainer(config, model)
            feat = ds.inter_feat
            batches = [A.Interaction({k: v[i * B:(i + 1) * B].to(dev) for k, v in feat.interaction.items()}) for i in range(2)]
            it = [0]

            graphed = bool(getattr(model, 'GRAPH_SAFE_STEP', False))

            def eager_step():
                trainer.train_step(batches[it[0] % 2])
                it[0] += 1

            hbatches = [A.Interaction({k: v[i * B:(i + 1) * B].clone().pin_memory() for k, v in feat.interaction.items()}) for i in range(2)]

            def step():
                if graphed:
                    # the captured step as the trainer's epoch loop runs it: a pinned host batch (what the loader yields) is copied into
                    # the static buffers and the graph replayed; AcBERT4Rec's python masking of the NEXT batch overlaps this replay
                    trainer.graphed_step(hbatches[it[0] % 2])
                    it[0] += 1
                else:
                    eager_step()

            def ev():
                b = batches[it[0] % 2]
                with torch.no_grad():
                    trainer.eval_batch((b, None, None, b['item_id']))
                it[0] += 1

            def timed(fn, n):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(n):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / n
            model.train()
            for _ in range(3):
                step()
            ms = timed(step, K)
            ms_eager = timed(eager_step, K) if graphed else ms
            model.eval()
            for _ in range(3):
                ev()
            ms_eval = timed(ev, K)
            # CPU: the oracle restatement of this model's reference step on Bc rows
            torch.set_num_threads(os.cpu_count() or 1)
            cfg = {k: d[k] for k in base}
            cfg.update({k: v for k, v in extra.items()})
            params = {k: v.detach().cpu() for k, v in model.state_dict().items()}
            seq, ln, tgt = (feat[k][:Bc] for k in ('item_id_list', 'item_length', 'item_id'))
            rnd = O.draw_rand(dict(cfg, hidden_size=model.hidden_size), Bc, Lm, 5)
            if name == 'AcBERT4Rec':
                import random
                random.seed(1)
                ms_, pi_, _, mi_ = model.reconstruct_train_data(seq)
                cpu_fn = lambda: O.bert_train_grads(params, cfg, ms_, pi_, mi_, rnd)
            elif name == 'ACSSEPT':
                cpu_fn = lambda: O.ssept_train_grads(params, cfg, seq, ln, feat['user_id'][:Bc], tgt, rnd)
            else:
                cpu_fn = lambda: O.ti_train_grads(params, cfg, seq, ln, feat['timestamp_list'][:Bc], tgt, rnd)
            cpu_fn()
            n, dt = _timed_cpu(cpu_fn, 4.0, 3)
            out[name] = {'train': {'value': round(B / (ms / 1e3), 1), 'unit': 'seq/s', 'ms_per_step': round(ms, 3),
                                   'eager_ms_per_step': round(ms_eager, 3),
                                   'launch': ('CUDA graph replay of the autograd step' + (' after the host-side masking of acbert4rec.py:86-150 (python, inside the timed region, overlapping the previous replay)'
                                                                                    if name == 'AcBERT4Rec' else '')) if graphed else 'eager launches'},
                         'eval': {'value': round(B / (ms_eval / 1e3), 1), 'unit': 'users/s', 'ms_per_batch': round(ms_eval, 3)},
                         'cpu_baseline': {'value': round(Bc * n / dt, 2), 'unit': 'seq/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                                          'sample': '%d oracle training steps (gradients, no optimizer) of B=%d' % (n, Bc)},
                         'config': 'V=%d B=%d L=%d hidden=%d layers=2 heads=2 %s' % (V, B, Lm, model.hidden_size, extra)}
            del trainer, model
            torch.cuda.empty_cache()
        except Exception as e:                                          # a sub-record must never sink the bench line
            out[name] = {'error': '%s: %s' % (type(e).__name__, str(e)[:300])}
    out['launch'] = 'train: the autograd Functions (routed double backward) + fused Adam; eval: CUDA graph replay'
    return out


def cpu_baseline(cfg, B, L, V, budget_s=20.0):
    torch.set_num_threads(os.cpu_count() or 1)
    n, dt = _timed_cpu(oracle_step_fn(cfg, B, L, V), budget_s, 10)
    return {'value': round(B * n / dt, 2), 'unit': 'seq/s', 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': '%d training steps of B=%d (oracle/acsr_oracle.py: CPU restatement of the reference step, all host threads; anomaly '
                      'mode OFF -- the reference as shipped runs with autograd anomaly detection ON (sine.py:25) and measured 1.3-1.8x '
                      'slower in the build container, BASELINE.md section 2)' % (n, B)}


def cpu_baseline_eval(cfg, B, L, V, k, budget_s=8.0):
    torch.set_num_threads(os.cpu_count() or 1)
    n, dt = _timed_cpu(oracle_eval_fn(cfg, B, L, V, k), budget_s, 20)
    return {'value': round(B * n / dt, 2), 'unit': 'users/s', 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': '%d full-sort eval batches of B=%d (oracle port: forward + scores + top-%d + hit flags)' % (n, B, k)}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    cfg = model_cfg()
    B, L, V, K, W = WORKLOAD['B'], WORKLOAD['L'], WORKLOAD['V'], args.steps, args.warmup
    torch.set_num_threads(os.cpu_count() or 1)
    step = oracle_step_fn(cfg, B, L, V)
    t0 = time.time()
    step()
    t1 = time.time() - t0
    Bs = B
    budget = 150.0
    if (K + W) * t1 > budget:                    # bounded sample: shrink the per-step batch so the run ends in minutes
        Bs = max(8, int(B * budget / ((K + W) * t1)))
        step = oracle_step_fn(cfg, Bs, L, V)
    for _ in range(W):
        step()
    t0 = time.time()
    for _ in range(K):
        step()
    dt = time.time() - t0
    val = round(Bs * K / dt, 2)
    cb = {'value': val, 'unit': 'seq/s', 'cores': torch.get_num_threads(), 'kind': 'port',
          'sample': '%d steps of B=%d of the workload (oracle port of the reference CPU path, anomaly mode OFF; /root/reference is Python and '
                    'cannot travel to the GPU box)' % (K, Bs)}
    ev = cpu_baseline_eval(cfg, Bs, L, V, WORKLOAD['topk'], budget_s=15.0)
    print(json.dumps({
        'impl': 'reference', 'metric': 'AC-SASRec train seq/s', 'value': val, 'unit': 'seq/s', 'n_gpus': int(args.gpus), 'steps': K,
        'warmup': W, 'ms_per_step': round(dt / K * 1e3, 3), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_string(bool(args.full_len))},
        'notes': {'cpu_sample_batch': Bs},
        'cpu_baseline': cb, 'e2e': {'value': val, 'unit': 'seq/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'eval': {'metric': 'AC-SASRec full-sort eval users/s', 'value': ev['value'], 'unit': 'users/s', 'cpu_baseline': ev,
                 'e2e': {'value': ev['value'], 'unit': 'users/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-parity', action='store_true', help='skip the in-run parity check against the CPU oracle')
    ap.add_argument('--no-large-batch', action='store_true', help='skip the B=2048 sub-record')
    ap.add_argument('--no-vocab-sharded', action='store_true', help='skip the 1M-item vocab-sharded sub-record')
    ap.add_argument('--no-siblings', action='store_true', help='skip the sibling-model (AcBERT4Rec / ACSSEPT / ACTiSASRec) sub-record')
    ap.add_argument('--no-long-seq', action='store_true', help='skip the long-sequence (config #5) sub-record')
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS), help='c2 = the headline configuration (default)')
    ap.add_argument('--full-len', action='store_true', help='every sequence has the maximum length (worst case) instead of LogNormal lengths')
    ap.add_argument('--batch', type=int, default=0, help='override the per-GPU batch of the workload')
    ap.add_argument('--dp-graph', type=int, default=1, help='capture the NCCL all-reduce inside the CUDA graph at N>1 (0 = eager launches)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what their callers receive: the two losses of the last timed training '
                         'step and the hit flags of the last timed eval batch, as DIR/<name>.npy')
    ap.add_argument('--profile', action='store_true',
                    help='launch-list mode for ncu: W+K eager training steps and K eval batches, nothing else')
    args = ap.parse_args()
    if args.dump_outputs and (args.profile or args.impl != 'ours'):
        ap.error('--dump-outputs writes the outputs of the timed steps of --impl ours')
    WORKLOAD.clear()
    WORKLOAD.update(WORKLOADS[args.workload])
    if args.batch > 0:
        WORKLOAD['B'] = args.batch
    if args.profile:
        return run_profile(args)
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
