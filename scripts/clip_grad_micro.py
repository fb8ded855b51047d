"""Cost of gradient clipping by global norm (`clip_grad_norm`) on one GPU:

    python scripts/clip_grad_micro.py [--out DIR] [--steps N]

Prints one JSON line (and writes it to DIR/clip_grad_micro.json):
  - the in-graph time per launch (each launch captured `reps` times back to back in one CUDA graph and replayed, as bench.py
    times kernels) of acsr_grad_norm_partial (norm_type 2), acsr_adam_step_clipped and plain acsr_adam_step, at the C2 flat
    size (the AC-SASRec parameters of the C2 shape, ~0.9 M floats, L2-resident) and at the C4 size (64 M floats, a 256 MB
    gradient), with their algorithmic bytes;
  - the C2 training step (V = 12 102, B = 256, L = 50, d = 64, 2 layers) in ms: the fused graphed step without clipping, the
    same step with clip_grad_norm on the device, and the clipped step as it ran before the device clip (torch's clip_grad_norm_
    on the autograd path, eager launches: `fused_step: False` plus an extra clip_grad_norm_ key keeps that path); the three are
    timed in alternating rounds;
  - the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import ac_tsr_b200 as A  # noqa: E402
from ac_tsr_b200 import _lib  # noqa: E402
from oracle import acsr_oracle as O  # noqa: E402


def gpu_info():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def kernel_us(n, dev, reps=16):
    """in-graph us per launch of the norm, the clipped Adam and the plain Adam over a flat buffer of n floats"""
    g = torch.Generator(device=dev).manual_seed(n % 997)
    grad = torch.randn(n, device=dev, generator=g) * 1e-3
    param = torch.randn(n, device=dev, generator=g)
    m, v = torch.zeros_like(param), torch.zeros_like(param)
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    work = A.ops.grad_norm_work(dev)
    part = torch.zeros(1, dtype=torch.float64, device=dev)
    timer = _lib.KernelTimer(keep_calls=True)
    A.LIB.timer = timer
    try:
        A.ops.grad_norm_partial(grad, 2.0, out=part, work=work)
        # max_norm far above the norm: coefficient 1, so the replays do not shrink the gradient (the same work either way)
        A.ops.adam_step_clipped(param, grad, m, v, step, 1e-4, part, 2.0, 1e30)
        A.ops.adam_step(param, grad, m, v, step, 1e-4)
    finally:
        A.LIB.timer = None
    torch.cuda.synchronize()
    out = _lib.replay_in_graph(A.LIB, timer.calls, reps=reps, skip=())
    res = {}
    for name, (cnt, us, ab) in out.items():
        res[name] = dict(us=round(us / cnt, 2), bytes=ab // cnt if name != 'acsr_adam_step' else 28 * n,
                         gbps=round((ab // cnt if name != 'acsr_adam_step' else 28 * n) / (us / cnt) / 1e3, 1))
    return res


def c2_trainer(dev, clip, fused):
    cfg = O.default_cfg()
    V, B, L = 12102, 256, 50
    d = dict(cfg, USER_ID_FIELD='user_id', ITEM_ID_FIELD='item_id', LIST_SUFFIX='_list', ITEM_LIST_LENGTH_FIELD='item_length',
             NEG_PREFIX='neg_', device=dev, seed=42, learning_rate=1e-4, epochs=1, train_batch_size=B, eval_batch_size=B,
             topk=[10], metrics=['Hit'], valid_metric='Hit@10', checkpoint_dir='/tmp/acsr_clip_micro', cuda_graph=True,
             fused_step=fused, clip_grad_norm=clip, MAX_ITEM_LIST_LENGTH=L)
    config = A.Config(model='ACSASRec', config_dict=d)

    class DS:
        item_num = V

        def num(self, f):
            return V
    torch.manual_seed(42)
    model = A.ACSASRec(config, DS()).to(dev)
    trainer = A.ACSASRecTrainer(config, model)
    model.train()
    g = torch.Generator().manual_seed(7)
    inter = A.Interaction({'item_id_list': torch.randint(1, V, (B, L), generator=g).to(dev), 'item_length': torch.full((B,), L).to(dev),
                           'item_id': torch.randint(1, V, (B,), generator=g).to(dev)})
    return trainer, inter


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('clip_grad_micro.py measures on the GPU; no CUDA device here')
    dev = torch.device('cuda')
    A.LIB.load()
    res = {'gpus': gpu_info()}
    arms = {'fused_graphed_no_clip': (None, True), 'fused_graphed_device_clip': ({'max_norm': 0.5, 'norm_type': 2}, True),
            'autograd_eager_torch_clip': ({'max_norm': 0.5, 'norm_type': 2, 'foreach': None}, False)}
    runs = {}
    for name, (clip, fused) in arms.items():
        tr, inter = c2_trainer(dev, clip, fused)
        assert (tr.fused is not None) == fused and tr.torch_clip == (name == 'autograd_eager_torch_clip')
        step = (lambda tr=tr, inter=inter: tr.train_step(inter)) if tr.torch_clip else (lambda tr=tr, inter=inter: tr.graphed_step(inter))
        for _ in range(10):
            step()
        runs[name] = (tr, step)
    flat_c2 = runs['fused_graphed_no_clip'][0].optimizer.flat_grad.numel()
    res['kernels'] = {'c2_flat_%d' % flat_c2: kernel_us(flat_c2, dev), 'c4_flat_%d' % (64 * 2 ** 20): kernel_us(64 * 2 ** 20, dev)}
    times = {k: [] for k in arms}
    for _ in range(a.rounds):
        for name, (tr, step) in runs.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(round(e0.elapsed_time(e1) / a.steps, 4))
    res['c2_step_ms'] = {k: dict(rounds=v, min=min(v)) for k, v in times.items()}
    res['c2_step_ms']['note'] = 'V=12102, B=256, L=50, d=64, 2 layers, 2 heads, dropout 0.5; %d steps per round, arms alternating' % a.steps
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'clip_grad_micro.json'), 'w') as fh:
            fh.write(line + '\n')


if __name__ == '__main__':
    main()
