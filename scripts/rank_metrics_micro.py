"""Cost of counting the positive's rank (GAUC) inside the full-sort top-k: one graphed evaluation batch (B = 256 users, k = 50,
hidden size 64) of ops.full_sort_topk with and without counts, at C2 (V = 12,102: tensor-core scores + dense select) and C4
(V = 1,000,001: the fused tcgen05 logits + streaming top-k).  The two variants are captured as CUDA graphs and replayed in
alternating rounds in one process; the result line carries the card name and its power limit.

    python scripts/rank_metrics_micro.py [--rounds 9] [--reps 200] [--out results/rank_metrics_micro.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=9)
    ap.add_argument('--reps', type=int, default=200)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('rank_metrics_micro: needs a CUDA device')
    import ac_tsr_b200 as A
    A.LIB.load()
    res = {'card': card(), 'B': 256, 'k': 50, 'd': 64, 'rounds': a.rounds, 'reps_per_round': a.reps, 'cases': {}}
    g = torch.Generator(device='cuda').manual_seed(0)
    for name, V in (('C2', 12102), ('C4', 1000001)):
        B = 256
        out = torch.randn(B, 64, generator=g, device='cuda')
        E = torch.randn(V, 64, generator=g, device='cuda') * 0.1
        pos = torch.randint(1, V, (B,), generator=g, device='cuda')
        graphs = {}
        for variant, counts in (('plain', False), ('counts', True)):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    A.ops.full_sort_topk(out, E, 50, pos, counts=counts)
            torch.cuda.current_stream().wait_stream(side)
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                r = A.ops.full_sort_topk(out, E, 50, pos, counts=counts)
            graphs[variant] = (gr, r)
        gr_p, r_p = graphs['plain']
        gr_c, r_c = graphs['counts']
        gr_p.replay(); gr_c.replay()
        torch.cuda.synchronize()
        same = all(torch.equal(x, y) for x, y in zip(r_p[:3], r_c[:3]))
        times = {'plain': [], 'counts': []}
        for rnd in range(a.rounds):
            order = ('plain', 'counts') if rnd % 2 == 0 else ('counts', 'plain')
            for v in order:
                gr = graphs[v][0]
                for _ in range(10):
                    gr.replay()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.reps):
                    gr.replay()
                e1.record()
                torch.cuda.synchronize()
                times[v].append(e0.elapsed_time(e1) * 1e3 / a.reps)
        med = {v: sorted(t)[len(t) // 2] for v, t in times.items()}
        res['cases'][name] = {'V': V, 'us_per_batch_median': {v: round(x, 2) for v, x in med.items()},
                              'us_per_batch_min_max': {v: [round(min(t), 2), round(max(t), 2)] for v, t in times.items()},
                              'added_us': round(med['counts'] - med['plain'], 2),
                              'added_pct': round(100.0 * (med['counts'] / med['plain'] - 1.0), 2),
                              'topk_bitwise_equal': bool(same)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as fh:
            fh.write(line + '\n')


if __name__ == '__main__':
    main()
