"""Exact tests of the full-sort top-k kernels: the fused tcgen05 streaming top-k (hidden size 64, with and without the per-row
bound its CTAs share), the fp32 SIMT streaming top-k (other hidden sizes), the dense radix select, the merge of per-chunk and
per-shard lists, and the vocab-parallel composition of dist.py.

`out` and the item table hold small integers, so every score is an integer far below 2^24 whose operands are exact in TF32: the
3xTF32 split has a zero low half, the fp32 accumulators and the SIMT FMAs are exact, and every path has to match a float64
reference with no tolerance.  The rows follow score patterns that Gaussian scores never produce: the best items in the last
tiles of the streams, k-1 items above a plateau (the k-th best equal to the shared bound), exactly k items above a flat
background in k different streams, constant rows and heavy random ties.

Contract checked for every row: `val` is the k largest reference scores, sorted descending (column 0 excluded when skipped);
the ids are distinct, lie in [idx_offset, idx_offset + V), are never column 0 when it is skipped, and score exactly `val`;
rec = hit flags of the returned ids + pos_len 1.  The dense select also keeps its documented tie order (lowest id first); the
fused paths promise the ids only up to exact ties."""
import json
import os
import sys
import time

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

from oracle import acsr_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATTERNS = ('rising', 'steps', 'falling', 'plateau_first', 'plateau_last', 'k_above', 'constant', 'random')
N_PAT_COLS = 5             # item-table columns 0..4 carry the designed patterns, the others random integers in [-4, 4]


@pytest.fixture(scope='module')
def A():
    import ac_tsr_b200 as pkg
    pkg.LIB.load()
    return pkg


# ---- integer cases -------------------------------------------------------------------------------
def _k_above_items(V, k, nc):
    """k distinct items, one in the last tile of each of k different streams (2 streams per chunk: the two 32-column halves of
    its 64-item tiles; chunk c owns tiles c, c + nc, ...).  Streams that hold more than one item, or items that fall outside
    the catalogue, are topped up with the last items of the catalogue."""
    n_tiles = (V + 63) // 64
    items = []
    for j in range(k):
        s = j % (2 * nc)
        c, h = s // 2, s % 2
        t = c + ((n_tiles - 1 - c) // nc) * nc
        item = t * 64 + h * 32 + 1 + j // (2 * nc)
        if 0 < item < V and item not in items:
            items.append(item)
    it = V - 1
    while len(items) < k:
        if it not in items:
            items.append(it)
        it -= 1
    return items


def make_case(V, d, k, M, seed, nc=None, dev='cuda'):
    """(out [M,d], E [V,d], pattern name of every row) on `dev`, all small integers.  Row r follows PATTERNS[(r + seed) % 8]:
      rising        score = item id (the best items in the last tile of every stream)
      steps         score = id // 128 (128-item plateaus, heavy ties at the top)
      falling       score = -id
      plateau_first k-1 items score 1 inside the first tile, every other item 0: the answer is those k-1 plus one plateau item
      plateau_last  the same inside the last full tile of the catalogue
      k_above       exactly k items score 1, one in the last tile of each of k different streams, every other item 0
      constant      every item scores 0
      random        random integer weights on the random columns"""
    assert d > N_PAT_COLS and V >= k + 1
    g = torch.Generator(device=dev).manual_seed(seed)
    E = torch.randint(-4, 5, (V, d), generator=g, device=dev).float()
    ids = torch.arange(V, device=dev)
    E[:, 0] = (ids // 128).float()
    E[:, 1] = (ids % 128).float()
    E[:, 2:N_PAT_COLS] = 0.0
    E[1:k, 2] = 1.0
    t_last = max(0, V // 64 - 1) * 64
    E[t_last + 1:t_last + k, 3] = 1.0
    E[torch.tensor(_k_above_items(V, k, nc or 1), device=dev), 4] = 1.0
    out = torch.zeros(M, d)
    names = []
    for r in range(M):
        p = PATTERNS[(r + seed) % len(PATTERNS)]
        names.append(p)
        if p == 'rising':
            out[r, 0], out[r, 1] = 128.0, 1.0
        elif p == 'steps':
            out[r, 0] = 1.0
        elif p == 'falling':
            out[r, 0], out[r, 1] = -128.0, -1.0
        elif p == 'plateau_first':
            out[r, 2] = 1.0
        elif p == 'plateau_last':
            out[r, 3] = 1.0
        elif p == 'k_above':
            out[r, 4] = 1.0
    rnd = [r for r, p in enumerate(names) if p == 'random']
    if rnd:
        out[rnd, N_PAT_COLS:] = torch.randint(-4, 5, (len(rnd), d - N_PAT_COLS), generator=torch.Generator().manual_seed(seed)).float()
    return out.to(dev), E, names


def chunk_has_fewer_than_k(V, nc, k, skip_col0):
    """whether some chunk of a launch with nc chunks (tiles c, c + nc, ... of 64 items) holds fewer than k candidates"""
    n_tiles = (V + 63) // 64
    for c in range(nc):
        n = sum(min(64, V - t * 64) for t in range(c, n_tiles, nc)) - (1 if c == 0 and skip_col0 else 0)
        if n < k:
            return True
    return False


def reference(out, E, k, skip_col0=True, stable=False):
    """float64 top-k of out.E^T in row blocks -> (values [M,k] float64, ids [M,k]); stable=True: ties to the lowest id"""
    o64, E64 = out.double(), E.double()
    vals, idxs = [], []
    for i in range(0, out.shape[0], 256):
        s = o64[i:i + 256] @ E64.t()
        if skip_col0:
            s[:, 0] = -float('inf')
        if stable:
            v, ix = torch.sort(s, dim=1, descending=True, stable=True)
            v, ix = v[:, :k], ix[:, :k]
        else:
            v, ix = torch.topk(s, k, dim=1)
        vals.append(v)
        idxs.append(ix)
    return torch.cat(vals), torch.cat(idxs)


def exact_scores(out, E, cols):
    """float64 scores of row r against item table row cols[r, j]"""
    return torch.einsum('rd,rjd->rj', out.double(), E.double()[cols])


def make_positives(ref_idx, V, seed, lo=0):
    """even rows: the reference's best item (a hit); odd rows: a random item of [lo, V)"""
    g = torch.Generator(device=ref_idx.device).manual_seed(seed)
    pos = torch.randint(lo, V, (ref_idx.shape[0],), generator=g, device=ref_idx.device)
    pos[0::2] = ref_idx[0::2, 0]
    return pos


def _rows(mask, names):
    bad = torch.nonzero(mask).view(-1)[:5].tolist()
    return ', '.join('row %d (%s)' % (r, names[r] if names else '-') for r in bad)


def check_contract(val, idx, rec, out, E, k, pos, ref_val, idx_offset=0, skip_col0=True, ref_idx=None, names=None, what=''):
    dev = out.device
    val, idx = val.to(dev), idx.to(dev)
    M, V = out.shape[0], E.shape[0]
    assert val.shape == (M, k) and idx.shape == (M, k), what
    bad = (val.double() != ref_val).any(1)
    assert not bad.any(), '%s: top-k values differ from the reference at %s' % (what, _rows(bad, names))
    inside = (idx >= idx_offset) & (idx < idx_offset + V)
    if skip_col0:
        inside &= idx != idx_offset
    assert inside.all(), '%s: ids outside the catalogue (or column 0) at %s' % (what, _rows(~inside.all(1), names))
    if k > 1:
        s = idx.sort(1).values
        dup = (s[:, 1:] == s[:, :-1]).any(1)
        assert not dup.any(), '%s: repeated ids at %s' % (what, _rows(dup, names))
    wrong = (exact_scores(out, E, idx - idx_offset) != val.double()).any(1)
    assert not wrong.any(), '%s: returned values are not the scores of the returned ids at %s' % (what, _rows(wrong, names))
    if ref_idx is not None:
        order = (idx != ref_idx + idx_offset).any(1)
        assert not order.any(), '%s: ties not resolved to the lowest id at %s' % (what, _rows(order, names))
    if rec is not None:
        rec = rec.to(dev)
        assert rec.shape == (M, k + 1), what
        assert torch.equal(rec[:, :k], (idx == pos.to(dev).view(-1, 1)).int()), '%s: hit flags' % what
        assert (rec[:, k] == 1).all(), '%s: pos_len column' % what


def check_lists(pv, pi, out, E, lo, skip_col0, what=''):
    """every entry of the per-chunk partial lists is padding (-inf, -1) or an id of [lo, lo + V) with its exact score"""
    M, nc, k = pv.shape
    valid = pi >= 0
    assert torch.equal(pv[~valid], torch.full_like(pv[~valid], -float('inf'))), '%s: padding entries must be -inf' % what
    cols = (pi - lo).clamp(min=0)
    assert ((cols < E.shape[0]) | ~valid).all(), '%s: list ids beyond the shard' % what
    if skip_col0:
        assert not (valid & (pi == lo)).any(), '%s: column 0 in a list' % what
    got = exact_scores(out, E, cols.clamp(max=E.shape[0] - 1).view(M, nc * k)).view(M, nc, k)
    assert torch.equal(pv.double()[valid], got[valid]), '%s: list values are not the scores of their ids' % what


def fused(A, out, E, k, pos, idx_offset, skip_col0, passes, share_bound):
    pv, pi = A.ops.logits_topk_partial(out, E, k, idx_offset, skip_col0, passes, share_bound=share_bound)
    assert pv.shape == (out.shape[0], A.ops.logits_num_chunks(out.shape[0], E.shape[0]), k)
    val, idx, rec = A.ops.topk_merge(pv, pi, k, pos)
    return pv, pi, val, idx, rec


def bound_on(A, M, V, k):
    """whether the CTAs of a hidden-size-64 launch share the per-row bound: two streams per CTA, at least k of them"""
    return 2 * A.ops.logits_num_chunks(M, V) >= k


# ---- fused tcgen05 path (hidden size 64) ---------------------------------------------------------
V_FUSED = 200003
FUSED_M = (1, 129, 512, 640, 768, 2048)


def test_fused_grid_covers_both_sides_of_the_shared_bound(A):
    for k in (50, 64):
        sides = {bound_on(A, M, V_FUSED, k) for M in FUSED_M}
        assert sides == {True, False}, (k, sides)


@pytest.mark.parametrize('M', FUSED_M)
@pytest.mark.parametrize('passes', [3, 1])
@pytest.mark.parametrize('k', [1, 10, 50, 57, 64])
def test_fused_topk_exact(A, k, passes, M):
    V = V_FUSED
    seed = 1000 * k + 10 * passes + M
    nc = A.ops.logits_num_chunks(M, V)
    out, E, names = make_case(V, 64, k, M, seed, nc)
    # odd M: a later vocab shard (ids offset, column 0 kept)
    idx_offset, skip_col0 = (3 * V + 5, False) if M % 2 else (0, True)
    ref_val, ref_idx = reference(out, E, k, skip_col0)
    pos = make_positives(ref_idx, V, seed) + idx_offset
    vals = []
    for share in (True, False):
        what = 'k=%d passes=%d M=%d bound %s' % (k, passes, M, 'shared (on)' if share and bound_on(A, M, V, k) else 'off')
        pv, pi, val, idx, rec = fused(A, out, E, k, pos, idx_offset, skip_col0, passes, share)
        check_lists(pv, pi, out, E, idx_offset, skip_col0, what)
        check_contract(val, idx, rec, out, E, k, pos, ref_val, idx_offset, skip_col0, names=names, what=what)
        vals.append(val)
    assert torch.equal(vals[0], vals[1])


# ---- fp32 SIMT path (other hidden sizes) ---------------------------------------------------------
@pytest.mark.parametrize('M', [129, 640])
@pytest.mark.parametrize('k', [50, 64])
@pytest.mark.parametrize('d', [32, 128])
def test_simt_topk_exact(A, d, k, M):
    V = 60001
    seed = 7 * d + k + M
    out, E, names = make_case(V, d, k, M, seed, A.ops.logits_num_chunks(M, V))
    idx_offset, skip_col0 = (V + 11, False) if M % 2 else (0, True)
    ref_val, ref_idx = reference(out, E, k, skip_col0)
    pos = make_positives(ref_idx, V, seed) + idx_offset
    pv, pi = A.ops.logits_topk_partial(out, E, k, idx_offset, skip_col0, 3)
    assert pv.shape == (M, A.ops.logits_num_chunks(M, V), k)
    check_lists(pv, pi, out, E, idx_offset, skip_col0, 'simt d=%d' % d)
    val, idx, rec = A.ops.topk_merge(pv, pi, k, pos)
    check_contract(val, idx, rec, out, E, k, pos, ref_val, idx_offset, skip_col0, names=names, what='simt d=%d k=%d M=%d' % (d, k, M))


# ---- ragged chunks: lists with fewer than k valid items, padded with -1 --------------------------
@pytest.mark.parametrize('M', [1, 300])
@pytest.mark.parametrize('V', [65, 129, 128 * 9 + 1, 128 * 74 + 1])
def test_ragged_chunks_exact(A, V, M):
    k = 64
    for d in (64, 128):
        seed = V + M + d
        out, E, names = make_case(V, d, k, M, seed, A.ops.logits_num_chunks(M, V))
        ref_val, ref_idx = reference(out, E, k, True)
        pos = make_positives(ref_idx, V, seed)
        for share in ((True, False) if d == 64 else (True,)):
            what = 'd=%d V=%d M=%d share_bound=%s' % (d, V, M, share)
            pv, pi, val, idx, rec = fused(A, out, E, k, pos, 0, True, 3, share)
            # a chunk with fewer than k items pads its list; with the bound shared, items at or below it are dropped as well
            short, padded = chunk_has_fewer_than_k(V, pv.shape[1], k, True), bool((pi < 0).any())
            if short or not (share and d == 64 and bound_on(A, M, V, k)):
                assert padded == short, what + ': padding of the lists'
            check_lists(pv, pi, out, E, 0, True, what)
            check_contract(val, idx, rec, out, E, k, pos, ref_val, names=names, what=what)


# ---- scores + dense radix select (small catalogues) -----------------------------------------------
def select_max(A):
    return A.LIB.query('acsr_topk_select_max_items')


@pytest.mark.parametrize('d', [64, 256])
@pytest.mark.parametrize('V', [65, 129, 12102, 'max'])
def test_select_topk_exact_and_lowest_id_on_ties(A, V, d):
    V = select_max(A) if V == 'max' else V
    M = 264
    for k in (50, 64):
        seed = V + d + k
        out, E, names = make_case(V, d, k, M, seed, A.ops.logits_num_chunks(M, V))
        scores = A.ops.logits_scores(out, E, 3)
        for idx_offset, skip_col0 in ((0, True), (12345, False)):
            ref_val, ref_idx = reference(out, E, k, skip_col0, stable=True)
            pos = make_positives(ref_idx, V, seed) + idx_offset
            val, idx, rec = A.ops.topk_select(scores, k, pos, skip_col0, idx_offset)
            check_contract(val, idx, rec, out, E, k, pos, ref_val, idx_offset, skip_col0, ref_idx=ref_idx, names=names,
                           what='select V=%d d=%d k=%d skip_col0=%s' % (V, d, k, skip_col0))


@pytest.mark.parametrize('d', [64, 256])
def test_full_sort_topk_both_sides_of_the_select_limit(A, d):
    """ops.full_sort_topk takes scores + select up to acsr_topk_select_max_items() items and the streaming top-k + merge above"""
    n = select_max(A)
    with pytest.raises(A.AcsrError):
        A.ops.topk_select(torch.zeros(2, n + 1, device='cuda'), 10)
    M, k = 136, 50
    for V in sorted({n, n + 1, 57344, 57345}):
        seed = V + d
        out, E, names = make_case(V, d, k, M, seed, A.ops.logits_num_chunks(M, V))
        ref_val, ref_idx = reference(out, E, k, True, stable=True)
        pos = make_positives(ref_idx, V, seed)
        for passes in (3, 1):
            val, idx, rec = A.ops.full_sort_topk(out, E, k, pos, passes)
            check_contract(val, idx, rec, out, E, k, pos, ref_val, ref_idx=ref_idx if V <= n else None, names=names,
                           what='full_sort_topk V=%d d=%d passes=%d' % (V, d, passes))


# ---- one Gaussian case per path, at shapes the kernel tests do not use ---------------------------
@pytest.mark.parametrize('path', ['fused', 'simt', 'select'])
def test_gaussian_topk_modulo_ties(A, path):
    V, d, M, k = {'fused': (V_FUSED, 64, 300, 64), 'simt': (60001, 128, 300, 64), 'select': (select_max(A), 256, 64, 64)}[path]
    g = torch.Generator(device='cuda').manual_seed(V + d)
    out = torch.randn(M, d, generator=g, device='cuda')
    E = torch.randn(V, d, generator=g, device='cuda') * 0.5
    scores = out.double() @ E.double().t()
    pos = torch.randint(1, V, (M,), generator=g, device='cuda')
    if path == 'select':
        val, idx, rec = A.ops.topk_select(A.ops.logits_scores(out, E, 3), k, pos)
    else:
        if path == 'fused':
            assert bound_on(A, M, V, k)
        pv, pi = A.ops.logits_topk_partial(out, E, k, 0, True, 3)
        val, idx, rec = A.ops.topk_merge(pv, pi, k, pos)
    idx, val, rec, scores = idx.cpu(), val.cpu(), rec.cpu(), scores.cpu()
    assert (idx > 0).all() and (val[:, :-1] >= val[:, 1:]).all()
    exact = torch.gather(scores, 1, idx)
    assert float((val.double() - exact).abs().max()) <= 3e-6 * float(scores.abs().max())
    _, ref_idx = O.full_sort_topk(scores.float(), k)
    ok, nbad = O.topk_equal_modulo_ties(idx, ref_idx, scores.float())
    assert ok, nbad
    assert torch.equal(rec[:, :-1], O.hit_flags(idx, pos.cpu())) and (rec[:, -1] == 1).all()


# ---- vocab shards on one GPU: per-shard lists (ids offset, column 0 kept) + one merge -------------
def shard_bounds(V, W, k):
    """W row ranges; the last one holds fewer rows than k"""
    small = k - 27
    per = (V - small + W - 2) // (W - 1)
    b = [min(V - small, i * per) for i in range(W)] + [V]
    return list(zip(b[:-1], b[1:]))


@pytest.mark.parametrize('d', [64, 128])
@pytest.mark.parametrize('W', [2, 3, 8])
def test_vocab_shards_merge_exact(A, W, d):
    V, M, k = 60001, 200, 64
    seed = 31 * W + d
    out, E, names = make_case(V, d, k, M, seed)
    ref_val, ref_idx = reference(out, E, k, True)
    bounds = shard_bounds(V, W, k)
    assert bounds[-1][1] - bounds[-1][0] < k and all(hi > lo for lo, hi in bounds)
    pos = make_positives(ref_idx, V, seed, lo=bounds[-1][0])           # odd rows: a positive in the last shard
    ncmax = max(A.ops.logits_num_chunks(M, hi - lo) for lo, hi in bounds)
    assert W * ncmax * k <= select_max(A)
    pvs, pis = [], []
    for lo, hi in bounds:
        pv, pi = A.ops.logits_topk_partial(out, E[lo:hi].contiguous(), k, lo, lo == 0, 3)
        check_lists(pv, pi, out, E[lo:hi], lo, lo == 0, 'shard [%d, %d)' % (lo, hi))
        padn = ncmax - pv.shape[1]                                     # padded as dist.py pads ragged chunk counts
        pvs.append(torch.cat((pv, pv.new_full((M, padn, k), -float('inf'))), 1))
        pis.append(torch.cat((pi, pi.new_full((M, padn, k), -1)), 1))
    val, idx, rec = A.ops.topk_merge(torch.cat(pvs, 1), torch.cat(pis, 1), k, pos)
    check_contract(val, idx, rec, out, E, k, pos, ref_val, names=names, what='W=%d d=%d' % (W, d))
    assert bool((idx >= bounds[-1][0]).any()) and bool(rec[:, :k].any())     # the last shard holds some winners and positives


# ---- the real VocabParallel (dist.py) with the CUDA kernels, gloo collectives on CPU tensors ------
def _vp_worker(rank, world, port, V, d, k, Rs, outdir):
    sys.path.insert(0, ROOT)
    ret = {}
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        import ac_tsr_b200 as A
        A.LIB.load()

        class GpuCompute(A.dist.CudaCompute):
            """the CUDA kernels on the one GPU, their results handed back on the CPU for gloo"""

            def topk_partial(self, out, table, k, idx_offset, skip_col0):
                pv, pi = super().topk_partial(out.cuda(), table.cuda(), k, idx_offset, skip_col0)
                return pv.cpu(), pi.cpu()

            def topk_merge(self, pv, pi, k, positive):
                r = super().topk_merge(pv.cuda(), pi.cuda(), k, positive.cuda() if positive is not None else None)
                return tuple(t.cpu() if t is not None else None for t in r)

        for R in Rs:
            seed = 17 * R + world + d
            out_all, E, names = make_case(V, d, k, world * R, seed)
            mine = slice(rank * R, (rank + 1) * R)
            out = out_all[mine]
            ref_val, ref_idx = reference(out, E, k, True)
            pos = make_positives(ref_idx, V, seed)
            for sharded in (False, True):
                key = '%d R=%d %s' % (rank, R, 'sharded' if sharded else 'replicated')
                try:
                    vp = A.dist.VocabParallel(V, compute=GpuCompute(3, d), sharded=sharded)
                    table = vp.make_shard(E) if sharded else E
                    val, idx, rec = vp.full_sort_topk(out.cpu(), table, k, pos.cpu())
                    check_contract(val, idx, rec, out, E, k, pos, ref_val, names=names[mine], what=key)
                    ret[key] = 'ok'
                except Exception as e:          # every rank fails alike, so the collectives of the next case still match
                    ret[key] = '%s: %s' % (type(e).__name__, str(e)[:300])
    finally:
        dist.destroy_process_group()
    with open(os.path.join(outdir, 'rank%d.json' % rank), 'w') as fh:
        json.dump(ret, fh)


@pytest.mark.parametrize('W,d', [(2, 64), (8, 64), (8, 128)])
def test_vocab_parallel_full_sort_topk_cuda(W, d, tmp_path):
    """W ranks share the one GPU.  V = 160,001 gives shards of 313 (W = 8) or 1251 tiles; at R <= 16 users per rank the W*R
    gathered rows form one 128-row tile, so every shard runs 148 chunks."""
    V, k, Rs = 160001, 50, (1, 16, 17)
    port = 29300 + (os.getpid() + 7 * W + d) % 300
    ctx = mp.start_processes(_vp_worker, args=(W, port, V, d, k, Rs, str(tmp_path)), nprocs=W, join=False, start_method='spawn')
    deadline = time.time() + 900
    try:
        while not ctx.join(timeout=5):
            assert time.time() < deadline, 'vocab-parallel workers did not finish in time'
    finally:
        for p in ctx.processes:
            if p.is_alive():
                p.terminate()
            p.join()
    want = {'%d R=%d %s' % (r, R, s) for r in range(W) for R in Rs for s in ('replicated', 'sharded')}
    got = {}
    for r in range(W):
        with open(os.path.join(str(tmp_path), 'rank%d.json' % r)) as fh:
            got.update(json.load(fh))
    assert set(got) == want, sorted(want - set(got))
    bad = {key: v for key, v in got.items() if v != 'ok'}
    assert not bad, bad
