"""ctypes binding of libacsr.so, generated from the prototypes in include/acsr.h.

There is NO fallback: if the library cannot be built/loaded, every op raises.
"""
import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HEADER = os.path.join(ROOT, 'include', 'acsr.h')
LIB_PATH = os.path.join(HERE, 'csrc', 'libacsr.so')

_CTYPES = {
    'int': ctypes.c_int, 'float': ctypes.c_float, 'double': ctypes.c_double,
    'int64_t': ctypes.c_int64, 'uint32_t': ctypes.c_uint32, 'int32_t': ctypes.c_int32,
}


def parse_header(path=HEADER):
    """-> {name: (restype, [(argname, ctype)])} for every `acsr_*` prototype."""
    src = open(path).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    protos = {}
    for m in re.finditer(r'(const\s+char\s*\*|int64_t|int)\s+(acsr_\w+)\s*\(([^)]*)\)\s*;', src, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        restype = ctypes.c_char_p if 'char' in ret else (ctypes.c_int64 if ret == 'int64_t' else ctypes.c_int)
        argl = []
        args = ' '.join(args.split())
        if args and args != 'void':
            for a in args.split(','):
                a = a.strip()
                mm = re.match(r'(.*?)(\w+)$', a)
                typ, aname = mm.group(1).strip(), mm.group(2)
                if '*' in typ:
                    argl.append((aname, ctypes.c_void_p))
                else:
                    argl.append((aname, _CTYPES[typ.replace('const', '').strip()]))
        protos[name] = (restype, argl)
    return protos



class GemmProblem(ctypes.Structure):
    """mirror of `acsr_gemm_problem` (include/acsr.h); strides in floats, pointers are device addresses."""
    _fields_ = [
        ('A', ctypes.c_void_p), ('a_row_stride', ctypes.c_int64), ('a_k_stride', ctypes.c_int64), ('a_kb_stride', ctypes.c_int64),
        ('B', ctypes.c_void_p), ('b_row_stride', ctypes.c_int64), ('b_k_stride', ctypes.c_int64), ('b_kb_stride', ctypes.c_int64),
        ('C', ctypes.c_void_p), ('ldc', ctypes.c_int64),
        ('M', ctypes.c_int64),
        ('bias', ctypes.c_void_p), ('colsum', ctypes.c_void_p), ('C2', ctypes.c_void_p),
        ('res', ctypes.c_void_p), ('res_rows', ctypes.c_int64),
        ('ln_w', ctypes.c_void_p), ('ln_b', ctypes.c_void_p),
        ('mask', ctypes.c_void_p), ('rng', ctypes.c_void_p),
        ('out', ctypes.c_void_p), ('stats', ctypes.c_void_p),
        ('a_kblk', ctypes.c_int32), ('b_kblk', ctypes.c_int32),
        ('N', ctypes.c_int32), ('K', ctypes.c_int32),
        ('epilogue', ctypes.c_int32), ('accumulate', ctypes.c_int32), ('k_splits', ctypes.c_int32), ('act', ctypes.c_int32),
        ('rng_stream', ctypes.c_uint32), ('eps', ctypes.c_float), ('p_drop', ctypes.c_float), ('reserved', ctypes.c_int32),
    ]


EPI_STORE, EPI_ATOMIC, EPI_ACT, EPI_BDRL = 0, 1, 2, 3
GEMM_MAX_PROBLEMS = 16

class AcsrError(RuntimeError):
    pass


class _Lib:
    def __init__(self):
        self._dll = None
        self.protos = parse_header()
        self.timer = None            # KernelTimer while bench.py measures per-kernel device time

    def load(self):
        if self._dll is not None:
            return self._dll
        if not os.path.exists(LIB_PATH):
            raise AcsrError(
                'libacsr.so is not built (%s). Run `python -c "import __graft_entry__ as g; g.build()"` '
                'or `python ac-tsr_b200/build.py`. There is no CPU / PyTorch fallback for the hot path.' % LIB_PATH)
        dll = ctypes.CDLL(LIB_PATH)
        for name, (restype, argl) in self.protos.items():
            fn = getattr(dll, name)          # AttributeError if a declared symbol is missing
            fn.restype = restype
            fn.argtypes = [t for _, t in argl]
        if dll.acsr_version() != 1:
            raise AcsrError('libacsr.so ABI version mismatch')
        self._dll = dll
        return dll

    def call(self, name, *args):
        dll = self.load()
        if self.timer is not None:
            return self.timer.timed_call(self, dll, name, args)
        rc = getattr(dll, name)(*args)
        if rc != 0:
            msg = dll.acsr_last_error()
            raise AcsrError('%s failed (%d): %s' % (name, rc, msg.decode() if msg else ''))

    def query(self, name, *args):
        return getattr(self.load(), name)(*args)

    def ensure_workspace(self, nbytes, device):
        """caller-owned scratch of `device` (acsr_set_workspace): one torch allocation, grown on demand, never shrunk."""
        import torch
        if not hasattr(self, '_ws'):
            self._ws = {}
        idx = device.index if device.index is not None else torch.cuda.current_device()
        cur = self._ws.get(idx)
        if cur is not None and cur.numel() >= nbytes:
            return cur
        if torch.cuda.is_current_stream_capturing():
            raise AcsrError('the attention workspace (%d bytes) must be allocated before CUDA-graph capture: run one eager step first' % nbytes)
        with torch.cuda.device(idx):
            torch.cuda.synchronize()
            buf = torch.empty(int(nbytes), dtype=torch.uint8, device=torch.device('cuda', idx))
            rc = self.load().acsr_set_workspace(buf.data_ptr(), int(nbytes))
            if rc != 0:
                raise AcsrError('acsr_set_workspace failed (%d)' % rc)
        self._ws[idx] = buf
        return buf


def _ab_linear_tok(a):
    # (X, ldx, xkb, rows, K, W, w_sn, w_sk, wkb, N, bias, accumulate, Y, ldy, batch, ...)
    rows, K, N, acc, batch = a[3], a[4], a[9], a[11], a[14]
    return 4 * batch * (rows * K + rows * N * (2 if acc else 1) + N * K)


def _ab_dense_bwd(a):
    # (d_out, rows, act_rows, res_rows, param_rows, d, I, ...): d_out, the saved z2 / h / hz [., 64], z1 [., I], stats and the residual
    # in; d_xres, d_ctx [rows, 64] out, d_z2 / d_hz [param_rows, 64] and d_z1 [param_rows, I] out; weights in
    rows, act_rows, res_rows, keep, d, I = a[1], a[2], a[3], a[4], a[5], a[6]
    ra = min(rows, act_rows)
    return 4 * (rows * d + ra * (3 * d + I + 4) + min(rows, res_rows) * d + 2 * rows * d + keep * (2 * d + I) + d * d + 2 * d * I)


def _ab_linear_tok_bdrl(a):
    # (X, ldx, rows, K, W, bias, res, res_rows, ...): X, W in; HZ, out, stats out; residual in
    rows, K = a[2], a[3]
    return 4 * (rows * K + 64 * K + 3 * rows * 64 + 2 * rows)


def _ab_proj_input_grad(a):
    # (d_qkv, d_aqk, plane_rows, d_gl, L, Wqkv, Waqk, Wg, d, rows, rows_keep, d_x, ...): d_aq, d_ak, d_mq, d_mk, d_mv (+ d_gl) in,
    # rows_keep rows of d_mq / d_mk written back, d_x read and written, weights in
    L, d, rows, keep = (a[4] if a[3] else 0), a[8], a[9], a[10]
    return 4 * (rows * (5 * d + L) + 2 * keep * d + 2 * rows * d + 5 * d * d + L * d)


def _ab_linear_wgrad(a):
    # (dY, X, T, N, K, dW, db, stream)
    T, N, K = a[2], a[3], a[4]
    return 4 * (T * (N + K) + N * K)


def _ab_linear_wgrad_batched(a):
    # (dY, X, T, N, K, dW, db, batch, ...)
    T, N, K, batch = a[2], a[3], a[4], a[7]
    return 4 * batch * (T * (N + K) + N * K)


def _ab_gemm_batch(a):
    # (problems array, n, passes, stream): operands read once, result written once (read-modify-write when accumulating)
    arr, n = a[0], a[1]
    tot = 0
    for i in range(n):
        p = arr[i]
        out_mult = 2 if (p.accumulate or p.epilogue in (EPI_ATOMIC, EPI_ACT)) else 1
        tot += 4 * (p.M * p.K + p.N * p.K + p.M * p.N * out_mult)
        if p.epilogue == EPI_BDRL:
            tot += 4 * (2 * p.M * p.N + 2 * p.M)       # residual in, normalised row out, stats
    return tot


def _ab_neg_sample(a):
    # (users, positives, perm, cursor, n_rows, M, N, ...): per row the user id, positive, permutation entry and two offsets in;
    # the M*N negatives out (the used-set probes of the binary searches are L2-resident and not counted)
    M, N = a[5], a[6]
    return 8 * (M * N + 5 * M)


def _ab_candidate_rank(a):
    # (out, table, V, d, cand, M, n_cand, kmax, rec, scores, stream): out rows and candidate ids in, one table row per candidate
    # gathered, hit flags (and scores) out
    d, M, C, kmax = a[3], a[5], a[6], a[7]
    return 4 * M * d + M * C * (8 + 4 * d) + 4 * M * (kmax + 1) + (4 * M * C if a[9] else 0)


def _ab_candidate_rank_counts(a):
    # (out, table, V, d, cand, M, n_cand, kmax, rec, scores, counts, stream): acsr_candidate_rank + three counts per row out
    return _ab_candidate_rank(a) + 12 * a[5]


def _ab_candidate_scores_shard(a):
    # (out, shard, lo, hi, V, d, cand, M, n_cand, scores, stream): out rows and candidate ids in, the owned candidates' rows
    # gathered (counted as all of them: the owned share is data-dependent), scores out
    d, M, C = a[5], a[7], a[8]
    return 4 * M * d + M * C * (8 + 4 * d) + 4 * M * C


def _ab_candidate_rank_scores(a):
    # (scores, cand, V, M, n_cand, kmax, rec, counts, stream): scores and ids in, hit flags (and counts) out
    M, C, kmax = a[3], a[4], a[5]
    return 12 * M * C + 4 * M * (kmax + 1) + (12 * M if a[7] else 0)


def _ab_bpr_dots_shard(a):
    # (out, shard, lo, hi, V, pos, neg, M, d, dots, stream): out rows, two ids and two table rows per row in, two dots out
    M, d = a[7], a[8]
    return 4 * M * 3 * d + 16 * M + 8 * M


def _ab_bpr_loss_from_dots(a):
    # (dots, M, n_groups, gamma, row_x, row_loss, loss, stream): dots in, row_x / row_loss out, row_loss read back for the means
    M = a[1]
    return 8 * M + 8 * M + 4 * M


def _ab_bpr_loss_bwd_shard(a):
    # (out, shard, lo, hi, V, pos, neg, row_x, row_scale, M, d, gamma, begin, end, d_out, d_shard, stream): per row two ids, x,
    # scale and two table rows in, d_out out; the training rows also read out and add into two gradient rows
    M, d, n_tab = a[9], a[10], max(0, a[13] - a[12])
    return M * (24 + 4 * 2 * d + (4 * d if a[14] else 0)) + n_tab * 4 * (d + 4 * d)


def _ab_grad_norm_partial(a):
    # (grad, n, ranges, n_ranges, norm_type, block_partials, counter, out, stream): the ranges' gradients read once, the norm out
    rg, nr = a[2], a[3]
    return 4 * sum(rg[2 * r + 1] - rg[2 * r] for r in range(nr)) + 8


def _ab_adam_step_clipped(a):
    # (param, grad, exp_avg, exp_avg_sq, n, lr, b1, b2, eps, wd, step_count, partials, n_partials, ...): Adam's 28 B per parameter,
    # the clipped gradient written back, the norm partials read
    return 32 * a[4] + 8 * a[12]


# ALGORITHMIC bytes of one launch, from the call's own arguments (DESIGN.md section 4)
ALGO_BYTES = {'acsr_linear_tok': _ab_linear_tok, 'acsr_linear_tok_bdrl': _ab_linear_tok_bdrl,
              'acsr_proj_input_grad': _ab_proj_input_grad, 'acsr_dense_bwd': _ab_dense_bwd,
              'acsr_linear_wgrad': _ab_linear_wgrad, 'acsr_linear_wgrad_batched': _ab_linear_wgrad_batched,
              'acsr_gemm_batch': _ab_gemm_batch, 'acsr_neg_sample': _ab_neg_sample, 'acsr_candidate_rank': _ab_candidate_rank,
              'acsr_candidate_rank_counts': _ab_candidate_rank_counts, 'acsr_candidate_scores_shard': _ab_candidate_scores_shard,
              'acsr_candidate_rank_scores': _ab_candidate_rank_scores, 'acsr_bpr_dots_shard': _ab_bpr_dots_shard,
              'acsr_bpr_loss_from_dots': _ab_bpr_loss_from_dots, 'acsr_bpr_loss_bwd_shard': _ab_bpr_loss_bwd_shard,
              'acsr_grad_norm_partial': _ab_grad_norm_partial, 'acsr_adam_step_clipped': _ab_adam_step_clipped}


class KernelTimer:
    """Brackets every C-ABI launch with CUDA events on the launching (current torch) stream.
    Used by bench.py for the per-kernel share / roofline numbers; never active in the timed step."""

    def __init__(self, keep_calls=False):
        self.events = []             # (name, start, stop)
        self.launches = 0
        self.calls = [] if keep_calls else None      # (name, args, algorithmic bytes) of every launch, for replay_in_graph

    def timed_call(self, lib, dll, name, args):
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(dll, name)(*args)
        e1.record()
        if rc != 0:
            msg = dll.acsr_last_error()
            raise AcsrError('%s failed (%d): %s' % (name, rc, msg.decode() if msg else ''))
        fn = ALGO_BYTES.get(name)
        ab = fn(args) if fn is not None else None
        self.events.append((name, e0, e1, ab))
        if self.calls is not None:
            self.calls.append((name, args, ab, torch.cuda.current_stream()))
        self.launches += 1

    def summary(self):
        """-> {name: (n_calls, total_ms)} after a device synchronize; self.bytes = {name: algorithmic bytes or None}."""
        import torch
        torch.cuda.synchronize()
        out, self.bytes = {}, {}
        for name, e0, e1, ab in self.events:
            n, t = out.get(name, (0, 0.0))
            out[name] = (n + 1, t + e0.elapsed_time(e1))
            if ab is not None:
                self.bytes[name] = self.bytes.get(name, 0) + ab
        return out


def replay_in_graph(lib, calls, reps=16, skip=('acsr_adam_step', 'acsr_rng_advance'), per_call=None):
    """Device time of every recorded launch INSIDE a CUDA graph: each call (same arguments, same buffers) is captured `reps`
    times back to back into its own graph and the replay is bracketed by events -- no host launch path and no event-record
    overhead between the kernels (an event pair around one eager launch costs ~12 us on B200, more than most kernels of the
    step), warm L2 as in the real step, programmatic dependent launch between the copies as between the step's kernels.
    -> {name: [n_calls, total_us, total_algorithmic_bytes]}.  Calls that change persistent state (optimizer, rng) are skipped."""
    import torch
    dll = lib.load()
    out = {}
    side = torch.cuda.Stream()
    for name, args, ab, _ in calls:
        if name in skip:
            continue
        a = list(args)
        fn = getattr(dll, name)
        argl = lib.protos[name][1]
        si = [i for i, (an, _) in enumerate(argl) if an == 'stream']
        g = torch.cuda.CUDAGraph()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            if si:
                a[si[0]] = side.cuda_stream
            rc = fn(*a)                                        # warm-up outside the capture (function attributes, L2)
            side.synchronize()
            with torch.cuda.graph(g, stream=side):
                if si:
                    a[si[0]] = torch.cuda.current_stream().cuda_stream
                for _ in range(reps):
                    rc |= fn(*a)
            if rc != 0:
                raise AcsrError('%s failed during the in-graph replay' % name)
            g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            g.replay()
            e1.record()
            side.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / (2 * reps)
        rec = out.setdefault(name, [0, 0.0, 0])
        rec[0] += 1
        rec[1] += us
        rec[2] += ab or 0
        if per_call is not None:
            per_call.append((name, [x for x in args if isinstance(x, int) and abs(x) < (1 << 24)][:12], round(us, 2), ab))
        del g
    torch.cuda.current_stream().wait_stream(side)
    return out


LIB = _Lib()
