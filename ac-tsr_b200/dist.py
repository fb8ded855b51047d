"""Vocab-parallel item table and logits for the multi-GPU path (SURVEY section 8e; north_star: "batches are data-parallel,
and the item table and logits are vocab-sharded with NCCL-over-NVLink allreduce of the per-row max/sum (training) and an
allgather of partial top-k (eval)").  One process per GPU; the encoder is batch data-parallel; the reference has no
distributed code at all (single process, configurator.py:344-348), so everything here is new.

Two storage modes:
  replicated (small catalogues): every rank keeps the whole table; only the logits / CE / top-k WORK is split by item rows.
  sharded    (large catalogues): rank r keeps rows [lo, hi) of the table, their gradient and their Adam moments.
      embedding rows of a rank's own tokens: all-gather of the item ids, each owner answers with the rows it holds (zeros
      elsewhere: acsr_shard_gather_rows), reduce-scatter(sum) delivers them; backward: all-gather of the per-token gradient
      rows, each owner adds the rows it owns (acsr_shard_scatter_add_rows).  The table never moves and the data-parallel
      all-reduce shrinks to the encoder parameters.  Break-even against replication: 2 * W * B * L rows exchanged per step
      versus V rows all-reduced, i.e. sharding pays for V > ~2*W*B*L (204,800 items at 8 ranks, B=256, L=50).

  training  : all-gather `out` -> every rank runs the fused tcgen05 CE-partial kernel on ITS table rows for ALL rows ->
              all-gather of the per-row (max, sum-exp) pairs and of the owner's target logit -> local combine (log-sum-exp);
              backward: d_out partial = G.E_shard and dE_shard = G^T.out_calibrated with the shard-local G recomputed tile by
              tile inside the two kernels (acsr_ce_bwd_dout / _dtable: no gradient matrix in HBM); reduce-scatter(sum) of
              d_out; dE_shard needs no traffic.
  evaluation: all-gather `out` -> fused top-k on the shard (indices offset by the shard start, column 0 skipped on shard 0)
              -> merge of the shard's chunk lists into one list per row -> all-gather of those lists -> merge of the rank's own rows.

The collective plumbing is backend-agnostic: `compute` supplies the local kernels (CUDA ops by default; the gloo CPU tests
inject torch restatements), so world_size-2 tests run without a GPU.  Nothing here allocates by value from the host inside the
step (no torch.tensor(...) constructors), so the whole vocab-parallel step is CUDA-graph capturable.
"""
import torch
import torch.distributed as dist


class CudaCompute(object):
    """the local kernels, bound to libacsr.so through ops.py"""

    def __init__(self, passes=3, d=64):
        from . import ops
        from ._lib import LIB
        self.ops, self.passes, self.LIB, self.d = ops, passes, LIB, d

    def num_chunks(self, rows, shard_rows):
        return self.ops.logits_num_chunks(rows, shard_rows, self.d) if shard_rows > 0 else 1

    def ce_partial(self, out, table):
        return self.ops.ce_partial(out, table, self.passes)

    def ce_backward_local(self, out_all, table, lse, target_local, row_scale, row_begin, n_rows, table_grad):
        """-> d_out_all [M,d] = G . table over this shard's items, G = (softmax - onehot(target_local)) * row_scale; when
        table_grad is given, table_grad += G[row_begin:row_begin+n_rows]^T . out_all[row_begin:row_begin+n_rows].  Hidden size
        64: G is recomputed tile by tile and stays in registers (acsr_ce_bwd_dout / _dtable); other widths write the shard-local
        Gt [rows, M] once and run both contractions as two problems of ONE tcgen05 launch."""
        ops = self.ops
        M, d = out_all.shape
        V = table.shape[0]
        d_out = torch.zeros((M, d), dtype=torch.float32, device=out_all.device)
        if d == 64:
            ops.ce_bwd_dout(out_all, table, lse, target_local, row_scale, d_out, self.passes)
            if table_grad is not None and n_rows > 0:
                sl = slice(row_begin, row_begin + n_rows)
                ops.ce_bwd_dtable(out_all[sl], table, lse[sl], target_local[sl], row_scale[sl], table_grad, self.passes)
            return d_out
        Gt = ops.ce_grad_matrix_t(out_all, table, lse, target_local, row_scale, self.passes)
        pr = [ops.wgrad_problem(Gt, table, V, M, d, d_out)]
        if table_grad is not None and n_rows > 0:
            pr.append(ops.gemm_problem(Gt[:, row_begin:], out_all[row_begin:], table_grad, V, d, n_rows, a_strides=(M, 1, 0, n_rows),
                                       b_strides=(1, d, 0, n_rows), accumulate=True))
        ops.gemm_batch(pr, passes=self.passes)
        return d_out

    def topk_partial(self, out, table, k, idx_offset, skip_col0):
        return self.ops.logits_topk_partial(out, table, k, idx_offset, skip_col0, self.passes)

    def topk_merge(self, pv, pi, k, positive):
        return self.ops.topk_merge(pv, pi, k, positive)

    def row_dot(self, out, table, ids, idx_offset):
        return self.ops.row_dot(out, table, ids, idx_offset)

    def topk_rank_partial(self, out, table, k, positive, pos_score, idx_offset, skip_col0):
        return self.ops.logits_topk_rank_partial(out, table, k, positive, pos_score, idx_offset, skip_col0, self.passes)

    def topk_merge_rank(self, pv, pi, k, pc, positive):
        return self.ops.topk_merge_rank(pv, pi, k, pc, positive)

    def gather_rows(self, ids, shard, lo, hi):
        out = torch.empty((ids.numel(), shard.shape[1]), dtype=torch.float32, device=shard.device)
        self.LIB.call('acsr_shard_gather_rows', self.ops._p(ids, torch.int64), ids.numel(), self.ops._p(shard), lo, hi, shard.shape[1],
                      self.ops._p(out), self.ops._stream())
        return out

    def scatter_add_rows(self, ids, rows, lo, hi, shard_grad):
        self.LIB.call('acsr_shard_scatter_add_rows', self.ops._p(ids, torch.int64), ids.numel(), self.ops._p(rows), lo, hi, rows.shape[1],
                      self.ops._p(shard_grad), self.ops._stream())


class VocabParallel(object):
    def __init__(self, n_items, group=None, compute=None, align=64, sharded=False):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        per = (n_items + self.world - 1) // self.world
        per = (per + align - 1) // align * align                 # whole 64-row tiles per shard
        self.V, self.per = n_items, per
        self.lo = min(n_items, self.rank * per)
        self.hi = min(n_items, self.lo + per)
        self.compute = compute or CudaCompute()
        self.shard_rows = [max(0, min(n_items, (r + 1) * per) - min(n_items, r * per)) for r in range(self.world)]
        self.sharded = bool(sharded)          # the table handed to the methods below IS this rank's shard ([per, d], rows >= hi-lo unused)
        if min(self.shard_rows) == 0:
            raise ValueError('vocab-parallel: %d items in shards of %d rows leave some of the %d ranks without rows' % (n_items, per, self.world))

    def _ncmax(self, rows):
        """largest per-shard chunk count, computed on the host from the shard sizes (no sync, graph-capturable)"""
        return max(self.compute.num_chunks(rows, sr) for sr in self.shard_rows)

    # ------------------------------------------------------------------------------------------
    def _all_gather(self, t):
        t = t.contiguous()
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t, group=self.group)
        return out.view((self.world,) + tuple(t.shape))

    def _reduce_scatter(self, t_all, rows):
        """t_all [W*rows, ...] summed over ranks -> this rank's block [rows, ...]"""
        if dist.get_backend(self.group) == 'nccl':
            out = torch.empty((rows,) + tuple(t_all.shape[1:]), dtype=t_all.dtype, device=t_all.device)
            dist.reduce_scatter_tensor(out, t_all.contiguous(), op=dist.ReduceOp.SUM, group=self.group)
            return out
        t_all = t_all.contiguous()                                           # gloo (CPU tests): no reduce-scatter
        dist.all_reduce(t_all, group=self.group)
        return t_all[self.rank * rows:(self.rank + 1) * rows].clone()

    def shard(self, table):
        """this rank's rows of the table (a view): of the full table (replicated storage) or of the stored shard"""
        return table[:self.hi - self.lo] if self.sharded else table[self.lo:self.hi]

    def make_shard(self, full_table):
        """[per, d] copy of this rank's rows, zero padded to the common shard size (equal collective sizes on every rank)"""
        s = torch.zeros((self.per, full_table.shape[1]), dtype=full_table.dtype, device=full_table.device)
        s[:self.hi - self.lo].copy_(full_table[self.lo:self.hi])
        return s

    def gather_full(self, shard):
        """all ranks' shards -> the full [V, d] table in the reference layout (checkpoints, state_dict)"""
        return self._all_gather(shard.detach()).reshape(self.world * self.per, -1)[:self.V].clone()

    # ---- sharded storage: embedding rows of this rank's tokens ---------------------------------------
    def fetch_rows(self, ids_local, shard, out=None):
        """ids_local [T] int64 -> (rows [T,d] = table[ids_local], ids of every rank [W,T] for scatter_grad_rows)"""
        T = ids_local.numel()
        ids_all = self._all_gather(ids_local.reshape(T))
        rows_all = self.compute.gather_rows(ids_all.reshape(-1), shard, self.lo, self.hi)        # [W*T, d], zeros where not owned
        rows = self._reduce_scatter(rows_all, T)
        if out is not None:
            out.copy_(rows)
            rows = out
        return rows, ids_all

    def scatter_grad_rows(self, ids_all, d_rows_local, shard_grad):
        """gradient rows of this rank's tokens [T,d] -> added into the owners' gradient shards (padding id 0 skipped)"""
        rows_all = self._all_gather(d_rows_local)
        self.compute.scatter_add_rows(ids_all.reshape(-1), rows_all.reshape(-1, rows_all.shape[-1]), self.lo, self.hi, shard_grad)

    # ------------------------------------------------------------------------------------------
    def ce_forward(self, out_local, table, target_local, n_groups):
        """-> (loss [n_groups] over this rank's rows, saved state for ce_backward).  Rows of every rank are laid out group-major
        ([group][rank][row]) so that the rows that train the table form one contiguous range for the backward GEMM."""
        R, d = out_local.shape
        W, per = self.world, R // n_groups
        out_all = self._all_gather(out_local.view(n_groups, per, d)).permute(1, 0, 2, 3).reshape(W * R, d).contiguous()
        tgt_all = self._all_gather(target_local.view(n_groups, per)).permute(1, 0, 2).reshape(W * R).contiguous()
        E_s = self.shard(table)
        rows_s = E_s.shape[0]
        ncmax = self._ncmax(W * R)
        part = self.compute.ce_partial(out_all, E_s)                         # [W*R, nc, 2]
        if part.shape[1] < ncmax:                                            # ragged chunk counts: pad with (-inf, 0)
            pad = part.new_zeros((part.shape[0], ncmax - part.shape[1], 2))
            pad[..., 0] = -float('inf')
            part = torch.cat((part, pad), 1)
        # the owner of a row's target item contributes the target logit (the other shards add 0)
        t_loc = tgt_all - self.lo
        own = (t_loc >= 0) & (t_loc < rows_s)
        dot = (out_all * E_s[t_loc.clamp(0, rows_s - 1)]).sum(1) * own.to(out_all.dtype)
        packed = torch.cat((part.reshape(W * R, ncmax * 2), dot.view(W * R, 1)), 1)               # one collective for both
        gathered = self._all_gather(packed).view(W, n_groups, W, per, ncmax * 2 + 1)
        mine = gathered[:, :, self.rank].permute(1, 2, 0, 3).reshape(R, W, ncmax * 2 + 1)       # my rows on every shard
        tgt_logit = mine[..., -1].sum(1)
        pm = mine[..., :-1].reshape(R, W * ncmax, 2)
        m = pm[..., 0].max(dim=1).values
        s = (pm[..., 1] * torch.exp(pm[..., 0] - m.unsqueeze(1))).sum(1)
        lse = m + torch.log(s)
        row_loss = lse - tgt_logit
        loss = row_loss.view(n_groups, per).mean(1)
        return loss, dict(out_all=out_all, tgt_all=tgt_all, lse=lse, R=R, n_groups=n_groups)

    def ce_backward(self, st, table, row_scale_local, table_grad=None, table_half=None, n_groups=2):
        """row_scale_local [R]: d loss / d row_loss of this rank's rows.  -> d_out_local [R,d]; when table_grad is given, dE of
        the owned rows is accumulated into it (the stored gradient shard, or rows [lo,hi) of a full-size gradient) from the
        row group `table_half` -- the calibrated rows (trainer.py:672-686)."""
        R, W = st['R'], self.world
        per = R // n_groups
        d = table.shape[1]
        lse_all = self._all_gather(st['lse'].view(n_groups, per)).permute(1, 0, 2).reshape(W * R).contiguous()
        scale_all = self._all_gather(row_scale_local.view(n_groups, per)).permute(1, 0, 2).reshape(W * R).contiguous()
        E_s = self.shard(table)
        tg = self.shard(table_grad) if table_grad is not None else None
        # [W*R, d] partial over my item rows; dE of my rows from the training group of every rank (no traffic)
        d_out_all = self.compute.ce_backward_local(st['out_all'], E_s, lse_all, (st['tgt_all'] - self.lo).contiguous(), scale_all,
                                                   (table_half or 0) * W * per, W * per, tg)
        # back to [rank][group][row] blocks, then every rank receives the sum of its own rows
        d_out_all = d_out_all.view(n_groups, W, per, d).permute(1, 0, 2, 3).reshape(W * R, d)
        return self._reduce_scatter(d_out_all, R)

    # ------------------------------------------------------------------------------------------
    def full_sort_topk(self, out_local, table, k, positive_local=None, counts=False):
        """all-gather of partial top-k lists (north_star eval path) -> (val [R,k], idx [R,k], rec|None).  Each rank first merges
        its shard's per-chunk lists into one list per row, so the final merge sees W*k candidates however many chunks a shard
        runs (W * 148 chunk lists of k would exceed the merge's capacity).  counts=True: also counts [R, 2] int32 (GAUC's rank
        inputs, ops.full_sort_topk) -- every shard counts its own items against the positive's score, which the owner of the
        positive's row computes (the others contribute 0 to a sum, like the CE target logit), and the per-row counts are summed."""
        R, d = out_local.shape
        out_all = self._all_gather(out_local).view(self.world * R, d)
        if counts:
            E_s = self.shard(table)
            pos_all = self._all_gather(positive_local.reshape(R)).view(self.world * R)
            s_pos = self.compute.row_dot(out_all, E_s, pos_all, self.lo)
            dist.all_reduce(s_pos, group=self.group)
            pv, pi, pc = self.compute.topk_rank_partial(out_all, E_s, k, pos_all, s_pos, self.lo, self.lo == 0)
            sv, si, _, sc = self.compute.topk_merge_rank(pv, pi, k, pc, None)                     # [W*R, k], [W*R, 2]
            sl = slice(self.rank * R, (self.rank + 1) * R)
            mv = self._all_gather(sv)[:, sl].permute(1, 0, 2).contiguous()                         # [R, W, k]
            mi = self._all_gather(si)[:, sl].permute(1, 0, 2).contiguous()
            mc = self._all_gather(sc)[:, sl].permute(1, 0, 2).contiguous()                         # [R, W, 2]
            return self.compute.topk_merge_rank(mv, mi, k, mc, positive_local)
        pv, pi = self.compute.topk_partial(out_all, self.shard(table), k, self.lo, self.lo == 0)   # [W*R, nc, k]
        sv, si, _ = self.compute.topk_merge(pv, pi, k, None)                                      # [W*R, k]
        sl = slice(self.rank * R, (self.rank + 1) * R)
        mv = self._all_gather(sv)[:, sl].permute(1, 0, 2).contiguous()                             # [R, W, k]
        mi = self._all_gather(si)[:, sl].permute(1, 0, 2).contiguous()
        return self.compute.topk_merge(mv, mi, k, positive_local)
