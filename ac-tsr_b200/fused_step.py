"""Explicit (autograd-free) AC-SASRec training step.

The reference trainer runs two backward traversals with requires_grad toggling (trainer.py:672-686):
attack_{query,key}_transform receive d(attacked_loss), every other parameter d(calibrated_loss).
Backward is linear in the cotangent, so here BOTH cotangent streams travel together as the two halves
of every gradient buffer ([stream 0 = calibrated loss ; stream 1 = attacked loss], 2T rows), each
kernel / GEMM is launched once for both, and every weight gradient reads the half that owns it and
accumulates straight into the flat gradient buffer (no autograd tape, no temporaries, no adds).

Dead work the reference performs is skipped without changing any result: the attacked branch of
non-final layers, the attacked branch's weight gradients, the attacked stream below the first layer.

At B=256 every kernel of the step is latency-bound (a few hundred CTAs, ~10 us each), so the step is
laid out as a DAG instead of a chain: the batch is cut into `step_branches` groups of sequences whose
encoder forward and backward run on parallel CUDA streams (parallel branches of the captured graph;
sequences only meet in the full-catalogue cross entropy, in the penalty norm and in the gradient
buffers, which are accumulated with atomics), and inside a branch the weight-gradient reductions,
which nothing consumes before Adam, run on a second stream next to the input-gradient chain.

All buffers are allocated once per batch size, so the step is CUDA-graph capturable as is.
"""
import math

import torch

from . import ops
from ._lib import LIB
from .ops import _p, _stream


class _RandSlice(object):
    """explicit masks / noise of a parity test ({key: full-batch tensor}), restricted to one branch's sequences."""

    def __init__(self, rand, sl):
        self.rand, self.sl = rand, sl

    def get(self, key):
        t = self.rand.get(key)
        return None if t is None else t[self.sl].contiguous()


class FusedTrainStep(object):
    def __init__(self, model, optimizer):
        if model.loss_type not in ('CE', 'BPR'):
            raise NotImplementedError("Make sure 'loss_type' in ['BPR', 'CE']!")
        self.m, self.opt = model, optimizer
        self.buf = {}
        self.vp = None            # dist.VocabParallel when the logits are sharded over ranks
        # d == 64: every encoder GEMM runs on the tcgen05 token-tile kernel (3xTF32) with its epilogue fused.  Every other width
        # (d = 128 of the shipped yelp / sports / toys configs, d = 256 of BASELINE config #5): the K-streamed tcgen05 kernel
        # (gemm_ks.cu) through problem lists.  At every width the weight gradients of a layer go through it as ONE launch (token
        # axis on K, split over the CTAs).  No library GEMM is left on the step.
        self.tc = model.hidden_size == 64 and model.inner_size <= 256 and model.inner_size % 4 == 0
        self.passes = 3                                   # encoder GEMMs: 3xTF32 (fp32-level accuracy)
        self.overlap_wgrad = True                         # weight gradients on a second stream next to the input-gradient chain
        self.n_branches = int(getattr(model, 'step_branches', 1))
        self._streams = {}
        self.pdl = True                                   # programmatic dependent launch between the step's kernels
        # last layer's dense part on the compact rows as ONE launch per direction (acsr_tail_fwd / _bwd); other inner sizes: six launches
        self.tail_fused = self.tc and model.inner_size % 16 == 0
        # backward of a layer's dense part (two LayerNorm backwards, the activation backward, three input-gradient GEMMs) as ONE
        # tcgen05 launch (acsr_dense_bwd: d_a1 / d_z1 stay in tensor memory); other inner sizes: the six launches
        self.dense_bwd = self.tc and model.inner_size % 64 == 0
        # CE backward without the [2B,V] gradient matrix (acsr_ce_bwd_dout / _dtable); other widths go through Gt
        self.ce_fused_bwd = model.hidden_size == 64

    # ------------------------------------------------------------------------------------------
    def _stream_for(self, dev, key):
        if key not in self._streams:
            self._streams[key] = torch.cuda.Stream(device=dev)
        return self._streams[key]

    def _branch_buffers(self, Bs, L, dev, idx, grads=True):
        """activations saved for the backward + (grads) gradient buffers of one group of Bs sequences."""
        key = ('branch', Bs, L, idx)
        if key in self.buf:
            return self.buf[key]
        m = self.m
        d, I, N = m.hidden_size, m.inner_size, m.n_layers
        T = Bs * L

        def f(*s):
            return torch.empty(s, dtype=torch.float32, device=dev)
        b = dict(T=T, x0=f(T, d), st_e=f(T, 2), layers=[], order=torch.empty(Bs, dtype=torch.int32, device=dev))
        for l in range(N):
            last = l == N - 1
            # mixed_q, mixed_k, mixed_v, attack_q, attack_k: one batched GEMM writes all
            qkv5 = f(5, T, d)
            qkv, aqk = qkv5[:3], qkv5[3:]
            lb = dict(qkv5=qkv5, qkv=qkv, aqk=aqk, mq=qkv[0], mk=qkv[1], mv=qkv[2], aq=aqk[0], ak=aqk[1], gl=f(T, L),
                      ctx=f(2 * T if last else T, d))
            if not last:                       # the last layer's dense part runs on the compact rows of b['c']
                lb.update(hz=f(T, d), st_a=f(T, 2), h=f(T, d), z1=f(T, I), a1=f(T, I), z2=f(T, d), st_f=f(T, 2), out=f(T, d))
            # buffers read by the weight-gradient kernels are per layer: the side stream may still be reading layer l's
            # while the branch stream already writes layer l-1's
            if grads:
                lb['d_gl'] = f(2 * T, L)
                if not last:
                    lb['d_z2'], lb['d_z1'], lb['d_hz'] = f(2 * T, d), f(2 * T, I), f(2 * T, d)
                lb['d_qkv'], lb['d_aqk'] = f(3, 2 * T, d), f(2, 2 * T, d)
                lb['d_mq'], lb['d_mk'], lb['d_mv'] = lb['d_qkv'][0], lb['d_qkv'][1], lb['d_qkv'][2]
                lb['d_aq'], lb['d_ak'] = lb['d_aqk'][0], lb['d_aqk'][1]
            b['layers'].append(lb)
        # last layer: only position len-1 of each sequence feeds the losses, so everything after its attention runs on
        # 2*Bs compact rows ([calibrated ; attacked]) instead of 2*T
        C = 2 * Bs
        b['c'] = dict(ctx=f(C, d), x=f(Bs, d), hz=f(C, d), st_a=f(C, 2), h=f(C, d), z1=f(C, I), a1=f(C, I), z2=f(C, d), st_f=f(C, 2),
                      out=f(C, d), d_out=f(C, d), d_z2=f(C, d), d_h=f(C, d), d_a1=f(C, I), d_z1=f(C, I), d_hz=f(C, d), d_x=f(C, d),
                      d_ctx=f(C, d))
        if grads:
            for n, w in (('d_out', d), ('d_a1', I), ('d_h', d), ('d_x', d), ('d_ctx', d)):
                b[n] = f(2 * T, w)
        self.buf[key] = b
        return b

    def _joint_buffers(self, B, dev):
        """full-batch buffers of the part where the sequences meet: last-position outputs, cross entropy, penalty."""
        key = ('joint', B)
        if key in self.buf:
            return self.buf[key]
        m = self.m
        d, N, V = m.hidden_size, m.n_layers, m.n_items

        def f(*s):
            return torch.empty(s, dtype=torch.float32, device=dev)
        nc = ops.logits_num_chunks(2 * B, V, d)
        loss3 = f(3)              # [CE(calibrated), CE(attacked), final attacked loss]: one buffer, one read-back
        j = dict(pen=torch.zeros(N, dtype=torch.float64, device=dev), out2=f(2 * B, d), partial=f(2 * B, nc, 2), lse=f(2 * B),
                 tgt=f(2 * B), row_loss=f(2 * B), loss3=loss3, loss=loss3[:2], loss_att=loss3[2:], dpen=f(N), Gt=None,      # [V, 2B] transposed CE gradient: allocated on first use (never under vocab-parallel / BPR)
                 d_out2=f(2 * B, d),
                 target2=torch.empty(2 * B, dtype=torch.int64, device=dev), ce_cnt=torch.zeros(1, dtype=torch.int32, device=dev),
                 neg2=torch.empty(2 * B, dtype=torch.int64, device=dev), row_x=f(2 * B),
                 row_scale=torch.cat((torch.full((B,), 1.0 / B), torch.full((B,), -1.0 / B))).to(dev))
        self.buf[key] = j
        return j

    # ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def __call__(self, interaction):
        """-> (final_attacked_loss, calibrated_loss) detached 0-d tensors; gradients land in the flat grad buffer."""
        was = LIB.query('acsr_set_pdl', 1 if self.pdl else 0)
        try:
            return self._step(interaction)
        finally:
            LIB.query('acsr_set_pdl', was)

    def _step(self, interaction):
        m, opt = self.m, self.opt
        seq = interaction[m.ITEM_SEQ].contiguous()
        ln = interaction[m.ITEM_SEQ_LEN].contiguous()
        pos_items = interaction[m.POS_ITEM_ID]
        B, L = seq.shape
        dev = seq.device
        d, N, V = m.hidden_size, m.n_layers, m.n_items
        rt = m._runtime(dev)
        rng, rand = rt.rng, rt.rand
        training = m.training
        E = m.item_embedding.weight
        main = torch.cuda.current_stream()
        # (sequences longer than 64: the attention backward's workspace is one per device, so the branches would race on it)
        nb = self.n_branches if (self.n_branches > 1 and B % self.n_branches == 0 and L <= 64 and self.vp is None) else 1
        Bs = B // nb
        jb = self._joint_buffers(B, dev)
        branches = []
        for s in range(nb):
            sl = slice(s * Bs, (s + 1) * Bs)
            branches.append(dict(idx=s, sl=sl, seq=seq[sl], ln=ln[sl], buf=self._branch_buffers(Bs, L, dev, s),
                                 rand=rand if (rand is None or nb == 1) else _RandSlice(rand, sl),
                                 stream=main if s == 0 else self._stream_for(dev, ('branch', s)),
                                 side=self._stream_for(dev, ('side', s)) if self.overlap_wgrad else None))
        rng.advance()
        jb['pen'].zero_()
        torch.cat((pos_items, pos_items), out=jb['target2'])      # targets of the [calibrated ; attacked] rows: off the CE's critical path
        zero_done = None
        if training:
            # every buffer the backward accumulates into is cleared on its own stream while the forward runs
            zs = self._stream_for(dev, ('zero',))
            zs.wait_stream(main)
            with torch.cuda.stream(zs):
                opt.zero_grad()
                jb['d_out2'].zero_()
                for br in branches:
                    bb = br['buf']
                    if self._sharded():
                        self._shard_buffers(bb, dev)['d_xrows'].zero_()
                    bb['d_ctx'].zero_()
                    bb['d_x'].zero_()
                    for l, layer in enumerate(m.trm_encoder.layer):
                        if layer.combine_option == 'gate':
                            bb['layers'][l]['d_gl'].zero_()
            zero_done = torch.cuda.Event()
            zero_done.record(zs)
        # ---------------- forward: parallel branches ----------------
        for br in branches:
            if br['stream'] is not main:
                br['stream'].wait_stream(main)
            with torch.cuda.stream(br['stream']):
                self._forward_branch(br, jb, B, L, rt, training)
        for br in branches:
            if br['stream'] is not main:
                main.wait_stream(br['stream'])
        if getattr(self, '_stop_after', None) == 'fwd':      # timeline probes (scripts/step_timeline.py)
            if zero_done is not None:
                main.wait_event(zero_done)
            return jb['loss'][0], jb['loss'][0]
        # ---------------- where the sequences meet: full-catalogue cross entropy + penalty norm ----------------
        st = _stream()
        passes = m.logits_passes
        vst = None
        if self.vp is not None:       # all-gather out -> shard-local partial CE -> all-gather (max, sum-exp) -> combine
            loss2, vst = self.vp.ce_forward(jb['out2'], E, jb['target2'], 2)
            jb['loss'].copy_(loss2)
        wp = m.mask_loss_weight.detach() if m.trainable_mask_loss_weight else None
        wv = 0.0 if wp is not None else float(m.mask_loss_weight)
        bpr = m.loss_type == 'BPR'
        if bpr:
            # acsasrec.py:109-116: one sampled negative per row; rows [0,B) calibrated, [B,2B) attacked share the two kernels
            if self.vp is not None:
                raise NotImplementedError('vocab-parallel logits are a CE construct; loss_type BPR touches two table rows per sequence')
            neg_items = interaction[m.NEG_ITEM_ID]
            torch.cat((neg_items, neg_items), out=jb['neg2'])
            LIB.call('acsr_bpr_loss_fwd', _p(jb['out2']), _p(E), _p(jb['target2'], torch.int64), _p(jb['neg2'], torch.int64), 2 * B, d, 2,
                     float(m.loss_fct.gamma), _p(jb['row_x']), _p(jb['row_loss']), _p(jb['loss']), st)
            LIB.call('acsr_loss_combine', jb['pen'].data_ptr(), N, _p(jb['loss'][1:]), _p(wp), wv, _p(jb['loss_att']), _p(jb['dpen']), st)
        elif self.vp is None:
            # per-chunk (max, sum-exp) -> lse / target logit / row losses -> the two CE means -> pen_l = sqrt(sum (1-M_l)^2),
            # loss_att = -CE(attacked) + w * mean_l pen_l, d loss_att / d pen_sq_l: one single-CTA launch after the GEMM
            LIB.call('acsr_logits_ce_partial', _p(jb['out2']), _p(E), 2 * B, V, d, passes, _p(jb['partial']), st)
            LIB.call('acsr_ce_finalize_losses', _p(jb['partial']), jb['partial'].shape[1], _p(jb['out2']), _p(E),
                     _p(jb['target2'], torch.int64), 2 * B, d, V, 0, 2, _p(jb['lse']), _p(jb['tgt']), _p(jb['row_loss']),
                     _p(jb['loss']), jb['pen'].data_ptr(), N, _p(wp), wv, _p(jb['loss_att']), _p(jb['dpen']),
                     jb['ce_cnt'].data_ptr(), st)
        else:
            LIB.call('acsr_loss_combine', jb['pen'].data_ptr(), N, _p(jb['loss'][1:]), _p(wp), wv, _p(jb['loss_att']), _p(jb['dpen']), st)
        loss_cal = jb['loss'][0]
        loss_att = jb['loss_att'][0]
        self.last_losses = jb['loss3']
        if not training or getattr(self, '_stop_after', None) == 'ce':
            if zero_done is not None:
                main.wait_event(zero_done)
            return loss_att, loss_cal
        # ---------------- backward ----------------
        dpen = jb['dpen']
        main.wait_event(zero_done)
        if bpr:                       # d_out2 = +-g (E[pos] - E[neg]) / B ; the calibrated rows scatter +-g.out into dE[pos], dE[neg]
            LIB.call('acsr_bpr_loss_bwd', _p(jb['out2']), _p(E), _p(jb['target2'], torch.int64), _p(jb['neg2'], torch.int64),
                     _p(jb['row_x']), _p(jb['row_scale']), 2 * B, d, float(m.loss_fct.gamma), 0, B, _p(jb['d_out2']), _p(E.grad), st)
        elif self.vp is not None:       # shard-local G^T, reduce-scatter of d_out, dE into the owner's rows
            jb['d_out2'].copy_(self.vp.ce_backward(vst, E, jb['row_scale'], E.grad, table_half=0, n_groups=2))
        elif self.ce_fused_bwd:
            # no [2B,V] gradient matrix: the logits are recomputed tile by tile and G = (softmax - onehot) * row_scale lives in
            # registers; d_out2 += G . E on the critical path (d_out2 was cleared on the zeroing stream)
            ops.ce_bwd_dout(jb['out2'], E, jb['lse'], jb['target2'], jb['row_scale'], jb['d_out2'], passes)
        else:
            if jb['Gt'] is None:
                jb['Gt'] = torch.empty((V, 2 * B), dtype=torch.float32, device=dev)
            LIB.call('acsr_logits_ce_grad', _p(jb['out2']), _p(E), _p(jb['lse']), _p(jb['target2'], torch.int64),
                     _p(jb['row_scale']), 2 * B, V, d, passes, _p(jb['Gt']), 2 * B, st)
            # d_out2 [2B,d] += Gt^T . E : contraction over the catalogue, split over the CTAs
            ops.gemm_batch([ops.wgrad_problem(jb['Gt'], E, V, 2 * B, d, jb['d_out2'])])
        for br in branches:
            if br['stream'] is not main:
                br['stream'].wait_stream(main)
        if self.vp is None and not bpr:
            # dE += Gt[:, :B] . out[:B]: only the calibrated rows train the item table.  It reads and writes dE without
            # atomics, so every branch's embedding scatter waits for it (dE_done).  Nothing else consumes it: with a single
            # branch it runs on that branch's weight-gradient stream.
            dE_stream = branches[0]['side'] if (nb == 1 and branches[0]['side'] is not None) else main
            if dE_stream is not main:
                dE_stream.wait_stream(main)
            with torch.cuda.stream(dE_stream):
                if self.ce_fused_bwd:     # dE += G[:B]^T . out[:B], G recomputed (table rows on the UMMA M axis)
                    ops.ce_bwd_dtable(jb['out2'][:B], E, jb['lse'][:B], jb['target2'][:B], jb['row_scale'][:B], E.grad, passes)
                else:                  # dE [V,d] += Gt[:, :B] . out[:B]  (rows of the table on the M axis, K = B)
                    ops.gemm_batch([ops.gemm_problem(jb['Gt'], jb['out2'], E.grad, V, d, B, a_strides=(2 * B, 1, 0, B),
                                                     b_strides=(1, d, 0, B), accumulate=True)])
        else:
            dE_stream = main
        dE_done = torch.cuda.Event()
        dE_done.record(dE_stream)
        for br in branches:
            with torch.cuda.stream(br['stream']):
                self._backward_branch(br, jb, B, L, rt, dpen, dE_done)
        for br in branches:
            if br['stream'] is not main:
                main.wait_stream(br['stream'])
        return loss_att, loss_cal

    # ------------------------------------------------------------------------------------------
    def _forward_branch(self, br, jb, B, L, rt, training, need_att=True):
        m = self.m
        b, seq, ln, s = br['buf'], br['seq'], br['ln'], br['idx']
        Bs = seq.shape[0]
        T, d, I, N, V, H = b['T'], m.hidden_size, m.inner_size, m.n_layers, m.n_items, m.n_heads
        dh = d // H
        rng, rand = rt.rng, br['rand']
        rngp = rng.ptr
        st = _stream()
        p_h = m.dropout.p if training else 0.0
        soff = 4096 * s                                           # Philox stream ids of this branch

        def mask(key):
            return None if (rand is None or p_h == 0.0) else rand.get(key)

        def mask2(l, k_cal, k_att, last):
            if rand is None or p_h == 0.0:
                return None
            a = rand.get((l, k_cal))
            return torch.cat((a.reshape(T, d), rand.get((l, k_att)).reshape(T, d))) if last else a

        E = m.item_embedding.weight
        posw = m.position_embedding.weight if m.use_position_embedding else None
        b['me'] = mask('emb')
        # longest sequences first: order of the attention CTAs of this batch (forward and backward).  Only the attention
        # kernels read it, so the single-CTA sort runs next to the embedding and the first projections, not in front of them.
        cur = torch.cuda.current_stream()
        so = self._stream_for(seq.device, ('order', s))
        so.wait_stream(cur)
        folded = {}
        if self.tc:                                       # first on the side stream: the first projection launch needs layer 0's
            for l in range(N):
                st3 = self._stacked(l)
                if st3 is None:
                    continue
                fw = self._folded_buffers(l, seq.device)
                LIB.call('acsr_fold_attack_weights', _p(st3['Wqkv']), _p(st3['bqkv']), _p(st3['Waqk']), _p(st3['baqk']), d,
                         _p(fw['W']), _p(fw['b']), so.cuda_stream)
                fw['done'] = torch.cuda.Event()
                fw['done'].record(so)
                folded[l] = fw
        bwd_ops = {}
        if self.dense_bwd and training:
            # the layers' dense weights transposed for acsr_dense_bwd (the last layer's dense part runs on the compact rows, see
            # acsr_tail_bwd).  Enqueued ahead of the sequence ordering, whose event the first attention launch waits for: complete
            # before any backward kernel starts (and static for its PDL chain)
            for l in range(N - 1):
                lay = m.trm_encoder.layer[l]
                dbuf = self._dense_bwd_ops_buffer(l, s, seq.device)
                LIB.call('acsr_dense_bwd_prep', _p(lay.attack_attention.dense.weight), _p(lay.feed_forward.dense_1.weight),
                         _p(lay.feed_forward.dense_2.weight), d, I, _p(dbuf), so.cuda_stream)
                bwd_ops[l] = dbuf
        b['dense_bwd_ops'] = bwd_ops
        LIB.call('acsr_seq_order', _p(seq, torch.int64), Bs, L, _p(b['order'], torch.int32), so.cuda_stream)
        order_done = torch.cuda.Event()
        order_done.record(so)
        if self._sharded():
            # the table rows of my tokens live on their owners: ids all-gathered, owners answer, reduce-scatter delivers (dist.py).
            # The rows land in xrows[1:], and the kernel gathers row t+1 for token t (ids 1..T: no token looks like padding)
            sb = self._shard_buffers(b, seq.device)
            _, b['ids_all'] = self.vp.fetch_rows(seq.reshape(-1), E, out=sb['xrows'][1:])
            LIB.call('acsr_embed_ln_dropout_fwd', _p(sb['iota1'], torch.int64), _p(sb['xrows']), _p(posw), _p(m.LayerNorm.weight),
                     _p(m.LayerNorm.bias), m.LayerNorm.eps, T, L, d, T + 1, p_h, _p(b['me']), rngp, soff + 1, _p(b['x0']), _p(b['st_e']), st)
        else:
            LIB.call('acsr_embed_ln_dropout_fwd', _p(seq, torch.int64), _p(E), _p(posw), _p(m.LayerNorm.weight), _p(m.LayerNorm.bias),
                     m.LayerNorm.eps, T, L, d, V, p_h, _p(b['me']), rngp, soff + 1, _p(b['x0']), _p(b['st_e']), st)
        x = b['x0']
        b['xs'] = []
        act_id = ops.ACT_IDS[m.hidden_act]
        for l, layer in enumerate(m.trm_encoder.layer):
            last = l == N - 1 and need_att                 # the attacked branch only matters on the last layer (and not in eval)
            lb = b['layers'][l]
            aa, ff = layer.attack_attention, layer.feed_forward
            base = soff + 16 * (l + 1)
            b['xs'].append(x)
            fw = folded.get(l)
            if fw is not None:
                # all five projections read x: one batched tcgen05 launch over the folded weights (prepared at the start of the
                # step on the ordering stream, next to the embedding kernel)
                cur.wait_event(fw['done'])
                ops.linear_tok(x, T, d, fw['W'], d, lb['qkv5'], d, bias=fw['b'], batch=5, sx=0, sw=d * d, sb=d, sy=T * d)
            else:
                # any width: Q / K / V in one launch of the K-streamed tcgen05 kernel, then the attack pair (+ the gate logits,
                # which read mixed_q as well) in a second one
                gp = ops.gemm_problem
                ops.gemm_batch([gp(x, lin.weight, lb[k], T, d, d, bias=lin.bias)
                                for lin, k in ((aa.query, 'mq'), (aa.key, 'mk'), (aa.value, 'mv'))], passes=self.passes)
                second = [gp(lb['mq'], aa.attack_query_transform.weight, lb['aq'], T, d, d, bias=aa.attack_query_transform.bias),
                          gp(lb['mk'], aa.attack_key_transform.weight, lb['ak'], T, d, d, bias=aa.attack_key_transform.bias)]
                if layer.combine_option == 'gate' and not self.tc:
                    if layer.gate.out_features != L:
                        raise ValueError('gate width %d != sequence length %d' % (layer.gate.out_features, L))
                    second.append(gp(lb['mq'], layer.gate.weight, lb['gl'], T, L, d, bias=layer.gate.bias))
                ops.gemm_batch(second, passes=self.passes)
            gate = layer.combine_option == 'gate'
            comb_scalar = 0.0
            if gate:
                if layer.gate.out_features != L:
                    raise ValueError('gate width %d != sequence length %d' % (layer.gate.out_features, L))
                if self.tc:
                    ops.linear_tok(lb['mq'], T, d, layer.gate.weight, L, lb['gl'], L, bias=layer.gate.bias)
            elif layer.combine_option == 'annealing':
                comb_scalar = math.exp(-layer.anneal_step / 100000)
                if s == 0:
                    layer.anneal_step += 1
            p_attn = aa.attn_dropout.p if training else 0.0
            lb['attn_args'] = self._attn_args(layer, lb, seq, Bs, L, H, dh, comb_scalar, p_attn, rand, l, rngp, base)
            ctx_cal, ctx_att = lb['ctx'][:T], (lb['ctx'][T:] if last else None)
            if l == 0:
                cur.wait_event(order_done)         # sequence order (side stream) is ready
            LIB.call('acsr_attn_calib_fwd', *lb['attn_args'], _p(ctx_att), _p(ctx_cal),
                     jb['pen'][l:].data_ptr() if need_att else None, None, _p(b['order'], torch.int32),
                     _p(ln, torch.int64) if l == N - 1 else None, st)
            m_a, m_f = mask2(l, 'D5', 'D4', last), mask2(l, 'D7', 'D6', last)
            if l == N - 1:
                # ---- last layer: gather position len-1 of every sequence, then the dense part on the compact rows ----
                cb = b['c']
                C = 2 * Bs if need_att else Bs
                if m_a is not None or m_f is not None:           # explicit masks of a parity test: the same rows
                    idx = torch.arange(Bs, device=seq.device) * L + ln - 1
                    rows = torch.cat((idx, T + idx)) if need_att else idx
                    m_a = None if m_a is None else m_a.reshape(-1, d)[rows].contiguous()
                    m_f = None if m_f is None else m_f.reshape(-1, d)[rows].contiguous()
                cb['m_a'], cb['m_f'] = m_a, m_f
                out_buf = jb['out2'] if Bs == B else cb['out']   # a single branch writes the joint buffer directly
                if self.tail_fused:
                    # gather + out-projection + LayerNorm + feed-forward + LayerNorm of the 2*Bs rows: one launch
                    LIB.call('acsr_tail_fwd', _p(lb['ctx'][:T]), _p(lb['ctx'][T:]) if need_att else None, _p(x), _p(ln, torch.int64),
                             Bs, L, d, I, act_id, _p(aa.dense.weight), _p(aa.dense.bias), _p(aa.LayerNorm.weight), _p(aa.LayerNorm.bias),
                             aa.LayerNorm.eps, _p(ff.dense_1.weight), _p(ff.dense_1.bias), _p(ff.dense_2.weight), _p(ff.dense_2.bias),
                             _p(ff.LayerNorm.weight), _p(ff.LayerNorm.bias), ff.LayerNorm.eps, p_h, _p(m_a), _p(m_f), rngp, base + 3,
                             base + 5, _p(cb['ctx']), _p(cb['x']), _p(cb['hz']), _p(cb['st_a']), _p(cb['h']), _p(cb['z1']), _p(cb['a1']),
                             _p(cb['z2']), _p(cb['st_f']), _p(out_buf), st)
                else:
                    LIB.call('acsr_gather_last_fwd', _p(lb['ctx'][:T]) if need_att else None, _p(lb['ctx'][T:] if need_att else lb['ctx'][:T]),
                             _p(ln, torch.int64), Bs, L, d, _p(cb['ctx']), st)
                    LIB.call('acsr_gather_last_fwd', None, _p(x), _p(ln, torch.int64), Bs, L, d, _p(cb['x']), st)
                    self._post_attn_fwd(layer, cb, cb['x'], Bs, C, out_buf, p_h, rngp, base, act_id, st)
                if Bs != B:
                    lo = br['sl'].start
                    jb['out2'][lo:lo + Bs].copy_(cb['out'][:Bs])
                    if need_att:
                        jb['out2'][B + lo:B + lo + Bs].copy_(cb['out'][Bs:C])
                return
            lb['m_a'], lb['m_f'] = m_a, m_f
            self._post_attn_fwd(layer, lb, x, T, T, lb['out'], p_h, rngp, base, act_id, st)
            x = lb['out']

    def _post_attn_fwd(self, layer, bf, x_res, res_rows, R, out, p_h, rngp, base, act_id, st):
        """out-projection + dropout + residual + LayerNorm, then the feed-forward block, on R rows of bf['ctx']
        (layers.py:676-684, 790-798).  x_res [res_rows, d] is the layer input (residual)."""
        m = self.m
        d, I = m.hidden_size, m.inner_size
        aa, ff = layer.attack_attention, layer.feed_forward
        if self.tc:
            # out-projection + bias + dropout + residual + LayerNorm in one kernel; FFN: GEMM, bias + activation, then
            # GEMM + bias + dropout + residual + LayerNorm
            ops.linear_tok_bdrl(bf['ctx'], R, d, aa.dense.weight, aa.dense.bias, x_res, res_rows, aa.LayerNorm.weight,
                                aa.LayerNorm.bias, aa.LayerNorm.eps, p_h, bf['m_a'], rngp, base + 3, bf['hz'], bf['h'], bf['st_a'])
            # (a bias + activation epilogue on the GEMM measured slower at I=256: four epilogue warps cannot hide the erf latency)
            ops.linear_tok(bf['h'], R, d, ff.dense_1.weight, I, bf['z1'], I)
            LIB.call('acsr_bias_act_fwd', _p(bf['z1']), _p(ff.dense_1.bias), R, I, act_id, _p(bf['a1']), st)
            ops.linear_tok_bdrl(bf['a1'], R, I, ff.dense_2.weight, ff.dense_2.bias, bf['h'], R, ff.LayerNorm.weight,
                                ff.LayerNorm.bias, ff.LayerNorm.eps, p_h, bf['m_f'], rngp, base + 5, bf['z2'], out, bf['st_f'])
        else:
            # any width: three launches of the K-streamed tcgen05 kernel, everything that follows a GEMM in the reference fused
            # into its TMEM epilogue (bias + dropout + residual + LayerNorm; bias + activation)
            gp, ps = ops.gemm_problem, self.passes
            ops.gemm_batch([gp(bf['ctx'], aa.dense.weight, bf['hz'], R, d, d, bias=aa.dense.bias, epilogue=ops.EPI_BDRL, res=x_res,
                               res_rows=res_rows, ln_w=aa.LayerNorm.weight, ln_b=aa.LayerNorm.bias, eps=aa.LayerNorm.eps, p_drop=p_h,
                               mask=bf['m_a'], rngp=rngp, rng_stream=base + 3, out=bf['h'], stats=bf['st_a'])], passes=ps)
            ops.gemm_batch([gp(bf['h'], ff.dense_1.weight, bf['z1'], R, I, d, bias=ff.dense_1.bias, epilogue=ops.EPI_ACT, act=act_id,
                               C2=bf['a1'])], passes=ps)
            ops.gemm_batch([gp(bf['a1'], ff.dense_2.weight, bf['z2'], R, d, I, bias=ff.dense_2.bias, epilogue=ops.EPI_BDRL, res=bf['h'],
                               res_rows=R, ln_w=ff.LayerNorm.weight, ln_b=ff.LayerNorm.bias, eps=ff.LayerNorm.eps, p_drop=p_h,
                               mask=bf['m_f'], rngp=rngp, rng_stream=base + 5, out=out, stats=bf['st_f'])], passes=ps)

    @torch.no_grad()
    def encode_eval(self, item_seq, item_seq_len):
        """calibrated last-position outputs [B,d] of an eval batch through the fused forward (no attacked branch, no
        dropout, no saved-for-backward traffic beyond the reused buffers): ACSASRec.forward for full_sort_predict."""
        m = self.m
        seq, ln = item_seq.contiguous(), item_seq_len.contiguous()
        B, L = seq.shape
        dev = seq.device
        rt = m._runtime(dev)
        jb = self._joint_buffers(B, dev)
        br = dict(idx=0, sl=slice(0, B), seq=seq, ln=ln, buf=self._branch_buffers(B, L, dev, 'eval', grads=False), rand=rt.rand,
                  stream=torch.cuda.current_stream(), side=None)
        jb['pen'].zero_()
        self._forward_branch(br, jb, B, L, rt, False, need_att=False)
        return jb['out2'][:B]

    # ------------------------------------------------------------------------------------------
    def _backward_branch(self, br, jb, B, L, rt, dpen, dE_done):
        m = self.m
        b, seq, ln, s = br['buf'], br['seq'], br['ln'], br['idx']
        Bs = seq.shape[0]
        T, d, I, N, V = b['T'], m.hidden_size, m.inner_size, m.n_layers, m.n_items
        rngp = rt.rng.ptr
        st = _stream()
        main = torch.cuda.current_stream()
        side = br['side']
        p_h = m.dropout.p
        soff = 4096 * s
        act_id = ops.ACT_IDS[m.hidden_act]
        E = m.item_embedding.weight
        posw = m.position_embedding.weight if m.use_position_embedding else None

        def fork():
            """-> stream handle for a weight-gradient launch: the side stream, ordered after everything enqueued so far"""
            if side is None:
                return st
            side.wait_stream(main)
            return side.cuda_stream

        d_out, d_x = b['d_out'], b['d_x']
        lo = br['sl'].start
        T2 = 2 * T
        for l in reversed(range(N)):
            last = l == N - 1
            lb = b['layers'][l]
            layer = m.trm_encoder.layer[l]
            aa, ff = layer.attack_attention, layer.feed_forward
            base = soff + 16 * (l + 1)
            x = b['xs'][l]
            gate = layer.combine_option == 'gate'
            wg = []                                          # weight-gradient problems of this layer (one launch at its end)
            if last:
                # the dense part of the last layer on the 2*Bs rows that carry a cotangent, then scatter into the zeroed
                # token-major buffers the attention backward (d_ctx) and the layer below (residual path, d_x) read
                cb = b['c']
                C = 2 * Bs
                if Bs == B:
                    dc_out = jb['d_out2']
                else:
                    dc_out = cb['d_out']
                    dc_out[:Bs].copy_(jb['d_out2'][lo:lo + Bs])
                    dc_out[Bs:].copy_(jb['d_out2'][B + lo:B + lo + Bs])
                if self.tail_fused:
                    g = lambda t: _p(t.grad)     # noqa: E731
                    LIB.call('acsr_tail_bwd', _p(dc_out), _p(ln, torch.int64), Bs, L, d, I, act_id, 2, _p(cb['x']), _p(cb['hz']),
                             _p(cb['st_a']), _p(cb['h']), _p(cb['z1']), _p(cb['z2']), _p(cb['st_f']), _p(aa.dense.weight), _p(aa.dense.bias),
                             _p(aa.LayerNorm.weight), _p(ff.dense_1.weight), _p(ff.dense_1.bias), _p(ff.dense_2.weight),
                             _p(ff.dense_2.bias), _p(ff.LayerNorm.weight), p_h, _p(cb['m_a']), _p(cb['m_f']), rngp, base + 3, base + 5,
                             _p(cb['d_z2']), _p(cb['d_z1']), _p(cb['d_hz']), _p(d_x[:T]), _p(d_x[T:]), _p(b['d_ctx'][:T]),
                             _p(b['d_ctx'][T:]), g(aa.dense.bias), g(aa.LayerNorm.weight), g(aa.LayerNorm.bias), g(ff.dense_1.bias),
                             g(ff.dense_2.bias), g(ff.LayerNorm.weight), g(ff.LayerNorm.bias), st)
                    self._wgrad(cb['d_z2'], cb['a1'], Bs, ff.dense_2.weight.grad, None, wg)
                    self._wgrad(cb['d_z1'], cb['h'], Bs, ff.dense_1.weight.grad, None, wg)
                    self._wgrad(cb['d_hz'], cb['ctx'], Bs, aa.dense.weight.grad, None, wg)
                else:
                    self._post_attn_bwd(layer, cb, cb, dc_out, cb['x'], C, C, Bs, Bs, cb['d_x'], cb['d_ctx'], p_h, rngp, base, act_id, st, wg)
                    LIB.call('acsr_gather_last_bwd', _p(cb['d_ctx']), _p(ln, torch.int64), Bs, L, d, _p(b['d_ctx'][:T]), _p(b['d_ctx'][T:]), st)
                    LIB.call('acsr_gather_last_bwd', _p(cb['d_x']), _p(ln, torch.int64), Bs, L, d, _p(d_x[:T]), _p(d_x[T:]), st)
            else:
                self._post_attn_bwd(layer, lb, lb, d_out, x, T2, T, T, T, d_x, b['d_ctx'], p_h, rngp, base, act_id, st, wg, b=b,
                                    dops=b['dense_bwd_ops'].get(l))
            if wg and l == 0:
                # the out-projection / feed-forward weight gradients are complete here: their launch runs on the side stream
                # under the attention backward, so the launch left for the end of the layer (the projections') is short --
                # the first layer's is the tail of the step's critical path
                ops.gemm_batch(wg, passes=self.passes, stream=fork())
                wg = []
            # fused attention backward (d_gate_logit accumulates over heads: cleared at the start of the step)
            g = lambda t: None if t is None else t.grad     # noqa: E731
            ow, ob_ = (aa.order_affine.weight, aa.order_affine.bias) if aa.use_order else (None, None)
            dw, db_, sc = (aa.distance_affine.weight, aa.distance_affine.bias, aa.scalar) if aa.use_distance else (None, None, None)
            rr = getattr(layer, 'rich_calibrated_combine_ratio', None) if not layer.two_level else None
            dc = b['d_ctx']
            # both cotangent streams in one launch: stream 0 = d(calibrated loss), stream 1 = d(attacked loss) which
            # enters through the attacked context on the last layer, through the calibrated chain below, plus the penalty
            d_att1, d_cal1 = (dc[T:], None) if last else (None, dc[T:])
            ops.attn_workspace(Bs, L, m.n_heads, 2, seq.device)          # only sequences longer than 64 need one
            LIB.call('acsr_attn_calib_bwd2', _p(dc[:T]), None, _p(d_att1), _p(d_cal1), _p(dpen[l:l + 1]), *lb['attn_args'],
                     _p(lb['d_mq']), _p(lb['d_mk']), _p(lb['d_mv']), _p(lb['d_aq']), _p(lb['d_ak']),
                     _p(lb['d_gl']) if gate else None, _p(g(ow)), _p(g(ob_)), _p(g(dw)), _p(g(db_)), _p(g(sc)), _p(g(rr)),
                     _p(b['order'], torch.int32), _p(ln, torch.int64) if last else None, st)
            # projections: input gradients for both streams, weight gradients from the owning stream
            aqt, akt = aa.attack_query_transform, aa.attack_key_transform
            # weight gradients of the projections: attack transforms are trained by the attacked-loss stream (rows [T,2T)), the
            # gate by both halves of d_gl's stream-0 rows, Q / K / V by the calibrated-loss stream.  (A third launch for the attack pair
            # + gate, whose operands are final right after the attention backward, measured no further gain: 0.7162 vs 0.7179 ms.)
            self._wgrad(lb['d_aq'][T:], lb['mq'], T, aqt.weight.grad, aqt.bias.grad, wg)
            self._wgrad(lb['d_ak'][T:], lb['mk'], T, akt.weight.grad, akt.bias.grad, wg)
            if gate:
                self._wgrad(lb['d_gl'], lb['mq'], T, layer.gate.weight.grad, layer.gate.bias.grad, wg)

            st3 = self._stacked(l)
            gp = ops.gemm_problem
            rows_x = T2 if l > 0 else T                      # below the first layer only the calibrated stream trains anything
            if self.tc and st3 is not None and (not gate or L <= d):
                # d_mq += d_aq.Waq (+ d_gl.Wg), d_mk += d_ak.Wak, d_x += [d_mq d_mk d_mv] . [Wq; Wk; Wv]: one launch.  Only rows
                # [0,T) of the summed d_mq / d_mk are read afterwards (the Q / K weight gradients): the kernel writes back those.
                LIB.call('acsr_proj_input_grad', _p(lb['d_qkv']), _p(lb['d_aqk']), T2, _p(lb['d_gl']) if gate else None, L,
                         _p(st3['Wqkv']), _p(st3['Waqk']), _p(layer.gate.weight) if gate else None, d, rows_x, T, _p(d_x),
                         self.passes, st)
            else:
                # any width, or a gate wider than the hidden size (K-streamed tcgen05 kernel): d_mq += d_aq.Waq, d_mk += d_ak.Wak in
                # one launch; the gate's d_mq += d_gl.Wg accumulates into the same rows, so it follows in its own launch; then d_x +=
                # sum of the three projections
                ops.gemm_batch([gp(lb['d_aq'], aqt.weight, lb['d_mq'], T2, d, d, b_strides=(1, d, 0, d), accumulate=True),
                                gp(lb['d_ak'], akt.weight, lb['d_mk'], T2, d, d, b_strides=(1, d, 0, d), accumulate=True)],
                               passes=self.passes)
                if gate:
                    ops.gemm_batch([gp(lb['d_gl'], layer.gate.weight, lb['d_mq'], T2, d, L, b_strides=(1, d, 0, L), accumulate=True)],
                                   passes=self.passes)
                if st3 is not None:                          # K-concatenated: [d_mq d_mk d_mv] . [Wq; Wk; Wv]
                    ops.gemm_batch([gp(lb['d_qkv'], st3['Wqkv'], d_x, rows_x, d, 3 * d, a_strides=(d, 1, T2 * d, d),
                                       b_strides=(1, d, d * d, d), accumulate=True)], passes=self.passes)
                else:
                    for lin, dk in ((aa.query, 'd_mq'), (aa.key, 'd_mk'), (aa.value, 'd_mv')):
                        ops.gemm_batch([gp(lb[dk], lin.weight, d_x, rows_x, d, d, b_strides=(1, d, 0, d), accumulate=True)],
                                       passes=self.passes)
            for lin, dk in ((aa.query, 'd_mq'), (aa.key, 'd_mk'), (aa.value, 'd_mv')):
                self._wgrad(lb[dk], x, T, lin.weight.grad, lin.bias.grad, wg)
            if wg:                                           # all weight gradients of the layer: ONE launch on the side stream
                ops.gemm_batch(wg, passes=self.passes, stream=fork())
            if l > 0:
                d_out, d_x = d_x, d_out                       # this layer's input gradient is the next one's output gradient
        main.wait_event(dE_done)                              # the dE GEMM is a plain read-modify-write of the table gradient
        if self._sharded():
            # per-token gradient rows (LayerNorm backward), then home to the owners of the table rows (padding id 0 gets none)
            sb = self._shard_buffers(b, seq.device)
            LIB.call('acsr_embed_ln_dropout_bwd', _p(d_x[:T]), _p(sb['iota1'], torch.int64), _p(sb['xrows']), _p(posw), _p(m.LayerNorm.weight),
                     _p(b['st_e']), T, L, d, T + 1, p_h, _p(b['me']), rngp, soff + 1, _p(sb['d_xrows']),
                     _p(posw.grad if posw is not None else None), _p(m.LayerNorm.weight.grad), _p(m.LayerNorm.bias.grad), st)
            self.vp.scatter_grad_rows(b['ids_all'], sb['d_xrows'][1:], E.grad)
        else:
            LIB.call('acsr_embed_ln_dropout_bwd', _p(d_x[:T]), _p(seq, torch.int64), _p(E), _p(posw), _p(m.LayerNorm.weight),
                     _p(b['st_e']), T, L, d, V, p_h, _p(b['me']), rngp, soff + 1, _p(E.grad), _p(posw.grad if posw is not None else None),
                     _p(m.LayerNorm.weight.grad), _p(m.LayerNorm.bias.grad), st)
        if side is not None:
            main.wait_stream(side)                            # join: every weight gradient of this branch landed

    def _post_attn_bwd(self, layer, bf, gb, d_out, x_res, R2, P, res_rows, w_rows, d_xres, d_ctx, p_h, rngp, base, act_id, st, wg, b=None,
                       dops=None):
        """backward of _post_attn_fwd over R2 cotangent rows ([stream 0 ; stream 1]); the saved forward tensors of bf repeat
        with period P, the residual x_res with period res_rows; rows [0, w_rows) (stream 0) feed the parameter gradients.
        Writes the gradient of the attention context to d_ctx and of the residual input to d_xres; weight-gradient problems
        are appended to wg (launched together at the end of the layer).  dops: the layer's weights prepared by acsr_dense_bwd_prep
        (the whole chain as one launch)."""
        m = self.m
        d, I = m.hidden_size, m.inner_size
        aa, ff = layer.attack_attention, layer.feed_forward
        if dops is not None:
            # only rows [0, w_rows) of d_z2 / d_z1 / d_hz leave the SM; the three bias gradients are their column sums, taken by
            # the weight-gradient launch
            LIB.call('acsr_dense_bwd', _p(d_out), R2, P, res_rows, w_rows, d, I, act_id, _p(dops), _p(bf['z2']), _p(ff.dense_2.bias),
                     _p(bf['h']), _p(ff.LayerNorm.weight), _p(bf['st_f']), _p(bf['z1']), _p(ff.dense_1.bias), _p(bf['hz']),
                     _p(aa.dense.bias), _p(x_res), _p(aa.LayerNorm.weight), _p(bf['st_a']), p_h, _p(bf['m_a']), _p(bf['m_f']), rngp,
                     base + 3, base + 5, _p(gb['d_z2']), _p(gb['d_z1']), _p(gb['d_hz']), _p(d_xres), _p(d_ctx),
                     _p(ff.LayerNorm.weight.grad), _p(ff.LayerNorm.bias.grad), _p(aa.LayerNorm.weight.grad),
                     _p(aa.LayerNorm.bias.grad), self.passes, st)
            self._wgrad(gb['d_z2'], bf['a1'], w_rows, ff.dense_2.weight.grad, ff.dense_2.bias.grad, wg)
            self._wgrad(gb['d_z1'], bf['h'], w_rows, ff.dense_1.weight.grad, ff.dense_1.bias.grad, wg)
            self._wgrad(gb['d_hz'], bf['ctx'], w_rows, aa.dense.weight.grad, aa.dense.bias.grad, wg)
            return
        d_h = gb['d_h'] if b is None else b['d_h']
        d_a1 = gb['d_a1'] if b is None else b['d_a1']
        gp, ps = ops.gemm_problem, self.passes
        # FFN
        LIB.call('acsr_bias_dropout_res_ln_bwd', _p(d_out), _p(bf['z2']), _p(ff.dense_2.bias), _p(bf['h']),
                 _p(ff.LayerNorm.weight), _p(bf['st_f']), R2, d, P, P, w_rows, p_h, _p(bf['m_f']), rngp, base + 5,
                 _p(gb['d_z2']), _p(d_h), _p(ff.dense_2.bias.grad), _p(ff.LayerNorm.weight.grad),
                 _p(ff.LayerNorm.bias.grad), st)
        self._wgrad(gb['d_z2'], bf['a1'], w_rows, ff.dense_2.weight.grad, None, wg)
        if self.tc:                                          # d_a1 = d_z2.W2 : the weight is read transposed
            ops.linear_tok(gb['d_z2'], R2, d, ff.dense_2.weight, I, d_a1, I, w_sn=1, w_sk=I, wkb=64 * I)
        else:
            ops.gemm_batch([gp(gb['d_z2'], ff.dense_2.weight, d_a1, R2, I, d, b_strides=(1, I, 0, d))], passes=ps)
        LIB.call('acsr_bias_act_bwd', _p(d_a1), _p(bf['z1']), _p(ff.dense_1.bias), R2, I, act_id, P, w_rows, _p(gb['d_z1']),
                 _p(ff.dense_1.bias.grad), st)
        self._wgrad(gb['d_z1'], bf['h'], w_rows, ff.dense_1.weight.grad, None, wg)
        if self.tc:
            ops.linear_tok(gb['d_z1'], R2, I, ff.dense_1.weight, d, d_h, d, w_sn=1, w_sk=d, wkb=64 * d, accumulate=True)
        else:
            ops.gemm_batch([gp(gb['d_z1'], ff.dense_1.weight, d_h, R2, d, I, b_strides=(1, d, 0, I), accumulate=True)], passes=ps)
        # attention output projection
        LIB.call('acsr_bias_dropout_res_ln_bwd', _p(d_h), _p(bf['hz']), _p(aa.dense.bias), _p(x_res),
                 _p(aa.LayerNorm.weight), _p(bf['st_a']), R2, d, P, res_rows, w_rows, p_h, _p(bf['m_a']), rngp, base + 3,
                 _p(gb['d_hz']), _p(d_xres), _p(aa.dense.bias.grad), _p(aa.LayerNorm.weight.grad), _p(aa.LayerNorm.bias.grad), st)
        self._wgrad(gb['d_hz'], bf['ctx'], w_rows, aa.dense.weight.grad, None, wg)
        if self.tc:
            ops.linear_tok(gb['d_hz'], R2, d, aa.dense.weight, d, d_ctx, d, w_sn=1, w_sk=d, wkb=64 * d)
        else:
            ops.gemm_batch([gp(gb['d_hz'], aa.dense.weight, d_ctx, R2, d, d, b_strides=(1, d, 0, d))], passes=ps)

    @staticmethod
    def _wgrad(dY, X, rows, dW, db, wg):
        """weight-gradient reduction dW [N,K] += dY[:rows]^T . X[:rows] (+ db += column sums): a problem of the layer's single
        tcgen05 launch (gemm_ks.cu, token axis on K, split over the CTAs)."""
        wg.append(ops.wgrad_problem(dY, X, rows, dY.shape[-1], X.shape[-1], dW, db))

    def _sharded(self):
        return self.vp is not None and self.vp.sharded

    def _shard_buffers(self, b, dev):
        """buffers of the sharded-table row exchange of one branch: fetched rows / their gradients (row 0 unused), ids 1..T"""
        if 'shard' not in b:
            T, d = b['T'], self.m.hidden_size
            b['shard'] = dict(xrows=torch.zeros((T + 1, d), dtype=torch.float32, device=dev),
                              d_xrows=torch.zeros((T + 1, d), dtype=torch.float32, device=dev),
                              iota1=torch.arange(1, T + 1, dtype=torch.int64, device=dev))
        return b['shard']

    def _folded_buffers(self, l, dev):
        key = ('folded', l)
        if key not in self.buf:
            d = self.m.hidden_size
            self.buf[key] = dict(W=torch.zeros((5, d, d), dtype=torch.float32, device=dev), b=torch.zeros((5, 1, d), dtype=torch.float32, device=dev))
            # written once per step by acsr_fold_attack_weights, which completes (full event dependency) before the first kernel
            # of the chain that reads them starts: safe to read ahead of programmatic-launch synchronisation
            for t in list(self.buf[key].values()):
                LIB.query('acsr_register_static', t.data_ptr(), t.numel() * 4)
        return self.buf[key]

    def _dense_bwd_ops_buffer(self, l, s, dev):
        key = ('dense_bwd_ops', l, s)
        if key not in self.buf:
            t = torch.empty(LIB.query('acsr_dense_bwd_prep_floats', int(self.m.inner_size)), dtype=torch.float32, device=dev)
            # written once per step by acsr_dense_bwd_prep, complete before its reader starts: static for the PDL chain
            LIB.query('acsr_register_static', t.data_ptr(), t.numel() * 4)
            self.buf[key] = t
        return self.buf[key]

    def _stacked(self, l):
        """stacked views [3,d,d]/[2,d,d] of the Q/K/V and attack-pair parameters (adjacent in FlatAdam's layout)."""
        if not hasattr(self, '_st'):
            self._st = {}
        if l not in self._st:
            aa = self.m.trm_encoder.layer[l].attack_attention
            opt = self.opt
            if not hasattr(opt, 'stacked'):
                self._st[l] = None
            else:
                qkv_w, qkv_b = [aa.query.weight, aa.key.weight, aa.value.weight], [aa.query.bias, aa.key.bias, aa.value.bias]
                aqk_w = [aa.attack_query_transform.weight, aa.attack_key_transform.weight]
                aqk_b = [aa.attack_query_transform.bias, aa.attack_key_transform.bias]
                v = dict(Wqkv=opt.stacked(qkv_w), bqkv=opt.stacked(qkv_b), Waqk=opt.stacked(aqk_w), baqk=opt.stacked(aqk_b),
                         gWqkv=opt.stacked(qkv_w, True), gbqkv=opt.stacked(qkv_b, True), gWaqk=opt.stacked(aqk_w, True),
                         gbaqk=opt.stacked(aqk_b, True))
                if any(t is None for t in v.values()):
                    self._st[l] = None
                else:
                    v['bqkv'] = v['bqkv'].unsqueeze(1)
                    v['baqk'] = v['baqk'].unsqueeze(1)
                    self._st[l] = v
        return self._st[l]

    @staticmethod
    def _attn_args(layer, lb, seq, B, L, H, dh, comb_scalar, p_attn, rand, l, rngp, base):
        """positional arguments shared by acsr_attn_calib_fwd / _bwd between the cotangents and the outputs."""
        aa = layer.attack_attention
        r = (lambda k: None) if (rand is None) else (lambda k: rand.get((l, k)))
        drop = p_attn > 0.0
        D1, D2, D3 = (r('D1'), r('D2'), r('D3')) if drop else (None, None, None)
        lb['_keep'] = (D1, D2, D3, r('noise'))              # keep explicit tensors alive until the backward ran
        two_level = int(bool(layer.two_level))
        rich = ops.RICH_IDS.get(layer.rich_calibrated_combine, 0) if not layer.two_level else 0
        rr = getattr(layer, 'rich_calibrated_combine_ratio', None) if not layer.two_level else None
        return (_p(lb['mq']), _p(lb['mk']), _p(lb['mv']), _p(lb['aq']), _p(lb['ak']),
                _p(lb['gl']) if layer.combine_option == 'gate' else None, _p(seq, torch.int64),
                _p(aa.order_affine.weight) if aa.use_order else None, _p(aa.order_affine.bias) if aa.use_order else None,
                _p(aa.distance_affine.weight) if aa.use_distance else None, _p(aa.distance_affine.bias) if aa.use_distance else None,
                _p(aa.scalar) if aa.use_distance else None,
                B, L, H, dh, two_level, ops.COMBINE_IDS[layer.combine_option], float(comb_scalar), rich, _p(rr),
                float(p_attn), _p(D1), _p(D2), _p(D3), _p(lb['_keep'][3]), rngp, base)
