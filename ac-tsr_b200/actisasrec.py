"""ACTiSASRec -- drop-in for recbole/model/sequential_recommender/actisasrec.py:20-224 (SURVEY section 8 f-4): AC-SASRec with
TiSASRec's time-interval aware attention.  Keys get an absolute-position and a time-interval embedding added, values likewise
(transformer_layers.py:1116-1134, 1085-1091); the layer is the transformer_layers.py variant (no re-normalising softmaxes).
Same class name, constructor keys, parameter names / shapes (reference checkpoints load unchanged), tuple returns.

The reference gathers time_matrix_emb_K/V[t_ij] into two [B,L,L,d] tensors per forward (41 MB each at B=256, L=50, d=64), drops
them out element-wise and contracts them with q / the attention matrices.  Here the interval matrix t_ij is built by one kernel
and the embeddings are read from their [time_span+1, d] tables inside the pair kernels of csrc/timeaware.cu; the dropout
multipliers come from Philox counters (or explicit tensors in parity tests).  As for ACSSEPT the reference registers no trainer
of this name; ACTiSASRecTrainer is the AC step (trainer.py:505-1036).
"""
import torch
import torch.nn as nn

from . import ops
from .acsasrec import BPRLoss
from .compat import SequentialRecommender, cfg_get
from .layers import Runtime
from .transformer_layers import ACTimeAwareTransformerEncoder, TimeTerms


class ACTiSASRec(SequentialRecommender):
    def __init__(self, config, dataset):
        super().__init__(config, dataset)
        self.n_layers = config['n_layers']
        self.n_heads = config['n_heads']
        self.hidden_size = config['hidden_size']
        self.inner_size = config['inner_size']
        self.hidden_dropout_prob = config['hidden_dropout_prob']
        self.attn_dropout_prob = config['attn_dropout_prob']
        self.hidden_act = config['hidden_act']
        self.layer_norm_eps = config['layer_norm_eps']
        self.time_span = config['time_span']
        self.timestamp = config['TIME_FIELD'] + '_list'
        self.initializer_range = config['initializer_range']
        self.loss_type = config['loss_type']
        self.combine_option = config['combine_option']
        self.rich_calibrated_combine = config['rich_calibrated_combine']
        self.two_level = config['two_level']
        self.use_position_embedding = config['use_position_embedding']        # read, never used (actisasrec.py:47, 104-144)
        self.use_order = config['use_order']
        self.use_distance = config['use_distance']
        self.trainable_mask_loss_weight = config['trainable_mask_loss_weight']
        self.EXTRA_FIELDS = [self.timestamp]                 # read by the training step besides sequence / length / target
        self.GRAPH_SAFE_STEP = True                      # no host-side work in the step: the trainer may capture it in a CUDA graph
        self.EVAL_FIELDS = [self.ITEM_SEQ, self.ITEM_SEQ_LEN, self.timestamp]   # what an evaluation batch must carry

        self.item_embedding = nn.Embedding(self.n_items, self.hidden_size, padding_idx=0)
        self.absolute_pos_K_embedding = nn.Embedding(self.max_seq_length, self.hidden_size, padding_idx=0)
        self.absolute_pos_V_embedding = nn.Embedding(self.max_seq_length, self.hidden_size, padding_idx=0)
        self.time_matrix_emb_K_embedding = nn.Embedding(self.time_span + 1, self.hidden_size, padding_idx=0)
        self.time_matrix_emb_V_embedding = nn.Embedding(self.time_span + 1, self.hidden_size, padding_idx=0)
        self.ti_trm_encoder = ACTimeAwareTransformerEncoder(
            n_layers=self.n_layers, n_heads=self.n_heads, hidden_size=self.hidden_size, inner_size=self.inner_size,
            hidden_dropout_prob=self.hidden_dropout_prob, attn_dropout_prob=self.attn_dropout_prob, hidden_act=self.hidden_act,
            layer_norm_eps=self.layer_norm_eps, combine_option=self.combine_option, use_order=self.use_order,
            use_distance=self.use_distance, two_level=self.two_level, rich_calibrated_combine=self.rich_calibrated_combine)
        self.LayerNorm = nn.LayerNorm(self.hidden_size, eps=self.layer_norm_eps)
        self.dropout = nn.Dropout(self.hidden_dropout_prob)
        if self.trainable_mask_loss_weight:
            self.mask_loss_weight = nn.Parameter(torch.FloatTensor([0.3]), requires_grad=True)
        else:
            self.mask_loss_weight = config['mask_loss_weight']
        if self.loss_type == 'BPR':
            self.loss_fct = BPRLoss()
        elif self.loss_type == 'CE':
            self.loss_fct = nn.CrossEntropyLoss()      # kept as an attribute; CE runs fused with the logits GEMM
        else:
            raise NotImplementedError("Make sure 'loss_type' in ['BPR', 'CE']!")
        self.apply(self._init_weights)

        self.logits_passes = int(cfg_get(config, 'logits_passes', 3))
        self._seed = int(cfg_get(config, 'seed', 2020) or 0)
        self._rng = None
        self._debug_rand = None            # explicit dropout masks / noise (parity tests)

    def _init_weights(self, module):
        """actisasrec.py:92-102."""
        if isinstance(module, (nn.Linear, nn.Embedding)):
            module.weight.data.normal_(mean=0.0, std=self.initializer_range)
        elif isinstance(module, nn.LayerNorm):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)
        if isinstance(module, nn.Linear) and module.bias is not None:
            module.bias.data.zero_()

    # ------------------------------------------------------------------------------------------
    def _runtime(self, device):
        if self._rng is None or self._rng.state.device != device:
            self._rng = ops.DeviceRng(self._seed, device)
        return Runtime(rng=self._rng, rand=self._debug_rand, attacked_last_only=True)

    def get_time_matrix(self, time_seq):
        """actisasrec.py:146-155: [B, L] time stamps -> int32 [B, L, L], |t_i - t_j| clipped to time_span"""
        if time_seq.size(1) != self.max_seq_length:
            raise ValueError('time_seq is %d long, MAX_ITEM_LIST_LENGTH is %d (actisasrec.py:149-150)' % (time_seq.size(1), self.max_seq_length))
        return ops.time_matrix(time_seq, self.time_span)

    def _encode(self, item_seq, item_seq_len, time_matrix, need_attacked=True):
        if not item_seq.is_cuda:
            raise ops.AcsrError('ACTiSASRec runs on CUDA only (got %s tensors); there is no CPU fallback' % item_seq.device)
        B, L = item_seq.shape
        if L > 64:
            raise ops.AcsrError('ACTiSASRec: the time-aware attention is implemented for sequences up to 64 long')
        rt = self._runtime(item_seq.device)
        if self.training:
            rt.rng.advance()
        p = self.dropout.p if self.training else 0.0
        x = ops.EmbedLnDropoutFn.apply(item_seq, self.item_embedding.weight, None, self.LayerNorm.weight, self.LayerNorm.bias,
                                       self.LayerNorm.eps, p, rt.mask('emb') if p > 0 else None, rt.rng, 1)
        pk, pv = self.absolute_pos_K_embedding.weight, self.absolute_pos_V_embedding.weight
        if L != pk.size(0):                # (the reference only runs L == MAX_ITEM_LIST_LENGTH, actisasrec.py:149-150)
            pk, pv = pk[:L], pv[:L]
        tt = TimeTerms(pk, pv,
                       self.time_matrix_emb_K_embedding.weight, self.time_matrix_emb_V_embedding.weight,
                       time_matrix.to(torch.int32), self.n_heads, p, rt)
        masks, att, cal = [], None, None
        n = len(self.ti_trm_encoder.layer)
        for l, layer in enumerate(self.ti_trm_encoder.layer):
            att, cal, m, _ = layer(x, item_seq, tt, rt=rt, layer_idx=l, need_attacked=(need_attacked and l == n - 1))
            x = cal
            masks.append(m)
        return ops.GatherLastFn.apply(att, cal, item_seq_len), masks

    def forward(self, item_seq, item_seq_len, time_matrix):
        """actisasrec.py:104-144 -> (attacked_output [B,d], calibrated_output [B,d], all_attack_masks)."""
        out, masks = self._encode(item_seq, item_seq_len, time_matrix, need_attacked=True)
        B = item_seq.size(0)
        return out[:B], out[B:], masks

    def calculate_loss(self, interaction):
        """actisasrec.py:173-193 -> (final_attacked_loss, calibrated_loss)."""
        item_seq = interaction[self.ITEM_SEQ]
        time_matrix = self.get_time_matrix(interaction[self.timestamp])
        out, masks = self._encode(item_seq, interaction[self.ITEM_SEQ_LEN], time_matrix, need_attacked=True)
        pos_items = interaction[self.POS_ITEM_ID]
        if self.loss_type == 'CE':
            ce = ops.LogitsCEFn.apply(out, self.item_embedding.weight, torch.cat((pos_items, pos_items)), 2, self.logits_passes)
        else:
            neg_items = interaction[self.NEG_ITEM_ID]
            ce = ops.BprLossFn.apply(out, self.item_embedding.weight, torch.cat((pos_items, pos_items)),
                                     torch.cat((neg_items, neg_items)), 2, self.loss_fct.gamma)
        mask_penalty = torch.mean(torch.stack([m.penalty() for m in masks], dim=0))
        w = self.mask_loss_weight[0] if self.trainable_mask_loss_weight else self.mask_loss_weight
        return -ce[0] + mask_penalty * w, ce[1]

    def predict(self, interaction):
        """actisasrec.py:195-209 -> (attacked_scores [B], scores [B])."""
        item_seq = interaction[self.ITEM_SEQ]
        time_matrix = self.get_time_matrix(interaction[self.timestamp])
        out, _ = self._encode(item_seq, interaction[self.ITEM_SEQ_LEN], time_matrix, need_attacked=True)
        B = item_seq.size(0)
        e = self.item_embedding(interaction[self.ITEM_ID])
        return torch.mul(out[:B], e).sum(dim=1), torch.mul(out[B:], e).sum(dim=1)

    def full_sort_predict(self, interaction):
        """actisasrec.py:211-224 -> (attacked_scores [B, n_items], scores [B, n_items])."""
        item_seq = interaction[self.ITEM_SEQ]
        time_matrix = self.get_time_matrix(interaction[self.timestamp])
        out, _ = self._encode(item_seq, interaction[self.ITEM_SEQ_LEN], time_matrix, need_attacked=True)
        B = item_seq.size(0)
        both = ops.logits_scores(out, self.item_embedding.weight, self.logits_passes)
        return both[:B], both[B:]

    def full_sort_topk(self, interaction, k, positive=None, counts=False):
        """fused scores -> scores[:,0] = -inf -> top-k -> hit flags of the calibrated stream (trainer.py:941-942, collector.py:145-153);
        counts=True: + the positive's rank counts [B, 2] (ops.full_sort_topk)"""
        item_seq = interaction[self.ITEM_SEQ]
        time_matrix = self.get_time_matrix(interaction[self.timestamp])
        cal, _ = self._encode(item_seq, interaction[self.ITEM_SEQ_LEN], time_matrix, need_attacked=False)
        return ops.full_sort_topk(cal.contiguous(), self.item_embedding.weight, k, positive, self.logits_passes, counts=counts)

    def sampled_topk(self, interaction, candidates, k, positive=None, counts=False):
        """sampled-candidate ranking of the calibrated stream (candidates [B, 1+N], positive in column 0, written there from
        `positive` when given) -> (scores [B, 1+N], rec_topk [B, k+1]) (+ counts [B, 3] of ops.candidate_rank with counts=True)"""
        if positive is not None:
            candidates[:, 0].copy_(positive)
        time_matrix = self.get_time_matrix(interaction[self.timestamp])
        cal, _ = self._encode(interaction[self.ITEM_SEQ], interaction[self.ITEM_SEQ_LEN], time_matrix, need_attacked=False)
        r = ops.candidate_rank(cal, self.item_embedding.weight, candidates, k, want_scores=True, want_counts=counts)
        return (r[1], r[0]) + tuple(r[2:])
