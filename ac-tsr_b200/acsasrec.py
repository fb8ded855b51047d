"""ACSASRec -- drop-in for recbole/model/sequential_recommender/acsasrec.py:9-164.

Same constructor `(config, dataset)`, config keys, parameter names/shapes (reference checkpoints
load unchanged) and return conventions: calculate_loss -> (final_attacked_loss, calibrated_loss),
predict -> (attacked_scores, scores), full_sort_predict -> (None, scores[B, n_items]).
The compute runs in libacsr.so (hand-written sm_100a kernels); CPU tensors raise.
"""
import torch
from torch import nn

from . import ops
from .compat import SequentialRecommender, cfg_get
from .layers import AttackRTransformerEncoder, Runtime


class BPRLoss(nn.Module):
    """recbole/model/loss.py:21-47 (only reached with loss_type: BPR; shipped configs use CE)."""

    def __init__(self, gamma=1e-10):
        super().__init__()
        self.gamma = gamma

    def forward(self, pos_score, neg_score):
        return -torch.log(self.gamma + torch.sigmoid(pos_score - neg_score)).mean()


class ACSASRec(SequentialRecommender):
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
        self.initializer_range = config['initializer_range']
        self.loss_type = config['loss_type']
        self.combine_option = config['combine_option']
        self.rich_calibrated_combine = config['rich_calibrated_combine']
        self.two_level = config['two_level']
        self.use_position_embedding = config['use_position_embedding']
        self.use_order = config['use_order']
        self.use_distance = config['use_distance']
        self.trainable_mask_loss_weight = config['trainable_mask_loss_weight']

        self.item_embedding = nn.Embedding(self.n_items, self.hidden_size, padding_idx=0)
        if self.use_position_embedding:
            self.position_embedding = nn.Embedding(self.max_seq_length, self.hidden_size)
        # The reference never forwards seq_length (gate hard-wired to 50, layers.py:878); sizing the gate
        # by MAX_ITEM_LIST_LENGTH is identical at L=50 and lets longer sequences run.
        self.trm_encoder = AttackRTransformerEncoder(
            n_layers=self.n_layers, n_heads=self.n_heads, hidden_size=self.hidden_size, inner_size=self.inner_size,
            hidden_dropout_prob=self.hidden_dropout_prob, attn_dropout_prob=self.attn_dropout_prob,
            hidden_act=self.hidden_act, layer_norm_eps=self.layer_norm_eps, combine_option=self.combine_option,
            use_order=self.use_order, use_distance=self.use_distance, two_level=self.two_level,
            rich_calibrated_combine=self.rich_calibrated_combine, seq_length=self.max_seq_length)
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

        # B200 runtime state (not parameters, not in the state_dict)
        self.logits_passes = int(cfg_get(config, 'logits_passes', 3))
        self.step_branches = int(cfg_get(config, 'step_branches', 1))     # parallel sequence groups of the fused step (measured: no gain at B=256)
        self._seed = int(cfg_get(config, 'seed', 2020))
        self._rng = None
        self._debug_rand = None      # {key: tensor}: explicit dropout masks / noise for parity tests

    def _init_weights(self, module):
        """acsasrec.py:74-84."""
        if isinstance(module, (nn.Linear, nn.Embedding)):
            module.weight.data.normal_(mean=0.0, std=self.initializer_range)
        elif isinstance(module, nn.LayerNorm):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)
        if isinstance(module, nn.Linear) and module.bias is not None:
            module.bias.data.zero_()

    def flat_groups(self):
        """parameters the fused step views as stacked tensors (one batched GEMM for Q/K/V and for the attack pair)."""
        out = []
        for layer in self.trm_encoder.layer:
            aa = layer.attack_attention
            out += [[aa.query.weight, aa.key.weight, aa.value.weight], [aa.query.bias, aa.key.bias, aa.value.bias],
                    [aa.attack_query_transform.weight, aa.attack_key_transform.weight],
                    [aa.attack_query_transform.bias, aa.attack_key_transform.bias]]
        return out

    # ------------------------------------------------------------------------------------------
    def _runtime(self, device, attacked_last_only=True):
        if self._rng is None or self._rng.state.device != device:
            self._rng = ops.DeviceRng(self._seed, device)
        return Runtime(rng=self._rng, rand=self._debug_rand, attacked_last_only=attacked_last_only)

    def _encode(self, item_seq, item_seq_len, need_attacked=True):
        """-> stacked [2B,d] (attacked rows first) or [B,d] (calibrated only), and the per-layer AttackMask list."""
        dev = self.item_embedding.weight.device
        if not item_seq.is_cuda:
            raise ops.AcsrError('ACSASRec runs on CUDA only (got %s tensors); there is no CPU fallback' % item_seq.device)
        fused = getattr(self, '_fused_step', None)
        if (fused is not None and not self.training and not need_attacked and not torch.is_grad_enabled()
                and item_seq.dim() == 2):
            return fused.encode_eval(item_seq, item_seq_len), []      # eval: the fused forward (same kernels as training)
        rt = self._runtime(dev)
        if self.training:
            rt.rng.advance()
        p = self.dropout.p if self.training else 0.0
        pos = self.position_embedding.weight if self.use_position_embedding else None
        if pos is not None and item_seq.size(1) != pos.size(0):
            pos = pos[: item_seq.size(1)].contiguous()
        x = ops.EmbedLnDropoutFn.apply(item_seq, self.item_embedding.weight, pos, self.LayerNorm.weight, self.LayerNorm.bias,
                                       self.LayerNorm.eps, p, rt.mask('emb') if p > 0 else None, rt.rng, 1)
        if not need_attacked:
            rt.attacked_last_only = True
        layers, masks = self._run_encoder(x, item_seq, rt, need_attacked)
        att, cal = layers
        out = ops.GatherLastFn.apply(att, cal, item_seq_len)
        return out, masks

    def _run_encoder(self, x, item_seq, rt, need_attacked):
        enc = self.trm_encoder
        n = len(enc.layer)
        masks, att, cal = [], None, None
        for l, layer in enumerate(enc.layer):
            na = need_attacked and l == n - 1
            att, cal, m, _ = layer(x, item_seq, rt=rt, layer_idx=l, need_attacked=na)
            x = cal
            masks.append(m)
        return (att, cal), masks

    def forward(self, item_seq, item_seq_len, is_train=False):
        """acsasrec.py:86-104 -> (attacked_output[B,d], calibrated_output[B,d], all_attack_masks)."""
        out, masks = self._encode(item_seq, item_seq_len, need_attacked=True)
        B = item_seq.size(0)
        return out[:B], out[B:], masks

    def _cal_loss(self, output, interaction, attack_loss=False):
        """acsasrec.py:107-121."""
        pos_items = interaction[self.POS_ITEM_ID]
        if self.loss_type == 'BPR':
            neg_items = interaction[self.NEG_ITEM_ID]
            return ops.BprLossFn.apply(output, self.item_embedding.weight, pos_items, neg_items, 1, self.loss_fct.gamma)[0]
        return ops.LogitsCEFn.apply(output, self.item_embedding.weight, pos_items, 1, self.logits_passes)[0]

    def calculate_loss(self, interaction):
        """acsasrec.py:123-144 -> (final_attacked_loss, calibrated_loss)."""
        item_seq = interaction[self.ITEM_SEQ]
        item_seq_len = interaction[self.ITEM_SEQ_LEN]
        out, masks = self._encode(item_seq, item_seq_len, need_attacked=True)
        B = item_seq.size(0)
        if self.loss_type == 'CE':
            pos_items = interaction[self.POS_ITEM_ID]
            # attacked and calibrated rows share ONE pass over the item table
            ce = ops.LogitsCEFn.apply(out, self.item_embedding.weight, torch.cat((pos_items, pos_items)), 2,
                                      self.logits_passes)
            attacked_ce, calibrated_loss = ce[0], ce[1]
        else:                                   # BPR: both row groups through one pair of kernels
            pos_items, neg_items = interaction[self.POS_ITEM_ID], interaction[self.NEG_ITEM_ID]
            bl = ops.BprLossFn.apply(out, self.item_embedding.weight, torch.cat((pos_items, pos_items)),
                                     torch.cat((neg_items, neg_items)), 2, self.loss_fct.gamma)
            attacked_ce, calibrated_loss = bl[0], bl[1]
        assert len(masks) > 0
        mask_penalty = torch.mean(torch.stack([m.penalty() for m in masks], dim=0))
        w = self.mask_loss_weight[0] if self.trainable_mask_loss_weight else self.mask_loss_weight
        final_attacked_loss = -attacked_ce + mask_penalty * w
        return final_attacked_loss, calibrated_loss

    def predict(self, interaction):
        """acsasrec.py:146-155."""
        item_seq = interaction[self.ITEM_SEQ]
        item_seq_len = interaction[self.ITEM_SEQ_LEN]
        test_item = interaction[self.ITEM_ID]
        out, _ = self._encode(item_seq, item_seq_len, need_attacked=True)
        B = item_seq.size(0)
        test_item_emb = self.item_embedding(test_item)
        attacked_scores = torch.mul(out[:B], test_item_emb).sum(dim=1)
        scores = torch.mul(out[B:], test_item_emb).sum(dim=1)
        return attacked_scores, scores

    def full_sort_predict(self, interaction):
        """acsasrec.py:157-164 -> (None, scores[B, n_items]); the dead attacked branch is skipped."""
        item_seq = interaction[self.ITEM_SEQ]
        item_seq_len = interaction[self.ITEM_SEQ_LEN]
        out, _ = self._encode(item_seq, item_seq_len, need_attacked=False)
        vp = getattr(self, '_vp', None)
        if vp is not None and vp.sharded:         # vocab-sharded table: every shard scores all ranks' rows, my rows are gathered back
            B = out.shape[0]
            out_all = vp._all_gather(out).reshape(vp.world * B, -1)
            part = ops.logits_scores(out_all, vp.shard(self.item_embedding.weight).contiguous(), self.logits_passes)
            padded = part.new_zeros((vp.world * B, vp.per))
            padded[:, :part.shape[1]] = part
            mine = vp._all_gather(padded)[:, vp.rank * B:(vp.rank + 1) * B]               # [W, B, per]
            return None, mine.permute(1, 0, 2).reshape(B, vp.world * vp.per)[:, :self.n_items].contiguous()
        scores = ops.logits_scores(out, self.item_embedding.weight, self.logits_passes)
        return None, scores

    def full_sort_topk(self, interaction, k, positive=None, counts=False):
        """Fused replacement of full_sort_predict + `scores[:,0]=-inf` + topk + hit flags
        (trainer.py:941-942, collector.py:145-153): -> (topk_scores[B,k], topk_idx[B,k], rec_topk[B,k+1]|None), and with
        counts=True the positive's rank counts [B, 2] (ops.full_sort_topk) as a fourth entry."""
        item_seq = interaction[self.ITEM_SEQ]
        item_seq_len = interaction[self.ITEM_SEQ_LEN]
        # programmatic dependent launch between the eval kernels (prologues overlap the previous kernel's tail), as in the training
        # step: measured +1 % eval users/s on B200
        was = ops.LIB.query('acsr_set_pdl', 1)
        try:
            out, _ = self._encode(item_seq, item_seq_len, need_attacked=False)
            vp = getattr(self, '_vp', None)
            if vp is not None:                        # vocab-parallel: partial top-k per shard, all-gather, merge (dist.py)
                return vp.full_sort_topk(out, self.item_embedding.weight, k, positive, counts=counts)
            return ops.full_sort_topk(out, self.item_embedding.weight, k, positive, self.logits_passes, counts=counts)
        finally:
            ops.LIB.query('acsr_set_pdl', was)

    def sampled_topk(self, interaction, candidates, k, positive=None, counts=False):
        """Sampled-candidate ranking (`eval_args.mode: uniN / popN`; trainer.py _neg_sample_batch_eval + collector.py
        eval_batch_collect): candidates [B, 1+N] int64 with the positive in column 0 (written there from `positive` when
        given).  Encodes each sequence once (the reference predicts on the interaction repeated 1+N times) and ranks the
        calibrated scores -> (scores [B, 1+N], rec_topk [B, k+1]), and with counts=True the counts [B, 3] of ops.candidate_rank."""
        vp = getattr(self, '_vp', None)
        if vp is not None and vp.sharded:
            raise ValueError('sampled evaluation is not implemented for a vocab-sharded item table')
        if positive is not None:
            candidates[:, 0].copy_(positive)
        was = ops.LIB.query('acsr_set_pdl', 1)
        try:
            out, _ = self._encode(interaction[self.ITEM_SEQ], interaction[self.ITEM_SEQ_LEN], need_attacked=False)
            r = ops.candidate_rank(out, self.item_embedding.weight, candidates, k, want_scores=True, want_counts=counts)
            return (r[1], r[0]) + tuple(r[2:])
        finally:
            ops.LIB.query('acsr_set_pdl', was)
