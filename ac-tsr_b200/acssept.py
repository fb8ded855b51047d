"""ACSSEPT -- drop-in for recbole/model/sequential_recommender/acssept.py:21-228 (SURVEY section 8 f-4): the SSE-PT sibling of
AC-SASRec.  A user embedding is concatenated to the item embedding of every position (hidden = item_hidden_size +
user_hidden_size, acssept.py:124-128) and the encoder is the one of recbole/model/transformer_layers.py:742-1007 -- the AC layer
WITHOUT the re-normalising softmaxes of layers.py:917-925 (see transformer_layers.py here, ACSR_ATTN_PLAIN in include/acsr.h).
Same class name, constructor keys, parameter names / shapes (reference checkpoints load unchanged) and tuple returns.

Scoring a candidate item v for row b is seq_output[b] . cat(E[v], user_vec[b]) (acssept.py:164-171, 212-224); the reference
expands a [B, n_items, hidden] tensor for it.  Here it is split as  out[:, :di] . E^T  +  (out[:, di:] . user_vec)  : the first
term is the fused tcgen05 logits kernel over the item table, the second one number per row.  That per-row constant shifts all
logits of a row alike, so it cancels in the cross entropy, in the BPR difference and in the top-k order; it is added where the
reference returns raw scores (predict, full_sort_predict).

(The reference only runs with user_hidden_size == item_hidden_size: acssept.py:127 expands the user vector "as" the item
embeddings.  Any pair of widths works here.)

Trainer: the reference registers no ACSSEPTTrainer (recbole/trainer/trainer.py:1038-1048 lists AttackRSASRec, ACSASRec and
AcBERT4Rec; utils.py:89-100 then falls back to the stock Trainer, whose evaluation cannot take the tuple full_sort_predict
returns, trainer.py:397).  ACSSEPTTrainer here is the AC step the model's tuple API is written for (trainer.py:505-1036).
"""
import torch
import torch.nn as nn

from . import ops
from .acsasrec import BPRLoss
from .compat import SequentialRecommender, cfg_get
from .layers import Runtime
from .transformer_layers import AttackRTransformerEncoder


class _NoGradRow0(torch.autograd.Function):
    """nn.Embedding(padding_idx=0): row 0 never receives a gradient through a lookup (acssept.py:57-59)."""

    @staticmethod
    def forward(ctx, table):
        return table.view_as(table)

    @staticmethod
    def backward(ctx, g):
        g = g.clone()
        g[0].zero_()
        return g


class ACSSEPT(SequentialRecommender):
    def __init__(self, config, dataset):
        super().__init__(config, dataset)
        self.n_layers = config['n_layers']
        self.n_heads = config['n_heads']
        self.user_hidden_size = config['user_hidden_size']
        self.item_hidden_size = config['item_hidden_size']
        self.hidden_size = self.user_hidden_size + self.item_hidden_size
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
        self.n_users = dataset.num(self.USER_ID)
        self.EXTRA_FIELDS = [self.USER_ID]                 # read by the training step besides sequence / length / target
        self.GRAPH_SAFE_STEP = True                      # no host-side work in the step: the trainer may capture it in a CUDA graph
        self.EVAL_FIELDS = [self.ITEM_SEQ, self.ITEM_SEQ_LEN, self.USER_ID]      # what an evaluation batch must carry

        self.user_embedding = nn.Embedding(self.n_users, self.user_hidden_size, padding_idx=0)         # concatenated to item_seq
        self.user_test_embedding = nn.Embedding(self.n_users, self.user_hidden_size, padding_idx=0)    # ... to the test items
        self.item_embedding = nn.Embedding(self.n_items, self.item_hidden_size, padding_idx=0)
        if self.use_position_embedding:
            self.position_embedding = nn.Embedding(self.max_seq_length, self.hidden_size)
        self.trm_encoder = AttackRTransformerEncoder(
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
        """acssept.py:111-122 (the padding rows are drawn too: normal_ overwrites the zeros of padding_idx)."""
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

    def _rows(self, table, ids):
        """table[ids] with nn.Embedding(padding_idx=0) gradient semantics, through the row gather / scatter-add kernels"""
        return ops.GatherRowsFn.apply(_NoGradRow0.apply(table), ids.reshape(-1))

    def _encode(self, item_seq, item_seq_len, user_id, need_attacked=True):
        """-> [2B, hidden] (attacked rows first) or [B, hidden] (calibrated only) at position item_seq_len - 1, [AttackMask]"""
        if not item_seq.is_cuda:
            raise ops.AcsrError('ACSSEPT runs on CUDA only (got %s tensors); there is no CPU fallback' % item_seq.device)
        if item_seq.size(1) > 64:
            raise ops.AcsrError('ACSSEPT: the transformer_layers.py attention variant is implemented for sequences up to 64 long')
        rt = self._runtime(item_seq.device)
        if self.training:
            rt.rng.advance()
        B, L = item_seq.shape
        d = self.hidden_size
        item_emb = self._rows(self.item_embedding.weight, item_seq).view(B, L, self.item_hidden_size)
        user_emb = self._rows(self.user_embedding.weight, user_id)
        # acssept.py:125-128: [item ; user] per position.  The rows then go through the gather + position add + LayerNorm + dropout
        # kernel (K1) as a B*L-row table read in order (ids 1..B*L; row 0 is the kernel's padding row)
        tokens = torch.cat((item_emb, user_emb.view(B, 1, -1).expand(B, L, self.user_hidden_size)), dim=-1).reshape(B * L, d)
        table = torch.cat((tokens.new_zeros(1, d), tokens))
        ids = torch.arange(1, B * L + 1, device=item_seq.device, dtype=torch.int64).view(B, L)
        p = self.dropout.p if self.training else 0.0
        pos = self.position_embedding.weight if self.use_position_embedding else None
        if pos is not None and L != pos.size(0):
            pos = pos[:L].contiguous()
        x = ops.EmbedLnDropoutFn.apply(ids, table, pos, self.LayerNorm.weight, self.LayerNorm.bias, self.LayerNorm.eps, p,
                                       rt.mask('emb') if p > 0 else None, rt.rng, 1)
        masks, att, cal = [], None, None
        n = len(self.trm_encoder.layer)
        for l, layer in enumerate(self.trm_encoder.layer):
            att, cal, m, _ = layer(x, item_seq, rt=rt, layer_idx=l, need_attacked=(need_attacked and l == n - 1))
            x = cal
            masks.append(m)
        return ops.GatherLastFn.apply(att, cal, item_seq_len), masks

    def forward(self, item_seq, item_seq_len, user_id):
        """acssept.py:124-145 -> (attacked_output [B, hidden], calibrated_output [B, hidden], all_attack_masks)."""
        out, masks = self._encode(item_seq, item_seq_len, user_id, need_attacked=True)
        B = item_seq.size(0)
        return out[:B], out[B:], masks

    def _item_part(self, out):
        return out[:, :self.item_hidden_size].contiguous()

    def _user_term(self, out, user_vec):
        """the per-row constant (out[:, di:] . user_vec) every candidate's score carries"""
        return torch.mul(out[:, self.item_hidden_size:], user_vec).sum(dim=1)

    def calculate_loss(self, interaction):
        """acssept.py:174-190 -> (final_attacked_loss, calibrated_loss).  The user half of a candidate row adds the same number to
        every logit of a sequence (and to both BPR scores), so both losses are functions of out[:, :di] . E^T alone."""
        item_seq = interaction[self.ITEM_SEQ]
        item_seq_len = interaction[self.ITEM_SEQ_LEN]
        user_id = interaction[self.USER_ID]
        out, masks = self._encode(item_seq, item_seq_len, user_id, need_attacked=True)
        out_i = self._item_part(out)
        pos_items = interaction[self.POS_ITEM_ID]
        if self.loss_type == 'CE':
            ce = ops.LogitsCEFn.apply(out_i, self.item_embedding.weight, torch.cat((pos_items, pos_items)), 2, self.logits_passes)
        else:
            neg_items = interaction[self.NEG_ITEM_ID]
            ce = ops.BprLossFn.apply(out_i, self.item_embedding.weight, torch.cat((pos_items, pos_items)),
                                     torch.cat((neg_items, neg_items)), 2, self.loss_fct.gamma)
        mask_penalty = torch.mean(torch.stack([m.penalty() for m in masks], dim=0))
        w = self.mask_loss_weight[0] if self.trainable_mask_loss_weight else self.mask_loss_weight
        return -ce[0] + mask_penalty * w, ce[1]

    def predict(self, interaction):
        """acssept.py:192-207 -> (attacked_scores [B], scores [B]); scored against user_test_embedding."""
        item_seq = interaction[self.ITEM_SEQ]
        user_id = interaction[self.USER_ID]
        out, _ = self._encode(item_seq, interaction[self.ITEM_SEQ_LEN], user_id, need_attacked=True)
        B = item_seq.size(0)
        e = torch.cat((self.item_embedding(interaction[self.ITEM_ID]), self.user_test_embedding(user_id)), dim=-1)
        return torch.mul(out[:B], e).sum(dim=1), torch.mul(out[B:], e).sum(dim=1)

    def full_sort_predict(self, interaction):
        """acssept.py:209-228 -> (attacked_scores [B, n_items], scores [B, n_items])."""
        item_seq = interaction[self.ITEM_SEQ]
        user_id = interaction[self.USER_ID]
        out, _ = self._encode(item_seq, interaction[self.ITEM_SEQ_LEN], user_id, need_attacked=True)
        B = item_seq.size(0)
        ut = self.user_test_embedding(user_id)
        both = ops.logits_scores(self._item_part(out), self.item_embedding.weight, self.logits_passes)
        both += self._user_term(out, torch.cat((ut, ut))).view(-1, 1)
        return both[:B], both[B:]

    def full_sort_topk(self, interaction, k, positive=None, counts=False):
        """fused scores -> scores[:,0] = -inf -> top-k -> hit flags of the calibrated stream (trainer.py:941-942,
        collector.py:145-153).  The user term is added to the k returned scores; it cannot change their order.  counts=True: + the
        positive's rank counts [B, 2] (ops.full_sort_topk), taken on the item part of the score for the same reason."""
        item_seq = interaction[self.ITEM_SEQ]
        user_id = interaction[self.USER_ID]
        cal, _ = self._encode(item_seq, interaction[self.ITEM_SEQ_LEN], user_id, need_attacked=False)
        r = ops.full_sort_topk(self._item_part(cal), self.item_embedding.weight, k, positive, self.logits_passes, counts=counts)
        return (r[0] + self._user_term(cal, self.user_test_embedding(user_id)).view(-1, 1),) + tuple(r[1:])

    def sampled_topk(self, interaction, candidates, k, positive=None, counts=False):
        """sampled-candidate ranking of the calibrated stream (candidates [B, 1+N], positive in column 0, written there from
        `positive` when given) -> (scores [B, 1+N], rec_topk [B, k+1]).  The user term is added to the returned scores; it is
        the same for every candidate of a row and cannot change the rank.  counts=True: + counts [B, 3] of ops.candidate_rank."""
        if positive is not None:
            candidates[:, 0].copy_(positive)
        user_id = interaction[self.USER_ID]
        cal, _ = self._encode(interaction[self.ITEM_SEQ], interaction[self.ITEM_SEQ_LEN], user_id, need_attacked=False)
        r = ops.candidate_rank(self._item_part(cal), self.item_embedding.weight, candidates, k, want_scores=True, want_counts=counts)
        return (r[1] + self._user_term(cal, self.user_test_embedding(user_id)).view(-1, 1), r[0]) + tuple(r[2:])
