"""AcBERT4Rec -- drop-in for recbole/model/sequential_recommender/acbert4rec.py:11-267 (SURVEY section 8 f-4): the
bidirectional, masked-item sibling of AC-SASRec on the SAME kernels.  Same class name, constructor keys, parameter names /
shapes (the item table has n_items + 1 rows: the last one is the mask token, acbert4rec.py:41-45), the same host-side
masking procedure (python `random`, so a seeded run masks the same positions as the reference), the same tuple returns.

What runs where: the encoder is AttackRTransformerEncoder with the bidirectional attention mask (ACSR_ATTN_BIDIRECTIONAL:
only padded keys are masked); the hidden states of the masked positions are gathered by a row-gather kernel instead of the
reference's one-hot bmm (acbert4rec.py:214-222); the masked-item cross entropy over table[:n_items] is the fused tcgen05
logits + CE kernel with per-row weights (acbert4rec.py:198-205).  Training uses the reference trainer semantics (two routed
backward passes, trainer.py:672-686) through the autograd Functions of ops.py.

Reference quirk kept on purpose: evaluation appends one position (reconstruct_test_data makes the sequence L+1 long), so a
`combine_option: gate` model -- whose gate is Linear(hidden, seq_length) -- cannot be evaluated in the reference either
(shape mismatch at layers.py:887-888); here that raises the same kind of ValueError.  `fixed` / `annealing` work.
"""
import random

import torch
import torch.nn as nn

from . import ops
from .compat import SequentialRecommender, cfg_get
from .layers import AttackRTransformerEncoder, Runtime


class AcBERT4Rec(SequentialRecommender):
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
        self.mask_ratio = config['mask_ratio']
        self.loss_type = config['loss_type']
        self.initializer_range = config['initializer_range']
        self.combine_option = config['combine_option']
        self.rich_calibrated_combine = config['rich_calibrated_combine']
        self.two_level = config['two_level']
        self.use_position_embedding = config['use_position_embedding']
        self.use_order = config['use_order']
        self.use_distance = config['use_distance']
        self.trainable_mask_loss_weight = config['trainable_mask_loss_weight']
        self.logits_passes = int(cfg_get(config, 'logits_passes', 3))

        self.mask_token = self.n_items
        self.mask_item_length = int(self.mask_ratio * self.max_seq_length)

        self.item_embedding = nn.Embedding(self.n_items + 1, self.hidden_size, padding_idx=0)      # + the mask token
        if self.use_position_embedding:
            self.position_embedding = nn.Embedding(self.max_seq_length, self.hidden_size)
        self.trm_encoder = AttackRTransformerEncoder(
            n_layers=self.n_layers, n_heads=self.n_heads, hidden_size=self.hidden_size, inner_size=self.inner_size,
            hidden_dropout_prob=self.hidden_dropout_prob, attn_dropout_prob=self.attn_dropout_prob, hidden_act=self.hidden_act,
            layer_norm_eps=self.layer_norm_eps, combine_option=self.combine_option, use_order=self.use_order,
            use_distance=self.use_distance, two_level=self.two_level, rich_calibrated_combine=self.rich_calibrated_combine,
            seq_length=int(cfg_get(config, 'gate_seq_length', 50)))                                # layers.py:878: Linear(hidden, 50)
        self.LayerNorm = nn.LayerNorm(self.hidden_size, eps=self.layer_norm_eps)
        self.dropout = nn.Dropout(self.hidden_dropout_prob)
        if self.trainable_mask_loss_weight:
            self.mask_loss_weight = nn.Parameter(torch.FloatTensor([0.3]), requires_grad=True)
        else:
            self.mask_loss_weight = config['mask_loss_weight']
        if self.loss_type not in ['BPR', 'CE']:
            raise AssertionError("Make sure 'loss_type' in ['BPR', 'CE']!")
        self._seed = int(cfg_get(config, 'seed', 2020) or 0)
        self._rng = None
        self._debug_rand = None            # explicit dropout masks / noise (parity tests)
        self._debug_masked = None          # explicit (masked_item_seq, pos_items, neg_items, masked_index) (parity tests)
        # the training step split for the trainer's CUDA graph: prepare_batch (host: the reference's python masking) fills these
        # fields, the rest of the step (calculate_loss on them + routed backward + Adam) has no host-side work
        self.EXTRA_FIELDS = ['bert_masked_seq', 'bert_pos_items', 'bert_neg_items', 'bert_masked_index']
        self.GRAPH_SAFE_STEP = True
        self.apply(self._init_weights)

    def _init_weights(self, module):
        if isinstance(module, (nn.Linear, nn.Embedding)):
            module.weight.data.normal_(mean=0.0, std=self.initializer_range)
        elif isinstance(module, nn.LayerNorm):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)
        if isinstance(module, nn.Linear) and module.bias is not None:
            module.bias.data.zero_()

    # ---- host-side masking: the same procedure and the same `random` call sequence as acbert4rec.py:86-150 ----
    def _neg_sample(self, item_set):
        item = random.randint(1, self.n_items - 1)
        while item in item_set:
            item = random.randint(1, self.n_items - 1)
        return item

    def _padding_sequence(self, sequence, max_length):
        pad_len = max_length - len(sequence)
        sequence = [0] * pad_len + sequence
        return sequence[-max_length:]

    def reconstruct_train_data(self, item_seq):
        device = item_seq.device
        batch_size = item_seq.size(0)
        masked_item_sequence, pos_items, neg_items, masked_index = [], [], [], []
        for instance in item_seq.cpu().numpy().tolist():
            masked_sequence = instance.copy()
            pos_item, neg_item, index_ids = [], [], []
            for index_id, item in enumerate(instance):
                if item == 0:
                    break
                if random.random() < self.mask_ratio:
                    pos_item.append(item)
                    neg_item.append(self._neg_sample(instance))
                    masked_sequence[index_id] = self.mask_token
                    index_ids.append(index_id)
            masked_item_sequence.append(masked_sequence)
            pos_items.append(self._padding_sequence(pos_item, self.mask_item_length))
            neg_items.append(self._padding_sequence(neg_item, self.mask_item_length))
            masked_index.append(self._padding_sequence(index_ids, self.mask_item_length))

        def t(x):
            return torch.tensor(x, dtype=torch.long, device=device).view(batch_size, -1)
        return t(masked_item_sequence), t(pos_items), t(neg_items), t(masked_index)

    def prepare_batch(self, interaction):
        """host half of the training step: reconstruct_train_data (acbert4rec.py:86-150, python `random`, one call per step as in the
        reference) -> the interaction plus the four masked tensors, which calculate_loss then takes as given"""
        from .compat import Interaction
        masked = self.reconstruct_train_data(interaction[self.ITEM_SEQ])
        fields = {k: interaction[k] for k in (self.ITEM_SEQ, self.ITEM_SEQ_LEN, self.POS_ITEM_ID)}
        fields.update(zip(self.EXTRA_FIELDS, masked))
        return Interaction(fields)

    def reconstruct_test_data(self, item_seq, item_seq_len):
        """mask token appended at position item_seq_len of a sequence one longer (acbert4rec.py:152-160), vectorised"""
        padding = torch.zeros(item_seq.size(0), 1, dtype=torch.long, device=item_seq.device)
        item_seq = torch.cat((item_seq, padding), dim=-1)
        item_seq.scatter_(1, item_seq_len.view(-1, 1), self.mask_token)
        return item_seq

    # ------------------------------------------------------------------------------------------
    def _runtime(self, device):
        if self._rng is None or self._rng.state.device != device:
            self._rng = ops.DeviceRng(self._seed, device)
        return Runtime(rng=self._rng, rand=self._debug_rand, attacked_last_only=True, bidirectional=True)

    def forward(self, item_seq):
        """acbert4rec.py:162-179 -> (attacked_output [B,L,d], calibrated_output [B,L,d], all_attack_masks)."""
        if not item_seq.is_cuda:
            raise ops.AcsrError('AcBERT4Rec runs on CUDA only (got %s tensors); there is no CPU fallback' % item_seq.device)
        rt = self._runtime(item_seq.device)
        if self.training:
            rt.rng.advance()
        p = self.dropout.p if self.training else 0.0
        pos = self.position_embedding.weight if self.use_position_embedding else None
        if pos is not None:
            if item_seq.size(1) > pos.size(0):          # the reference indexes past the table here (acbert4rec.py:165-167)
                raise IndexError('position_embedding has %d rows, the sequence is %d long' % (pos.size(0), item_seq.size(1)))
            pos = pos[: item_seq.size(1)].contiguous()
        x = ops.EmbedLnDropoutFn.apply(item_seq, self.item_embedding.weight, pos, self.LayerNorm.weight, self.LayerNorm.bias,
                                       self.LayerNorm.eps, p, rt.mask('emb') if p > 0 else None, rt.rng, 1)
        masks, att, cal = [], None, None
        n = len(self.trm_encoder.layer)
        for l, layer in enumerate(self.trm_encoder.layer):
            att, cal, m, _ = layer(x, item_seq, rt=rt, layer_idx=l, need_attacked=(l == n - 1))
            x = cal
            masks.append(m)
        return att, cal, masks

    def multi_hot_embed(self, masked_index, max_length):
        masked_index = masked_index.view(-1)
        multi_hot = torch.zeros(masked_index.size(0), max_length, device=masked_index.device)
        multi_hot[torch.arange(masked_index.size(0)), masked_index] = 1
        return multi_hot

    def _cal_loss(self, seq_output, pos_items, targets):
        """acbert4rec.py:198-205: CE over table[:n_items] at the masked slots, weighted by `targets`, without the [B*m, V] logits"""
        E = self.item_embedding.weight[:self.n_items]
        out = seq_output.reshape(-1, self.hidden_size)
        return ops.LogitsCEFn.apply(out, E, pos_items.reshape(-1), 1, self.logits_passes, targets)[0]

    def calculate_loss(self, interaction):
        """acbert4rec.py:207-245 -> (final_attacked_loss, calibrated_loss)."""
        item_seq = interaction[self.ITEM_SEQ]
        if self._debug_masked is not None:
            masked_item_seq, pos_items, neg_items, masked_index = self._debug_masked
        elif self.EXTRA_FIELDS[0] in interaction:          # prepared on the host by prepare_batch (the trainer's graphed step)
            masked_item_seq, pos_items, neg_items, masked_index = (interaction[k] for k in self.EXTRA_FIELDS)
        else:
            masked_item_seq, pos_items, neg_items, masked_index = self.reconstruct_train_data(item_seq)
        attacked_output, calibrated_output, all_attack_masks = self.forward(masked_item_seq)
        B, L = masked_item_seq.shape
        # hidden states of the masked positions: a row gather (the reference multiplies by a one-hot [B, m, L] matrix)
        flat = (torch.arange(B, device=item_seq.device).view(B, 1) * L + masked_index).reshape(-1)
        both = ops.GatherRowsFn.apply(torch.cat((attacked_output.reshape(B * L, -1), calibrated_output.reshape(B * L, -1))),
                                      torch.cat((flat, flat + B * L)))
        targets = (masked_index > 0).float().view(-1)
        # attacked and calibrated rows share ONE pass over the item table
        E = self.item_embedding.weight[:self.n_items]
        ce = ops.LogitsCEFn.apply(both, E, torch.cat((pos_items.reshape(-1), pos_items.reshape(-1))), 2, self.logits_passes,
                                  torch.cat((targets, targets)))
        mask_penalty = torch.mean(torch.stack([m.penalty() for m in all_attack_masks], dim=0))
        w = self.mask_loss_weight[0] if self.trainable_mask_loss_weight else self.mask_loss_weight
        final_attacked_loss = -ce[0] + mask_penalty * w
        return final_attacked_loss, ce[1]

    def _test_outputs(self, interaction):
        item_seq = interaction[self.ITEM_SEQ]
        item_seq_len = interaction[self.ITEM_SEQ_LEN]
        seq = self.reconstruct_test_data(item_seq, item_seq_len)
        attacked_output, calibrated_output, _ = self.forward(seq)
        B, L1 = seq.shape
        idx = torch.arange(B, device=seq.device) * L1 + item_seq_len            # gather_indexes(output, item_seq_len)
        both = ops.GatherRowsFn.apply(torch.cat((attacked_output.reshape(B * L1, -1), calibrated_output.reshape(B * L1, -1))),
                                      torch.cat((idx, idx + B * L1)))
        return both[:B], both[B:]

    def predict(self, interaction):
        """acbert4rec.py:247-258 -> (attacked_scores [B], scores [B])."""
        att, cal = self._test_outputs(interaction)
        e = self.item_embedding(interaction[self.ITEM_ID])
        return torch.mul(att, e).sum(dim=1), torch.mul(cal, e).sum(dim=1)

    def full_sort_predict(self, interaction):
        """acbert4rec.py:260-267 -> (attacked_scores [B, n_items], scores [B, n_items]) (the mask-token row is left out)."""
        att, cal = self._test_outputs(interaction)
        E = self.item_embedding.weight[:self.n_items]
        both = ops.logits_scores(torch.cat((att, cal)), E, self.logits_passes)
        B = att.shape[0]
        return both[:B], both[B:]

    def full_sort_topk(self, interaction, k, positive=None, counts=False):
        """fused scores -> scores[:,0] = -inf -> top-k -> hit flags of the calibrated stream (trainer.py:941-942, collector.py:145-153);
        counts=True: + the positive's rank counts [B, 2] (ops.full_sort_topk)"""
        _, cal = self._test_outputs(interaction)
        return ops.full_sort_topk(cal.contiguous(), self.item_embedding.weight[:self.n_items], k, positive, self.logits_passes,
                                  counts=counts)

    def sampled_topk(self, interaction, candidates, k, positive=None, counts=False):
        """sampled-candidate ranking of the calibrated stream (candidates [B, 1+N], positive in column 0, written there from
        `positive` when given) over the table without the mask-token row -> (scores [B, 1+N], rec_topk [B, k+1]) (+ counts [B, 3]
        of ops.candidate_rank with counts=True)"""
        if positive is not None:
            candidates[:, 0].copy_(positive)
        _, cal = self._test_outputs(interaction)
        r = ops.candidate_rank(cal, self.item_embedding.weight[:self.n_items], candidates, k, want_scores=True, want_counts=counts)
        return (r[1], r[0]) + tuple(r[2:])
