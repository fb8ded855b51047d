"""ACSASRecTrainer -- drop-in for recbole/trainer/trainer.py:505-1044 (AttackSASRecTrainer /
ACSASRecTrainer) restricted to what AC-SASRec uses: the adversarial two-loss step (:660-687), the
full-sort evaluation driver (:926-945, :964-1019) with the collector's top-k (evaluator/collector.py:
145-153), early stopping and the checkpoint format (:710-761, :809-924).

B200-native choices: parameters, gradients and Adam moments live in three flat fp32 buffers so the
optimizer is ONE fused kernel and zero_grad ONE memset; the whole step (H2D'd batch -> both losses ->
both routed backward passes -> Adam) is captured once in a CUDA graph and replayed, with dropout /
noise streams advanced on the device; evaluation uses the fused logits+top-k kernel, so neither
the [B,V] scores nor the [B,V] int pos_matrix of the reference exist.
"""
import contextlib
import os
import time
from logging import getLogger

import numpy as np
import torch

from . import ops
from .compat import Interaction, PackedInteraction, cfg_get
from .evaluator import Evaluator

ATTACK_KEYS = ('attack_key_transform', 'attack_query_transform')      # trainer.py:673


def is_attack_param(name):
    return any(k in name for k in ATTACK_KEYS)


def early_stopping(value, best, cur_step, max_step, bigger=True):
    """recbole/utils/utils.py:103-144."""
    stop_flag = update_flag = False
    better = value >= best if bigger else value <= best
    if better:
        cur_step, best, update_flag = 0, value, True
    else:
        cur_step += 1
        if cur_step > max_step:
            stop_flag = True
    return best, cur_step, stop_flag, update_flag


class FlatAdam(object):
    """torch.optim.Adam semantics (trainer.py:614-615) over flat buffers; step() is one fused kernel.  With `clip` (device_clip of
    the `clip_grad_norm` setting) step() first clips the gradient as torch.nn.utils.clip_grad_norm_ does: one norm launch over the
    flat gradient, and the scale folded into the Adam kernel."""

    @staticmethod
    def device_clip(clip_grad_norm):
        """`clip_grad_norm` (clip_grad_norm_'s keyword arguments) -> (max_norm, norm_type) when step() can clip on the device, else
        None (unset, or settings only torch's clip_grad_norm_ handles: other keys such as error_if_nonfinite, which needs a host
        sync, norm_type <= 0, max_norm <= 0)"""
        if not isinstance(clip_grad_norm, dict) or 'max_norm' not in clip_grad_norm or set(clip_grad_norm) - {'max_norm', 'norm_type'}:
            return None
        try:
            max_norm, norm_type = float(clip_grad_norm['max_norm']), float(clip_grad_norm.get('norm_type', 2.0))
        except (TypeError, ValueError):
            return None
        return (max_norm, norm_type) if max_norm > 0 and norm_type > 0 else None

    def __init__(self, model, lr, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8, clip=None):
        params = [p for p in model.parameters()]
        dev = params[0].device
        align = 64                      # floats: every group starts on a 256-byte boundary (float4 / bulk-copy loads)
        # groups of parameters that must be adjacent (no padding) so they can be viewed as one stacked tensor
        groups, seen = [], set()
        for g in (model.flat_groups() if hasattr(model, 'flat_groups') else []):
            groups.append(list(g))
            seen.update(id(p) for p in g)
        layout = []
        gi = {id(g[0]): g for g in groups}
        for p in params:
            if id(p) in gi:
                layout.append(gi[id(p)])
            elif id(p) not in seen:
                layout.append([p])
        n = sum((sum(p.numel() for p in g) + align - 1) // align * align for g in layout)
        self.flat_param = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        self.step_count = torch.zeros(1, dtype=torch.int64, device=dev)
        self.offsets = {}
        off = 0
        with torch.no_grad():
            for g in layout:
                start = off
                for p in g:
                    k = p.numel()
                    if k % 4:
                        off = (off + 3) // 4 * 4
                    self.flat_param[off:off + k].copy_(p.data.reshape(-1))
                    p.data = self.flat_param[off:off + k].view(p.shape)
                    p.grad = self.flat_grad[off:off + k].view(p.shape)
                    self.offsets[id(p)] = off
                    off += k
                off = start + (off - start + align - 1) // align * align
        assert off <= n + align * len(layout)
        self.lr, self.weight_decay, self.betas, self.eps = float(lr), float(weight_decay or 0.0), betas, eps
        self.params = params
        if self.flat_param.is_cuda:
            # parameters: only this optimizer (the last node of a step) writes them -> kernels may read them ahead of
            # programmatic dependent launch synchronisation
            from ._lib import LIB
            LIB.query('acsr_register_static', self.flat_param.data_ptr(), self.flat_param.numel() * 4)
        self.no_grad_params = [p for n, p in model.named_parameters() if n == 'mask_loss_weight']
        self.clip = clip
        self._table_shard = None
        self._norm_partial = ops.grad_norm_partial       # the local norm kernel (the CPU gloo tests put a torch restatement here)
        if clip is not None:
            self._norm_work = ops.grad_norm_work(dev) if self.flat_param.is_cuda else None
            self._norm_parts = torch.zeros(2, dtype=torch.float64, device=dev)
            self.grad_norm = torch.zeros(1, dtype=torch.float32, device=dev)      # the total norm of the last step

    def stacked(self, plist, grad=False):
        """view of adjacent, equally shaped parameters (or their grads) as one [len, *shape] tensor; None if not adjacent."""
        k = plist[0].numel()
        off0 = self.offsets[id(plist[0])]
        for i, p in enumerate(plist):
            if p.shape != plist[0].shape or self.offsets[id(p)] != off0 + i * k:
                return None
        src = self.flat_grad if grad else self.flat_param
        return src[off0:off0 + len(plist) * k].view(len(plist), *plist[0].shape)

    def slot(self, p):
        """[begin, end) of the flat buffers reserved for a parameter that forms a group of its own (its padding included)"""
        a = self.offsets[id(p)]
        return a, a + (p.numel() + 63) // 64 * 64

    def set_table_shard(self, table, own_elems, all_gather):
        """the item table `table` is this rank's shard of a vocab-sharded table: its first own_elems gradient entries are this rank's
        rows, the rest of its slot is padding, and every other parameter is replicated.  The clip norm then combines the partial of
        the replicated ranges with every rank's shard partial, all_gather(t [1]) -> [world, 1] collecting those in rank order."""
        a, b = self.slot(table)
        self._table_shard = ([(0, a), (b, self.flat_grad.numel())], (a, a + int(own_elems)), all_gather)

    def _clip_partials(self):
        """-> float64 [n] norm partials of the whole (logical) gradient, combined in index order by the clipped Adam"""
        q, norm = self.clip[1], self._norm_partial
        if self._table_shard is None:
            return norm(self.flat_grad, q, out=self._norm_parts[:1], work=self._norm_work)
        replicated, own, all_gather = self._table_shard
        norm(self.flat_grad, q, [r for r in replicated if r[1] > r[0]] or [(0, 0)], out=self._norm_parts[:1], work=self._norm_work)
        norm(self.flat_grad, q, [own], out=self._norm_parts[1:], work=self._norm_work)
        return torch.cat((self._norm_parts[:1], all_gather(self._norm_parts[1:]).view(-1)))

    def zero_grad(self, set_to_none=False):
        self.flat_grad.zero_()

    def step(self):
        # torch.optim.Adam skips parameters whose .grad is None -- in the reference that is a trainable mask_loss_weight, which
        # only enters the attacked loss and is routed away (trainer.py:672-686): with weight decay the flat kernel would
        # still shrink it, so its value is put back after the step
        keep = [(p, p.detach().clone()) for p in self.no_grad_params] if (self.weight_decay and self.no_grad_params) else []
        if self.clip is None:
            ops.adam_step(self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step_count, self.lr,
                          self.betas[0], self.betas[1], self.eps, self.weight_decay)
        else:
            ops.adam_step_clipped(self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step_count, self.lr,
                                  self._clip_partials(), self.clip[1], self.clip[0], self.betas[0], self.betas[1], self.eps,
                                  self.weight_decay, total=self.grad_norm)
        for p, v in keep:
            p.data.copy_(v)

    def _view(self, flat, p):
        off = self.offsets[id(p)]
        return flat[off:off + p.numel()].view(p.shape)

    def state_dict(self, gather=None):
        """torch.optim.Adam's format (trainer.py:718-728 saves `self.optimizer.state_dict()`): per-parameter step / exp_avg /
        exp_avg_sq indexed by the position in model.parameters(), one param group -- a checkpoint written here resumes in
        the reference trainer and vice versa."""
        step = int(self.step_count.item())
        state = {}
        if step > 0:
            for i, p in enumerate(self.params):
                ea, es = self._view(self.exp_avg, p).detach(), self._view(self.exp_avg_sq, p).detach()
                if gather is not None:            # vocab-sharded item table: moments gathered into the reference layout
                    ea, es = gather(p, ea), gather(p, es)
                state[i] = {'step': torch.tensor(float(step)), 'exp_avg': ea.cpu().clone(), 'exp_avg_sq': es.cpu().clone()}
        group = {'lr': self.lr, 'betas': tuple(self.betas), 'eps': self.eps, 'weight_decay': self.weight_decay, 'amsgrad': False,
                 'maximize': False, 'foreach': None, 'capturable': False, 'differentiable': False, 'fused': None,
                 'params': list(range(len(self.params)))}
        return {'state': state, 'param_groups': [group]}

    def load_state_dict(self, sd, scatter=None):
        """accepts torch.optim.Adam's state_dict (a reference checkpoint's 'optimizer' entry) or the round-1 flat format"""
        if sd.get('flat_adam'):                       # checkpoints written by the first version of this trainer
            if sd['exp_avg'].numel() != self.exp_avg.numel():
                raise ValueError('flat optimizer state has %d elements, this model needs %d' % (sd['exp_avg'].numel(), self.exp_avg.numel()))
            self.exp_avg.copy_(sd['exp_avg'])
            self.exp_avg_sq.copy_(sd['exp_avg_sq'])
            self.step_count.fill_(sd['step'])
            return
        if 'state' not in sd or 'param_groups' not in sd:
            raise ValueError('optimizer state is neither a torch.optim.Adam state_dict nor a FlatAdam one')
        order = [i for g in sd['param_groups'] for i in g['params']]
        if len(order) != len(self.params):
            raise ValueError('optimizer state covers %d parameters, this model has %d' % (len(order), len(self.params)))
        steps = set()
        self.exp_avg.zero_()
        self.exp_avg_sq.zero_()
        for pos, key in enumerate(order):
            st = sd['state'].get(key)
            if st is None:                            # parameter that never received a gradient (torch keeps no state for it)
                continue
            p = self.params[pos]
            if scatter is not None:               # vocab-sharded item table: keep this rank's rows of the full-size moments
                st = dict(st, exp_avg=scatter(p, st['exp_avg']), exp_avg_sq=scatter(p, st['exp_avg_sq']))
            if tuple(st['exp_avg'].shape) != tuple(p.shape):
                raise ValueError('optimizer state %s has shape %s, parameter %d has %s' % (key, tuple(st['exp_avg'].shape), pos, tuple(p.shape)))
            self._view(self.exp_avg, p).copy_(st['exp_avg'])
            self._view(self.exp_avg_sq, p).copy_(st['exp_avg_sq'])
            steps.add(int(float(st['step'])))
        if len(steps) > 1:
            raise ValueError('per-parameter step counts differ (%s): not representable by the single-step flat Adam' % sorted(steps))
        self.step_count.fill_(steps.pop() if steps else 0)
        g0 = sd['param_groups'][0]
        self.lr, self.betas, self.eps = float(g0.get('lr', self.lr)), tuple(g0.get('betas', self.betas)), float(g0.get('eps', self.eps))
        self.weight_decay = float(g0.get('weight_decay', self.weight_decay) or 0.0)


class ACSASRecTrainer(object):
    def __init__(self, config, model):
        self.config, self.model = config, model
        self.logger = getLogger()
        self.learner = cfg_get(config, 'learner', 'adam')
        self.learning_rate = config['learning_rate']
        self.epochs = config['epochs']
        self.eval_step = min(cfg_get(config, 'eval_step', 1), self.epochs)
        self.stopping_step = cfg_get(config, 'stopping_step', 10)
        self.clip_grad_norm = config['clip_grad_norm']
        self.valid_metric = str(cfg_get(config, 'valid_metric', 'MRR@10')).lower()
        self.valid_metric_bigger = cfg_get(config, 'valid_metric_bigger', True)
        self.test_batch_size = config['eval_batch_size']
        self.device = config['device']
        self.checkpoint_dir = cfg_get(config, 'checkpoint_dir', 'saved')
        os.makedirs(self.checkpoint_dir, exist_ok=True)
        self.saved_model_file = os.path.join(self.checkpoint_dir, '{}-{}.pth'.format(
            cfg_get(config, 'model', 'ACSASRec'), time.strftime('%b-%d-%Y_%H-%M-%S')))
        self.weight_decay = cfg_get(config, 'weight_decay', 0.0)
        self.start_epoch, self.cur_step = 0, 0
        self.best_valid_score = -np.inf if self.valid_metric_bigger else np.inf
        self.best_valid_result = None
        self.train_loss_dict = dict()
        self.optimizer = self._build_optimizer()
        self.evaluator = Evaluator(config)
        self.topk = list(config['topk'])
        self.tot_item_num = None
        self.use_graph = bool(cfg_get(config, 'cuda_graph', True))
        self.fused_topk = bool(cfg_get(config, 'fused_topk', True))
        self._graph = None
        self._dgraph = None
        self._eval_graphs = {}
        self.dp_world = 1
        self.fused = None
        if (bool(cfg_get(config, 'fused_step', True)) and isinstance(self.optimizer, FlatAdam) and type(model).__name__ == 'ACSASRec'
                and getattr(model, 'loss_type', None) in ('CE', 'BPR') and not self.torch_clip):
            from .fused_step import FusedTrainStep
            self.fused = FusedTrainStep(model, self.optimizer)
            model._fused_step = self.fused          # eval batches reuse the fused forward (ACSASRec._encode)
        if self.clip_grad_norm:
            self.logger.info('clip_grad_norm by torch.nn.utils.clip_grad_norm_' if self.torch_clip else
                             'clip_grad_norm on the device (%s step)' % ('fused' if self.fused is not None else 'autograd'))
        self.nan_check_interval = int(cfg_get(config, 'nan_check_interval', 50))
        # BPR with `neg_sampling` on host-side batches: the ops.NegSampler that draws each step's negatives on the device
        # (set from the training loader by _train_epoch; a DeviceTrainDataLoader draws inside its own gather instead)
        self.train_neg_sampler = None
        # training rows per target item (RecBole's data.count_items, collected from the training data by fit / set_item_counts):
        # AveragePopularity and TailPercentage read it
        self.item_counts = None
        self.logger.info('use attack trainer!!!')

    # ------------------------------------------------------------------------------------------
    def _build_optimizer(self, **kwargs):
        learner = str(kwargs.pop('learner', self.learner)).lower()
        lr = kwargs.pop('learning_rate', self.learning_rate)
        wd = kwargs.pop('weight_decay', self.weight_decay)
        if learner == 'adam':
            return FlatAdam(self.model, lr, wd, clip=FlatAdam.device_clip(self.clip_grad_norm))
        import torch.optim as optim         # other learners are outside the hot path: library optimizers
        params = self.model.parameters()
        if learner == 'sgd':
            return optim.SGD(params, lr=lr, weight_decay=wd or 0.0)
        if learner == 'adagrad':
            return optim.Adagrad(params, lr=lr, weight_decay=wd or 0.0)
        if learner == 'rmsprop':
            return optim.RMSprop(params, lr=lr, weight_decay=wd or 0.0)
        self.logger.warning('Received unrecognized optimizer, set default Adam optimizer')
        return FlatAdam(self.model, lr, 0.0, clip=FlatAdam.device_clip(self.clip_grad_norm))

    @property
    def torch_clip(self):
        """`clip_grad_norm` is set and the optimizer does not clip on the device (FlatAdam.device_clip): the step calls
        torch.nn.utils.clip_grad_norm_, which rules out the fused step and the captured graph"""
        return bool(self.clip_grad_norm) and getattr(self.optimizer, 'clip', None) is None

    def _route(self, attack):
        for name, p in self.model.named_parameters():
            p.requires_grad = is_attack_param(name) == attack

    def _step_body(self, interaction):
        """trainer.py:660-687 without the host syncs: -> (attacked_loss, calibrated_loss) tensors."""
        if self.fused is not None:
            attacked_loss, calibrated_loss = self.fused(interaction)      # both cotangent streams in one pass
            if self.dp_world > 1:
                self._allreduce_grads()
            self.optimizer.step()
            return attacked_loss.detach(), calibrated_loss.detach()
        self.optimizer.zero_grad()
        attacked_loss, calibrated_loss = self.model.calculate_loss(interaction)
        # parameter gradients go straight into the optimizer's gradient buffer (ops.direct_param_grads)
        with (ops.direct_param_grads() if isinstance(self.optimizer, FlatAdam) else contextlib.nullcontext()):
            self._route(attack=False)
            calibrated_loss.backward(retain_graph=True)
            if attacked_loss is not None:
                self._route(attack=True)
                attacked_loss.backward()
        for p in self.model.parameters():
            p.requires_grad = True
        if self.dp_world > 1:               # batch data-parallel: average the flat gradient over ranks (NCCL / NVLink)
            self._allreduce_grads()
        if self.torch_clip:
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), **self.clip_grad_norm)
        self.optimizer.step()
        return attacked_loss.detach(), calibrated_loss.detach()

    def enable_data_parallel(self, vocab_parallel=False, shard_table=None):
        """One process per GPU: broadcast rank 0's weights, then all-reduce gradients every step (batch data-parallel).
        vocab_parallel=True additionally splits the full-catalogue logits / CE / top-k by item rows across ranks
        (dist.VocabParallel: all-gather of `out`, all-gather of per-row (max, sum-exp, target logit), reduce-scatter of d_out);
        under loss_type BPR the two table rows of each row are scored by their owners (reduce-scatter of the dots and of d_out),
        and sampled evaluation scores each candidate on its owner's rows.
        shard_table=True (default for catalogues above the break-even 2*W*B*L rows, see dist.py) also shards the STORAGE: this
        rank keeps rows [lo, hi) of the item table, their gradient and their Adam moments; the embedding rows of its own tokens
        are exchanged every step and the data-parallel all-reduce shrinks to the encoder parameters."""
        import torch.distributed as dist
        if not isinstance(self.optimizer, FlatAdam):
            raise ValueError('data-parallel training needs the flat Adam optimizer')
        self.dp_world = dist.get_world_size()
        dist.broadcast(self.optimizer.flat_param, src=0)
        self.vp = None
        if not vocab_parallel:
            return
        if self.fused is None:
            raise ValueError('vocab-parallel logits need the fused step (loss_type CE or BPR)')
        from .dist import VocabParallel, CudaCompute
        m = self.model
        if shard_table is None:
            L = int(cfg_get(self.config, 'MAX_ITEM_LIST_LENGTH', 50))
            shard_table = m.n_items > 2 * self.dp_world * int(self.config['train_batch_size']) * L
        self.vp = VocabParallel(m.n_items, compute=CudaCompute(m.logits_passes, m.hidden_size), sharded=bool(shard_table))
        if shard_table:
            # swap the replicated table for this rank's shard and rebuild the flat optimizer state around it
            full = m.item_embedding.weight.detach()
            shard = self.vp.make_shard(full)
            step = int(self.optimizer.step_count.item())
            if step != 0:
                raise ValueError('shard the item table before the first optimisation step (or resume from a checkpoint afterwards)')
            m.item_embedding.weight = torch.nn.Parameter(shard)
            del full
            self.optimizer = self._build_optimizer()
            E = m.item_embedding.weight
            self.optimizer.set_table_shard(E, (self.vp.hi - self.vp.lo) * E.shape[1], self.vp._all_gather)
            from .fused_step import FusedTrainStep
            self.fused = FusedTrainStep(m, self.optimizer)
            m._fused_step = self.fused
            self._graph, self._eval_graphs = None, {}
            torch.cuda.empty_cache()
        self.fused.vp = self.vp
        m._vp = self.vp                           # eval: sharded top-k (ACSASRec.full_sort_topk / full_sort_predict)

    def _allreduce_grads(self):
        """average the gradients over the ranks (NCCL over NVLink).  With a sharded item table its gradient shard is already the
        owner's sum over all ranks' rows: only the other (replicated, encoder) parameters are all-reduced."""
        import torch.distributed as dist
        g = self.optimizer.flat_grad
        if self.vp is not None and self.vp.sharded:
            a, b = self.optimizer.slot(self.model.item_embedding.weight)
            if a > 0:
                dist.all_reduce(g[:a])
            if b < g.numel():
                dist.all_reduce(g[b:])
        else:
            dist.all_reduce(g)
        g.mul_(1.0 / self.dp_world)

    def train_step(self, interaction):
        """One optimisation step on a device-resident Interaction (eager launch path)."""
        return self._step_body(self._draw_negatives(interaction))

    def _needs_negatives(self, interaction):
        return self.train_neg_sampler is not None and self.model.NEG_ITEM_ID not in interaction

    def _draw_negatives(self, interaction):
        """a device batch without negatives under BPR + `neg_sampling`: the same batch plus one negative per row, drawn on the
        device by the training sampler (recbole/data/dataloader/general_dataloader.py's neg_sample_by, sampler.py)"""
        if not self._needs_negatives(interaction):
            return interaction
        m = self.model
        f = dict(interaction.interaction)
        f[m.NEG_ITEM_ID] = self.train_neg_sampler.draw(interaction[m.USER_ID], 1, positives=interaction[m.POS_ITEM_ID]).view(-1)
        return Interaction(f)

    # -------- CUDA-graph replay of the whole step ----------------------------------------------
    def _graph_key(self, interaction):
        return tuple((k, tuple(interaction[k].shape)) for k in self._fields() if k in interaction)

    def _fields(self):
        m = self.model
        f = [m.ITEM_SEQ, m.ITEM_SEQ_LEN, m.POS_ITEM_ID]
        if m.loss_type == 'BPR':
            f.append(m.NEG_ITEM_ID)
        if self.train_neg_sampler is not None and m.USER_ID not in f:
            f.append(m.USER_ID)                    # read by the negative sampler
        return f + [k for k in getattr(m, 'EXTRA_FIELDS', []) if k not in f]      # ACSSEPT: user id; ACTiSASRec: time stamps

    def _capture(self, interaction=None, loader=None):
        """capture the whole step as one CUDA graph.  interaction: the batch arrives by a copy into the static input buffers
        before each replay; loader (data.DeviceTrainDataLoader): the batch is gathered from the HBM-resident data by the first
        two nodes of the graph itself (acsr_batch_gather + acsr_cursor_advance) -- a replay needs no input at all."""
        dev = self.device
        m = self.model
        # BPR + neg_sampling on host batches: the static buffers get a neg slot the sampler fills inside the graph
        draw = loader is None and self._needs_negatives(interaction)
        present = [k for k in self._fields() if loader is not None or k in interaction]
        # static input buffers: one flat buffer with the fields as views, so a packed host batch arrives as ONE copy
        if loader is not None:
            lay, total = loader.layout()
        else:
            lay, total = None, 0
            if all(interaction[k].dtype == torch.int64 for k in present):
                lay, total = PackedInteraction.layout_of({k: interaction[k] for k in present})
                if draw:
                    B = int(interaction[m.POS_ITEM_ID].shape[0])
                    lay, total = lay + [(m.NEG_ITEM_ID, total, (B,))], total + B
        if loader is None and lay is None:        # a float field (ACTiSASRec's time stamps): one static tensor per field
            f = {k: torch.empty_like(interaction[k], device=dev) for k in present}
            if draw:
                f[m.NEG_ITEM_ID] = torch.empty_like(interaction[m.POS_ITEM_ID], device=dev)
            static_inter = Interaction(f)
        else:
            static_inter = PackedInteraction(torch.empty(total, dtype=torch.int64, device=dev), lay)
        static = {k: static_inter[k] for k in self._fields() if k in static_inter}
        if loader is None:
            for k in present:
                static[k].copy_(interaction[k])
        self.model._runtime(dev)               # creates the device RNG state, so the snapshot below covers it
        sampler = self.train_neg_sampler if draw else None
        if sampler is not None:
            sampler.to_device(dev)

        def body():
            if loader is not None:
                loader.gather_into(static_inter.packed)
            if sampler is not None:
                sampler.draw(static_inter[m.USER_ID], 1, positives=static_inter[m.POS_ITEM_ID],
                             out=static_inter[m.NEG_ITEM_ID].view(-1, 1), ld=1)
            return self._step_body(static_inter)
        loader_sampler = getattr(loader, 'neg_sampler', None) if loader is not None else None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):          # warm-up on a side stream (allocator + lazy inits), state restored after
            if loader_sampler is not None:
                loader_sampler.to_device(dev)
            rngs = [s.rng.state for s in (sampler, loader_sampler) if s is not None]
            snap = (self.optimizer.flat_param.clone(), self.optimizer.exp_avg.clone(), self.optimizer.exp_avg_sq.clone(),
                    self.optimizer.step_count.clone(), self.model._rng.state.clone() if self.model._rng else None,
                    loader.cursor.clone() if loader is not None else None, [r.clone() for r in rngs])
            for _ in range(2):
                body()
            self.optimizer.flat_param.copy_(snap[0]); self.optimizer.exp_avg.copy_(snap[1])
            self.optimizer.exp_avg_sq.copy_(snap[2]); self.optimizer.step_count.copy_(snap[3])
            if snap[4] is not None:
                self.model._rng.state.copy_(snap[4])
            if snap[5] is not None:
                loader.cursor.copy_(snap[5])
            for r, v in zip(rngs, snap[6]):
                r.copy_(v)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            la, lc = body()
        rec = dict(graph=g, static=static, static_inter=static_inter, la=la, lc=lc)
        if loader is not None:
            self._dgraph = dict(rec, loader=loader)
        else:
            self._graph = dict(rec, key=self._graph_key(interaction), sampler=sampler)

    def device_loader_step(self, loader):
        """one optimisation step on the next batch of a data.DeviceTrainDataLoader: a bare graph replay (the batch is gathered
        from HBM inside the graph; nothing crosses PCIe).  -> (attacked_loss, calibrated_loss) device tensors."""
        dg = getattr(self, '_dgraph', None)
        if dg is None or dg['loader'] is not loader:
            self._capture(loader=loader)
            dg = self._dgraph
        dg['graph'].replay()
        return dg['la'], dg['lc']

    def _host_schedule(self):
        """combine_option 'annealing' (layers.py:889-891): the mixing rate exp(-anneal_step / 1e5) is a host float that changes
        with EVERY forward, train or eval.  A captured graph would freeze it, so such models always launch eagerly."""
        enc = getattr(self.model, 'trm_encoder', None) or getattr(self.model, 'ti_trm_encoder', None)
        return enc is not None and any(getattr(l, 'combine_option', None) == 'annealing' for l in enc.layer)

    def graphed_step(self, interaction):
        """interaction: host (pinned) or device tensors of the captured shape.  Copies the batch into the
        static buffers on the current stream and replays the captured step."""
        if self._host_schedule() or int(interaction[self.model.ITEM_SEQ].shape[1]) > 64:
            # annealing: see _host_schedule; sequences longer than 64: the attention backward's workspace may have to grow
            return self.train_step(interaction.to(self.device))
        if self.fused is None and hasattr(self.model, 'prepare_batch'):
            if self._graph is not None and self._graph['key'][0][1] != tuple(interaction[self.model.ITEM_SEQ].shape):
                return self._step_body(interaction.to(self.device))      # ragged last batch: eager launch (masks itself)
            interaction = self.model.prepare_batch(interaction)          # host half of the step (AcBERT4Rec's python masking)
        if self._graph is not None and self._graph['sampler'] is not (self.train_neg_sampler if self._needs_negatives(interaction) else None):
            self._graph = None                     # the captured step draws from another sampler's device state: capture anew
        if self._graph is None or self._graph['key'] != self._graph_key(interaction):
            if self._graph is not None:
                return self.train_step(interaction.to(self.device))      # ragged last batch: eager launch
            self._capture(interaction)
        si = self._graph['static_inter']
        lay = getattr(interaction, 'layout', None)
        if lay is not None and lay == getattr(si, 'layout', [])[:len(lay)]:
            # packed batch: one copy (a trailing neg slot the captured sampler fills is not part of it)
            si.packed[:interaction.packed.numel()].copy_(interaction.packed, non_blocking=True)
        else:
            st = self._graph['static']
            for k in st:
                if k in interaction:
                    st[k].copy_(interaction[k], non_blocking=True)
        self._graph['graph'].replay()
        return self._graph['la'], self._graph['lc']

    # ------------------------------------------------------------------------------------------
    def _check_nan(self, loss):
        if torch.isnan(loss):
            raise ValueError('Training loss is nan')

    def _train_epoch(self, train_data, epoch_idx, loss_func=None, show_progress=False, attack=True, calibrate=True):
        assert attack or calibrate
        self.model.train()
        tot_a = torch.zeros((), dtype=torch.float64, device=self.device)
        tot_c = torch.zeros((), dtype=torch.float64, device=self.device)
        # the captured step: AC-SASRec's fused one-pass step, or -- for sibling models whose step has no host-side work
        # (GRAPH_SAFE_STEP) -- the autograd Functions' forward + routed double backward + Adam as they launch
        graph_ok = (self.use_graph and (self.fused is not None or getattr(self.model, 'GRAPH_SAFE_STEP', False))
                    and isinstance(self.optimizer, FlatAdam) and not self.torch_clip)
        if not getattr(train_data, 'device_resident', False):
            self.train_neg_sampler = getattr(train_data, 'neg_sampler', None)
        if (getattr(train_data, 'device_resident', False) and graph_ok and self.fused is not None and not self._host_schedule()
                and train_data.L <= 64 and train_data.full_batches > 0):
            # HBM-resident data (f-2): the epoch is graph replays + one eager step for the ragged tail
            train_data.new_epoch()
            for batch_idx in range(train_data.full_batches):
                la, lc = self.device_loader_step(train_data)
                tot_a += la
                tot_c += lc
                if self.nan_check_interval and (batch_idx + 1) % self.nan_check_interval == 0:
                    self._check_nan(tot_a + tot_c)
            tail = train_data.tail_batch()
            if tail is not None:
                la, lc = self.train_step(tail)
                tot_a += la
                tot_c += lc
            self._check_nan(tot_a + tot_c)
            return float(tot_a.item()), float(tot_c.item())
        for batch_idx, interaction in enumerate(train_data):
            if graph_ok:
                la, lc = self.graphed_step(interaction)
            else:
                la, lc = self.train_step(interaction.to(self.device))
            tot_a += la
            tot_c += lc
            if self.nan_check_interval and (batch_idx + 1) % self.nan_check_interval == 0:
                self._check_nan(tot_a + tot_c)
        self._check_nan(tot_a + tot_c)
        return float(tot_a.item()), float(tot_c.item())

    def _valid_epoch(self, valid_data, show_progress=False):
        valid_result = self.evaluate(valid_data, load_best_model=False, show_progress=show_progress)
        return valid_result[self.valid_metric] if self.valid_metric else valid_result['recall@10'], valid_result

    def _save_checkpoint(self, epoch, verbose=True, **kwargs):
        """trainer.py:710-731: same keys; 'optimizer' is in torch.optim.Adam's state_dict format (FlatAdam.state_dict)."""
        saved_model_file = kwargs.pop('saved_model_file', self.saved_model_file)
        state = {
            'config': self.config, 'epoch': epoch, 'cur_step': self.cur_step, 'best_valid_score': self.best_valid_score,
            'state_dict': self._full_state_dict(),
            'other_parameter': self.model.other_parameter(), 'optimizer': self.optimizer.state_dict(gather=self._gather_fn()),
        }
        torch.save(state, saved_model_file)
        if verbose:
            self.logger.info('Saving current: %s' % saved_model_file)

    def _sharded(self):
        return getattr(self, 'vp', None) is not None and self.vp.sharded

    def _gather_fn(self):
        """-> fn(param, tensor_of_param_shape) -> tensor in the reference layout: the item table's shard (or its moments) is
        gathered into the full [V, d] table; every rank takes part in the collective"""
        if not self._sharded():
            return None
        E = self.model.item_embedding.weight
        return lambda p, t: self.vp.gather_full(t) if p is E else t

    def _full_state_dict(self):
        """the model's state_dict in the reference layout (a sharded item table is gathered: SURVEY section 5, checkpoints)"""
        sd = {k: v.detach() for k, v in self.model.state_dict().items()}
        if self._sharded():
            sd['item_embedding.weight'] = self.vp.gather_full(sd['item_embedding.weight'])
        return {k: v.cpu().clone() for k, v in sd.items()}

    def _load_state(self, state_dict):
        with torch.no_grad():               # copy in place: parameters are views of the flat buffer
            own = self.model.state_dict()
            missing = set(own) - set(state_dict)
            if missing:
                raise KeyError('missing keys in checkpoint: %s' % sorted(missing))
            for k, v in own.items():
                src = state_dict[k]
                if k == 'item_embedding.weight' and self._sharded():
                    src = self.vp.make_shard(src.to(v.device))
                v.copy_(src)

    def resume_checkpoint(self, resume_file):
        """trainer.py:733-761."""
        resume_file = str(resume_file)
        self.saved_model_file = resume_file
        checkpoint = torch.load(resume_file, map_location='cpu', weights_only=False)
        self.start_epoch = checkpoint['epoch'] + 1
        self.cur_step = checkpoint['cur_step']
        self.best_valid_score = checkpoint['best_valid_score']
        self._load_state(checkpoint['state_dict'])
        self.model.load_other_parameter(checkpoint.get('other_parameter'))
        scatter = None
        if self._sharded():
            E = self.model.item_embedding.weight
            scatter = lambda p, t: self.vp.make_shard(t.to(E.device)) if p is E else t      # noqa: E731
        self.optimizer.load_state_dict(checkpoint['optimizer'], scatter=scatter)
        self.logger.info('Checkpoint loaded. Resume training from epoch {}'.format(self.start_epoch))

    def set_item_counts(self, train_data):
        """record the training item counts the popularity metrics need (collector.py data_collect(train_data): data.count_items)
        from a training loader or dataset (its inter_feat item ids), or take them as an array indexed by item id"""
        ds = getattr(train_data, 'dataset', train_data)
        feat = getattr(ds, 'inter_feat', None)
        if feat is not None:
            ids = feat[ds.iid_field]
            ids = (ids.cpu() if torch.is_tensor(ids) else torch.as_tensor(ids)).to(torch.int64).reshape(-1)
            n = int(getattr(ds, 'item_num', 0) or 0)
            self.item_counts = np.bincount(ids.numpy(), minlength=n).astype(np.int64)
        else:
            self.item_counts = np.asarray(train_data, dtype=np.int64)

    def fit(self, train_data, valid_data=None, verbose=True, saved=True, show_progress=False, callback_fn=None):
        """trainer.py:809-924 (epoch range 2*epochs, eval every eval_step, early stopping, checkpoint on improvement)."""
        self.set_item_counts(train_data)
        if saved and self.start_epoch >= self.epochs:
            self._save_checkpoint(-1, verbose=verbose)
        for epoch_idx in range(self.start_epoch, 2 * self.epochs):
            t0 = time.time()
            a, c = self._train_epoch(train_data, epoch_idx, show_progress=show_progress)
            self.train_loss_dict[epoch_idx] = (a, c)
            t1 = time.time()
            if verbose:
                des = self.config['loss_decimal_place'] or 4
                self.logger.info(('epoch %d training [time: %.2fs, train loss: %.' + str(des) + 'f]') % (epoch_idx, t1 - t0, a))
                self.logger.info(('epoch %d training [time: %.2fs, train loss: %.' + str(des) + 'f]') % (epoch_idx, t1 - t0, c))
            if self.eval_step <= 0 or not valid_data:
                if saved:
                    self._save_checkpoint(epoch_idx, verbose=verbose)
                continue
            if (epoch_idx + 1) % self.eval_step == 0:
                v0 = time.time()
                valid_score, valid_result = self._valid_epoch(valid_data, show_progress=show_progress)
                self.best_valid_score, self.cur_step, stop_flag, update_flag = early_stopping(
                    valid_score, self.best_valid_score, self.cur_step, max_step=self.stopping_step,
                    bigger=self.valid_metric_bigger)
                if verbose:
                    self.logger.info('epoch %d evaluating [time: %.2fs, valid_score: %f]' % (epoch_idx, time.time() - v0, valid_score))
                    self.logger.info('valid result: \n' + '    '.join('%s : %s' % kv for kv in valid_result.items()))
                if update_flag:
                    if saved:
                        self._save_checkpoint(epoch_idx, verbose=verbose)
                    self.best_valid_result = valid_result
                if callback_fn:
                    callback_fn(epoch_idx, valid_score)
                if stop_flag:
                    if verbose:
                        self.logger.info('Finished training, best eval result in epoch %d' %
                                         (epoch_idx - self.cur_step * self.eval_step))
                    break
        return self.best_valid_score, self.best_valid_result

    # ------------------------------------------------------------------------------------------
    def _full_sort_batch_eval(self, batched_data):
        """trainer.py:926-945 with the API-compatible materialised scores (used when fused_topk is off)."""
        interaction, history_index, positive_u, positive_i = batched_data
        _, scores = self.model.full_sort_predict(interaction.to(self.device))
        scores = scores.view(-1, self.tot_item_num or self.model.n_items)
        scores[:, 0] = -np.inf
        if history_index is not None:
            scores[history_index] = -np.inf
        return interaction, scores, positive_u, positive_i

    def eval_batch(self, batched_data, rec_out=None, neg_sampler=None, neg_num=0, need=None):
        """-> rec_topk [B, kmax+1] int32 on the device (collector.py:145-153 'rec.topk'); with rec_out (a pinned host tensor)
        the graphed path copies the result straight into it (no device-side clone) and returns rec_out.  With neg_sampler (the
        batch of a data.NegSampleEvalDataLoader, `eval_args.mode: uniN / popN`): the positive is ranked against neg_num
        negatives drawn on the device (trainer.py _neg_sample_batch_eval, collector.py eval_batch_collect).
        need = (counts, items) with either set (what GAUC / the item-distribution metrics read): -> (rec, counts [B, 2] int32 | None,
        user_len [B] int32 | None, items [B, kmax] int32 | None) instead, all on the device (collector.py rec.meanrank / rec.items)."""
        interaction, history_index, positive_u, positive_i = batched_data
        kmax = max(self.topk)
        need = tuple(bool(x) for x in need) if need is not None and any(need) else None
        if neg_sampler is not None:
            return self._sampled_eval(interaction, positive_i, neg_sampler, int(neg_num), kmax, rec_out, need)
        if self.fused_topk and history_index is None:
            if kmax > 64:                      # the fused top-k keeps at most 64 candidates per row: materialised scores + torch.topk
                return self._eval_materialised(batched_data, kmax, rec_out, need)
            if self.use_graph and not self.model.training and not self._host_schedule():
                return self._graphed_eval(interaction, positive_i, kmax, rec_out, need)
            inter = interaction.to(self.device)
            pos = inter[self.model.POS_ITEM_ID] if positive_i is interaction.interaction.get(self.model.POS_ITEM_ID) else \
                positive_i.to(self.device, non_blocking=True)
            if need is not None:
                return self._collect_full(self.model.full_sort_topk(inter, kmax, pos, counts=need[0]), need, rec_out)
            _, _, rec = self.model.full_sort_topk(inter, kmax, pos)
        else:
            return self._eval_materialised(batched_data, kmax, rec_out, need)
        if rec_out is not None:
            rec_out.copy_(rec, non_blocking=True)
            return rec_out
        return rec

    def _n_items(self):
        return int(self.tot_item_num or self.model.n_items)

    def _collect_full(self, res, need, rec_out=None):
        """(val, idx, rec[, counts]) of a full-sort top-k -> (rec, counts, user_len, items) of eval_batch(need=...).  Every
        score but column 0 is finite in full sort, so user_len = n_items - 1 (collector.py: argmin of the sorted row)."""
        rec = res[2]
        if rec_out is not None:
            rec_out.copy_(rec, non_blocking=True)
            rec = rec_out
        counts = res[3] if need[0] else None
        user_len = torch.full((rec.shape[0],), self._n_items() - 1, dtype=torch.int32, device=res[1].device) if need[0] else None
        items = res[1].to(torch.int32) if need[1] else None
        return rec, counts, user_len, items

    def _eval_materialised(self, batched_data, kmax, rec_out=None, need=None):
        """trainer.py:926-945 + collector.py:145-153 on materialised scores (API-compatible path).  need: the rank counts are
        taken on the scores this path holds (the positive's own column left out), the ids are torch.topk's."""
        interaction, scores, positive_u, positive_i = self._full_sort_batch_eval(batched_data)
        _, topk_idx = torch.topk(scores, kmax, dim=-1)
        pos = positive_i.to(self.device)
        flags = (topk_idx == pos.view(-1, 1)).to(torch.int32)
        rec = torch.cat((flags, torch.ones_like(flags[:, :1])), dim=1)
        if rec_out is not None:
            rec_out.copy_(rec, non_blocking=True)
            rec = rec_out
        if need is None:
            return rec
        counts = user_len = None
        if need[0]:
            s_pos = scores.gather(1, pos.view(-1, 1))
            counts = torch.stack(((scores > s_pos).sum(1), (scores == s_pos).sum(1) - 1), 1).to(torch.int32)
            user_len = torch.isfinite(scores).sum(1).to(torch.int32)
        return rec, counts, user_len, (topk_idx.to(torch.int32) if need[1] else None)

    @torch.no_grad()
    def _graphed_eval(self, interaction, positive_i, kmax, rec_out=None, need=None):
        """forward + fused logits/top-k + hit flags of one eval batch as a CUDA-graph replay (one graph per batch shape, and per
        `need` of eval_batch).  The batch (host or device) is copied into static buffers; the returned tensors are fresh copies."""
        m = self.model
        fields = list(getattr(m, 'EVAL_FIELDS', None) or [m.ITEM_SEQ, m.ITEM_SEQ_LEN])      # ACSSEPT also reads the user id
        key = tuple(tuple(interaction[k].shape) for k in fields) + (kmax,) + ((need,) if need is not None else ())
        g = self._eval_graphs.get(key)
        if g is None:
            dev = self.device
            # static inputs (sequence, length, held-out item) as views of one flat buffer: a packed batch is ONE copy
            if all(interaction[k].dtype == torch.int64 for k in fields):
                lay, total = PackedInteraction.layout_of({**{k: interaction[k] for k in fields}, m.POS_ITEM_ID: positive_i})
                inter = PackedInteraction(torch.empty(total, dtype=torch.int64, device=dev), lay)
            else:                             # a float field (ACTiSASRec's time stamps): one static tensor per field
                inter = Interaction({**{k: torch.empty_like(interaction[k], device=dev) for k in fields},
                                     m.POS_ITEM_ID: torch.empty_like(positive_i, device=dev)})
            static = {k: inter[k] for k in fields}
            for k in fields:
                static[k].copy_(interaction[k])
            pos = inter[m.POS_ITEM_ID]
            pos.copy_(positive_i)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            def body():
                if need is None:
                    return m.full_sort_topk(inter, kmax, pos)[2], None
                return None, self._collect_full(m.full_sort_topk(inter, kmax, pos, counts=need[0]), need)
            with torch.cuda.stream(side):
                for _ in range(2):
                    body()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                rec, extra = body()
            if extra is not None:
                rec = extra[0]
            g = dict(graph=graph, static=static, pos=pos, rec=rec, inter=inter, extra=extra)
            self._eval_graphs[key] = g
        if getattr(interaction, 'layout', None) == getattr(g['inter'], 'layout', ()) and positive_i is interaction.interaction.get(m.POS_ITEM_ID):
            g['inter'].packed.copy_(interaction.packed, non_blocking=True)
        else:
            for k in fields:
                g['static'][k].copy_(interaction[k], non_blocking=True)
            g['pos'].copy_(positive_i, non_blocking=True)
        g['graph'].replay()
        return self._graph_result(g, rec_out)

    @staticmethod
    def _graph_result(g, rec_out):
        """copies of a replayed eval graph's outputs: rec (into rec_out when given), and with a `need` the other three of eval_batch"""
        if rec_out is not None:
            rec_out.copy_(g['rec'], non_blocking=True)
            rec = rec_out
        else:
            rec = g['rec'].clone()
        if g.get('extra') is None:
            return rec
        return (rec,) + tuple(t.clone() if t is not None else None for t in g['extra'][1:])

    def _sampled_body(self, inter, pos, cand, sampler, kmax, need=None):
        """negatives into cand[:, 1:] (the sampler's state advances), the positive into column 0, rank -> rec [B, kmax+1];
        need (counts only: the item-distribution metrics are not defined here): -> (rec, counts [B, 2], user_len [B], None)"""
        m = self.model
        N = cand.shape[1] - 1
        sampler.draw(inter[m.USER_ID], N, positives=pos, out=cand[:, 1:], ld=N + 1)
        if need is None:
            _, rec = m.sampled_topk(inter, cand, kmax, pos)
            return rec
        _, rec, counts = m.sampled_topk(inter, cand, kmax, pos, counts=True)
        return rec, counts[:, :2], counts[:, 2], None

    @torch.no_grad()
    def _sampled_eval(self, interaction, positive_i, sampler, N, kmax, rec_out=None, need=None):
        """one batch of sampled-candidate evaluation: sampler -> encoder -> acsr_candidate_rank, eagerly or as a CUDA-graph
        replay (one graph per batch shape and `need`; every replay draws fresh negatives).  Vocab-parallel: every rank draws its
        own rows' negatives and the graph captures the collectives of VocabParallel.sampled_rank."""
        m = self.model
        if need is not None and need[1]:
            raise NotImplementedError('the item-distribution metrics (ItemCoverage, AveragePopularity, GiniIndex, ShannonEntropy, '
                                      'TailPercentage) are not available in sampled evaluation (eval_args.mode uniN / popN): '
                                      'use full-sort evaluation for them')
        if not hasattr(m, 'sampled_topk'):
            raise NotImplementedError('%s has no sampled_topk: sampled evaluation is not available for it' % type(m).__name__)
        dev = self.device
        sampler.to_device(dev)
        if not (self.use_graph and not m.training and not self._host_schedule()):
            inter = interaction.to(dev)
            pos = positive_i.to(dev)
            cand = torch.empty((pos.shape[0], N + 1), dtype=torch.int64, device=dev)
            res = self._sampled_body(inter, pos, cand, sampler, kmax, need)
            rec = res if need is None else res[0]
            if rec_out is not None:
                rec_out.copy_(rec, non_blocking=True)
                rec = rec_out
            return rec if need is None else (rec,) + tuple(res[1:])
        fields = list(getattr(m, 'EVAL_FIELDS', None) or [m.ITEM_SEQ, m.ITEM_SEQ_LEN])
        if m.USER_ID not in fields:
            fields.append(m.USER_ID)
        # the graph captures the sampler's device state (used sets, alias table, Philox state): one graph per sampler, which the
        # record keeps alive so its id cannot be reused by another
        key = ('sampled', id(sampler), N, kmax) + tuple(tuple(interaction[k].shape) for k in fields) + ((need,) if need is not None else ())
        g = self._eval_graphs.get(key)
        own = getattr(interaction, 'layout', None) is not None and positive_i is interaction.interaction.get(m.POS_ITEM_ID)
        if g is None:
            if own and all(k in interaction for k in fields):
                # a packed loader batch: the static buffer takes the batch's own layout, so each replay's input is ONE copy
                inter = PackedInteraction(torch.empty(interaction.packed.numel(), dtype=torch.int64, device=dev), interaction.layout)
            elif all(interaction[k].dtype == torch.int64 for k in fields):
                lay, total = PackedInteraction.layout_of({**{k: interaction[k] for k in fields}, m.POS_ITEM_ID: positive_i})
                inter = PackedInteraction(torch.empty(total, dtype=torch.int64, device=dev), lay)
            else:                             # a float field (ACTiSASRec's time stamps): one static tensor per field
                inter = Interaction({**{k: torch.empty_like(interaction[k], device=dev) for k in fields},
                                     m.POS_ITEM_ID: torch.empty_like(positive_i, device=dev)})
            for k in fields:
                inter[k].copy_(interaction[k])
            pos = inter[m.POS_ITEM_ID]
            pos.copy_(positive_i)
            cand = torch.empty((pos.shape[0], N + 1), dtype=torch.int64, device=dev)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):      # warm-up; the sampler's state is put back so the graph starts where eager would
                snap = sampler.rng.state.clone()
                for _ in range(2):
                    self._sampled_body(inter, pos, cand, sampler, kmax, need)
                sampler.rng.state.copy_(snap)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                res = self._sampled_body(inter, pos, cand, sampler, kmax, need)
            rec, extra = (res, None) if need is None else (res[0], res)
            g = dict(graph=graph, pos=pos, rec=rec, inter=inter, cand=cand, fields=fields, sampler=sampler, extra=extra)
            self._eval_graphs[key] = g
        assert g['sampler'] is sampler
        if own and interaction.layout == getattr(g['inter'], 'layout', ()):
            g['inter'].packed.copy_(interaction.packed, non_blocking=True)
        else:
            for k in fields:
                g['inter'][k].copy_(interaction[k], non_blocking=True)
            g['pos'].copy_(positive_i, non_blocking=True)
        g['graph'].replay()
        return self._graph_result(g, rec_out)

    @torch.no_grad()
    def evaluate(self, eval_data, load_best_model=True, model_file=None, show_progress=False):
        """trainer.py:964-1019."""
        if not eval_data:
            return
        if load_best_model:
            checkpoint_file = model_file or self.saved_model_file
            checkpoint = torch.load(checkpoint_file, map_location='cpu', weights_only=False)
            self._load_state(checkpoint['state_dict'])
            self.model.load_other_parameter(checkpoint.get('other_parameter'))
            self.logger.info('Loading model structure and parameters from {}'.format(checkpoint_file))
        self.model.eval()
        self.tot_item_num = eval_data.dataset.item_num
        sampler = getattr(eval_data, 'neg_sampler', None)      # data.NegSampleEvalDataLoader: sampled-candidate evaluation
        ev = self.evaluator
        if ev.need_items and sampler is not None:
            raise NotImplementedError('the item-distribution metrics (ItemCoverage, AveragePopularity, GiniIndex, ShannonEntropy, '
                                      'TailPercentage) are not available in sampled evaluation (eval_args.mode uniN / popN): '
                                      'use full-sort evaluation for them')
        if ev.need_item_counts and self.item_counts is None:
            raise ValueError('AveragePopularity / TailPercentage need the training item counts: call fit(train_data) first, or '
                             'trainer.set_item_counts(train_data) (a training loader, its dataset, or an array of counts by item id)')
        if not (ev.need_counts or ev.need_items):
            recs = [self.eval_batch(b, neg_sampler=sampler, neg_num=getattr(eval_data, 'neg_num', 0)) for b in eval_data]
            rec = torch.cat(recs, dim=0).cpu().numpy()
            return ev.evaluate(rec)
        need = (ev.need_counts, ev.need_items)
        parts = [self.eval_batch(b, neg_sampler=sampler, neg_num=getattr(eval_data, 'neg_num', 0), need=need) for b in eval_data]
        cat = [torch.cat([p[i] for p in parts], dim=0).cpu().numpy() if parts[0][i] is not None else None for i in range(4)]
        rec, counts, user_len, items = cat
        return ev.evaluate(rec, counts=counts, user_len=user_len, items=items, n_items=self._n_items(), item_counts=self.item_counts)


class AcBERT4RecTrainer(ACSASRecTrainer):
    """trainer.py:1046-1048: AcBERT4Rec trains with the same adversarial two-loss step (the routed double backward of
    trainer.py:672-686, here through the autograd Functions over the same kernels) and the same full-sort evaluation."""
    pass


class ACSSEPTTrainer(ACSASRecTrainer):
    """ACSSEPT (acssept.py) under the AC training step of trainer.py:505-1036.  The reference registers no trainer of this name
    (trainer.py:1038-1048), so get_trainer (utils.py:89-100) hands its ACSSEPT the stock Trainer, which sums the two losses and
    cannot evaluate the tuple full_sort_predict returns; this class is the trainer the model's (attacked, calibrated) API is
    written for, on the autograd Functions over the same kernels."""
    pass


class ACTiSASRecTrainer(ACSASRecTrainer):
    """ACTiSASRec (actisasrec.py) under the AC training step; like ACSSEPT the reference registers no trainer of this name."""
    pass
