"""Feeds of the hot path: synthetic Interaction-shaped batches (SURVEY.md §8d) and the two loaders
the trainer iterates (recbole/data/dataloader/general_dataloader.py:23-65, 161-253, sequential branch).
Only what AC-SASRec reads is carried: item_id_list int64[B,L], item_length int64[B], item_id int64[B]
(the reference moves 5 more unused fields per step, SURVEY a19)."""
import math
from contextlib import nullcontext as _nullcontext

import numpy as np
import torch

from .compat import Interaction


def synth_sequences(n_rows, L, V, seed=42, full_len=False):
    """lengths ~ clip(round(LogNormal(ln 7, 0.8)), 1, L); items Zipf(1) on [1, V-1]; right-padded with 0."""
    g = torch.Generator().manual_seed(seed)
    if full_len:
        ln = torch.full((n_rows,), L, dtype=torch.int64)
    else:
        ln = torch.exp(torch.randn(n_rows, generator=g) * 0.8 + math.log(7.0)).round().clamp(1, L).to(torch.int64)
    w = 1.0 / torch.arange(1, V, dtype=torch.float64)
    items = torch.multinomial(w, n_rows * (L + 1), replacement=True, generator=g).view(n_rows, L + 1) + 1
    seq = items[:, :L].clone()
    seq[torch.arange(L).view(1, L) >= ln.view(n_rows, 1)] = 0
    return seq, ln, items[:, L].clone()


class SyntheticSequentialDataset(object):
    """Stands in for SequentialDataset (recbole/data/dataset/sequential_dataset.py) with seeded synthetic rows."""

    def __init__(self, config, n_rows, n_items, seed=42, full_len=False, pin=True):
        self.config = config
        self.item_num = int(n_items)
        L = config['MAX_ITEM_LIST_LENGTH']
        self.iid_field = config['ITEM_ID_FIELD']
        self.uid_field = config['USER_ID_FIELD']
        seq, ln, tgt = synth_sequences(n_rows, L, n_items, seed, full_len)
        feat = {self.iid_field + config['LIST_SUFFIX']: seq, config['ITEM_LIST_LENGTH_FIELD']: ln, self.iid_field: tgt,
                self.uid_field: torch.arange(n_rows, dtype=torch.int64) % max(n_rows - 1, 1) + 1}
        if str(config.get('model', '')) == 'ACTiSASRec':    # increasing time stamps, 0 on the padding (sequential_dataset.py:128-132)
            g = torch.Generator().manual_seed(seed + 7)
            ts = (torch.cumsum(torch.randint(0, 40, (n_rows, L), generator=g), 1) + 1000).float()
            ts[seq == 0] = 0.0
            feat[config['TIME_FIELD'] + config['LIST_SUFFIX']] = ts
        if pin and torch.cuda.is_available():
            feat = {k: v.pin_memory() for k, v in feat.items()}
        self.inter_feat = Interaction(feat)

    def num(self, field):
        if field == self.iid_field or field == self.iid_field + self.config['LIST_SUFFIX']:
            return self.item_num
        return len(self.inter_feat)

    def __len__(self):
        return len(self.inter_feat)


def _model_fields(config):
    iid = config['ITEM_ID_FIELD']
    f = [iid + config['LIST_SUFFIX'], config['ITEM_LIST_LENGTH_FIELD'], iid]
    if str(config.get('model', '')) == 'ACSSEPT':          # the one model that reads the user id (acssept.py:177)
        f.append(config['USER_ID_FIELD'])
    if str(config.get('model', '')) == 'ACTiSASRec':       # ... and the one that reads the time stamps (actisasrec.py:177)
        f.append(config['TIME_FIELD'] + config['LIST_SUFFIX'])
    return f


def _with_user(config, fields):
    """fields + the user id, which the negative sampler reads (once)"""
    uid = config['USER_ID_FIELD']
    return list(fields) + ([uid] if uid not in fields else [])


class _PackedBatches(object):
    """The three int64 fields the model reads, re-laid out batch by batch in ONE pinned buffer (refilled in place after every
    shuffle), so that each batch is a single contiguous host->device copy.  Full batches only; a ragged tail stays unpacked."""

    def __init__(self, config, batch_size, fields=None):
        self.fields, self.bs, self.buf = (fields or _model_fields(config)), batch_size, None

    def fill(self, inter_feat):
        n = len(inter_feat)
        nb = n // self.bs
        if nb == 0 or any(f not in inter_feat or inter_feat[f].dtype != torch.int64 for f in self.fields):    # int64 fields only
            self.nb = 0
            return
        per = [int(np.prod(inter_feat[f].shape[1:])) for f in self.fields]
        P = self.bs * sum(per)
        if self.buf is None or self.buf.shape != (nb, P):
            self.buf = torch.empty((nb, P), dtype=torch.int64)
            if torch.cuda.is_available():
                self.buf = self.buf.pin_memory()
        off = 0
        self.layout = []
        for f, w in zip(self.fields, per):
            src = inter_feat[f][:nb * self.bs].reshape(nb, self.bs * w)
            self.buf[:, off:off + self.bs * w].copy_(src)
            self.layout.append((f, off, (self.bs,) + tuple(inter_feat[f].shape[1:])))
            off += self.bs * w
        self.nb = nb

    def batch(self, i):
        from .compat import PackedInteraction
        return PackedInteraction(self.buf[i], self.layout)


class TrainDataLoader(object):
    """general_dataloader.py:23-65: per-epoch CPU randperm shuffle, then contiguous batch slices."""

    def __init__(self, config, dataset, shuffle=True, batch_size=None, neg_sampler=None):
        self.config, self.dataset, self.shuffle = config, dataset, shuffle
        self.batch_size = batch_size or config['train_batch_size']
        self.pr = 0
        # BPR with `neg_sampling`: batches carry the user id; the trainer draws the negatives on the device (ops.NegSampler)
        self.neg_sampler = neg_sampler
        if neg_sampler is not None:
            neg_sampler.check_users(dataset.inter_feat[config['USER_ID_FIELD']])
        fields = _with_user(config, _model_fields(config)) if neg_sampler is not None else None
        self._packed = _PackedBatches(config, self.batch_size, fields) if config.get('packed_batches', True) else None
        self._filled = False

    @property
    def pr_end(self):
        return len(self.dataset)

    def __len__(self):
        return math.ceil(self.pr_end / self.batch_size)

    def __iter__(self):
        if self.shuffle:
            self.dataset.inter_feat.shuffle()
            self._filled = False
        if self._packed is not None and not self._filled:
            self._packed.fill(self.dataset.inter_feat)
            self._filled = True
        elif self.shuffle and torch.cuda.is_available():
            self.dataset.inter_feat = Interaction({k: v.pin_memory() for k, v in self.dataset.inter_feat.interaction.items()})
        return self

    def __next__(self):
        if self.pr >= self.pr_end:
            self.pr = 0
            raise StopIteration()
        i = self.pr // self.batch_size
        if self._packed is not None and self._filled and i < self._packed.nb:
            cur = self._packed.batch(i)
        else:
            cur = self.dataset.inter_feat[self.pr:self.pr + self.batch_size]
        self.pr += self.batch_size
        return cur



class DeviceTrainDataLoader(object):
    """TrainDataLoader with the data resident in HBM (SURVEY section 8 f-2): the fields the model reads are uploaded once, the
    epoch permutation is drawn ON the device (sort order of uniform keys from the CUDA generator seeded with the config seed; the reference
    uses a CPU randperm, interaction.py:293-297, so the order differs the way any two seeds differ), and acsr_batch_gather
    writes batch `cursor` into a packed device buffer.  The trainer captures gather + cursor advance inside its CUDA graph, so
    an epoch is nothing but graph replays: no host->device traffic, no host work per step.  Iterating the loader the usual
    way also works (each batch is gathered eagerly) and yields the same batches, including the ragged last one."""

    device_resident = True

    def __init__(self, config, dataset, shuffle=True, batch_size=None, device=None, neg_sampler=None):
        from ._lib import LIB
        from .compat import PackedInteraction
        self.LIB, self.PackedInteraction = LIB, PackedInteraction
        self.config, self.dataset, self.shuffle = config, dataset, shuffle
        self.batch_size = int(batch_size or config['train_batch_size'])
        self.device = torch.device(device if device is not None else config['device'])
        if self.device.type != 'cuda':
            raise ValueError('DeviceTrainDataLoader needs a CUDA device (got %s); use TrainDataLoader for host-side batches' % self.device)
        if len(_model_fields(config)) != 3:
            raise ValueError('DeviceTrainDataLoader serves the three fields of ACSASRec / AcBERT4Rec; use TrainDataLoader for %s' % config.get('model'))
        f = _model_fields(config)
        feat = dataset.inter_feat
        self.fields = list(f)
        self.seqs = feat[f[0]].to(self.device).contiguous()
        self.lens = feat[f[1]].to(self.device).contiguous()
        self.tgts = feat[f[2]].to(self.device).contiguous()
        neg_field = config['NEG_PREFIX'] + config['ITEM_ID_FIELD']
        self.negs = feat[neg_field].to(self.device).contiguous() if neg_field in feat else None
        # BPR with `neg_sampling`: the user ids stay in HBM too, and the sampler fills the neg slot of every gathered batch
        self.neg_sampler = neg_sampler if self.negs is None else None
        self.uids = None
        if self.neg_sampler is not None:
            self.neg_sampler.check_users(feat[config['USER_ID_FIELD']])
            self.uids = feat[config['USER_ID_FIELD']].to(self.device).contiguous()
        if self.negs is not None or self.neg_sampler is not None:
            self.fields.append(neg_field)
        self.n, self.L = int(self.seqs.shape[0]), int(self.seqs.shape[1])
        self.perm = torch.arange(self.n, dtype=torch.int64, device=self.device)
        self.cursor = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.gen = torch.Generator(device=self.device)
        self.gen.manual_seed(int(config['seed'] if config['seed'] is not None else 0))
        self.pr = 0
        self._out = None

    # ---- layout of one packed batch (what the trainer's static input buffer looks like) ----
    def layout(self, rows=None):
        B = self.batch_size if rows is None else rows
        lay, off = [], 0
        for k, shape in zip(self.fields, [(B, self.L), (B,), (B,), (B,)]):
            lay.append((k, off, shape))
            off += int(np.prod(shape))
        return lay, off

    @property
    def pr_end(self):
        return self.n

    @property
    def full_batches(self):
        return self.n // self.batch_size

    def __len__(self):
        return math.ceil(self.n / self.batch_size)

    def new_epoch(self):
        """draws the epoch's permutation on the device and rewinds the cursor"""
        if self.shuffle:
            # a uniformly random permutation as the sort order of i.i.d. keys, entirely on the device and asynchronous
            # (torch.randperm on CUDA synchronises / detours through the host for small n: ~80 ms per epoch on the GPU box)
            if getattr(self, '_keys', None) is None:
                self._keys = torch.empty(self.n, dtype=torch.float64, device=self.device)
            self._keys.uniform_(generator=self.gen)
            self.perm.copy_(torch.sort(self._keys).indices)
        self.cursor.zero_()
        self.pr = 0

    def gather_into(self, packed, stream=None):
        """enqueue: packed <- batch `cursor` of the permutation; with a negative sampler its draws for the same rows into the
        neg slot; cursor += 1  (two or three launches; graph-capturable)"""
        st = torch.cuda.current_stream().cuda_stream if stream is None else stream
        self.LIB.call('acsr_batch_gather', self.seqs.data_ptr(), self.lens.data_ptr(), self.tgts.data_ptr(),
                      self.negs.data_ptr() if self.negs is not None else None, self.perm.data_ptr(), self.cursor.data_ptr(), self.n,
                      self.batch_size, self.L, packed.data_ptr(), st)
        if self.neg_sampler is not None:
            lay = dict((k, off) for k, off, _ in self.layout()[0])
            off = lay[self.fields[3]]
            with torch.cuda.stream(torch.cuda.ExternalStream(st)) if stream is not None else _nullcontext():
                self.neg_sampler.draw(self.uids, 1, positives=self.tgts, out=packed[off:off + self.batch_size].view(-1, 1), ld=1,
                                      perm=self.perm, cursor=self.cursor, n_rows=self.n, rows=self.batch_size)
        self.LIB.call('acsr_cursor_advance', self.cursor.data_ptr(), st)

    def tail_batch(self):
        """the ragged last batch (n % batch_size rows) as a device Interaction, or None"""
        r = self.n % self.batch_size
        if r == 0:
            return None
        idx = self.perm[self.n - r:]
        f = {self.fields[0]: self.seqs[idx], self.fields[1]: self.lens[idx], self.fields[2]: self.tgts[idx]}
        if self.negs is not None:
            f[self.fields[3]] = self.negs[idx]
        elif self.neg_sampler is not None:
            f[self.fields[3]] = self.neg_sampler.draw(self.uids[idx], 1, positives=f[self.fields[2]]).view(-1)
        return Interaction(f)

    def __iter__(self):
        self.new_epoch()
        return self

    def __next__(self):
        if self.pr >= self.n:
            self.pr = 0
            raise StopIteration()
        if self.pr + self.batch_size <= self.n:
            lay, total = self.layout()
            out = torch.empty(total, dtype=torch.int64, device=self.device)
            self.gather_into(out)
            cur = self.PackedInteraction(out, lay)
        else:
            cur = self.tail_batch()
        self.pr += self.batch_size
        return cur


class FullSortEvalDataLoader(object):
    """general_dataloader.py:246-253: (interaction, history_index=None, positive_u=arange(B), positive_i=item_id)."""

    def __init__(self, config, dataset, batch_size=None):
        self.config, self.dataset = config, dataset
        self.batch_size = batch_size or config['eval_batch_size']
        self.iid_field = config['ITEM_ID_FIELD']
        self.pr = 0
        self._packed = _PackedBatches(config, self.batch_size) if config.get('packed_batches', True) else None
        if self._packed is not None:
            self._packed.fill(dataset.inter_feat)

    @property
    def pr_end(self):
        return len(self.dataset)

    def __len__(self):
        return math.ceil(self.pr_end / self.batch_size)

    def __iter__(self):
        return self

    def __next__(self):
        if self.pr >= self.pr_end:
            self.pr = 0
            raise StopIteration()
        i = self.pr // self.batch_size
        if self._packed is not None and i < self._packed.nb:
            interaction = self._packed.batch(i)
        else:
            interaction = self.dataset.inter_feat[self.pr:self.pr + self.batch_size]
        n = len(interaction)
        self.pr += self.batch_size
        return interaction, None, torch.arange(n), interaction[self.iid_field]


class NegSampleEvalDataLoader(FullSortEvalDataLoader):
    """`eval_args.mode: uniN / popN` (general_dataloader.py NegSampleEvalDataLoader, sequential branch): yields
    (interaction, None, positive_u=arange(B), positive_i=item_id) like FullSortEvalDataLoader, with the user id in every batch.
    The N negatives of a batch are not drawn here but on the device by the trainer (`neg_sampler`, an ops.NegSampler holding
    this phase's used sets), fresh for every batch of every pass."""

    def __init__(self, config, dataset, neg_sampler, neg_num, batch_size=None):
        self.neg_sampler, self.neg_num = neg_sampler, int(neg_num)
        neg_sampler.check_users(dataset.inter_feat[config['USER_ID_FIELD']])
        self.uid_field = config['USER_ID_FIELD']
        self.config, self.dataset = config, dataset
        self.batch_size = batch_size or config['eval_batch_size']
        self.iid_field = config['ITEM_ID_FIELD']
        self.pr = 0
        self._packed = (_PackedBatches(config, self.batch_size, _with_user(config, _model_fields(config)))
                        if config.get('packed_batches', True) else None)
        if self._packed is not None:
            self._packed.fill(dataset.inter_feat)
