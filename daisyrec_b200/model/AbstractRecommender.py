"""Host side of the B200 recommenders: the reference's plug-in surface
(daisy/model/AbstractRecommender.py:10-137) without nn.Module / autograd / torch.optim.

``GeneralRecommender.fit(train_loader)`` keeps the reference contract -- a
``torch.utils.data.DataLoader`` over ``BasicDataset(samples)``, ``batch_size`` and ``shuffle`` read
from the loader, epoch loss accumulated from per-step losses, ``ValueError`` on a NaN loss, early
stop on |delta epoch loss| < 1e-5 -- but runs each epoch as ONE persistent kernel launch:
the epoch's permutation is produced with the DataLoader's own RNG protocol (so batches are the
reference's batches), gathered into SoA index planes on the device, and consumed by
``drb_mf_bpr_train_steps``.
"""
import os

import numpy as np
import torch
from torch.utils.data import RandomSampler, SequentialSampler, BatchSampler
from tqdm import tqdm

from .. import ops
from ..utils.sampler import fingerprint


# 'torch': the DataLoader's own permutation -- the reference's batches bit for bit -- computed ON THE DEVICE
#          (drb_randperm_torch: MT19937 stream + parallel Fisher-Yates, same result as torch.randperm on the CPU generator);
# 'torch-cpu': the same permutation from torch.randperm on the host (what the line above is tested against);
# 'device': torch.randperm on the GPU, seeded from the global RNG (same distribution, another order)
DEFAULT_SHUFFLE_ENGINE = 'torch'
RANDPERM_DEVICE_MAX = 0xFFFFFFFF // 20          # ATen switches algorithm above this n; the host path covers it


class _Table:
    """Stand-in for nn.Embedding: ``.weight`` is the raw fp32 [rows, factors] table."""

    def __init__(self, weight):
        self.weight = weight

    @property
    def num_embeddings(self):
        return self.weight.shape[0]

    @property
    def embedding_dim(self):
        return self.weight.shape[1]


def _init_table(rows, cols, method):
    """Reproduce the reference's CPU init stream: nn.Embedding's own N(0,1) reset first
    (torch/nn/modules/sparse.py reset_parameters), re-initialised later by ``_apply_init``."""
    return torch.empty(rows, cols, dtype=torch.float32).normal_(0.0, 1.0)


_INIT = {
    # AbstractRecommender.py:19-31 (initializer_param_config / initializer_config)
    'normal': lambda w: torch.nn.init.normal_(w, mean=0.0, std=0.01),
    'uniform': lambda w: torch.nn.init.uniform_(w, a=0.0, b=1.0),
    'xavier_normal': lambda w: torch.nn.init.xavier_normal_(w, gain=1.0),
    'xavier_uniform': lambda w: torch.nn.init.xavier_uniform_(w, gain=1.0),
}


def epoch_seed(shuffle, generator=None):
    """The DataLoader's RNG protocol for one epoch (torch/utils/data/dataloader.py:706-710 draws ``_base_seed``;
    sampler.py RandomSampler.__iter__ draws the seed of a private generator).  Consumes the global torch RNG exactly as
    iterating the loader would.  -> the RandomSampler's seed, or None without shuffling."""
    torch.empty((), dtype=torch.int64).random_(generator=generator)           # _base_seed (discarded)
    if not shuffle:
        return None
    return int(torch.empty((), dtype=torch.int64).random_().item())


def epoch_permutation(n, shuffle, generator=None, seed=None):
    """Index order of one DataLoader epoch: ``torch.randperm(n, generator)`` of a private generator seeded as
    RandomSampler.__iter__ seeds it (``seed`` given: already drawn with epoch_seed)."""
    if seed is None:
        seed = epoch_seed(shuffle, generator)
    if not shuffle or seed is None:
        return None
    g = torch.Generator()
    g.manual_seed(seed)
    return torch.randperm(n, generator=g)


def loader_plan(train_loader):
    """Decode a DataLoader into (triples ndarray, batch_size, shuffle, drop_last, generator), or None when it is not the
    plain ``DataLoader(BasicDataset(int[T,3]), batch_size, shuffle)`` of run_examples/test.py:93-94 (then fit() falls back
    to iterating it batch by batch)."""
    ds = getattr(train_loader, 'dataset', None)
    data = getattr(ds, 'data', None)
    bs = getattr(train_loader, 'batch_size', None)
    if not isinstance(data, np.ndarray) or data.ndim != 2 or data.shape[1] != 3 or bs is None:
        return None
    sampler = getattr(train_loader, 'sampler', None)
    if not isinstance(getattr(train_loader, 'batch_sampler', None), BatchSampler):
        return None
    if isinstance(sampler, RandomSampler) and not sampler.replacement and sampler._num_samples is None:
        shuffle, gen = True, sampler.generator
    elif isinstance(sampler, SequentialSampler):
        shuffle, gen = False, None
    else:
        return None
    if gen is not None:
        return None
    return data, int(bs), shuffle, bool(train_loader.drop_last), train_loader.generator


class AbstractRecommender(object):
    def __init__(self):
        self.optimizer = None
        self.initializer = None
        self.loss_type = None
        self.lr = 0.01
        self.logger = None
        self.training = False

    # -- reference surface (AbstractRecommender.py:33-46)
    def calc_loss(self, batch):
        raise NotImplementedError

    def fit(self, train_loader):
        raise NotImplementedError

    def rank(self, test_loader):
        raise NotImplementedError

    def full_rank(self, u):
        raise NotImplementedError

    def predict(self, u, i):
        raise NotImplementedError

    # -- nn.Module look-alikes used by drivers
    def train(self, mode=True):
        self.training = mode
        return self

    def eval(self):
        return self.train(False)

    SUPPORTED_OPTIMIZERS = ('sgd', 'adam')

    def _optimizer_name(self):
        """AbstractRecommender.py:48-67: unknown names fall back to Adam with a log line."""
        name = str(self.optimizer).lower()
        if name in self.SUPPORTED_OPTIMIZERS:
            return name
        if name == 'sparse_adam':       # what optim.SparseAdam.step() raises on nn.Embedding's dense gradients (:61-62)
            raise RuntimeError('SparseAdam does not support dense gradients, please consider Adam instead')
        if name in ('adagrad', 'rmsprop'):
            raise NotImplementedError(f"optimizer '{name}' is outside the B200 hot path of {type(self).__name__} "
                                      f"(native: {', '.join(self.SUPPORTED_OPTIMIZERS)})")
        if self.logger is not None:
            self.logger.info('Received unrecognized optimizer, set default Adam optimizer')
        return 'adam'

    SUPPORTED_LOSSES = ('BPR',)

    def _check_loss_type(self):
        lt = str(self.loss_type).upper()
        if lt in self.SUPPORTED_LOSSES:
            return
        if lt in ('CL', 'SL', 'HL', 'TL', 'BPR'):
            raise NotImplementedError(f"loss_type '{lt}' is outside the B200 hot path of {type(self).__name__} "
                                      f"(native: {', '.join(self.SUPPORTED_LOSSES)})")
        raise NotImplementedError(f'Invalid loss type: {self.loss_type}...')


class GeneralRecommender(AbstractRecommender):
    def __init__(self, config):
        super().__init__()
        gpu = str(config.get('gpu', '') or '')
        if gpu and not torch.cuda.is_initialized() and 'LOCAL_RANK' not in os.environ:
            os.environ['CUDA_VISIBLE_DEVICES'] = gpu             # AbstractRecommender.py:99
        ops.require_cuda()
        local = int(os.environ.get('LOCAL_RANK', torch.cuda.current_device()))
        self.device = torch.device('cuda', local if local < torch.cuda.device_count() else 0)
        torch.cuda.set_device(self.device)
        self.logger = config['logger']
        self.steps_per_launch = int(config.get('steps_per_launch', 0))   # 0 = whole epoch in one launch
        self.show_progress = bool(config.get('progress', True))
        # 'torch' (default): the DataLoader's own CPU permutation -> the reference's batches bit for bit;
        # 'device': torch.randperm on the GPU seeded from the global RNG (same distribution, no 8-byte/triple H2D)
        self.shuffle_engine = str(config.get('shuffle_engine', DEFAULT_SHUFFLE_ENGINE))
        # one process per GPU (torchrun): user-sharded training / ranking, see daisyrec_b200/parallel.py
        import torch.distributed as dist
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.rank_id = dist.get_rank() if self.world > 1 else 0

    def _loader_plan(self, train_loader):
        return loader_plan(train_loader)

    def fit(self, train_loader):
        self._check_loss_type()
        opt = self._optimizer_name()
        self._begin_fit(opt)
        plan = self._loader_plan(train_loader)
        last_loss = 0.
        for epoch in range(1, self.epochs + 1):
            self.train()
            if plan is not None and self.world > 1:
                current_loss = self._fit_epoch_sharded(plan, epoch)
            elif plan is not None:
                current_loss = self._fit_epoch_bulk(plan, epoch)
            else:
                current_loss = self._fit_epoch_generic(train_loader, epoch)
            self.eval()
            delta_loss = float(current_loss - last_loss)
            if (abs(delta_loss) < 1e-5) and self.early_stop:
                self.logger.info('Satisfy early stop mechanism')
                break
            else:
                last_loss = current_loss

    def _fit_epoch_bulk(self, plan, epoch):
        data, bs, shuffle, drop_last, gen = plan
        T = data.shape[0]
        # the epoch's order is computed on a side stream while the rows upload (first epoch) / are stamped: the one-CTA
        # MT19937 stream leaves the copy engines and 147 SMs free
        exact_on_device = shuffle and self.shuffle_engine == 'torch' and T < RANDPERM_DEVICE_MAX
        if exact_on_device:
            # buffers are allocated on the main stream and kept for the model's lifetime (no cross-stream allocator traffic)
            if getattr(self, '_perm_bufs', None) is None or self._perm_bufs[0].numel() < T:
                self._perm_bufs = ops.randperm_workspace(T, self.device)
            main = torch.cuda.current_stream(self.device)
            if getattr(self, '_side_stream', None) is None:
                self._side_stream = torch.cuda.Stream(self.device)
            self._side_stream.wait_stream(main)
            with torch.cuda.stream(self._side_stream):
                d_perm = self._device_permutation(T, shuffle, gen)
            d_triples = self._device_triples(data)
            main.wait_stream(self._side_stream)
        else:
            d_triples = self._device_triples(data)
            d_perm = self._device_permutation(T, shuffle, gen)
        bu, bi, bj = ops.gather_triples(d_triples, d_perm)
        n_use = (T // bs) * bs if drop_last else T
        nsteps = (n_use + bs - 1) // bs
        if n_use != T:
            bu, bi, bj = bu[:n_use], bi[:n_use], bj[:n_use]
        chunk = self.steps_per_launch if self.steps_per_launch > 0 else nsteps
        pbar = tqdm(total=nsteps, disable=not self.show_progress)
        pbar.set_description(f'[Epoch {epoch:03d}]')
        current_loss = 0.
        for first in range(0, nsteps, chunk):
            k = min(chunk, nsteps - first)
            losses = self._train_steps(bu, bi, bj, bs, first, k)           # raises ValueError on NaN
            current_loss += float(losses.sum().item())
            pbar.update(k)
        pbar.set_postfix(loss=current_loss)
        pbar.close()
        return current_loss

    def _device_permutation(self, T, shuffle, gen, seed=None):
        """The epoch's index order as a device int64 tensor (None = sequential); consumes the global RNG like the DataLoader."""
        if seed is None:
            seed = epoch_seed(shuffle, gen)
        if not shuffle:
            return None
        if self.shuffle_engine == 'device':
            g = torch.Generator(device=self.device)
            g.manual_seed(seed)
            return torch.randperm(T, generator=g, device=self.device)
        if self.shuffle_engine == 'torch' and T < RANDPERM_DEVICE_MAX:
            return ops.randperm_torch(seed, T, self.device, out=getattr(self, '_perm_bufs', None))
        return epoch_permutation(T, shuffle, gen, seed=seed).to(self.device, non_blocking=False)

    def _device_triples(self, data):
        """Device copy of the loader's [T,3] rows: the sampler's own device twin when the host array still carries the stamp
        it was attached with, else an upload cached per (array, stamp) -- an in-place edit of the host rows re-uploads."""
        stamp = fingerprint(data)
        d_triples = getattr(data, '_drb_device', None)
        if not (d_triples is not None and d_triples.device == self.device and getattr(data, '_drb_stamp', None) == stamp):
            if getattr(self, '_triples_key', None) != (id(data), stamp):
                host = np.ascontiguousarray(data, dtype=np.int32)
                self._triples_dev = torch.from_numpy(host if host.flags.writeable else host.copy()).to(self.device)
                self._triples_key = (id(data), stamp)
            d_triples = self._triples_dev
        if d_triples.is_cuda and getattr(self, '_range_ok', None) != (id(data), stamp):
            # nn.Embedding's IndexError (the kernels index raw tables): one pass over the ids per uploaded array
            ops.check_index_range(d_triples, *self._triple_columns())
            self._range_ok = (id(data), stamp)
        return d_triples

    def _triple_columns(self):
        """(upper bounds, names) of the loader rows' three columns, for the range check of _device_triples."""
        pointwise = str(self.loss_type).upper() in ('CL', 'SL')
        return ((self.user_num, self.item_num, (1 << 62) if pointwise else self.item_num),
                ('user', 'item', 'label' if pointwise else 'negative item'))

    def _fit_epoch_sharded(self, plan, epoch):
        """N > 1: same global batches as the single-GPU run; this rank trains the triples of its users."""
        data, bs, shuffle, drop_last, gen = plan
        T = data.shape[0]
        d_triples = self._device_triples(data)
        trainer = self._sharded_trainer(d_triples)
        # every rank advances its own RNG as the DataLoader would, but rank 0's seed decides the epoch's order: the ranks
        # keep disjoint shares of ONE permutation whatever their RNG histories were
        from ..parallel import broadcast_int
        seed = epoch_seed(shuffle, gen)
        if shuffle:
            seed = broadcast_int(seed, self.device)
        d_perm = self._device_permutation(T, shuffle, gen, seed=seed if shuffle else 0)
        nsteps = trainer.prepare_epoch(d_triples, d_perm, bs)
        if drop_last and T % bs:
            nsteps -= 1
        pbar = tqdm(total=nsteps, disable=not self.show_progress or self.rank_id != 0)
        pbar.set_description(f'[Epoch {epoch:03d}]')
        losses = trainer.train_steps(0, nsteps)
        trainer.check_nan()
        current_loss = float(losses.sum().item())
        pbar.update(nsteps)
        pbar.set_postfix(loss=current_loss)
        pbar.close()
        return current_loss

    def _fit_epoch_generic(self, train_loader, epoch):
        """Any other iterable of (user, pos, neg) batches: one end-to-end step per batch."""
        current_loss = 0.
        pbar = tqdm(train_loader, disable=not self.show_progress)
        pbar.set_description(f'[Epoch {epoch:03d}]')
        for batch in pbar:
            current_loss += self.train_step(batch)
        pbar.set_postfix(loss=current_loss)
        return current_loss
