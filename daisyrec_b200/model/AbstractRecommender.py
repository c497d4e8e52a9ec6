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


def loader_plan(train_loader, shape_ok=lambda data: data.ndim == 2 and data.shape[1] == 3):
    """Decode a DataLoader into (rows ndarray, batch_size, shuffle, drop_last, generator), or None when it is not a plain
    ``DataLoader(dataset, batch_size, shuffle)`` over a dataset whose ``.data`` ndarray passes ``shape_ok`` -- by default
    the ``BasicDataset(int[T,3])`` of run_examples/test.py:93-94 (then fit() falls back to iterating it batch by batch)."""
    ds = getattr(train_loader, 'dataset', None)
    data = getattr(ds, 'data', None)
    bs = getattr(train_loader, 'batch_size', None)
    if not isinstance(data, np.ndarray) or not shape_ok(data) or bs is None:
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


def candidate_rows(test_loader):
    """Decode a test loader into (users int64 ndarray [n], candidates int64 ndarray [n, C]): the (user, candidates) rows of
    a CandidatesDataset are read directly, any other iterable of (users, candidates) batches is iterated."""
    data = getattr(getattr(test_loader, 'dataset', None), 'data', None)
    if isinstance(data, (list, tuple)) and len(data) and len(data[0]) == 2:
        users = np.fromiter((int(r[0]) for r in data), np.int64, len(data))
        return users, np.stack([np.asarray(r[1], dtype=np.int64) for r in data])
    us, cs = [], []
    for b_us, b_c in test_loader:
        us.append(torch.as_tensor(b_us).reshape(-1).to(torch.int64))
        cs.append(torch.as_tensor(b_c).to(torch.int64).reshape(us[-1].numel(), -1))
    if not us:
        return np.zeros(0, np.int64), np.zeros((0, 0), np.int64)
    return torch.cat(us).numpy(), torch.cat(cs).numpy()


def mask_segments(n_rows, batch, first, n_steps, bytes_per_step, cap=64 << 20):
    """Split steps first .. first+n_steps-1 over n_rows index rows (``batch`` rows a step, the last step may hold fewer)
    into calls whose host-drawn dropout masks take at most ``cap`` bytes -> (first_step, count, rows) in step order: count
    steps of ``rows = batch`` rows, or the ragged last step alone (count 1, rows < batch), which gets its own draws."""
    chunk = max(1, cap // max(1, bytes_per_step))
    s, end = first, first + n_steps
    while s < end:
        k = min(chunk, end - s)
        full = k if (s + k) * batch <= n_rows else k - 1
        if full > 0:
            yield s, full, batch
        if full < k:
            yield s + full, 1, n_rows - (s + full) * batch
        s += k


def tower_dtype(config, allowed=('fp32', 'bf16')):
    """config['tower_dtype'] -> its kernel code: the index in ``allowed`` (0 fp32, 1 bf16, 2 fused)."""
    td = str(config.get('tower_dtype', 'fp32')).lower()
    if td not in allowed:
        names = [f"'{a}'" for a in allowed]
        raise ValueError(f"tower_dtype must be {', '.join(names[:-1])} or {names[-1]}, got {td!r}")
    return allowed.index(td)


def dropout_engine(config):
    """config['dropout_engine']: 'auto' | 'torch' (host masks from the global CPU generator) | 'philox' (device masks)."""
    engine = str(config.get('dropout_engine', 'auto')).lower()
    if engine not in ('auto', 'torch', 'philox'):
        raise ValueError(f"dropout_engine must be 'auto', 'torch' or 'philox', got {engine!r}")
    return engine


def dropout_rate(p):
    """A dropout probability as nn.Dropout takes it (None -> 0.0)."""
    p = float(p or 0.0)
    if not 0.0 <= p < 1.0:
        raise ValueError(f"dropout probability has to be in [0, 1), but got {p}")
    return p


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
        self._ws, self._hp, self._opt_steps = None, None, 0

    # ------------------------------------------------------------------ state
    _BUFFERS = ()                               # state_dict() keys that hold statistics, not trained parameters

    def parameters(self):
        return [t for k, t in self.state_dict().items() if k not in self._BUFFERS]

    def load_state_dict(self, sd):
        """Copy every state_dict() key from sd (reshaped to the parameter's shape)."""
        for k, t in self.state_dict().items():
            t.copy_(torch.as_tensor(sd[k]).reshape(t.shape))
        self._tables_changed()

    def to(self, device):
        """The parameters live on self.device from construction on; kept for drivers that call model.to(device)."""
        return self

    def _tables_changed(self):
        """Called when the parameters changed: drop whatever was computed from them."""

    # ------------------------------------------------------------------ set-up
    def _hyper(self, opt):
        return ops.hyper(self.lr, self.reg_1, self.reg_2, opt)

    def _begin_fit(self, opt):
        """fit() builds a fresh optimizer (AbstractRecommender.py:105): fresh optimiser state and step count.  Classes whose
        scratch grows with the batch allocate it in _ensure."""
        self._hp = self._hyper(opt)
        self._opt_steps = 0
        self._fit_opt = opt
        self._ws = None

    def _ensure(self, rows):
        """Optimiser state and scratch for a call outside fit() that will hold up to ``rows`` index rows (classes without
        scratch ignore it): a fresh fit's state the first time."""
        if self._ws is None:
            self._begin_fit(self._optimizer_name())

    # ------------------------------------------------------------------ ids (nn.Embedding's IndexError: kernels index raw tables)
    def _users(self, ids):
        """Host-checked user ids -> int64 device tensor."""
        u = torch.as_tensor(ids).reshape(-1).to(torch.int64)
        if u.numel() and (int(u.min()) < 0 or int(u.max()) >= self.user_num):
            raise IndexError(f'index out of range in self: user id outside [0, {self.user_num})')
        return u.to(self.device)

    def _planes(self, cols, dtype=torch.int32):
        """A batch's id columns -> contiguous device planes of ``dtype``, checked against the bounds of _triple_columns()
        before any kernel sees them."""
        planes = [torch.as_tensor(c).to(self.device, dtype).reshape(-1).contiguous() for c in cols]
        bounds, names = self._triple_columns()
        ops.check_index_range(torch.stack(planes, 1), bounds[:len(planes)], names[:len(planes)])
        return planes

    # ------------------------------------------------------------------ reference surface
    def forward(self, user, item):
        """Scores of the (user[k], item[k]) pairs for index tensors."""
        return self._score_pairs(*self._planes((user, item)))

    def __call__(self, *args):
        return self.forward(*args)

    def train_step(self, batch):
        """zero_grad + calc_loss + backward + optimizer.step on one batch in train mode (AbstractRecommender.py:119-128)
        -> loss.item()."""
        self._check_loss_type()
        bu, bi, bj = self._planes(batch[:3])
        self._ensure(2 * bu.numel())
        was = self.training
        self.train()
        try:
            return float(self._train_steps(bu, bi, bj, max(1, bu.numel()), 0, 1).item())
        finally:
            self.train(was)

    def rank(self, test_loader):
        """-> float32 ndarray [n_test_users, topk] of candidate ids, best first, rows in loader order."""
        users, cands = candidate_rows(test_loader)
        if len(users) == 0:
            return np.zeros((0,), np.float32)
        users = self._users(users)
        d_cands = torch.from_numpy(np.ascontiguousarray(cands)).to(self.device)
        ops.check_index_range(d_cands.reshape(-1, 1), (self.item_num,), ('candidate item',))
        return self._rank_rows(users, d_cands, min(self.topk, cands.shape[1])).cpu().numpy()

    def full_rank(self, u):
        """-> int64 ndarray [topk] over every item; no masking of train items."""
        return self._full_rank_rows(self._users([int(u)]), min(self.topk, self.item_num))[0].cpu().numpy()

    def predict(self, u, i):
        """-> python float."""
        users = self._users([int(u)])
        if not 0 <= int(i) < self.item_num:
            raise IndexError(f'index out of range in self: item id outside [0, {self.item_num})')
        return float(self._score_pairs(users, torch.tensor([int(i)], dtype=torch.int32, device=self.device)).item())

    # per-class scoring on checked device ids; the defaults run the MF kernels on _score_tables()
    def _score_tables(self):
        """(user table, item table) the MF scoring kernels read."""
        return self.embed_user.weight, self.embed_item.weight

    def _rank_rows(self, users, cands, k):
        """users int64 [n], cands int64 [n, C] -> float32 [n, k] candidate ids, best first."""
        return ops.mf_rank(*self._score_tables(), users, cands, k)

    def _full_rank_rows(self, users, k):
        """users int64 [n] -> int64 [n, k] item ids, best first."""
        return ops.mf_full_rank(*self._score_tables(), users, k)

    def _score_pairs(self, u, i):
        """-> float32 [n] scores of the (u[k], i[k]) pairs."""
        return ops.mf_predict(*self._score_tables(), u.to(torch.int32), i.to(torch.int32))

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
