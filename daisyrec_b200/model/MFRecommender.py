"""BPR-MF on the B200 path, with the reference's class name, config keys and methods
(daisy/model/MFRecommender.py:25-133).

No nn.Embedding, no autograd, no torch.optim: the two factor tables are raw fp32 device tensors
(still reachable as ``embed_user.weight`` / ``embed_item.weight``) and every method forwards to
hand-written CUDA through the C ABI (include/daisyrec_b200.h):

    fit        -> drb_gather_triples + drb_mf_bpr_train_steps   (one persistent launch per epoch)
    calc_loss  -> drb_mf_bpr_loss
    train_step -> drb_mf_bpr_train_step_host                     (host batch in, loss out)
    rank       -> drb_mf_rank        full_rank -> drb_mf_full_rank        predict -> drb_mf_predict
"""
import numpy as np
import torch

from .. import ops
from .AbstractRecommender import GeneralRecommender, _Table, _init_table, _INIT


class MF(GeneralRecommender):
    # the pair-wise criteria of AbstractRecommender.py:83-88 and the point-wise ones of :79-82 (batch[2] = label)
    SUPPORTED_LOSSES = ('BPR', 'HL', 'TL', 'CL', 'SL')
    SUPPORTED_OPTIMIZERS = ('sgd', 'adam', 'adagrad', 'rmsprop')     # AbstractRecommender.py:53-60

    def __init__(self, config):
        """Same keys as the reference (MFRecommender.py:46-59): lr, reg_1, reg_2, epochs, topk,
        user_num, item_num, factors, loss_type, optimizer, init_method, early_stop (+ gpu, logger)."""
        super().__init__(config)
        self.lr = config['lr']
        self.reg_1 = config['reg_1']
        self.reg_2 = config['reg_2']
        self.epochs = config['epochs']
        self.topk = config['topk']
        self.user_num, self.item_num, self.factors = config['user_num'], config['item_num'], config['factors']

        self.loss_type = config['loss_type']
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'sgd'
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'normal'
        self.early_stop = config['early_stop']

        # Same CPU RNG consumption as the reference: two nn.Embedding constructors (N(0,1) each),
        # then self.apply(_init_weight) over embed_user, embed_item (AbstractRecommender.py:69-77).
        wu = _init_table(self.user_num, self.factors, None)
        wi = _init_table(self.item_num, self.factors, None)
        _INIT[self.initializer](wu)
        _INIT[self.initializer](wi)
        if self.world > 1:
            # every rank drew the tables from its own CPU RNG; rank 0's draw is THE model (replicas of Q must start
            # bit-identical and the shards of P must come from one table whatever the ranks' RNG histories were)
            from ..parallel import broadcast_cpu_
            broadcast_cpu_(wu, self.device)
            broadcast_cpu_(wi, self.device)
        self.embed_item = _Table(wi.to(self.device))
        if self.world > 1:
            # user rows are sharded at fit()/rank() time, once the interaction counts are known
            self._P_full_cpu, self.embed_user, self._bounds, self._trainer = wu, None, None, None
        else:
            self.embed_user = _Table(wu.to(self.device))
        self._stage = None
        self.step_variant = ops.mf_step_variant(self.factors, self.user_num + self.item_num)   # runs the one-off on-device selection
        # optional B200 key: True = every cross-thread sum of a step in fixed point (bitwise reproducible runs); single GPU
        self.deterministic = bool(config.get('deterministic', False))
        if self.deterministic and (self.world > 1 or str(config.get('neg_sampling', 'table')) == 'fused'):
            raise NotImplementedError("deterministic=True covers single-GPU training on the sampler's triples")
        # optional B200 key (torchrun only): 'p2p' = one persistent launch per epoch with the exchange inside the kernel over
        # peer-mapped memory; 'nccl' = phase 1 -> grouped NCCL all-reduce -> phase 2 per step (also the automatic fallback)
        self.sharded_comm = str(config.get('sharded_comm', 'auto'))   # auto: p2p on 2 GPUs, nccl beyond (parallel.py)
        # optional B200 key: 'table' (default; the reference's per-user-once negatives, taken from the loader's triples) |
        # 'fused' (throughput mode: a fresh negative per triple and step is drawn inside the step kernel from the
        # complement of the user's train row; the loader's third column is ignored)
        self.neg_sampling = str(config.get('neg_sampling', 'table'))
        self._csr_dev = None
        if self.neg_sampling == 'fused':
            from ..utils.sampler import csr_from_ur
            row_ptr, col = config['train_csr'] if config.get('train_csr') is not None else csr_from_ur(config['train_ur'], self.user_num)
            if int(np.max(np.diff(row_ptr))) >= self.item_num:
                raise ValueError("'a' cannot be empty unless no samples are taken")
            self._csr_dev = (torch.from_numpy(np.ascontiguousarray(row_ptr, np.int64)).to(self.device),
                             torch.from_numpy(np.ascontiguousarray(col, np.int32)).to(self.device))
            self._neg_seed = int(torch.empty((), dtype=torch.int64).random_().item()) & ((1 << 63) - 1)

    # ------------------------------------------------------------------ plumbing
    def state_dict(self):
        return {'embed_user.weight': self._full_user_table(), 'embed_item.weight': self.embed_item.weight}

    def load_state_dict(self, sd):
        pu = sd['embed_user.weight']
        if self.world > 1:                                            # keep this rank's rows of the full table
            if self._bounds is None:
                self._shard(self._default_bounds())
            lo, hi = int(self._bounds[self.rank_id]), int(self._bounds[self.rank_id + 1])
            pu = pu[lo:hi]
        self.embed_user.weight.copy_(pu)
        self.embed_item.weight.copy_(sd['embed_item.weight'])

    # ------------------------------------------------------------------ multi-GPU (user-sharded P)
    def _shard(self, bounds):
        from ..parallel import ShardedTrainer
        if self._bounds is not None and np.array_equal(bounds, self._bounds):
            return
        if self._bounds is not None:                               # re-shard: collect the current rows first
            self._P_full_cpu = self.gather_user_table().cpu()
        self._bounds = np.asarray(bounds, np.int64)
        lo, hi = int(bounds[self.rank_id]), int(bounds[self.rank_id + 1])
        self.embed_user = _Table(self._P_full_cpu[lo:hi].contiguous().to(self.device))
        self._P_full_cpu = None
        if self._trainer is not None:
            self._trainer.close()
            self.embed_item = _Table(self._trainer.Q)
        self._trainer = None

    def _default_bounds(self):
        from ..parallel import partition_users
        return partition_users(np.ones(self.user_num, np.int64), self.world)

    def _sharded_trainer(self, d_triples):
        from ..parallel import ShardedTrainer, partition_users
        if self._bounds is None:
            w = torch.bincount(d_triples[:, 0].to(torch.int64), minlength=self.user_num).cpu().numpy()
            self._shard(partition_users(w, self.world))
        if self._trainer is None:
            self._trainer = ShardedTrainer(self.embed_user.weight, self.embed_item.weight, self._bounds, self.rank_id,
                                           self.world, self._hp, self._optimizer_name(), comm=self.sharded_comm)
            self.embed_item = _Table(self._trainer.Q)             # p2p: the replica lives in the peer-visible buffer
        return self._trainer

    def gather_user_table(self):
        """Full [user_num, factors] user table on every rank (one all-gather of the shards)."""
        if self.world == 1:
            return self.embed_user.weight
        from ..parallel import allgather_rows
        lo, hi = int(self._bounds[self.rank_id]), int(self._bounds[self.rank_id + 1])
        pos = torch.arange(lo, hi, device=self.device)
        return allgather_rows(self.embed_user.weight, pos, self.user_num)

    def _hyper(self, opt):
        return ops.hyper(self.lr, self.reg_1, self.reg_2, opt, loss=str(self.loss_type).upper())

    def _begin_fit(self, opt):
        """fit() builds a fresh optimizer (AbstractRecommender.py:105): fresh Adam moments / step count."""
        if str(self.loss_type).upper() in ('CL', 'SL') and (self.world > 1 or self.neg_sampling == 'fused'):
            raise NotImplementedError('the point-wise losses (CL / SL) run on one GPU with sampler-made rows; the sharded '
                                      'step and the fused negative sampler cover the pair-wise losses')
        super()._begin_fit(opt)
        if self.world > 1:
            if self._trainer is not None:
                self._trainer.close()                              # keeps a private copy of Q; frees the peer buffers
                self.embed_item = _Table(self._trainer.Q)
            self._trainer = None                                   # fresh optimiser state per fit()
            return
        self._ws = ops.MFWorkspace(self.user_num, self.item_num, self.factors, opt, self.device, deterministic=self.deterministic)

    def _train_steps(self, bu, bi, bj, batch, first, n_steps):
        if self.neg_sampling == 'fused':
            losses = ops.mf_bpr_train_steps_fused_neg(self.embed_user.weight, self.embed_item.weight, self._ws, bu, bi,
                                                      self._csr_dev[0], self._csr_dev[1], self._neg_seed + self._opt_steps,
                                                      batch, first, n_steps, self._hp, adam_step0=self._opt_steps)
            self._opt_steps += n_steps
            return losses
        losses = ops.mf_bpr_train_steps(self.embed_user.weight, self.embed_item.weight, self._ws, bu, bi, bj, batch,
                                        first, n_steps, self._hp, adam_step0=self._opt_steps)
        self._opt_steps += n_steps
        return losses

    @staticmethod
    def _host_i32(x):
        if isinstance(x, torch.Tensor):
            x = x.detach().cpu().numpy()
        return np.ascontiguousarray(x, dtype=np.int32)

    # ------------------------------------------------------------------ reference surface
    def _full_user_table(self):
        """[user_num, factors] user table: the local tensor on one GPU, an all-gather of the shards under torchrun
        (a collective: like every driver call in SPMD mode it must be reached by all ranks)."""
        if self.world == 1:
            return self.embed_user.weight
        if self._bounds is None:
            self._shard(self._default_bounds())
        return self.gather_user_table()

    def _score_tables(self):
        return self._full_user_table(), self.embed_item.weight

    def calc_loss(self, batch):
        """MFRecommender.py:70-97: 0-d fp32 loss of one (user, pos, neg) -- or, for CL / SL, (user, item, label) --
        batch; no update."""
        self._check_loss_type()
        if self.world > 1:
            raise NotImplementedError('calc_loss / train_step on single batches are single-GPU entry points; under torchrun '
                                      'use fit(train_loader) (user-sharded global steps)')
        bu, bi, bj = self._planes(batch[:3])
        self._ensure(0)
        loss = ops.mf_bpr_loss(self.embed_user.weight, self.embed_item.weight, self._ws, bu, bi, bj, self._hp)
        return loss.to(torch.float32).reshape(())

    def train_step(self, batch):
        """zero_grad + calc_loss + backward + optimizer.step on one HOST batch
        (AbstractRecommender.py:119-128); returns loss.item().  The ids are range-checked on the host: the kernel reads
        them from there."""
        self._check_loss_type()
        if self.world > 1:
            raise NotImplementedError('train_step is a single-GPU entry point; under torchrun use fit(train_loader)')
        hb = [self._host_i32(b) for b in batch[:3]]
        for h, hi, name in zip(hb, *self._triple_columns()):
            if len(h) and (int(h.min()) < 0 or int(h.max()) >= hi):
                raise IndexError(f'index out of range in self: {name} id(s) outside [0, {hi})')
        self._ensure(0)
        n = len(hb[0])
        if self._stage is None or self._stage.numel() < 3 * ((n + 3) // 4 * 4) + 4:
            self._stage = ops.stage_buffer(n, self.device)
        loss = ops.mf_bpr_train_step_host(self.embed_user.weight, self.embed_item.weight, self._ws, hb[0], hb[1], hb[2],
                                          self._hp, self._stage, adam_step0=self._opt_steps)
        self._opt_steps += 1
        return loss

    def fit_host_batches(self, h_bu, h_bi, h_bj, batch_size, n_steps=None):
        """Train on pre-collated HOST index planes (pinned CPU int32 tensors holding consecutive batches of
        ``batch_size`` triples): the step loop of AbstractRecommender.py:116-128 with the per-step
        ``.to(device)`` copies and ``loss.item()`` reads kept, but pipelined (copy of batch s+1 under the
        kernel of batch s).  Returns the per-step losses (CPU float64 tensor)."""
        self._check_loss_type()
        self._ensure(0)
        n = h_bu.numel()
        if n_steps is None:
            n_steps = (n + batch_size - 1) // batch_size
        losses = ops.mf_bpr_train_steps_host(self.embed_user.weight, self.embed_item.weight, self._ws, h_bu, h_bi, h_bj,
                                             batch_size, n_steps, self._hp, adam_step0=self._opt_steps)
        self._opt_steps += n_steps
        return losses

    def _rank_rows(self, users, cands, k):
        if self.world > 1:
            return self._rank_sharded(users, cands, k)
        return super()._rank_rows(users, cands, k)

    def _rank_sharded(self, users, cands, k):
        """Each rank scores the test users it owns; one all-gather assembles [n_users, k] in loader order."""
        from ..parallel import allgather_rows, owner_of
        if self._bounds is None:
            self._shard(self._default_bounds())
        mine = torch.from_numpy(np.flatnonzero(owner_of(users.cpu().numpy(), self._bounds) == self.rank_id)).to(self.device)
        if len(mine):
            loc = ops.mf_rank(self.embed_user.weight, self.embed_item.weight, users[mine] - int(self._bounds[self.rank_id]),
                              cands[mine], k)
        else:
            loc = torch.zeros((0, k), dtype=torch.float32, device=self.device)
        return allgather_rows(loc, mine, len(users))

    def full_rank_users(self, users):
        """Batched full_rank (B200 extension): int64 ndarray [len(users), topk]."""
        users = self._users(np.asarray(users, dtype=np.int64))
        return self._full_rank_rows(users, min(self.topk, self.item_num)).cpu().numpy()
