"""Item2Vec on the B200 path, with the reference's class name, config keys and methods
(daisy/model/Item2VecRecommender.py).

Skip-gram with negative sampling over ONE item table: the loss of a (target, context, label) row is
BCEWithLogitsLoss(sum) of <shared[target], shared[context]>, so both rows are read from and both gradients land in
``shared_embedding``.  After training, a user's row is the sum of the item rows of their train items.

    fit        -> drb_gather_triples + drb_item2vec_train_steps (one persistent launch per epoch) + drb_item2vec_user_embed
    calc_loss  -> drb_item2vec_train_steps(apply=0)         train_step -> drb_item2vec_train_steps
    rank       -> drb_mf_rank        full_rank -> drb_mf_full_rank        predict -> drb_mf_predict
"""
import numpy as np
import torch

from .. import ops
from .AbstractRecommender import GeneralRecommender, _Table, _init_table, _INIT


class Item2Vec(GeneralRecommender):
    SUPPORTED_LOSSES = ('CL',)
    SUPPORTED_OPTIMIZERS = ('sgd', 'adam', 'adagrad', 'rmsprop')     # AbstractRecommender.py:53-60

    def __init__(self, config):
        """Same keys as the reference: user_num, item_num, factors, train_ur, lr, epochs, optimizer ('default' -> adam),
        init_method ('default' -> normal), early_stop, topk (+ gpu, logger; train_csr optional).  loss_type is always CL."""
        super().__init__(config)
        if self.world > 1:
            raise NotImplementedError('Item2Vec runs as independent replicas only (the sharded step covers MF)')
        if config.get('deterministic', False):
            raise NotImplementedError('deterministic=True covers MF only')
        self.user_num, self.item_num, self.factors = config['user_num'], config['item_num'], config['factors']
        self.ur = config['train_ur']
        self.csr = config.get('train_csr', None)
        self.lr = config['lr']
        self.epochs = config['epochs']
        self.loss_type = 'CL'                                      # cross-entropy, whatever the config says
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'adam'
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'normal'
        self.early_stop = config['early_stop']
        self.topk = config['topk']

        # The reference's CPU RNG consumption: the two nn.Embedding constructors (user, then shared; N(0,1) each), then
        # self.apply(_init_weight) re-initialises them in registration order.
        wu = _init_table(self.user_num, self.factors, None)
        wi = _init_table(self.item_num, self.factors, None)
        _INIT[self.initializer](wu)
        _INIT[self.initializer](wi)
        self.user_embedding = _Table(wu.to(self.device))
        self.shared_embedding = _Table(wi.to(self.device))
        self._ws = None
        self._opt_steps = 0

    # ------------------------------------------------------------------ plumbing
    def parameters(self):
        return [self.user_embedding.weight, self.shared_embedding.weight]

    def state_dict(self):
        return {'user_embedding.weight': self.user_embedding.weight, 'shared_embedding.weight': self.shared_embedding.weight}

    def load_state_dict(self, sd):
        for k, t in self.state_dict().items():
            t.copy_(torch.as_tensor(sd[k]).reshape(t.shape))

    def to(self, device):
        return self

    def _hyper(self, opt=None):
        return ops.hyper(self.lr, 0.0, 0.0, opt or self._optimizer_name(), loss='CL')

    def _begin_fit(self, opt):
        """fit() builds a fresh optimizer (AbstractRecommender.py:105): fresh optimiser state / step count."""
        self._hp = self._hyper(opt)
        self._opt_steps = 0
        self._ws = ops.Item2VecWorkspace(self.item_num, self.factors, opt, self.device)

    def _ensure_ws(self):
        if self._ws is None:
            self._begin_fit(self._optimizer_name())

    def _train_steps(self, bu, bi, bj, batch, first, n_steps):
        losses = ops.item2vec_train_steps(self.shared_embedding.weight, self._ws, bu, bi, bj, batch, first, n_steps, self._hp,
                                          adam_step0=self._opt_steps)
        self._opt_steps += n_steps
        return losses

    def _triple_columns(self):
        return (self.item_num, self.item_num, 1 << 62), ('target item', 'context item', 'label')

    def _batch(self, batch):
        planes = [torch.as_tensor(b).to(self.device, torch.int32).reshape(-1).contiguous() for b in batch[:3]]
        ops.check_index_range(torch.stack(planes[:2], 1).contiguous(), (self.item_num, self.item_num),
                              ('target item', 'context item'))
        return planes

    # ------------------------------------------------------------------ reference surface
    def fit(self, train_loader):
        """The epoch loop (AbstractRecommender.py:103-137), then every user of train_ur gets the sum of their items' rows --
        also after an early stop."""
        super().fit(train_loader)
        if self.csr is not None:
            row_ptr, col = self.csr
        else:
            from ..utils.sampler import csr_from_ur
            row_ptr, col = csr_from_ur(self.ur, self.user_num)
        col = np.ascontiguousarray(col, np.int32)
        ops.item2vec_user_embed(torch.from_numpy(np.ascontiguousarray(row_ptr, np.int64)).to(self.device),
                                torch.from_numpy(col if len(col) else np.zeros(1, np.int32)).to(self.device),
                                self.shared_embedding.weight, self.user_embedding.weight)

    def forward(self, target_i, context_j):
        """<shared[target], shared[context]> for index tensors."""
        t = torch.as_tensor(target_i).to(self.device, torch.int32).reshape(-1).contiguous()
        c = torch.as_tensor(context_j).to(self.device, torch.int32).reshape(-1).contiguous()
        return ops.mf_predict(self.shared_embedding.weight, self.shared_embedding.weight, t, c)

    __call__ = forward

    def calc_loss(self, batch):
        """0-d fp32 BCEWithLogitsLoss(sum) of one (target, context, label) batch; no update."""
        self._ensure_ws()
        bt, bc, bl = self._batch(batch)
        loss = ops.item2vec_train_steps(self.shared_embedding.weight, self._ws, bt, bc, bl, max(1, bt.numel()), 0, 1, self._hp,
                                        adam_step0=self._opt_steps, apply=False)
        return loss.to(torch.float32).reshape(())

    def train_step(self, batch):
        """zero_grad + calc_loss + backward + optimizer.step on one batch (AbstractRecommender.py:119-128) -> loss.item()."""
        self._ensure_ws()
        bt, bc, bl = self._batch(batch)
        return float(self._train_steps(bt, bc, bl, max(1, bt.numel()), 0, 1).item())

    def predict(self, u, i):
        """(user_embedding[u] * shared_embedding[i]).sum() -> python float."""
        d_u = torch.tensor([int(u)], dtype=torch.int32, device=self.device)
        d_i = torch.tensor([int(i)], dtype=torch.int32, device=self.device)
        return float(ops.mf_predict(self.user_embedding.weight, self.shared_embedding.weight, d_u, d_i).item())

    def rank(self, test_loader):
        """float32 ndarray [n_test_users, topk], rows in loader order (MF's ranking on (user_embedding, shared_embedding))."""
        data = getattr(getattr(test_loader, 'dataset', None), 'data', None)
        if isinstance(data, (list, tuple)) and len(data) and len(data[0]) == 2:
            users = np.fromiter((int(r[0]) for r in data), np.int64, len(data))
            cands = np.stack([np.asarray(r[1], dtype=np.int64) for r in data])
        else:
            us, cs = [], []
            for b_us, b_c in test_loader:
                us.append(torch.as_tensor(b_us).reshape(-1).to(torch.int64))
                cs.append(torch.as_tensor(b_c).to(torch.int64).reshape(us[-1].numel(), -1))
            if not us:
                return np.zeros((0,), np.float32)
            users, cands = torch.cat(us).numpy(), torch.cat(cs).numpy()
        if len(users) == 0:
            return np.zeros((0,), np.float32)
        if users.min() < 0 or users.max() >= self.user_num:
            raise IndexError('index out of range in self: test user id outside [0, user_num)')
        d_cands = torch.from_numpy(np.ascontiguousarray(cands)).to(self.device)
        ops.check_index_range(d_cands.reshape(-1, 1), (self.item_num,), ('candidate item',))
        k = min(self.topk, cands.shape[1])
        out = ops.mf_rank(self.user_embedding.weight, self.shared_embedding.weight, torch.from_numpy(users).to(self.device),
                          d_cands, k)
        return out.cpu().numpy()

    def full_rank(self, u):
        """int64 ndarray [topk] over every item; no masking of train items."""
        users = torch.tensor([int(u)], dtype=torch.int64, device=self.device)
        k = min(self.topk, self.item_num)
        return ops.mf_full_rank(self.user_embedding.weight, self.shared_embedding.weight, users, k)[0].cpu().numpy()
