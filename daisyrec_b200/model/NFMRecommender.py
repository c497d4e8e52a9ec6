"""NFM + BPR on the B200 path, with the reference's class name, config keys and methods
(daisy/model/NFMRecommender.py:14-209).

Factor tables ``embed_user.weight`` / ``embed_item.weight``, the first-order terms in one packed vector (``u_bias.weight``,
``i_bias.weight``, ``bias_`` are views of it), the network (FM_layers' BatchNorm, the hidden Linear / BatchNorm layers and
``prediction.weight``) in one flat fp32 block ``net`` in module-registration order, the BatchNorm running statistics in
``running`` (mean, var per BatchNorm).  Training goes through ``drb_nfm_bpr_train_steps``; rank / full_rank / predict score
in eval mode (running statistics) through ``drb_nfm_scores`` + ``drb_topk_from_scores``.

Dropout (``config['dropout']``, reference default 0.5, :67,:88): in train mode the host draws exactly the masks torch's Dropout
modules would -- ``bernoulli_(1 - p)`` on the global CPU generator, forward(user, pos) first (FM_layers' Dropout, then the one
behind each activation), then forward(user, neg) -- and uploads them as bytes with the batch, so a step equals the reference's
and the global RNG ends where the reference's does.  That is a parity mechanism (one byte per activation and step through the
host); ``dropout = 0`` is the throughput configuration.

Two reference behaviours are NOT mirrored because they are failures, not results: with ``dropout = 0`` today's torch makes
the reference's own ``backward()`` raise (the in-place ``fm += ...`` of :120 aliases the activation output), and
``predict()`` with ``batch_norm`` feeds a 1-D row to BatchNorm1d, which rejects it.  Both work here.
"""
import numpy as np
import torch

from .. import ops
from .AbstractRecommender import GeneralRecommender, _Table, _init_table, _INIT


class NFM(GeneralRecommender):
    def __init__(self, config):
        super().__init__(config)
        if self.world > 1:
            raise NotImplementedError('NFM runs as independent replicas only (DESIGN.md, multi-GPU section)')
        self.factors = config['factors']
        self.act_function = config['act_function']
        self.num_layers = config['num_layers']
        self.batch_norm = bool(config['batch_norm'])
        self.dropout = float(config['dropout'] or 0.0)
        if not 0.0 <= self.dropout < 1.0:
            raise ValueError(f"dropout probability has to be in [0, 1), but got {self.dropout}")
        if self.act_function not in ops.NFM_ACT:
            raise NotImplementedError(f"act_function={self.act_function!r}: expected one of {sorted(ops.NFM_ACT)}")
        self.lr = config['lr']
        self.reg_1 = config['reg_1']
        self.reg_2 = config['reg_2']
        self.epochs = config['epochs']
        self.loss_type = config['loss_type']
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'xavier_normal'
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'sgd'
        self.early_stop = config['early_stop']
        self.topk = config['topk']
        self.user_num, self.item_num = config['user_num'], config['item_num']
        U, I, F, Ln = self.user_num, self.item_num, self.factors, self.num_layers

        # reference RNG stream (:55-108): constructors in registration order, then _init_weight
        import torch.nn as nn
        wu, wi = _init_table(U, F, None), _init_table(I, F, None)
        _init_table(U, 1, None); _init_table(I, 1, None)                 # u_bias / i_bias constructors (zeroed by _init_weight)
        linears = [nn.Linear(F, F) for _ in range(Ln)]                   # BatchNorm1d / Dropout constructors draw nothing
        prediction = nn.Linear(F, 1, bias=False)
        init = _INIT[self.initializer]
        with torch.no_grad():
            init(wu)
            init(wi)
            if Ln > 0:
                for lin in linears:
                    init(lin.weight)                                     # biases keep nn.Linear's own draw (:101-104)
                init(prediction.weight)
            else:
                prediction.weight.fill_(1.0)
            parts = []
            one, zero = torch.ones(F), torch.zeros(F)
            if self.batch_norm:
                parts += [one, zero]
            for lin in linears:
                parts += [lin.weight.reshape(-1), lin.bias.reshape(-1)]
                if self.batch_norm:
                    parts += [one, zero]
            parts.append(prediction.weight.reshape(-1))
            net = torch.cat(parts).contiguous()
        assert net.numel() == ops.nfm_param_count(F, Ln, self.batch_norm)
        self.embed_user = _Table(wu.to(self.device))
        self.embed_item = _Table(wi.to(self.device))
        self.bias = torch.zeros(U + I + 1, dtype=torch.float32, device=self.device)
        self.u_bias = _Table(self.bias[:U].view(U, 1))
        self.i_bias = _Table(self.bias[U:U + I].view(I, 1))
        self.bias_ = self.bias[U + I:]
        self.net = net.to(self.device)
        n_bn = (1 + Ln) if self.batch_norm else 0
        run = torch.zeros(n_bn * 2 * F, dtype=torch.float32)
        for k in range(n_bn):
            run[k * 2 * F + F:(k + 1) * 2 * F] = 1.0                     # running_var starts at 1
        self.running = run.to(self.device)
        td = str(config.get('tower_dtype', 'fp32')).lower()
        if td not in ('fp32', 'bf16'):
            raise ValueError(f"tower_dtype must be 'fp32' or 'bf16', got {td!r}")
        self._tower_dtype = 1 if td == 'bf16' else 0
        self._act = ops.NFM_ACT[self.act_function]
        self._rows = int(config.get('nfm_scratch_rows', 1 << 16))
        self._ws = None
        self._opt_steps = 0

    # ------------------------------------------------------------------ plumbing
    def parameters(self):
        return [self.embed_user.weight, self.embed_item.weight, self.u_bias.weight, self.i_bias.weight, self.bias_, self.net]

    def state_dict(self):
        return {'embed_user.weight': self.embed_user.weight, 'embed_item.weight': self.embed_item.weight,
                'u_bias.weight': self.u_bias.weight, 'i_bias.weight': self.i_bias.weight, 'bias_': self.bias_,
                'net': self.net, 'running': self.running}

    def load_state_dict(self, sd):
        for k, t in self.state_dict().items():
            if k in sd:
                t.copy_(torch.as_tensor(sd[k]).reshape(t.shape))

    def to(self, device):
        return self

    def _hyper(self, opt=None):
        return ops.hyper(self.lr, self.reg_1, self.reg_2, opt or self._optimizer_name())

    def _workspace(self, rows, opt, fresh=False):
        rows = max(int(rows), self._rows, 2)
        if fresh or self._ws is None or self._ws.max_rows < rows:
            if not fresh and self._ws is not None:
                raise RuntimeError('NFM scratch too small; set config["nfm_scratch_rows"] >= 2 * batch_size')
            self._ws = ops.NfmWorkspace(self.user_num, self.item_num, self.factors, self.num_layers, self.batch_norm, opt, rows,
                                        self.device)
        return self._ws

    def _begin_fit(self, opt):
        self._hp = self._hyper(opt)
        self._opt_steps = 0
        self._fit_opt = opt
        self._ws = None                                              # fresh optimiser state per fit()

    def _ensure(self, rows):
        if getattr(self, '_hp', None) is None or self._ws is None:
            if getattr(self, '_hp', None) is None:
                self._begin_fit(self._optimizer_name())
            self._workspace(rows, self._fit_opt, fresh=True)
        elif self._ws.max_rows < rows:
            self._workspace(rows, self._fit_opt)

    def _host_keep(self, rows_per_step):
        """The masks nn.Dropout would draw for steps of rows_per_step[k] triples, drawn by torch on the global CPU generator in
        the reference's order -> uint8 CUDA tensor [step][forward call][site][rows][F] (drb_nfm_bpr_train_steps)."""
        F, sites, keep = self.factors, 1 + self.num_layers, 1.0 - self.dropout
        parts = []
        for B in rows_per_step:
            for _side in (0, 1):                                          # forward(user, pos) draws first, then forward(user, neg)
                for _site in range(sites):
                    parts.append(torch.empty(B, F, dtype=torch.float32).bernoulli_(keep).to(torch.uint8).reshape(-1))
        return torch.cat(parts).to(self.device)

    def _dropping(self):
        return self.training and self.dropout > 0.0

    def _steps(self, bu, bi, bj, batch, first, n_steps, apply=True):
        """n_steps steps; in train mode with dropout > 0 the masks of every step are drawn first (in step order)."""
        kw = dict(adam_step0=self._opt_steps, tower_dtype=self._tower_dtype, apply=apply)
        args = (self.embed_user.weight, self.embed_item.weight, self.bias, self.net, self.running, self._ws, self._act)
        if not self._dropping():
            return ops.nfm_bpr_train_steps(*args, bu, bi, bj, batch, first, n_steps, self._hp, **kw)
        n = bu.numel()
        per_step = 2 * (1 + self.num_layers) * batch * self.factors
        chunk = max(1, (64 << 20) // per_step)                           # at most 64 MB of masks per call
        out, s = [], first
        while s < first + n_steps:
            k = min(chunk, first + n_steps - s)
            full = k if (s + k) * batch <= n else k - 1                   # a ragged last batch gets its own masks + call
            if full > 0:
                out.append(ops.nfm_bpr_train_steps(*args, bu, bi, bj, batch, s, full, self._hp, dropout=self.dropout,
                                                   keep=self._host_keep([batch] * full),
                                                   **dict(kw, adam_step0=self._opt_steps + (s - first))))
            if full < k:
                base = (s + full) * batch
                last = n - base
                out.append(ops.nfm_bpr_train_steps(*args, bu[base:], bi[base:], bj[base:], last, 0, 1, self._hp, dropout=self.dropout,
                                                   keep=self._host_keep([last]),
                                                   **dict(kw, adam_step0=self._opt_steps + (s + full - first))))
            s += k
        return torch.cat(out)

    def _train_steps(self, bu, bi, bj, batch, first, n_steps):
        if self._ws is None:
            self._workspace(2 * batch, self._fit_opt, fresh=True)
        losses = self._steps(bu, bi, bj, batch, first, n_steps)
        self._opt_steps += n_steps
        return losses

    # ------------------------------------------------------------------ reference surface
    def _scores(self, u, i):
        self._ensure(2)
        return ops.nfm_scores(self.embed_user.weight, self.embed_item.weight, self.bias, self.net, self.running, self._ws,
                              self._act, u, i, self._tower_dtype)

    def forward(self, user, item):
        """NFMRecommender.py:110-123 in eval mode (running statistics) for index tensors."""
        u = torch.as_tensor(user).to(self.device, torch.int32).reshape(-1).contiguous()
        i = torch.as_tensor(item).to(self.device, torch.int32).reshape(-1).contiguous()
        return self._scores(u, i)

    __call__ = forward

    def calc_loss(self, batch):
        """NFMRecommender.py:125-151 under train(): 0-d fp32 loss; the BatchNorm running statistics move as they do there."""
        self._check_loss_type()
        bu, bi, bj = (torch.as_tensor(b).to(self.device, torch.int32).contiguous() for b in batch[:3])
        self._ensure(2 * bu.numel())
        loss = self._steps(bu, bi, bj, bu.numel(), 0, 1, apply=False)
        return loss.to(torch.float32).reshape(())

    def train_step(self, batch):
        self._check_loss_type()
        bu, bi, bj = (torch.as_tensor(b).to(self.device, torch.int32).contiguous() for b in batch[:3])
        self._ensure(2 * bu.numel())
        was = self.training
        self.train()                                                 # a training step runs in train mode (dropout on)
        try:
            return float(self._train_steps(bu, bi, bj, bu.numel(), 0, 1).item())
        finally:
            self.train(was)

    def predict(self, u, i):
        return float(self.forward([int(u)], [int(i)]).item())

    def rank(self, test_loader):
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
        n, C = cands.shape
        d_cands = torch.from_numpy(np.ascontiguousarray(cands)).to(self.device)
        u_rep = torch.from_numpy(np.repeat(users, C).astype(np.int32)).to(self.device)
        scores = self._scores(u_rep, d_cands.reshape(-1).to(torch.int32).contiguous()).view(n, C).contiguous()
        return ops.topk_from_scores(scores, d_cands, min(self.topk, C)).cpu().numpy()

    def full_rank(self, u):
        items = torch.arange(self.item_num, dtype=torch.int32, device=self.device)
        users = torch.full((self.item_num,), int(u), dtype=torch.int32, device=self.device)
        scores = self._scores(users, items).view(1, -1).contiguous()
        return ops.topk_from_scores(scores, None, min(self.topk, self.item_num))[0].cpu().numpy()
