"""Multi-VAE on the B200 path, with the reference's class name, config keys and methods (daisy/model/VAECFRecommender.py).

Every parameter lives in ONE flat fp32 block ``net`` in module-registration order (encoder Linears, then decoder Linears;
weight then bias each, each zero-padded to a multiple of 4 floats so that it starts 16-byte aligned), so one dense optimiser
launch moves them all.  The first encoder weight is stored transposed, [item_num, h_1], so that the sparse encoder reads an
item's row contiguously; ``state_dict()`` hands out torch's [out, in] views of the block.  The rating rows R are a device CSR built once from ``config['history_item_id' / 'history_item_value']``
(or from ``config['train_csr']``), never a dense [batch, item_num] matrix.

    fit / calc_loss / train_step -> drb_vae_train_steps (one launch per epoch with the Philox engine)
    rank      -> drb_vae_forward(hidden rows) + drb_vae_candidate_scores + drb_topk_from_scores
    full_rank / predict / forward -> drb_vae_forward (eval mode: no dropout, z = mu)

Dropout and the reparameterisation noise in train mode (``config['dropout_engine']``, as NeuMF's):
    'torch'  : torch draws them on the host from the global CPU generator in the reference's order -- per step the
               [B, item_num] keep-mask (``bernoulli_(1 - p)``; nothing with dropout 0), then ``randn(B, latent_dim // 2)`` --
               so a step equals the reference's and the global RNG ends where the reference's does.  The masks are bit-packed
               and uploaded: one host bernoulli_ per step, meant for small item counts.
    'philox' : counter-based masks and Box-Muller noise generated inside the kernels (same distributions, another stream).
    'auto'   : 'torch' while a step's mask stays under 4 M elements (ml-100k at batch 256: 0.43 M), 'philox' above.
"""
import math

import numpy as np
import torch
from tqdm import tqdm

from .. import ops
from .AbstractRecommender import GeneralRecommender, _INIT, dropout_engine, dropout_rate, loader_plan, mask_segments, tower_dtype


def rating_csr(history_item_id, history_item_value, item_num, device):
    """The rating rows get_user_rating_matrix builds (AbstractRecommender.py:147-158), as a device CSR.  index_put_ without
    accumulate writes a row's padded history in order, so the LAST write to a (user, item) cell wins -- including the
    (item 0, 0.0) padding written after a shorter row's real entries, which erases item 0 from that row -- and a zero value
    leaves the cell empty.  -> ops.VaeRatings (row_ptr int64 [U+1], ascending col int32, val float32)."""
    hid = torch.as_tensor(history_item_id).to(device, torch.int64)
    hval = torch.as_tensor(history_item_value).to(device, torch.float32)
    if hid.dim() != 2 or hval.shape != hid.shape:
        raise ValueError('history_item_id / history_item_value must be two [user_num, max_len] tensors of the same shape')
    U, W = hid.shape
    if hid.numel() and (int(hid.min()) < 0 or int(hid.max()) >= item_num):
        raise IndexError(f'history_item_id holds an item id outside [0, {item_num})')
    key = (torch.arange(U, device=device, dtype=torch.int64)[:, None] * item_num + hid).reshape(-1)
    skey, order = torch.sort(key, stable=True)                      # a cell's writes stay in write order
    val = hval.reshape(-1)[order]
    last = torch.ones_like(skey, dtype=torch.bool)
    last[:-1] = skey[1:] != skey[:-1]
    keep = last & (val != 0)
    skey, val = skey[keep], val[keep].contiguous()
    row = skey // item_num
    col = (skey - row * item_num).to(torch.int32).contiguous()
    row_ptr = torch.zeros(U + 1, dtype=torch.int64, device=device)
    row_ptr[1:] = torch.cumsum(torch.bincount(row, minlength=U), 0)
    return ops.VaeRatings(row_ptr, col, val)


def _pad4(t):
    """A block part followed by zeros up to a multiple of 4 floats (the device layout's alignment)."""
    return torch.cat([t, t.new_zeros((-t.numel()) % 4)])


class VAECF(GeneralRecommender):
    def __init__(self, config):
        """Same keys as the reference: user_num, item_num, history_item_id, history_item_value, mlp_hidden_size (None ->
        [600]), latent_dim, dropout, anneal_cap, total_anneal_steps, lr, epochs, optimizer ('default' -> adam), init_method
        ('default' -> xavier_normal), early_stop, topk (+ gpu, logger).  Optional: train_csr = (row_ptr, col) stands in for the
        padded history (every rating 1.0; the padding's erasure of item 0 does not happen then), tower_dtype ('fp32' | 'bf16'),
        dropout_engine ('auto' | 'torch' | 'philox'), vae_scratch_rows (rows of activation scratch, default 256)."""
        super().__init__(config)
        if self.world > 1:
            raise NotImplementedError('VAECF runs as independent replicas only (DESIGN.md, multi-GPU section)')
        self.epochs = config['epochs']
        self.lr = config['lr']
        self.dropout = dropout_rate(config['dropout'])
        self.layers = list(config['mlp_hidden_size']) if config['mlp_hidden_size'] is not None else [600]
        self.lat_dim = int(config['latent_dim'])
        self.anneal_cap = config['anneal_cap']
        self.total_anneal_steps = config['total_anneal_steps']
        self.user_num, self.item_num = config['user_num'], config['item_num']
        self.update = 0
        self.encode_layer_dims = [self.item_num] + self.layers + [self.lat_dim]
        self.decode_layer_dims = [int(self.lat_dim / 2)] + self.encode_layer_dims[::-1][1:]
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'adam'
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'xavier_normal'
        self.early_stop = config['early_stop']
        self.topk = config['topk']
        if self.lat_dim < 2 or len(self.layers) > 8:
            raise ValueError('VAECF: latent_dim >= 2 and at most 8 hidden layers')

        # the reference's CPU RNG stream: every nn.Linear constructor in registration order (encoder, then decoder), then
        # self.apply(_init_weight) re-initialises each weight in the same order and zeroes the biases
        import torch.nn as nn
        E, D = self.encode_layer_dims, self.decode_layer_dims
        lins = [nn.Linear(a, b) for a, b in zip(E[:-1], E[1:])] + [nn.Linear(a, b) for a, b in zip(D[:-1], D[1:])]
        init = _INIT[self.initializer]
        with torch.no_grad():
            parts = []
            for k, lin in enumerate(lins):
                init(lin.weight)
                w = lin.weight.t() if k == 0 else lin.weight                 # encoder.0 is stored [item_num, h_1]
                parts += [_pad4(w.reshape(-1)), _pad4(torch.zeros(lin.out_features))]
            net = torch.cat(parts).contiguous()
        del lins
        assert net.numel() == ops.vae_param_count(self.item_num, self.layers, self.lat_dim)
        self.net = net.to(self.device)
        self._views = self._param_views()

        csr = config.get('train_csr', None)
        if csr is not None:
            row_ptr, col = csr
            col = torch.from_numpy(np.ascontiguousarray(col, np.int32)).to(self.device)
            self.R = ops.VaeRatings(torch.from_numpy(np.ascontiguousarray(row_ptr, np.int64)).to(self.device), col,
                                    torch.ones(col.numel(), dtype=torch.float32, device=self.device))
        else:
            self.R = rating_csr(config['history_item_id'], config['history_item_value'], self.item_num, self.device)

        self._tower_dtype = tower_dtype(config)
        self.dropout_engine = dropout_engine(config)
        self._rows = int(config.get('vae_scratch_rows', 256))
        self._philox_seed = None

    # ------------------------------------------------------------------ plumbing
    def _param_views(self):
        """state_dict names -> views of the flat block, in torch's layout ([out, in] weights)."""
        views, o = {}, 0
        for side, dims in (('encoder', self.encode_layer_dims), ('decoder', self.decode_layer_dims)):
            for k, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
                w = self.net[o:o + a * b]
                views[f'{side}.{2 * k}.weight'] = w.view(a, b).t() if (side == 'encoder' and k == 0) else w.view(b, a)
                o += -(-a * b // 4) * 4
                views[f'{side}.{2 * k}.bias'] = self.net[o:o + b]
                o += -(-b // 4) * 4
        return views

    def state_dict(self):
        return dict(self._views)

    def _check_loss_type(self):
        """The ELBO is VAECF's only loss: its config has no loss_type."""

    def _hyper(self, opt):
        return ops.hyper(self.lr, 0.0, 0.0, opt)

    def _ensure(self, rows):
        if self._hp is None:
            self._begin_fit(self._optimizer_name())
        rows = max(int(rows), self._rows, 1)
        if self._ws is None or self._ws.max_rows < rows:
            if self._ws is not None and self._opt_steps > 0:
                raise RuntimeError('VAECF scratch too small; set config["vae_scratch_rows"] >= batch_size')
            self._ws = ops.VaeWorkspace(self.item_num, self.layers, self.lat_dim, self._fit_opt, rows, self.device)

    def _host_rng(self, batch):
        """True when the step's dropout mask and eps come from torch's global CPU generator (the reference's stream)."""
        if not self.training:
            return False
        if self.dropout_engine == 'auto':
            return batch * self.item_num <= (1 << 22)
        return self.dropout_engine == 'torch'

    def _seed(self):
        """Philox key: drawn from torch's global RNG the first time the kernels need it, so torch.manual_seed makes runs
        reproducible."""
        if self._philox_seed is None:
            self._philox_seed = int(torch.empty((), dtype=torch.int64).random_().item())
        return self._philox_seed

    def _host_draws(self, rows_per_step):
        """Per step, in the reference's order: the keep-mask F.dropout draws (none when dropout = 0), then the reparameterisation
        noise -> (int32 bit-packed masks or None, float32 eps) CUDA tensors."""
        words, eps = [], []
        half = self.lat_dim // 2
        for B in rows_per_step:
            if self.dropout > 0.0:
                m = torch.empty(B, self.item_num, dtype=torch.float32).bernoulli_(1 - self.dropout).numpy() != 0
                bits = np.packbits(m.reshape(-1), bitorder='little')
                words.append(np.pad(bits, (0, (-len(bits)) % 4)).view(np.int32))
            eps.append(torch.randn(B, half, dtype=torch.float32).reshape(-1))
        keep = torch.from_numpy(np.concatenate(words)).to(self.device) if words else None
        return keep, torch.cat(eps).to(self.device)

    def _steps(self, users, batch, n_steps, apply=True):
        """n_steps steps over the int32 device ids `users` (a ragged last batch holds the rest) -> float64 losses [n_steps]."""
        kw = dict(apply=apply, training=self.training, tower_dtype=self._tower_dtype, dropout=self.dropout,
                  anneal_cap=float(self.anneal_cap), total_anneal_steps=int(self.total_anneal_steps))
        args = (self.net, self._ws, self.R)
        if not self._host_rng(batch):
            seed = self._seed() if self.training else 0
            out = ops.vae_train_steps(*args, users, batch, 0, n_steps, self._hp, adam_step0=self._opt_steps, seed=seed,
                                      update0=self.update, **kw)
            self.update += n_steps
            if apply:
                self._opt_steps += n_steps
            return out
        out = []
        for s, k, rows in mask_segments(users.numel(), batch, 0, n_steps, batch * self.item_num // 8):
            keep, eps = self._host_draws([rows] * k)
            out.append(ops.vae_train_steps(*args, users[s * batch:s * batch + k * rows], rows, 0, k, self._hp,
                                           adam_step0=self._opt_steps, keep=keep, eps=eps, update0=self.update, **kw))
            self.update += k
            if apply:
                self._opt_steps += k
        return torch.cat(out)

    def _users(self, batch):
        """Host-checked user ids -> int32 device ids; ids in [-user_num, 0) wrap as history_item_id[user] does."""
        u = torch.as_tensor(batch).reshape(-1).to(torch.int64)
        if u.numel() and (int(u.min()) < -self.user_num or int(u.max()) >= self.user_num):
            raise IndexError(f'index out of range: user id outside [0, {self.user_num})')
        u = torch.where(u < 0, u + self.user_num, u)                     # torch indexing semantics of history_item_id[user]
        return u.to(self.device, torch.int32).contiguous()

    # ------------------------------------------------------------------ training
    def _loader_plan(self, train_loader):
        """A plain DataLoader(AEDataset): a 1-D array of user ids read in DataLoader order."""
        return loader_plan(train_loader, lambda data: data.ndim == 1)

    def _fit_epoch_bulk(self, plan, epoch):
        """One epoch over the loader's own permutation of the user ids, so the batches are the reference's."""
        data, bs, shuffle, drop_last, gen = plan
        T = len(data)
        key = (id(data), data.ctypes.data, T)
        if getattr(self, '_users_key', None) != key:
            self._users_dev = self._users(torch.from_numpy(np.ascontiguousarray(data, np.int64)))
            self._users_key = key
        d_perm = self._device_permutation(T, shuffle, gen)              # consumes the global RNG as the DataLoader does
        users = self._users_dev if d_perm is None else self._users_dev.index_select(0, d_perm).contiguous()
        n_use = (T // bs) * bs if drop_last else T
        nsteps = (n_use + bs - 1) // bs
        pbar = tqdm(total=nsteps, disable=not self.show_progress)
        pbar.set_description(f'[Epoch {epoch:03d}]')
        current_loss = 0.
        if nsteps:
            self._ensure(bs)
            current_loss = float(self._steps(users[:n_use], bs, nsteps).sum().item())   # raises ValueError on NaN
        pbar.update(nsteps)
        pbar.set_postfix(loss=current_loss)
        pbar.close()
        return current_loss

    def calc_loss(self, batch):
        """VAECFRecommender.py:92-110 in the current mode: 0-d fp32 loss; counts one update of the KL anneal; no parameter
        change."""
        users = self._users(batch)
        self._ensure(users.numel())
        return self._steps(users, max(1, users.numel()), 1, apply=False).to(torch.float32).reshape(())

    def train_step(self, batch):
        """zero_grad + calc_loss + backward + optimizer.step on one batch of user ids (train mode) -> loss.item()."""
        users = self._users(batch)
        self._ensure(users.numel())
        was = self.training
        self.train()
        try:
            return float(self._steps(users, max(1, users.numel()), 1).item())
        finally:
            self.train(was)

    # ------------------------------------------------------------------ inference (eval mode)
    def forward(self, user):
        """forward() of VAECFRecommender.py:79-90 in eval mode for the rating rows of `user` -> (decoder output
        [n, item_num], mu, logvar).  Unlike the reference, whose forward() takes a dense [B, item_num] rating matrix, this
        takes the users' ids (integers, 0-d or 1-d): the rating rows already live on the device."""
        t = torch.as_tensor(user)
        if t.is_floating_point() or t.is_complex() or t.dim() > 1:
            raise TypeError('VAECF.forward takes user ids (an integer scalar or 1-d array), not a dense rating matrix; '
                            f'got a {t.dim()}-d {t.dtype} tensor')
        u = self._users(t)
        scores = self._scores(u)
        h = ops.vae_forward(self.net, self._ws, self.R, u, 'latent', self._tower_dtype)
        return scores, h[:, :int(self.lat_dim / 2)], h[:, math.ceil(self.lat_dim / 2):]

    def _scores(self, users):
        self._ensure(1)
        return ops.vae_forward(self.net, self._ws, self.R, users, 'scores', self._tower_dtype)

    def _score_pairs(self, u, i):
        return self._scores(u).gather(1, i.to(torch.int64).reshape(-1, 1)).reshape(-1)

    def _rank_rows(self, users, cands, k):
        """The decoder output at the candidates only."""
        self._ensure(1)
        hidden = ops.vae_forward(self.net, self._ws, self.R, users, 'hidden', self._tower_dtype)
        return ops.topk_from_scores(ops.vae_candidate_scores(self.net, self._ws, hidden, cands), cands, k)

    def _full_rank_rows(self, users, k):
        return ops.topk_from_scores(self._scores(users), None, k)
