"""NGCF + BPR on the B200 path, with the reference's class name, config keys and methods
(daisy/model/NGCFRecommender.py:61-252; node_dropout = 0).

The ego table E0 = cat(embed_user.weight, embed_item.weight) is one contiguous device tensor; the BiGNN layers live in
one flat fp32 block (``gnn``: per layer W1, b1, W2, b2 in module-registration order); the normalised adjacency is
LightGCN's (``get_norm_adj_mat`` :125-146 is the same arithmetic) as segmented CSR on the device.  A step runs through
``drb_ngcf_bpr_train_steps`` (sparse products, GEMMs, the row-wise LeakyReLU / normalise kernels and the shared BPR /
optimiser phases); rank / full_rank / predict score the cached concatenated representation (``restore_user_e`` /
``restore_item_e``, :99-100) with the MF rank kernels.

Message dropout (``mess_dropout``, reference default 0.1): forward() builds ``nn.Dropout(mess_dropout)`` per layer (:164), a
module in training mode, so the reference drops on EVERY forward() -- the one behind rank() / full_rank() / predict() as well.
The host draws exactly those masks (one ``bernoulli_(1 - p)`` per layer over its [n, width] output, torch's global CPU
generator) and uploads them as bytes; the kernels apply them between LeakyReLU and the row normalisation, forward and backward.
That is a parity mechanism (one byte per node and width through the host per forward); ``mess_dropout = 0`` is the throughput
configuration.  ``node_dropout`` (reference default 0; a sparse dropout of the adjacency) is refused when non-zero.
"""
import numpy as np
import torch

from .. import ops
from .AbstractRecommender import GeneralRecommender, _Table, _init_table, _INIT, dropout_rate, tower_dtype


class NGCF(GeneralRecommender):
    def __init__(self, config):
        super().__init__(config)
        if self.world > 1:
            raise NotImplementedError('NGCF runs as independent replicas only (DESIGN.md, multi-GPU section)')
        self.epochs = config['epochs']
        self.lr = config['lr']
        self.topk = config['topk']
        self.user_num = config['user_num']
        self.item_num = config['item_num']
        self.interaction_matrix = config['inter_matrix']            # scipy COO from utils.get_inter_matrix
        self.embedding_size = config['factors']
        hidden = config['hidden_size_list'] if config.get('hidden_size_list') is not None else [64, 64, 64]
        self.hidden_size_list = [self.embedding_size] + list(hidden)
        self.node_dropout = config['node_dropout']
        self.message_dropout = config['mess_dropout']
        if float(self.node_dropout or 0.0) != 0.0:
            raise NotImplementedError('NGCF on the B200 path runs with node_dropout = 0 (the reference default; a sparse dropout '
                                      'of the adjacency drawn from the torch RNG)')
        self.message_dropout = dropout_rate(self.message_dropout)
        self.reg_1 = config['reg_1']
        self.reg_2 = config['reg_2']
        self.loss_type = config['loss_type']
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'adam'
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'xavier_normal'
        self.early_stop = config['early_stop']
        dims = self.hidden_size_list
        if any(int(d) < 1 or int(d) > 256 for d in dims):
            raise NotImplementedError('NGCF on the B200 path supports layer widths up to 256')

        # reference RNG stream (:95-116): two nn.Embedding constructors, per BiGNN layer two nn.Linear constructors, then
        # apply(_init_weight) over embed_user, embed_item and every (linear, interact_transform) pair
        import torch.nn as nn
        wu = _init_table(self.user_num, self.embedding_size, None)
        wi = _init_table(self.item_num, self.embedding_size, None)
        layers = [(nn.Linear(i, o), nn.Linear(i, o)) for i, o in zip(dims[:-1], dims[1:])]
        init = _INIT[self.initializer]
        with torch.no_grad():
            init(wu)
            init(wi)
            parts = []
            for lin, inter in layers:
                for mod in (lin, inter):
                    init(mod.weight)
                    mod.bias.zero_()
                parts += [lin.weight.reshape(-1), lin.bias.reshape(-1), inter.weight.reshape(-1), inter.bias.reshape(-1)]
            gnn = torch.cat(parts).contiguous()
        assert gnn.numel() == ops.ngcf_param_count(dims)
        self.E0 = torch.cat([wu, wi]).contiguous().to(self.device)
        self.embed_user = _Table(self.E0[:self.user_num])
        self.embed_item = _Table(self.E0[self.user_num:])
        self.gnn = gnn.to(self.device)
        self.restore_user_e = None
        self.restore_item_e = None
        m = self.interaction_matrix
        row_ptr, col, val = ops.lgcn_norm_adj(np.asarray(m.row), np.asarray(m.col), self.user_num, self.item_num)
        self.graph = ops.LgcnGraph(row_ptr, col, val, self.device)
        self._tower_dtype = tower_dtype(config)

    # ------------------------------------------------------------------ plumbing
    def state_dict(self):
        return {'embed_user.weight': self.embed_user.weight, 'embed_item.weight': self.embed_item.weight, 'gnn': self.gnn}

    def _tables_changed(self):
        self.restore_user_e = self.restore_item_e = None             # NGCFRecommender.py:175-176

    def _begin_fit(self, opt):
        super()._begin_fit(opt)
        self._ws = ops.NgcfWorkspace(self.user_num, self.item_num, self.hidden_size_list, opt, self.device)

    def _host_keep(self, n_forwards):
        """The masks nn.Dropout(mess_dropout) draws for n_forwards forward() calls: per call one bernoulli_ per layer over its
        [n, width] output on torch's global CPU generator -> uint8 CUDA tensor (None without message dropout)."""
        if self.message_dropout <= 0.0:
            return None
        n, keep = self.user_num + self.item_num, 1.0 - self.message_dropout
        parts = []
        for _ in range(n_forwards):
            for width in self.hidden_size_list[1:]:
                parts.append(torch.empty(n, int(width), dtype=torch.float32).bernoulli_(keep).to(torch.uint8).reshape(-1))
        return torch.cat(parts).to(self.device)

    def _train_steps(self, bu, bi, bj, batch, first, n_steps):
        self._tables_changed()
        kw = dict(tower_dtype=self._tower_dtype, dropout=self.message_dropout)
        if self.message_dropout <= 0.0:
            losses = ops.ngcf_bpr_train_steps(self.E0, self.gnn, self._ws, self.graph, bu, bi, bj, batch, first, n_steps, self._hp,
                                              adam_step0=self._opt_steps, **kw)
        else:                                                        # masks of at most 64 MB per call, drawn in step order
            chunk = max(1, (64 << 20) // max(1, ops.ngcf_keep_bytes(self._ws)))
            out = []
            for s in range(first, first + n_steps, chunk):
                k = min(chunk, first + n_steps - s)
                out.append(ops.ngcf_bpr_train_steps(self.E0, self.gnn, self._ws, self.graph, bu, bi, bj, batch, s, k, self._hp,
                                                    adam_step0=self._opt_steps + (s - first), keep=self._host_keep(k), **kw))
            losses = torch.cat(out)
        self._opt_steps += n_steps
        return losses

    # ------------------------------------------------------------------ reference surface
    def forward(self):
        """NGCFRecommender.py:157-172 -> (user_all_embeddings, item_all_embeddings): the concatenated layer outputs."""
        self._ensure(0)
        rep = ops.ngcf_forward(self.E0, self.gnn, self._ws, self.graph, self._tower_dtype, dropout=self.message_dropout,
                               keep=self._host_keep(1))              # the reference's forward() always drops (:164)
        return rep[:self.user_num], rep[self.user_num:]

    def calc_loss(self, batch):
        self._check_loss_type()
        bu, bi, bj = self._planes(batch[:3])
        self._ensure(0)
        self._tables_changed()
        loss = ops.ngcf_bpr_train_steps(self.E0, self.gnn, self._ws, self.graph, bu, bi, bj, bu.numel(), 0, 1, self._hp,
                                        apply=False, tower_dtype=self._tower_dtype, dropout=self.message_dropout,
                                        keep=self._host_keep(1))
        return loss.to(torch.float32).reshape(())

    def _score_tables(self):
        """The propagated tables (restore_user_e / restore_item_e), recomputed after a step or a load."""
        if self.restore_user_e is None or self.restore_item_e is None:
            self.restore_user_e, self.restore_item_e = self.forward()
        return self.restore_user_e, self.restore_item_e
