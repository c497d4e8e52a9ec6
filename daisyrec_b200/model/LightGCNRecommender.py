"""LightGCN + BPR on the B200 path, with the reference's class name, config keys and methods
(daisy/model/LightGCNRecommender.py:23-211).

The ego table E0 = cat(embed_user.weight, embed_item.weight) is one contiguous device tensor
(``embed_user.weight`` / ``embed_item.weight`` are views of it); the normalised adjacency is built once
on the host exactly as ``get_norm_adj_mat`` does (:73-107, values bit-identical) and lives on the device as
segmented CSR.  Every step runs L forward + L backward sparse products and the fused BPR / Adam kernels
through ``drb_lgcn_bpr_train_steps``; rank / full_rank / predict score with the cached propagated
tables (``restore_user_e`` / ``restore_item_e``, :64-65) through the MF rank kernels.
"""
import numpy as np
import torch

from .. import ops
from .AbstractRecommender import GeneralRecommender, _Table, _init_table, _INIT


class LightGCN(GeneralRecommender):
    def __init__(self, config):
        super().__init__(config)
        if self.world > 1:
            raise NotImplementedError('LightGCN runs as independent replicas only (DESIGN.md, multi-GPU section)')
        self.epochs = config['epochs']
        self.lr = config['lr']
        self.topk = config['topk']
        self.user_num = config['user_num']
        self.item_num = config['item_num']
        self.interaction_matrix = config['inter_matrix']            # scipy COO from utils.get_inter_matrix
        self.factors = config['factors']
        self.num_layers = config['num_layers']
        self.reg_1 = config['reg_1']
        self.reg_2 = config['reg_2']
        self.loss_type = config['loss_type']
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'adam'
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'xavier_uniform'
        self.early_stop = config['early_stop']

        # reference init stream: two nn.Embedding constructors, then apply(_init_weight) (LightGCNRecommender.py:53-68)
        wu = _init_table(self.user_num, self.factors, None)
        wi = _init_table(self.item_num, self.factors, None)
        _INIT[self.initializer](wu)
        _INIT[self.initializer](wi)
        self.E0 = torch.cat([wu, wi]).contiguous().to(self.device)
        self.embed_user = _Table(self.E0[:self.user_num])
        self.embed_item = _Table(self.E0[self.user_num:])
        self.restore_user_e = None
        self.restore_item_e = None

        m = self.interaction_matrix
        # optional B200 key 'adj_builder': 'host' (default; numpy restatement of get_norm_adj_mat, values bit-identical to
        # scipy's) | 'device' (sorted CSR + transpose + D^-1/2 A D^-1/2 built by csr.cu; 1/sqrt instead of pow: fp32
        # values equal except on rare rounding ties)
        if str(config.get('adj_builder', 'host')) == 'device':
            row_ptr, col, val = ops.lgcn_build_adj(torch.from_numpy(np.ascontiguousarray(m.row, np.int32)).to(self.device),
                                                   torch.from_numpy(np.ascontiguousarray(m.col, np.int32)).to(self.device),
                                                   self.user_num, self.item_num)
        else:
            row_ptr, col, val = ops.lgcn_norm_adj(np.asarray(m.row), np.asarray(m.col), self.user_num, self.item_num)
        self.graph = ops.LgcnGraph(row_ptr, col, val, self.device)

    # ------------------------------------------------------------------ plumbing
    def state_dict(self):
        return {'embed_user.weight': self.embed_user.weight, 'embed_item.weight': self.embed_item.weight}

    def _tables_changed(self):
        self.restore_user_e = self.restore_item_e = None             # LightGCNRecommender.py:133-134

    def _begin_fit(self, opt):
        super()._begin_fit(opt)
        self._ws = ops.LgcnWorkspace(self.user_num, self.item_num, self.factors, opt, self.device)

    def _train_steps(self, bu, bi, bj, batch, first, n_steps):
        self._tables_changed()
        losses = ops.lgcn_bpr_train_steps(self.E0, self._ws, self.graph, self.num_layers, bu, bi, bj, batch, first,
                                          n_steps, self._hp, adam_step0=self._opt_steps)
        self._opt_steps += n_steps
        return losses

    # ------------------------------------------------------------------ reference surface
    def forward(self):
        """LightGCNRecommender.py:117-129 -> (user_embedding, item_embedding) after propagation + layer mean."""
        self._ensure(0)
        Em = ops.lgcn_propagate(self.E0, self._ws, self.graph, self.num_layers)
        return Em[:self.user_num], Em[self.user_num:]

    def calc_loss(self, batch):
        self._check_loss_type()
        bu, bi, bj = self._planes(batch[:3])
        self._ensure(0)
        self._tables_changed()
        loss = ops.lgcn_bpr_train_steps(self.E0, self._ws, self.graph, self.num_layers, bu, bi, bj, bu.numel(), 0, 1,
                                        self._hp, apply=False)
        return loss.to(torch.float32).reshape(())

    def _score_tables(self):
        """The propagated tables (restore_user_e / restore_item_e), recomputed after a step or a load."""
        if self.restore_user_e is None or self.restore_item_e is None:
            self.restore_user_e, self.restore_item_e = self.forward()
        return self.restore_user_e, self.restore_item_e
