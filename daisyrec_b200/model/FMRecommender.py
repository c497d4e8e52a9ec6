"""FM on the B200 path, with the reference's class name, config keys and methods
(daisy/model/FMRecommender.py:16-131).

FM here is MF's factor product plus first-order terms: ``pred = <p_u, q_i> + (u_bias[u] + i_bias[i]) + bias_``
(:61-68); the regulariser covers the factor rows only (:76-95), so the step is the MF step kernel
(``csrc/mf_bpr.cu``, GEN instantiation) with three extra scalar loads per score, three scalar ``RED``s per triple
and a sweep over the ``U + I + 1`` bias scalars in phase 2.  The biases live in ONE packed device vector
``[u_bias (U), i_bias (I), bias_ (1)]``; ``u_bias.weight`` / ``i_bias.weight`` / ``bias_`` are views of it.

    fit -> drb_gather_triples + drb_fm_train_steps     calc_loss -> drb_fm_train_steps(apply=0)
    rank -> drb_fm_rank     full_rank -> drb_fm_full_rank     predict / forward -> drb_fm_predict
"""
import torch

from .. import ops
from .AbstractRecommender import GeneralRecommender, _Table, _init_table, _INIT


class FM(GeneralRecommender):
    SUPPORTED_LOSSES = ('BPR', 'HL', 'TL', 'CL', 'SL')               # AbstractRecommender.py:79-88
    SUPPORTED_OPTIMIZERS = ('sgd', 'adam', 'adagrad', 'rmsprop')     # AbstractRecommender.py:53-60

    def __init__(self, config):
        """Same keys as the reference (FMRecommender.py:38-56): epochs, lr, reg_1, reg_2, user_num, item_num, factors,
        loss_type, optimizer ('default' -> sgd), init_method ('default' -> normal), early_stop, topk (+ gpu, logger)."""
        super().__init__(config)
        if self.world > 1:
            raise NotImplementedError('FM runs as independent replicas only (the sharded step covers MF)')
        self.epochs = config['epochs']
        self.lr = config['lr']
        self.reg_1 = config['reg_1']
        self.reg_2 = config['reg_2']
        self.user_num, self.item_num, self.factors = config['user_num'], config['item_num'], config['factors']
        self.loss_type = config['loss_type']
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'sgd'
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'normal'
        self.early_stop = config['early_stop']
        self.topk = config['topk']

        # The reference's CPU RNG consumption (:43-59): four nn.Embedding constructors (N(0,1) each, in this order), then
        # self.apply(_init_weight) re-initialises all four in registration order, then the two bias tables are zeroed.
        U, I, F = self.user_num, self.item_num, self.factors
        wu, wi = _init_table(U, F, None), _init_table(I, F, None)
        bu_, bi_ = _init_table(U, 1, None), _init_table(I, 1, None)
        for w in (wu, wi, bu_, bi_):
            _INIT[self.initializer](w)
        self.embed_user = _Table(wu.to(self.device))
        self.embed_item = _Table(wi.to(self.device))
        self.bias = torch.zeros(U + I + 1, dtype=torch.float32, device=self.device)
        self.u_bias = _Table(self.bias[:U].view(U, 1))
        self.i_bias = _Table(self.bias[U:U + I].view(I, 1))
        self.bias_ = self.bias[U + I:]

    # ------------------------------------------------------------------ plumbing
    def state_dict(self):
        return {'embed_user.weight': self.embed_user.weight, 'embed_item.weight': self.embed_item.weight,
                'u_bias.weight': self.u_bias.weight, 'i_bias.weight': self.i_bias.weight, 'bias_': self.bias_}

    def _hyper(self, opt):
        return ops.hyper(self.lr, self.reg_1, self.reg_2, opt, loss=str(self.loss_type).upper())

    def _begin_fit(self, opt):
        super()._begin_fit(opt)
        self._ws = ops.FMWorkspace(self.user_num, self.item_num, self.factors, opt, self.device)

    def _train_steps(self, bu, bi, bj, batch, first, n_steps):
        losses = ops.fm_train_steps(self.embed_user.weight, self.embed_item.weight, self.bias, self._ws, bu, bi, bj, batch,
                                    first, n_steps, self._hp, adam_step0=self._opt_steps)
        self._opt_steps += n_steps
        return losses

    # ------------------------------------------------------------------ reference surface (FMRecommender.py:61-131)
    def calc_loss(self, batch):
        """FMRecommender.py:70-97: 0-d fp32 loss of one (user, pos, neg) / (user, item, label) batch; no update."""
        self._check_loss_type()
        bu, bi, bj = self._planes(batch[:3])
        self._ensure(0)
        loss = ops.fm_train_steps(self.embed_user.weight, self.embed_item.weight, self.bias, self._ws, bu, bi, bj,
                                  max(1, bu.numel()), 0, 1, self._hp, adam_step0=self._opt_steps, apply=False)
        return loss.to(torch.float32).reshape(())

    def _rank_rows(self, users, cands, k):
        return ops.fm_rank(self.embed_user.weight, self.embed_item.weight, self.bias, users, cands, k)

    def _full_rank_rows(self, users, k):
        return ops.fm_full_rank(self.embed_user.weight, self.embed_item.weight, self.bias, users, k)

    def _score_pairs(self, u, i):
        return ops.fm_predict(self.embed_user.weight, self.embed_item.weight, self.bias, u.to(torch.int32), i.to(torch.int32))
