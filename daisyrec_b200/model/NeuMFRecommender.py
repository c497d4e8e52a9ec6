"""NeuMF + BPR on the B200 path, with the reference's class name, config keys and methods
(daisy/model/NeuMFRecommender.py:15-232; model_name 'NeuMF', 'GMF', 'MLP' and 'NeuMF-pre').

Four raw fp32 embedding tables (``embed_user_GMF/embed_item_GMF/embed_user_MLP/embed_item_MLP`` ``.weight``)
and the tower as one flat fp32 block (``tower``; per layer weight then bias, then predict weight and bias).
No nn.Module in the compute path, no autograd, no torch.optim: fit / calc_loss / rank / full_rank / predict
forward to ``drb_neumf_*`` (include/daisyrec_b200.h).  torch.nn is touched at construction time only, to
consume the global CPU RNG exactly as the reference's constructor does (bit-identical initial weights).
"""
import numpy as np
import torch

from .. import ops
from .AbstractRecommender import GeneralRecommender, _Table, _INIT, dropout_engine, dropout_rate, mask_segments, tower_dtype


class NeuMF(GeneralRecommender):
    def __init__(self, config):
        super().__init__(config)
        if self.world > 1:
            raise NotImplementedError('NeuMF runs as independent replicas only (DESIGN.md, multi-GPU section)')
        self.lr = config['lr']
        self.epochs = config['epochs']
        self.reg_1 = config['reg_1']
        self.reg_2 = config['reg_2']
        self.model = config['model_name']
        self.user_num, self.item_num = config['user_num'], config['item_num']
        self.factors, self.num_layers = config['factors'], config['num_layers']
        self.loss_type = config['loss_type']
        self.optimizer = config['optimizer'] if config['optimizer'] != 'default' else 'adam'
        self.initializer = config['init_method'] if config['init_method'] != 'default' else 'xavier_normal'
        self.early_stop = config['early_stop']
        self.topk = config['topk']
        if self.model not in ops.NEUMF_MODE:
            raise ValueError(f"model_name={self.model!r}: expected one of {sorted(ops.NEUMF_MODE)}")
        self._mode = ops.NEUMF_MODE[self.model]                       # 0 NeuMF / NeuMF-pre, 1 GMF, 2 MLP
        self.GMF_model = config.get('GMF_model', None)
        self.MLP_model = config.get('MLP_model', None)
        self.dropout = dropout_rate(config['dropout'])
        if self.factors % 4 != 0:
            raise NotImplementedError('NeuMF on the B200 path needs factors to be a multiple of 4 (128-bit rows)')
        F, Ln = self.factors, self.num_layers
        D = F * (2 ** (Ln - 1))
        self.mlp_dim = D

        # ---- reference RNG stream (NeuMFRecommender.py:52-71 constructors, :81-96 _init_weight) on the CPU
        import torch.nn as nn
        embs = [nn.Embedding(self.user_num, F), nn.Embedding(self.item_num, F),
                nn.Embedding(self.user_num, D), nn.Embedding(self.item_num, D)]
        linears = [nn.Linear(F * (2 ** (Ln - i)), F * (2 ** (Ln - i)) // 2) for i in range(Ln)]
        predict = nn.Linear(F if self.model in ('MLP', 'GMF') else 2 * F, 1)          # :63-68
        init = _INIT[self.initializer]
        with torch.no_grad():
            if self.model != 'NeuMF-pre':
                for e in embs:
                    init(e.weight)
                bare = {'normal': torch.nn.init.normal_, 'uniform': torch.nn.init.uniform_,
                        'xavier_normal': torch.nn.init.xavier_normal_, 'xavier_uniform': torch.nn.init.xavier_uniform_}
                for lin in linears:
                    bare[self.initializer](lin.weight)  # :88-90 passes NO param config to the hidden layers: 'normal' is N(0, 1)
                init(predict.weight)
                for lin in linears + [predict]:
                    lin.bias.zero_()
            else:
                self._load_pretrained(embs, linears, predict)
            parts = []
            for lin in linears:
                parts += [lin.weight.reshape(-1), lin.bias.reshape(-1)]
            parts += [predict.weight.reshape(-1), predict.bias.reshape(-1)]
            tower = torch.cat(parts).contiguous()
        assert tower.numel() == ops.neumf_param_count(F, Ln, self._mode)
        self.embed_user_GMF = _Table(embs[0].weight.detach().to(self.device).contiguous())
        self.embed_item_GMF = _Table(embs[1].weight.detach().to(self.device).contiguous())
        self.embed_user_MLP = _Table(embs[2].weight.detach().to(self.device).contiguous())
        self.embed_item_MLP = _Table(embs[3].weight.detach().to(self.device).contiguous())
        self.tower = tower.to(self.device)
        self._rows = int(config.get('neumf_scratch_rows', 1 << 16))
        # optional B200 key: 'fp32' (CUDA cores, parity path, default) | 'bf16' (tcgen05 tensor cores, BASELINE config 3)
        #                   | 'fused' (bf16 tcgen05, the whole tower step of a 64-triple tile inside one CTA: activations stay in
        #                     shared / tensor memory; factors = 32, num_layers = 2, dropout 0 -- other shapes run as 'bf16')
        self._tower_dtype = tower_dtype(config, ('fp32', 'bf16', 'fused'))
        # optional B200 key: how nn.Dropout's masks (:61) are produced in train mode.
        #   'torch'  : torch itself draws them on the host, in the reference's order (per step: the pos forward's L masks, then
        #              the neg forward's), from the global CPU generator; they are bit-packed and uploaded -- the reference's
        #              masks bit for bit.  Costs one host bernoulli_ per layer and forward: meant for small batches.
        #   'philox' : counter-based masks generated inside the kernels (same distribution, another stream).
        #   'auto'   : 'torch' while a step's masks stay under 4 M elements (the reference's default batch of 256 is 74 K),
        #              'philox' above (throughput).
        self.dropout_engine = dropout_engine(config)

    def _load_pretrained(self, embs, linears, predict):
        """'NeuMF-pre' (NeuMFRecommender.py:97-116): tables and tower copied from config['GMF_model'] / config['MLP_model'];
        predict weight and bias as the reference leaves them -- :115 writes 0.5 * cat(w_gmf, w_mlp) into the weight and :116
        overwrites it with 0.5 * (b_gmf + b_mlp) broadcast over all 2F entries, while the bias keeps nn.Linear's own
        initial draw (mirrored: the quirk is what the reference trains from)."""
        g, m = self.GMF_model, self.MLP_model
        if g is None or m is None:
            raise ValueError("model_name='NeuMF-pre' needs config['GMF_model'] and config['MLP_model']")

        def cpu(t):
            return torch.as_tensor(t).detach().to('cpu', torch.float32)

        def tower_parts(model):
            """(per-layer (weight, bias) list, predict weight [1, k], predict bias [1]) of a B200 NeuMF or an nn.Module one."""
            if hasattr(model, 'tower'):
                flat, F, Ln = cpu(model.tower), model.factors, model.num_layers
                out, o = [], 0
                for i in range(Ln):
                    n_in = F * (2 ** (Ln - i))
                    w = flat[o:o + n_in * (n_in // 2)].view(n_in // 2, n_in); o += n_in * (n_in // 2)
                    b = flat[o:o + n_in // 2]; o += n_in // 2
                    out.append((w, b))
                pw = flat[o:-1].view(1, -1)
                return out, pw, flat[-1:]
            lins = [mod for mod in model.MLP_layers if isinstance(mod, torch.nn.Linear)]
            return [(cpu(l.weight), cpu(l.bias)) for l in lins], cpu(model.predict_layer.weight), cpu(model.predict_layer.bias)

        embs[0].weight.copy_(cpu(g.embed_user_GMF.weight)); embs[1].weight.copy_(cpu(g.embed_item_GMF.weight))
        embs[2].weight.copy_(cpu(m.embed_user_MLP.weight)); embs[3].weight.copy_(cpu(m.embed_item_MLP.weight))
        m_layers, m_pw, m_pb = tower_parts(m)
        _, g_pw, g_pb = tower_parts(g)
        for lin, (w, b) in zip(linears, m_layers):
            lin.weight.copy_(w); lin.bias.copy_(b)
        predict.weight.copy_(0.5 * torch.cat([g_pw, m_pw], dim=1))
        predict.weight.copy_((0.5 * (g_pb + m_pb)).expand_as(predict.weight))        # :116 (bias into weight)

    # ------------------------------------------------------------------ plumbing
    def _tabs(self):
        return (self.embed_user_GMF.weight, self.embed_item_GMF.weight, self.embed_user_MLP.weight,
                self.embed_item_MLP.weight)

    def state_dict(self):
        return {'embed_user_GMF.weight': self.embed_user_GMF.weight, 'embed_item_GMF.weight': self.embed_item_GMF.weight,
                'embed_user_MLP.weight': self.embed_user_MLP.weight, 'embed_item_MLP.weight': self.embed_item_MLP.weight,
                'tower': self.tower}

    def _ensure(self, rows):
        if self._hp is None:
            self._begin_fit(self._optimizer_name())
        rows = max(int(rows), self._rows)
        if self._ws is None:
            self._ws = ops.NeumfWorkspace(self.user_num, self.item_num, self.factors, self.num_layers, self._fit_opt, rows,
                                          self.device)
        elif self._ws.max_rows < rows:
            # growing the scratch would drop the optimiser state: size it up front instead
            raise RuntimeError('NeuMF scratch too small; set config["neumf_scratch_rows"] >= 2 * batch_size')

    def _begin_fit(self, opt):
        super()._begin_fit(opt)
        self._philox_seed = None                                     # drawn lazily: the host-mask engine must not move the RNG here

    def _host_masks(self, rows_per_step):
        """Parity dropout: the keep-masks nn.Dropout would draw for steps of rows_per_step[k] triples, drawn by torch on the CPU
        generator in the reference's order and bit-packed (layout: drb_neumf_mask_words) -> int32 CUDA tensor."""
        F, Ln, keep = self.factors, self.num_layers, 1.0 - self.dropout
        widths = [F * (2 ** (Ln - i)) for i in range(Ln)]
        words = []
        for B in rows_per_step:
            per_layer = [[None, None] for _ in range(Ln)]
            for side in (0, 1):                                           # forward(user, pos) draws first, then forward(user, neg)
                for l, n in enumerate(widths):
                    per_layer[l][side] = torch.empty(B, n, dtype=torch.float32).bernoulli_(keep).numpy() != 0
            for l in range(Ln):
                bits = np.packbits(np.concatenate(per_layer[l]).reshape(-1), bitorder='little')
                pad = (-len(bits)) % 4
                words.append(np.pad(bits, (0, pad)).view(np.int32))
        return torch.from_numpy(np.concatenate(words)).to(self.device)

    def _drop_seed(self):
        """Key of the counter-based (Philox) masks: drawn from torch's global RNG the first time a fit needs it, so that
        torch.manual_seed makes runs reproducible."""
        if self.dropout <= 0.0 or not self.training or self._mode == 1:
            return 0                                                      # 'GMF' never calls a Dropout module: no draw at all
        if getattr(self, '_philox_seed', None) is None:
            self._philox_seed = int(torch.empty((), dtype=torch.int64).random_().item())
        return self._philox_seed

    def _mask_bits(self, batch):
        """Dropout mask elements of one step: both forward calls over every tower layer."""
        return 2 * batch * (4 * self.mlp_dim - 2 * self.factors)

    def _use_host_masks(self, batch):
        if not self.training or self.dropout <= 0.0 or self._mode == 1:
            return False                                                  # 'GMF' never runs the tower: no Dropout is called
        if self.dropout_engine == 'auto':
            return self._mask_bits(batch) <= (1 << 22)
        return self.dropout_engine == 'torch'

    def _train_steps(self, bu, bi, bj, batch, first, n_steps):
        self._ensure(2 * batch)
        p = self.dropout if self.training else 0.0
        kw = dict(tower_dtype=self._tower_dtype, dropout=p, mode=self._mode)
        if self._use_host_masks(batch):
            out = []
            for s, k, rows in mask_segments(bu.numel(), batch, first, n_steps, self._mask_bits(batch) // 8):
                lo, s0 = (s * batch, 0) if rows < batch else (0, s)   # a ragged last step runs as a batch of its own
                out.append(ops.neumf_bpr_train_steps(self._tabs(), self.tower, self._ws, bu[lo:], bi[lo:], bj[lo:], rows, s0, k,
                                                     self._hp, adam_step0=self._opt_steps + (s - first),
                                                     drop_masks=self._host_masks([rows] * k), **kw))
            losses = torch.cat(out)
        else:
            losses = ops.neumf_bpr_train_steps(self._tabs(), self.tower, self._ws, bu, bi, bj, batch, first, n_steps, self._hp,
                                               adam_step0=self._opt_steps, dropout_seed=self._drop_seed(), **kw)
        self._opt_steps += n_steps
        return losses

    # ------------------------------------------------------------------ reference surface
    def calc_loss(self, batch):
        self._check_loss_type()
        bu, bi, bj = self._planes(batch[:3])
        self._ensure(2 * bu.numel())
        masks = self._host_masks([bu.numel()]) if self._use_host_masks(bu.numel()) else None
        loss = ops.neumf_bpr_train_steps(self._tabs(), self.tower, self._ws, bu, bi, bj, bu.numel(), 0, 1, self._hp,
                                         apply=False, tower_dtype=self._tower_dtype, adam_step0=self._opt_steps,
                                         dropout=self.dropout if self.training else 0.0,
                                         dropout_seed=0 if masks is not None else self._drop_seed(), drop_masks=masks,
                                         mode=self._mode)
        return loss.to(torch.float32).reshape(())

    def _scores(self, users, items, per_user):
        self._ensure(1)
        return ops.neumf_scores(self._tabs(), self.tower, self._ws, users, items, per_user, self._tower_dtype, self._mode)

    def _score_pairs(self, u, i):
        return self._scores(u.to(torch.int64), i.to(torch.int64).reshape(-1, 1), 1).reshape(-1)

    def _rank_rows(self, users, cands, k):
        return ops.topk_from_scores(self._scores(users, cands, cands.shape[1]), cands, k)

    def _full_rank_rows(self, users, k):
        return ops.topk_from_scores(self._scores(users, None, self.item_num), None, k)
