"""Negative sampler with the reference's class name and config keys
(daisy/utils/sampler.py:3-103), computed on the device through the C ABI.

Reference semantics kept bit for bit: per USER, ``num_ng`` draws (with replacement) using numpy's
global legacy RandomState -- uniform over the sorted complement of the user's train positives
(:84-89), or, for ``sample_method`` 'low-pop' / 'high-pop', ``num_ng - int(sample_ratio*num_ng)``
such draws followed by popularity-weighted draws over all items (:43-53, :64-81); every positive
row is then paired with its user's negatives (``explode``): [T,3] triples for BPR / HL / TL
(:99-101), or positives-then-negatives labelled rows for CL / SL (:93-98).  The global numpy RNG is
advanced exactly as the reference would advance it.
"""
import numpy as np
import torch

from .. import ops


def fingerprint(a):
    """Cheap content stamp of a host index array: shape, an int64 sum over <= 65 536 evenly strided elements and the two
    end rows.  It lets fit() notice that a host array whose device copy is cached was edited in place (shuffled, filtered,
    relabelled) and re-upload it; a stamp, not a checksum."""
    flat = np.asarray(a).reshape(-1)
    step = max(1, flat.size // 65536)
    while step > 1 and step % 3 == 0:        # [T,3] rows: a stride that is a multiple of 3 would only ever see one column
        step += 1
    return (tuple(a.shape), int(flat[::step].sum(dtype=np.int64)), flat[:3].tobytes(), flat[-3:].tobytes())


class TripleArray(np.ndarray):
    """int32 [T,3] host array that remembers its device twin (saves fit() a 12*T-byte H2D).  Views / copies forget
    the twin; an in-place edit is caught by the stamp taken when the twin was attached."""
    _drb_device = None
    _drb_stamp = None

    def __array_finalize__(self, obj):
        self._drb_device = None
        self._drb_stamp = None

    @staticmethod
    def attach(host, device_tensor):
        out = host.view(TripleArray)
        out._drb_device = device_tensor
        out._drb_stamp = fingerprint(out)
        return out


def csr_from_ur(ur, user_num):
    """config['train_ur'] (dict[int -> set[int]], daisy/utils/utils.py:19-34) -> sorted CSR."""
    lens = np.fromiter((len(ur[u]) if u in ur else 0 for u in range(user_num)), np.int64, user_num)
    row_ptr = np.zeros(user_num + 1, np.int64)
    np.cumsum(lens, out=row_ptr[1:])
    total = int(row_ptr[-1])
    col = np.fromiter((i for u in range(user_num) if u in ur for i in ur[u]), np.int64, total)
    key = np.repeat(np.arange(user_num, dtype=np.int64), lens) * (1 << 32) + col
    key.sort()
    return row_ptr, (key & 0xFFFFFFFF).astype(np.int32)


class AbstractSampler(object):
    def __init__(self, config):
        self.uid_name = config['UID_NAME']
        self.iid_name = config['IID_NAME']
        self.item_num = config['item_num']
        self.ur = config['train_ur']

    def sampling(self):
        raise NotImplementedError


class BasicNegtiveSampler(AbstractSampler):
    def __init__(self, df, config):
        super().__init__(config)
        self.user_num = config['user_num']
        self.num_ng = config['num_ng']
        self.inter_name = config['INTER_NAME']
        self.sample_method = config['sample_method']
        self.sample_ratio = config['sample_ratio']
        self.loss_type = config['loss_type'].upper()
        # optional B200 keys (absent == reference behaviour)
        self.rng_engine = config.get('sampler_rng', 'numpy')       # 'numpy' (MT19937 replay) | 'philox'
        self.csr = config.get('train_csr', None)                   # (row_ptr int64, col int32) to skip the dict walk

        assert self.sample_method in ['uniform', 'low-pop', 'high-pop'], f'Invalid sampling method: {self.sample_method}'
        assert 0 <= self.sample_ratio <= 1, 'Invalid sample ratio value'
        self.df = df
        self.pop_prob = None
        if self.sample_method in ['high-pop', 'low-pop']:          # sampler.py:43-53
            cnt = np.bincount(np.asarray(df[self.iid_name].values, dtype=np.int64), minlength=self.item_num)
            seen = cnt > 0
            pop = cnt[seen] / cnt.sum()                            # groupby(item).size() rescaled to [0, 1]
            if self.sample_method == 'high-pop':
                norm_pop = np.zeros(self.item_num)
                norm_pop[seen] = pop
            else:
                norm_pop = np.ones(self.item_num)
                norm_pop[seen] = 1 - pop
            self.pop_prob = norm_pop / norm_pop.sum()

    def _pointwise(self, d_coo_u, d_coo_i, d_js):
        """CL / SL rows (sampler.py:58-59, :93-98): positives (u, i, rating) then negatives (u, j, 0), int32."""
        label = np.array(self.df[self.inter_name].values).astype(np.int32)
        d_rows = ops.sampler_explode_pointwise(d_coo_u, d_coo_i, torch.from_numpy(label).cuda(), d_js)
        return TripleArray.attach(d_rows.cpu().numpy(), d_rows)

    def sampling(self):
        if self.loss_type not in ('BPR', 'HL', 'TL', 'CL', 'SL'):
            raise NotImplementedError
        coo_u = np.array(self.df[self.uid_name].values, dtype=np.int32)        # a writable copy: pandas >= 3
        coo_i = np.array(self.df[self.iid_name].values, dtype=np.int32)        # hands out read-only views
        if self.num_ng == 0:
            if self.loss_type in ('CL', 'SL'):
                ops.require_cuda()
                d_js = torch.zeros((self.user_num, 0), dtype=torch.int32, device='cuda')
                return self._pointwise(torch.from_numpy(coo_u).cuda(), torch.from_numpy(coo_i).cuda(), d_js)
            raise NotImplementedError('loss function (BPR, TL, HL) need num_ng > 0')
        ops.require_cuda()
        U, I, G = self.user_num, self.item_num, self.num_ng
        row_ptr, col = self.csr if self.csr is not None else csr_from_ur(self.ur, U)
        d_row_ptr = torch.from_numpy(np.ascontiguousarray(row_ptr, np.int64)).cuda()
        d_col = torch.from_numpy(np.ascontiguousarray(col, np.int32)).cuda()
        if self.pop_prob is not None:
            if self.rng_engine != 'numpy':
                raise NotImplementedError("sampler_rng='philox' covers the uniform branch only")
            other_num = int(self.sample_ratio * G)                 # sampler.py:65-66
            state = ops.mt19937_from_numpy()
            draws, u01 = ops.sampler_draw_mt19937_mixed(state, row_ptr, U, I, G - other_num, other_num)
            ops.mt19937_to_numpy(state)
            cdf = self.pop_prob.cumsum()                           # RandomState.choice(p=...) ahead of searchsorted
            cdf /= cdf[-1]
            d_js = ops.sampler_assemble_mixed(d_row_ptr, d_col, torch.from_numpy(draws).cuda(),
                                              torch.from_numpy(cdf).cuda(), torch.from_numpy(u01).cuda(), I)
            d_draws = None
        elif self.rng_engine == 'numpy':
            state = ops.mt19937_from_numpy()
            draws = ops.sampler_draw_mt19937(state, row_ptr, U, I, G)         # host: sequential MT19937 words
            ops.mt19937_to_numpy(state)                                       # numpy's stream moves on as in the reference
            d_draws = torch.from_numpy(draws).cuda()
        else:
            seed = int(np.random.randint(0, 2 ** 31 - 1))
            d_draws, bad = ops.sampler_draw_philox(seed, 0, d_row_ptr, U, I, G)
            if int(bad.item()) < U:
                raise ValueError("'a' cannot be empty unless no samples are taken")
        if d_draws is not None:
            d_js = ops.sampler_kth_complement(d_row_ptr, d_col, d_draws, I)
        self.js = d_js
        if self.loss_type in ('CL', 'SL'):
            return self._pointwise(torch.from_numpy(coo_u).cuda(), torch.from_numpy(coo_i).cuda(), d_js)
        d_tr = ops.sampler_explode(torch.from_numpy(coo_u).cuda(), torch.from_numpy(coo_i).cuda(), d_js)
        return TripleArray.attach(d_tr.cpu().numpy(), d_tr)


class SkipGramNegativeSampler(AbstractSampler):
    """Skip-gram rows <target, context, label> for Item2Vec (daisy/utils/sampler.py:105-160), built on the device.

    Every df row is a position of its user's sequence (users ascending, df row order inside a user, duplicates kept).  A
    position contributes its window's context items as positives [target, context, 1] in ascending position, then as many
    negatives [target, item, 0] drawn uniformly with replacement from the items outside config['train_ur'][user] -- the same
    numpy MT19937 words np.random.choice would consume, so numpy's global state moves on exactly as in the reference.
    ``sampling()`` returns the int64 [T, 3] host array with its int32 device twin attached (fit() does not upload it again).
    """

    def __init__(self, df, config, discard=False):
        super().__init__(config)
        self.context_window = int(config['context_window'])
        self.csr = config.get('train_csr', None)                   # (row_ptr int64, col int32) to skip the dict walk
        freq = df[self.iid_name].value_counts()
        prob_discard = 1 - np.sqrt(config['rho'] / freq)           # computed (and 'rho' required) with or without discard
        if discard:                                                # one uniform per df row, before any negative is drawn
            rnd_p = np.random.uniform(low=0., high=1., size=len(df))
            df = df[rnd_p >= df[self.iid_name].map(prob_discard).values]
        self.users = np.array(df[self.uid_name].values, dtype=np.int32)
        self.items = np.array(df[self.iid_name].values, dtype=np.int32)

    def sampling(self):
        ops.require_cuda()
        n, I, w = len(self.users), self.item_num, self.context_window
        if self.csr is not None:
            row_ptr, col = self.csr
        else:
            row_ptr, col = csr_from_ur(self.ur, int(self.users.max()) + 1 if n else 0)
        col = np.ascontiguousarray(col, np.int32)
        d_row_ptr = torch.from_numpy(np.ascontiguousarray(row_ptr, np.int64)).cuda()
        d_col = torch.from_numpy(col if len(col) else np.zeros(1, np.int32)).cuda()
        d_su, order = torch.sort(torch.from_numpy(self.users).cuda(), stable=True)     # groupby(uid): stable, users ascending
        d_si = torch.from_numpy(self.items).cuda()[order].contiguous()
        count, bound = ops.sgns_positions(d_su, d_row_ptr, I, w)
        d_off = torch.zeros(n + 1, dtype=torch.int64, device=d_su.device)
        torch.cumsum(count, 0, out=d_off[1:])
        state = ops.mt19937_from_numpy()
        try:                                                       # host: one np.random.choice(cands, size=c) per position
            draws = ops.bounded_draws_mt19937(state, bound.cpu().numpy(), d_off.cpu().numpy())
        finally:
            ops.mt19937_to_numpy(state)                            # numpy's stream moves on as in the reference
        d_draws = torch.from_numpy(draws if len(draws) else np.zeros(1, np.int32)).cuda()
        d_rows = ops.sgns_explode(d_su, d_si, w, d_off, d_row_ptr, d_col, d_draws)
        if d_rows.shape[0] == 0:
            return np.array([])                                    # np.array of no rows: float64 (0,)
        return TripleArray.attach(d_rows.cpu().numpy().astype(np.int64), d_rows)
