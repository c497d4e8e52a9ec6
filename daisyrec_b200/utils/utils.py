"""Boundary producers around the hot path, with the reference's function names
(daisy/utils/utils.py:19-34,53-85,125-144).

``build_candidates_set`` reproduces the reference's candidate lists bit for bit (same global
numpy RNG stream, ground-truth ids appended in ``list(set)`` order) but finds the k-th
un-interacted item with a device binary search instead of ``np.setdiff1d(arange(item_num), ...)``
per user.
"""
from collections import defaultdict

import numpy as np
import torch

from .. import ops


def get_ur(df):
    """daisy/utils/utils.py:19-34: dict[user -> set(items)] (vectorised instead of iterrows)."""
    ur = defaultdict(set)
    users = np.asarray(df['user'].values, dtype=np.int64)
    items = np.asarray(df['item'].values, dtype=np.int64)
    if len(users) == 0:
        return ur
    order = np.argsort(users, kind='stable')
    us, its = users[order], items[order]
    cuts = np.flatnonzero(np.diff(us)) + 1
    starts = np.concatenate([[0], cuts])
    groups = {int(us[s]): its[s:e] for s, e in zip(starts, np.concatenate([cuts, [len(us)]]))}
    # dict insertion order of the reference = first appearance of each user in df; the items of a user are added in df
    # order (stable sort), so each set goes through the same insertions as the reference's `ur[u].add(i)` loop
    uniq, first_idx = np.unique(users, return_index=True)
    for u in uniq[np.argsort(first_idx, kind='stable')].tolist():
        ur[u] = set(groups[u].tolist())
    return ur


def get_inter_matrix(df, config, form='coo'):
    """daisy/utils/utils.py:125-144: the whole sparse interaction matrix (scipy), what LightGCN's config['inter_matrix']
    holds (run_examples/test.py:89)."""
    import scipy.sparse as sp
    src, tar = df[config['UID_NAME']].values, df[config['IID_NAME']].values
    data = df[config['INTER_NAME']].values
    mat = sp.coo_matrix((data, (src, tar)), shape=(config['user_num'], config['item_num']))
    if form == 'coo':
        return mat
    elif form == 'csr':
        return mat.tocsr()
    raise NotImplementedError(f'Sparse matrix format [{form}] has not been implemented...')


def build_train_csr(df, config):
    """Sorted, duplicate-free user->item CSR of the train set, built on the device from the two DataFrame columns
    (drb_csr_build): the same object as ``csr_from_ur(get_ur(df))`` without the dict-of-sets walk.  Hand it to the
    sampler / MF as ``config['train_csr']``.  -> (row_ptr int64[user_num+1], col int32) numpy arrays."""
    ops.require_cuda()
    d_u = torch.from_numpy(np.array(df[config['UID_NAME']].values, dtype=np.int32)).cuda()
    d_i = torch.from_numpy(np.array(df[config['IID_NAME']].values, dtype=np.int32)).cuda()
    row_ptr, col = ops.csr_build(d_u, d_i, config['user_num'], config['item_num'])
    return row_ptr.cpu().numpy(), col.cpu().numpy()


def build_candidates_set(test_ur, train_ur, config, drop_past_inter=True):
    """daisy/utils/utils.py:53-85 -> (test_u, test_ucands) with test_ucands[k] = [u, int64[cand_num]]."""
    ops.require_cuda()
    item_num = config['item_num']
    candidates_num = config['cand_num']

    test_u, gts, excl, n_pop, n_draw, from_gt = [], [], [], [], [], []
    for u, r in test_ur.items():
        gt = list(r)                                            # set iteration order, as the reference
        sample_num = candidates_num - len(r) if len(r) <= candidates_num else 0
        test_u.append(u)
        gts.append(np.asarray(gt, dtype=np.int64))
        from_gt.append(sample_num == 0)
        if sample_num == 0:                                     # np.random.choice(list(r), candidates_num)
            excl.append(np.zeros(0, np.int32))
            n_pop.append(len(gt))
            n_draw.append(candidates_num)
        else:
            pos = gt + list(train_ur[u]) if drop_past_inter else gt
            ex = np.unique(np.asarray(pos, dtype=np.int64))
            ex = ex[(ex >= 0) & (ex < item_num)].astype(np.int32)
            excl.append(ex)
            n_pop.append(item_num - len(ex))
            n_draw.append(sample_num)
    m = len(test_u)
    if m == 0:
        return test_u, []
    offsets = np.zeros(m + 1, np.int64)
    np.cumsum(n_draw, out=offsets[1:])
    row_ptr = np.zeros(m + 1, np.int64)
    np.cumsum([len(e) for e in excl], out=row_ptr[1:])
    col = np.concatenate(excl) if row_ptr[-1] else np.zeros(1, np.int32)

    state = ops.mt19937_from_numpy()
    draws = ops.bounded_draws_mt19937(state, np.asarray(n_pop, np.int64), offsets)   # numpy's stream, in user order
    ops.mt19937_to_numpy(state)
    picked = ops.kth_complement_var(torch.from_numpy(row_ptr).cuda(), torch.from_numpy(col).cuda(),
                                    torch.from_numpy(offsets).cuda(), torch.from_numpy(draws).cuda()).cpu().numpy()

    test_ucands = []
    for k, u in enumerate(test_u):
        lo, hi = offsets[k], offsets[k + 1]
        if from_gt[k]:
            samples = gts[k][draws[lo:hi]]                      # choice from the ground truth itself
        else:
            samples = np.concatenate((picked[lo:hi].astype(np.int64), gts[k]), axis=None)
        test_ucands.append([u, samples])
    return test_u, test_ucands


def get_history_matrix(df, config, row='user', use_config_value_name=False):
    """daisy/utils/utils.py:87-123, vectorised: (history_matrix int64 [row_num, max_len], history_value float32 [row_num,
    max_len], history_len int64 [row_num]).  A row's entries keep their df order and are padded with (0, 0.0)."""
    logger = config['logger']
    assert row in df.columns, f'invalid name {row}: not in columns of history dataframe'
    uid_name, iid_name = config['UID_NAME'], config['IID_NAME']
    user_ids, item_ids = df[uid_name].values, df[iid_name].values
    value_name = config['INTER_NAME'] if use_config_value_name else None
    user_num, item_num = config['user_num'], config['item_num']
    values = np.ones(len(df)) if value_name is None else df[value_name].values
    if row == 'user':
        row_num, max_col_num = user_num, item_num
        row_ids, col_ids = user_ids, item_ids
    else:
        row_num, max_col_num = item_num, user_num
        row_ids, col_ids = item_ids, user_ids
    row_ids = np.asarray(row_ids, dtype=np.int64)
    history_len = np.bincount(row_ids, minlength=row_num).astype(np.int64) if len(row_ids) else np.zeros(row_num, np.int64)
    if len(history_len) > row_num:
        raise IndexError(f'index {len(history_len) - 1} is out of bounds for axis 0 with size {row_num}')
    col_num = np.max(history_len)
    if col_num > max_col_num * 0.2:
        logger.info(f'Max value of {row}\'s history interaction records has reached: {col_num / max_col_num * 100:.4f}% of the total.')
    order = np.argsort(row_ids, kind='stable')
    starts = np.zeros(row_num + 1, np.int64)
    np.cumsum(history_len, out=starts[1:])
    pos = np.empty(len(row_ids), np.int64)
    pos[order] = np.arange(len(row_ids), dtype=np.int64) - starts[row_ids[order]]      # rank of each entry inside its row
    history_matrix = np.zeros((row_num, col_num), dtype=np.int64)
    history_value = np.zeros((row_num, col_num))
    history_matrix[row_ids, pos] = np.asarray(col_ids, dtype=np.int64)
    history_value[row_ids, pos] = values
    return torch.LongTensor(history_matrix), torch.FloatTensor(history_value), torch.LongTensor(history_len)
