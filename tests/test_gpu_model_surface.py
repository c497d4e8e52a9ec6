"""The public surface every recommender shares, on tiny models of all eight classes: rank on either loader form, the
IndexError of nn.Embedding for an out-of-range id at every entry point (raised before any kernel indexes a table with it),
and the state_dict / load_state_dict / to() plumbing."""
import logging

import numpy as np
import pytest
import scipy.sparse as sp
import torch
from torch.utils.data import DataLoader

from daisyrec_b200.utils.dataset import CandidatesDataset, get_dataloader

pytestmark = pytest.mark.gpu

U, I, TOPK = 20, 30, 5
MODELS = ["MF", "FM", "LightGCN", "NGCF", "NFM", "NeuMF", "Item2Vec", "VAECF"]


@pytest.fixture(params=MODELS)
def model(request):
    import daisyrec_b200.model as M
    rs = np.random.RandomState(0)
    cu = np.repeat(np.arange(U), 3)
    ci = rs.randint(0, I, len(cu))
    cfg = dict(gpu="", logger=logging.getLogger("t"), epochs=1, lr=0.01, reg_1=0.001, reg_2=0.001, user_num=U, item_num=I,
               factors=8, loss_type="BPR", optimizer="adam", init_method="default", early_stop=False, topk=TOPK, progress=False)
    name = request.param
    if name in ("LightGCN", "NGCF"):
        cfg.update(inter_matrix=sp.coo_matrix((np.ones(len(cu)), (cu, ci)), shape=(U, I)), num_layers=2, hidden_size_list=[8, 8],
                   node_dropout=0.0, mess_dropout=0.0)
    elif name == "NFM":
        cfg.update(num_layers=1, batch_norm=True, act_function="relu", dropout=0.0)
    elif name == "NeuMF":
        cfg.update(num_layers=2, dropout=0.0, model_name="NeuMF")
    elif name == "Item2Vec":
        cfg.update(train_ur={u: set(ci[cu == u].tolist()) for u in range(U)})
    elif name == "VAECF":
        cfg.update(history_item_id=torch.from_numpy(ci.reshape(U, 3)), history_item_value=torch.ones(U, 3), mlp_hidden_size=[16],
                   latent_dim=8, dropout=0.0, total_anneal_steps=100, anneal_cap=0.2)
    torch.manual_seed(0)
    return getattr(M, name)(cfg)


def _name(m):
    return type(m).__name__


def _batch(m, n=16):
    rs = np.random.RandomState(1)
    if _name(m) == "VAECF":
        return rs.randint(0, U, n)
    if _name(m) == "Item2Vec":
        return [rs.randint(0, I, n), rs.randint(0, I, n), rs.randint(0, 2, n)]        # (target, context, label)
    return [rs.randint(0, U, n), rs.randint(0, I, n), rs.randint(0, I, n)]            # (user, pos, neg)


def _bad_batches(m):
    """The batch with one id out of range, for every id column and both ends."""
    if _name(m) == "VAECF":
        out = []
        for v in (U, -U - 1):
            b = _batch(m)
            b[5] = v
            out.append(b)
        return out
    bounds = (I, I) if _name(m) == "Item2Vec" else (U, I, I)
    out = []
    for c, hi in enumerate(bounds):
        for v in (hi, -1):
            b = [x.copy() for x in _batch(m)]
            b[c][5] = v
            out.append(b)
    return out


def _rows(n=9, C=7):
    rs = np.random.RandomState(2)
    return [[int(u), rs.randint(0, I, C)] for u in rs.randint(0, U, n)]


def _loader(rows):
    return get_dataloader(CandidatesDataset(rows), batch_size=4, shuffle=False)


def test_rank_on_list_and_iterable_loaders(model):
    rows = _rows()
    a = model.rank(_loader(rows))
    b = model.rank(list(DataLoader(CandidatesDataset(rows), batch_size=4, shuffle=False)))
    assert a.shape == (len(rows), TOPK) and a.dtype == np.float32
    assert np.array_equal(a, b)
    assert model.rank(_loader([])).shape == (0,)
    assert model.rank([]).shape == (0,)


def test_out_of_range_ids_raise_index_error(model):
    rows = _rows()
    for r in ([[U, rows[0][1]]] + rows[1:], [[-U - 1, rows[0][1]]] + rows[1:],
              rows[:1] + [[rows[1][0], np.r_[rows[1][1][:-1], I]]] + rows[2:],
              rows[:1] + [[rows[1][0], np.r_[rows[1][1][:-1], -1]]] + rows[2:]):
        with pytest.raises(IndexError):
            model.rank(_loader(r))
    for u in (U, -U - 1):
        with pytest.raises(IndexError):
            model.full_rank(u)
    for u, i in ((U, 0), (-U - 1, 0), (0, I), (0, -1)):
        with pytest.raises(IndexError):
            model.predict(u, i)
    for bad in _bad_batches(model):
        with pytest.raises(IndexError):
            model.calc_loss(bad)
        with pytest.raises(IndexError):
            model.train_step(bad)
    if _name(model) in ("MF", "FM", "NFM", "NeuMF", "Item2Vec"):
        first = I if _name(model) == "Item2Vec" else U
        with pytest.raises(IndexError):
            model.forward([0, first], [0, 0])
        with pytest.raises(IndexError):
            model.forward([0, 0], [0, I])
    # the model still answers in-range calls
    assert model.full_rank(U - 1).shape == (TOPK,)
    assert np.isfinite(model.predict(U - 1, I - 1))
    assert np.isfinite(float(model.calc_loss(_batch(model))))


def test_refused_train_step_leaves_tables_unchanged(model):
    model.train_step(_batch(model))                                  # optimiser state and scratch exist from here on
    before = {k: v.clone() for k, v in model.state_dict().items()}
    for bad in _bad_batches(model):
        with pytest.raises(IndexError):
            model.train_step(bad)
    torch.cuda.synchronize()
    for k, v in model.state_dict().items():
        assert torch.equal(v, before[k]), k


def test_state_dict_round_trip_and_to(model):
    assert model.to("cuda") is model
    loader = _loader(_rows())
    preds = model.rank(loader)
    saved = {k: v.clone() for k, v in model.state_dict().items()}
    model.train_step(_batch(model))
    assert any(not torch.equal(v, saved[k]) for k, v in model.state_dict().items())
    model.load_state_dict(saved)
    for k, v in model.state_dict().items():
        assert torch.equal(v, saved[k]), k
    assert np.array_equal(model.rank(loader), preds)                 # nothing computed from the trained tables survives
    params = {p.data_ptr() for p in model.parameters()}
    assert params and params <= {t.data_ptr() for t in model.state_dict().values()}
