"""GPU suite for Item2Vec: the skip-gram sampler, the shared-table step, the user rows and the ranking, through the C ABI and
the classes, against the reference's outputs (tests/golden/item2vec.npz) and the C oracle (oracle/item2vec_oracle.c)."""
import hashlib
import logging
import tempfile

import numpy as np
import pandas as pd
import pytest
import torch

from conftest import golden, csr_from_coo

pytestmark = pytest.mark.gpu
OPTS = ("sgd", "adam", "adagrad", "rmsprop")


@pytest.fixture(scope="module")
def g():
    return golden("item2vec")


@pytest.fixture(scope="module")
def i2v():
    from oracle import item2vec_oracle
    item2vec_oracle.build()
    return item2vec_oracle


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cfg(U, I, train_ur, **kw):
    cfg = dict(UID_NAME="user", IID_NAME="item", user_num=U, item_num=I, train_ur=train_ur, context_window=2, rho=0.3,
               factors=16, lr=0.05, epochs=1, optimizer="default", init_method="default", early_stop=False, topk=10,
               gpu="0", logger=logging.getLogger("t"), progress=False)
    cfg.update(kw)
    return cfg


def _close(got, want, opt, lr):
    d = np.abs(got - want)
    if opt == "sgd":
        assert d.max() <= 3e-6, d.max()
    else:                       # DESIGN section 4: a gradient of pure rounding noise may become a step of up to lr
        assert (d > 3e-5).sum() <= 4 and d.max() <= 2 * lr + 1e-6, ((d > 3e-5).sum(), d.max())


def test_sampler_matches_reference(g):
    from daisyrec_b200.utils.sampler import SkipGramNegativeSampler
    from daisyrec_b200.utils.utils import get_ur
    from daisyrec_b200 import ops
    for k in range(int(g["n_sampler_cases"])):
        U, I, w, discard, seed = (int(x) for x in g[f"s{k}_meta"])
        df = pd.DataFrame({"user": g[f"s{k}_users"].astype(np.int64), "item": g[f"s{k}_items"].astype(np.int64)})
        ops.mt19937_to_numpy(g[f"s{k}_state0"])
        cfg = _cfg(U, I, get_ur(df), context_window=w)
        rows = SkipGramNegativeSampler(df, cfg, discard=bool(discard)).sampling()
        assert rows.dtype == np.int64 and np.array_equal(rows, g[f"s{k}_rows"]), k
        assert np.array_equal(ops.mt19937_from_numpy(), g[f"s{k}_state1"]), k
        assert np.array_equal(rows._drb_device.cpu().numpy(), rows.astype(np.int32))      # the int32 device twin


def test_sampler_empty_complement_and_empty_result():
    from daisyrec_b200.utils.sampler import SkipGramNegativeSampler
    df = pd.DataFrame({"user": [0, 0], "item": [0, 1]})
    with pytest.raises(ValueError, match="cannot be empty"):
        SkipGramNegativeSampler(df, _cfg(1, 2, {0: {0, 1}})).sampling()
    one = SkipGramNegativeSampler(df.iloc[:1], _cfg(1, 2, {0: {0, 1}})).sampling()
    assert one.shape == (0,) and one.dtype == np.float64
    with pytest.raises(KeyError):
        SkipGramNegativeSampler(df, {k: v for k, v in _cfg(1, 2, {0: {0}}).items() if k != "rho"})


def test_constructor_tables_match_reference(g):
    from daisyrec_b200.model.Item2VecRecommender import Item2Vec
    U, I, F, seed = (int(x) for x in g["step_meta"])
    torch.manual_seed(seed)
    model = Item2Vec(_cfg(U, I, {}, factors=F))
    assert model.loss_type == "CL" and model._optimizer_name() == "adam"
    assert np.array_equal(model.user_embedding.weight.cpu().numpy(), g["P0"])
    assert np.array_equal(model.shared_embedding.weight.cpu().numpy(), g["Q0"])
    with pytest.raises(NotImplementedError):
        Item2Vec(_cfg(U, I, {}, factors=F, deterministic=True))


def test_steps_match_reference_and_oracle(g, i2v):
    from daisyrec_b200 import ops
    lr = float(g["step_lr"])
    I, F = g["Q0"].shape
    for opt in OPTS:
        Q = _dev(g["Q0"].copy())
        Qo = g["Q0"].copy()
        state = {}
        ws = ops.Item2VecWorkspace(I, F, opt, "cuda")
        hp = ops.hyper(lr, 0.0, 0.0, opt, loss="CL")
        for s, b in enumerate(g["step_batches"]):
            b32 = b.astype(np.int32)
            l = ops.item2vec_train_steps(Q, ws, _dev(b32[:, 0]), _dev(b32[:, 1]), _dev(b32[:, 2]), len(b), 0, 1, hp,
                                         adam_step0=s).item()
            lo = i2v.item2vec_step(Qo, b, opt, lr, state, step_count=s + 1)
            ref = g[f"{opt}_losses"][s]
            assert abs(l - ref) <= 1e-5 * abs(ref) and abs(l - lo) <= 2e-6 * abs(lo), (opt, s, l, ref, lo)
            _close(Q.cpu().numpy(), g[f"{opt}_Q"][s], opt, lr)
            _close(Q.cpu().numpy(), Qo, opt, lr)


def test_apply0_and_target_equals_context_and_nan():
    from daisyrec_b200 import ops
    rng = np.random.default_rng(3)
    I, F, lr = 20, 16, 0.1
    Q0 = (rng.standard_normal((I, F)) * 0.3).astype(np.float32)
    Q = _dev(Q0.copy())
    ws = ops.Item2VecWorkspace(I, F, "sgd", "cuda")
    hp = ops.hyper(lr, 0.0, 0.0, "sgd", loss="CL")
    one = lambda *v: _dev(np.array(v, np.int32))
    l0 = ops.item2vec_train_steps(Q, ws, one(5, 2), one(5, 7), one(1, 0), 2, 0, 1, hp, apply=False).item()
    assert np.array_equal(Q.cpu().numpy(), Q0) and l0 > 0
    l = ops.item2vec_train_steps(Q, ws, one(5), one(5), one(1), 1, 0, 1, hp).item()
    x = float(np.dot(Q0[5].astype(np.float64), Q0[5]))
    d = 1 / (1 + np.exp(-x)) - 1.0
    assert abs(l - (np.log1p(np.exp(-x)))) <= 1e-5 * l
    want = Q0.copy()
    want[5] = Q0[5] - lr * (2 * d * Q0[5])                           # both contributions land on the one row
    np.testing.assert_allclose(Q.cpu().numpy(), want, rtol=0, atol=2e-6)
    Qn = _dev(np.full((I, F), np.nan, np.float32))
    with pytest.raises(ValueError, match="Nan"):
        ops.item2vec_train_steps(Qn, ws, one(1), one(2), one(1), 1, 0, 1, hp)


def test_model_user_rows_rank_and_predict(i2v, orc):
    from daisyrec_b200.model.Item2VecRecommender import Item2Vec
    from daisyrec_b200.utils.dataset import BasicDataset, get_dataloader
    from daisyrec_b200.utils.sampler import SkipGramNegativeSampler
    from daisyrec_b200.utils.utils import get_ur
    rng = np.random.default_rng(9)
    U, I = 40, 60
    df = pd.DataFrame({"user": rng.integers(0, U - 5, 400), "item": rng.integers(0, I, 400)})   # users U-5.. have no rows
    cfg = _cfg(U, I, get_ur(df), factors=32, epochs=2, optimizer="adam", lr=0.01)
    np.random.seed(1); torch.manual_seed(1)
    model = Item2Vec(cfg)
    P0 = model.user_embedding.weight.cpu().numpy().copy()
    rows = SkipGramNegativeSampler(df, cfg).sampling()
    model.fit(get_dataloader(BasicDataset(rows), batch_size=128, shuffle=True, num_workers=0))
    P = model.user_embedding.weight.cpu().numpy()
    Q = model.shared_embedding.weight.cpu().numpy()
    row_ptr, col = csr_from_coo(df["user"].values, df["item"].values, U)
    Po = i2v.user_embed(row_ptr, col, Q, P0.copy())
    np.testing.assert_allclose(P, Po, rtol=1e-6, atol=1e-7)
    assert np.array_equal(P[U - 5:], P0[U - 5:])                     # outside train_ur: initial rows, bit for bit
    users = np.arange(U, dtype=np.int64)
    cands = rng.integers(0, I, size=(U, 25)).astype(np.int64)
    from daisyrec_b200.utils.dataset import CandidatesDataset
    preds = model.rank(get_dataloader(CandidatesDataset([[int(u), cands[u]] for u in users]), batch_size=16, shuffle=False,
                                      num_workers=0))
    assert preds.dtype == np.float32 and np.array_equal(preds, orc.mf_rank(P, Q, users, cands, 10))
    full = model.full_rank(3)
    assert full.dtype == np.int64 and np.array_equal(full, orc.mf_full_rank(P, Q, np.array([3], np.int64), 10)[0])
    assert model.predict(3, 7) == float(orc.mf_predict(P, Q, np.array([3], np.int32), np.array([7], np.int32))[0])
    with pytest.raises(IndexError, match="target item"):
        model.fit(get_dataloader(BasicDataset(np.array([[I, 0, 1]] * 4, np.int64)), batch_size=2, shuffle=False,
                                 num_workers=0))


def test_ml100k_driver_sequence(g):
    """run_examples/test.py with algo_name=item2vec, 1 epoch at batch 256, against the reference's run."""
    from daisyrec_b200.model.Item2VecRecommender import Item2Vec
    from daisyrec_b200.utils.sampler import SkipGramNegativeSampler
    from daisyrec_b200.utils.dataset import BasicDataset, CandidatesDataset, get_dataloader
    from daisyrec_b200.utils.utils import get_ur, build_candidates_set
    from daisyrec_b200.utils.metrics import calc_ranking_results
    from daisyrec_b200 import ops
    U, I, F, B, seed, w, topk = (int(x) for x in g["ml_meta"])
    s = golden("ml100k_sampler")
    r = golden("ml100k_rank")
    coo = np.stack([s["coo_u"], s["coo_i"]]).astype(np.int64)
    assert hashlib.sha256(coo.tobytes()).digest() == bytes(g["ml_coo_sha256"])      # the same train split
    train = pd.DataFrame({"user": coo[0], "item": coo[1]})
    train_ur = get_ur(train)
    test_ur, k = {}, 0
    for u, n in zip(r["test_u"], r["gt_len"]):
        test_ur[int(u)] = set(int(x) for x in r["gt_flat"][k:k + n])
        k += n
    cfg = _cfg(U, I, train_ur, factors=F, lr=float(g["ml_lr"]), context_window=w, topk=topk, cand_num=1000,
               metrics=["recall", "mrr", "ndcg", "hit", "precision"], res_path=tempfile.mkdtemp() + "/")
    np.random.seed(seed); torch.manual_seed(seed)
    model = Item2Vec(cfg)
    rows = SkipGramNegativeSampler(train, cfg).sampling()
    assert rows.shape[0] == int(g["ml_T"]) and hashlib.sha256(rows.tobytes()).digest() == bytes(g["ml_sha256"])
    assert np.array_equal(ops.mt19937_from_numpy(), g["ml_state1"])
    losses = []
    orig = model._train_steps
    model._train_steps = lambda *a: losses.append(orig(*a)) or losses[-1]
    model.fit(get_dataloader(BasicDataset(rows), batch_size=B, shuffle=True, num_workers=0))
    loss = float(sum(float(t.sum()) for t in losses))
    ref = float(g["ml_epoch_loss"])
    assert abs(loss - ref) <= 1e-4 * abs(ref), (loss, ref)       # measured on a B200: 2.9e-8 relative
    test_u, test_ucands = build_candidates_set(test_ur, train_ur, cfg)
    preds = model.rank(get_dataloader(CandidatesDataset(test_ucands), batch_size=128, shuffle=False, num_workers=0))
    same = (preds.astype(np.int64) == g["ml_preds"].astype(np.int64)).mean()
    print(f"ml-100k item2vec: epoch loss {loss:.6f} (reference {ref:.6f}), rank positions equal {same:.4f}")
    assert same >= 0.95, same                                        # measured on a B200: 0.9999
    res = calc_ranking_results(test_ur, preds, test_u, cfg)
    kpi = res.values[:, 1:].astype(np.float64)
    assert np.abs(kpi - g["ml_kpi"]).max() <= 0.005, np.abs(kpi - g["ml_kpi"]).max()
