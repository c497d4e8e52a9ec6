"""CPU suite for Item2Vec: the C oracle (oracle/item2vec_oracle.c) and the library's host draws against the reference's
outputs in tests/golden/item2vec.npz (oracle/gen_item2vec.py).

Bars: sampler rows and numpy's MT19937 state bit-exact; constructor tables bit-identical; step losses 1e-5 relative; tables
after each step 3e-6 absolute for SGD and 3e-5 for the stateful optimisers (DESIGN section 4: Adam turns a gradient that is
pure rounding noise into a step of up to lr, so a few such entries may differ by up to 2 lr)."""
import hashlib

import numpy as np
import pytest

from conftest import golden, csr_from_coo

OPTS = ("sgd", "adam", "adagrad", "rmsprop")


@pytest.fixture(scope="module")
def g():
    return golden("item2vec")


@pytest.fixture(scope="module")
def i2v():
    from oracle import item2vec_oracle
    item2vec_oracle.build()
    return item2vec_oracle


def _case(g, k):
    U, I, w, discard, seed = (int(x) for x in g[f"s{k}_meta"])
    users, items = g[f"s{k}_users"], g[f"s{k}_items"]
    row_ptr, col = csr_from_coo(users, items, U)
    return U, I, w, bool(discard), users, items, row_ptr, col


def _discard(g, k, users, items, st):
    """The reference's discard step, on numpy's generator at state st (rho = 0.3 in the fixture)."""
    import pandas as pd
    from daisyrec_b200 import ops
    ops.mt19937_to_numpy(st)
    df = pd.DataFrame({"user": users, "item": items})
    prob = 1 - np.sqrt(0.3 / df["item"].value_counts())
    keep = np.random.uniform(low=0., high=1., size=len(df)) >= df["item"].map(prob).values
    return users[keep], items[keep], ops.mt19937_from_numpy()


def test_oracle_sampler_matches_reference(g, i2v):
    for k in range(int(g["n_sampler_cases"])):
        U, I, w, discard, users, items, row_ptr, col = _case(g, k)
        st = g[f"s{k}_state0"].copy()
        if discard:
            users, items, st = _discard(g, k, users, items, st)
        rows = i2v.sgns_sample(st, users, items, row_ptr, col, I, w)
        assert np.array_equal(rows, g[f"s{k}_rows"]), k
        assert np.array_equal(st, g[f"s{k}_state1"]), k


def test_oracle_sampler_empty_complement_raises(i2v):
    st = np.zeros(625, np.uint32)
    st[624] = 624
    row_ptr, col = np.array([0, 3], np.int64), np.arange(3, dtype=np.int32)
    with pytest.raises(ValueError, match="cannot be empty"):
        i2v.sgns_sample(st, np.zeros(2, np.int32), np.array([0, 1], np.int32), row_ptr, col, 3, 1)
    one = i2v.sgns_sample(st, np.zeros(1, np.int32), np.array([0], np.int32), row_ptr, col, 3, 1)
    assert one.shape == (0,) and one.dtype == np.float64           # no context, no draw: numpy's empty array


def test_library_host_draws_match_reference_words(g):
    """The library's bounded draws, one row per position, consume the words the reference's np.random.choice calls do."""
    from daisyrec_b200 import ops
    for k in range(int(g["n_sampler_cases"])):
        U, I, w, discard, users, items, row_ptr, col = _case(g, k)
        st = g[f"s{k}_state0"].copy()
        if discard:
            users, items, st = _discard(g, k, users, items, st)
        order = np.argsort(users, kind="stable")
        su = users[order]
        start = np.searchsorted(su, su, "left")
        end = np.searchsorted(su, su, "right")
        i = np.arange(len(su)) - start
        L = end - start
        count = np.minimum(i + w, L - 1) - np.maximum(i - w, 0)
        off = np.concatenate([[0], np.cumsum(count)]).astype(np.int64)
        bound = I - (row_ptr[su + 1] - row_ptr[su])
        draws = ops.bounded_draws_mt19937(st, bound, off)
        assert np.array_equal(st, g[f"s{k}_state1"]), k
        rows = g[f"s{k}_rows"]
        assert len(draws) * 2 == len(rows)
        neg = rows[rows[:, 2] == 0]
        for p in range(len(su)):                                    # k-th complement of each draw == the stored negative
            cands = np.setdiff1d(np.arange(I), col[row_ptr[su[p]]:row_ptr[su[p] + 1]])
            assert np.array_equal(cands[draws[off[p]:off[p + 1]]], neg[off[p]:off[p + 1], 1]), (k, p)


def test_ml100k_sampler_digest_is_consistent(g):
    rows_head, rows_tail = g["ml_head"], g["ml_tail"]
    assert int(g["ml_T"]) % 2 == 0 and rows_head.shape == (64, 3) and rows_tail.shape == (64, 3)
    assert len(bytes(g["ml_sha256"])) == len(hashlib.sha256().digest())


def test_oracle_steps_match_reference(g, i2v):
    lr = float(g["step_lr"])
    for opt in OPTS:
        Q = g["Q0"].copy()
        state = {}
        for s, b in enumerate(g["step_batches"]):
            loss = i2v.item2vec_step(Q, b, opt, lr, state, step_count=s + 1)
            assert abs(loss - g[f"{opt}_losses"][s]) <= 1e-5 * abs(g[f"{opt}_losses"][s]), (opt, s)
            want = g[f"{opt}_Q"][s]
            d = np.abs(Q - want)
            if opt == "sgd":
                assert d.max() <= 3e-6, (opt, s, d.max())
            else:
                bad = d > 3e-5
                assert bad.sum() <= 4 and d.max() <= 2 * lr + 1e-6, (opt, s, bad.sum(), d.max())


def test_oracle_user_embed(g, i2v):
    P = g["P0"].copy()
    Q = g["sgd_Q"][-1]
    row_ptr = np.array([0, 2, 2, 5] + [5] * (P.shape[0] - 3), np.int64)
    col = np.array([1, 7, 0, 3, 29], np.int32)
    i2v.user_embed(row_ptr, col, Q, P)
    assert np.allclose(P[0], Q[1] + Q[7], rtol=1e-6, atol=0)
    assert np.allclose(P[2], Q[0] + Q[3] + Q[29], rtol=1e-6, atol=1e-7)
    assert np.array_equal(P[1], g["P0"][1]) and np.array_equal(P[3:], g["P0"][3:])


def test_constructor_init_stream_matches_reference(g):
    """Item2Vec's tables come from two nn.Embedding draws (user, then shared) and _init_weight on each, in that order."""
    import torch
    from daisyrec_b200.model.AbstractRecommender import _init_table, _INIT
    U, I, F, seed = (int(x) for x in g["step_meta"])
    torch.manual_seed(seed)
    wu, wi = _init_table(U, F, None), _init_table(I, F, None)
    _INIT["normal"](wu)
    _INIT["normal"](wi)
    assert np.array_equal(wu.numpy(), g["P0"]) and np.array_equal(wi.numpy(), g["Q0"])
