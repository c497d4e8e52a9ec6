"""CPU checks for Multi-VAE: the vectorised get_history_matrix and the fp64 oracle (oracle/vae_oracle.py) against the
reference's own runs (tests/golden/vae.npz, written by oracle/gen_vae.py)."""
import hashlib
import logging

import numpy as np
import pandas as pd
import pytest
import torch

from conftest import golden
from oracle import vae_oracle as vo


@pytest.fixture(scope="module")
def g():
    return golden("vae")


def _cfg(U, I):
    return dict(UID_NAME="user", IID_NAME="item", INTER_NAME="rating", user_num=U, item_num=I, logger=logging.getLogger("t"))


def case(g, c):
    nh, lat, opt = (int(x) for x in g["case_meta"][c])
    return [int(h) for h in g["case_hidden"][c][:nh]], lat, ("sgd", "adam")[opt], float(g["case_dropout"][c])


def replay(state, B, I, lat, p):
    """The masks and noise the reference drew in one step, from the generator state before it."""
    torch.set_rng_state(torch.from_numpy(state))
    mask = torch.empty(B, I, dtype=torch.float32).bernoulli_(1 - p).numpy().astype(np.float64) if p > 0 else None
    eps = torch.randn(B, lat // 2, dtype=torch.float32).numpy().astype(np.float64)
    return mask, eps


def test_history_matrix_matches_reference(g, caplog):
    from daisyrec_b200.utils.utils import get_history_matrix
    U, I = int(g["small_meta"][0]), int(g["small_meta"][1])
    df = pd.DataFrame({"user": g["df_user"], "item": g["df_item"]})
    hid, hval, hlen = get_history_matrix(df, _cfg(U, I), row="user")
    assert hid.dtype == torch.int64 and hval.dtype == torch.float32 and hlen.dtype == torch.int64
    assert np.array_equal(hid.numpy(), g["hist_id"]) and np.array_equal(hval.numpy(), g["hist_val"])
    assert np.array_equal(hlen.numpy(), g["hist_len"])
    with caplog.at_level(logging.INFO, logger="t"):
        get_history_matrix(df, _cfg(U, I), row="user")
    assert any("history interaction records has reached" in r.message for r in caplog.records)   # 20 of 40 items > 20 %


def test_ml100k_history_matrix_matches_reference(g):
    from daisyrec_b200.utils.utils import get_history_matrix
    s = golden("ml100k_sampler")
    U, I = int(g["ml_meta"][0]), int(g["ml_meta"][1])
    df = pd.DataFrame({"user": s["coo_u"].astype(np.int64), "item": s["coo_i"].astype(np.int64)})
    got = get_history_matrix(df, _cfg(U, I), row="user")
    for k, t in enumerate(got):
        assert hashlib.sha256(np.ascontiguousarray(t.numpy()).tobytes()).digest() == bytes(g["ml_hist_sha"][k]), k


def test_rating_matrix_last_write_wins(g):
    I = int(g["small_meta"][1])
    R = vo.rating_matrix(g["hist_id"], g["hist_val"], I)
    assert np.array_equal(R, g["R"])
    short = g["hist_len"] < g["hist_len"].max()
    assert (R[short, 0] == 0).all()                                    # the padding erased item 0 from every shorter row
    assert R[~short, 0].any() and (R <= 1).all()                       # the duplicate row is written once, not summed


@pytest.mark.parametrize("c", range(5))
def test_oracle_steps_match_reference(g, c):
    hidden, lat, opt, p = case(g, c)
    U, I, total, _ = (int(x) for x in g["small_meta"])
    R = vo.rating_matrix(g["hist_id"], g["hist_val"], I)
    net = g[f"c{c}_N0"].astype(np.float64)
    state = {}
    for s, b in enumerate(g["batches"]):
        mask, eps = replay(g[f"c{c}_rng"][s], len(b), I, lat, p)
        loss, grad = vo.loss_grad(net, R[b], I, hidden, lat, p, mask, eps, vo.anneal(s + 1, 0.2, total))
        net = vo.step(net, grad, opt, 0.01, state, s + 1)
        ref = g[f"c{c}_losses"][s]
        assert abs(loss - ref) <= 2e-6 * abs(ref), (s, loss, ref)
        d = np.abs(net - g[f"c{c}_N"][s])
        if opt == "sgd":
            assert d.max() <= 1e-6, (s, d.max())
        else:                   # a gradient of pure rounding noise may become an Adam step of up to lr (DESIGN section 4)
            assert (d > 1e-5).sum() <= 4 and d.max() <= 2 * 0.01 + 1e-6, (s, (d > 1e-5).sum(), d.max())
    loss, _ = vo.loss_grad(g[f"c{c}_N"][-1], R[g["batches"][0]], I, hidden, lat, ann=vo.anneal(4, 0.2, total), training=False,
                           want_grad=False)
    assert abs(loss - float(g[f"c{c}_eval_loss"])) <= 2e-6 * abs(loss)


def test_odd_latent_middle_column_gets_no_gradient(g):
    hidden, lat, _, p = case(g, 4)
    assert lat % 2 == 1
    I = int(g["small_meta"][1])
    R = vo.rating_matrix(g["hist_id"], g["hist_val"], I)
    b = g["batches"][0]
    mask, eps = replay(g["c4_rng"][0], len(b), I, lat, p)
    _, grad = vo.loss_grad(g["c4_N0"], R[b], I, hidden, lat, p, mask, eps, 0.1)
    enc, _ = vo.unpack(grad, I, hidden, lat)
    W, bias = enc[-1]
    assert not W[lat // 2].any() and bias[lat // 2] == 0
