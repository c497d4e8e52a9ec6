"""GPU suite for Multi-VAE (VAECF): constructor, rating rows, steps, the ml-100k driver sequence, inference and the Philox /
bf16 modes, against the reference's runs (tests/golden/vae.npz) and the fp64 oracle (oracle/vae_oracle.py)."""
import hashlib
import logging

import numpy as np
import pandas as pd
import pytest
import torch

from conftest import golden
from oracle import vae_oracle as vo

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def g():
    return golden("vae")


def _case(g, c):
    nh, lat, opt = (int(x) for x in g["case_meta"][c])
    return [int(h) for h in g["case_hidden"][c][:nh]], lat, ("sgd", "adam")[opt], float(g["case_dropout"][c])


def _cfg(U, I, **kw):
    cfg = dict(UID_NAME="user", IID_NAME="item", user_num=U, item_num=I, mlp_hidden_size=None, latent_dim=128, dropout=0.5,
               lr=1e-3, epochs=10, total_anneal_steps=100000, anneal_cap=0.2, optimizer="default", init_method="default",
               early_stop=False, topk=50, gpu="0", logger=logging.getLogger("t"), progress=False)
    cfg.update(kw)
    return cfg


def _small_model(g, c, **kw):
    from daisyrec_b200.model.VAECFRecommender import VAECF
    hidden, lat, opt, p = _case(g, c)
    U, I, total, seed = (int(x) for x in g["small_meta"])
    torch.manual_seed(seed)
    cfg = _cfg(U, I, history_item_id=torch.from_numpy(g["hist_id"]), history_item_value=torch.from_numpy(g["hist_val"]),
               mlp_hidden_size=hidden, latent_dim=lat, optimizer=opt, dropout=p, lr=0.01, total_anneal_steps=total)
    cfg.update(kw)
    return VAECF(cfg)


def _flat(model):
    """The model's parameter block in the packed (unpadded) layout of the fixture and the oracle."""
    return vo.from_device(model.net.cpu().numpy(), model.item_num, model.layers, model.lat_dim)


def _dense(R, U, I):
    rp, col, val = R.row_ptr.cpu().numpy(), R.col.cpu().numpy(), R.val.cpu().numpy()
    out = np.zeros((U, I), np.float32)
    for u in range(U):
        out[u, col[rp[u]:rp[u + 1]]] = val[rp[u]:rp[u + 1]]
    return out


def _close(got, want, opt, lr):
    d = np.abs(got - want)
    if opt == "sgd":
        assert d.max() <= 3e-6, d.max()
    else:                       # DESIGN section 4: a gradient of pure rounding noise may become a step of up to lr
        assert (d > 3e-5).sum() <= 4 and d.max() <= 2 * lr + 1e-6, ((d > 3e-5).sum(), d.max())


@pytest.mark.parametrize("c", range(5))
def test_constructor_and_rating_rows_bit_exact(g, c):
    model = _small_model(g, c)
    U, I = int(g["small_meta"][0]), int(g["small_meta"][1])
    assert np.array_equal(_flat(model), g[f"c{c}_N0"])
    assert np.array_equal(_dense(model.R, U, I), g["R"])                    # item 0 erased by the padding, duplicates once
    sd = model.state_dict()
    assert tuple(sd["encoder.0.weight"].shape) == (model.layers[0], I)
    assert model._optimizer_name() == _case(g, c)[2]


@pytest.mark.parametrize("c", range(5))
def test_steps_match_reference(g, c):
    hidden, lat, opt, p = _case(g, c)
    U, I, total, _ = (int(x) for x in g["small_meta"])
    model = _small_model(g, c)
    R = vo.rating_matrix(g["hist_id"], g["hist_val"], I)
    net_o, state = g[f"c{c}_N0"].astype(np.float64), {}
    torch.set_rng_state(torch.from_numpy(g[f"c{c}_rng"][0]))
    for s, b in enumerate(g["batches"]):
        torch_state = torch.get_rng_state()
        loss = model.train_step(torch.from_numpy(b))
        ref = g[f"c{c}_losses"][s]
        torch.set_rng_state(torch_state)
        mask = torch.empty(len(b), I).bernoulli_(1 - p).numpy().astype(np.float64) if p > 0 else None
        eps = torch.randn(len(b), lat // 2).numpy().astype(np.float64)
        lo, grad = vo.loss_grad(net_o, R[b], I, hidden, lat, p, mask, eps, vo.anneal(s + 1, 0.2, total))
        net_o = vo.step(net_o, grad, opt, 0.01, state, s + 1)
        assert abs(loss - ref) <= 1e-5 * abs(ref) and abs(loss - lo) <= 1e-5 * abs(lo), (s, loss, ref, lo)
        _close(_flat(model), g[f"c{c}_N"][s], opt, 0.01)
        _close(_flat(model), net_o, opt, 0.01)
    assert np.array_equal(torch.get_rng_state().numpy(), g[f"c{c}_rng_end"])   # the reference's draws, no more, no fewer
    model.eval()
    le = float(model.calc_loss(torch.from_numpy(g["batches"][0])))
    assert abs(le - float(g[f"c{c}_eval_loss"])) <= 1e-5 * abs(le)


def test_inference_agrees_with_forward(g):
    model = _small_model(g, 4)
    model.eval()
    U, I = int(g["small_meta"][0]), int(g["small_meta"][1])
    scores, mu, logvar = model.forward(torch.arange(U))
    hidden, lat, _, _ = _case(g, 4)
    enc, dec = vo.unpack(_flat(model), I, hidden, lat)
    R = vo.rating_matrix(g["hist_id"], g["hist_val"], I).astype(np.float64)
    h = R / np.maximum(np.sqrt((R * R).sum(1)), 1e-12)[:, None]
    for k, (W, b) in enumerate(enc):
        h = h @ W.T + b
        h = np.tanh(h) if k < len(enc) - 1 else h
    y = h[:, :lat // 2]
    for k, (W, b) in enumerate(dec):
        y = y @ W.T + b
        y = np.tanh(y) if k < len(dec) - 1 else y
    np.testing.assert_allclose(scores.cpu().numpy(), y, rtol=0, atol=2e-5)
    np.testing.assert_allclose(mu.cpu().numpy(), h[:, :lat // 2], rtol=0, atol=2e-5)
    np.testing.assert_allclose(logvar.cpu().numpy(), h[:, lat - lat // 2:], rtol=0, atol=2e-5)
    s = scores.cpu().numpy()
    assert model.predict(3, 7) == float(s[3, 7])
    model.topk = 10
    full = model.full_rank(3)
    assert full.dtype == np.int64 and np.array_equal(np.sort(s[3][full])[::-1], np.sort(s[3])[::-1][:10])
    cands = np.stack([np.random.default_rng(u).choice(I, 20, replace=False) for u in range(U)]).astype(np.int64)
    from daisyrec_b200.utils.dataset import CandidatesDataset, get_dataloader
    preds = model.rank(get_dataloader(CandidatesDataset([[u, cands[u]] for u in range(U)]), batch_size=5, shuffle=False))
    want = np.stack([cands[u][np.argsort(-s[u][cands[u]], kind="stable")[:10]] for u in range(U)])
    assert preds.dtype == np.float32 and (preds.astype(np.int64) == want).mean() >= 0.99


def test_nan_loss_raises(g):
    model = _small_model(g, 0)
    model.net.fill_(float("nan"))
    with pytest.raises(ValueError, match="Nan"):
        model.train_step(torch.arange(4))


def test_philox_is_deterministic_and_keeps_one_minus_p():
    from daisyrec_b200.model.VAECFRecommender import VAECF
    U, I, n = 1, 2000, 1000
    hid = torch.arange(n).reshape(1, n)
    cfg = _cfg(U, I, history_item_id=hid, history_item_value=torch.ones(1, n), mlp_hidden_size=[32], latent_dim=16,
               dropout=0.5, optimizer="sgd", lr=0.5, dropout_engine="philox")
    nets = []
    for _ in range(2):
        torch.manual_seed(7)
        m = VAECF(cfg)
        w0 = m.net[:I * 32].view(I, 32).clone()
        m.train_step(torch.zeros(1, dtype=torch.int64))
        nets.append(m.net.cpu().numpy())
        changed = (m.net[:I * 32].view(I, 32) != w0).any(1).cpu().numpy()
    assert np.array_equal(nets[0], nets[1])
    assert not changed[n:].any()                                             # only the user's items can move
    frac = changed[:n].mean()
    assert 0.45 <= frac <= 0.55, frac


@pytest.mark.parametrize("hidden,lat", [([600], 128), ([600], 50), ([600], 15), ([600, 150], 64)])
def test_bf16_loss_within_measured_bar(g, hidden, lat):
    """Three ml-100k-sized Adam steps: the loss with bf16 tensor-core GEMMs against the fp32 path.  latent_dim 50 and 15 and
    the [600, 150] stack put the packed weight offsets off a 4-float boundary; the block pads every part to one."""
    from daisyrec_b200.model.VAECFRecommender import VAECF
    s = golden("ml100k_sampler")
    U, I = int(g["ml_meta"][0]), int(g["ml_meta"][1])
    from daisyrec_b200.utils.utils import get_history_matrix
    df = pd.DataFrame({"user": s["coo_u"].astype(np.int64), "item": s["coo_i"].astype(np.int64)})
    cfg = _cfg(U, I, mlp_hidden_size=hidden, latent_dim=lat, dropout_engine="philox")
    cfg["history_item_id"], cfg["history_item_value"], _ = get_history_matrix(df, cfg, row="user")
    losses = {}
    for td in ("fp32", "bf16"):
        torch.manual_seed(1)
        m = VAECF(dict(cfg, tower_dtype=td))
        assert all(t.data_ptr() % 16 == 0 for t in m.parameters())           # every weight and bias 16-byte aligned
        losses[td] = [m.train_step(torch.arange(k * 300, (k + 1) * 300)) for k in range(3)]
    rel = max(abs(a - b) / abs(a) for a, b in zip(losses["fp32"], losses["bf16"]))
    print(f"bf16 vs fp32 loss {hidden}/{lat}, relative: {rel:.3e}  ({losses})")
    assert rel <= 2e-5, rel                                         # measured on a B200: 2.0e-6 at [600] / 128


def test_forward_rejects_a_dense_rating_matrix(g):
    model = _small_model(g, 0)
    U, I = int(g["small_meta"][0]), int(g["small_meta"][1])
    with pytest.raises(TypeError, match="user ids"):
        model.forward(torch.from_numpy(g["R"][:2]))
    scores, _, _ = model.forward(3)
    assert tuple(scores.shape) == (1, I)


def test_ml100k_driver_sequence(g):
    """run_examples/test.py with algo_name=multi-vae, mlp_hidden_size=[64], latent_dim=32, 2 epochs, against the reference."""
    from daisyrec_b200.model.VAECFRecommender import VAECF
    from daisyrec_b200.utils.dataset import AEDataset, CandidatesDataset, get_dataloader
    from daisyrec_b200.utils.utils import build_candidates_set, get_history_matrix, get_ur
    U, I, B, seed, topk, epochs = (int(x) for x in g["ml_meta"])
    s = golden("ml100k_sampler")
    r = golden("ml100k_rank")
    train = pd.DataFrame({"user": s["coo_u"].astype(np.int64), "item": s["coo_i"].astype(np.int64)})
    test_ur, k = {}, 0
    for u, n in zip(r["test_u"], r["gt_len"]):
        test_ur[int(u)] = set(int(x) for x in r["gt_flat"][k:k + n])
        k += n
    cfg = _cfg(U, I, mlp_hidden_size=[64], latent_dim=32, epochs=epochs, topk=topk, cand_num=1000)
    np.random.seed(seed); torch.manual_seed(seed)
    cfg["history_item_id"], cfg["history_item_value"], _ = get_history_matrix(train, cfg, row="user")
    model = VAECF(cfg)
    assert hashlib.sha256(_flat(model).tobytes()).digest() == bytes(g["ml_N0_sha"])
    losses = []
    orig = model._steps
    model._steps = lambda *a, **kw: losses.append(orig(*a, **kw)) or losses[-1]
    model.fit(get_dataloader(AEDataset(train, yield_col="user"), batch_size=B, shuffle=True, num_workers=4))
    got = torch.cat(losses).cpu().numpy()
    ref = g["ml_step_losses"]
    assert got.shape == ref.shape and np.abs(got - ref).max() <= 1e-4 * np.abs(ref).max(), (got, ref)
    assert np.array_equal(torch.get_rng_state().numpy(), g["ml_rng_end"])
    d = np.abs(_flat(model) - g["ml_N1"])
    print(f"ml-100k multi-vae: step losses {got.tolist()} (reference {ref.tolist()}); params |d| max {d.max():.3e}, "
          f"mean {d.mean():.3e}, > 1e-4: {(d > 1e-4).mean():.2e}")
    assert d.mean() <= 1e-5 and (d > 1e-4).mean() <= 1e-3
    test_u, test_ucands = build_candidates_set(test_ur, get_ur(train), cfg)
    preds = model.rank(get_dataloader(CandidatesDataset(test_ucands), batch_size=128, shuffle=False, num_workers=0))
    same = (preds.astype(np.int64) == g["ml_preds"].astype(np.int64)).mean()
    print(f"ml-100k multi-vae: rank positions equal {same:.4f}")
    assert same >= 0.95, same
