"""GPU drop-in test: the reference driver's call sequence (run_examples/test.py:41-120) executed on
the B200 classes, checked against the golden artefacts of the same sequence run on the reference.
"""
import logging

import numpy as np
import pandas as pd
import pytest
import torch

from conftest import golden

pytestmark = pytest.mark.gpu


def _config(**kw):
    cfg = dict(gpu='0', seed=2022, topk=50, cand_num=1000, sample_method='uniform', sample_ratio=0, num_ng=4,
               batch_size=256, loss_type='BPR', init_method='default', optimizer='default', early_stop=False,
               UID_NAME='user', IID_NAME='item', INTER_NAME='rating', TID_NAME='timestamp',
               factors=32, epochs=1, lr=0.01, reg_1=0.001, reg_2=0.001, logger=logging.getLogger('t'), progress=False)
    cfg.update(kw)
    return cfg


def test_ml100k_driver_sequence():
    from daisyrec_b200.model.MFRecommender import MF
    from daisyrec_b200.utils.sampler import BasicNegtiveSampler
    from daisyrec_b200.utils.dataset import BasicDataset, CandidatesDataset, get_dataloader
    from daisyrec_b200.utils.utils import get_ur, build_candidates_set
    gs, gf, gr = golden("ml100k_sampler"), golden("ml100k_fit"), golden("ml100k_rank")
    U, I, G, seed = (int(v) for v in gs["meta"])
    train_set = pd.DataFrame({"user": gs["coo_u"].astype(np.int64), "item": gs["coo_i"].astype(np.int64), "rating": 1.0,
                              "timestamp": np.arange(len(gs["coo_u"]))})
    off = np.concatenate([[0], np.cumsum(gr["gt_len"])])
    test_ur = {int(u): gr["gt_flat"][off[k]:off[k + 1]].tolist() for k, u in enumerate(gr["test_u"])}

    cfg = _config(user_num=U, item_num=I)
    np.random.seed(seed); torch.manual_seed(seed)                     # init_seed, config.py:32-36
    train_ur = get_ur(train_set)
    cfg['train_ur'] = train_ur
    model = MF(cfg)                                                   # test.py:90
    assert np.array_equal(model.embed_user.weight.cpu().numpy(), gf["P0"])
    assert np.array_equal(model.embed_item.weight.cpu().numpy(), gf["Q0"])
    samples = BasicNegtiveSampler(train_set, cfg).sampling()          # test.py:91-92
    assert samples.dtype == np.int32 and samples.shape == (313452, 3)
    assert np.array_equal(samples[:, 2], gs["triples_j"].astype(np.int32))
    loader = get_dataloader(BasicDataset(samples), batch_size=cfg['batch_size'], shuffle=True, num_workers=4)
    model.fit(loader)                                                 # test.py:95
    for got, want in ((model.embed_user.weight.cpu().numpy(), gf["P1"]), (model.embed_item.weight.cpu().numpy(), gf["Q1"])):
        err = np.abs(got - want)
        assert err.max() < 1e-4 and (err < 5e-6).mean() > 0.999
    test_u, test_ucands = build_candidates_set(test_ur, train_ur, cfg)  # test.py:112
    assert test_u == [int(u) for u in gr["test_u"]]
    assert np.array_equal(np.stack([c[1] for c in test_ucands]), gr["cands"].astype(np.int64))
    assert np.array_equal(np.random.randint(0, 2 ** 31 - 1, size=3), gr["next"])   # numpy stream in lock-step
    test_loader = get_dataloader(CandidatesDataset(test_ucands), batch_size=128, shuffle=False, num_workers=0)
    preds = model.rank(test_loader)                                   # test.py:120
    assert preds.dtype == np.float32 and preds.shape == (304, 50)
    # After GPU training the tables differ from the reference's by fp32 re-association noise (the reference's own autograd
    # sums in ANOTHER fp32 order than any other implementation), so a list can differ from the reference's exactly where two
    # candidates are tied to within that noise.  Checked position by position: wherever the ids differ, the REFERENCE's own
    # scores (its trained tables gf[P1], gf[Q1], fp64 dot) of the two candidates are closer than the score perturbation the
    # observed table difference can cause -- i.e. every mismatch is a near-tie, there is no mis-ranking.
    ref = gr["preds"]
    assert (preds == ref).mean() > 0.98
    Pr, Qr = gf["P1"].astype(np.float64), gf["Q1"].astype(np.float64)
    dP = np.abs(model.embed_user.weight.cpu().numpy() - gf["P1"]).max()
    dQ = np.abs(model.embed_item.weight.cpu().numpy() - gf["Q1"]).max()
    noise = 2.0 * cfg['factors'] * (dP * np.abs(Qr).max() + dQ * np.abs(Pr).max()) + 1e-7
    rows, cols = np.nonzero(preds != ref)
    users_arr = np.asarray(test_u)
    for r, k in zip(rows, cols):
        u = users_arr[r]
        gap = abs(Pr[u] @ Qr[int(preds[r, k])] - Pr[u] @ Qr[int(ref[r, k])])
        # the candidate we placed at k is within noise of the reference's k-th candidate, or the lists are shifted by one
        # around a near-tie: compare against the neighbouring reference positions too
        near = min(abs(Pr[u] @ Qr[int(preds[r, k])] - Pr[u] @ Qr[int(ref[r, kk])])
                   for kk in range(max(0, k - 1), min(ref.shape[1], k + 2)))
        assert min(gap, near) <= noise, (int(r), int(k), float(gap), float(near), float(noise))
    # with the reference's own trained tables the ids are bit-identical
    model.load_state_dict({'embed_user.weight': torch.from_numpy(gf["P1"]).cuda(),
                           'embed_item.weight': torch.from_numpy(gf["Q1"]).cuda()})
    assert np.array_equal(model.rank(test_loader), gr["preds"])
    assert np.array_equal(np.stack([model.full_rank(int(u)) for u in test_u[:16]]), gr["full"])
    assert abs(model.predict(int(test_u[0]), int(gr["cands"][0][-1])) - float(gr["pred_pairs"][0])) < 1e-6


def test_generic_loader_and_calc_loss_paths():
    """A plain iterable of collated batches takes the per-batch host path (train_step)."""
    from daisyrec_b200.model.MFRecommender import MF
    rng = np.random.default_rng(0)
    U, I = 300, 200
    cfg = _config(user_num=U, item_num=I, factors=64, epochs=2)
    torch.manual_seed(1)
    a, b = MF(cfg), None
    torch.manual_seed(1)
    b = MF(cfg)
    data = np.stack([rng.integers(U, size=5000), rng.integers(I, size=5000), rng.integers(I, size=5000)], 1).astype(np.int32)
    batches = [[torch.from_numpy(data[s:s + 512, k].copy()) for k in range(3)] for s in range(0, 5000, 512)]
    l0 = float(a.calc_loss(batches[0]))
    a.fit(batches)                                                    # generic path
    from daisyrec_b200.utils.dataset import BasicDataset, get_dataloader
    b.fit(get_dataloader(BasicDataset(data), batch_size=512, shuffle=False))   # bulk path, same order
    np.testing.assert_allclose(a.embed_user.weight.cpu().numpy(), b.embed_user.weight.cpu().numpy(), atol=3e-6)
    assert l0 > 0 and float(a.calc_loss(batches[0])) < l0             # training reduced the loss


def test_unsupported_options_fail_loudly():
    from daisyrec_b200.model.MFRecommender import MF
    with pytest.raises(NotImplementedError):                           # AbstractRecommender.py:90-91
        MF(_config(user_num=10, item_num=10, loss_type='nope')).fit([])
    with pytest.raises(RuntimeError):                                  # optim.SparseAdam.step() on dense gradients
        MF(_config(user_num=10, item_num=10, optimizer='sparse_adam')).fit([])
    with pytest.raises(NotImplementedError):                           # point-wise rows come from the sampler, not the fused draw
        MF(_config(user_num=10, item_num=10, loss_type='CL', neg_sampling='fused',
                   train_ur={u: {0} for u in range(10)})).fit([])


def test_edge_cases_small_inputs():
    """Inputs the reference mishandles or never sees: one test user (the reference's .squeeze() breaks, MFRecommender.py:115),
    fewer triples than one batch, topk larger than the candidate list, a user without any train interaction."""
    from daisyrec_b200.model.MFRecommender import MF
    from daisyrec_b200.utils.sampler import BasicNegtiveSampler
    from daisyrec_b200.utils.dataset import BasicDataset, CandidatesDataset, get_dataloader
    U, I = 12, 20
    cfg = _config(user_num=U, item_num=I, factors=8, topk=50, cand_num=7)
    torch.manual_seed(0); np.random.seed(0)
    model = MF(cfg)
    loader1 = get_dataloader(CandidatesDataset([[3, np.array([1, 5, 5, 9, 0, 2, 19])]]), batch_size=128, shuffle=False)
    out = model.rank(loader1)
    assert out.shape == (1, 7) and sorted(out[0].tolist()) == [0, 1, 2, 5, 5, 9, 19]      # topk clipped to cand_num
    df = pd.DataFrame({"user": [0, 0, 1, 3, 3, 3], "item": [1, 2, 3, 4, 5, 6], "rating": 1.0, "timestamp": range(6)})
    ur = {0: {1, 2}, 1: {3}, 3: {4, 5, 6}}
    from collections import defaultdict
    cfg['train_ur'] = defaultdict(set, ur)                              # users 2, 4..11 have no interactions
    tri = BasicNegtiveSampler(df, cfg).sampling()
    assert tri.shape == (24, 3)
    for u, i, j in tri:
        assert j not in ur[int(u)] and 0 <= j < I
    model.fit(get_dataloader(BasicDataset(tri), batch_size=256, shuffle=True))          # 24 triples < one batch
    assert np.isfinite(model.embed_user.weight.cpu().numpy()).all()
    assert model.rank(get_dataloader(CandidatesDataset([]), batch_size=128, shuffle=False)).shape[0] == 0


def test_deterministic_mode_is_bitwise_reproducible(orc):
    """deterministic=True: every cross-thread sum of a step is taken in fixed point (integer atomics are associative), so two
    fits from the same state give bitwise identical tables and epoch losses; the default mode (float RED in arrival order)
    agrees with it to fp32 noise; and the oracle, which accumulates the same sums in fp64, stays within 1e-6 of it."""
    from daisyrec_b200.model.MFRecommender import MF
    from daisyrec_b200.utils.dataset import BasicDataset, get_dataloader
    rng = np.random.default_rng(12)
    U, I, T, B = 400, 300, 40_000, 512
    users = np.minimum(U - 1, rng.zipf(1.3, size=T) - 1)                 # hot rows: many contributions per row and step
    data = np.stack([users, rng.integers(I, size=T), rng.integers(I, size=T)], 1).astype(np.int32)
    runs = []
    for det in (True, True, False):
        cfg = _config(user_num=U, item_num=I, factors=64, epochs=2, batch_size=B, deterministic=det)
        torch.manual_seed(7)
        m = MF(cfg)
        P0, Q0 = m.embed_user.weight.cpu().numpy().copy(), m.embed_item.weight.cpu().numpy().copy()
        m.fit(get_dataloader(BasicDataset(data), batch_size=B, shuffle=False))
        runs.append((m.embed_user.weight.cpu().numpy(), m.embed_item.weight.cpu().numpy()))
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])       # bitwise
    for a, b in zip(runs[0], runs[2]):
        d = np.abs(a - b)
        assert (d > 5e-6).mean() < 2e-3 and d.max() < 1e-3
    Po, Qo = P0.copy(), Q0.copy()
    for _ in range(2):
        orc.mf_bpr_epoch(Po, Qo, np.ascontiguousarray(data), None, B, orc.hyper(0.01, 0.001, 0.001))
    for got, want, equal in ((runs[0][0], Po, 0.6), (runs[0][1], Qo, 0.15)):
        # Measured on a B200 (1000 W limit): 0.70 of P and 0.18 of Q bit-equal, largest differences 3e-7 and 1.1e-8.  A single step leaves
        # some entries one fp32 ulp apart (the default mode the same ones), and later steps carry them on; an item row takes
        # few contributions per step, so a larger share of Q carries one.
        assert (got == want).mean() > equal and np.abs(got - want).max() < 1e-6, \
            (float((got == want).mean()), float(np.abs(got - want).max()))
