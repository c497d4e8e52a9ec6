"""Generate tests/golden/item2vec.npz by RUNNING THE REAL REFERENCE (build container only).

TEST INFRASTRUCTURE.  Usage:  python -m oracle.gen_item2vec
SkipGramNegativeSampler.sampling() iterates ``Series.iteritems``, which pandas 2 removed; ``Series.items`` yields the same
(index, value) pairs in the same order, so it stands in for it here (the other shims are those of oracle/ref_harness.py).
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_harness as rh  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
OPTS = ("sgd", "adam", "adagrad", "rmsprop")


def _reference():
    import pandas as pd
    rh.import_reference()
    if not hasattr(pd.Series, "iteritems"):
        pd.Series.iteritems = pd.Series.items


def _mt_state():
    s = np.random.get_state()
    return np.concatenate([s[1].astype(np.uint32), np.array([s[2]], np.uint32)])


def _sampler_cases(out):
    """Synthetic cases: shuffled df order, duplicate rows, a one-interaction user, a user whose complement has one item,
    windows 1 / 2 / 3, discard on and off."""
    import pandas as pd
    from daisy.utils.sampler import SkipGramNegativeSampler
    from daisy.utils.utils import get_ur
    rng = np.random.default_rng(11)
    specs = [(1, False, 7), (2, False, 8), (3, False, 9), (2, True, 10), (1, True, 12)]
    for k, (w, discard, seed) in enumerate(specs):
        U, I = 9, 14
        u = rng.integers(0, U, size=60)
        it = rng.integers(0, I, size=60)
        u = np.concatenate([u, [U, U, U], [U + 1] * (I - 1)])                     # a duplicate pair; a near-full user
        it = np.concatenate([it, [3, 3, 5], np.arange(I - 1)])
        u = np.concatenate([u, [U + 2]])                                           # one interaction
        it = np.concatenate([it, [6]])
        perm = rng.permutation(len(u))
        df = pd.DataFrame({"user": u[perm].astype(np.int64), "item": it[perm].astype(np.int64)})
        cfg = dict(UID_NAME="user", IID_NAME="item", item_num=I, train_ur=get_ur(df), context_window=w, rho=0.3)
        np.random.seed(seed)
        state0 = _mt_state()
        rows = np.asarray(SkipGramNegativeSampler(df, cfg, discard=discard).sampling())
        out[f"s{k}_users"] = df["user"].values.astype(np.int32)
        out[f"s{k}_items"] = df["item"].values.astype(np.int32)
        out[f"s{k}_meta"] = np.array([U + 3, I, w, int(discard), seed], np.int64)
        out[f"s{k}_state0"] = state0
        out[f"s{k}_rows"] = rows.astype(np.int64)
        out[f"s{k}_state1"] = _mt_state()
    out["n_sampler_cases"] = np.array(len(specs))


def _steps(out):
    """Constructor tables and 3 reference steps per optimiser on a small problem."""
    import torch
    from daisy.model.Item2VecRecommender import Item2Vec
    U, I, F, B = 12, 30, 16, 48
    rng = np.random.default_rng(5)
    batches = np.stack([np.stack([rng.integers(0, I, B), rng.integers(0, I, B), rng.integers(0, 2, B)], 1)
                        for _ in range(3)]).astype(np.int64)
    batches[0, :4, 1] = batches[0, :4, 0]                                         # target == context rows
    out["step_batches"] = batches
    out["step_meta"] = np.array([U, I, F, 2022], np.int64)
    out["step_lr"] = np.array(0.05, np.float64)
    for opt in OPTS:
        cfg = rh.make_config("item2vec", user_num=U, item_num=I, factors=F, optimizer=opt, lr=0.05, train_ur={})
        rh.seed_everything(2022)
        model = Item2Vec(cfg)
        if opt == OPTS[0]:
            out["P0"] = model.user_embedding.weight.detach().numpy().copy()
            out["Q0"] = model.shared_embedding.weight.detach().numpy().copy()
        model.criterion = model._build_criterion("CL")
        optim = model._build_optimizer(optimizer=opt, lr=0.05)
        losses, tabs = [], []
        for b in batches:
            model.zero_grad()
            loss = model.calc_loss(torch.from_numpy(b).T)
            loss.backward()
            optim.step()
            losses.append(float(loss.item()))
            tabs.append(model.shared_embedding.weight.detach().numpy().copy())
            assert model.user_embedding.weight.grad is None
        out[f"{opt}_losses"] = np.array(losses, np.float64)
        out[f"{opt}_Q"] = np.stack(tabs)


def _ml100k(out):
    """run_examples/test.py with algo_name=item2vec: 1 epoch at batch 256, build_candidates_set, rank, KPIs."""
    import torch
    from daisy.model.Item2VecRecommender import Item2Vec
    from daisy.utils.sampler import SkipGramNegativeSampler
    from daisy.utils.dataset import BasicDataset, CandidatesDataset, get_dataloader
    from daisy.utils.utils import build_candidates_set
    from daisy.utils.metrics import calc_ranking_results
    cfg = rh.make_config("item2vec", epochs=1, batch_size=256)
    rh.seed_everything(cfg["seed"])
    art = rh.load_ml100k(cfg)
    train_set, test_ur, train_ur = art["train_set"], art["test_ur"], art["train_ur"]
    model = Item2Vec(cfg)
    rows = np.asarray(SkipGramNegativeSampler(train_set, cfg).sampling())
    out["ml_state1"] = _mt_state()
    out["ml_T"] = np.array(rows.shape[0], np.int64)
    out["ml_sha256"] = np.frombuffer(hashlib.sha256(np.ascontiguousarray(rows, np.int64).tobytes()).digest(), np.uint8)
    out["ml_head"] = rows[:64].astype(np.int64)
    out["ml_tail"] = rows[-64:].astype(np.int64)
    coo = np.stack([train_set["user"].values, train_set["item"].values]).astype(np.int64)
    out["ml_coo_sha256"] = np.frombuffer(hashlib.sha256(coo.tobytes()).digest(), np.uint8)
    loader = get_dataloader(BasicDataset(rows), batch_size=cfg["batch_size"], shuffle=True, num_workers=0)
    epoch_loss = []
    orig = model.calc_loss

    def rec_loss(batch):
        loss = orig(batch)
        epoch_loss.append(float(loss.item()))
        return loss

    model.calc_loss = rec_loss
    model.fit(loader)
    out["ml_epoch_loss"] = np.array(sum(epoch_loss), np.float64)
    out["ml_P1"] = model.user_embedding.weight.detach().numpy().copy()
    out["ml_Q1"] = model.shared_embedding.weight.detach().numpy().copy()
    test_u, test_ucands = build_candidates_set(test_ur, train_ur, cfg)
    preds = model.rank(get_dataloader(CandidatesDataset(test_ucands), batch_size=128, shuffle=False, num_workers=0))
    cfg["res_path"] = tempfile.mkdtemp() + "/"
    res = calc_ranking_results(test_ur, preds, test_u, cfg)
    out["ml_test_u"] = np.array(test_u, np.int32)
    out["ml_preds"] = np.asarray(preds).astype(np.int16)
    out["ml_kpi"] = res.values[:, 1:].astype(np.float64)
    out["ml_meta"] = np.array([cfg["user_num"], cfg["item_num"], cfg["factors"], cfg["batch_size"], cfg["seed"],
                               cfg["context_window"], cfg["topk"]], np.int64)
    out["ml_lr"] = np.array(cfg["lr"], np.float64)
    print(res)


def main():
    _reference()
    out = {}
    _sampler_cases(out)
    _steps(out)
    _ml100k(out)
    path = os.path.join(GOLD, "item2vec.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


if __name__ == "__main__":
    main()
