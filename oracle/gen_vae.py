"""Generate tests/golden/vae.npz by RUNNING THE REAL REFERENCE (build container only).

TEST INFRASTRUCTURE.  Usage:  python -m oracle.gen_vae
The reference runs single-threaded: CPU index_put_ without accumulate is parallel, so the item-0 overwrite of
get_user_rating_matrix is only well defined with one thread.
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_harness as rh  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
# (hidden, latent_dim, optimizer, dropout)
CASES = [([32], 16, "sgd", 0.5), ([32], 16, "sgd", 0.0), ([32], 16, "adam", 0.5), ([32], 16, "adam", 0.0),
         ([24, 16], 15, "adam", 0.5)]


def flat(model):
    """state_dict -> the device block layout (encoder.0 weight transposed)."""
    sd = model.state_dict()
    parts = []
    for side, n in (("encoder", len(model.encode_layer_dims) - 1), ("decoder", len(model.decode_layer_dims) - 1)):
        for k in range(n):
            w = sd[f"{side}.{2 * k}.weight"].detach().numpy()
            parts += [(w.T if (side == "encoder" and k == 0) else w).reshape(-1), sd[f"{side}.{2 * k}.bias"].detach().numpy()]
    return np.concatenate(parts).astype(np.float32)


def _sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def _small_df():
    """Users with histories of different lengths, item 0 in some of them, a duplicate (user, item) row."""
    import pandas as pd
    rng = np.random.default_rng(17)
    U, I = 12, 40
    users, items = [], []
    for u in range(U):
        n = int(rng.integers(1, 9))
        its = rng.choice(I, size=n, replace=False)
        if u % 3 == 0:
            its[0] = 0                                                           # item 0 in a short row: erased by padding
        users += [u] * n
        items += its.tolist()
    users += [5, 5, 11]                                                          # a duplicate pair and a longest row
    items += [items[users.index(5)], 0, 0]
    users += [11] * 12
    items += list(range(20, 32))
    perm = rng.permutation(len(users))
    return pd.DataFrame({"user": np.array(users)[perm], "item": np.array(items)[perm]}), U, I


def _small(out):
    import torch
    from daisy.model.VAECFRecommender import VAECF
    from daisy.utils.utils import get_history_matrix
    df, U, I = _small_df()
    base = rh.make_config("multi-vae", user_num=U, item_num=I, lr=0.01, total_anneal_steps=10)
    hid, hval, hlen = get_history_matrix(df, base, row="user")
    out["df_user"] = df["user"].values.astype(np.int64)
    out["df_item"] = df["item"].values.astype(np.int64)
    out["hist_id"], out["hist_val"], out["hist_len"] = hid.numpy(), hval.numpy(), hlen.numpy()
    out["small_meta"] = np.array([U, I, 10, 2022], np.int64)
    rng = np.random.default_rng(3)
    batches = np.stack([rng.permutation(U)[:8] for _ in range(3)]).astype(np.int64)
    out["batches"] = batches
    for c, (hidden, lat, opt, p) in enumerate(CASES):
        cfg = dict(base, history_item_id=hid, history_item_value=hval, mlp_hidden_size=hidden, latent_dim=lat, optimizer=opt,
                   dropout=p)
        rh.seed_everything(2022)
        model = VAECF(cfg)
        if c == 0:
            out["R"] = model.get_user_rating_matrix(torch.arange(U)).numpy()
        out[f"c{c}_N0"] = flat(model)
        optim = model._build_optimizer(optimizer=opt, lr=cfg["lr"])
        model.train()
        states, losses, nets = [], [], []
        for b in batches:
            states.append(torch.get_rng_state().numpy())
            model.zero_grad()
            loss = model.calc_loss(torch.from_numpy(b))
            loss.backward()
            optim.step()
            losses.append(float(loss.item()))
            nets.append(flat(model))
        model.eval()
        out[f"c{c}_eval_loss"] = np.array(float(model.calc_loss(torch.from_numpy(batches[0])).item()))
        out[f"c{c}_rng"] = np.stack(states)
        out[f"c{c}_rng_end"] = torch.get_rng_state().numpy()
        out[f"c{c}_losses"] = np.array(losses, np.float64)
        out[f"c{c}_N"] = np.stack(nets)
    out["n_cases"] = np.array(len(CASES))
    out["case_hidden"] = np.array([h + [0] * (2 - len(h)) for h, _, _, _ in CASES], np.int64)
    out["case_meta"] = np.array([[len(h), lat, 0 if o == "sgd" else 1] for h, lat, o, _ in CASES], np.int64)
    out["case_dropout"] = np.array([p for _, _, _, p in CASES], np.float64)


def _ml100k(out):
    """run_examples/test.py with algo_name=multi-vae, mlp_hidden_size=[64], latent_dim=32, 2 epochs."""
    import torch
    from daisy.model.VAECFRecommender import VAECF
    from daisy.utils.dataset import AEDataset, CandidatesDataset, get_dataloader
    from daisy.utils.utils import build_candidates_set, get_history_matrix
    cfg = rh.make_config("multi-vae", epochs=2, mlp_hidden_size=[64], latent_dim=32)
    rh.seed_everything(cfg["seed"])
    art = rh.load_ml100k(cfg)
    train_set, test_ur, train_ur = art["train_set"], art["test_ur"], art["train_ur"]
    hid, hval, hlen = get_history_matrix(train_set, cfg, row="user")
    out["ml_hist_sha"] = np.stack([_sha(hid.numpy()), _sha(hval.numpy()), _sha(hlen.numpy())])
    cfg["history_item_id"], cfg["history_item_value"] = hid, hval
    model = VAECF(cfg)
    out["ml_N0_sha"] = _sha(flat(model))
    loader = get_dataloader(AEDataset(train_set, yield_col=cfg["UID_NAME"]), batch_size=cfg["batch_size"], shuffle=True,
                            num_workers=0)
    losses = []
    orig = model.calc_loss

    def rec(batch):
        loss = orig(batch)
        losses.append(float(loss.item()))
        return loss

    model.calc_loss = rec
    model.fit(loader)
    out["ml_step_losses"] = np.array(losses, np.float64)
    out["ml_N1"] = flat(model)
    out["ml_rng_end"] = torch.get_rng_state().numpy()
    test_u, test_ucands = build_candidates_set(test_ur, train_ur, cfg)
    preds = model.rank(get_dataloader(CandidatesDataset(test_ucands), batch_size=128, shuffle=False, num_workers=0))
    out["ml_preds"] = np.asarray(preds).astype(np.int16)
    out["ml_meta"] = np.array([cfg["user_num"], cfg["item_num"], cfg["batch_size"], cfg["seed"], cfg["topk"], 2], np.int64)


def main():
    import torch
    torch.set_num_threads(1)
    rh.import_reference()
    out = {}
    _small(out)
    _ml100k(out)
    path = os.path.join(GOLD, "vae.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


if __name__ == "__main__":
    main()
