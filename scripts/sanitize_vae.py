"""Tiny run of every Multi-VAE kernel, meant for `compute-sanitizer --tool memcheck python scripts/sanitize_vae.py`:
fp32 and bf16, dropout on (host masks and Philox), a ragged last batch, an odd latent_dim and a two-layer stack whose packed
offsets are off a 4-float boundary, then rank / full_rank / predict / forward."""
import logging
import sys

import numpy as np
import pandas as pd
import torch

sys.path.insert(0, ".")
from daisyrec_b200.model.VAECFRecommender import VAECF  # noqa: E402
from daisyrec_b200.utils.dataset import AEDataset, CandidatesDataset, get_dataloader  # noqa: E402
from daisyrec_b200.utils.utils import get_history_matrix  # noqa: E402

rng = np.random.default_rng(0)
U, I = 50, 300
users = rng.integers(0, U, 1500)
df = pd.DataFrame({"user": np.concatenate([np.arange(U), users]), "item": rng.integers(0, I, U + 1500)})
cfg = dict(UID_NAME="user", IID_NAME="item", user_num=U, item_num=I, mlp_hidden_size=[64, 24], latent_dim=15, dropout=0.5,
           lr=1e-3, epochs=2, total_anneal_steps=10, anneal_cap=0.2, optimizer="adam", init_method="default", early_stop=False,
           topk=10, gpu="", logger=logging.getLogger("s"), progress=False)
cfg["history_item_id"], cfg["history_item_value"], _ = get_history_matrix(df, cfg, row="user")
cands = [[u, rng.choice(I, 40, replace=False)] for u in range(U)]
for td in ("fp32", "bf16"):
    for engine in ("torch", "philox"):
        torch.manual_seed(1)
        m = VAECF(dict(cfg, tower_dtype=td, dropout_engine=engine))
        m.fit(get_dataloader(AEDataset(df), batch_size=16, shuffle=True))       # 50 users: the last batch holds 2
        m.train()
        m.calc_loss(torch.arange(7))
        m.eval()
        preds = m.rank(get_dataloader(CandidatesDataset(cands), batch_size=16, shuffle=False))
        full = m.full_rank(3)
        p = m.predict(3, 5)
        scores, mu, logvar = m.forward(torch.arange(U))
        torch.cuda.synchronize()
        assert np.isfinite(scores.cpu().numpy()).all() and preds.shape == (U, 10), (td, engine)
        print(f"{td} {engine}: ok (predict {p:.4f}, full_rank head {full[:3].tolist()})")
