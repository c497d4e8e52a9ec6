"""Secondary measurements (not the driver's bench): BASELINE configs 3, 4, 5 on one GPU.

    python scripts/bench_models.py lightgcn|neumf|mf-netflix|item2vec|vae [--batch B] [--steps K]
Prints one JSON line per run: triples/s with CUDA events around K steps after warm-up.
"""
import argparse
import json
import sys

import torch

sys.path.insert(0, ".")
from daisyrec_b200 import ops  # noqa: E402
from daisyrec_b200.utils.synthetic import SHAPES, make_interactions  # noqa: E402


def timed(fn, warm, steps):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def batches(U, I, n, dev, d=None):
    g = torch.Generator(device=dev); g.manual_seed(3)
    if d is not None:                                       # real (u,i) pairs + uniform negatives
        idx = torch.randint(0, d["coo_u"].numel(), (n,), device=dev, generator=g)
        bu, bi = d["coo_u"][idx].contiguous(), d["coo_i"][idx].contiguous()
    else:
        bu = torch.randint(0, U, (n,), device=dev, dtype=torch.int32, generator=g)
        bi = torch.randint(0, I, (n,), device=dev, dtype=torch.int32, generator=g)
    bj = torch.randint(0, I, (n,), device=dev, dtype=torch.int32, generator=g)
    return bu, bi, bj


def card():
    """Name and power limit of the card the numbers below come from (read in the same process as the measurement)."""
    import subprocess
    try:
        watts = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        watts = "unknown"
    return {"gpu": torch.cuda.get_device_name(), "power_limit": watts}


def bench_item2vec(dev, steps):
    """Item2Vec at the ml-20m shape: the skip-gram sampler (window 2) stage by stage and end to end, then the shared-table
    Adam step (F = 100) at B = 1 048 576 and B = 256, and a check of both against the C oracle at a small seeded size."""
    import time
    import numpy as np
    import pandas as pd
    from daisyrec_b200.utils.sampler import SkipGramNegativeSampler
    from oracle import item2vec_oracle as orc
    out = card()
    U, I, nnz = SHAPES["ml-20m"]
    F, w = 100, 2
    d = make_interactions(U, I, nnz, device=dev)
    df = pd.DataFrame({"user": d["coo_u"].cpu().numpy(), "item": d["coo_i"].cpu().numpy()})
    cfg = dict(UID_NAME="user", IID_NAME="item", item_num=I, train_ur=None, context_window=w, rho=1e-5,
               train_csr=(d["row_ptr"].cpu().numpy(), d["col"].cpu().numpy()))
    sampler = SkipGramNegativeSampler(df, cfg)
    # stages: device positions + scan, host MT19937 draws, device explode (the rows stay on the device)
    np.random.seed(1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d_su, order = torch.sort(torch.from_numpy(sampler.users).to(dev), stable=True)
    d_si = torch.from_numpy(sampler.items).to(dev)[order].contiguous()
    count, bound = ops.sgns_positions(d_su, d["row_ptr"], I, w)
    d_off = torch.zeros(len(sampler.users) + 1, dtype=torch.int64, device=dev)
    torch.cumsum(count, 0, out=d_off[1:])
    h_off, h_bound = d_off.cpu().numpy(), bound.cpu().numpy()
    t1 = time.perf_counter()
    st = ops.mt19937_from_numpy()
    draws = ops.bounded_draws_mt19937(st, h_bound, h_off)
    t2 = time.perf_counter()
    d_draws = torch.from_numpy(draws).to(dev)
    rows = ops.sgns_explode(d_su, d_si, w, d_off, d["row_ptr"], d["col"], d_draws)
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    T = rows.shape[0]
    del rows, d_draws, draws
    np.random.seed(1)
    t4 = time.perf_counter()
    host_rows = sampler.sampling()                      # the class end to end, int64 host array included
    t5 = time.perf_counter()
    assert host_rows.shape[0] == T
    out["sampler"] = {"shape": "ml-20m", "window": w, "positions": len(sampler.users), "T": T,
                      "device_ms": round(1e3 * ((t1 - t0) + (t3 - t2)), 2), "host_draw_ms": round(1e3 * (t2 - t1), 2),
                      "wall_ms": round(1e3 * (t5 - t4), 2)}
    d_rows = host_rows._drb_device
    del host_rows
    # steps: Adam, F = 100; the item table (10.7 MB) and its state stay L2-resident, the index planes stream
    g = torch.Generator(device=dev); g.manual_seed(5)
    Q0 = (torch.randn(I, F, device=dev, generator=g) * 0.01).contiguous()
    hp = ops.hyper(0.001, 0.0, 0.0, "adam", loss="CL")
    out["step"] = []
    for B in (1 << 20, 256):
        k = max(2, steps)
        n = B * k
        perm = torch.randint(0, T, (n,), device=dev, generator=g)
        bt, bc, bl = (d_rows[perm, c].contiguous() for c in range(3))
        Q = Q0.clone()
        ws = ops.Item2VecWorkspace(I, F, "adam", dev)
        ms = timed(lambda: ops.item2vec_train_steps(Q, ws, bt, bc, bl, B, 0, k, hp, check=False), 1, 3) / k
        bytes_step = (16 * F + 12) * B + 2 * 4 * 4 * I * F      # rows + indices, and theta, g, m, v of every item row in + out
        out["step"].append({"B": B, "F": F, "opt": "adam", "steps_per_launch": k, "ms_per_step": round(ms, 4),
                            "samples_per_s": round(B / ms * 1e3), "achieved_GBps": round(bytes_step / ms / 1e6, 1)})
    # outputs against the C oracle at a small seeded size (3 Adam steps)
    Is, B = 500, 4096
    gs = torch.Generator(device=dev); gs.manual_seed(7)
    trip = torch.stack([torch.randint(0, Is, (3 * B,), device=dev, generator=gs),
                        torch.randint(0, Is, (3 * B,), device=dev, generator=gs),
                        torch.randint(0, 2, (3 * B,), device=dev, generator=gs)], 1).to(torch.int32)
    Qs = (torch.randn(Is, F, device=dev, generator=gs) * 0.1).contiguous()
    Qo = Qs.cpu().numpy().copy()
    ws = ops.Item2VecWorkspace(Is, F, "adam", dev)
    losses = ops.item2vec_train_steps(Qs, ws, *(trip[:, c].contiguous() for c in range(3)), B, 0, 3, hp).cpu().numpy()
    state, lo = {}, []
    h = trip.cpu().numpy()
    for s in range(3):
        lo.append(orc.item2vec_step(Qo, h[s * B:(s + 1) * B], "adam", 0.001, state, step_count=s + 1))
    out["oracle_check"] = {"I": Is, "F": F, "B": B, "steps": 3,
                           "max_rel_loss_diff": float(np.max(np.abs(losses - lo) / np.abs(lo))),
                           "max_abs_table_diff": float(np.abs(Qs.cpu().numpy() - Qo).max())}
    return out


def _vae_model(U, I, row_ptr, col, dev, **kw):
    import logging
    from daisyrec_b200.model.VAECFRecommender import VAECF
    cfg = dict(gpu="", logger=logging.getLogger("b"), user_num=U, item_num=I, mlp_hidden_size=None, latent_dim=128, dropout=0.5,
               lr=1e-3, epochs=1, total_anneal_steps=100000, anneal_cap=0.2, optimizer="adam", init_method="default",
               early_stop=False, topk=50, train_csr=(row_ptr, col), progress=False)
    cfg.update(kw)
    return VAECF(cfg)


def bench_vae(dev, steps, batch):
    """Multi-VAE at the ml-20m shape (defaults: mlp_hidden_size [600], latent_dim 128, dropout 0.5, Adam): ms/step and users/s
    for fp32 / bf16 x torch / philox at B = 256 and one larger B, the per-kernel split (torch.profiler), FLOP and byte counts
    from shapes, the reference VAECF on CUDA (oracle/_ref) at B = 256, and an fp64-oracle parity check at a small shape."""
    import time
    import numpy as np
    from oracle import vae_oracle as vo
    out = [dict(card())]
    U, I, nnz = SHAPES["ml-20m"]
    d = make_interactions(U, I, nnz, device=dev)
    row_ptr, col = d["row_ptr"].cpu().numpy(), d["col"].cpu().numpy()
    deg = np.diff(row_ptr)
    H, lat = 600, 128
    nN = ops.vae_param_count(I, [H], lat)
    g = torch.Generator(); g.manual_seed(11)
    for B in (256, batch or 2048):
        K = max(2, steps)
        users = torch.randperm(U, generator=g)[:B * K].to(torch.int32).to(dev)
        nnz_b = float(deg[users.cpu().numpy()].mean()) * B
        wide = 3 * 2.0 * B * I * H                                                     # decoder out, dW_out, d hidden
        small = 3 * 2.0 * B * (H * lat + (lat // 2) * H)
        sparse = 2 * 2.0 * nnz_b * H
        adam_bytes = 32.0 * nN                                                         # W, g, m, v read + written
        logit_bytes = 4.0 * B * I * 5                                                  # GEMM write, 2 softmax reads, 1 write, 1 GEMM read
        for td in ("fp32", "bf16"):
            for eng in ("torch", "philox"):
                torch.manual_seed(1)
                m = _vae_model(U, I, row_ptr, col, dev, tower_dtype=td, dropout_engine=eng)
                m.train()
                m._begin_fit("adam")
                m._ensure(B)
                m._steps(users[:B], B, 1)                                              # warm-up
                torch.cuda.synchronize()
                t0 = time.time()
                losses = m._steps(users, B, K)
                torch.cuda.synchronize()
                ms = (time.time() - t0) * 1e3 / K
                out.append(dict(model="VAECF", shape="ml-20m", batch=B, tower_dtype=td, dropout_engine=eng, ms_per_step=ms,
                                users_per_s=B / ms * 1e3, loss_last=float(losses[-1]), flop_per_step=wide + small + sparse,
                                TFLOPs=(wide + small + sparse) / ms / 1e9, adam_and_logit_bytes=adam_bytes + logit_bytes,
                                GBps=(adam_bytes + logit_bytes) / ms / 1e6, params=nN, nnz_per_step=nnz_b))
                del m
                torch.cuda.empty_cache()
    # per-kernel split of one Philox step at B = 256 per dtype
    from torch.profiler import profile, ProfilerActivity
    for td in ("fp32", "bf16"):
        torch.manual_seed(1)
        m = _vae_model(U, I, row_ptr, col, dev, tower_dtype=td, dropout_engine="philox")
        m.train()
        m._begin_fit("adam")
        m._ensure(256)
        us = torch.randperm(U, generator=g)[:256 * 8].to(torch.int32).to(dev)
        m._steps(us, 256, 2)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m._steps(us, 256, 8)
            torch.cuda.synchronize()
        split = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and getattr(e, "device_time_total", 0) > 0:
                split[e.key[:60]] = round(e.device_time_total / 8 / 1e3, 4)
        out.append(dict(model="VAECF", batch=256, tower_dtype=td, kernel_ms_per_step=dict(sorted(split.items(), key=lambda kv: -kv[1])[:14])))
        del m
    # the reference VAECF on CUDA (installed copy), on the first 4096 users (its padded history lives on the device)
    try:
        from oracle import ref_harness as rh
        rh.use_root(rh.INSTALLED_ROOT)
        rh.import_reference()
        from daisy.model.VAECFRecommender import VAECF as RefVAE
        Ur = 4096
        L = int(deg[:Ur].max())
        hid = np.zeros((Ur, L), np.int64)
        for u in range(Ur):
            hid[u, :deg[u]] = col[row_ptr[u]:row_ptr[u + 1]]
        hval = (np.arange(L)[None, :] < deg[:Ur, None]).astype(np.float32)
        cfg = rh.make_config("multi-vae", user_num=Ur, item_num=I, history_item_id=torch.from_numpy(hid),
                             history_item_value=torch.from_numpy(hval))
        cfg["gpu"] = "0"
        ref = RefVAE(cfg).cuda()
        opt = ref._build_optimizer(optimizer="adam", lr=1e-3)
        ref.train()

        def ref_step(b):
            ref.zero_grad()
            loss = ref.calc_loss(b)
            loss.backward()
            opt.step()
        ub = [torch.randint(0, Ur, (256,), generator=g) for _ in range(steps + 2)]
        ref_step(ub[0]); ref_step(ub[1])
        torch.cuda.synchronize()
        t0 = time.time()
        for b in ub[2:]:
            ref_step(b)
        torch.cuda.synchronize()
        ms = (time.time() - t0) * 1e3 / steps
        out.append(dict(model="reference VAECF (torch, CUDA)", batch=256, ms_per_step=ms, users_per_s=256 / ms * 1e3))
    except Exception as e:                                  # the installed reference copy is optional
        out.append(dict(model="reference VAECF (torch, CUDA)", error=repr(e)[:200]))
    # parity against the fp64 oracle at a small shape (host masks and eps, one Adam step)
    Us, Is = 64, 500
    rng = np.random.default_rng(0)
    hid = rng.integers(0, Is, size=(Us, 30))
    hval = (rng.random((Us, 30)) < 0.8).astype(np.float32)
    from daisyrec_b200.model.VAECFRecommender import VAECF
    import logging
    torch.manual_seed(3)
    m = VAECF(dict(gpu="", logger=logging.getLogger("b"), user_num=Us, item_num=Is, mlp_hidden_size=[64], latent_dim=32,
                   dropout=0.5, lr=1e-3, epochs=1, total_anneal_steps=100, anneal_cap=0.2, optimizer="adam", init_method="default",
                   early_stop=False, topk=10, history_item_id=torch.from_numpy(hid), history_item_value=torch.from_numpy(hval),
                   dropout_engine="torch"))
    N0 = vo.from_device(m.net.cpu().numpy(), Is, [64], 32).astype(np.float64)
    b = np.arange(32)
    st = torch.get_rng_state()
    loss = m.train_step(torch.from_numpy(b))
    torch.set_rng_state(st)
    mask = torch.empty(32, Is).bernoulli_(0.5).numpy().astype(np.float64)
    eps = torch.randn(32, 16).numpy().astype(np.float64)
    R = vo.rating_matrix(hid, hval, Is)
    lo, grad = vo.loss_grad(N0, R[b], Is, [64], 32, 0.5, mask, eps, vo.anneal(1, 0.2, 100))
    Nn = vo.step(N0, grad, "adam", 1e-3, {}, 1)
    dN = np.abs(vo.from_device(m.net.cpu().numpy(), Is, [64], 32) - Nn)
    out.append(dict(check="oracle parity, 64 users x 500 items, one Adam step", loss=loss, oracle_loss=lo,
                    loss_rel=abs(loss - lo) / abs(lo), params_max_abs=float(dN.max()), params_over_1e5=int((dN > 1e-5).sum())))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["lightgcn", "neumf", "mf-netflix", "mf-fit", "mf-fused", "item2vec", "vae"])
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--tower", default="fp32", choices=["fp32", "bf16"])
    a = ap.parse_args()
    dev = torch.device("cuda")
    if a.what == "item2vec":
        print(json.dumps(bench_item2vec(dev, a.steps)))
        return
    if a.what == "vae":
        for line in bench_vae(dev, a.steps, a.batch):
            print(json.dumps(line))
        return
    if a.what == "lightgcn":
        U, I, nnz = SHAPES["amazon-book"]
        F, L = 64, 3
        B = a.batch or 65536
        d = make_interactions(U, I, nnz, device=dev)
        row_ptr, col, val = ops.lgcn_norm_adj(d["coo_u"].cpu().numpy(), d["coo_i"].cpu().numpy(), U, I)
        graph = ops.LgcnGraph(row_ptr, col, val, dev)
        E0 = (torch.randn(U + I, F, device=dev) * 0.05).contiguous()
        ws = ops.LgcnWorkspace(U, I, F, "adam", dev)
        hp = ops.hyper(0.01, 0.0, 0.0, "adam")
        bu, bi, bj = batches(U, I, B * 4, dev, d)
        step = [0]

        def fn():
            ops.lgcn_bpr_train_steps(E0, ws, graph, L, bu, bi, bj, B, step[0] % 4, 1, hp, adam_step0=step[0], check=False)
            step[0] += 1
        ms = timed(fn, 3, a.steps)
        nnzA = int(row_ptr[-1])
        alg = 2 * L * (nnzA * (8 + 4 * F) + (U + I) * 4 * F) + B * (24 * F + 12)
        print(json.dumps(dict(model="LightGCN", shape="amazon-book", U=U, I=I, nnzA=nnzA, F=F, L=L, batch=B, ms_per_step=ms,
                              triples_per_s=B / ms * 1e3, alg_bytes_per_step=alg, alg_GBps=alg / ms / 1e6,
                              spmm_segments=graph.nseg)))
    elif a.what == "neumf":
        U, I, _ = SHAPES["ml-20m"]
        F, L = 32, 2
        B = a.batch or 262144
        D = F * 2 ** (L - 1)
        tabs = [(torch.randn(s, device=dev) * 0.05).contiguous() for s in ((U, F), (I, F), (U, D), (I, D))]
        W = (torch.randn(ops.neumf_param_count(F, L), device=dev) * 0.1).contiguous()
        ws = ops.NeumfWorkspace(U, I, F, L, "adam", 2 * B, dev)
        hp = ops.hyper(0.001, 0.001, 0.001, "adam")
        bu, bi, bj = batches(U, I, B * 4, dev)
        step = [0]

        def fn():
            ops.neumf_bpr_train_steps(tabs, W, ws, bu, bi, bj, B, step[0] % 4, 1, hp, adam_step0=step[0], check=False,
                                      tower_dtype=1 if a.tower == 'bf16' else 0)
            step[0] += 1
        ms = timed(fn, 3, a.steps)
        flop = 0
        n_in = 2 * D
        for _ in range(L):
            flop += 2 * n_in * (n_in // 2)
            n_in //= 2
        flop_triple = 2 * 3 * flop                          # 2 items x (fwd + 2 bwd GEMMs)
        print(json.dumps(dict(model="NeuMF", shape="ml-20m", F=F, L=L, batch=B, ms_per_step=ms, triples_per_s=B / ms * 1e3,
                              tower_TFLOPs=B * flop_triple / ms / 1e9, tower="fp32 CUDA cores" if a.tower == "fp32" else "bf16 tcgen05 (TMEM accumulator)")))
    elif a.what == "mf-fused":
        # throughput mode: negatives drawn inside the step kernel (Philox + k-th complement over the CSR row)
        U, I, nnz = SHAPES["ml-20m"]
        F, B, K = 64, a.batch or (1 << 20), 16
        d = make_interactions(U, I, nnz, device=dev)
        P = (torch.randn(U, F, device=dev) * 0.01).contiguous(); Q = (torch.randn(I, F, device=dev) * 0.01).contiguous()
        ws = ops.MFWorkspace(U, I, F, "sgd", dev)
        hp = ops.hyper(0.01, 0.001, 0.001)
        g = torch.Generator(device=dev); g.manual_seed(5)
        idx = torch.randint(0, d["coo_u"].numel(), (B * K,), device=dev, generator=g)
        bu, bi = d["coo_u"][idx].contiguous(), d["coo_i"][idx].contiguous()
        bj = torch.randint(0, I, (B * K,), device=dev, dtype=torch.int32, generator=g)
        ms_f = timed(lambda: ops.mf_bpr_train_steps_fused_neg(P, Q, ws, bu, bi, d["row_ptr"], d["col"], 1, B, 0, K, hp, check=False), 1, 3) / K
        ms_t = timed(lambda: ops.mf_bpr_train_steps(P, Q, ws, bu, bi, bj, B, 0, K, hp, check=False), 1, 3) / K
        print(json.dumps(dict(model="MF", shape="ml-20m", F=F, batch=B, fused_sampler_ms_per_step=ms_f,
                              fused_sampler_triples_per_s=B / ms_f * 1e3, table_mode_ms_per_step=ms_t,
                              table_mode_triples_per_s=B / ms_t * 1e3)))
    elif a.what == "mf-fit":
        # wall-clock of the drop-in API at config-2 scale: MF(config).fit(DataLoader over the 80 M sampler triples)
        import logging, time as _t
        sys.path.insert(0, ".")
        import bench as Bn
        from daisyrec_b200.model.MFRecommender import MF
        from daisyrec_b200.utils.dataset import BasicDataset, get_dataloader
        from daisyrec_b200.utils.sampler import TripleArray
        d, triples = Bn.build_workload("ml-20m", dev, 4, 2022, "cuda")
        host = triples.cpu().numpy().view(TripleArray)
        host._drb_device = triples
        for engine in ("torch", "device"):
            cfg = dict(gpu="", logger=logging.getLogger("b"), lr=0.01, reg_1=0.001, reg_2=0.001, epochs=2, topk=50,
                       user_num=d["user_num"], item_num=d["item_num"], factors=64, loss_type="BPR", optimizer="default",
                       init_method="default", early_stop=False, progress=False, shuffle_engine=engine)
            model = MF(cfg)
            loader = get_dataloader(BasicDataset(host), batch_size=a.batch or (1 << 20), shuffle=True)
            torch.cuda.synchronize(); t0 = _t.time()
            model.fit(loader)
            torch.cuda.synchronize(); dt = _t.time() - t0
            print(json.dumps(dict(model="MF.fit drop-in", shuffle_engine=engine, epochs=2, triples=int(host.shape[0]),
                                  wall_s=dt, triples_per_s_wall=2 * host.shape[0] / dt)))
    else:
        U, I, nnz = SHAPES["netflix"]
        F = 128
        B = a.batch or (1 << 20)
        P = (torch.randn(U, F, device=dev) * 0.01).contiguous()
        Q = (torch.randn(I, F, device=dev) * 0.01).contiguous()
        ws = ops.MFWorkspace(U, I, F, "sgd", dev)
        hp = ops.hyper(0.01, 0.001, 0.001)
        K = 16
        bu, bi, bj = batches(U, I, B * K, dev)
        bi = (I * torch.rand(B * K, device=dev).pow(2.0)).to(torch.int32).clamp_(0, I - 1)

        def fn():
            ops.mf_bpr_train_steps(P, Q, ws, bu, bi, bj, B, 0, K, hp, check=False)
        ms = timed(fn, 1, max(1, a.steps // 4)) / K
        print(json.dumps(dict(model="MF", shape="netflix", U=U, I=I, F=F, batch=B, ms_per_step=ms, triples_per_s=B / ms * 1e3,
                              alg_GBps=B * (24 * F + 12) / ms / 1e6)))


if __name__ == "__main__":
    main()
