"""NFM on the device (daisy/model/NFMRecommender.py:14-209; SURVEY 8(f) rank 4) against the reference-generated fixture
tests/golden/nfm.npz (5 cases: with / without BatchNorm, relu / sigmoid / tanh, 1-3 layers, SGD / Adam) and the pinned oracle."""
import logging

import numpy as np
import pytest
import torch

from conftest import golden

pytestmark = pytest.mark.gpu
SEEDS = [51, 52, 53, 54, 55]
ACTS = ["relu", "sigmoid", "tanh"]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_nfm_steps_match_reference_fixture(orc):
    from daisyrec_b200 import ops
    g = golden("nfm")
    for c in range(int(g["ncases"])):
        L, bn, act, lr, r1, r2, opt = g[f"c{c}_hyper"]
        L, bn, act = int(L), bool(bn), int(act)
        optn = "sgd" if opt == 0 else "adam"
        Ps, Qs, Bs, Ns, Rs = g[f"c{c}_P"], g[f"c{c}_Q"], g[f"c{c}_bias"], g[f"c{c}_N"], g[f"c{c}_R"]
        bs, losses = g[f"c{c}_batches"], g[f"c{c}_loss"]
        U, F = Ps.shape[1:]
        I = Qs.shape[1]
        assert Ns.shape[1] == ops.nfm_param_count(F, L, bn)
        hp = ops.hyper(float(lr), float(r1), float(r2), optn)
        ws = ops.NfmWorkspace(U, I, F, L, bn, optn, 2 * bs.shape[2], "cuda")       # optimiser state carried across the steps
        for s in range(bs.shape[0]):
            P, Q, bias, N = dev(Ps[s]), dev(Qs[s]), dev(Bs[s]), dev(Ns[s])
            R = dev(Rs[s]) if bn else None
            b = [dev(bs[s][k]) for k in range(3)]
            loss = ops.nfm_bpr_train_steps(P, Q, bias, N, R, ws, act, *b, b[0].numel(), 0, 1, hp, adam_step0=s).item()
            assert abs(loss - losses[s]) <= 3e-5 * abs(losses[s]), (c, s, loss, losses[s])
            # A Linear bias in front of a BatchNorm has a mathematically zero gradient (the batch mean is removed), and so has the
            # bias (beta) of FM_layers' BatchNorm when a Linear + BatchNorm follows it directly (dropout 0: a constant shift of
            # the Linear's input is a constant shift of its output).  What any implementation computes for those slots is
            # cancellation noise, and Adam turns noise into +-lr steps (different signs here and in the reference).  They are only
            # required to stay within 2.1 lr; everything else must agree.
            noisy = np.zeros(Ns.shape[1], bool)
            if bn and optn == "adam":
                if L >= 1:
                    noisy[F:2 * F] = True                                 # beta of BatchNorm 0
                o = 2 * F
                for _l in range(L):
                    noisy[o + F * F:o + F * F + F] = True                 # Linear bias
                    o += F * F + F + 2 * F
            if optn == "adam":
                # The same holds batch by batch: the bias of a unit that is active for both items of every triple shifts both
                # scores alike, so its gradient is zero.  The reference's sums cancel to exactly 0 there and its Adam leaves
                # the slot where it was; any other summation order leaves noise.
                noisy |= Ns[s + 1] == Ns[s]
            for got, want, nm in ((P, Ps[s + 1], "P"), (Q, Qs[s + 1], "Q"), (bias, Bs[s + 1], "bias"), (N, Ns[s + 1], "N")):
                err = np.abs(got.cpu().numpy() - want)
                tol = (1e-5 if optn == "sgd" else 1e-4) * max(1.0, np.abs(want).max())
                keep = ~noisy if nm == "N" else np.ones(err.shape, bool)
                assert (err[keep] <= tol).mean() >= 0.99 and err.max() <= 2.1 * float(lr) + tol, \
                    (c, s, nm, float((err[keep] <= tol).mean()), float(err.max()))
            if bn:
                np.testing.assert_allclose(R.cpu().numpy(), Rs[s + 1], rtol=2e-5, atol=2e-6, err_msg=f"running stats {c} {s}")
        # eval-mode scores on the reference's final state
        P, Q, bias, N = dev(Ps[-1]), dev(Qs[-1]), dev(Bs[-1]), dev(Ns[-1])
        R = dev(Rs[-1]) if bn else None
        users, cands = g[f"c{c}_users"], g[f"c{c}_cands"].astype(np.int64)
        n, C = cands.shape
        sc = ops.nfm_scores(P, Q, bias, N, R, ws, act, dev(np.repeat(users, C).astype(np.int32)),
                            dev(cands.reshape(-1).astype(np.int32))).view(n, C).contiguous()
        want_sc = np.stack([orc.nfm_scores(Ps[-1], Qs[-1], Bs[-1], Ns[-1], Rs[-1], L, bn, act, np.full(C, u, np.int32),
                                           cands[r].astype(np.int32)) for r, u in enumerate(users)])
        np.testing.assert_allclose(sc.cpu().numpy(), want_sc, rtol=3e-5, atol=3e-6)
        preds = ops.topk_from_scores(sc, dev(cands), 10).cpu().numpy()
        assert (preds == g[f"c{c}_preds"]).mean() >= 0.97, c


def test_nfm_class_drop_in():
    from daisyrec_b200.model import NFM
    from daisyrec_b200.utils.dataset import BasicDataset, CandidatesDataset, get_dataloader
    g = golden("nfm")
    for c in range(int(g["ncases"])):
        L, bn, act, lr, r1, r2, opt = g[f"c{c}_hyper"]
        L, bn, act = int(L), bool(bn), int(act)
        U, F = g[f"c{c}_P"].shape[1:]
        I = g[f"c{c}_Q"].shape[1]
        cfg = dict(gpu="", logger=logging.getLogger("t"), epochs=1, lr=float(lr), reg_1=float(r1), reg_2=float(r2), user_num=U,
                   item_num=I, factors=F, num_layers=L, batch_norm=bn, act_function=ACTS[act], dropout=0.0, loss_type="BPR",
                   optimizer="sgd" if opt == 0 else "adam", init_method="default", early_stop=False, topk=10, progress=False)
        torch.manual_seed(SEEDS[c])
        m = NFM(cfg)
        # the generator spreads the tables by 3x and re-draws the biases; the network block is the constructor's own
        np.testing.assert_allclose(m.embed_user.weight.cpu().numpy() * 3.0, g[f"c{c}_P"][0], rtol=1e-6, atol=0)
        np.testing.assert_allclose(m.embed_item.weight.cpu().numpy() * 3.0, g[f"c{c}_Q"][0], rtol=1e-6, atol=0)
        assert np.array_equal(m.net.cpu().numpy(), g[f"c{c}_N"][0]), c
        if bn:
            assert np.array_equal(m.running.cpu().numpy(), g[f"c{c}_R"][0])
        Bs = g[f"c{c}_bias"]
        m.load_state_dict({"embed_user.weight": g[f"c{c}_P"][0], "embed_item.weight": g[f"c{c}_Q"][0], "u_bias.weight": Bs[0][:U],
                           "i_bias.weight": Bs[0][U:U + I], "bias_": Bs[0][U + I:]})
        b = g[f"c{c}_batches"]
        rows = np.ascontiguousarray(np.concatenate([b[s].T for s in range(3)]).astype(np.int32))
        m.fit(get_dataloader(BasicDataset(rows), batch_size=b.shape[2], shuffle=False))
        want = g[f"c{c}_P"][3]
        err = np.abs(m.embed_user.weight.cpu().numpy() - want)
        tol = (3e-5 if opt == 0 else 3e-4) * max(1.0, np.abs(want).max())
        assert (err <= tol).mean() >= 0.98, (c, float((err <= tol).mean()))
        if bn:
            # a Linear bias in front of a BatchNorm has a mathematically zero gradient; what autograd / the kernels compute
            # for it is cancellation noise, which Adam turns into +-lr steps (in the reference as well, with another sign
            # pattern).  The bias does not change any output, but it shifts the running MEAN of the BatchNorm behind it by
            # momentum x the accumulated bias drift: bounded, not comparable bit for bit.
            # Only the running MEANS of the BatchNorms that follow a Linear are affected (layout: per BatchNorm mean F, var F;
            # BatchNorm 0 follows the bi-interaction, not a Linear); the rest compares as tightly as under SGD.
            got_r, want_r = m.running.cpu().numpy().reshape(-1, 2, F), g[f"c{c}_R"][3].reshape(-1, 2, F)
            loose = np.zeros(got_r.shape, bool)
            if opt != 0:
                loose[1:, 0, :] = True
            np.testing.assert_allclose(got_r[~loose], want_r[~loose], rtol=2e-4, atol=2e-5)
            if loose.any():
                assert np.abs(got_r[loose] - want_r[loose]).max() <= 10 * float(lr), float(np.abs(got_r[loose] - want_r[loose]).max())
        m.load_state_dict({"embed_user.weight": g[f"c{c}_P"][3], "embed_item.weight": g[f"c{c}_Q"][3], "u_bias.weight": Bs[3][:U],
                           "i_bias.weight": Bs[3][U:U + I], "bias_": Bs[3][U + I:], "net": g[f"c{c}_N"][3],
                           "running": g[f"c{c}_R"][3]})
        users, cands = g[f"c{c}_users"], g[f"c{c}_cands"].astype(np.int64)
        loader = get_dataloader(CandidatesDataset([[int(u), cands[r]] for r, u in enumerate(users)]), batch_size=128,
                                shuffle=False)
        preds = m.rank(loader)
        assert preds.dtype == np.float32 and (preds == g[f"c{c}_preds"]).mean() >= 0.97, c
        full = np.stack([m.full_rank(int(u)) for u in users[:4]])
        assert (full == g[f"c{c}_full"]).mean() >= 0.9
        if not bn:
            pp = np.array([m.predict(int(users[q]), int(cands[q][0])) for q in range(4)], np.float32)
            np.testing.assert_allclose(pp, g[f"c{c}_pred_pairs"], rtol=3e-5, atol=3e-6)
        else:
            assert isinstance(m.predict(int(users[0]), int(cands[0][0])), float)      # the reference's predict() cannot run here
        with pytest.raises(ValueError):                                    # nn.Dropout's own range check (dropout > 0 itself runs:
            NFM(dict(cfg, dropout=1.5))                                    # tests/test_gpu_zzz_late.py)
