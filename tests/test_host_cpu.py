"""CPU suite for the host side: the C-ABI library loads and exports every symbol the header declares
(no compute calls without a GPU), host-only entry points (MT19937 seeding / bounded draws) match
numpy, the DataLoader permutation protocol, the init stream, and loud failure without a device.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, golden, csr_from_coo


def test_library_exports_every_header_symbol():
    from daisyrec_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "daisyrec_b200.h")).read()
    declared = set(re.findall(r"\b(drb_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = C.CDLL(_lib.so_path()) if os.path.exists(_lib.so_path()) else _lib.lib()
    for name in declared:
        assert hasattr(L, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert _lib.lib().drb_version() >= 100


def test_host_mt19937_entry_points_match_numpy():
    from daisyrec_b200 import ops
    for seed in (0, 2022, 2 ** 32 - 1):
        st = ops.mt19937_seed(seed)
        assert np.array_equal(st, ops.mt19937_from_numpy(np.random.RandomState(seed)))
    # per-user bounded draws == np.random.choice(arange(n), size=G) user after user
    U, I, G = 40, 50, 4
    rng = np.random.default_rng(1)
    deg = rng.integers(0, 49, size=U)
    row_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int64)
    st = ops.mt19937_seed(5)
    draws = ops.sampler_draw_mt19937(st, row_ptr, U, I, G)
    np.random.seed(5)
    want = np.stack([np.random.choice(np.arange(I - d), size=G) for d in deg])
    assert np.array_equal(draws, want)
    assert np.array_equal(st, ops.mt19937_from_numpy())
    # variable-count form used by build_candidates_set
    n = np.array([7, 1, 1000, 33], np.int64)
    off = np.array([0, 5, 9, 9, 20], np.int64)
    st = ops.mt19937_seed(9)
    d = ops.bounded_draws_mt19937(st, n, off)
    np.random.seed(9)
    want = np.concatenate([np.random.choice(np.arange(n[k]), size=off[k + 1] - off[k]) for k in range(4)])
    assert np.array_equal(d, want)
    with pytest.raises(ValueError):
        ops.sampler_draw_mt19937(ops.mt19937_seed(1), np.array([0, 3], np.int64), 1, 3, 2)


def test_epoch_permutation_is_the_dataloaders():
    from torch.utils.data import DataLoader, TensorDataset
    from daisyrec_b200.model.AbstractRecommender import epoch_permutation
    n = 1000
    ds = TensorDataset(torch.arange(n))
    for shuffle in (True, False):
        torch.manual_seed(3)
        loader = DataLoader(ds, batch_size=64, shuffle=shuffle)
        want = [torch.cat([b[0] for b in loader]) for _ in range(2)]          # two epochs
        torch.manual_seed(3)
        for e in range(2):
            p = epoch_permutation(n, shuffle)
            got = torch.arange(n) if p is None else p
            assert torch.equal(got, want[e])
    g = golden("ml100k_fit")
    torch.set_rng_state(torch.from_numpy(g["torch_state"]))
    assert np.array_equal(epoch_permutation(313452, True).numpy().astype(np.int32), g["perm"])


def test_init_stream_matches_reference():
    from daisyrec_b200.model.AbstractRecommender import _init_table, _INIT
    g = golden("ml100k_fit")
    torch.manual_seed(2022)
    wu, wi = _init_table(943, 32, None), _init_table(1152, 32, None)
    _INIT['normal'](wu); _INIT['normal'](wi)
    assert np.array_equal(wu.numpy(), g["P0"]) and np.array_equal(wi.numpy(), g["Q0"])


def test_csr_from_ur_and_get_ur():
    import pandas as pd
    from daisyrec_b200.utils.sampler import csr_from_ur
    from daisyrec_b200.utils.utils import get_ur
    rng = np.random.default_rng(0)
    df = pd.DataFrame({"user": rng.integers(30, size=400), "item": rng.integers(50, size=400)})
    ur = get_ur(df)
    ref = {}
    for u, i in zip(df["user"], df["item"]):
        ref.setdefault(int(u), set()).add(int(i))
    assert dict(ur) == ref and list(ur.keys()) == list(ref.keys())
    # list(set) order feeds build_candidates_set (utils.py:72-80): same insertions => same iteration order as the reference
    assert all(list(ur[u]) == list(ref[u]) for u in ref)
    row_ptr, col = csr_from_ur(ur, 30)
    rp2, col2 = csr_from_coo(df["user"].values.astype(np.int32), df["item"].values.astype(np.int32), 30)
    assert np.array_equal(row_ptr, rp2) and np.array_equal(col, col2)


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_silent_cpu_fallback():
    import logging
    from daisyrec_b200.model.MFRecommender import MF
    cfg = dict(gpu='', logger=logging.getLogger(), lr=.01, reg_1=0, reg_2=0, epochs=1, topk=5, user_num=4, item_num=4,
               factors=8, loss_type='BPR', optimizer='default', init_method='default', early_stop=False)
    with pytest.raises(RuntimeError):
        MF(cfg)


def test_synthetic_generator_shape():
    from daisyrec_b200.utils.synthetic import make_interactions
    d = make_interactions(2000, 1500, 60000, seed=1)
    assert d["nnz"] == 60000 == int(d["row_ptr"][-1])
    key = d["coo_u"].to(torch.int64) * 1500 + d["coo_i"]
    assert torch.unique(key).numel() == 60000                         # unique pairs
    deg = d["row_ptr"][1:] - d["row_ptr"][:-1]
    assert int(deg.min()) >= 1


def test_loader_plan_decoding():
    """fit() takes the bulk path only for the reference's own loader shape; anything else is iterated batch by batch."""
    from torch.utils.data import DataLoader, RandomSampler, WeightedRandomSampler
    from daisyrec_b200.model.AbstractRecommender import loader_plan
    from daisyrec_b200.utils.dataset import BasicDataset, get_dataloader
    data = np.arange(30, dtype=np.int32).reshape(10, 3)
    plan = loader_plan(get_dataloader(BasicDataset(data), batch_size=4, shuffle=True, num_workers=4))
    assert plan is not None and plan[0] is data and plan[1:4] == (4, True, False)
    plan = loader_plan(DataLoader(BasicDataset(data), batch_size=3, shuffle=False, drop_last=True))
    assert plan[1:4] == (3, False, True)
    g = torch.Generator(); g.manual_seed(1)
    assert loader_plan(DataLoader(BasicDataset(data), batch_size=4, sampler=RandomSampler(data, generator=g))) is None
    assert loader_plan(DataLoader(BasicDataset(data), batch_size=4, sampler=WeightedRandomSampler([1.0] * 10, 10))) is None
    assert loader_plan(DataLoader(BasicDataset(data[:, :2]), batch_size=4)) is None           # not <u,i,j> rows
    assert loader_plan([[torch.zeros(4), torch.zeros(4), torch.zeros(4)]]) is None            # plain list of batches
    # the DataLoader and the plan consume the global RNG identically: same first batch
    from daisyrec_b200.model.AbstractRecommender import epoch_permutation
    torch.manual_seed(7)
    first = next(iter(get_dataloader(BasicDataset(data), batch_size=4, shuffle=True)))
    torch.manual_seed(7)
    perm = epoch_permutation(10, True)
    assert [int(x) for x in first[0]] == data[perm[:4].numpy(), 0].tolist()


def test_host_mixed_draws_replay_reference_fixture():
    """drb_sampler_draw_mt19937_mixed (host part of the 'low-pop' / 'high-pop' branch, sampler.py:64-81): ranks and
    doubles off numpy's stream; the device lookups are restated with numpy here (setdiff1d / searchsorted)."""
    import pandas as pd
    from daisyrec_b200 import ops
    from daisyrec_b200.utils.sampler import BasicNegtiveSampler, csr_from_ur
    from daisyrec_b200.utils.utils import get_ur
    g = golden("sampler_pop")
    for c in range(int(g["ncases"])):
        method, loss = str(g[f"c{c}_method"]), str(g[f"c{c}_loss"])
        if method == "uniform" or loss != "BPR":
            continue
        U, I, G, seed = (int(v) for v in g[f"c{c}_meta"])
        df = pd.DataFrame({"user": g[f"c{c}_coo_u"], "item": g[f"c{c}_coo_i"], "rating": g[f"c{c}_rating"]})
        ur = get_ur(df)
        cfg = dict(UID_NAME='user', IID_NAME='item', INTER_NAME='rating', user_num=U, item_num=I, num_ng=G,
                   sample_method=method, sample_ratio=float(g[f"c{c}_ratio"]), loss_type=loss, train_ur=ur)
        smp = BasicNegtiveSampler(df, cfg)
        assert np.array_equal(smp.pop_prob, g[f"c{c}_pop_prob"])
        other = int(float(g[f"c{c}_ratio"]) * G)
        row_ptr, col = csr_from_ur(ur, U)
        st = ops.mt19937_seed(seed)
        draws, u01 = ops.sampler_draw_mt19937_mixed(st, row_ptr, U, I, G - other, other)
        cdf = smp.pop_prob.cumsum()
        cdf /= cdf[-1]
        js = np.zeros((U, G), np.int32)
        for u in range(U):
            comp = np.setdiff1d(np.arange(I), col[row_ptr[u]:row_ptr[u + 1]])
            js[u, :G - other] = comp[draws[u]]
            js[u, G - other:] = cdf.searchsorted(u01[u], side='right')
        rows = g[f"c{c}_rows"]
        assert np.array_equal(js[rows[:, 0], np.tile(np.arange(G), len(rows) // G)], rows[:, 2])
        ops.mt19937_to_numpy(st)
        assert np.array_equal(np.random.randint(0, 2 ** 31 - 1, size=3), g[f"c{c}_next"])


def test_metrics_mirror_host_logic():
    from daisyrec_b200.utils.metrics import ground_truth_csr, calc_ranking_results, Metric, metrics_name_config
    test_ur = {7: {5, 1, 9}, 3: {2}, 11: set()}
    ptr, idx = ground_truth_csr(test_ur, [3, 7, 11])
    assert ptr.tolist() == [0, 1, 4, 4] and idx.tolist() == [2, 1, 5, 9] and idx.dtype == np.int32
    assert metrics_name_config["hit"] == 'Hit Ratio'
    import logging, tempfile
    cfg = dict(logger=logging.getLogger("t"), res_path=tempfile.mkdtemp() + "/", item_num=10, topk=5)
    with pytest.raises(KeyError):                                      # 'map' has no display name (metrics.py:5-16,38)
        calc_ranking_results(test_ur, np.zeros((3, 5), np.float32), [3, 7, 11], dict(cfg, metrics=["map"]))
    with pytest.raises(ValueError):                                    # 'f1' / 'auc' are unreachable (metrics.py:87-92)
        Metric(dict(cfg, metrics=["f1"])).run(test_ur, np.zeros((3, 5), np.float32), [3, 7, 11])
    if not torch.cuda.is_available():                                  # CPU-only behaviour: no CPU fallback for the KPIs either
        with pytest.raises(RuntimeError):
            Metric(dict(cfg, metrics=["recall"])).run(test_ur, np.zeros((3, 5), np.float32), [3, 7, 11])


def test_optimizer_names_mirror():
    from daisyrec_b200.model.MFRecommender import MF
    from daisyrec_b200.model.AbstractRecommender import GeneralRecommender
    assert MF.SUPPORTED_OPTIMIZERS == ('sgd', 'adam', 'adagrad', 'rmsprop') and GeneralRecommender.SUPPORTED_OPTIMIZERS == ('sgd', 'adam')
    m = MF.__new__(MF)
    m.logger = None
    for name, want in (('adagrad', 'adagrad'), ('RMSprop', 'rmsprop'), ('nonsense', 'adam')):
        m.optimizer = name
        assert m._optimizer_name() == want
    m.optimizer = 'sparse_adam'
    with pytest.raises(RuntimeError):
        m._optimizer_name()


def test_device_twin_is_dropped_after_an_in_place_edit():
    """fit() trusts the sampler's device twin only while the host rows still carry the stamp taken at attach time."""
    from daisyrec_b200.utils.sampler import TripleArray, fingerprint
    from daisyrec_b200.model.AbstractRecommender import GeneralRecommender
    rows = np.arange(3 * 5000, dtype=np.int32).reshape(-1, 3)
    twin = torch.from_numpy(rows.copy())                               # stands in for the CUDA tensor
    arr = TripleArray.attach(rows, twin)
    assert isinstance(arr, TripleArray) and arr._drb_device is twin and arr._drb_stamp == fingerprint(rows)
    assert arr[10:20]._drb_device is None and arr.copy()._drb_device is None        # views / copies forget the twin
    m = GeneralRecommender.__new__(GeneralRecommender)
    m.device = torch.device('cpu')
    assert m._device_triples(arr) is twin                                           # untouched -> the twin itself
    np.random.default_rng(0).shuffle(arr)                                           # in-place row shuffle
    up = m._device_triples(arr)
    assert up is not twin and np.array_equal(up.numpy(), np.asarray(arr))           # re-uploaded from the edited rows
    assert m._device_triples(arr) is up                                             # cached per (array, stamp)
    arr[::7, 2] += 1
    assert np.array_equal(m._device_triples(arr).numpy(), np.asarray(arr))
    plain = np.asarray(arr).copy()
    plain.flags.writeable = False                                                   # pandas >= 3 hands out read-only views
    assert np.array_equal(m._device_triples(plain).numpy(), plain)
    empty = np.zeros((0, 3), np.int32)
    assert fingerprint(empty)[0] == (0, 3) and m._device_triples(empty).shape == (0, 3)


def test_fingerprint_sees_every_column():
    """A stride that is a multiple of 3 would sample one column of the [T,3] rows only (T = 65536*k hits it)."""
    from daisyrec_b200.utils.sampler import fingerprint
    rows = np.zeros((65536 * 3, 3), np.int32)
    base = fingerprint(rows)
    for col in range(3):
        edited = rows.copy()
        edited[5:-5, col] += 1                                            # leave the end rows (stamped separately) alone
        assert fingerprint(edited) != base, col


def test_epoch_seed_and_permutation_follow_the_dataloader():
    """epoch_seed + epoch_permutation consume the global RNG exactly as iterating DataLoader(shuffle=True) does."""
    from torch.utils.data import DataLoader, TensorDataset
    from daisyrec_b200.model.AbstractRecommender import epoch_permutation, epoch_seed
    n = 1000
    torch.manual_seed(7)
    order = torch.cat([b[0] for b in DataLoader(TensorDataset(torch.arange(n)), batch_size=64, shuffle=True)])
    after = torch.get_rng_state()
    torch.manual_seed(7)
    assert torch.equal(epoch_permutation(n, True, seed=epoch_seed(True)), order)
    assert torch.equal(torch.get_rng_state(), after)
    torch.manual_seed(7)
    assert torch.equal(epoch_permutation(n, True), order)


def test_reference_arm_times_the_installed_reference(tmp_path):
    """bench.py --impl reference runs the REAL daisy MF.fit (oracle/_ref) over its own DataLoader; config is the own arm's."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    sys.path.insert(0, ROOT)
    import bench
    if bench.reference_root() is None:
        pytest.skip("oracle/_ref not installed (no /root/reference in this container)")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--shape", "tiny", "--batch",
                        "2048", "--steps", "3", "--warmup", "1", "--quick"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "reference" and line["value"] > 0
    assert line["steps"] == 3 and line["gpu_launches"] == 0
    ns = type("A", (), dict(shape="tiny", num_ng=4, factors=64, batch=2048))
    assert line["config"] == bench.workload_config(ns, 1)                  # same_config with the own arm


def test_step_kernel_geometry_and_tiles():
    """Host logic of the step-kernel launcher: the lean instantiation's lane geometry (W lanes x NCH chunks of 4 floats cover the
    row, W a power of two <= 32, 8 lanes = one 128-byte line per access where the row is long enough) and the equal-tile choice."""
    import ctypes as C
    from daisyrec_b200 import _lib as L
    lib = L.lib()
    w, n, t = C.c_int32(), C.c_int32(), C.c_int32()
    for F in range(4, 516, 4):
        rc = lib.drb_mf_step_geometry(F, 1, C.byref(w), C.byref(n), 3543, C.byref(t))
        if rc != 0:                                            # rows the lean body has no geometry for take the general kernel
            ch = F // 4
            assert ch > 32 and not any(ch % k == 0 and (ch // k) & (ch // k - 1) == 0 and ch // k <= 32 for k in (4, 2, 1)), F
            continue
        W, N = w.value, n.value
        assert W in (1, 2, 4, 8, 16, 32) and N in (1, 2, 4) and W * N * 4 >= F, (F, W, N)
        if N > 1:
            assert W >= 8, (F, W, N)                           # a group's 128-bit access covers whole 128-byte lines
    for F, want in ((16, (4, 1)), (32, (8, 1)), (64, (8, 2)), (128, (8, 4)), (256, (16, 4)), (100, (32, 1)), (48, (16, 1))):
        assert lib.drb_mf_step_geometry(F, 1, C.byref(w), C.byref(n), 3543, C.byref(t)) == 0 and (w.value, n.value) == want, F
        assert t.value == 512
    assert lib.drb_mf_step_geometry(64, 0, C.byref(w), C.byref(n), 3543, C.byref(t)) == 0 and (w.value, n.value) == (16, 1)
    assert lib.drb_mf_step_geometry(6, 1, C.byref(w), C.byref(n), 1, C.byref(t)) != 0          # not a multiple of 4: general kernel
    for per_cta, want in ((1, 16), (16, 16), (17, 32), (512, 512), (513, 272), (3543, 512), (1024, 512), (1025, 352)):
        lib.drb_mf_step_geometry(64, 1, None, None, per_cta, C.byref(t))
        assert t.value == want, (per_cta, t.value, want)
        k = -(-per_cta // t.value)
        assert t.value % 16 == 0 and k * t.value >= per_cta and (k - 1) * t.value < per_cta


def test_mt19937_jump_table_matches_numpy():
    """csrc/mt_jump_table.inc (scripts/gen_mt_jump.py): g_m(x) = x^(1680 * 624 * 2^m) mod phi(x).  The Horner walk the segmented
    kernel runs, restated on the host, must land on numpy's MT19937 state that many words ahead (levels 0 and 2 here; the
    generator script checks all eight), and every level must be the square of the one below modulo the same phi -- checked
    through the states: two jumps of level m == one jump of level m + 1."""
    import os
    import re
    from daisyrec_b200 import _build
    src = open(os.path.join(_build.CSRC, "mt_jump_table.inc")).read()
    seg_blocks = int(re.search(r"kMtSegBlocks = (\d+)", src).group(1))
    rows = re.findall(r"\{((?:0x[0-9a-f]{16}ull(?:, )?)+)\}", src)
    assert seg_blocks == 1680 and len(rows) == 8
    polys = []
    for r in rows:
        words = [int(w[:-3], 16) for w in r.split(", ")]
        assert len(words) == 312
        polys.append(sum(w << (64 * k) for k, w in enumerate(words)))
    UPPER, LOWER, MAG = 0x80000000, 0x7FFFFFFF, 0x9908B0DF

    def jump(g, s):
        s = [int(v) for v in s]
        h, p = list(s), 0
        for i in range(g.bit_length() - 2, -1, -1):
            y = (h[p] & UPPER) | (h[(p + 1) % 624] & LOWER)
            h[p] = h[(p + 397) % 624] ^ (y >> 1) ^ (MAG if y & 1 else 0)
            p = (p + 1) % 624
            if (g >> i) & 1:
                for j in range(624):
                    h[(p + j) % 624] ^= s[j]
        return np.array([h[(p + j) % 624] for j in range(624)], dtype=np.uint32)

    def same(a, b):                                   # word 0 of a block state: only its top bit is ever read again
        return (int(a[0]) ^ int(b[0])) & UPPER == 0 and np.array_equal(a[1:], b[1:])

    for m in (0, 2):
        rs = np.random.RandomState(77 + m)
        s0 = rs.get_state()[1].copy()
        rs.bytes(4 * seg_blocks * 624 * (1 << m))
        assert same(jump(polys[m], s0), rs.get_state()[1]), m
    s0 = np.random.RandomState(5).get_state()[1].copy()
    for m in (3, 6):
        assert same(jump(polys[m + 1], s0), jump(polys[m], jump(polys[m], s0))), m
