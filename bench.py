#!/usr/bin/env python
"""bench.py -- BPR training throughput on the BASELINE.json workloads (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--shape ml-20m] [--configs LIST]
                    [--dump-outputs DIR]

One "step" = one synchronous BPR-MF training step over one batch of ``--batch`` triples (u,i,j) per GPU
(the reference's zero_grad + calc_loss + backward + optimizer.step, AbstractRecommender.py:119-128).
Headline workload: BASELINE.json configs[1] -- MF + BPR, synthetic ML-20M shape (138,493 x 26,744, 20 M interactions,
num_ng=4 -> 80 M triples/epoch), factors=64, fp32, SGD lr .01, reg .001/.001.  Metric: BPR user-item pairs
(= training triples) per second, whole job.

Own arm
  value      K steps timed with CUDA events around the persistent step-kernel launches; index planes and tables resident
             in HBM (N > 1: per-GPU batch fixed, user-row-sharded P, replicated Q; max over ranks).
  e2e        the reference's plug-in call, wall clock: MF(cfg).fit(get_dataloader(BasicDataset(host_triples), B,
             shuffle=True)) for one full epoch from PINNED host triples -- upload, epoch permutation, gather, every step,
             loss read-back -- median of 3, for both shuffle engines (N > 1: the native sharded step loop fed from pinned
             host shares, H2D per step + loss D2H per step).  `fit_host_batches` (per-step H2D / D2H) is kept beside it.
  roofline   algorithmic bytes (24*F+12 per triple, SURVEY 8(d)) / event-timed launch duration vs MEASURED_PEAKS.json.
  configs    driver-visible lines for the other BASELINE configs and the kernels either side of the step: C3 NeuMF bf16
             tower, C4 LightGCN L=3, C5 shape on one GPU (and row-sharded when N > 1), rank / full_rank / KPIs / sampling /
             epoch permutation, and one step-time line each for FM, NFM, NGCF (SURVEY 8(f) ranks 3-4).
  parity_check (N > 1)  3 global steps on a 48 K-triple slice: sharded run vs the single-GPU kernel on the same batches.
  cpu_baseline  the REAL reference (oracle/_ref = /root/reference installed unmodified, oracle/build_ref.py) running
             daisy.model.MFRecommender.MF.fit over its own DataLoader on this host's cores, bounded sample, in a
             subprocess with the GPUs hidden.
Reference arm (--impl reference): the same real-reference run for K steps after W warm-up steps (rank 0 only).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bpr_train_triples_per_sec"
UNIT = "triples/s"
HYPER = dict(lr=0.01, reg_1=0.001, reg_2=0.001)


# ------------------------------------------------------------------------------- helpers
def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


class ClockSampler:
    """nvidia-smi sampler running beside the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.rows, self.proc, self.thr = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(dev)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._pump, daemon=True)
            self.thr.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons, n = [], None, set(), 0
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mxc = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= ts <= t1 + 0.05:
                n += 1
                sm.append(clk)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:                                      # region shorter than the sampling period
            sm = [float(x.split(",")[1]) for _, x in self.rows[-3:] if len(x.split(",")) > 2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples_in_region": n}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def profiled_traffic(factors, batch):
    """dram bytes per STEP from the committed ncu capture (profiles/traffic.json), else None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            t = json.load(open(p))
            if t.get("factors") == factors and t.get("batch") == batch:
                return t.get("dram_bytes_per_step"), t.get("source", "profiles/traffic.json")
        except Exception:  # noqa: BLE001
            pass
    return None, None


def build_workload(shape, device, num_ng, seed, sampler):
    """Synthetic interactions -> (data dict, triples int32 [T,3] on `device`).  sampler: 'cuda' | 'oracle'."""
    from daisyrec_b200.utils.synthetic import SHAPES, make_interactions
    U, I, nnz = SHAPES[shape]
    d = make_interactions(U, I, nnz, seed=seed, device=device)
    row_ptr_h = d["row_ptr"].cpu().numpy()
    if sampler == "cuda":
        from daisyrec_b200 import ops
        st = ops.mt19937_seed(seed)
        draws = ops.sampler_draw_mt19937(st, row_ptr_h, U, I, num_ng)
        js = ops.sampler_kth_complement(d["row_ptr"], d["col"], torch.from_numpy(draws).to(device), I)
        triples = ops.sampler_explode(d["coo_u"], d["coo_i"], js)
    else:
        from oracle import oracle as orc
        js = orc.sample_negatives(orc.mt_seed(seed), row_ptr_h, d["col"].cpu().numpy(), U, I, num_ng)
        triples = torch.from_numpy(orc.explode_triples(d["coo_u"].cpu().numpy(), d["coo_i"].cpu().numpy(), js))
    return d, triples


def workload_config(args, world):
    """The workload both arms are measured on (identical dict in the own and the reference arm)."""
    from daisyrec_b200.utils.synthetic import SHAPES
    U, I, nnz = SHAPES[args.shape]
    T = nnz * args.num_ng
    return {"workload": f"MF+BPR synthetic {args.shape} shape ({U}x{I}, nnz={nnz}, num_ng={args.num_ng} -> {T} "
                        f"triples/epoch), factors={args.factors}, SGD lr=0.01 reg=0.001/0.001",
            "batch_size": args.batch, "global_batch": args.batch * world, "factors": args.factors,
            "triples_per_epoch": T, "optimizer": "sgd",
            "parallelism": "single GPU" if world == 1 else f"user-row-sharded P x{world}, replicated Q",
            "l2": "index planes (12 B/triple, all K steps) exceed L2 and are streamed once; the factor tables "
                  "(42 MB at F=64) are persistent model state reused by every step and stay L2-resident by design"}


def timed_ms(fn, warm, reps):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


DUMP_BYTES = 64 << 20


def timed_outputs(tensors, seed=0):
    """Host copies of what the timed path returned, for --dump-outputs (float32 / float64 as computed).  When they exceed
    DUMP_BYTES in all, every 2-D table keeps the same fraction of its rows, drawn with a fixed seed: the same rows in every
    run with the same arguments."""
    total = sum(t.numel() * t.element_size() for t in tensors.values())
    tables = sum(t.numel() * t.element_size() for t in tensors.values() if t.dim() == 2)
    keep = 1.0 if total <= DUMP_BYTES else (DUMP_BYTES - (total - tables)) / tables
    rng = np.random.default_rng(seed)
    out = {}
    for name, t in tensors.items():
        if t.dim() == 2 and keep < 1.0:
            rows = np.sort(rng.choice(t.shape[0], max(1, int(t.shape[0] * keep)), replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        out[name] = t.detach().cpu().numpy()
    return out


def mf_config(U, I, F, **kw):
    import logging
    cfg = dict(gpu="", logger=logging.getLogger("bench"), epochs=1, topk=50, user_num=U, item_num=I, factors=F,
               loss_type="BPR", optimizer="default", init_method="default", early_stop=False, progress=False, **HYPER)
    cfg.update(kw)
    return cfg


# ------------------------------------------------------------------------------- reference arm (real daisyRec on the CPU)
class TimedLoader:
    """Pass-through around the reference's own DataLoader that notes when batch `warmup` is requested (= the moment the
    step before it finished) and when the epoch ends: the K steps in between run inside the reference's fit() loop
    untouched (tqdm, zero_grad, calc_loss, isnan, backward, optimizer.step, loss.item(); AbstractRecommender.py:112-128)."""

    def __init__(self, loader, warmup):
        self.loader, self.warmup = loader, warmup
        self.t0 = self.t1 = None
        self.steps = 0

    def __len__(self):
        return len(self.loader)

    def __iter__(self):
        k = 0
        it = iter(self.loader)
        while True:
            if k == self.warmup:
                self.t0 = time.perf_counter()
            try:
                b = next(it)
            except StopIteration:
                self.t1 = time.perf_counter()
                self.steps = k - self.warmup
                return
            k += 1
            yield b


def reference_root():
    p = os.path.join(ROOT, "oracle", "_ref")
    return p if os.path.isfile(os.path.join(p, "daisy", "model", "MFRecommender.py")) else None


def reference_fit(rows, U, I, F, batch, warmup, steps, num_workers, seed):
    batch = min(batch, max(256, rows.shape[0] // max(1, warmup + steps)))
    """daisy.model.MFRecommender.MF(config).fit(get_dataloader(BasicDataset(rows), batch, shuffle=True, num_workers)) on the
    CPU; rows = (warmup+steps)*batch sampler triples.  -> (seconds for the `steps` timed steps, steps)."""
    from oracle import ref_harness as RH
    RH.use_root(reference_root())
    RH.import_reference()
    from daisy.model.MFRecommender import MF
    from daisy.utils.dataset import BasicDataset, get_dataloader
    cfg = RH.make_config("mf", factors=F, epochs=1, batch_size=batch, user_num=U, item_num=I, **HYPER)
    RH.seed_everything(seed)
    model = MF(cfg)
    assert model.device == "cpu", "the reference arm must run with the GPUs hidden"
    n = (warmup + steps) * batch
    loader = get_dataloader(BasicDataset(rows[:n]), batch_size=batch, shuffle=True, num_workers=num_workers)
    tl = TimedLoader(loader, warmup)
    model.fit(tl)
    return tl.t1 - tl.t0, tl.steps


def reference_rows(args, n_rows):
    """First n_rows triples of one seeded epoch permutation of the workload (CPU only)."""
    if args.rows_file:
        rows = np.load(args.rows_file)
    else:
        d, triples = build_workload(args.shape, "cpu", args.num_ng, args.seed, "oracle")
        g = torch.Generator()
        g.manual_seed(args.seed)
        perm = torch.randperm(triples.shape[0], generator=g)[:n_rows]
        rows = triples[perm].numpy()
    if rows.shape[0] < n_rows:                                       # wrap (more steps than the sample holds)
        rows = np.concatenate([rows] * ((n_rows + rows.shape[0] - 1) // rows.shape[0]))
    return np.ascontiguousarray(rows[:n_rows], dtype=np.int32)


def run_reference(args):
    rank, local, world = dist_env()
    if rank != 0:
        return 0
    os.environ["CUDA_VISIBLE_DEVICES"] = ""            # before any CUDA call: the reference picks 'cuda' when it sees one
    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    from daisyrec_b200.utils.synthetic import SHAPES
    U, I, _ = SHAPES[args.shape]
    world = max(world, args.gpus)
    cfg = workload_config(args, world)
    if reference_root() is None:
        return run_reference_port(args, cfg, cores)
    W, K, F = args.warmup, args.steps, args.factors
    Bg = args.batch * world                                           # the own arm's global step
    rows = reference_rows(args, (W + K) * min(Bg, 4 << 20))            # larger global batches get a shrunk sample anyway
    # calibrate with ONE step (at most 1 M triples, scaled linearly); shrink the per-step sample only if K+W steps of the own
    # arm's global batch would not fit the time budget.  --quick: the caller sized the sample, no calibration.
    batch = Bg
    if not args.quick:
        Bc = min(Bg, 1 << 20)
        dt1, _ = reference_fit(rows, U, I, F, Bc, 0, 1, 0, args.seed)
        per_step = dt1 * Bg / Bc
        if per_step * (W + K) > args.ref_budget:
            batch = max(256, int(Bg * args.ref_budget / (per_step * (W + K))) // 256 * 256)
    dt, done = reference_fit(rows, U, I, F, batch, W, K, args.ref_workers, args.seed)
    value = done * batch / dt
    extra = {}
    if not args.quick:
        d0, k0 = reference_fit(rows, U, I, F, batch, 1, 2, 0, args.seed)
        extra["num_workers_0"] = {"value": k0 * batch / d0, "steps": k0, "batch": batch}
        db, kb = reference_fit(rows, U, I, F, 256, 20, 200, args.ref_workers, args.seed)
        extra["batch_256"] = {"value": kb * 256 / db, "steps": kb, "batch": 256, "ms_per_step": db / kb * 1e3,
                              "note": "the reference's default batch_size (assets/basic.yaml)"}
    sample = (f"{done} steps x {batch} triples after {W} warm-up steps inside daisy.model.MFRecommender.MF.fit over "
              f"get_dataloader(BasicDataset, batch_size={batch}, shuffle=True, num_workers={args.ref_workers}) "
              f"(own arm global batch {Bg}{'' if batch == Bg else ', per-step sample shrunk to fit the time budget'}); "
              f"unmodified reference installed in oracle/_ref, torch {torch.__version__} CPU, {cores} threads")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
            "warmup": W, "ms_per_step": dt / max(1, done) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample, **extra},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def run_reference_port(args, cfg, cores):
    """oracle/_ref missing (the recipe never ran where /root/reference exists): time the pinned PyTorch-CPU port."""
    from daisyrec_b200.utils.synthetic import SHAPES, init_tables
    from oracle.torch_port import TorchMFBaseline
    U, I, _ = SHAPES[args.shape]
    W, K, B = args.warmup, args.steps, args.batch
    rows = torch.from_numpy(reference_rows(args, (W + K) * B)).to(torch.int64)
    P0, Q0 = init_tables(U, I, args.factors, args.seed, "cpu")
    m = TorchMFBaseline(P0, Q0, optimizer="sgd", **HYPER)

    def step(s):
        r = rows[s * B:(s + 1) * B]
        return m.step(r[:, 0].contiguous(), r[:, 1].contiguous(), r[:, 2].contiguous())

    for s in range(W):
        step(s)
    t0 = time.perf_counter()
    for s in range(K):
        step(W + s)
    dt = time.perf_counter() - t0
    value = K * B / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
            "warmup": W, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{K} steps x {B} triples, oracle/torch_port.py (oracle/_ref absent)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def cpu_baseline_subprocess(args, rows, steps=2, warmup=1):
    """The reference arm on a bounded sample, GPUs hidden, in a child process -> its cpu_baseline dict."""
    with tempfile.TemporaryDirectory(prefix="drb_bench_") as tmp:
        f = os.path.join(tmp, "rows.npy")
        np.save(f, rows)
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--quick", "--rows-file", f,
               "--steps", str(steps), "--warmup", str(warmup), "--batch", str(args.batch), "--factors", str(args.factors),
               "--shape", args.shape, "--ref-budget", str(args.cpu_budget), "--gpus", "1"]
        try:
            r = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                               timeout=max(120.0, 6 * args.cpu_budget))
            for ln in reversed(r.stdout.strip().splitlines()):
                if ln.startswith("{"):
                    return json.loads(ln)["cpu_baseline"]
            return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference",
                    "sample": f"failed rc={r.returncode}: {r.stderr.strip()[-300:]}"}
        except Exception as e:  # noqa: BLE001
            return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {e!r}"}


# ------------------------------------------------------------------------------- secondary configs (driver-visible)
def step_kernel_info(F, table_rows=0):
    """Which instantiation of the step kernel the timed steps ran (a lean one only after its on-device selection)."""
    try:
        from daisyrec_b200 import ops
        lean, lanes, chunks = ops.mf_step_variant(F, table_rows)
        ms_gen, ms_lean, tile_cap = ops.mf_step_selfcheck_ms(F, table_rows)
    except Exception as e:  # noqa: BLE001  (reporting only: never let it cost the line)
        return {"instantiation": "mf_bpr_steps_kernel", "error": repr(e)}
    return {"instantiation": "mf_bpr_steps_lean_kernel" if lean else "mf_bpr_steps_kernel", "lanes_per_row": lanes,
            "chunks_per_lane": chunks,
            "index_tile_cap": tile_cap,
            "selection": "on-device, once per process: every lean candidate geometry must equal the general instantiation on a "
                         "seeded problem (loss 1e-5 rel, tables 1e-5 abs); candidates and the general kernel are timed on 3 steps "
                         "x 524 288 triples; the fastest correct candidate runs only if it beats the general one",
            "selection_ms": {"general": ms_gen, "best_lean": ms_lean}}


def roof(achieved_gbs, kernel, alg_bytes, note=None):
    peak, src = measured_peaks()
    r = {"bound": "hbm", "achieved": achieved_gbs, "peak": peak, "unit": "GB/s", "frac": achieved_gbs / peak,
         "kernel": kernel, "algorithmic_bytes": alg_bytes, "peak_source": src}
    if note:
        r["note"] = note
    return r


def cfg_c3_neumf(args, dev, d, planes):
    """BASELINE config 3: NeuMF + BPR, ML-20M shape, F=32, tower 128->64->32, Adam, bf16 tcgen05 tower."""
    from daisyrec_b200 import ops
    U, I = d["user_num"], d["item_num"]
    F, L, B = 32, 2, args.batch
    D = F * 2 ** (L - 1)
    g = torch.Generator(device=dev); g.manual_seed(11)
    tabs = [(torch.randn(s, device=dev, generator=g) * 0.05).contiguous() for s in ((U, F), (I, F), (U, D), (I, D))]
    W = (torch.randn(ops.neumf_param_count(F, L), device=dev, generator=g) * 0.1).contiguous()
    hp = ops.hyper(0.001, 0.001, 0.001, "adam")
    bu, bi, bj = (p_[:4 * B] for p_ in planes)
    out = {}
    for name, td in (("fused", 2), ("bf16", 1), ("fp32", 0)):
        ws = ops.NeumfWorkspace(U, I, F, L, "adam", 2 * B, dev)
        step = [0]

        def fn():
            ops.neumf_bpr_train_steps(tabs, W, ws, bu, bi, bj, B, step[0] % 4, 1, hp, adam_step0=step[0], check=False,
                                      tower_dtype=td)
            step[0] += 1
        ms = timed_ms(fn, 3, 8 if td else 4)
        bpt = 3 * (F + D) * 4 * 2 + 12
        kern = {2: "neumf_fused_kernel (gather + tower fwd/bwd + head + scatter in one CTA per tile) + table sweeps",
                1: "layer-wise tcgen05 GEMMs + head + table sweeps", 0: "layer-wise fp32 GEMMs + head + table sweeps"}[td]
        out[name] = {"value": B / ms * 1e3, "unit": UNIT, "ms_per_step": ms, "batch": B,
                     "roofline": roof(B * bpt / ms / 1e6, kern, bpt)}
        del ws
    res = out["fused"]
    res["workload"] = (f"NeuMF+BPR synthetic ml-20m shape, factors={F}, num_layers={L} (tower {2*D}->{D}->{F}), Adam, bf16 tcgen05 "
                       "tower fused per 64-triple tile (activations in shared / tensor memory)")
    res["layerwise_bf16_tower"] = out["bf16"]
    res["fp32_tower"] = out["fp32"]
    return res


def cfg_c4_lightgcn(args, dev):
    """BASELINE config 4: LightGCN L=3 + BPR, Amazon-Book shape, F=64, Adam."""
    from daisyrec_b200 import ops
    from daisyrec_b200.utils.synthetic import SHAPES, make_interactions
    U, I, nnz = SHAPES["amazon-book"]
    F, L = 64, 3
    d = make_interactions(U, I, nnz, seed=args.seed, device=dev)
    adj = ops.lgcn_build_adj(d["coo_u"], d["coo_i"], U, I)
    graph = ops.LgcnGraph(*adj, dev)
    nnzA = int(adj[1].numel())
    g = torch.Generator(device=dev); g.manual_seed(7)
    E0 = (torch.randn(U + I, F, device=dev, generator=g) * 0.05).contiguous()
    hp = ops.hyper(0.01, 0.0, 0.0, "adam")
    out = {"workload": f"LightGCN+BPR synthetic amazon-book shape ({U}x{I}, nnz={d['nnz']}), factors={F}, num_layers={L}, Adam",
           "spmm_segments": graph.nseg, "adjacency_nnz": nnzA}
    for B in (65536, 1 << 20):
        idx = torch.randint(0, d["coo_u"].numel(), (4 * B,), device=dev, generator=g)
        bu, bi = d["coo_u"][idx].contiguous(), d["coo_i"][idx].contiguous()
        bj = torch.randint(0, I, (4 * B,), device=dev, dtype=torch.int32, generator=g)
        ws = ops.LgcnWorkspace(U, I, F, "adam", dev)
        step = [0]

        def fn():
            ops.lgcn_bpr_train_steps(E0, ws, graph, L, bu, bi, bj, B, step[0] % 4, 1, hp, adam_step0=step[0], check=False)
            step[0] += 1
        ms = timed_ms(fn, 3, 10)
        alg = 2 * L * (nnzA * (8 + 4 * F) + (U + I) * 4 * F) + B * (24 * F + 12)
        out[f"batch_{B}"] = {"value": B / ms * 1e3, "unit": UNIT, "ms_per_step": ms, "batch": B,
                             "roofline": roof(alg / ms / 1e6, "spmm_seg_kernel x 2L + BPR phases + Adam sweep (per step)", alg,
                                              "upper-bound algorithmic bytes: neighbour-row gathers are mostly L2 hits")}
        del ws
    out["value"], out["unit"], out["ms_per_step"] = out["batch_65536"]["value"], UNIT, out["batch_65536"]["ms_per_step"]
    return out


def cfg_c5_single(args, dev, steps=24):
    """BASELINE config 5's shape on ONE GPU: MF + BPR, Netflix shape, F=128 -- tables (255 MB) >> L2: the HBM regime."""
    from daisyrec_b200 import ops
    from daisyrec_b200.utils.synthetic import init_tables
    a5 = argparse.Namespace(**vars(args)); a5.shape, a5.factors = "netflix", 128
    d, triples = build_workload("netflix", dev, args.num_ng, args.seed, "cuda")
    U, I, F, B = d["user_num"], d["item_num"], 128, args.batch
    T = triples.shape[0]
    g = torch.Generator(device=dev); g.manual_seed(args.seed)
    perm = torch.randperm(T, generator=g, device=dev)[:(steps + 4) * B].contiguous()
    bu, bi, bj = ops.gather_triples(triples, perm)
    del triples, perm
    P, Q = init_tables(U, I, F, args.seed, dev)
    ws = ops.MFWorkspace(U, I, F, "sgd", dev)
    hp = ops.hyper(**HYPER)
    ops.mf_bpr_train_steps(P, Q, ws, bu, bi, bj, B, 0, 4, hp, check=False)
    ms = timed_ms(lambda: ops.mf_bpr_train_steps(P, Q, ws, bu, bi, bj, B, 4, steps, hp, check=False), 1, 2) / steps
    bpt = 24 * F + 12
    return {"workload": workload_config(a5, 1)["workload"], "value": B / ms * 1e3, "unit": UNIT, "ms_per_step": ms,
            "batch": B, "n_gpus": 1, "roofline": roof(B * bpt / ms / 1e6, "mf_bpr_steps_kernel", bpt),
            "step_kernel": step_kernel_info(F, U + I)}


def cfg_inference(args, dev, d, P, Q):
    """rank (4 096 users x 1 000 candidates, top-50), full_rank_users (4 096 users x all items), KPIs of the rank output."""
    from daisyrec_b200 import ops
    U, I, F = d["user_num"], d["item_num"], P.shape[1]
    g = torch.Generator(device=dev); g.manual_seed(5)
    n, C, K = 4096, 1000, 50
    users = torch.randint(0, U, (n,), device=dev, generator=g)
    cands = torch.randint(0, I, (n, C), device=dev, generator=g)
    ms_r = timed_ms(lambda: ops.mf_rank(P, Q, users, cands, K), 2, 10)
    alg_r = n * (C * (4 * F + 8) + 4 * F + 4 * K)
    ms_f = timed_ms(lambda: ops.mf_full_rank(P, Q, users, K), 1, 5)
    alg_f = n * (I * 4 * F + 4 * F + 8 * K)
    preds = ops.mf_rank(P, Q, users, cands, K)
    lens = torch.randint(1, 21, (n,), device=dev, generator=g)
    ptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    ptr[1:] = torch.cumsum(lens, 0)
    rows = torch.repeat_interleave(torch.arange(n, device=dev), lens)
    key, _ = torch.sort(rows * I + torch.randint(0, I, (rows.numel(),), device=dev, generator=g))
    gt_idx = (key % I).to(torch.int32).contiguous()
    ks = [1, 5, 10, 20, 30, 50]
    ms_k = timed_ms(lambda: ops.rank_metrics(preds, ptr, gt_idx, ks, I), 2, 10)
    alg_k = n * K * 4 + rows.numel() * 4 + (n + 1) * 8
    return {"kpis": {"users": n, "topk": K, "ks": ks, "ms": ms_k, "users_per_s": n / ms_k * 1e3,
                     "roofline": roof(alg_k / ms_k / 1e6, "kpi_kernel (+ coverage / finish)", alg_k,
                                      "preds + ground-truth CSR read once; launch-latency-sized at 4 096 users")},
            "rank": {"users": n, "cand_num": C, "topk": K, "ms": ms_r, "users_per_s": n / ms_r * 1e3,
                     "roofline": roof(alg_r / ms_r / 1e6, "rank_kernel", alg_r, "per user: cand_num x (row + id) + own row + out")},
            "full_rank_users": {"users": n, "item_num": I, "topk": K, "ms": ms_f, "users_per_s": n / ms_f * 1e3,
                                "roofline": roof(alg_f / ms_f / 1e6, "rank_kernel (chunked merge)", alg_f,
                                                 "item table (6.8 MB) is L2-resident: algorithmic bytes are L2 reads")}}


def cfg_sampling(args, dev, d):
    """BasicNegtiveSampler.sampling() at the ML-20M shape: host MT19937 replay + k-th complement + explode."""
    from daisyrec_b200 import ops
    U, I, G = d["user_num"], d["item_num"], args.num_ng
    row_ptr_h = d["row_ptr"].cpu().numpy()
    t0 = time.perf_counter()
    draws = ops.sampler_draw_mt19937(ops.mt19937_seed(args.seed), row_ptr_h, U, I, G)
    t_host = time.perf_counter() - t0
    d_draws = torch.from_numpy(draws).to(dev)
    ms_k = timed_ms(lambda: ops.sampler_kth_complement(d["row_ptr"], d["col"], d_draws, I), 1, 5)
    js = ops.sampler_kth_complement(d["row_ptr"], d["col"], d_draws, I)
    ms_e = timed_ms(lambda: ops.sampler_explode(d["coo_u"], d["coo_i"], js), 1, 3)
    nnz = d["coo_u"].numel()
    T = nnz * G
    alg_e = T * 12 + nnz * 8
    return {"triples": T, "host_mt19937_draws_s": t_host, "kth_complement_ms": ms_k, "explode_ms": ms_e,
            "triples_per_s": T / (t_host + (ms_k + ms_e) * 1e-3),
            "roofline": roof(alg_e / ms_e / 1e6, "explode_kernel", alg_e, "12 B written per triple + 8 B read per COO row")}


def cfg_shuffle(args, dev, d):
    """The DataLoader's epoch permutation of the 80 M triples, bit-exact on the device: MT19937 stream + parallel Fisher-Yates."""
    from daisyrec_b200 import ops
    T = d["coo_u"].numel() * args.num_ng
    ms_mt = timed_ms(lambda: ops.mt19937_stream(args.seed, T, dev), 1, 3)
    ms_all = timed_ms(lambda: ops.randperm_torch(args.seed, T, dev), 1, 3)
    t0 = time.perf_counter()
    g = torch.Generator(); g.manual_seed(args.seed)
    ref = torch.randperm(T, generator=g)
    t_cpu = time.perf_counter() - t0
    same = bool(torch.equal(ops.randperm_torch(args.seed, T, dev).cpu(), ref))
    variant = ops.mt19937_stream_variant(T)
    return {"n": T, "mt19937_kernel": variant, "mt19937_stream_ms": ms_mt, "randperm_total_ms": ms_all, "fisher_yates_ms": ms_all - ms_mt,
            "torch_cpu_randperm_s": t_cpu, "equals_torch_randperm": same,
            "roofline": roof(T * 4 / ms_mt / 1e6, "mt19937_segments_kernel (one CTA per 1 680 blocks of 624 words, jump-ahead polynomials)"
                             if variant == "segmented" else "mt19937_stream_kernel (one CTA)", T * 4,
                             "bounded by the Horner jump (19 937 single steps per set bit of the segment index), not by bytes")}


# SURVEY 8(f) ranks 3-4 on the device, one step-time line each.  Random-init parameters of the reference's shapes; parity is
# the business of tests/test_gpu_{fm,ngcf,nfm}.py.
def cfg_f_fm(args, dev, d, planes):
    """FM + BPR, ML-20M shape, F=64, SGD: the first-order terms ride in the GEN step instantiation."""
    from daisyrec_b200 import ops
    from daisyrec_b200.utils.synthetic import init_tables
    bu, bi, bj = planes
    U, I, F, B = d["user_num"], d["item_num"], 64, args.batch
    P, Q = init_tables(U, I, F, args.seed + 3, dev)
    bias = torch.zeros(U + I + 1, dtype=torch.float32, device=dev)
    ws = ops.FMWorkspace(U, I, F, "sgd", dev)
    hp = ops.hyper(0.01, 0.001, 0.001, "sgd")
    nst, k = min(8, bu.numel() // B), [0]

    def step():
        ops.fm_train_steps(P, Q, bias, ws, bu, bi, bj, B, k[0] % nst, 1, hp, check=False)
        k[0] += 1
    ms = timed_ms(step, 3, 10)
    alg = B * (24 * F + 12 + 24)
    return {"workload": f"FM+BPR synthetic ml-20m shape, factors={F}, SGD", "value": B / ms * 1e3, "unit": UNIT,
            "ms_per_step": ms, "batch": B,
            "roofline": roof(alg / ms / 1e6, "mf_bpr_steps_kernel<GEN> with the packed bias vector", alg,
                             "24 F + 12 B per triple + 3 bias scalars read and written")}


def cfg_f_nfm(args, dev, d, planes):
    """NFM + BPR, ML-20M shape, F=64, one hidden layer + BatchNorm, relu, Adam (fp32 layer-wise path)."""
    from daisyrec_b200 import ops
    from daisyrec_b200.utils.synthetic import init_tables
    bu, bi, bj = planes
    U, I, F = d["user_num"], d["item_num"], 64
    Ln, bn, B = 1, True, min(args.batch, 1 << 18)
    g = torch.Generator(device=dev); g.manual_seed(11)
    P, Q = init_tables(U, I, F, args.seed + 4, dev)
    P.mul_(10.0); Q.mul_(10.0)
    bias = torch.zeros(U + I + 1, dtype=torch.float32, device=dev)
    N = (torch.randn(ops.nfm_param_count(F, Ln, bn), device=dev, generator=g) * 0.1).contiguous()
    N[0:F] = 1.0                                        # BatchNorm 0 weight (layout: NFMRecommender module-registration order)
    o = 2 * F + F * F + F
    N[o:o + F] = 1.0                                    # BatchNorm 1 weight
    R = torch.zeros(2 * 2 * F, dtype=torch.float32, device=dev)
    R[F:2 * F] = 1.0; R[3 * F:4 * F] = 1.0              # running variances start at 1
    ws = ops.NfmWorkspace(U, I, F, Ln, bn, "adam", 2 * B, dev)
    hp = ops.hyper(0.001, 0.0, 0.001, "adam")
    nst, k = min(8, bu.numel() // B), [0]

    def step():
        ops.nfm_bpr_train_steps(P, Q, bias, N, R, ws, ops.NFM_ACT["relu"], bu, bi, bj, B, k[0] % nst, 1, hp, adam_step0=k[0],
                                check=False)
        k[0] += 1
    ms = timed_ms(step, 3, 10)
    alg = B * (3 * 4 * F * 2 + 12) + 2 * B * 4 * F * 2 * (3 + 4 * Ln)
    return {"workload": f"NFM+BPR synthetic ml-20m shape, factors={F}, num_layers={Ln}, batch_norm, relu, Adam", "value": B / ms * 1e3,
            "unit": UNIT, "ms_per_step": ms, "batch": B,
            "roofline": roof(alg / ms / 1e6, "nfm_* kernels: layer-wise, activations through HBM", alg,
                             "row gathers / scatters + one read and one write of every [2B, F] activation and gradient")}


def cfg_f_ngcf(args, dev):
    """NGCF + BPR, Amazon-Book shape, widths 64/64/64/64, Adam, dropout 0."""
    from daisyrec_b200 import ops
    from daisyrec_b200.utils.synthetic import SHAPES, make_interactions
    U, I, nnz = SHAPES["amazon-book"]
    g = torch.Generator(device=dev); g.manual_seed(12)
    da = make_interactions(U, I, nnz, seed=args.seed, device=dev)
    adj = ops.lgcn_build_adj(da["coo_u"], da["coo_i"], U, I)
    graph = ops.LgcnGraph(*adj, dev)
    nnzA = int(adj[1].numel())
    dims = [64, 64, 64, 64]
    E0 = (torch.randn(U + I, dims[0], device=dev, generator=g) * 0.05).contiguous()
    W = (torch.randn(ops.ngcf_param_count(dims), device=dev, generator=g) * 0.1).contiguous()
    ws = ops.NgcfWorkspace(U, I, dims, "adam", dev)
    B = 65536
    idx = torch.randint(0, da["coo_u"].numel(), (4 * B,), device=dev, generator=g)
    bu, bi = da["coo_u"][idx].contiguous(), da["coo_i"][idx].contiguous()
    bj = torch.randint(0, I, (4 * B,), device=dev, dtype=torch.int32, generator=g)
    hp = ops.hyper(0.001, 0.0, 0.001, "adam")
    k = [0]

    def step():
        ops.ngcf_bpr_train_steps(E0, W, ws, graph, bu, bi, bj, B, k[0] % 4, 1, hp, adam_step0=k[0], check=False)
        k[0] += 1
    ms = timed_ms(step, 3, 10)
    Lg = len(dims) - 1
    alg = 2 * Lg * (nnzA * (8 + 4 * 64) + (U + I) * 4 * 64 * 6) + B * (24 * sum(dims) + 12)
    return {"workload": f"NGCF+BPR synthetic amazon-book shape ({U}x{I}, nnz={da['nnz']}), widths {dims}, Adam, dropout 0",
            "value": B / ms * 1e3, "unit": UNIT, "ms_per_step": ms, "batch": B, "adjacency_nnz": nnzA,
            "roofline": roof(alg / ms / 1e6, "spmm_seg_kernel + BiGNN GEMMs / row kernels x 2L + BPR phases + Adam", alg,
                             "upper-bound algorithmic bytes (sparse products + 6 [N, F] streams per layer and direction)")}


def run_configs(args, dev, d, planes, P, Q, which):
    out = {}

    def section(name, fn):
        if which != ["all"] and name not in which:
            return
        try:
            out[name] = fn()
        except Exception as e:  # noqa: BLE001  (keep the headline line whatever a secondary config does)
            import traceback
            out[name] = {"error": repr(e), "trace": traceback.format_exc()[-400:]}
        torch.cuda.empty_cache()

    section("c3_neumf", lambda: cfg_c3_neumf(args, dev, d, planes))
    section("c4_lightgcn", lambda: cfg_c4_lightgcn(args, dev))
    section("inference", lambda: cfg_inference(args, dev, d, P, Q))
    section("sampling", lambda: cfg_sampling(args, dev, d))
    section("shuffle", lambda: cfg_shuffle(args, dev, d))
    section("f_fm", lambda: cfg_f_fm(args, dev, d, planes))
    section("f_nfm", lambda: cfg_f_nfm(args, dev, d, planes))
    section("f_ngcf", lambda: cfg_f_ngcf(args, dev))
    return out


# ------------------------------------------------------------------------------- own arm, one GPU
def run_own(args):
    rank, local, world = dist_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (own arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs writes the single-GPU path's outputs; run it with one process")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        return run_sharded(args, rank, local, world, dev)
    from daisyrec_b200 import ops
    from daisyrec_b200.model.MFRecommender import MF
    from daisyrec_b200.utils.dataset import BasicDataset, get_dataloader
    from daisyrec_b200.utils.synthetic import init_tables
    which = [w for w in args.configs.split(",") if w]

    d, triples = build_workload(args.shape, dev, args.num_ng, args.seed, "cuda")
    U, I, F, B = d["user_num"], d["item_num"], args.factors, args.batch
    T = triples.shape[0]
    g = torch.Generator(device=dev); g.manual_seed(args.seed)
    perm = torch.randperm(T, generator=g, device=dev)
    bu, bi, bj = ops.gather_triples(triples, perm)
    del perm
    spe = (T + B - 1) // B                                           # steps per epoch
    ncpu = min(T, 3 * B)                                             # the CPU baseline's sample: 3 batches of this epoch
    cpu_rows = torch.stack([bu[:ncpu], bi[:ncpu], bj[:ncpu]], 1).cpu().numpy()

    model = MF(mf_config(U, I, F))
    P0, Q0 = init_tables(U, I, F, args.seed, dev)
    model.load_state_dict({"embed_user.weight": P0, "embed_item.weight": Q0})
    model._begin_fit("sgd")
    P, Q, ws, hp = model.embed_user.weight, model.embed_item.weight, model._ws, model._hp

    def run_steps(first, k, timed):
        """k steps starting at global step `first`, walking the epoch cyclically; one launch per epoch segment.
        -> (events, launches, per-step losses of the last launch)."""
        evs, launches, s, losses = [], 0, first, None
        while k > 0:
            pos = s % spe
            seg = min(k, spe - pos)
            if timed:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            losses = ops.mf_bpr_train_steps(P, Q, ws, bu, bi, bj, B, pos, seg, hp, check=False)
            if timed:
                e1.record()
                evs.append((e0, e1, seg, pos))
            launches += 1
            s += seg
            k -= seg
        return evs, launches, losses

    clocks = ClockSampler(local)
    run_steps(0, args.warmup, False)
    torch.cuda.synchronize()
    t_region0 = time.time()
    evs, launches, losses = run_steps(args.warmup, args.steps, True)
    torch.cuda.synchronize()
    t_region1 = time.time()
    # snapshot now: fit_host_batches below trains the same tables further
    outputs = timed_outputs({"embed_user.weight": P, "embed_item.weight": Q, "loss": losses[-1:]}) if args.dump_outputs else None
    ms = sum(e0.elapsed_time(e1) for e0, e1, _, _ in evs)
    done_triples = 0
    for _, _, seg, pos in evs:
        done_triples += min(T, (pos + seg) * B) - pos * B
    value = done_triples / ms * 1e3
    nan_check = ops.mf_bpr_loss(P, Q, ws, bu[:B], bi[:B], bj[:B], hp).item()
    if not np.isfinite(nan_check):
        raise RuntimeError("bench: loss became non-finite during the timed steps")

    # ---- end to end = the reference's plug-in call (run_examples/test.py:91-95): fit(DataLoader) over PINNED host triples,
    #      one full epoch, wall clock: upload + id check + epoch permutation + gather + all steps + loss read-back
    host_t = torch.empty((T, 3), dtype=torch.int32).pin_memory()
    host_t.copy_(triples)
    host_np = host_t.numpy()
    del triples
    torch.cuda.empty_cache()
    e2e_runs = {}
    for engine in ("torch", "torch-cpu", "device"):
        walls = []
        for rep in range((1 if engine == "torch-cpu" else args.e2e_reps) + 1):   # first repetition = warm-up (allocator, page-in)
            torch.manual_seed(args.seed + rep)
            m = MF(mf_config(U, I, F, shuffle_engine=engine))
            loader = get_dataloader(BasicDataset(host_np), batch_size=B, shuffle=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.fit(loader)
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
            del m, loader
        walls = walls[1:]
        med = float(np.median(walls))
        e2e_runs[engine] = {"value": T / med, "wall_s_median": med, "wall_s": walls, "epochs_per_run": 1,
                            "h2d_bytes_per_step": (12 + (8 if engine == "torch-cpu" else 0)) * B, "steps": spe}
    from daisyrec_b200.model.AbstractRecommender import DEFAULT_SHUFFLE_ENGINE as default_engine
    e2e_main = e2e_runs[default_engine]

    # fit_host_batches: per-step H2D of the batch + per-step loss D2H (pipelined), >= 0.25 s of steps
    ke = spe - 1
    planes_h = [t[:ke * B].cpu().pin_memory() for t in (bu, bi, bj)]
    model.fit_host_batches(*[p_[:3 * B] for p_ in planes_h], B, 3)   # warm-up
    torch.cuda.synchronize()
    rounds, t0 = 0, time.perf_counter()
    while True:
        host_losses = model.fit_host_batches(*planes_h, B, ke)
        rounds += 1
        if time.perf_counter() - t0 >= 0.25 and rounds >= 2:
            break
    torch.cuda.synchronize()
    hb_s = time.perf_counter() - t0
    assert bool(torch.isfinite(host_losses).all())
    t_e1 = time.time()
    clk = clocks.stop(t_region0, t_e1)

    # ---- the other BASELINE configs + the kernels either side of the step
    cfgs = {}
    if which != ["none"]:
        cfgs = run_configs(args, dev, d, (bu, bi, bj), P, Q, which)
        if which == ["all"] or "c5_netflix_1gpu" in which:
            del bu, bi, bj, planes_h
            torch.cuda.empty_cache()
            try:
                cfgs["c5_netflix_1gpu"] = cfg_c5_single(args, dev)
            except Exception as e:  # noqa: BLE001
                cfgs["c5_netflix_1gpu"] = {"error": repr(e)}

    # ---- CPU baseline: the real reference's fit on this host's cores (child process, GPUs hidden, bounded sample)
    cpu = cpu_baseline_subprocess(args, cpu_rows)

    peak, peak_src = measured_peaks()
    bytes_per_triple = 24 * F + 12
    avg_launch_ms = ms / len(evs)
    avg_launch_triples = done_triples / len(evs)
    achieved = avg_launch_triples * bytes_per_triple / (avg_launch_ms * 1e-3) / 1e9
    traffic, traffic_src = profiled_traffic(F, B)
    sk = step_kernel_info(F, U + I)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, 1), "steps_per_epoch": spe,
            "clocks": clk,
            "e2e": {"value": e2e_main["value"], "unit": UNIT, "h2d_bytes_per_step": e2e_main["h2d_bytes_per_step"],
                    "d2h_bytes_per_step": 8.0 / spe, "steps": spe * args.e2e_reps, "wall_s_median": e2e_main["wall_s_median"],
                    "api": "MF(config).fit(get_dataloader(BasicDataset(pinned host int32[T,3]), batch_size, shuffle=True)): one "
                           "epoch per run, wall clock around fit() incl. the 12 B/triple upload, id range check, epoch "
                           "permutation, gather, all steps and the epoch-loss read-back; median of "
                           f"{args.e2e_reps} runs after one warm-up run; shuffle_engine={default_engine!r} (the default)",
                    "engines": e2e_runs,
                    "fit_host_batches": {"value": rounds * ke * B / hb_s, "steps": rounds * ke, "wall_s": hb_s,
                                         "h2d_bytes_per_step": 12 * B, "d2h_bytes_per_step": 8,
                                         "api": "MF.fit_host_batches(pinned host planes): per step H2D of the batch + step "
                                                "kernel + D2H of the loss, copy of batch s+1 under the kernel of batch s"}},
            "gpu_launches": launches,
            "gpu_launches_note": "persistent cooperative kernel: one launch runs up to steps_per_epoch synchronous steps",
            "step_kernel": sk,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": None if traffic is None else traffic * (args.steps / len(evs)),
                         "traffic_note": f"dram__bytes_read+write per step ({traffic_src}: ncu capture of the general "
                                         "instantiation mf_bpr_steps_kernel<4,16,1>; a lean instantiation moves the same rows) x "
                                         "steps per launch; the 85 MB working set is L2-resident, so the limiter at this shape is "
                                         "L2/issue, not HBM -- configs.c5_netflix_1gpu is the HBM-regime figure",
                         "peak_source": peak_src, "algorithmic_bytes_per_triple": bytes_per_triple,
                         "kernel": sk["instantiation"], "avg_launch_ms": avg_launch_ms},
            "cpu_baseline": cpu,
            "configs": cfgs}
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------- own arm, N GPUs (one process each)
def sharded_parity_check(d, triples, perm, bounds, rank, world, dev, F, seed, comm):
    """3 global steps on a 48 K-triple slice: every rank trains its share (sharded path), rank 0 also runs the single-GPU
    kernel on the same global batches (the single-GPU run is the pinned oracle of N > 1).  All ranks return the verdict."""
    import torch.distributed as dist
    from daisyrec_b200 import ops
    from daisyrec_b200.parallel import ShardedTrainer, allgather_rows
    from daisyrec_b200.utils.synthetic import init_tables
    U, I = d["user_num"], d["item_num"]
    Bs, K = 16384, 3
    sl = perm[:Bs * K].contiguous()
    P0, Q0 = init_tables(U, I, F, seed + 1, dev)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    tr = ShardedTrainer(P0[lo:hi].clone(), Q0.clone(), bounds, rank, world, ops.hyper(**HYPER), comm=comm)   # clone: a slice's .contiguous() aliases P0
    m = tr.prepare_epoch(triples, sl, Bs)
    assert m == K
    losses = tr.train_steps(0, K).clone()
    tr.check_nan()
    P_all = allgather_rows(tr.P[:hi - lo], torch.arange(lo, hi, device=dev), U)
    qsum = tr.Q.view(torch.int32).to(torch.int64).sum().reshape(1)
    qs = [torch.zeros_like(qsum) for _ in range(world)]
    dist.all_gather(qs, qsum)
    q_same = all(int(q.item()) == int(qs[0].item()) for q in qs)
    q_sharded = tr.Q.clone()
    tr.close()
    verdict = torch.zeros(4, dtype=torch.float64, device=dev)
    if rank == 0:
        P1, Q1 = P0.clone(), Q0.clone()
        ws = ops.MFWorkspace(U, I, F, "sgd", dev)
        bu, bi, bj = ops.gather_triples(triples, sl)
        ref = ops.mf_bpr_train_steps(P1, Q1, ws, bu, bi, bj, Bs, 0, K, ops.hyper(**HYPER))
        rel = float(((losses - ref).abs() / ref.abs()).max().item())
        dP = float((P_all - P1).abs().max().item())
        dQ = float((q_sharded - Q1).abs().max().item())
        moved = float((P1 - P0).abs().max().item())
        verdict = torch.tensor([rel, max(dP, dQ), moved, 1.0 if q_same else 0.0], dtype=torch.float64, device=dev)
    dist.broadcast(verdict, 0)
    rel, dtab, moved, qok = (float(x) for x in verdict.tolist())
    ok = rel <= 1e-5 and dtab <= 1e-6 and qok == 1.0 and moved > 0
    return {"ok": ok, "max_rel_loss": rel, "max_abs_table": dtab, "q_replicas_identical": bool(qok), "steps": K,
            "global_batch": Bs, "max_abs_update": moved,
            "how": "sharded N-rank run vs the single-GPU step kernel on the same 3 global batches (tolerances: loss rel 1e-5, "
                   "tables abs 1e-6; item replicas compared bit for bit across ranks)"}


def run_sharded(args, rank, local, world, dev):
    """Weak scaling: per-GPU batch fixed (args.batch), global batch = world * batch."""
    import torch.distributed as dist
    from daisyrec_b200 import ops
    from daisyrec_b200.parallel import ShardedTrainer, partition_users
    from daisyrec_b200.utils.synthetic import init_tables

    def shape_run(shape, F, steps, warmup, with_e2e):
        a = argparse.Namespace(**vars(args)); a.shape, a.factors = shape, F
        d, triples = build_workload(shape, dev, args.num_ng, args.seed, "cuda")     # identical on every rank
        U, I = d["user_num"], d["item_num"]
        T = triples.shape[0]
        Bg = args.batch * world
        deg = (d["row_ptr"][1:] - d["row_ptr"][:-1]).cpu().numpy()
        bounds = partition_users(deg, world)
        g = torch.Generator(device=dev); g.manual_seed(args.seed)
        perm = torch.randperm(T, generator=g, device=dev)
        P0, Q0 = init_tables(U, I, F, args.seed, dev)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        progress["stage"] = f"{shape}: trainer setup ({comm})"
        tr = ShardedTrainer(P0[lo:hi].contiguous(), Q0.contiguous(), bounds, rank, world, ops.hyper(**HYPER), comm=comm)
        del P0
        spe = tr.prepare_epoch(triples, perm, Bg)
        par_sl = perm[:16384 * 3].clone()
        del perm
        torch.cuda.empty_cache()
        local_counts = np.diff(tr.offsets_host)
        scratch_losses = torch.empty(spe + 1, dtype=torch.float64, device=dev)

        def run(first, k):
            n_loc, s = 0, first
            while k > 0:
                pos = s % spe
                seg = min(k, spe - pos)
                tr.train_steps(pos, seg, scratch_losses)
                n_loc += int(local_counts[pos:pos + seg].sum())
                s += seg
                k -= seg
            return n_loc

        progress["stage"] = f"{shape}: warm-up steps ({comm})"
        run(0, warmup)
        torch.cuda.synchronize(); dist.barrier()
        progress["stage"] = f"{shape}: timed steps ({comm})"
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        n_loc = run(warmup, steps)
        e1.record()
        torch.cuda.synchronize(); dist.barrier()
        t1 = time.time()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        tot = torch.tensor([n_loc], dtype=torch.float64, device=dev)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        tr.check_nan()
        res = {"d": d, "T": T, "spe": spe, "ms": float(ms.item()), "value": float(tot.item()) / float(ms.item()) * 1e3,
               "t0": t0, "t1": t1, "parity": None, "cfg": workload_config(a, world), "steps": steps}
        progress[shape] = res                                    # the watchdog can print from here on
        progress["stage"] = f"{shape}: parity check ({comm})"
        res["parity"] = sharded_parity_check(d, triples, par_sl, bounds, rank, world, dev, F, args.seed, comm)
        del triples
        if with_e2e:
            progress["stage"] = f"{shape}: e2e host-fed steps ({comm})"
            # e2e: pinned host share of every global batch of one epoch segment -> native loop (H2D per step, loss D2H per step)
            ke = min(spe - 1, 64)
            offs = tr.offsets_host[:ke + 1].copy()
            nloc = int(offs[-1])
            h = [t[:nloc].cpu().pin_memory() for t in (tr.bu, tr.bi, tr.bj)]
            tr.train_steps_host(*h, offs, 0, min(3, ke))
            torch.cuda.synchronize(); dist.barrier()
            rounds, tw0 = 0, time.perf_counter()
            stop = torch.zeros(1, device=dev)
            while True:
                hl = tr.train_steps_host(*h, offs, 0, ke)
                rounds += 1
                stop[0] = 1.0 if (time.perf_counter() - tw0 >= 0.25 and rounds >= 2) else 0.0
                dist.all_reduce(stop, op=dist.ReduceOp.MIN)              # every rank leaves after the same round
                if float(stop.item()) > 0:
                    break
            torch.cuda.synchronize(); dist.barrier()
            wall = torch.tensor([time.perf_counter() - tw0], dtype=torch.float64, device=dev)
            dist.all_reduce(wall, op=dist.ReduceOp.MAX)
            etot = torch.tensor([float(nloc) * rounds], dtype=torch.float64, device=dev)
            dist.all_reduce(etot, op=dist.ReduceOp.SUM)
            assert bool(torch.isfinite(hl).all())
            res["e2e"] = {"value": float(etot.item()) / float(wall.item()), "unit": UNIT,
                          "h2d_bytes_per_step": 12.0 * float(etot.item()) / (rounds * ke), "d2h_bytes_per_step": 8 * world,
                          "steps": rounds * ke, "wall_s": float(wall.item()),
                          "api": "ShardedTrainer.train_steps_host(pinned host shares): native loop, per global step H2D of "
                                 "each rank's share + phase 1 + exchange + phase 2 + D2H of the global loss; copy of step "
                                 "s+1 under step s"}
            res["t1"] = time.time()
        tr.close()
        del tr
        torch.cuda.empty_cache()
        return res

    comm = args.comm if args.comm != "auto" else ("p2p" if world == 2 else "nccl")
    progress = {"stage": "start"}
    clocks = ClockSampler(local) if rank == 0 else None
    printed = threading.Event()

    def emit(main, c5, incomplete=None):
        """rank 0: the driver's JSON line from whatever has been measured."""
        if printed.is_set():
            return
        printed.set()
        if main is None:
            print(json.dumps({"metric": METRIC, "value": None, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                              "warmup": args.warmup, "higher_is_better": True, "comm": comm,
                              "incomplete": incomplete}), flush=True)
            return
        clk = clocks.stop(main["t0"], main["t1"])
        peak, peak_src = measured_peaks()
        F = args.factors
        bpt = 24 * F + 12
        achieved = main["value"] / world * bpt / 1e9                      # per-GPU algorithmic GB/s of the step
        exchange = ("ONE grouped NCCL all-reduce of gQ/counters/norms enqueued by the library between the phase-1 and "
                    "phase-2 kernels" if comm == "nccl" else
                    "in-kernel peer exchange over NVLink (no NCCL, no relaunch per step)")
        line = {"metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": main["ms"] / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": main["cfg"],
                "steps_per_epoch": main["spe"], "exchange": exchange, "comm": comm,
                "clocks": clk, "e2e": main.get("e2e"), "parity_check": main["parity"],
                "gpu_launches": 2 * args.steps if comm == "nccl" else 1,
                "step_kernel": step_kernel_info(F, main["d"]["user_num"] // world + main["d"]["item_num"]),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_triple": bpt,
                             "kernel": "mf_bpr_steps_kernel (per GPU)"}}
        if c5 is not None:
            b5 = 24 * 128 + 12
            a5 = c5["value"] / world * b5 / 1e9
            line["configs"] = {"c5": {"workload": c5["cfg"]["workload"], "value": c5["value"], "unit": UNIT, "n_gpus": world,
                                      "ms_per_step": c5["ms"] / c5["steps"], "steps": c5["steps"],
                                      "per_gpu_batch": args.batch, "parity_check": c5["parity"],
                                      "roofline": roof(a5, "mf_bpr_steps_kernel (per GPU)", b5)}}
        if incomplete:
            line["incomplete"] = incomplete
        print(json.dumps(line), flush=True)

    def watchdog():
        # a stage that never returns (a collective or a mapping call that blocks) must not cost the line: after --watchdog
        # seconds rank 0 prints what has been measured and every rank leaves without waiting for the others
        if printed.wait(args.watchdog):
            return
        why = f"watchdog after {args.watchdog:.0f} s in stage '{progress.get('stage')}'"
        if rank == 0:
            emit(progress.get(args.shape), progress.get("netflix") if progress.get(args.shape) else None, why)
        sys.stderr.write(f"[bench rank {rank}] {why}\n")
        sys.stderr.flush()
        os._exit(0 if progress.get(args.shape) else 4)

    threading.Thread(target=watchdog, daemon=True).start()
    main = shape_run(args.shape, args.factors, args.steps, args.warmup, True)
    c5 = None
    if args.c5 == "on" or (args.c5 == "auto" and world >= 8):
        c5 = shape_run("netflix", 128, max(100, args.steps), max(10, args.warmup), False)
    ok = main["parity"]["ok"] and (c5 is None or c5["parity"]["ok"])
    if rank == 0:
        emit(main, c5)
    printed.set()
    dist.barrier()
    dist.destroy_process_group()
    return 0 if ok else 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20)
    ap.add_argument("--factors", type=int, default=64)
    ap.add_argument("--shape", default="ml-20m")
    ap.add_argument("--num-ng", dest="num_ng", type=int, default=4)
    ap.add_argument("--seed", type=int, default=2022)
    ap.add_argument("--e2e-reps", dest="e2e_reps", type=int, default=3)
    ap.add_argument("--configs", default="all", help="all | none | comma list of c3_neumf,c4_lightgcn,c5_netflix_1gpu,inference,sampling,shuffle,f_fm,f_nfm,f_ngcf")
    ap.add_argument("--c5", default="auto", choices=["auto", "on", "off"], help="N > 1: also run config 5 (netflix F=128)")
    ap.add_argument("--comm", default="auto", choices=["auto", "nccl", "p2p"],
                    help="N > 1: auto = in-kernel peer exchange on 2 GPUs (validated), the NCCL step beyond; or force one")
    ap.add_argument("--watchdog", type=float, default=420.0,
                    help="N > 1: seconds after which rank 0 prints the line with what has been measured and every rank exits")
    ap.add_argument("--cpu-budget", dest="cpu_budget", type=float, default=45.0)
    ap.add_argument("--ref-budget", dest="ref_budget", type=float, default=330.0)
    ap.add_argument("--ref-workers", dest="ref_workers", type=int, default=4, help="DataLoader workers of the reference (test.py:94)")
    ap.add_argument("--rows-file", dest="rows_file", default=None, help="reference arm: .npy of sampler triples to train on")
    ap.add_argument("--quick", action="store_true", help="reference arm: main measurement only")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="own arm, one GPU: after the timed steps write DIR/<name>.npy of what the last timed step returned "
                         "(embed_user.weight, embed_item.weight, loss); above 64 MB a fixed seeded sample of table rows")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the own arm's outputs")
    if args.impl == "reference":
        args.steps = 8 if args.steps is None else args.steps
        args.warmup = 2 if args.warmup is None else args.warmup
        return run_reference(args)
    args.steps = 760 if args.steps is None else args.steps
    args.warmup = 76 if args.warmup is None else max(args.warmup, 3)
    return run_own(args)


if __name__ == "__main__":
    sys.exit(main())
