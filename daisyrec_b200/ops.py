"""Tensor-level bindings of the C ABI (include/daisyrec_b200.h).

torch is plumbing here: device memory (``tensor.data_ptr()``) and the current CUDA stream.
Every function forwards to libdaisyrec_b200.so; nothing is computed by torch ops.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _dev(t, dtype, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == dtype and t.is_contiguous()):
        raise TypeError(f"{name}: expected a contiguous CUDA tensor of dtype {dtype}")
    return t


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("daisyrec_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def hyper(lr, reg_1, reg_2, opt="sgd", beta1=0.9, beta2=0.999, eps=1e-8, loss="BPR"):
    return L.Hyper(lr, reg_1, reg_2, L.OPT_KIND[opt], beta1, beta2, eps, L.LOSS_KIND[loss.upper()])


def device_query():
    sm, ma, mi, l2 = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    L.check(L.lib().drb_device_query(C.byref(sm), C.byref(ma), C.byref(mi), C.byref(l2)))
    return dict(sm_count=sm.value, cc=(ma.value, mi.value), l2_bytes=l2.value)


def mf_step_variant(factors, table_rows=0):
    """-> (lean, lanes_per_row, chunks_per_lane) of the BPR + SGD / Adam step kernel for this factor count and table size
    (user_num + item_num; 0 = the L2 regime).  Runs the one-off on-device selection if it has not run yet."""
    w, n = C.c_int32(0), C.c_int32(0)
    lean = L.lib().drb_mf_step_variant(int(factors), int(table_rows), C.byref(w), C.byref(n))
    return bool(lean), int(w.value), int(n.value)


def mf_step_selfcheck_ms(factors, table_rows=0):
    """-> (ms_general, ms_lean, tile_cap) of the on-device selection for this factor count and table size."""
    a, b, t = C.c_float(0), C.c_float(0), C.c_int32(0)
    L.lib().drb_mf_step_selfcheck_ms(int(factors), int(table_rows), C.byref(a), C.byref(b), C.byref(t))
    return float(a.value), float(b.value), int(t.value)


def check_index_range(ids, bounds, what):
    """IndexError (what nn.Embedding raises in the reference) when a column of the device index array ``ids`` [n, len(bounds)]
    holds an id outside [0, bounds[c]).  One kernel + one 64-byte read-back."""
    if not (isinstance(ids, torch.Tensor) and ids.is_cuda and ids.is_contiguous() and ids.dtype in (torch.int32, torch.int64)):
        raise TypeError("check_index_range: expected a contiguous CUDA int32 / int64 tensor")
    ncols = len(bounds)
    n = ids.numel() // ncols
    hi = (C.c_int64 * 4)(*([int(b) for b in bounds] + [0] * (4 - ncols)))
    bad = (C.c_int64 * 4)()
    L.check(L.lib().drb_index_range_check(_ptr(ids), ids.element_size(), n, ncols, hi, bad, _stream()))
    for c in range(ncols):
        if bad[c]:
            raise IndexError(f"index out of range in self: {bad[c]} {what[c]} id(s) outside [0, {int(bounds[c])})")


# ------------------------------------------------------------------ sampler
def mt19937_seed(seed):
    st = np.zeros(625, np.uint32)
    L.check(L.lib().drb_mt19937_seed(st.ctypes.data, C.c_uint32(seed & 0xFFFFFFFF)))
    return st


def mt19937_from_numpy(rs=None):
    s = (np.random if rs is None else rs).get_state()
    st = np.zeros(625, np.uint32)
    st[:624] = s[1]
    st[624] = s[2]
    return st


def mt19937_to_numpy(st, rs=None):
    tgt = np.random if rs is None else rs
    old = tgt.get_state()
    tgt.set_state(("MT19937", st[:624].copy(), int(st[624]), old[3], old[4]))


def sampler_draw_mt19937(state, row_ptr, user_num, item_num, num_ng):
    """Host: the reference's per-user bounded draws (advances ``state`` in place)."""
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    draws = np.empty((user_num, num_ng), np.int32)
    bad = C.c_int32(-1)
    rc = L.lib().drb_sampler_draw_mt19937(state.ctypes.data, row_ptr.ctypes.data, user_num, item_num, num_ng,
                                          draws.ctypes.data, C.byref(bad))
    if rc == L.DRB_ERR_EMPTY_SET:
        raise ValueError("'a' cannot be empty unless no samples are taken")
    L.check(rc)
    return draws


def sampler_draw_philox(seed, offset, d_row_ptr, user_num, item_num, num_ng):
    _dev(d_row_ptr, torch.int64, "row_ptr")
    draws = torch.empty((user_num, num_ng), dtype=torch.int32, device=d_row_ptr.device)
    bad = torch.empty(1, dtype=torch.int32, device=d_row_ptr.device)
    L.check(L.lib().drb_sampler_draw_philox(C.c_uint64(seed), C.c_uint64(offset), _ptr(d_row_ptr), user_num, item_num,
                                            num_ng, _ptr(draws), _ptr(bad), _stream()))
    return draws, bad


def sampler_kth_complement(d_row_ptr, d_col, d_draws, item_num):
    _dev(d_row_ptr, torch.int64, "row_ptr"); _dev(d_col, torch.int32, "col"); _dev(d_draws, torch.int32, "draws")
    U, G = d_draws.shape
    js = torch.empty_like(d_draws)
    L.check(L.lib().drb_sampler_kth_complement(_ptr(d_row_ptr), _ptr(d_col), _ptr(d_draws), U, item_num, G, _ptr(js),
                                               _stream()))
    return js


def sampler_explode(d_coo_u, d_coo_i, d_js):
    _dev(d_coo_u, torch.int32, "coo_u"); _dev(d_coo_i, torch.int32, "coo_i"); _dev(d_js, torch.int32, "js")
    nnz, G = d_coo_u.numel(), d_js.shape[1]
    tr = torch.empty((nnz * G, 3), dtype=torch.int32, device=d_js.device)
    L.check(L.lib().drb_sampler_explode(_ptr(d_coo_u), _ptr(d_coo_i), nnz, _ptr(d_js), G, _ptr(tr), _stream()))
    return tr


def sample_triples_host(state, row_ptr, col, coo_u, coo_i, user_num, item_num, num_ng):
    """All-host-buffer convenience call (H2D/D2H inside the library)."""
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    col = np.ascontiguousarray(col, np.int32)
    coo_u = np.ascontiguousarray(coo_u, np.int32)
    coo_i = np.ascontiguousarray(coo_i, np.int32)
    js = np.empty((user_num, num_ng), np.int32)
    tr = np.empty((len(coo_u) * num_ng, 3), np.int32)
    bad = C.c_int32(-1)
    rc = L.lib().drb_sample_triples_host(state.ctypes.data, row_ptr.ctypes.data, col.ctypes.data, coo_u.ctypes.data,
                                         coo_i.ctypes.data, len(coo_u), user_num, item_num, num_ng, js.ctypes.data,
                                         tr.ctypes.data, C.byref(bad))
    if rc == L.DRB_ERR_EMPTY_SET:
        raise ValueError("'a' cannot be empty unless no samples are taken")
    L.check(rc)
    return js, tr


def bounded_draws_mt19937(state, n, offsets):
    """Host: row m draws offsets[m+1]-offsets[m] values from [0, n[m]) off numpy's MT19937 stream."""
    n = np.ascontiguousarray(n, np.int64)
    offsets = np.ascontiguousarray(offsets, np.int64)
    draws = np.empty(int(offsets[-1]), np.int32)
    bad = C.c_int64(-1)
    rc = L.lib().drb_bounded_draws_mt19937(state.ctypes.data, n.ctypes.data, offsets.ctypes.data, len(n),
                                           draws.ctypes.data, C.byref(bad))
    if rc == L.DRB_ERR_EMPTY_SET:
        raise ValueError("'a' cannot be empty unless no samples are taken")
    L.check(rc)
    return draws


def kth_complement_var(d_row_ptr, d_col, d_offsets, d_draws):
    _dev(d_row_ptr, torch.int64, "row_ptr"); _dev(d_col, torch.int32, "col")
    _dev(d_offsets, torch.int64, "offsets"); _dev(d_draws, torch.int32, "draws")
    out = torch.empty_like(d_draws)
    L.check(L.lib().drb_kth_complement_var(_ptr(d_row_ptr), _ptr(d_col), _ptr(d_offsets), _ptr(d_draws),
                                           d_row_ptr.numel() - 1, _ptr(out), _stream()))
    return out


def sampler_draw_mt19937_mixed(state, row_ptr, user_num, item_num, uniform_num, other_num):
    """Host: numpy-stream replay of the popularity-mixed branch (sampler.py:71-80) -> (ranks i32, doubles f64)."""
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    draws = np.empty((user_num, uniform_num), np.int32)
    u01 = np.empty((user_num, other_num), np.float64)
    bad = C.c_int32(-1)
    rc = L.lib().drb_sampler_draw_mt19937_mixed(state.ctypes.data, row_ptr.ctypes.data, user_num, item_num, uniform_num,
                                                other_num, draws.ctypes.data, u01.ctypes.data, C.byref(bad))
    if rc == L.DRB_ERR_EMPTY_SET:
        raise ValueError("'a' cannot be empty unless no samples are taken")
    L.check(rc)
    return draws, u01


def sampler_assemble_mixed(d_row_ptr, d_col, d_draws, d_cdf, d_u01, item_num):
    _dev(d_row_ptr, torch.int64, "row_ptr"); _dev(d_col, torch.int32, "col")
    _dev(d_draws, torch.int32, "draws"); _dev(d_cdf, torch.float64, "cdf"); _dev(d_u01, torch.float64, "u01")
    U, un, on = d_row_ptr.numel() - 1, d_draws.shape[1], d_u01.shape[1]
    js = torch.empty((U, un + on), dtype=torch.int32, device=d_row_ptr.device)
    L.check(L.lib().drb_sampler_assemble_mixed(_ptr(d_row_ptr), _ptr(d_col), _ptr(d_draws), _ptr(d_cdf), _ptr(d_u01), U,
                                               item_num, un, on, _ptr(js), _stream()))
    return js


def sampler_explode_pointwise(d_coo_u, d_coo_i, d_label, d_js):
    _dev(d_coo_u, torch.int32, "coo_u"); _dev(d_coo_i, torch.int32, "coo_i")
    _dev(d_label, torch.int32, "label"); _dev(d_js, torch.int32, "js")
    nnz, G = d_coo_u.numel(), d_js.shape[1]
    rows = torch.empty((nnz * (1 + G), 3), dtype=torch.int32, device=d_coo_u.device)
    L.check(L.lib().drb_sampler_explode_pointwise(_ptr(d_coo_u), _ptr(d_coo_i), _ptr(d_label), nnz, _ptr(d_js), G,
                                                  _ptr(rows), _stream()))
    return rows


def sgns_positions(d_su, d_row_ptr, item_num, window):
    """Skip-gram positions (users ascending): -> (context counts int64 [n], complement sizes int64 [n]) on the device."""
    _dev(d_su, torch.int32, "su"); _dev(d_row_ptr, torch.int64, "row_ptr")
    n = d_su.numel()
    count = torch.empty(max(n, 1), dtype=torch.int64, device=d_su.device)
    bound = torch.empty(max(n, 1), dtype=torch.int64, device=d_su.device)
    L.check(L.lib().drb_sgns_positions(_ptr(d_su), n, _ptr(d_row_ptr), item_num, window, _ptr(count), _ptr(bound), _stream()))
    return count[:n], bound[:n]


def sgns_explode(d_su, d_si, window, d_offsets, d_row_ptr, d_col, d_draws):
    """-> int32 [2 * offsets[-1], 3] skip-gram rows on the device (positives then negatives of every position)."""
    _dev(d_su, torch.int32, "su"); _dev(d_si, torch.int32, "si"); _dev(d_offsets, torch.int64, "offsets")
    _dev(d_row_ptr, torch.int64, "row_ptr"); _dev(d_col, torch.int32, "col"); _dev(d_draws, torch.int32, "draws")
    n = d_su.numel()
    T = 2 * int(d_offsets[-1].item())
    rows = torch.empty((max(T, 1), 3), dtype=torch.int32, device=d_su.device)
    L.check(L.lib().drb_sgns_explode(_ptr(d_su), _ptr(d_si), n, window, _ptr(d_offsets), _ptr(d_row_ptr), _ptr(d_col),
                                     _ptr(d_draws), _ptr(rows), _stream()))
    return rows[:T]


# ------------------------------------------------------------------ CSR / adjacency builders
def csr_build(d_row, d_col, n_rows, n_cols):
    """COO int32 pairs on the device -> (row_ptr int64[n_rows+1], col int32[nnz_unique]) sorted + duplicate-free."""
    _dev(d_row, torch.int32, "row"); _dev(d_col, torch.int32, "col")
    nnz = d_row.numel()
    ws = torch.empty(L.lib().drb_csr_workspace_bytes(n_rows, nnz), dtype=torch.uint8, device=d_row.device)
    row_ptr = torch.empty(n_rows + 1, dtype=torch.int64, device=d_row.device)
    col = torch.empty(max(nnz, 1), dtype=torch.int32, device=d_row.device)
    kept = C.c_int64(0)
    L.check(L.lib().drb_csr_build(_ptr(d_row), _ptr(d_col), nnz, n_rows, n_cols, _ptr(ws), _ptr(row_ptr), _ptr(col),
                                  C.byref(kept), _stream()))
    return row_ptr, col[:kept.value]


def lgcn_build_adj(d_coo_u, d_coo_i, user_num, item_num):
    """Train COO on the device -> A_hat CSR (row_ptr i64, col i32, val f32) of get_norm_adj_mat, built on the device."""
    ui_ptr, ui_col = csr_build(d_coo_u, d_coo_i, user_num, item_num)
    iu_ptr, iu_col = csr_build(d_coo_i, d_coo_u, item_num, user_num)
    nnz = ui_col.numel()
    assert iu_col.numel() == nnz
    dev = d_coo_u.device
    adj_ptr = torch.empty(user_num + item_num + 1, dtype=torch.int64, device=dev)
    adj_col = torch.empty(max(2 * nnz, 1), dtype=torch.int32, device=dev)
    adj_val = torch.empty(max(2 * nnz, 1), dtype=torch.float32, device=dev)
    L.check(L.lib().drb_lgcn_build_adj(_ptr(ui_ptr), _ptr(ui_col), _ptr(iu_ptr), _ptr(iu_col), user_num, item_num, nnz,
                                       _ptr(adj_ptr), _ptr(adj_col), _ptr(adj_val), _stream()))
    return adj_ptr, adj_col[:2 * nnz], adj_val[:2 * nnz]


# ------------------------------------------------------------------ evaluation KPIs
def rank_metrics(d_preds, d_gt_ptr, d_gt_idx, ks, item_num, d_item_pop=None):
    """calc_ranking_results' numbers for rank()'s device output: -> float64 CUDA tensor [len(ks), 8] (L.KPI_NAMES)."""
    _dev(d_preds, torch.float32, "preds"); _dev(d_gt_ptr, torch.int64, "gt_ptr"); _dev(d_gt_idx, torch.int32, "gt_idx")
    if d_item_pop is not None:
        _dev(d_item_pop, torch.float64, "item_pop")
    ks = np.ascontiguousarray(ks, np.int32)
    n, ld = d_preds.shape
    ws = torch.empty(L.lib().drb_rank_metrics_workspace_bytes(item_num, len(ks)), dtype=torch.uint8, device=d_preds.device)
    out = torch.empty((len(ks), len(L.KPI_NAMES)), dtype=torch.float64, device=d_preds.device)
    L.check(L.lib().drb_rank_metrics(_ptr(d_preds), n, ld, _ptr(d_gt_ptr), _ptr(d_gt_idx), ks.ctypes.data, len(ks),
                                     item_num, None if d_item_pop is None else _ptr(d_item_pop), _ptr(ws), _ptr(out),
                                     _stream()))
    return out


def rank_metrics_host(preds, gt_ptr, gt_idx, ks, item_num, item_pop=None):
    """Same through host buffers (H2D/D2H inside the library) -> float64 numpy [len(ks), 8]."""
    preds = np.ascontiguousarray(preds, np.float32)
    gt_ptr = np.ascontiguousarray(gt_ptr, np.int64)
    gt_idx = np.ascontiguousarray(gt_idx, np.int32)
    ks = np.ascontiguousarray(ks, np.int32)
    pop = None if item_pop is None else np.ascontiguousarray(item_pop, np.float64)
    out = np.empty((len(ks), len(L.KPI_NAMES)), np.float64)
    L.check(L.lib().drb_rank_metrics_host(preds.ctypes.data, preds.shape[0], preds.shape[1], gt_ptr.ctypes.data,
                                          gt_idx.ctypes.data, ks.ctypes.data, len(ks), item_num,
                                          None if pop is None else pop.ctypes.data, out.ctypes.data))
    return out


# ------------------------------------------------------------------ epoch permutation
def mt19937_stream(seed, n, device):
    out = torch.empty(max(n, 1), dtype=torch.int32, device=device)
    L.check(L.lib().drb_mt19937_stream(C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), n, _ptr(out), _stream()))
    return out[:n]


def mt19937_stream_variant(n):
    """'segmented' when drb_mt19937_stream runs the many-CTA jump-ahead kernel for n words (after its one-off device check),
    'one-cta' otherwise."""
    return "segmented" if L.lib().drb_mt19937_stream_variant(int(n)) else "one-cta"


def randperm_workspace(n, device):
    """(perm int64 [n], scratch) for randperm_torch(out=...): lets a caller keep them across epochs."""
    return (torch.empty(max(n, 1), dtype=torch.int64, device=device),
            torch.empty(L.lib().drb_randperm_workspace_bytes(n), dtype=torch.uint8, device=device))


def randperm_torch(seed, n, device, out=None):
    """torch.randperm(n, generator=G) for a CPU generator G with G.manual_seed(seed) -- computed on the device, bit-exact."""
    perm, ws = out if out is not None else randperm_workspace(n, device)
    L.check(L.lib().drb_randperm_torch(C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), n, _ptr(perm), _ptr(ws), _stream()))
    return perm[:n]


# ------------------------------------------------------------------ train feed
def gather_triples(d_triples, d_perm=None):
    _dev(d_triples, torch.int32, "triples")
    n = d_triples.shape[0] if d_perm is None else d_perm.numel()
    if d_perm is not None:
        _dev(d_perm, torch.int64, "perm")
    n4 = (n + 3) // 4 * 4                                   # 16-byte aligned planes for the TMA path
    soa = torch.empty((3, n4), dtype=torch.int32, device=d_triples.device)
    L.check(L.lib().drb_gather_triples(_ptr(d_triples), None if d_perm is None else _ptr(d_perm), n, _ptr(soa[0]),
                                       _ptr(soa[1]), _ptr(soa[2]), _stream()))
    return soa[0][:n], soa[1][:n], soa[2][:n]


# ------------------------------------------------------------------ training
def _check_step(rc):
    """A NaN / infinite loss raises ValueError, as the reference's fit() does; any other failure DrbError."""
    if rc == L.DRB_ERR_NAN_LOSS:
        raise ValueError("Loss=Nan or Infinity: current settings does not fit the recommender")
    L.check(rc)


class MFWorkspace:
    """Device scratch of the step kernel: gradient accumulators, row counters, optimiser state (Adam m, v; Adagrad /
    RMSprop one table)."""

    def __init__(self, user_num, item_num, factors, opt, device, deterministic=False):
        self.U, self.I, self.F = user_num, item_num, factors
        self.opt = L.OPT_KIND[opt]
        self.det = bool(deterministic)
        nbytes = (L.lib().drb_mf_workspace_bytes_det if self.det else L.lib().drb_mf_workspace_bytes)(user_num, item_num, factors,
                                                                                                     self.opt)
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        self.reset()

    def reset(self):
        if self.det:
            self.buf.zero_()               # the int64 images behind the regular layout as well
        else:
            L.check(L.lib().drb_mf_workspace_init(_ptr(self.buf), self.U, self.I, self.F, self.opt, _stream()))


def mf_bpr_train_steps(P, Q, ws, bu, bi, bj, batch, first_step, n_steps, hp, adam_step0=0, check=True, out=None):
    _dev(P, torch.float32, "P"); _dev(Q, torch.float32, "Q")
    for t, nm in ((bu, "bu"), (bi, "bi"), (bj, "bj")):
        _dev(t, torch.int32, nm)
    n = bu.numel()
    losses = out if out is not None else torch.empty(max(n_steps, 1), dtype=torch.float64, device=P.device)
    nan_step = C.c_int64(-1)
    fn = L.lib().drb_mf_bpr_train_steps_det if getattr(ws, "det", False) else L.lib().drb_mf_bpr_train_steps
    rc = fn(_ptr(P), _ptr(Q), _ptr(ws.buf), ws.U, ws.I, ws.F, _ptr(bu), _ptr(bi), _ptr(bj), n, batch, first_step, n_steps,
            C.byref(hp), adam_step0, _ptr(losses), 1 if check else 0, C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


def mf_bpr_train_steps_fused_neg(P, Q, ws, bu, bi, d_row_ptr, d_col, seed, batch, first_step, n_steps, hp, adam_step0=0,
                                 neg_out=None, check=True):
    """Throughput mode: negatives are drawn inside the step kernel (fresh per triple and step) from the complement of the
    user's CSR row.  neg_out (optional int32 [n]) receives them."""
    _dev(P, torch.float32, "P"); _dev(Q, torch.float32, "Q"); _dev(bu, torch.int32, "bu"); _dev(bi, torch.int32, "bi")
    _dev(d_row_ptr, torch.int64, "row_ptr"); _dev(d_col, torch.int32, "col")
    losses = torch.empty(max(n_steps, 1), dtype=torch.float64, device=P.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_mf_bpr_train_steps_fused_neg(_ptr(P), _ptr(Q), _ptr(ws.buf), ws.U, ws.I, ws.F, _ptr(bu), _ptr(bi),
                                                  _ptr(d_row_ptr), _ptr(d_col), C.c_uint64(seed),
                                                  None if neg_out is None else _ptr(neg_out), bu.numel(), batch, first_step,
                                                  n_steps, C.byref(hp), adam_step0, _ptr(losses), 1 if check else 0,
                                                  C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


def mf_bpr_loss(P, Q, ws, bu, bi, bj, hp):
    _dev(P, torch.float32, "P"); _dev(Q, torch.float32, "Q")
    loss = torch.empty(1, dtype=torch.float64, device=P.device)
    L.check(L.lib().drb_mf_bpr_loss(_ptr(P), _ptr(Q), _ptr(ws.buf), ws.U, ws.I, ws.F, _ptr(bu), _ptr(bi), _ptr(bj),
                                    bu.numel(), C.byref(hp), _ptr(loss), _stream()))
    return loss


def stage_buffer(batch, device):
    stride = (batch + 3) // 4 * 4
    return torch.empty(3 * stride + 4, dtype=torch.int32, device=device)


def mf_bpr_train_step_host(P, Q, ws, h_bu, h_bi, h_bj, hp, stage, adam_step0=0):
    """One end-to-end step from HOST batch arrays (numpy int32 or CPU tensors, ideally pinned)."""
    def hp_(a):
        return a.data_ptr() if isinstance(a, torch.Tensor) else a.ctypes.data
    n = len(h_bu)
    loss = C.c_double(0.0)
    rc = L.lib().drb_mf_bpr_train_step_host(_ptr(P), _ptr(Q), _ptr(ws.buf), ws.U, ws.I, ws.F, hp_(h_bu), hp_(h_bi),
                                            hp_(h_bj), n, C.byref(hp), adam_step0, _ptr(stage), C.byref(loss), _stream())
    _check_step(rc)
    return loss.value


def mf_bpr_train_steps_host(P, Q, ws, h_bu, h_bi, h_bj, batch, n_steps, hp, adam_step0=0):
    """Pipelined end-to-end steps from pinned HOST planes (CPU int32 tensors).  Returns float64 losses [n_steps]."""
    for t in (h_bu, h_bi, h_bj):
        if not (isinstance(t, torch.Tensor) and not t.is_cuda and t.dtype == torch.int32 and t.is_contiguous()):
            raise TypeError("host planes must be contiguous CPU int32 tensors (pin them for overlap)")
    n = h_bu.numel()
    stride = (batch + 3) // 4 * 4
    stage = torch.empty(2 * 3 * stride, dtype=torch.int32, device=P.device)
    d_loss = torch.empty(max(1, n_steps), dtype=torch.float64, device=P.device)
    h_loss = torch.empty(max(1, n_steps), dtype=torch.float64).pin_memory()
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_mf_bpr_train_steps_host(_ptr(P), _ptr(Q), _ptr(ws.buf), ws.U, ws.I, ws.F, h_bu.data_ptr(),
                                             h_bi.data_ptr(), h_bj.data_ptr(), n, batch, n_steps, C.byref(hp), adam_step0,
                                             _ptr(stage), _ptr(d_loss), h_loss.data_ptr(), C.byref(nan_step), _stream())
    _check_step(rc)
    return h_loss[:n_steps]


# ------------------------------------------------------------------ FM
class FMWorkspace:
    """MF workspace + gradient accumulator / optimiser state of the packed bias vector."""

    def __init__(self, user_num, item_num, factors, opt, device):
        self.U, self.I, self.F = user_num, item_num, factors
        self.opt = L.OPT_KIND[opt]
        self.buf = torch.empty(L.lib().drb_fm_workspace_bytes(user_num, item_num, factors, self.opt), dtype=torch.uint8,
                               device=device)
        L.check(L.lib().drb_fm_workspace_init(_ptr(self.buf), user_num, item_num, factors, self.opt, _stream()))


def fm_train_steps(P, Q, bias, ws, bu, bi, bj, batch, first_step, n_steps, hp, adam_step0=0, apply=True, check=True):
    _dev(P, torch.float32, "P"); _dev(Q, torch.float32, "Q"); _dev(bias, torch.float32, "bias")
    for t, nm in ((bu, "bu"), (bi, "bi"), (bj, "bj")):
        _dev(t, torch.int32, nm)
    if bias.numel() != ws.U + ws.I + 1:
        raise ValueError("bias must hold user_num + item_num + 1 floats")
    losses = torch.empty(max(n_steps, 1), dtype=torch.float64, device=P.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_fm_train_steps(_ptr(P), _ptr(Q), _ptr(bias), _ptr(ws.buf), ws.U, ws.I, ws.F, _ptr(bu), _ptr(bi), _ptr(bj),
                                    bu.numel(), batch, first_step, n_steps, C.byref(hp), adam_step0, 1 if apply else 0,
                                    _ptr(losses), 1 if check else 0, C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


def fm_rank(P, Q, bias, users, cands, topk):
    _dev(users, torch.int64, "users"); _dev(cands, torch.int64, "cands"); _dev(bias, torch.float32, "bias")
    n, Cn = cands.shape
    out = torch.empty((n, topk), dtype=torch.float32, device=P.device)
    L.check(L.lib().drb_fm_rank(_ptr(P), _ptr(Q), _ptr(bias), P.shape[0], Q.shape[0], P.shape[1], _ptr(users), n, _ptr(cands),
                                Cn, topk, _ptr(out), _stream()))
    return out


def fm_full_rank(P, Q, bias, users, topk):
    _dev(users, torch.int64, "users"); _dev(bias, torch.float32, "bias")
    out = torch.empty((users.numel(), topk), dtype=torch.int64, device=P.device)
    L.check(L.lib().drb_fm_full_rank(_ptr(P), _ptr(Q), _ptr(bias), P.shape[0], Q.shape[0], P.shape[1], _ptr(users),
                                     users.numel(), topk, _ptr(out), _stream()))
    return out


def fm_predict(P, Q, bias, u, i):
    _dev(u, torch.int32, "u"); _dev(i, torch.int32, "i"); _dev(bias, torch.float32, "bias")
    out = torch.empty(u.numel(), dtype=torch.float32, device=P.device)
    L.check(L.lib().drb_fm_predict(_ptr(P), _ptr(Q), _ptr(bias), P.shape[0], Q.shape[0], P.shape[1], _ptr(u), _ptr(i),
                                   u.numel(), _ptr(out), _stream()))
    return out


# ------------------------------------------------------------------ Item2Vec
class Item2VecWorkspace:
    """Step-kernel scratch of the shared item table: accumulator, row counters and optimiser state of the item rows."""

    def __init__(self, item_num, factors, opt, device):
        self.I, self.F = item_num, factors
        self.opt = L.OPT_KIND[opt]
        self.buf = torch.empty(L.lib().drb_item2vec_workspace_bytes(item_num, factors, self.opt), dtype=torch.uint8,
                               device=device)
        L.check(L.lib().drb_item2vec_workspace_init(_ptr(self.buf), item_num, factors, self.opt, _stream()))


def item2vec_train_steps(Q, ws, bt, bc, blabel, batch, first_step, n_steps, hp, adam_step0=0, apply=True, check=True):
    """Steps of BCEWithLogitsLoss(sum) on (target, context, label) planes, both rows from the one table Q -> float64 losses."""
    _dev(Q, torch.float32, "Q")
    for t, nm in ((bt, "target"), (bc, "context"), (blabel, "label")):
        _dev(t, torch.int32, nm)
    losses = torch.empty(max(n_steps, 1), dtype=torch.float64, device=Q.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_item2vec_train_steps(_ptr(Q), _ptr(ws.buf), ws.I, ws.F, _ptr(bt), _ptr(bc), _ptr(blabel), bt.numel(),
                                          batch, first_step, n_steps, C.byref(hp), adam_step0, 1 if apply else 0,
                                          _ptr(losses), 1 if check else 0, C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


def item2vec_user_embed(d_row_ptr, d_col, Q, P):
    """P[u] = sum of Q over user u's train CSR row, for every user whose row is not empty (in place)."""
    _dev(d_row_ptr, torch.int64, "row_ptr"); _dev(d_col, torch.int32, "col")
    _dev(Q, torch.float32, "Q"); _dev(P, torch.float32, "P")
    L.check(L.lib().drb_item2vec_user_embed(_ptr(d_row_ptr), _ptr(d_col), _ptr(Q), P.shape[0], P.shape[1], _ptr(P),
                                            _stream()))
    return P


# ------------------------------------------------------------------ inference
def mf_rank(P, Q, users, cands, topk):
    _dev(users, torch.int64, "users"); _dev(cands, torch.int64, "cands")
    n, Cn = cands.shape
    out = torch.empty((n, topk), dtype=torch.float32, device=P.device)
    L.check(L.lib().drb_mf_rank(_ptr(P), _ptr(Q), P.shape[1], _ptr(users), n, _ptr(cands), Cn, topk, _ptr(out),
                                _stream()))
    return out


def mf_full_rank(P, Q, users, topk):
    _dev(users, torch.int64, "users")
    out = torch.empty((users.numel(), topk), dtype=torch.int64, device=P.device)
    L.check(L.lib().drb_mf_full_rank(_ptr(P), _ptr(Q), P.shape[1], Q.shape[0], _ptr(users), users.numel(), topk,
                                     _ptr(out), _stream()))
    return out


def mf_predict(P, Q, u, i):
    _dev(u, torch.int32, "u"); _dev(i, torch.int32, "i")
    out = torch.empty(u.numel(), dtype=torch.float32, device=P.device)
    L.check(L.lib().drb_mf_predict(_ptr(P), _ptr(Q), P.shape[1], _ptr(u), _ptr(i), u.numel(), _ptr(out), _stream()))
    return out


def mf_rank_host(P, Q, users, cands, topk):
    users = np.ascontiguousarray(users, np.int64)
    cands = np.ascontiguousarray(cands, np.int64)
    out = np.empty((len(users), topk), np.float32)
    L.check(L.lib().drb_mf_rank_host(_ptr(P), _ptr(Q), P.shape[1], users.ctypes.data, len(users), cands.ctypes.data,
                                     cands.shape[1], topk, out.ctypes.data))
    return out


# ------------------------------------------------------------------ LightGCN
def lgcn_norm_adj(coo_u, coo_i, user_num, item_num):
    """get_norm_adj_mat (LightGCNRecommender.py:73-107) as CSR over the U+I nodes, values bit-identical to the
    reference: float64 (deg + 1e-7) ** -0.5, (D*A)*D in float64, cast to fp32.  One-off host build (numpy)."""
    n = user_num + item_num
    u = np.asarray(coo_u, np.int64)
    i = np.asarray(coo_i, np.int64) + user_num
    key = np.unique(np.concatenate([u * n + i, i * n + u]))
    row, col = key // n, key % n
    cnt = np.bincount(row, minlength=n)
    dinv = np.power(cnt.astype(np.float64) + 1e-7, -0.5)
    val = ((dinv[row] * 1.0) * dinv[col]).astype(np.float32)
    row_ptr = np.zeros(n + 1, np.int64)
    np.cumsum(cnt, out=row_ptr[1:])
    return row_ptr, col.astype(np.int32), val


class LgcnGraph:
    """Device copy of the normalised adjacency + its segment list."""

    def __init__(self, row_ptr, col, val, device):
        d_row_ptr = d_col = d_val = None
        if isinstance(row_ptr, torch.Tensor):                    # lgcn_build_adj's device arrays: only the segment
            d_row_ptr, d_col, d_val = row_ptr, col, val          # list is derived on the host (from row_ptr)
            row_ptr = row_ptr.cpu().numpy()
        n = len(row_ptr) - 1
        row_ptr = np.ascontiguousarray(row_ptr, np.int64)
        nseg = int(L.lib().drb_lgcn_segment_count(row_ptr.ctypes.data, n))
        seg_row = np.empty(max(1, nseg), np.int32)
        seg_ptr = np.empty(nseg + 1, np.int64)
        L.check(L.lib().drb_lgcn_segments(row_ptr.ctypes.data, n, seg_row.ctypes.data, seg_ptr.ctypes.data))
        self.n, self.nseg = n, nseg
        if d_row_ptr is not None:
            self.row_ptr, self.col, self.val = d_row_ptr.to(device), d_col.to(device), d_val.to(device)
        else:
            self.row_ptr = torch.from_numpy(row_ptr).to(device)
            self.col = torch.from_numpy(np.ascontiguousarray(col, np.int32)).to(device)
            self.val = torch.from_numpy(np.ascontiguousarray(val, np.float32)).to(device)
        self.seg_row = torch.from_numpy(seg_row).to(device)
        self.seg_ptr = torch.from_numpy(seg_ptr).to(device)

    def args(self):
        return (_ptr(self.row_ptr), _ptr(self.col), _ptr(self.val), _ptr(self.seg_row), _ptr(self.seg_ptr), self.nseg)


class LgcnWorkspace:
    def __init__(self, user_num, item_num, factors, opt, device):
        self.U, self.I, self.F = user_num, item_num, factors
        self.opt = L.OPT_SGD if opt == "sgd" else L.OPT_ADAM
        self.buf = torch.empty(L.lib().drb_lgcn_workspace_bytes(user_num, item_num, factors, self.opt), dtype=torch.uint8,
                               device=device)
        L.check(L.lib().drb_lgcn_workspace_init(_ptr(self.buf), user_num, item_num, factors, self.opt, _stream()))


def lgcn_propagate(E0, ws, graph, num_layers, out=None):
    _dev(E0, torch.float32, "E0")
    Em = out if out is not None else torch.empty_like(E0)
    L.check(L.lib().drb_lgcn_propagate(_ptr(E0), _ptr(ws.buf), ws.U, ws.I, ws.F, num_layers, *graph.args(), _ptr(Em),
                                       _stream()))
    return Em


def lgcn_bpr_train_steps(E0, ws, graph, num_layers, bu, bi, bj, batch, first_step, n_steps, hp, adam_step0=0, apply=True,
                         check=True):
    _dev(E0, torch.float32, "E0")
    for t, nm in ((bu, "bu"), (bi, "bi"), (bj, "bj")):
        _dev(t, torch.int32, nm)
    losses = torch.empty(max(1, n_steps), dtype=torch.float64, device=E0.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_lgcn_bpr_train_steps(_ptr(E0), _ptr(ws.buf), ws.U, ws.I, ws.F, num_layers, *graph.args(), _ptr(bu),
                                          _ptr(bi), _ptr(bj), bu.numel(), batch, first_step, n_steps, C.byref(hp),
                                          adam_step0, 1 if apply else 0, _ptr(losses), 1 if check else 0,
                                          C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


# ------------------------------------------------------------------ NGCF
def _dims_arr(dims):
    return (C.c_int32 * len(dims))(*[int(d) for d in dims])


def ngcf_param_count(dims):
    return int(L.lib().drb_ngcf_param_count(_dims_arr(dims), len(dims) - 1))


class NgcfWorkspace:
    def __init__(self, user_num, item_num, dims, opt, device):
        self.U, self.I, self.dims = user_num, item_num, [int(d) for d in dims]
        self.opt = L.OPT_SGD if opt == "sgd" else L.OPT_ADAM
        nbytes = L.lib().drb_ngcf_workspace_bytes(user_num, item_num, _dims_arr(self.dims), len(self.dims) - 1, self.opt)
        if nbytes == 0:
            raise ValueError("NGCF: layer widths must be in 1..256 and 1 <= layers <= 8")
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        L.check(L.lib().drb_ngcf_workspace_init(_ptr(self.buf), user_num, item_num, _dims_arr(self.dims), len(self.dims) - 1,
                                                self.opt, _stream()))


def ngcf_keep_bytes(ws):
    """bytes of dropout masks one forward() consumes: one per element of every layer output."""
    return (ws.U + ws.I) * sum(ws.dims[1:])


def ngcf_forward(E0, W, ws, graph, tower_dtype=0, dropout=0.0, keep=None):
    """keep (with mess_dropout > 0): uint8 CUDA tensor, the masks torch's nn.Dropout draws per layer, layers concatenated."""
    _dev(E0, torch.float32, "E0"); _dev(W, torch.float32, "W")
    if keep is not None:
        _dev(keep, torch.uint8, "keep")
        if keep.numel() != ngcf_keep_bytes(ws):
            raise ValueError("keep must hold (user_num + item_num) x sum(hidden widths) bytes")
    out = torch.empty((ws.U + ws.I, sum(ws.dims)), dtype=torch.float32, device=E0.device)
    L.check(L.lib().drb_ngcf_forward(_ptr(E0), _ptr(W), _ptr(ws.buf), ws.U, ws.I, _dims_arr(ws.dims), len(ws.dims) - 1,
                                             *graph.args(), tower_dtype, None if keep is None else _ptr(keep),
                                             C.c_float(dropout if keep is not None else 0.0), _ptr(out), _stream()))
    return out


def ngcf_bpr_train_steps(E0, W, ws, graph, bu, bi, bj, batch, first_step, n_steps, hp, adam_step0=0, apply=True, check=True,
                         tower_dtype=0, dropout=0.0, keep=None):
    _dev(E0, torch.float32, "E0"); _dev(W, torch.float32, "W")
    for t, nm in ((bu, "bu"), (bi, "bi"), (bj, "bj")):
        _dev(t, torch.int32, nm)
    if keep is not None:
        _dev(keep, torch.uint8, "keep")
        if keep.numel() != max(1, n_steps) * ngcf_keep_bytes(ws):
            raise ValueError("keep must hold n_steps x (user_num + item_num) x sum(hidden widths) bytes")
    losses = torch.empty(max(1, n_steps), dtype=torch.float64, device=E0.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_ngcf_bpr_train_steps(_ptr(E0), _ptr(W), _ptr(ws.buf), ws.U, ws.I, _dims_arr(ws.dims), len(ws.dims) - 1,
                                                  *graph.args(), _ptr(bu), _ptr(bi), _ptr(bj), bu.numel(), batch, first_step,
                                                  n_steps, C.byref(hp), adam_step0, 1 if apply else 0, tower_dtype,
                                                  None if keep is None else _ptr(keep),
                                                  C.c_float(dropout if keep is not None else 0.0), _ptr(losses),
                                                  1 if check else 0, C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


# ------------------------------------------------------------------ NFM
NFM_ACT = {"relu": 0, "sigmoid": 1, "tanh": 2}


def nfm_param_count(factors, num_layers, batch_norm):
    return int(L.lib().drb_nfm_param_count(factors, num_layers, 1 if batch_norm else 0))


class NfmWorkspace:
    def __init__(self, user_num, item_num, factors, num_layers, batch_norm, opt, max_rows, device):
        self.U, self.I, self.F, self.Ln, self.bn, self.max_rows = user_num, item_num, factors, num_layers, 1 if batch_norm else 0, int(max_rows)
        self.opt = L.OPT_SGD if opt == "sgd" else L.OPT_ADAM
        nbytes = L.lib().drb_nfm_workspace_bytes(user_num, item_num, factors, num_layers, self.bn, self.opt, self.max_rows)
        if nbytes == 0:
            raise ValueError("NFM: factors must be in 1..256, 0 <= num_layers <= 8 and max_rows >= 2")
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        L.check(L.lib().drb_nfm_workspace_init(_ptr(self.buf), user_num, item_num, factors, num_layers, self.bn, self.opt,
                                               self.max_rows, _stream()))


def nfm_bpr_train_steps(P, Q, bias, N, Rs, ws, act, bu, bi, bj, batch, first_step, n_steps, hp, adam_step0=0, apply=True,
                        check=True, tower_dtype=0, dropout=0.0, keep=None):
    """keep (with dropout > 0): uint8 CUDA tensor of the masks torch's Dropout modules draw, per step
    [forward call][site][batch][F] (drb_nfm_bpr_train_steps)."""
    for t in (P, Q, bias, N):
        _dev(t, torch.float32, "parameter")
    for t, nm in ((bu, "bu"), (bi, "bi"), (bj, "bj")):
        _dev(t, torch.int32, nm)
    if keep is not None:
        _dev(keep, torch.uint8, "keep")
        rows = batch if n_steps != 1 else min(batch, bu.numel() - first_step * batch)
        if keep.numel() != max(1, n_steps) * 2 * (1 + ws.Ln) * rows * ws.F:
            raise ValueError("keep must hold n_steps x 2 x (1 + num_layers) x batch x factors bytes")
    losses = torch.empty(max(1, n_steps), dtype=torch.float64, device=P.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_nfm_bpr_train_steps(
        _ptr(P), _ptr(Q), _ptr(bias), _ptr(N), None if Rs is None or Rs.numel() == 0 else _ptr(Rs), _ptr(ws.buf), ws.U, ws.I, ws.F,
        ws.Ln, ws.bn, act, ws.max_rows, _ptr(bu), _ptr(bi), _ptr(bj), bu.numel(), batch, first_step, n_steps, C.byref(hp), adam_step0,
        1 if apply else 0, tower_dtype, None if keep is None else _ptr(keep), C.c_float(dropout if keep is not None else 0.0),
        _ptr(losses), 1 if check else 0, C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


def nfm_scores(P, Q, bias, N, Rs, ws, act, u, i, tower_dtype=0):
    """eval-mode scores of the (u[k], i[k]) pairs (int32 CUDA tensors)."""
    _dev(u, torch.int32, "u"); _dev(i, torch.int32, "i")
    out = torch.empty(u.numel(), dtype=torch.float32, device=P.device)
    L.check(L.lib().drb_nfm_scores(_ptr(P), _ptr(Q), _ptr(bias), _ptr(N), None if Rs is None or Rs.numel() == 0 else _ptr(Rs),
                                   _ptr(ws.buf), ws.U, ws.I, ws.F, ws.Ln, ws.bn, act, ws.opt, ws.max_rows, _ptr(u), _ptr(i),
                                   u.numel(), tower_dtype, _ptr(out), _stream()))
    return out


# ------------------------------------------------------------------ Multi-VAE
def _hidden_arr(hidden):
    arr = (C.c_int32 * max(1, len(hidden)))(*[int(h) for h in hidden])
    return arr, len(hidden)


def vae_param_count(item_num, hidden, latent_dim):
    arr, n = _hidden_arr(hidden)
    return int(L.lib().drb_vae_param_count(item_num, arr, n, latent_dim))


class VaeWorkspace:
    def __init__(self, item_num, hidden, latent_dim, opt, max_rows, device):
        self.I, self.hidden, self.lat, self.max_rows = item_num, [int(h) for h in hidden], int(latent_dim), int(max_rows)
        self.opt = L.OPT_SGD if opt == "sgd" else L.OPT_ADAM
        self._arr, self.Ln = _hidden_arr(self.hidden)
        nbytes = L.lib().drb_vae_workspace_bytes(item_num, self._arr, self.Ln, self.lat, self.opt, self.max_rows)
        if nbytes == 0:
            raise ValueError("VAECF: item_num > 0, at most 8 positive hidden sizes, latent_dim >= 2 and max_rows >= 1")
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        L.check(L.lib().drb_vae_workspace_init(_ptr(self.buf), item_num, self._arr, self.Ln, self.lat, self.opt, self.max_rows,
                                               _stream()))


class VaeRatings:
    """The rating rows as a device CSR: row_ptr int64 [U+1], col int32, val float32 (duplicate-free, no zeros)."""

    def __init__(self, row_ptr, col, val):
        self.row_ptr = _dev(row_ptr, torch.int64, "row_ptr")
        self.col = _dev(col, torch.int32, "col") if col.numel() else torch.zeros(1, dtype=torch.int32, device=row_ptr.device)
        self.val = _dev(val, torch.float32, "val") if val.numel() else torch.zeros(1, dtype=torch.float32, device=row_ptr.device)
        self.U = row_ptr.numel() - 1

    def args(self):
        return _ptr(self.row_ptr), _ptr(self.col), _ptr(self.val), self.U


def vae_train_steps(N, ws, R, users, batch, first_step, n_steps, hp, adam_step0=0, apply=True, training=True, tower_dtype=0,
                    dropout=0.0, keep=None, eps=None, seed=0, anneal_cap=0.2, total_anneal_steps=0, update0=0, check=True):
    """keep: int32 CUDA tensor of bit-packed torch keep-masks (ceil(batch * item_num / 32) words per step) or None (Philox);
    eps: float32 CUDA tensor [n_steps, batch, latent_dim // 2] or None (Philox).  -> float64 losses [n_steps]."""
    _dev(N, torch.float32, "N"); _dev(users, torch.int32, "users")
    if keep is not None:
        _dev(keep, torch.int32, "keep")
        if keep.numel() < n_steps * ((batch * ws.I + 31) // 32):
            raise ValueError("keep too short for n_steps batches")
    if eps is not None:
        _dev(eps, torch.float32, "eps")
        last = min(batch, users.numel() - (first_step + n_steps - 1) * batch)
        if eps.numel() < ((n_steps - 1) * batch + last) * (ws.lat // 2):
            raise ValueError("eps too short for n_steps batches")
    losses = torch.empty(max(1, n_steps), dtype=torch.float64, device=N.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_vae_train_steps(_ptr(N), _ptr(ws.buf), ws.I, ws._arr, ws.Ln, ws.lat, ws.max_rows, *R.args(), _ptr(users),
                                     users.numel(), batch, first_step, n_steps, C.byref(hp), adam_step0, 1 if apply else 0,
                                     1 if training else 0, tower_dtype, C.c_float(dropout),
                                     None if keep is None else _ptr(keep), None if eps is None else _ptr(eps),
                                     C.c_uint64(seed), C.c_double(anneal_cap), int(total_anneal_steps), int(update0),
                                     _ptr(losses), 1 if check else 0, C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


VAE_OUT = {"scores": 0, "hidden": 1, "latent": 2}


def vae_forward(N, ws, R, users, what="scores", tower_dtype=0):
    """eval-mode forward for int32 CUDA user ids: 'scores' [n, item_num], 'hidden' (last decoder hidden) or 'latent'
    (encoder output: mu, logvar)."""
    _dev(N, torch.float32, "N"); _dev(users, torch.int32, "users")
    width = {"scores": ws.I, "hidden": ws.hidden[0] if ws.hidden else ws.lat // 2, "latent": ws.lat}[what]
    out = torch.empty((users.numel(), width), dtype=torch.float32, device=N.device)
    L.check(L.lib().drb_vae_forward(_ptr(N), _ptr(ws.buf), ws.I, ws._arr, ws.Ln, ws.lat, ws.opt, ws.max_rows, *R.args(),
                                    _ptr(users), users.numel(), VAE_OUT[what], tower_dtype, _ptr(out), _stream()))
    return out


def vae_candidate_scores(N, ws, hidden_rows, cands):
    """decoder output at the candidates only: hidden_rows [n, K] from vae_forward(.., 'hidden'), cands int64 [n, C]."""
    _dev(hidden_rows, torch.float32, "hidden_rows"); _dev(cands, torch.int64, "cands")
    n, Cn = cands.shape
    out = torch.empty((n, Cn), dtype=torch.float32, device=N.device)
    L.check(L.lib().drb_vae_candidate_scores(_ptr(N), ws.I, ws._arr, ws.Ln, ws.lat, _ptr(hidden_rows), n, _ptr(cands), Cn,
                                             _ptr(out), _stream()))
    return out


# ------------------------------------------------------------------ NeuMF
NEUMF_MODE = {"NeuMF": 0, "NeuMF-pre": 0, "GMF": 1, "MLP": 2}       # config['model_name'] (NeuMFRecommender.py:48-50)


def neumf_param_count(factors, num_layers, mode=0):
    return int(L.lib().drb_neumf_param_count(factors, num_layers, mode))


def neumf_mask_words(factors, num_layers, batch):
    return int(L.lib().drb_neumf_mask_words(factors, num_layers, batch))


class NeumfWorkspace:
    def __init__(self, user_num, item_num, factors, num_layers, opt, max_rows, device):
        self.U, self.I, self.F, self.Ln, self.max_rows = user_num, item_num, factors, num_layers, int(max_rows)
        self.opt = L.OPT_SGD if opt == "sgd" else L.OPT_ADAM
        nbytes = L.lib().drb_neumf_workspace_bytes(user_num, item_num, factors, num_layers, self.opt, self.max_rows)
        if nbytes == 0:
            raise ValueError("NeuMF: factors must be a positive multiple of 4 and 1 <= num_layers <= 8")
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        L.check(L.lib().drb_neumf_workspace_init(_ptr(self.buf), user_num, item_num, factors, num_layers, self.opt,
                                                 self.max_rows, _stream()))


def neumf_bpr_train_steps(tabs, W, ws, bu, bi, bj, batch, first_step, n_steps, hp, adam_step0=0, apply=True, check=True,
                          tower_dtype=0, dropout=0.0, dropout_seed=0, drop_masks=None, mode=0):
    """drop_masks: int32 CUDA tensor [n_steps * neumf_mask_words(F, L, batch)] of host-generated keep-masks (parity mode)."""
    if drop_masks is not None:
        _dev(drop_masks, torch.int32, "drop_masks")
        if drop_masks.numel() < n_steps * neumf_mask_words(ws.F, ws.Ln, batch):
            raise ValueError("drop_masks too short for n_steps batches")
    for t in list(tabs) + [W]:
        _dev(t, torch.float32, "table")
    for t, nm in ((bu, "bu"), (bi, "bi"), (bj, "bj")):
        _dev(t, torch.int32, nm)
    losses = torch.empty(max(1, n_steps), dtype=torch.float64, device=W.device)
    nan_step = C.c_int64(-1)
    rc = L.lib().drb_neumf_bpr_train_steps(_ptr(tabs[0]), _ptr(tabs[1]), _ptr(tabs[2]), _ptr(tabs[3]), _ptr(W), _ptr(ws.buf),
                                           ws.U, ws.I, ws.F, ws.Ln, ws.max_rows, _ptr(bu), _ptr(bi), _ptr(bj), bu.numel(),
                                           batch, first_step, n_steps, C.byref(hp), adam_step0, 1 if apply else 0,
                                           tower_dtype, C.c_float(dropout), C.c_uint64(dropout_seed),
                                           None if drop_masks is None else _ptr(drop_masks), mode, _ptr(losses),
                                           1 if check else 0, C.byref(nan_step), _stream())
    _check_step(rc)
    return losses[:n_steps]


def neumf_scores(tabs, W, ws, users, items, per_user, tower_dtype=0, mode=0):
    """scores [n_users, per_user]: items = int64 [n_users, per_user] candidate ids, or None for all item ids."""
    _dev(users, torch.int64, "users")
    if items is not None:
        _dev(items, torch.int64, "items")
    out = torch.empty((users.numel(), per_user), dtype=torch.float32, device=W.device)
    L.check(L.lib().drb_neumf_scores(_ptr(tabs[0]), _ptr(tabs[1]), _ptr(tabs[2]), _ptr(tabs[3]), _ptr(W), _ptr(ws.buf), ws.U,
                                     ws.I, ws.F, ws.Ln, ws.opt, ws.max_rows, _ptr(users), users.numel(),
                                     None if items is None else _ptr(items), per_user, tower_dtype, mode, _ptr(out),
                                     _stream()))
    return out


def topk_from_scores(scores, cands, topk):
    _dev(scores, torch.float32, "scores")
    n, cnt = scores.shape
    if cands is not None:
        _dev(cands, torch.int64, "cands")
        out = torch.empty((n, topk), dtype=torch.float32, device=scores.device)
        L.check(L.lib().drb_topk_from_scores(_ptr(scores), _ptr(cands), n, cnt, topk, _ptr(out), None, _stream()))
    else:
        out = torch.empty((n, topk), dtype=torch.int64, device=scores.device)
        L.check(L.lib().drb_topk_from_scores(_ptr(scores), None, n, cnt, topk, None, _ptr(out), _stream()))
    return out


def gemm_test(variant, dtype, A, B, C_out, M, N, K, bias=None, ref=None):
    """Tower GEMM dispatcher (tests): variant 0 NT+bias+ReLU, 1 NN+mask, 2 NN, 3 TN split-K accumulate."""
    L.check(L.lib().drb_gemm_test(variant, dtype, M, N, K, _ptr(A), A.stride(0), _ptr(B), B.stride(0), _ptr(C_out),
                                  C_out.stride(0), None if bias is None else _ptr(bias), None if ref is None else _ptr(ref),
                                  0 if ref is None else ref.stride(0), _stream()))
    return C_out
