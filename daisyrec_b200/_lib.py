"""ctypes loader for libdaisyrec_b200.so -- the C ABI declared in include/daisyrec_b200.h.

The product path has NO CPU fallback: if the shared object is missing (and cannot be built
because nvcc is absent) or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

from . import _build

_lib = None

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u32p = C.POINTER(C.c_uint32)
c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
vp = C.c_void_p

DRB_OK, DRB_ERR_INVALID, DRB_ERR_CUDA, DRB_ERR_NAN_LOSS, DRB_ERR_EMPTY_SET, DRB_ERR_NO_DEVICE, DRB_ERR_PEER = range(7)
OPT_SGD, OPT_ADAM, OPT_ADAGRAD, OPT_RMSPROP = 0, 1, 2, 3
OPT_KIND = {"sgd": 0, "adam": 1, "adagrad": 2, "rmsprop": 3}
LOSS_KIND = {"BPR": 0, "HL": 1, "TL": 2, "CL": 3, "SL": 4}


class Hyper(C.Structure):
    """struct drb_hyper"""
    _fields_ = [("lr", C.c_float), ("reg_1", C.c_float), ("reg_2", C.c_float), ("opt", C.c_int32),
                ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("loss", C.c_int32)]


# name -> (restype, argtypes); every symbol of include/daisyrec_b200.h
SIGNATURES = {
    "drb_version": (C.c_int, []),
    "drb_last_error": (C.c_char_p, []),
    "drb_device_query": (C.c_int, [c_i32p, c_i32p, c_i32p, c_i64p]),
    "drb_index_range_check": (C.c_int, [vp, C.c_int32, C.c_int64, C.c_int32, c_i64p, c_i64p, vp]),
    "drb_mf_step_variant": (C.c_int, [C.c_int32, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "drb_mf_step_selfcheck_ms": (C.c_int, [C.c_int32, C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "drb_mf_step_geometry": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int64,
                                       C.POINTER(C.c_int32)]),
    "drb_mt19937_seed": (C.c_int, [vp, C.c_uint32]),
    "drb_sampler_draw_mt19937": (C.c_int, [vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, c_i32p]),
    "drb_sampler_draw_philox": (C.c_int, [C.c_uint64, C.c_uint64, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp]),
    "drb_sampler_kth_complement": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp]),
    "drb_sampler_explode": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int32, vp, vp]),
    "drb_sample_triples_host": (C.c_int, [vp, vp, vp, vp, vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, vp, vp,
                                          c_i32p]),
    "drb_bounded_draws_mt19937": (C.c_int, [vp, vp, vp, C.c_int64, vp, c_i64p]),
    "drb_kth_complement_var": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp, vp]),
    "drb_gather_triples": (C.c_int, [vp, vp, C.c_int64, vp, vp, vp, vp]),
    "drb_mf_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "drb_mf_workspace_init": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]),
    "drb_mf_bpr_train_steps": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64, C.c_int64,
                                         C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64, vp, C.c_int32, c_i64p, vp]),
    "drb_mf_workspace_bytes_det": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "drb_mf_bpr_train_steps_det": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64, C.c_int64,
                                             C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64, vp, C.c_int32, c_i64p, vp]),
    "drb_mf_bpr_train_steps_fused_neg": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp, C.c_uint64, vp,
                                                   C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64, vp,
                                                   C.c_int32, c_i64p, vp]),
    "drb_mf_bpr_loss": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64, C.POINTER(Hyper),
                                  vp, vp]),
    "drb_mf_bpr_train_step_host": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64,
                                             C.POINTER(Hyper), C.c_int64, vp, c_f64p, vp]),
    "drb_mf_bpr_train_steps_host": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64,
                                              C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64, vp, vp, vp, c_i64p, vp]),
    "drb_randperm_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "drb_mt19937_stream": (C.c_int, [C.c_uint64, C.c_int64, vp, vp]),
    "drb_mt19937_stream_variant": (C.c_int, [C.c_int64]),
    "drb_randperm_torch": (C.c_int, [C.c_uint64, C.c_int64, vp, vp, vp]),
    "drb_fm_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "drb_fm_workspace_init": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]),
    "drb_fm_train_steps": (C.c_int, [vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64, C.c_int64,
                                     C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64, C.c_int32, vp, C.c_int32, c_i64p, vp]),
    "drb_fm_rank": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, C.c_int64, vp, C.c_int32, C.c_int32, vp, vp]),
    "drb_fm_full_rank": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, C.c_int64, C.c_int32, vp, vp]),
    "drb_fm_predict": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, C.c_int64, vp, vp]),
    "drb_mf_workspace_layout": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_i64p]),
    "drb_mf_bpr_phase": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64, C.c_int64,
                                   C.c_int32, C.POINTER(Hyper), C.c_int64, vp, vp]),
    "drb_shard_gather_triples": (C.c_int, [vp, vp, C.c_int64, C.c_int32, C.c_int32, C.c_int64, vp, vp, vp, vp, vp, vp]),
    "drb_lgcn_segment_count": (C.c_int64, [vp, C.c_int64]),
    "drb_lgcn_segments": (C.c_int, [vp, C.c_int64, vp, vp]),
    "drb_lgcn_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "drb_lgcn_workspace_init": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp]),
    "drb_lgcn_propagate": (C.c_int, [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, C.c_int64, vp,
                                     vp]),
    "drb_lgcn_bpr_train_steps": (C.c_int, [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp, vp,
                                           C.c_int64, vp, vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                           C.POINTER(Hyper), C.c_int64, C.c_int32, vp, C.c_int32, c_i64p, vp]),
    "drb_ngcf_param_count": (C.c_int64, [c_i32p, C.c_int32]),
    "drb_ngcf_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, c_i32p, C.c_int32, C.c_int32]),
    "drb_ngcf_workspace_init": (C.c_int, [vp, C.c_int32, C.c_int32, c_i32p, C.c_int32, C.c_int32, vp]),
    "drb_ngcf_forward": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, c_i32p, C.c_int32, vp, vp, vp, vp, vp, C.c_int64, C.c_int32,
                                   vp, C.c_float, vp, vp]),
    "drb_ngcf_bpr_train_steps": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, c_i32p, C.c_int32, vp, vp, vp, vp, vp, C.c_int64,
                                           vp, vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64,
                                           C.c_int32, C.c_int32, vp, C.c_float, vp, C.c_int32, c_i64p, vp]),
    "drb_nfm_param_count": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "drb_nfm_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64]),
    "drb_nfm_workspace_init": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64, vp]),
    "drb_nfm_bpr_train_steps": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_int64, vp, vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                          C.POINTER(Hyper), C.c_int64, C.c_int32, C.c_int32, vp, C.c_float, vp, C.c_int32, c_i64p,
                                          vp]),
    "drb_nfm_scores": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_int32, C.c_int64, vp, vp, C.c_int64, C.c_int32, vp, vp]),
    "drb_comm_unique_id": (C.c_int, [vp]),
    "drb_comm_init": (C.c_int, [vp, C.c_int32, C.c_int32]),
    "drb_comm_destroy": (C.c_int, []),
    "drb_mf_bpr_train_steps_sharded": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp, C.c_int64,
                                                 C.c_int64, C.POINTER(Hyper), C.c_int64, vp, vp]),
    "drb_mf_bpr_train_steps_sharded_host": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp, vp, vp,
                                                      C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64, vp, C.c_int64, vp,
                                                      vp, vp]),
    "drb_p2p_buffer_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "drb_p2p_q_offset": (C.c_size_t, [C.c_int32, C.c_int32]),
    "drb_p2p_alloc": (C.c_int, [C.c_size_t, C.POINTER(vp), vp]),
    "drb_p2p_open": (C.c_int, [vp, C.POINTER(vp)]),
    "drb_p2p_close": (C.c_int, [vp]),
    "drb_p2p_free": (C.c_int, [vp]),
    "drb_mf_bpr_train_steps_p2p": (C.c_int, [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp), C.c_int32, C.c_int32,
                                             vp, vp, vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.POINTER(Hyper),
                                             C.c_int64, vp, C.c_double, C.c_int32, c_i64p, vp]),
    "drb_neumf_param_count": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "drb_neumf_mask_words": (C.c_int64, [C.c_int32, C.c_int32, C.c_int64]),
    "drb_neumf_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64]),
    "drb_neumf_workspace_init": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64, vp]),
    "drb_neumf_bpr_train_steps": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                                            vp, vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.POINTER(Hyper),
                                            C.c_int64, C.c_int32, C.c_int32, C.c_float, C.c_uint64, vp, C.c_int32, vp,
                                            C.c_int32, c_i64p, vp]),
    "drb_neumf_scores": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                                   vp, C.c_int64, vp, C.c_int32, C.c_int32, C.c_int32, vp, vp]),
    "drb_gemm_test": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, vp, C.c_int64, vp, C.c_int64, vp,
                                C.c_int64, vp, vp, C.c_int64, vp]),
    "drb_topk_from_scores": (C.c_int, [vp, vp, C.c_int64, C.c_int32, C.c_int32, vp, vp, vp]),
    "drb_mf_rank": (C.c_int, [vp, vp, C.c_int32, vp, C.c_int64, vp, C.c_int32, C.c_int32, vp, vp]),
    "drb_mf_full_rank": (C.c_int, [vp, vp, C.c_int32, C.c_int32, vp, C.c_int64, C.c_int32, vp, vp]),
    "drb_mf_predict": (C.c_int, [vp, vp, C.c_int32, vp, vp, C.c_int64, vp, vp]),
    "drb_mf_rank_host": (C.c_int, [vp, vp, C.c_int32, vp, C.c_int64, vp, C.c_int32, C.c_int32, vp]),
    "drb_sampler_draw_mt19937_mixed": (C.c_int, [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp, c_i32p]),
    "drb_sampler_assemble_mixed": (C.c_int, [vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, vp, vp]),
    "drb_sampler_explode_pointwise": (C.c_int, [vp, vp, vp, C.c_int64, vp, C.c_int32, vp, vp]),
    "drb_sgns_positions": (C.c_int, [vp, C.c_int64, vp, C.c_int32, C.c_int32, vp, vp, vp]),
    "drb_sgns_explode": (C.c_int, [vp, vp, C.c_int64, C.c_int32, vp, vp, vp, vp, vp, vp]),
    "drb_item2vec_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "drb_item2vec_workspace_init": (C.c_int, [vp, C.c_int32, C.c_int32, C.c_int32, vp]),
    "drb_item2vec_train_steps": (C.c_int, [vp, vp, C.c_int32, C.c_int32, vp, vp, vp, C.c_int64, C.c_int64, C.c_int64,
                                           C.c_int64, C.POINTER(Hyper), C.c_int64, C.c_int32, vp, C.c_int32, c_i64p, vp]),
    "drb_item2vec_user_embed": (C.c_int, [vp, vp, vp, C.c_int32, C.c_int32, vp, vp]),
    "drb_vae_param_count": (C.c_int64, [C.c_int32, vp, C.c_int32, C.c_int32]),
    "drb_vae_workspace_bytes": (C.c_size_t, [C.c_int32, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64]),
    "drb_vae_workspace_init": (C.c_int, [vp, C.c_int32, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64, vp]),
    "drb_vae_train_steps": (C.c_int, [vp, vp, C.c_int32, vp, C.c_int32, C.c_int32, C.c_int64, vp, vp, vp, C.c_int32, vp,
                                      C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.POINTER(Hyper), C.c_int64, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_float, vp, vp, C.c_uint64, C.c_double, C.c_int64, C.c_int64,
                                      vp, C.c_int32, c_i64p, vp]),
    "drb_vae_forward": (C.c_int, [vp, vp, C.c_int32, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64, vp, vp, vp, C.c_int32,
                                  vp, C.c_int64, C.c_int32, C.c_int32, vp, vp]),
    "drb_vae_candidate_scores": (C.c_int, [vp, C.c_int32, vp, C.c_int32, C.c_int32, vp, C.c_int64, vp, C.c_int32, vp, vp]),
    "drb_csr_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int64]),
    "drb_csr_build": (C.c_int, [vp, vp, C.c_int64, C.c_int32, C.c_int32, vp, vp, vp, c_i64p, vp]),
    "drb_lgcn_build_adj": (C.c_int, [vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int64, vp, vp, vp, vp]),
    "drb_rank_metrics_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "drb_rank_metrics": (C.c_int, [vp, C.c_int64, C.c_int32, vp, vp, vp, C.c_int32, C.c_int32, vp, vp, vp, vp]),
    "drb_rank_metrics_host": (C.c_int, [vp, C.c_int64, C.c_int32, vp, vp, vp, C.c_int32, C.c_int32, vp, vp]),
}

KPI_NAMES = ("recall", "mrr", "ndcg", "hit", "precision", "map", "coverage", "popularity")   # DRB_KPI_* order


def so_path():
    # DRB_LIB_PATH: developer override used by scripts/tune_variants.sh to A/B kernel builds
    return os.environ.get("DRB_LIB_PATH") or _build.SO


def _cuda_device_count():
    """Devices the driver reports, without touching the runtime of this process (0 when there is no driver)."""
    try:
        cu = C.CDLL("libcuda.so.1")
        n = C.c_int(0)
        if cu.cuInit(0) != 0 or cu.cuDeviceGetCount(C.byref(n)) != 0:
            return 0
        return n.value
    except OSError:
        return 0


_CANARY = r"""
import ctypes, sys
l = ctypes.CDLL(sys.argv[1])
l.drb_mf_step_variant.argtypes = [ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
l.drb_mt19937_stream_variant.argtypes = [ctypes.c_int64]
a = l.drb_mf_step_variant(64, 0, None, None)                 # step-kernel selection, tables inside L2
b = l.drb_mf_step_variant(128, 1 << 20, None, None)          # ... streamed from HBM
c = l.drb_mt19937_stream_variant(3 << 20)                    # segmented MT19937 kernel's device check
print("CANARY OK", a, b, c, flush=True)
"""


def _canary(path):
    """The kernels that select themselves on the device (lean step instantiations, segmented MT19937) first run in a sacrificial
    child process: if that child crashes or does not come back, this process keeps the kernels that have a GPU record
    (DRB_NO_LEAN / DRB_MT_SEQUENTIAL are set before the library reads them).  Skipped without a device and under DRB_NO_CANARY."""
    if os.environ.get("DRB_NO_CANARY") or os.environ.get("DRB_NO_LEAN") or _cuda_device_count() == 0:
        return
    import subprocess
    import sys
    env = dict(os.environ)
    local = int(env.get("LOCAL_RANK", "0") or 0)
    vis = [v for v in env.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
    env["CUDA_VISIBLE_DEVICES"] = vis[local] if local < len(vis) else (vis[0] if vis else str(local))
    ok = False
    try:
        r = subprocess.run([sys.executable, "-c", _CANARY, path], env=env, capture_output=True, text=True, timeout=90)
        ok = r.returncode == 0 and "CANARY OK" in r.stdout
        why = (r.stdout + r.stderr)[-300:]
    except Exception as e:  # noqa: BLE001  (timeout, spawn failure)
        why = repr(e)
    if not ok:
        os.environ["DRB_NO_LEAN"] = "1"
        os.environ["DRB_MT_SEQUENTIAL"] = "1"
        sys.stderr.write(f"[daisyrec_b200] canary run of the self-selecting kernels failed ({why!r}): keeping the general step "
                         "kernel and the one-CTA MT19937 kernel in this process\n")


def lib():
    """Load (building first if the .so is absent and nvcc is present).  Fails loudly otherwise."""
    global _lib
    if _lib is not None:
        return _lib
    path = so_path()
    if not os.path.exists(path):
        try:
            _build.build()
        except Exception as e:  # noqa: BLE001
            raise RuntimeError(
                f"libdaisyrec_b200.so is missing ({path}) and could not be built: {e}. "
                "The B200 path has no CPU fallback; run `python -c 'import __graft_entry__ as g; g.build()'`.") from e
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)          # AttributeError here == header and library out of sync
        fn.restype, fn.argtypes = res, args
    _canary(path)
    _lib = L
    return L


class DrbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[libdaisyrec_b200 rc={code}] {msg}")
        self.code = code


def check(rc):
    if rc != DRB_OK:
        raise DrbError(rc, (lib().drb_last_error() or b"").decode(errors="replace"))
