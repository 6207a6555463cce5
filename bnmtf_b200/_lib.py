"""ctypes binding of libbnmtf_b200.so (include/bnmtf_b200.h).  There is no CPU fallback: if the shared
library is missing or a call fails, an exception is raised."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# BNMTF_LIB: another build of the same library (A/B runs of build options such as -DBNMTF_DIGITS=7, tools/gpu_margins.py)
LIB_PATH = os.environ.get("BNMTF_LIB") or os.path.join(_HERE, "libbnmtf_b200.so")

c_i, c_i64, c_u64, c_d, c_p = ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double, ctypes.c_void_p

# name -> argument types (all return int unless listed in _RESTYPES)
SIGNATURES = {
    "bnmtf_version": [],
    "bnmtf_last_error": [],
    "bnmtf_ld_for": [c_i64],
    "bnmtf_kp_for": [c_i],
    "bnmtf_gram_len": [c_i],
    "bnmtf_pack_dataset_f64": [c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_p],
    "bnmtf_pack_mask_f64": [c_p, c_i64, c_i64, c_i64, c_p, c_p],
    "bnmtf_transpose_dataset_f64": [c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_i64, c_p],
    "bnmtf_pad_factor_f64": [c_p, c_p, c_i64, c_i, c_i64, c_p, c_p, c_p],
    "bnmtf_stats_rx_f64": [c_p, c_p, c_i64, c_i64, c_p, c_i, c_i, c_p, c_p],
    "bnmtf_fixed_point_digits": [],
    "bnmtf_rx_planes_bytes": [c_i64, c_i64],
    "bnmtf_rx_planes_pack_f64": [c_p, c_p, c_i64, c_i64, c_p, c_p, c_p, c_p, c_p],
    "bnmtf_peer_sync_bytes": [],
    "bnmtf_peer_sync_f64": [c_p, c_p, c_i, c_i, c_i, c_p, c_i, c_p],
    "bnmtf_peer_put_f64": [c_p, c_p, c_i64, c_i64, c_i, c_i, c_p],
    "bnmtf_accumulate_f64": [c_p, c_p, c_i64, c_p],
    "bnmtf_sample_mean_f64": [c_p, c_i64, c_i, c_i, c_i, c_p, c_p],
    "bnmtf_range_guard_f64": [c_p, c_i, c_i64, c_p, c_i, c_i, c_i64, c_p, c_p, c_p, c_p],
    "bnmtf_stats_gated_f64": [c_p, c_p, c_p, c_i64, c_i64, c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p],
    "bnmtf_rx_umma_workspace_bytes": [c_i, c_i64],
    "bnmtf_stats_rx_umma_f64": [c_p, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_i, c_i, c_i, c_p, c_p, c_i64, c_p],
    "bnmtf_stats_gram_f64": [c_p, c_i64, c_i64, c_p, c_p, c_i, c_i, c_i, c_p, c_p, c_p],
    "bnmtf_gram_full_f64": [c_p, c_p, c_i64, c_i, c_i64, c_p, c_p, c_p],
    "bnmtf_small_cluster_size": [c_i64, c_i64, c_i, c_i],
    "bnmtf_small_sweeps_f64": [c_i, c_p, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                               c_p, c_p, c_p, c_p, c_p, c_i64, c_d, c_d, c_d, c_d, c_d, c_d, c_u64, c_i, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p],
    "bnmtf_small_tri_cluster_size": [c_i64, c_i64, c_i, c_i, c_i],
    "bnmtf_small_tri_sweeps_f64": [c_i, c_p, c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_i64,
                                   c_d, c_d, c_d, c_d, c_d, c_d, c_u64, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "bnmtf_kmeans_distances_f64": [c_p, c_p, c_i64, c_i64, c_p, c_p, c_i, c_p, c_p],
    "bnmtf_csr_kmeans_distances_f64": [c_p, c_p, c_p, c_i64, c_i64, c_p, c_p, c_i, c_p, c_p],
    "bnmtf_csr_kmeans_sums_f64": [c_p, c_p, c_p, c_i64, c_p, c_i, c_i, c_p, c_p, c_p],
    "bnmtf_gram_umma_workspace_bytes": [c_i, c_i, c_i64],
    "bnmtf_stats_gram_umma_f64": [c_p, c_i64, c_i64, c_i64, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_i64, c_p],
    "bnmf_row_solve_f64": [c_i, c_i64, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                           c_i, c_i, c_d, c_u64, c_p, c_u64, c_i64, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p],
    "bnmtf_masked_metrics_f64": [c_p, c_p, c_i64, c_i64, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p],
    "bnmtf_mstat_reduce_f64": [c_p, c_i64, c_p, c_p, c_p],
    "bnmtf_csr_stats_f64": [c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_i, c_p, c_p, c_i64, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p,
                            c_p, c_p],
    "bnmtf_csr_metrics_f64": [c_p, c_p, c_p, c_i64, c_p, c_p, c_i, c_p, c_i, c_p, c_p, c_p],
    "bnmtf_metrics_from_sums_f64": [c_p, c_p, c_d, c_p, c_p, c_p],
    "bnmtf_select_metrics_f64": [c_p, c_p, c_p, c_p],
    "bnmtf_dense_metrics_f64": [c_p, c_p, c_p, c_i64, c_p, c_i, c_p, c_p],
    "bnmtf_vb_factor_terms_f64": [c_p, c_p, c_p, c_p, c_p, c_i64, c_p, c_i, c_p],
    "bnmtf_reduce8_f64": [c_p, c_i, c_p, c_p],
    "bnmtf_reduce1_f64": [c_p, c_i64, c_p, c_p],
    "bnmf_finish_sweep_f64": [c_i, c_d, c_d, c_d, c_d, c_d, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_u64, c_i, c_p, c_p],
    "bnmtf_nmtf_transform_f64": [c_i64, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "bnmtf_nmtf_sq_f64": [c_i64, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p],
    "bnmtf_nmtf_sq_scratch_len": [c_i, c_i, c_i],
    "bnmtf_nmtf_sq_parts": [c_i64, c_i, c_i, c_i],
    "bnmtf_coord_solve_f64": [c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_d, c_u64, c_p, c_u64, c_p],
    "bnmtf_nmtf_extra_f64": [c_i64, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "bnmtf_nmtf_mstat_f64": [c_i64, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "bnmtf_np_build_pred_f64": [c_p, c_p, c_i64, c_i64, c_i64, c_i, c_p, c_p],
    "bnmtf_np_row_update_f64": [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_i, c_p],
    "bnmtf_np_s_update_f64": [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_i, c_i, c_p, c_i, c_i, c_p, c_p, c_i, c_p],
    "bnmtf_np_metrics_f64": [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_p, c_i, c_p, c_p],
    "bnmtf_csr_np_row_update_f64": [c_p, c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_p, c_p, c_p, c_i, c_i,
                                    c_i, c_p, c_p],
    "bnmtf_csr_np_s_update_f64": [c_p, c_p, c_p, c_p, c_p, c_i64, c_i, c_p, c_p, c_i, c_p, c_i, c_p, c_i, c_p, c_p, c_p, c_i,
                                  c_p],
    "bnmtf_csr_np_metrics_f64": [c_p, c_p, c_p, c_i64, c_p, c_p, c_i, c_p, c_i, c_p, c_p],
    "bnmtf_small_matmul_f64": [c_p, c_p, c_i64, c_i, c_i, c_i, c_p, c_p],
    "bnmtf_tn_moments_f64": [c_p, c_p, c_i64, c_p, c_p, c_p],
    "bnmtf_tn_draw_f64": [c_p, c_p, c_i64, c_u64, c_u64, c_p, c_p],
    "bnmtf_gamma_draw_f64": [c_d, c_d, c_i64, c_u64, c_u64, c_p, c_p],
    "bnmtf_exponential_draw_f64": [c_p, c_i64, c_u64, c_u64, c_p, c_p],
}
_RESTYPES = {"bnmtf_nmtf_sq_scratch_len": c_i64, "bnmtf_last_error": ctypes.c_char_p, "bnmtf_ld_for": c_i64, "bnmtf_gram_len": c_i64,
             "bnmtf_gram_umma_workspace_bytes": c_i64, "bnmtf_rx_planes_bytes": c_i64,
             "bnmtf_rx_umma_workspace_bytes": c_i64, "bnmtf_peer_sync_bytes": c_i64}
_PLAIN = {"bnmtf_nmtf_sq_scratch_len", "bnmtf_nmtf_sq_parts", "bnmtf_small_cluster_size", "bnmtf_small_tri_cluster_size", "bnmtf_fixed_point_digits", "bnmtf_version", "bnmtf_last_error", "bnmtf_ld_for", "bnmtf_kp_for", "bnmtf_gram_len",
          "bnmtf_gram_umma_workspace_bytes", "bnmtf_rx_planes_bytes", "bnmtf_rx_umma_workspace_bytes", "bnmtf_peer_sync_bytes"}

_lib = None

# kernels launched per entry point (for bench.py's gpu_launches count)
KERNELS_PER_CALL = {"bnmtf_pack_dataset_f64": 1, "bnmtf_pack_mask_f64": 1, "bnmtf_transpose_dataset_f64": 1,
                    "bnmtf_pad_factor_f64": 1, "bnmtf_stats_rx_f64": 1, "bnmtf_stats_rx_umma_f64": 5,
                    "bnmtf_rx_planes_pack_f64": 2, "bnmtf_range_guard_f64": 1, "bnmtf_stats_gated_f64": 2, "bnmtf_stats_gram_f64": 1, "bnmtf_kmeans_distances_f64": 1, "bnmtf_csr_kmeans_distances_f64": 1, "bnmtf_csr_kmeans_sums_f64": 1, "bnmtf_small_sweeps_f64": 1, "bnmtf_small_tri_sweeps_f64": 1, "bnmtf_stats_gram_umma_f64": 4, "bnmtf_mstat_reduce_f64": 2,
                    "bnmtf_metrics_from_sums_f64": 1, "bnmtf_select_metrics_f64": 1,
                    "bnmtf_gram_full_f64": 2, "bnmf_row_solve_f64": 1, "bnmtf_masked_metrics_f64": 3, "bnmtf_csr_stats_f64": 2, "bnmtf_csr_metrics_f64": 2,
                    "bnmtf_dense_metrics_f64": 2, "bnmtf_vb_factor_terms_f64": 1, "bnmtf_reduce8_f64": 1,
                    "bnmtf_reduce1_f64": 1, "bnmf_finish_sweep_f64": 1, "bnmtf_tn_moments_f64": 1, "bnmtf_np_build_pred_f64": 1,
                    "bnmtf_np_row_update_f64": 1, "bnmtf_np_s_update_f64": 2, "bnmtf_np_metrics_f64": 2,
                    "bnmtf_small_matmul_f64": 1, "bnmtf_csr_np_metrics_f64": 2,
                    # one launch per non-empty plan class / per pair plus one: the engine adds the rest
                    "bnmtf_csr_np_row_update_f64": 0, "bnmtf_csr_np_s_update_f64": 1, "bnmtf_nmtf_transform_f64": 1, "bnmtf_nmtf_sq_f64": 2,
                    "bnmtf_coord_solve_f64": 1, "bnmtf_nmtf_extra_f64": 1, "bnmtf_nmtf_mstat_f64": 1,
                    "bnmtf_tn_draw_f64": 1, "bnmtf_gamma_draw_f64": 1, "bnmtf_exponential_draw_f64": 1}
launch_count = [0]


class BnmtfError(RuntimeError):
    pass


_seed_calls = [0]


def derive_seed():
    """A Philox seed for the device-side draws that is a deterministic function of numpy's global random state and of
    how many seeds were asked for so far, WITHOUT consuming from that stream: the host random numbers the reference
    draws (initialisations, folds, K-means) keep their positions, so seeded runs with several models stay aligned
    with the reference."""
    import numpy as np
    st = np.random.get_state()
    keys, pos = st[1], int(st[2])
    _seed_calls[0] += 1
    h = (int(keys[pos % 624]) * 2654435761 + int(keys[(pos + 311) % 624]) * 40503 + pos * 97 + _seed_calls[0] * 1000003)
    return int(h % (2 ** 31 - 1))


def load():
    """Load the shared library (once) and declare every prototype of include/bnmtf_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BnmtfError("libbnmtf_b200.so not built (run `python -m bnmtf_b200.build` or __graft_entry__.build()); "
                         "there is no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.argtypes = args
        fn.restype = _RESTYPES.get(name, c_i)
    _lib = lib
    return lib


def call(name, *args):
    """Invoke an int-returning entry point; raise with the library's message on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if name in _PLAIN:
        return rc
    if rc != 0:
        raise BnmtfError("%s failed (%d): %s" % (name, rc, lib.bnmtf_last_error().decode()))
    launch_count[0] += KERNELS_PER_CALL.get(name, 1)
    return 0
