"""ctypes loader for libsoundsym_b200.so (the C ABI declared in include/soundsym_b200.h).

The library is the product; this module only declares argument types. There is no Python or CPU fallback: if the
shared library is missing, loading raises, and without a CUDA device ss_ctx_create fails with SS_ERR_CUDA.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SS_B200_LIB") or os.path.join(_HERE, "libsoundsym_b200.so")  # override: development A/B builds

SS_OK, SS_ERR_INVALID, SS_ERR_CUDA, SS_ERR_NOMEM, SS_ERR_NOT_TRAINED, SS_ERR_EMPTY_DICT, SS_ERR_TOO_FEW_ROWS = 0, -1, -2, -3, -4, -5, -6
SS_COSINE_REF, SS_DTW = 0, 1
SS_MAX_TOPK = 8
SS_COMM_ID_BYTES = 128

# every symbol include/soundsym_b200.h declares (tests/test_abi.py checks the header against this list and the .so)
SYMBOLS = [
    "ss_version", "ss_ctx_create", "ss_ctx_destroy", "ss_last_error", "ss_ctx_stream", "ss_ctx_sync", "ss_ctx_device",
    "ss_ctx_launch_count", "ss_frame_count", "ss_decode_pcm", "ss_sound_analyze", "ss_sound_analyze_pcm", "ss_sound_analyze_batch", "ss_mfcc", "ss_max_power", "ss_mfcc_dev",
    "ss_symbols", "ss_gmm_train", "ss_vote_split", "ss_partition", "ss_dict_create", "ss_dict_destroy", "ss_dict_len", "ss_dict_match",
    "ss_queries_create", "ss_queries_destroy", "ss_dict_match_dev", "ss_topk_merge_dev", "ss_dict_last_work", "ss_dict_last_scan_kind",
    "ss_dict_last_uncertified", "ss_dict_last_tc_fallback", "ss_dict_last_exhaustive", "ss_queries_invalidate", "ss_dict_last_scan_ms", "ss_resynth", "ss_sequence_distances", "ss_dict_debug_tc_scan", "ss_dict_debug_h2_scan", "ss_dict_set_scan", "ss_dict_match_finish",
    "ss_dict_set_dtw_band", "ss_dict_dtw_band", "ss_sharded_dict_set_dtw_band",
    "ss_dict_walk", "ss_dict_walk_dev", "ss_dict_align", "ss_dict_align_dev",
    "ss_shard_bounds", "ss_comm_unique_id", "ss_comm_create", "ss_comm_create_all", "ss_comm_destroy", "ss_comm_rank", "ss_comm_nranks",
    "ss_queries_create_sharded", "ss_dict_match_sharded_dev", "ss_dict_match_sharded", "ss_dict_create_sharded", "ss_sharded_dict_match",
    "ss_sharded_dict_destroy", "ss_sharded_dict_len", "ss_sharded_dict_nshards",
]


class ss_gmm(C.Structure):
    _fields_ = [("ncomp", C.c_int), ("ncoeffs", C.c_int), ("means", C.c_void_p), ("covs", C.c_void_p), ("weights", C.c_void_p)]


_lib = None


def load():
    """Loads the shared library (building it in-tree first if the sources are newer and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OSError("libsoundsym_b200.so is not built: run `python -m soundsym_b200.build` (needs nvcc). "
                      "There is no CPU fallback.")
    if "SS_NCCL_LIB" not in os.environ:
        # the multi-GPU entry points bind NCCL at run time: point them at the copy PyTorch ships (if there is one), so that
        # whichever of {this library, torch} touches NCCL first, the process ends up with the same libnccl.so.2
        try:
            import importlib.util
            spec = importlib.util.find_spec("nvidia.nccl")
            for base in (list(spec.submodule_search_locations) if spec and spec.submodule_search_locations else []):
                cand = os.path.join(base, "lib", "libnccl.so.2")
                if os.path.exists(cand):
                    os.environ["SS_NCCL_LIB"] = cand
                    break
        except Exception:
            pass
    L = C.CDLL(LIB_PATH)
    vp, sz, u64, u32, dbl, i = C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32, C.c_double, C.c_int
    P = C.POINTER
    L.ss_version.restype = C.c_char_p
    L.ss_ctx_create.argtypes = [i, P(vp)]
    L.ss_ctx_destroy.argtypes = [vp]
    L.ss_ctx_destroy.restype = None
    L.ss_last_error.argtypes = [vp]
    L.ss_last_error.restype = C.c_char_p
    L.ss_ctx_stream.argtypes = [vp]
    L.ss_ctx_stream.restype = vp
    L.ss_ctx_sync.argtypes = [vp]
    L.ss_ctx_device.argtypes = [vp]
    L.ss_ctx_launch_count.argtypes = [vp]
    L.ss_ctx_launch_count.restype = u64
    L.ss_frame_count.argtypes = [sz, P(sz)]
    L.ss_decode_pcm.argtypes = [vp, vp, sz, i, vp]
    L.ss_sound_analyze.argtypes = [vp, vp, sz, dbl, i, vp, P(sz), P(dbl), vp]
    L.ss_sound_analyze_pcm.argtypes = [vp, vp, sz, i, dbl, i, vp, vp, P(sz), P(dbl), vp]
    L.ss_sound_analyze_batch.argtypes = [vp, vp, vp, sz, dbl, i, vp, vp, vp, vp]
    L.ss_mfcc.argtypes = [vp, vp, sz, dbl, i, vp, P(sz)]
    L.ss_max_power.argtypes = [vp, vp, sz, P(dbl)]
    L.ss_mfcc_dev.argtypes = [vp, vp, sz, dbl, i, vp]
    L.ss_symbols.argtypes = [vp, vp, sz, P(ss_gmm), vp, vp]
    L.ss_gmm_train.argtypes = [vp, vp, sz, i, i, i, dbl, u64, vp, vp, vp]
    L.ss_vote_split.argtypes = [vp, vp, sz, i, i, vp, vp, P(sz)]
    L.ss_partition.argtypes = [vp, vp, sz, P(ss_gmm), i, i, vp, P(sz)]
    L.ss_dict_create.argtypes = [vp, vp, vp, sz, i, u32, P(vp)]
    L.ss_dict_destroy.argtypes = [vp]
    L.ss_dict_destroy.restype = None
    L.ss_dict_len.argtypes = [vp]
    L.ss_dict_len.restype = sz
    L.ss_dict_match.argtypes = [vp, vp, vp, sz, i, vp, i, vp, vp]
    L.ss_queries_create.argtypes = [vp, vp, vp, sz, i, P(vp)]
    L.ss_queries_destroy.argtypes = [vp]
    L.ss_queries_destroy.restype = None
    L.ss_dict_match_dev.argtypes = [vp, vp, i, vp, i, vp, vp]
    L.ss_topk_merge_dev.argtypes = [vp, vp, vp, i, sz, i, vp, vp]
    L.ss_dict_last_work.argtypes = [vp]
    L.ss_dict_last_scan_kind.argtypes = [vp]
    L.ss_dict_last_work.restype = u64
    L.ss_dict_last_uncertified.argtypes = [vp]
    L.ss_dict_last_uncertified.restype = u64
    L.ss_dict_last_tc_fallback.argtypes = [vp]
    L.ss_dict_last_tc_fallback.restype = u64
    L.ss_dict_last_exhaustive.argtypes = [vp]
    L.ss_dict_last_exhaustive.restype = u64
    L.ss_queries_invalidate.argtypes = [vp]
    L.ss_dict_last_scan_ms.argtypes = [vp]
    L.ss_dict_last_scan_ms.restype = dbl
    L.ss_dict_match_finish.argtypes = [vp]
    L.ss_dict_walk.argtypes = [vp, vp, sz, vp, sz, vp, vp]
    L.ss_dict_walk_dev.argtypes = [vp, vp, vp, sz, vp, vp]
    L.ss_dict_align.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp, vp]
    L.ss_dict_align_dev.argtypes = [vp, vp, vp, vp, sz, vp, vp]
    L.ss_dict_debug_h2_scan.argtypes = [vp, vp, vp, sz, vp, vp, P(C.c_float), P(C.c_float)]
    L.ss_dict_set_scan.argtypes = [vp, i]
    L.ss_dict_set_dtw_band.argtypes = [vp, u32]
    L.ss_dict_dtw_band.argtypes = [vp]
    L.ss_dict_dtw_band.restype = u32
    L.ss_sharded_dict_set_dtw_band.argtypes = [vp, u32]
    L.ss_shard_bounds.argtypes = [vp, sz, i, vp]
    L.ss_comm_unique_id.argtypes = [vp]
    L.ss_comm_create.argtypes = [vp, i, i, vp, P(vp)]
    L.ss_comm_create_all.argtypes = [P(vp), i, P(vp)]
    L.ss_comm_destroy.argtypes = [vp]
    L.ss_comm_destroy.restype = None
    L.ss_comm_rank.argtypes = [vp]
    L.ss_comm_nranks.argtypes = [vp]
    L.ss_queries_create_sharded.argtypes = [vp, vp, vp, sz, i, P(vp)]
    L.ss_dict_match_sharded_dev.argtypes = [vp, vp, vp, i, vp, i, vp, vp]
    L.ss_dict_match_sharded.argtypes = [vp, vp, vp, vp, sz, i, vp, i, vp, vp]
    L.ss_dict_create_sharded.argtypes = [P(vp), i, vp, vp, sz, i, P(vp)]
    L.ss_sharded_dict_match.argtypes = [vp, vp, vp, sz, i, vp, i, vp, vp]
    L.ss_sharded_dict_destroy.argtypes = [vp]
    L.ss_sharded_dict_destroy.restype = None
    L.ss_sharded_dict_len.argtypes = [vp]
    L.ss_sharded_dict_len.restype = sz
    L.ss_sharded_dict_nshards.argtypes = [vp]
    L.ss_dict_debug_tc_scan.argtypes = [vp, vp, vp, sz, vp, vp, P(C.c_float)]
    L.ss_resynth.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp]
    L.ss_sequence_distances.argtypes = [vp, vp, sz, i, vp]
    _lib = L
    return L


class SoundsymError(RuntimeError):
    """Maps the C ABI's negative status codes (CosError / Box<Error> on the Rust side, src/lib.rs:181-198)."""

    def __init__(self, code, message):
        super().__init__("%s (status %d)" % (message, code))
        self.code = code
        self.message = message
