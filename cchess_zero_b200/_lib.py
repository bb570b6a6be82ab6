"""ctypes loader of libcchess_b200.so (include/cchess_b200.h).  There is NO CPU fallback: if the
CUDA library cannot be loaded every entry point of the package raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcchess_b200.so")

NSQ, NLABEL, MAXCHILD, ENC_LEN, STATUS_BYTES, MT_WORDS = 90, 2086, 128, 1260, 112, 626
F32, BF16, F16, BOARD = 0, 1, 2, 3
ERR_NAMES = {1: "NOMOVES", 2: "NOLABEL", 4: "DEPTH", 8: "ARENA", 16: "CHILDREN", 32: "NOCHILD"}
NOMOVE = 0xFFFF

_lib = None


class EngineError(RuntimeError):
    pass


def _sig(L):
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.cz_last_error.restype = C.c_char_p
    L.cz_labels.argtypes = [vp]
    L.cz_label_index.argtypes = [i32, i32]
    L.cz_unflipped_index.argtypes = [vp]
    L.cz_from_state.argtypes = [C.c_char_p, vp]
    L.cz_to_state.argtypes = [vp, C.c_char_p]
    L.cz_legal_moves_batch.argtypes = [i32, vp, vp, i32, vp, vp]
    L.cz_apply_moves_batch.argtypes = [i32, vp, vp, i32, vp]
    L.cz_encode_batch.argtypes = [i32, vp, vp, i32, vp]
    L.cz_legal_moves_dev.argtypes = [vp, vp, i32, vp, vp, vp]
    L.cz_encode_dev.argtypes = [vp, vp, i32, vp, i32, vp]
    L.cz_engine_create.argtypes = [i32, i64, i32, C.POINTER(vp)]
    L.cz_engine_create_ex.argtypes = [i32, i64, i32, i32, C.POINTER(vp)]
    L.cz_engine_create_fifo.argtypes = [i32, i64, i32, i32, C.POINTER(vp)]
    L.cz_engine_is_fifo.argtypes = [vp]
    L.cz_engine_leaves.argtypes = [vp]
    L.cz_engine_destroy.argtypes = [vp]
    L.cz_engine_n_games.argtypes = [vp]
    L.cz_engine_reset.argtypes = [vp, vp, vp, vp, vp, vp]
    L.cz_engine_set_root_meta.argtypes = [vp, vp, vp, vp, vp]
    L.cz_engine_begin_search.argtypes = [vp, vp, vp, i32]
    L.cz_engine_wave.argtypes = [vp, vp, vp, i32, vp, vp]
    L.cz_engine_wave_compact.argtypes = [vp, vp, vp, vp, i32, vp, vp]
    L.cz_engine_live_rows.argtypes = [vp, vp, vp]
    L.cz_engine_select.argtypes = [vp, vp, vp, i32]
    L.cz_engine_expand_backup.argtypes = [vp, vp, vp, vp]
    L.cz_engine_enable_hashing.argtypes = [vp, i32]
    L.cz_engine_leaf_hashes.argtypes = [vp, vp]
    L.cz_engine_root_keys.argtypes = [vp, vp, vp]
    L.cz_engine_play_status.argtypes = [vp, vp, vp, vp]
    L.cz_engine_status_packed.argtypes = [vp, vp, vp]
    L.cz_engine_play_moves.argtypes = [vp, vp, vp, vp]
    L.cz_engine_unfinished.argtypes = [vp, vp, vp]
    L.cz_engine_unfinished_async.argtypes = [vp, vp, vp]
    L.cz_engine_root_children.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.cz_engine_play.argtypes = [vp, vp, vp]
    L.cz_engine_status.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.cz_engine_counters.argtypes = [vp, vp, vp]
    L.cz_engine_tree_signature.argtypes = [vp, vp, i32, vp, i64, vp]
    L.cz_net_first_conv.argtypes = [vp, i32, vp, vp, vp, vp]
    L.cz_net_first_conv_tc.argtypes = [vp, i32, vp, vp, vp, vp]
    L.cz_net_first_conv_mma.argtypes = [vp, i32, vp, vp, vp]
    L.cz_net_heads.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cz_host_choose_moves.argtypes = [i32, vp, vp, vp, i32, vp, vp, vp, vp, i32]
    L.cz_net_heads_tc.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cz_net_heads_fc.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.cz_net_split_tf32.argtypes = [vp, vp, vp, i64, vp]
    L.cz_net_epilogue_split.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, vp]
    L.cz_net_tower_blob_bytes.argtypes = [i32]
    L.cz_net_tower_blob_bytes.restype = i64
    L.cz_net_tower_small.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]


def lib():
    """Loads the shared library, building it with nvcc when it is missing or stale."""
    global _lib
    if _lib is None:
        from . import build as _build

        # Under torchrun (RANK set) several ranks import at once: never race nvcc there -- use the library that
        # __graft_entry__.build() / `python -m cchess_zero_b200.build` produced.  CCHESS_NO_REBUILD=1 forces the same.
        distributed = "RANK" in os.environ or os.environ.get("CCHESS_NO_REBUILD", "0") == "1"
        if not (distributed and os.path.exists(LIB_PATH)):
            try:
                _build.build()
            except Exception as e:  # stale/missing and not buildable
                if not os.path.exists(LIB_PATH):
                    raise EngineError("libcchess_b200.so is missing and could not be built: %s" % e)
        L = C.CDLL(LIB_PATH)
        _sig(L)
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        raise EngineError("%s failed (%d): %s" % (what or "cchess_b200 call", rc, lib().cz_last_error().decode()))
