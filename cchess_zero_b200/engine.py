"""Python handle on the batched device engine (cz_engine_* in include/cchess_b200.h).

torch is used for device buffers and streams only; all tree / rules work happens in the
sm_100a kernels of csrc/cz_engine.cu."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import BF16, BOARD, F16, F32, MAXCHILD, STATUS_BYTES, EngineError, check, lib

_DT = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16, torch.uint8: BOARD}


def _hp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Engine:
    def __init__(self, n_games, arena_words=0, device=None, leaves=1, search_threads=None):
        """leaves > 1: leaf-parallel engine (up to `leaves` leaves per game per wave; network rows = n_games*leaves).
        leaves == -1: the leaf-parallel kernel with one slot (test hook).
        search_threads = K: the reference's search_threads schedule in canonical FIFO form (bit-exact with the reference's
        uvloop runs wherever those are reproducible); network rows = n_games*K."""
        if not torch.cuda.is_available():
            raise EngineError("cchess_zero_b200 needs a CUDA device (no CPU fallback exists)")
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.B = int(n_games)
        self.fifo = search_threads is not None
        self.leaves = int(search_threads) if self.fifo else abs(int(leaves))
        self.rows = self.B * self.leaves
        h = C.c_void_p()
        if self.fifo:
            check(lib().cz_engine_create_fifo(self.B, int(arena_words), self.device, int(search_threads), C.byref(h)), "cz_engine_create_fifo")
        else:
            check(lib().cz_engine_create_ex(self.B, int(arena_words), self.device, int(leaves), C.byref(h)), "cz_engine_create_ex")
        self.h = h
        self.launches = 0   # kernels of csrc/cz_engine.cu launched through this handle
        self._count = torch.zeros(1, dtype=torch.int32, device="cuda:%d" % self.device)

    def close(self):
        if getattr(self, "h", None):
            lib().cz_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- game state -------------------------------------------------------------------
    def reset(self, mask=None, boards=None, sides=None, rr=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        b = None if boards is None else np.ascontiguousarray(boards, dtype=np.uint8).reshape(self.B, 90)
        s = None if sides is None else np.ascontiguousarray(sides, dtype=np.uint8)
        r = None if rr is None else np.ascontiguousarray(rr, dtype=np.int32)
        self.launches += 1
        check(lib().cz_engine_reset(self.h, _stream(), _hp(m), _hp(b), _hp(s), _hp(r)), "cz_engine_reset")

    def set_root_meta(self, sides=None, rr=None, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        s = None if sides is None else np.ascontiguousarray(sides, dtype=np.uint8)
        r = None if rr is None else np.ascontiguousarray(rr, dtype=np.int32)
        self.launches += 1
        check(lib().cz_engine_set_root_meta(self.h, _stream(), _hp(m), _hp(s), _hp(r)), "cz_engine_set_root_meta")

    def begin_search(self, playouts, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        self.launches += 1
        check(lib().cz_engine_begin_search(self.h, _stream(), _hp(m), int(playouts)), "cz_engine_begin_search")

    # ---- waves (device tensors) ---------------------------------------------------------
    def wave(self, nn_in, logits, value):
        self.launches += 1
        check(lib().cz_engine_wave(self.h, _stream(), nn_in.data_ptr(), _DT[nn_in.dtype], logits.data_ptr(), value.data_ptr()),
              "cz_engine_wave")

    def wave_compact(self, nn_stage, nn_dense, logits, value):
        """search_threads = K engines: a wave whose leaves are gathered densely into nn_dense (cz_engine_wave_compact); evaluate
        nn_dense[:live_rows()] into logits / value before the next call."""
        self.launches += 3           # k_wave_fifo, k_compact_scan, k_compact_rows
        check(lib().cz_engine_wave_compact(self.h, _stream(), nn_stage.data_ptr(), nn_dense.data_ptr(), _DT[nn_stage.dtype],
                                           logits.data_ptr(), value.data_ptr()), "cz_engine_wave_compact")

    def live_rows(self):
        out = C.c_int32(0)
        check(lib().cz_engine_live_rows(self.h, _stream(), C.byref(out)), "cz_engine_live_rows")
        return out.value

    def select(self, nn_in):
        self.launches += 1
        check(lib().cz_engine_select(self.h, _stream(), nn_in.data_ptr(), _DT[nn_in.dtype]), "cz_engine_select")

    def expand_backup(self, logits, value):
        self.launches += 1
        check(lib().cz_engine_expand_backup(self.h, _stream(), logits.data_ptr(), value.data_ptr()), "cz_engine_expand_backup")

    # ---- board hashing (Zobrist keys of the pending leaves; never used by the search) -------
    def enable_hashing(self, on=True):
        check(lib().cz_engine_enable_hashing(self.h, 1 if on else 0), "cz_engine_enable_hashing")

    def leaf_hashes(self):
        """int64 view (device tensor, [rows]) of the 64-bit Zobrist keys of the positions in the network batch rows."""
        ptr = C.c_void_p()
        check(lib().cz_engine_leaf_hashes(self.h, C.byref(ptr)), "cz_engine_leaf_hashes")
        n = self.rows

        class _Arr:                                            # __cuda_array_interface__ view of engine-owned memory
            __cuda_array_interface__ = dict(shape=(n,), typestr="<i8", data=(ptr.value, False), version=2)
        return torch.as_tensor(_Arr(), device="cuda:%d" % self.device)

    def root_keys(self):
        out = np.zeros(self.B, dtype=np.uint64)
        check(lib().cz_engine_root_keys(self.h, _stream(), _hp(out)), "cz_engine_root_keys")
        return out

    def unfinished(self):
        out = C.c_int32(0)
        self.launches += 1
        check(lib().cz_engine_unfinished(self.h, _stream(), C.byref(out)), "cz_engine_unfinished")
        return out.value

    def unfinished_async(self):
        self.launches += 1
        check(lib().cz_engine_unfinished_async(self.h, _stream(), self._count.data_ptr()), "cz_engine_unfinished_async")
        return self._count

    # ---- root statistics / moves ----------------------------------------------------------
    def root_children(self, want_wpq=True):
        B = self.B
        n = np.zeros(B, dtype=np.int32)
        mv = np.zeros((B, MAXCHILD), dtype=np.uint16)
        vis = np.zeros((B, MAXCHILD), dtype=np.int32)
        w = np.zeros((B, MAXCHILD), dtype=np.float32) if want_wpq else None
        p = np.zeros((B, MAXCHILD), dtype=np.float32) if want_wpq else None
        q = np.zeros((B, MAXCHILD), dtype=np.float32) if want_wpq else None
        self.launches += 1
        check(lib().cz_engine_root_children(self.h, _stream(), _hp(n), _hp(mv), _hp(vis), _hp(w), _hp(p), _hp(q)),
              "cz_engine_root_children")
        return dict(n=n, moves=mv, visits=vis, w=w, p=p, q=q)

    def play(self, child_index, want_status=True):
        """GameBoard update + update_tree for every game with child_index >= 0; returns the status of all games (see status())
        from the same call: one kernel, one device->host copy, one synchronisation."""
        ci = np.ascontiguousarray(child_index, dtype=np.int32)
        assert ci.shape == (self.B,)
        self.launches += 1
        rec = np.zeros((self.B, STATUS_BYTES), dtype=np.uint8) if want_status else None
        check(lib().cz_engine_play_status(self.h, _stream(), _hp(ci), _hp(rec)), "cz_engine_play_status")
        return self._unpack_status(rec) if want_status else None

    def play_moves(self, moves, want_status=True):
        """update_tree(act) keyed by the move code (src | dst << 7) + the board update for every game with moves[g] != NOMOVE:
        the tree follows a move chosen elsewhere (the opponent's, human_move main.py:1394-1430).  status()["q"] is Q(act) of this
        tree.  A move that is not a child of an expanded root leaves that game untouched and flags it with NOCHILD; with
        want_status the flag raises EngineError (the reference's KeyError, main.py:275)."""
        mv = np.ascontiguousarray(moves, dtype=np.uint16)
        assert mv.shape == (self.B,)
        self.launches += 1
        rec = np.zeros((self.B, STATUS_BYTES), dtype=np.uint8) if want_status else None
        check(lib().cz_engine_play_moves(self.h, _stream(), _hp(mv), _hp(rec)), "cz_engine_play_moves")
        if not want_status:
            return None
        self.raise_on_error()
        return self._unpack_status(rec)

    @staticmethod
    def _unpack_status(rec):
        tail = np.ascontiguousarray(rec[:, 96:112]).view(np.int32)
        return dict(boards=np.ascontiguousarray(rec[:, :90]), side=rec[:, 90].copy(), terminal=rec[:, 91].copy(),
                    winner=rec[:, 92].copy().view(np.int8), ply=tail[:, 0].copy(), rr=tail[:, 1].copy(),
                    q=np.ascontiguousarray(tail[:, 2]).view(np.float32), root_N=tail[:, 3].copy())

    def status(self, boards=True):
        """terminal / winner / ply / restrict_round / side / boards of every game (check_end, main.py:1380-1392)."""
        rec = np.zeros((self.B, STATUS_BYTES), dtype=np.uint8)
        self.launches += 1
        check(lib().cz_engine_status_packed(self.h, _stream(), _hp(rec)), "cz_engine_status_packed")
        return self._unpack_status(rec)

    def counters(self):
        out = np.zeros(9, dtype=np.int64)
        check(lib().cz_engine_counters(self.h, _stream(), _hp(out)), "cz_engine_counters")
        return dict(n_expand=int(out[0]), n_playout=int(out[1]), sum_L=int(out[2]), sum_c=int(out[3]), error=int(out[4]),
                    max_arena_words=int(out[5]), first_error_game=int(out[6]), max_depth=int(out[7]), sum_C=int(out[8]))

    def raise_on_error(self):
        c = self.counters()
        if c["error"]:
            names = [v for k, v in _lib.ERR_NAMES.items() if c["error"] & k]
            raise EngineError("engine error flags %s (first game %d)" % ("|".join(names), c["first_error_game"]))
        return c

    def tree_signature(self, game, cap=1 << 16):
        out = np.zeros((cap, 6), dtype=np.int64)
        n = C.c_int64(0)
        check(lib().cz_engine_tree_signature(self.h, _stream(), int(game), _hp(out), cap, C.byref(n)), "cz_engine_tree_signature")
        if n.value > cap:
            return self.tree_signature(game, int(n.value))
        return out[: n.value].copy()

    # ---- a whole search: MCTS_tree.main for every selected game ---------------------------
    def search(self, forward_dev, playouts, nn_in, logits, value, mask=None, check_every=1):
        """forward_dev(nn_in) must fill `logits` [B,2086] f32 and `value` [B] (or [B,1]) f32 in place
        (device tensors).  Runs waves until every selected game has finished `playouts` playouts."""
        self.begin_search(playouts, mask)
        waves = 0
        while True:
            self.wave(nn_in, logits, value)
            waves += 1
            first = playouts // self.leaves
            if waves > first and (waves - first) % check_every == 0 and self.unfinished() == 0:
                break
            forward_dev(nn_in)
            if waves > 4 * playouts + 64:
                self.raise_on_error()
                raise EngineError("search did not converge after %d waves" % waves)
        return waves
