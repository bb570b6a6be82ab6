"""Batched self-play driver (many games in lock-step on one GPU) and the reference-shaped
`cchess_main` facade (main.py:1118-1554).

Move choice stays on the host in numpy, exactly as the reference does it (get_action,
main.py:1332-1358): pi = softmax(log(visits)/T) in float64 and
np.random.choice(p = 0.75*pi + 0.25*Dirichlet(0.3)) on a legacy MT19937 RandomState -- one
RandomState per game slot stands in for the reference's global np.random (SURVEY H3).  The device
produces the integer visit counts; everything before them (select / expand / backup / encode /
move generation / re-rooting) runs in csrc/cz_engine.cu."""
import os
import pickle
import random
import time
from collections import defaultdict, deque

import numpy as np
import torch

from . import rules
from ._lib import MAXCHILD, MT_WORDS, NLABEL, EngineError
from .engine import Engine


def _flip_board(b):
    """try_flip (main.py:560-574): reverse the rows, swap the colours; files are not mirrored."""
    f = b.reshape(10, 9)[::-1].copy()
    red, blk = (f >= 1) & (f <= 7), f >= 8
    f[red] += 7
    f[blk] -= 7
    return f.reshape(90)


def _flip_move_label_index(mv):
    """label index of the rank-mirrored move (flipped_uci_labels, main.py:23-27 / 1507-1512)."""
    s, d = int(mv) & 127, (int(mv) >> 7) & 127
    s = (9 - s // 9) * 9 + s % 9
    d = (9 - d // 9) * 9 + d % 9
    return rules.label2i[rules.move_to_label(s | (d << 7))]


_LABEL_OF = None


def _label_table():
    """(src_sq, dst_sq) -> label index as a numpy table (cz_label_index); -1 where the pair is not a label."""
    global _LABEL_OF
    if _LABEL_OF is None:
        from ._lib import lib
        L = lib()
        _LABEL_OF = np.array([[L.cz_label_index(s, d) for d in range(90)] for s in range(90)], dtype=np.int64)
    return _LABEL_OF


class GameRecord:
    """(s, pi, z) tuples of one finished game in the reference's format (selfplay, main.py:1493-1554).

    During play nothing per game is recorded: SelfPlay keeps ONE log entry per ply for the whole batch (boards, sides, root moves
    and visit counts, chosen indices); a record only remembers its slot and ply span.  Boards, move lists, pi (recomputed from the
    integer visit counts with the very numpy operations get_action uses, so bit-identical) and the canonical state strings /
    label indices are materialised on first access."""

    def __init__(self, slot=None, logs=None, temperature=1):
        self._slot, self._logs, self._T = slot, logs if logs is not None else [], temperature
        self.players = []
        self.z = None
        self.winner = None
        self._boards = self._moves = self._chosen = self.visits = self.pi_val = None
        self._states = self._pi_idx = self._actions = None

    def __len__(self):
        return len(self.players)

    def _raw(self):
        if self._boards is not None:
            return
        g = self._slot
        logs = self._logs
        L = len(logs)
        self._boards = [lg["boards"][g] for lg in logs]
        nn = np.fromiter((lg["n"][g] for lg in logs), dtype=np.int32, count=L)
        self._chosen = [int(lg["choice"][g]) for lg in logs]
        V = np.stack([lg["visits"][g] for lg in logs]) if L else np.zeros((0, MAXCHILD), np.int32)
        M = np.stack([lg["moves"][g] for lg in logs]) if L else np.zeros((0, MAXCHILD), np.uint16)
        self._moves = [M[i, :nn[i]] for i in range(L)]
        self.visits = [V[i, :nn[i]] for i in range(L)]
        # pi = softmax(1/T * log(visits)) (main.py:1341, 1111-1116): element-wise log / exp for the whole game at once, the
        # order-sensitive row sums in csrc/cz_host.cu exactly as np.sum does them (the same call get_action's batch path uses)
        with np.errstate(divide="ignore", invalid="ignore"):
            lv = (1.0 / self._T) * np.log(V.astype(np.int64))
            lv[np.arange(MAXCHILD)[None, :] >= nn[:, None]] = -np.inf
            ex = np.ascontiguousarray(np.exp(lv - np.max(lv, axis=1, keepdims=True))) if L else np.zeros((0, MAXCHILD))
        probs = np.empty((L, MAXCHILD), dtype=np.float64)
        if L:
            import ctypes as C
            from ._lib import lib
            vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
            mt = np.zeros((L, MT_WORDS), dtype=np.uint32); mt[:, 624] = 624          # scratch generators: the draws are discarded
            ch, fb = np.zeros(L, np.int32), np.zeros(L, np.uint8)
            lib().cz_host_choose_moves(L, None, vp(nn), vp(ex), 0, vp(mt), vp(ch), vp(probs), vp(fb), 1)
            for i in np.nonzero(fb)[0]:                                               # (NaN rows: plain numpy, as get_action would)
                pr = ex[i, :nn[i]].copy(); pr /= np.sum(pr); probs[i, :nn[i]] = pr
        self.pi_val = [probs[i, :nn[i]] for i in range(L)]
        self._logs = None

    def _materialise(self):
        self._raw()
        if self._states is not None and len(self._states) == len(self.players):
            return
        tab = _label_table()
        st, ix = [], []
        for b, side, mv in zip(self._boards, self.players, self._moves):
            st.append(rules.board_to_state(_flip_board(b) if side == 1 else b))             # main.py:1504-1505
            src, dst = (mv & 127).astype(np.int64), (mv >> 7).astype(np.int64)
            if side == 1:   # flipped_uci_labels for black (main.py:1507-1512): rank y -> 9-y
                src = (9 - src // 9) * 9 + src % 9
                dst = (9 - dst // 9) * 9 + dst % 9
            li = tab[src, dst]
            if (li < 0).any():
                raise KeyError("move outside the label table")                                # label2i[...] KeyError in the reference
            ix.append(li)
        self._states, self._pi_idx = st, ix
        self._actions = [rules.move_to_label(mv[c]) for mv, c in zip(self._moves, self._chosen)]

    @classmethod
    def from_tuples(cls, states, pi_idx, pi_val, z):
        """A record built from already materialised tuples (tests, gathered data)."""
        r = cls()
        r._states, r._pi_idx, r.pi_val, r.z = list(states), list(pi_idx), list(pi_val), z
        r.players = [0] * len(r._states)
        r._boards = [None] * len(r._states)
        r._moves = r._chosen = r.visits = []
        return r

    @property
    def states(self):
        self._materialise()
        return self._states

    @property
    def pi_idx(self):
        self._materialise()
        return self._pi_idx

    @property
    def actions(self):
        self._materialise()
        return self._actions

    def dense_pi(self):
        self._raw()
        out = np.zeros((len(self), NLABEL))
        for i, (ix, v) in enumerate(zip(self.pi_idx, self.pi_val)):
            out[i, ix] = v
        return out

    def tuples(self):
        return zip(self.states, self.dense_pi(), self.z)


def choose_moves(n_children, visits, live, mt, exploration, temperature, n_threads=1):
    """get_action's move choice (main.py:1339-1348) for every game with live[g]: the index into the root's children drawn from
    softmax(1/T * log(visits)), with the reference's Dirichlet noise when `exploration`.  mt [B][MT_WORDS]: one legacy MT19937
    state per game, advanced in place exactly as numpy's RandomState would be.  -1 for the other games."""
    B = len(n_children)
    choice = np.full(B, -1, dtype=np.int32)
    with np.errstate(divide="ignore", invalid="ignore"):
        # softmax(1/T * log(visits)) of main.py:1341, 1111-1116.  log / exp / max are element-wise or exact, so they are
        # taken over the whole [B,128] batch at once (padding: visits 0 -> -inf -> exp 0); the order-sensitive row sum, the
        # Dirichlet / choice draws and the cumulative sums happen per game in csrc/cz_host.cu, operation for operation what
        # numpy does for `probs /= np.sum(probs)`, RandomState.dirichlet and RandomState.choice (main.py:1345-1348).
        lv = (1.0 / temperature) * np.log(visits.astype(np.int64))
        valid = np.arange(MAXCHILD)[None, :] < n_children[:, None]
        lv[~valid] = -np.inf
        ex = np.ascontiguousarray(np.exp(lv - np.max(lv, axis=1, keepdims=True)))
    probs = np.empty((B, MAXCHILD), dtype=np.float64)
    fallback = np.zeros(B, dtype=np.uint8)
    live8 = np.ascontiguousarray(live, dtype=np.uint8)
    nn = np.ascontiguousarray(n_children, dtype=np.int32)
    from ._lib import lib
    import ctypes as C
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rcode = lib().cz_host_choose_moves(B, vp(live8), vp(nn), vp(ex), 1 if exploration else 0, vp(mt), vp(choice), vp(probs),
                                       vp(fallback), n_threads)
    if rcode:
        raise EngineError("cz_host_choose_moves failed (%d)" % rcode)
    for g in np.nonzero(fallback)[0]:
        # a probability vector numpy would reject (NaN priors ...): let numpy raise exactly what the reference would raise
        n = int(nn[g])
        rs = np.random.RandomState()
        rs.set_state(("MT19937", mt[g, :624].copy(), int(mt[g, 624]), 0, 0.0))
        pr = ex[g, :n] / np.sum(ex[g, :n])
        choice[g] = int(rs.choice(n, p=pr))          # (the Dirichlet draws were consumed by the native sampler, as in the reference)
        st_ = rs.get_state()
        mt[g, :624], mt[g, 624] = st_[1], st_[2]
    return choice


class _Lane:
    """One half-batch of a pipelined SelfPlay: its own engine, I/O buffers and evaluator scratch."""

    def __init__(self, engine, lo, hi, nn_in, logits, value, forward):
        self.engine, self.lo, self.hi = engine, lo, hi
        self.nn_in, self.logits, self.value, self.forward = nn_in, logits, value, forward


class _MultiEngine:
    """Engine-shaped facade over the lanes' engines (games [lo, hi) of lane k live in engine k)."""

    def __init__(self, lanes, B):
        self.lanes, self.B = lanes, B
        self.device = lanes[0].engine.device

    @property
    def launches(self):
        return sum(l.engine.launches for l in self.lanes)

    def _m(self, mask, l):
        return None if mask is None else np.ascontiguousarray(mask[l.lo:l.hi], dtype=np.uint8)

    def reset(self, mask=None, boards=None, sides=None, rr=None):
        for l in self.lanes:
            if mask is not None and not np.any(mask[l.lo:l.hi]):
                continue
            l.engine.reset(self._m(mask, l), None if boards is None else boards[l.lo:l.hi],
                           None if sides is None else sides[l.lo:l.hi], None if rr is None else rr[l.lo:l.hi])

    def begin_search(self, playouts, mask=None):
        for l in self.lanes:
            l.engine.begin_search(playouts, self._m(mask, l))

    def unfinished(self):
        return sum(l.engine.unfinished() for l in self.lanes)

    def root_children(self, want_wpq=True):
        parts = [l.engine.root_children(want_wpq) for l in self.lanes]
        return {k: (np.concatenate([p[k] for p in parts]) if parts[0][k] is not None else None) for k in parts[0]}

    def play(self, child_index, want_status=True):
        parts = [l.engine.play(child_index[l.lo:l.hi], want_status) for l in self.lanes]
        return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]} if want_status else None

    def status(self, boards=True):
        parts = [l.engine.status(boards) for l in self.lanes]
        return {k: (np.concatenate([p[k] for p in parts]) if parts[0][k] is not None else None) for k in parts[0]}

    def counters(self):
        cs = [l.engine.counters() for l in self.lanes]
        out = {k: sum(c[k] for c in cs) for k in ("n_expand", "n_playout", "sum_L", "sum_c", "sum_C")}
        out["error"] = 0
        for c in cs:
            out["error"] |= c["error"]
        out["max_arena_words"] = max(c["max_arena_words"] for c in cs)
        out["max_depth"] = max(c["max_depth"] for c in cs)
        out["first_error_game"] = next((l.lo + c["first_error_game"] for l, c in zip(self.lanes, cs) if c["first_error_game"] >= 0), -1)
        return out

    def raise_on_error(self):
        for l in self.lanes:
            l.engine.raise_on_error()
        return self.counters()

    def tree_signature(self, game):
        for l in self.lanes:
            if l.lo <= game < l.hi:
                return l.engine.tree_signature(game - l.lo)
        raise IndexError(game)


class SelfPlay:
    """n_games concurrent self-play games on one engine, advanced in lock-step plies by step().

    Evaluator: pass `plan` (an InferencePlan / NativePlan: it owns the input buffer layout and writes logits / value in
    place), or `forward` = a callable (nn_in) -> (logits [B,2086] f32, value [B] f32) device tensors, which are copied
    into the static buffers the engine reads.  Finished games accumulate in `finished` (slot, GameRecord); long runs
    should drain them with pop_finished()."""

    def __init__(self, n_games, forward, playouts, seeds=None, exploration=True, temperature=1,
                 nn_dtype=torch.float32, arena_words=0, auto_reset=True, device=None, keep_records=True, plan=None,
                 plan_factory=None, lanes=1, engine=None, hashing=False, search_threads=1, compact=None):
        """plan: an InferencePlan / NativePlan (defines the input buffer, writes logits/value in place).
        plan_factory(n) + lanes=2: two half-batches, each with its own engine and plan; the search pipelines them so
        that one half's tree kernel runs under the other half's network (see capture_graph)."""
        self.B = n_games
        # search_threads = K > 1: every game runs the reference's K-coroutine schedule (k_wave_fifo); the network batch has K rows per game
        self.K = max(1, int(search_threads))
        # ... of which only the rows that carry a leaf are evaluated (row compaction, cz_engine_wave_compact): default for K > 1
        self.compact = (self.K > 1 and lanes == 1 and engine is None) if compact is None else bool(compact)
        assert not self.compact or (self.K > 1 and lanes == 1), "row compaction belongs to the search_threads = K engine"
        if lanes > 1:
            assert plan_factory is not None and n_games % lanes == 0
            per = n_games // lanes
            self.lanes = []
            for k in range(lanes):
                eng = Engine(per, arena_words, device)
                dev = torch.device("cuda", eng.device)
                pl = plan_factory(per)
                lg = torch.zeros((per, NLABEL), dtype=torch.float32, device=dev)
                vl = torch.zeros((per,), dtype=torch.float32, device=dev)
                ni = pl.make_input(per)
                self.lanes.append(_Lane(eng, k * per, (k + 1) * per, ni, lg, vl, (lambda x, pl=pl, lg=lg, vl=vl: pl(x, lg, vl))))
            self.engine = _MultiEngine(self.lanes, n_games)
            self.nn_in, self.logits, self.value, forward = None, None, None, None
        else:
            # `engine`: an object with the Engine interface (tests drive the host loop with a CPU stand-in); the product
            # always constructs the CUDA engine here
            self.engine = engine if engine is not None else (Engine(n_games, arena_words, device, search_threads=self.K) if self.K > 1
                                                             else Engine(n_games, arena_words, device))
            if hashing:                              # Zobrist keys of the pending leaves (must be on before a graph is captured)
                self.engine.enable_hashing(True)
            dev = torch.device("cuda", self.engine.device) if engine is None else torch.device(getattr(engine, "torch_device", "cpu"))
            rows = n_games * self.K
            if plan is None and plan_factory is not None:
                plan = plan_factory(rows)
            self.logits = torch.zeros((rows, NLABEL), dtype=torch.float32, device=dev)
            self.value = torch.zeros((rows,), dtype=torch.float32, device=dev)
            if plan is not None:
                self.nn_in = plan.make_input(rows)
                forward = lambda x: plan(x, self.logits, self.value)  # noqa: E731
            else:
                self.nn_in = torch.zeros((rows, 9, 10, 14), dtype=nn_dtype, device=dev)
            if self.compact:                                   # the engine writes every slot's row here; the leaves go densely to nn_in
                self.nn_stage = torch.zeros_like(self.nn_in)
                self._bucket_graphs, self._use_graphs, self._pool = {}, False, None
                self.rows_evaluated = 0
                # batch sizes the network is run at: multiples of the game count (K sizes, one lazily captured CUDA graph each).  Finer
                # buckets evaluate 3.5 % fewer rows but a search then meets dozens of sizes, and capturing their graphs costs more
                # than it saves in anything but a very long run (measured: 2.32 -> 1.81 M exp/s over 6 plies with 256-row buckets)
                self.bucket_rows = n_games
            self.lanes = None
        self.plan = plan
        self.forward = forward
        self.playouts = np.broadcast_to(np.asarray(playouts, dtype=np.int64), (n_games,)).copy()
        seeds = range(n_games) if seeds is None else seeds
        # one legacy MT19937 stream per game slot (stands in for the reference's global np.random, SURVEY H3), held as raw numpy
        # RandomState states: csrc/cz_host.cu draws from them exactly as RandomState.dirichlet / .choice would
        self._mt = np.zeros((n_games, MT_WORDS), dtype=np.uint32)
        for g, sd in enumerate(seeds):
            st = np.random.RandomState(int(sd)).get_state()
            self._mt[g, :624], self._mt[g, 624] = st[1], st[2]
        self._span = [[] for _ in range(n_games)]        # the log entries of each slot's current game
        self.exploration = exploration
        self.temperature = temperature
        self.auto_reset = auto_reset
        self.keep_records = keep_records
        self.records = [GameRecord(g, None, temperature) for g in range(n_games)]
        self._start_board = rules.state_to_board(rules.START_STATE)
        self.boards = np.tile(self._start_board, (n_games, 1))
        self.sides = np.zeros(n_games, dtype=np.uint8)
        self.live = np.ones(n_games, dtype=bool)
        self.finished = []
        self.plies = 0
        self.waves = 0
        self.graph = None
        self._threads = max(1, min(16, (len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else 4)))
        rules._init_tables()

    # -- evaluation step ---------------------------------------------------------------------
    def _eval(self, nn_in):
        out = self.forward(nn_in)
        if out is not None:
            lo, v = out
            self.logits.copy_(lo.reshape(self.B * self.K, NLABEL))
            self.value.copy_(v.reshape(self.B * self.K))

    def _capture_pipeline(self, warmup=3):
        """Two-lane software pipeline in ONE CUDA graph:
              stage 1:  network(A)  ||  k_wave(B)        stage 2:  network(B)  ||  k_wave(A)
        k_wave is a latency-bound kernel (one warp per game, ~17 % issue utilisation), so it runs on a side stream
        underneath the other half-batch's convolutions.  Data flow per replay: network(A) consumes the leaves lane A
        selected in the previous replay (or in the prologue wave), k_wave(B) consumes network(B)'s previous output."""
        A, Bn = self.lanes
        side = torch.cuda.Stream()
        cs = torch.cuda.Stream()
        cs.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(cs):
            for _ in range(warmup):
                A.forward(A.nn_in)
                Bn.forward(Bn.nn_in)
        torch.cuda.current_stream().wait_stream(cs)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=cs):
            side.wait_stream(cs)
            with torch.cuda.stream(side):
                Bn.engine.wave(Bn.nn_in, Bn.logits, Bn.value)
            A.forward(A.nn_in)
            cs.wait_stream(side)
            side.wait_stream(cs)
            with torch.cuda.stream(side):
                A.engine.wave(A.nn_in, A.logits, A.value)
            Bn.forward(Bn.nn_in)
            cs.wait_stream(side)
        self.graph = g

    def _search_pipeline(self, sel):
        e = self.engine
        A, Bn = self.lanes
        for p in np.unique(self.playouts[sel]):
            e.begin_search(int(p), (sel & (self.playouts == p)).astype(np.uint8))
        pmax = int(self.playouts[sel].max()) if sel.any() else 0
        A.engine.wave(A.nn_in, A.logits, A.value)      # prologue: lane A's first leaves
        waves = 1
        while True:
            if self.graph is not None:
                self.graph.replay()
                A.engine.launches += 1
                Bn.engine.launches += 1
            else:
                Bn.engine.wave(Bn.nn_in, Bn.logits, Bn.value)
                A.forward(A.nn_in)
                A.engine.wave(A.nn_in, A.logits, A.value)
                Bn.forward(Bn.nn_in)
            waves += 1
            if waves > pmax and e.unfinished() == 0:
                break
            if waves > 4 * pmax + 64:
                e.raise_on_error()
                raise EngineError("search did not converge")
        self.waves += waves
        return waves

    # -- search_threads = K with row compaction ---------------------------------------------------
    def _eval_rows(self, n):
        """Evaluate the first n rows of the dense batch into logits[:n] / value[:n]."""
        x = self.nn_in[:n]
        if self.plan is not None:
            self.plan(x, self.logits[:n], self.value[:n])
            return
        lo, v = self.forward(x)
        self.logits[:n].copy_(lo.reshape(n, NLABEL))
        self.value[:n].copy_(v.reshape(n))

    def _eval_bucket(self, n_live):
        """The network on n_live rows rounded up to the bucket size (one lazily captured CUDA graph per size, sharing a memory pool)."""
        n = min(self.B * self.K, -(-n_live // self.bucket_rows) * self.bucket_rows)
        self.rows_evaluated += n
        if not self._use_graphs:
            return self._eval_rows(n)
        g = self._bucket_graphs.get(n)
        if g is None:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    self._eval_rows(n)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            if self._pool is None:
                self._pool = torch.cuda.graph_pool_handle()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=self._pool, stream=torch.cuda.Stream()):
                self._eval_rows(n)
            self._bucket_graphs[n] = g
        g.replay()

    def _search_compact(self, sel):
        e = self.engine
        if self.plan is not None and hasattr(self.plan, "refresh_if_stale"):
            self.plan.refresh_if_stale()
        for p in np.unique(self.playouts[sel]):
            e.begin_search(int(p), (sel & (self.playouts == p)).astype(np.uint8))
        pmax = int(self.playouts[sel].max()) if sel.any() else 0
        waves = 0
        while True:
            e.wave_compact(self.nn_stage, self.nn_in, self.logits, self.value)
            n = e.live_rows()                               # stream sync: the host picks the bucket
            waves += 1
            if n > 0:
                self._eval_bucket(n)
            elif e.unfinished() == 0:                       # nothing to evaluate and every search complete
                break
            if waves > 4 * pmax + 64:
                e.raise_on_error()
                raise EngineError("search did not converge")
        self.waves += waves
        return waves

    def capture_graph(self, warmup=3):
        """Capture (wave kernel -> network) into one CUDA graph; the search loop then replays it."""
        if self.lanes is not None:
            return self._capture_pipeline(warmup)
        if self.compact:                                    # the wave runs eagerly (the host reads the row count); the network is one
            self._use_graphs = True                         # graph per bucket size, captured on first use
            return
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self._eval(self.nn_in)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        cs = torch.cuda.Stream()
        with torch.cuda.graph(g, stream=cs):
            self.engine.wave(self.nn_in, self.logits, self.value)
            self._eval(self.nn_in)
        self.graph = g

    def search(self, mask=None):
        """MCTS_tree.main for every live game (mask: only those live games with mask[g]): `playouts[g]` playouts each."""
        sel = self.live if mask is None else self.live & np.asarray(mask, dtype=bool)
        if self.lanes is not None:
            return self._search_pipeline(sel)
        if self.compact:
            return self._search_compact(sel)
        e = self.engine
        if self.plan is not None and hasattr(self.plan, "refresh_if_stale"):
            self.plan.refresh_if_stale()       # weights trained / restored since the last search (the graph reads them in place)
        for p in np.unique(self.playouts[sel]):
            e.begin_search(int(p), (sel & (self.playouts == p)).astype(np.uint8))
        pmax = int(self.playouts[sel].max()) if sel.any() else 0
        waves = 0
        while True:
            if self.graph is not None:
                self.graph.replay()
                e.launches += 1          # the captured k_wave launch
            else:
                e.wave(self.nn_in, self.logits, self.value)
            waves += 1
            if waves > pmax // self.K and e.unfinished() == 0:       # (K leaves per game and wave in the search_threads = K schedule)
                break
            if self.graph is None:
                self._eval(self.nn_in)
            if waves > 4 * pmax + 64:
                e.raise_on_error()
                raise EngineError("search did not converge")
        self.waves += waves
        return waves

    # -- one ply for every live game ------------------------------------------------------------
    def step(self):
        e = self.engine
        self.search()
        rc = e.root_children(want_wpq=False)                      # n, moves, visits: what get_action reads (main.py:1339)
        live = np.nonzero(self.live)[0]
        if (rc["n"][live] <= 0).any():
            e.raise_on_error()
            raise EngineError("game %d has no root children" % int(live[np.argmax(rc["n"][live] <= 0)]))
        nn = np.ascontiguousarray(rc["n"], dtype=np.int32)
        choice = choose_moves(nn, rc["visits"], self.live, self._mt, self.exploration, self.temperature, self._threads)
        if self.keep_records:
            entry = dict(boards=self.boards, n=nn, moves=rc["moves"], visits=rc["visits"], choice=choice)
            for g in live:
                self._span[g].append(entry)
        sides_now = self.sides
        for g in live:
            self.records[g].players.append(int(sides_now[g]))
        st = e.play(choice)                                          # board update + re-root + status, one synchronisation
        win_rate = np.where(choice >= 0, st["q"], 0.0).astype(np.float32)                 # mcts.Q(act), main.py:1350
        self.boards, self.sides = st["boards"], st["side"]
        self.plies += int(self.live.sum())
        done_now = []
        for g in np.nonzero(self.live & (st["terminal"] != 0))[0]:
            rec = self.records[g]
            players = np.asarray(rec.players)
            if st["terminal"][g] == 1:                                                   # main.py:1532-1541
                w = int(st["winner"][g])
                rec.z = np.where(players == w, 1.0, -1.0)
                rec.winner = "w" if w == 0 else "b"
            else:                                                                        # main.py:1542-1545
                rec.z = np.zeros(len(players))
                rec.winner = "t"
            rec._logs, rec._T = self._span[g], self.temperature
            self._span[g] = []
            done_now.append((int(g), rec))
            self.finished.append((int(g), rec))
            self.records[g] = GameRecord(int(g), None, self.temperature)
        if done_now:
            idx = [g for g, _ in done_now]
            if self.auto_reset:
                mask = np.zeros(self.B, dtype=np.uint8)
                mask[idx] = 1
                e.reset(mask)                                                            # GameBoard.reload + mcts.reload
                st = {k: v.copy() for k, v in st.items()}
                st["boards"][idx] = self._start_board                                    # what reload() leaves: no second status read
                st["side"][idx] = 0
                st["terminal"][idx] = 0
                st["winner"][idx] = -1
                st["ply"][idx] = 0
                st["rr"][idx] = 0
                self.boards, self.sides = st["boards"], st["side"]
            else:
                self.live[idx] = False
        return dict(choice=choice, win_rate=win_rate, finished=done_now, status=st)

    def pop_finished(self):
        """Hand over (and forget) the games finished so far: keeps memory flat in long self-play runs."""
        out, self.finished = self.finished, []
        return out

    def play_games(self, max_plies=100000):
        """Every slot plays ONE game to the end (auto_reset must be False)."""
        assert not self.auto_reset
        n = 0
        while self.live.any() and n < max_plies:
            self.step()
            n += 1
        self.engine.raise_on_error()
        return sorted(self.finished, key=lambda t: t[0])


# =================================================================================================
# Reference-shaped facade: cchess_main (main.py:1118-1554).  One game at a time through MCTS_tree,
# exactly the call sequence of the reference, so main.py's train loop runs unchanged on top of it.
# For throughput use SelfPlay (thousands of games per GPU); `selfplay_many` bridges the two.
# =================================================================================================
def save_replay(path, data_buffer, extra=None):
    """Persist the replay deque (main.py:1138-1139 keeps it in memory only) together with the global numpy / python RNG
    states, so that a training run can resume exactly where it stopped (SURVEY 8(f)2).  Atomic: write + rename."""
    blob = dict(data=list(data_buffer), maxlen=getattr(data_buffer, "maxlen", None), np_state=np.random.get_state(),
                py_state=random.getstate(), extra=dict(extra or {}))
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        pickle.dump(blob, f, protocol=pickle.HIGHEST_PROTOCOL)
    os.replace(tmp, path)


def load_replay(path, restore_rng=True):
    """-> (deque, extra).  With restore_rng the numpy / python global RNGs continue from the saved point."""
    with open(path, "rb") as f:
        blob = pickle.load(f)
    if restore_rng:
        np.random.set_state(blob["np_state"])
        random.setstate(blob["py_state"])
    return deque(blob["data"], maxlen=blob["maxlen"]), blob["extra"]


class cchess_main(object):

    def __init__(self, playout=400, in_batch_size=128, exploration=True, in_search_threads=16, processor="cpu",
                 num_gpus=1, res_block_nums=7, human_color="b", network=None, log_file=True, leaf_parallel=1):
        from .mcts import MCTS_tree
        from .net import policy_value_network, policy_value_network_gpus
        rules._init_tables()
        self.epochs = 5
        self.playout_counts = playout
        self.temperature = 1
        self.batch_size = in_batch_size
        self.game_batch = 400
        self.top_steps = 30
        self.top_temperature = 1
        self.eta = 0.03
        self.learning_rate = 0.001
        self.lr_multiplier = 1.0
        self.buffer_size = 10000
        self.data_buffer = deque(maxlen=self.buffer_size)
        self.game_borad = rules.GameBoard()
        if network is not None:
            self.policy_value_netowrk = network
        else:  # `processor` selected CPU/GPU TensorFlow in the reference (main.py:1142); both map to the CUDA net here
            self.policy_value_netowrk = policy_value_network(res_block_nums) if processor == "cpu" else policy_value_network_gpus(num_gpus, res_block_nums)
        self.search_threads = in_search_threads
        self.mcts = MCTS_tree(self.game_borad.state, self.policy_value_netowrk.forward, self.search_threads, leaf_parallel=leaf_parallel)
        self.exploration = exploration
        self.resign_threshold = -0.8
        self.global_step = 0
        self.kl_targ = 0.025
        self.log_file = open(os.path.join(os.getcwd(), "log_file.txt"), "w") if log_file else None
        self.human_color = human_color

    @staticmethod
    def flip_policy(prob):  # main.py:1152-1155
        prob = np.asarray(prob).flatten()
        return np.asarray([prob[i] for i in rules.unflipped_index])

    # ---- training (main.py:1157-1205) ------------------------------------------------------------
    def policy_update(self):
        mini_batch = random.sample(self.data_buffer, self.batch_size)
        state_batch = [d[0] for d in mini_batch]
        mcts_probs_batch = [d[1] for d in mini_batch]
        winner_batch = np.expand_dims([d[2] for d in mini_batch], 1)
        start_time = time.time()
        old_probs, old_v = self.mcts.forward(state_batch)
        kl, loss, accuracy, new_v = 0.0, 0.0, 0.0, old_v
        for _ in range(self.epochs):
            accuracy, loss, self.global_step = self.policy_value_netowrk.train_step(
                state_batch, mcts_probs_batch, winner_batch, self.learning_rate * self.lr_multiplier)
            new_probs, new_v = self.mcts.forward(state_batch)
            with np.errstate(all="ignore"):
                kl_tmp = old_probs * (np.log((old_probs + 1e-10) / (new_probs + 1e-10)))
            # main.py:1178-1182 drops the terms whose str() is 'nan' or 'inf' -- and therefore KEEPS '-inf' (logits are used as
            # probabilities, so negative old_probs are routine and a row sum can legitimately be -inf)
            kl = np.mean([np.sum(line[~(np.isnan(line) | np.isposinf(line))]) for line in kl_tmp])
            if kl > self.kl_targ * 4:
                break
        self.policy_value_netowrk.save(self.global_step)
        print("train using time {} s".format(time.time() - start_time))
        if kl > self.kl_targ * 2 and self.lr_multiplier > 0.1:
            self.lr_multiplier /= 1.5
        elif kl < self.kl_targ / 2 and self.lr_multiplier < 10:
            self.lr_multiplier *= 1.5
        wb = np.array(winner_batch)
        explained_var_old = 1 - np.var(wb - old_v.flatten()) / np.var(wb)
        explained_var_new = 1 - np.var(wb - new_v.flatten()) / np.var(wb)
        msg = "kl:{:.5f},lr_multiplier:{:.3f},loss:{},accuracy:{},explained_var_old:{:.3f},explained_var_new:{:.3f}".format(
            kl, self.lr_multiplier, loss, accuracy, explained_var_old, explained_var_new)
        print(msg)
        if self.log_file:
            self.log_file.write(msg + "\n")
            self.log_file.flush()

    def save_state(self, path):
        """Replay buffer + lr multiplier + step + RNG states (the reference checkpoints only the network weights)."""
        save_replay(path, self.data_buffer, dict(lr_multiplier=self.lr_multiplier, global_step=self.global_step))

    def load_state(self, path):
        self.data_buffer, extra = load_replay(path)
        self.lr_multiplier = extra.get("lr_multiplier", self.lr_multiplier)
        self.global_step = extra.get("global_step", self.global_step)

    def policy_evaluate(self, opponent, n_games=10):
        """main.py:1207-1222 (commented out in the reference): n_games matches of this object's network against `opponent` (a
        cchess_main or a network), colours alternating, both sides with this object's playout_counts / search_threads, played
        concurrently by arena.Arena.  Returns the reference's win_ratio = (win + 0.5 * tie) / n_games."""
        from .arena import Arena
        opp = getattr(opponent, "policy_value_netowrk", opponent)
        s = Arena(self.policy_value_netowrk, opp, n_games, self.playout_counts, search_threads_a=self.search_threads,
                  temperature=self.temperature).play().summary()
        print("num_playouts:{}, win: {}, lose: {}, tie:{}".format(self.playout_counts, s["w"], s["l"], s["d"]))
        return s["win_ratio"]

    def run(self, max_batches=None):  # main.py:1224-1248
        batch_iter = 0
        try:
            while max_batches is None or batch_iter < max_batches:
                batch_iter += 1
                play_data, episode_len = self.selfplay()
                print("batch i:{}, episode_len:{}".format(batch_iter, episode_len))
                extend_data = []
                for state, mcts_prob, winner in play_data:
                    extend_data.append((self.mcts.state_to_positions(state), mcts_prob, winner))
                self.data_buffer.extend(extend_data)
                if len(self.data_buffer) > self.batch_size:
                    self.policy_update()
        except KeyboardInterrupt:
            if self.log_file:
                self.log_file.close()
            self.policy_value_netowrk.save(self.global_step)

    # ---- move choice (main.py:1278-1358) -----------------------------------------------------------
    def _visit_probs(self):
        actions_visits = [(act, nod.N) for act, nod in self.mcts.root.child.items()]
        actions, visits = zip(*actions_visits)
        with np.errstate(divide="ignore"):
            probs = rules.softmax(1.0 / self.temperature * np.log(visits))
        return actions, probs

    def get_hint(self, mcts_or_net, reverse, disp_mcts_msg_handler):
        act_prob_dict = defaultdict(float)
        if mcts_or_net == "mcts":
            if self.mcts.root.child == {}:
                disp_mcts_msg_handler()
                self.mcts.main(self.game_borad.state, self.game_borad.current_player, self.game_borad.restrict_round, self.playout_counts)
            actions, probs = self._visit_probs()
            for i in range(len(actions)):
                action = "".join(rules.flipped_uci_labels(actions[i])) if self.human_color == "w" else actions[i]
                act_prob_dict[action] = probs[i]
        elif mcts_or_net == "net":
            moves, p, _ = self._net_priors()
            for action, mov_p in zip(moves, p):
                if self.human_color == "w":
                    action = "".join(rules.flipped_uci_labels(action))
                act_prob_dict[action] = mov_p
        return sorted(act_prob_dict.items(), key=lambda item: item[1], reverse=reverse)

    def _net_priors(self):
        """The 'net' branches of get_hint / select_move (main.py:1300-1324, 1437-1459)."""
        positions = self.mcts.generate_inputs(self.game_borad.state, self.game_borad.current_player)
        action_probs, value = self.mcts.forward(np.expand_dims(positions, 0))
        if self.mcts.is_black_turn(self.game_borad.current_player):
            action_probs = cchess_main.flip_policy(action_probs)
        moves = rules.GameBoard.get_legal_moves(self.game_borad.state, self.game_borad.current_player)
        action_probs = np.asarray(action_probs).flatten()
        tot_p = 1e-8
        p = []
        for action in moves:
            mov_p = action_probs[rules.label2i[action]]
            p.append(mov_p)
            tot_p += mov_p
        return moves, [x / tot_p for x in p], value

    def get_action(self, state, temperature=1e-3):
        self.mcts.main(state, self.game_borad.current_player, self.game_borad.restrict_round, self.playout_counts)
        actions_visits = [(act, nod.N) for act, nod in self.mcts.root.child.items()]
        actions, visits = zip(*actions_visits)
        with np.errstate(divide="ignore"):
            probs = rules.softmax(1.0 / temperature * np.log(visits))
        move_probs = [[actions, probs]]
        if self.exploration:
            act = np.random.choice(actions, p=0.75 * probs + 0.25 * np.random.dirichlet(0.3 * np.ones(len(probs))))
        else:
            act = np.random.choice(actions, p=probs)
        win_rate = self.mcts.Q(act)
        self.mcts.update_tree(act)
        return act, move_probs, win_rate

    # ---- game flow (main.py:1380-1554) -------------------------------------------------------------
    def check_end(self):
        st = self.game_borad.state
        if st.find("K") == -1 or st.find("k") == -1:
            if st.find("K") == -1:
                print("Green is Winner")
                return True, "b"
            print("Red is Winner")
            return True, "w"
        elif self.game_borad.restrict_round >= 60:
            print("TIE! No Winners!")
            return True, "t"
        return False, ""

    def _advance(self, action):
        """state / round / player / restrict_round bookkeeping shared by human_move, select_move, selfplay."""
        last_state = self.game_borad.state
        self.game_borad.state = rules.GameBoard.sim_do_action(action, self.game_borad.state)
        self.game_borad.round += 1
        self.game_borad.current_player = "w" if self.game_borad.current_player == "b" else "b"
        if rules.is_kill_move(last_state, self.game_borad.state) == 0:
            self.game_borad.restrict_round += 1
        else:
            self.game_borad.restrict_round = 0

    def human_move(self, coord, mcts_or_net):
        win_rate = 0
        action = "abcdefghi"[coord[0]] + str(coord[1]) + "abcdefghi"[coord[2]] + str(coord[3])
        if self.human_color == "w":
            action = "".join(rules.flipped_uci_labels(action))
        if mcts_or_net == "mcts":
            if self.mcts.root.child == {}:
                self.mcts.main(self.game_borad.state, self.game_borad.current_player, self.game_borad.restrict_round, self.playout_counts)
            win_rate = self.mcts.Q(action)
            self.mcts.update_tree(action)
        self._advance(action)
        return win_rate

    def select_move(self, mcts_or_net):
        if mcts_or_net == "mcts":
            action, probs, win_rate = self.get_action(self.game_borad.state, self.temperature)
        else:
            moves, p, value = self._net_priors()
            win_rate = value[0, 0]
            action = max(zip(moves, p), key=lambda t: t[1])[0]   # first maximum wins, main.py:1461
        print("Win rate for player {} is {:.4f}".format(self.game_borad.current_player, win_rate))
        print(self.game_borad.current_player, " now take a action : ", action, "[Step {}]".format(self.game_borad.round))
        self._advance(action)
        self.game_borad.print_borad(self.game_borad.state)
        if self.human_color == "w":
            action = "".join(rules.flipped_uci_labels(action))
        sx, sy, dx, dy = ord(action[0]) - 97, int(action[1]), ord(action[2]) - 97, int(action[3])
        return (sx, sy, dx - sx, dy - sy), win_rate

    def selfplay(self):
        self.game_borad.reload()
        states, mcts_probs, current_players = [], [], []
        z = None
        game_over = False
        start_time = time.time()
        while not game_over:
            action, probs, win_rate = self.get_action(self.game_borad.state, self.temperature)
            black = self.mcts.is_black_turn(self.game_borad.current_player)
            state, _ = self.mcts.try_flip(self.game_borad.state, self.game_borad.current_player, black)
            states.append(state)
            prob = np.zeros(rules.labels_len)
            for a, pr in zip(probs[0][0], probs[0][1]):
                prob[rules.label2i["".join(rules.flipped_uci_labels(a)) if black else a]] = pr
            mcts_probs.append(prob)
            current_players.append(self.game_borad.current_player)
            self._advance(action)
            st = self.game_borad.state
            if st.find("K") == -1 or st.find("k") == -1:
                winnner = "b" if st.find("K") == -1 else "w"
                z = np.zeros(len(current_players))
                z[np.array(current_players) == winnner] = 1.0
                z[np.array(current_players) != winnner] = -1.0
                game_over = True
                print("Game end. Winner is player : ", winnner, " In {} steps".format(self.game_borad.round - 1))
            elif self.game_borad.restrict_round >= 60:
                z = np.zeros(len(current_players))
                game_over = True
                print("Game end. Tie in {} steps".format(self.game_borad.round - 1))
            if game_over:
                self.mcts.reload()
        print("Using time {} s".format(time.time() - start_time))
        return zip(states, mcts_probs, z), len(z)

    # ---- batched bridge: many games at once on this rank's GPU ---------------------------------------
    def selfplay_many(self, n_games, seeds=None, arena_words=0):
        """Plays n_games concurrent games with the engine's lock-step waves and returns a list of
        (zip(states, mcts_probs, z), n) -- the same tuples selfplay() yields, one entry per game."""
        net = self.policy_value_netowrk
        plan = net.plan()
        sp = SelfPlay(n_games, None, self.playout_counts, seeds=seeds, exploration=self.exploration, temperature=self.temperature,
                      arena_words=arena_words, auto_reset=False, plan=plan)
        return [(rec.tuples(), len(rec)) for _, rec in sp.play_games()]
