"""Batched head-to-head matches between two networks on one GPU (the evaluation the reference planned as
cchess_main.policy_evaluate, main.py:1207-1222, and never finished).

One match is two play-mode cchess_main objects (exploration=False, temperature 1) facing each other, each with its own network,
MCTS_tree, playout_counts and search_threads.  Every ply:
  1. the mover runs select_move('mcts') = get_action(state, 1) (main.py:1332-1358): playout_counts more playouts on its reused
     tree, np.random.choice(actions, p=softmax(log(visits)/T)), win_rate = Q(act), update_tree(act);
  2. the other player runs human_move(coord, 'mcts') (main.py:1394-1430): if its root was never expanded it first searches
     playout_counts playouts on the PRE-move position (so black's tree searches the start position before red's first move is
     applied), then Q(act) and update_tree(act), which keeps the subtree;
  3. the game ends as check_end says (main.py:1380-1392): a king captured, or restrict_round >= 60 is a tie.
All M matches run in lock-step.  Each player is one SelfPlay-owned search path (its own engine, evaluator buffers and CUDA graphs;
row-compacted for search_threads > 1), searched on the games it has to search; the opponent's move reaches its tree through
cz_engine_play_moves.  One legacy MT19937 stream per match, seeded from seeds[m], stands in for the global np.random; only the
mover's choice draws from it.

    python -m cchess_zero_b200.arena --a CKPT_A --b CKPT_B --matches 400 --playouts 400 --search_threads 16 --seed 0
prints one JSON line: the summary from A's side, the settings and the device name."""
import argparse
import json
import math
import os
import sys

import numpy as np

from ._lib import MT_WORDS, NOMOVE, EngineError


def elo(score):
    """Elo difference of an expected score: -400 log10(1/score - 1); -inf at 0, +inf at 1."""
    if score <= 0.0:
        return -math.inf
    if score >= 1.0:
        return math.inf
    return -400.0 * math.log10(1.0 / score - 1.0)


def summarize(a_red, winners):
    """Result of a match set from A's side.  a_red[m]: A played red in match m; winners[m]: 'w' (red won), 'b' (black won) or 't'.

    score = (W + D/2) / n, the reference's win_ratio (main.py:1219); elo = -400 log10(1/score - 1); the 95 % interval maps
    score -+ 1.96 sqrt(var / n) through the same formula, var = (W (1-s)^2 + D (1/2-s)^2 + L s^2) / n the per-game score variance.
    When every game scored 1 (or 0) that variance is 0; the finite side of the interval is then the rule-of-three bound
    1 - 3/n (3/n) on the score.  los = 1/2 (1 + erf((W-L) / sqrt(2 (W+L)))), 1/2 when there are no decisive games."""
    a_red = np.asarray(a_red, dtype=bool)
    winners = np.asarray(winners)
    if a_red.shape != winners.shape or a_red.ndim != 1 or a_red.size == 0:
        raise ValueError("a_red and winners must be two non-empty lists of the same length")
    if not np.isin(winners, ["w", "b", "t"]).all():
        raise ValueError("winners must be 'w', 'b' or 't'")
    a_won = np.where(a_red, winners == "w", winners == "b")
    draw = winners == "t"
    a_lost = ~a_won & ~draw

    def wdl(sel):
        return dict(w=int((a_won & sel).sum()), d=int((draw & sel).sum()), l=int((a_lost & sel).sum()))

    n = int(a_red.size)
    W, D, L = int(a_won.sum()), int(draw.sum()), int(a_lost.sum())
    s = (W + 0.5 * D) / n
    var = (W * (1.0 - s) ** 2 + D * (0.5 - s) ** 2 + L * s ** 2) / n
    half = 1.96 * math.sqrt(var / n)
    lo, hi = s - half, s + half
    if var == 0.0 and s == 1.0:
        lo = 1.0 - 3.0 / n
    elif var == 0.0 and s == 0.0:
        hi = 3.0 / n
    red_score = (int((winners == "w").sum()) + 0.5 * D) / n
    los = 0.5 if W + L == 0 else 0.5 * (1.0 + math.erf((W - L) / math.sqrt(2.0 * (W + L))))
    return dict(n=n, w=W, d=D, l=L, as_red=wdl(a_red), as_black=wdl(~a_red), score=s, win_ratio=s, elo=elo(s),
                elo_95=[elo(lo), elo(hi)], los=los, red_score=red_score)


class ArenaResult:
    """Per match: A's colour, the winner ('w' / 'b' / 't'), the ply count, the moves (src | dst << 7) and both players' Q(act) of
    every move (A's tree and B's tree, float32)."""

    def __init__(self, a_red, winner, plies, moves, q_a, q_b):
        self.a_red, self.winner, self.plies, self.moves, self.q_a, self.q_b = a_red, winner, plies, moves, q_a, q_b

    def __len__(self):
        return len(self.a_red)

    def match(self, m):
        from . import rules
        return dict(a_colour="w" if self.a_red[m] else "b", winner=self.winner[m], plies=int(self.plies[m]),
                    moves=[rules.move_to_label(int(x)) for x in self.moves[m]],
                    q_a=np.asarray(self.q_a[m], dtype=np.float32), q_b=np.asarray(self.q_b[m], dtype=np.float32))

    def summary(self):
        return summarize(self.a_red, self.winner)


def _search_path(net, n, playouts, K, temperature, arena_words, device):
    """One player's SelfPlay-owned search path: its own engine, evaluator buffers and CUDA graphs.  `net`: a policy_value_network,
    an inference plan (make_input / __call__(x, logits, value)), or a callable x -> (logits, value) such as FakeNet."""
    from .selfplay import SelfPlay
    kw = dict(exploration=False, temperature=temperature, arena_words=arena_words, auto_reset=False, keep_records=False,
              device=device, search_threads=K)
    if hasattr(net, "native_plan"):             # policy_value_network: the evaluator the self-play benchmark uses for it
        factory = (lambda rows: net.native_plan(rows)) if net.precision == "fp16" else (lambda rows: net.plan())
        sp = SelfPlay(n, None, playouts, plan_factory=factory, **kw)
    elif hasattr(net, "make_input"):
        sp = SelfPlay(n, None, playouts, plan=net, **kw)
    elif callable(net):
        sp = SelfPlay(n, net, playouts, **kw)
    else:
        raise TypeError("a network must be a policy_value_network, an inference plan or a callable evaluator")
    sp.capture_graph()
    return sp


class Arena:
    def __init__(self, net_a, net_b, n_matches, playouts_a, playouts_b=None, search_threads_a=16, search_threads_b=None,
                 temperature=1, seeds=None, a_red=None, arena_words=0, device=None):
        """n_matches concurrent matches of net_a against net_b.  Unset *_b arguments copy the *_a value.  a_red[m]: A plays red in
        match m (default: even slots).  seeds[m]: seed of match m's MT19937 stream (default m)."""
        playouts_b = playouts_a if playouts_b is None else playouts_b
        search_threads_b = search_threads_a if search_threads_b is None else search_threads_b
        M = int(n_matches)
        if M < 1:
            raise ValueError("n_matches must be >= 1")
        for name, v, lo, hi in (("playouts_a", playouts_a, 1, None), ("playouts_b", playouts_b, 1, None),
                                ("search_threads_a", search_threads_a, 1, 32), ("search_threads_b", search_threads_b, 1, 32)):
            if int(v) != v or v < lo or (hi is not None and v > hi):
                raise ValueError("%s must be an integer in [%d, %s]" % (name, lo, hi or "inf"))
        self.M = M
        self.a_red = (np.arange(M) % 2 == 0) if a_red is None else np.asarray(a_red, dtype=bool).copy()
        seeds = range(M) if seeds is None else seeds
        if self.a_red.shape != (M,) or len(seeds) != M:
            raise ValueError("a_red and seeds need one entry per match")
        self.temperature = temperature
        self.settings = dict(matches=M, playouts_a=int(playouts_a), playouts_b=int(playouts_b), search_threads_a=int(search_threads_a),
                             search_threads_b=int(search_threads_b), temperature=temperature)
        self.players = (_search_path(net_a, M, int(playouts_a), int(search_threads_a), temperature, arena_words, device),
                        _search_path(net_b, M, int(playouts_b), int(search_threads_b), temperature, arena_words, device))
        self._mt = np.zeros((M, MT_WORDS), dtype=np.uint32)
        for m, sd in enumerate(seeds):
            st = np.random.RandomState(int(sd)).get_state()
            self._mt[m, :624], self._mt[m, 624] = st[1], st[2]
        self.side = np.zeros(M, dtype=np.uint8)           # side to move: 0 red ('w'), 1 black
        self.live = np.ones(M, dtype=bool)
        self.winner = np.full(M, "", dtype=object)
        self.plies = np.zeros(M, dtype=np.int64)
        self.moves = [[] for _ in range(M)]
        self.q_a = [[] for _ in range(M)]
        self.q_b = [[] for _ in range(M)]
        self.boards = None

    def step(self):
        """One ply of every running match.  Returns dict(a_moves (bool [M]: A was the mover), move (uint16 [M], NOMOVE where the
        match had already ended), n / visits (the mover's root children and visit counts, [M] / [M][128]), q_a / q_b (float32 [M]),
        status (A's engine status records after the move))."""
        A, B = self.players
        live = self.live.copy()
        a_moves = live & ((self.side == 0) == self.a_red)
        b_moves = live & ~a_moves
        # the mover searches (get_action); the other player searches first only where its root was never expanded (human_move)
        pre_a = A.engine.root_children(want_wpq=False)["n"] < 0
        pre_b = B.engine.root_children(want_wpq=False)["n"] < 0
        A.search(a_moves | (b_moves & pre_a))
        B.search(b_moves | (a_moves & pre_b))
        rca = A.engine.root_children(want_wpq=False)
        rcb = B.engine.root_children(want_wpq=False)
        n = np.where(a_moves, rca["n"], rcb["n"]).astype(np.int32)
        if (n[live] <= 0).any():
            for p in self.players:
                p.engine.raise_on_error()
            raise EngineError("match %d has no root children" % int(np.nonzero(live & (n <= 0))[0][0]))
        visits = np.where(a_moves[:, None], rca["visits"], rcb["visits"])
        root_moves = np.where(a_moves[:, None], rca["moves"], rcb["moves"])
        from .selfplay import choose_moves
        choice = choose_moves(n, visits, live, self._mt, False, self.temperature, A._threads)
        move = np.full(self.M, NOMOVE, dtype=np.uint16)
        idx = np.nonzero(live)[0]
        move[idx] = root_moves[idx, choice[idx]]
        sa = A.engine.play_moves(move)
        sb = B.engine.play_moves(move)
        if not np.array_equal(sa["boards"][idx], sb["boards"][idx]):
            raise EngineError("the two players' boards diverged")
        for m in idx:
            self.moves[m].append(int(move[m]))
            self.q_a[m].append(sa["q"][m])
            self.q_b[m].append(sb["q"][m])
        self.plies[idx] += 1
        self.side = sa["side"].copy()
        self.boards = sa["boards"]
        for m in np.nonzero(live & (sa["terminal"] != 0))[0]:
            self.live[m] = False
            self.winner[m] = "t" if sa["terminal"][m] == 2 else ("w" if sa["winner"][m] == 0 else "b")
        return dict(a_moves=a_moves, move=move, n=n, visits=visits, q_a=sa["q"].copy(), q_b=sb["q"].copy(), status=sa)

    def play(self):
        """Plays every match to its end (the rules bound a game's length) and returns the ArenaResult."""
        while self.live.any():
            self.step()
        return self.result()

    def result(self):
        return ArenaResult(self.a_red.copy(), list(self.winner), self.plies.copy(), [list(x) for x in self.moves],
                           [list(x) for x in self.q_a], [list(x) for x in self.q_b])


# ---- command line --------------------------------------------------------------------------------------------------------------
PRECISIONS = ("fp16", "bf16", "tf32", "tf32x3", "fp32")


def parse_args(argv=None):
    """Parses and checks the command line; every error is reported here, before any GPU work."""
    ap = argparse.ArgumentParser(prog="python -m cchess_zero_b200.arena", description=__doc__.split("\n\n")[0])
    ap.add_argument("--a", required=True, help="checkpoint of network A (policy_value_network.save)")
    ap.add_argument("--b", required=True, help="checkpoint of network B")
    ap.add_argument("--res_block_nums_a", type=int, default=7)
    ap.add_argument("--res_block_nums_b", type=int, default=None, help="default: --res_block_nums_a")
    ap.add_argument("--matches", type=int, default=400)
    ap.add_argument("--playouts", type=int, default=400)
    ap.add_argument("--playouts_b", type=int, default=None, help="default: --playouts")
    ap.add_argument("--search_threads", type=int, default=16)
    ap.add_argument("--search_threads_b", type=int, default=None, help="default: --search_threads")
    ap.add_argument("--seed", type=int, default=0, help="match m draws from a MT19937 stream seeded with seed + m")
    ap.add_argument("--precision", default="fp16", choices=PRECISIONS)
    ap.add_argument("--arena_words", type=int, default=0, help="tree storage per game and half, uint32 words (0: engine default)")
    a = ap.parse_args(argv)
    a.res_block_nums_b = a.res_block_nums_a if a.res_block_nums_b is None else a.res_block_nums_b
    a.playouts_b = a.playouts if a.playouts_b is None else a.playouts_b
    a.search_threads_b = a.search_threads if a.search_threads_b is None else a.search_threads_b
    for f in (a.a, a.b):
        if not os.path.isfile(f):
            ap.error("checkpoint not found: %s" % f)
    if a.matches < 1:
        ap.error("--matches must be >= 1")
    if min(a.playouts, a.playouts_b) < 1:
        ap.error("--playouts must be >= 1")
    if not (1 <= a.search_threads <= 32 and 1 <= a.search_threads_b <= 32):
        ap.error("--search_threads must be in [1, 32]")
    if min(a.res_block_nums_a, a.res_block_nums_b) < 1:
        ap.error("--res_block_nums must be >= 1")
    if a.arena_words < 0:
        ap.error("--arena_words must be >= 0")
    if a.seed < 0:
        ap.error("--seed must be >= 0")
    return a


def main(argv=None):
    a = parse_args(argv)
    import torch
    from .net import policy_value_network

    def load(path, blocks):
        # save_dir: a directory that cannot hold a `checkpoint` index, so the constructor restores nothing of its own
        net = policy_value_network(blocks, precision=a.precision, save_dir=os.devnull)
        net.restore(path)
        return net

    stdout = sys.stdout
    sys.stdout = sys.stderr                           # restore() and the network constructor print; the JSON line goes alone to stdout
    try:
        net_a, net_b = load(a.a, a.res_block_nums_a), load(a.b, a.res_block_nums_b)
        ar = Arena(net_a, net_b, a.matches, a.playouts, a.playouts_b, a.search_threads, a.search_threads_b,
                   seeds=[a.seed + m for m in range(a.matches)], arena_words=a.arena_words)
        res = ar.play()
    finally:
        sys.stdout = stdout
    out = dict(summary=res.summary(), settings=dict(ar.settings, a=a.a, b=a.b, res_block_nums_a=a.res_block_nums_a,
                                                        res_block_nums_b=a.res_block_nums_b, seed=a.seed, precision=a.precision),
               device=torch.cuda.get_device_name(), mean_plies=float(np.mean(res.plies)))
    print(json.dumps(out))
    return out


if __name__ == "__main__":
    main()
