"""TEST INFRASTRUCTURE ONLY -- the arena protocol (two play-mode cchess_main objects facing each other) restated over two C trees.

The executable specification of cchess_zero_b200.arena: per ply the mover runs get_action(state, 1) (main.py:1332-1358: search,
np.random.choice over softmax(log(visits)), Q(act), update_tree(act)); the other player runs human_move(coord, 'mcts')
(main.py:1394-1430: a search of its own first if its root was never expanded -- on the PRE-move position -- then Q(act) and
update_tree(act)).  tests/golden/arena.json.gz holds the same matches played by the unmodified reference (oracle/gen_golden_arena.py)."""
import hashlib

import numpy as np

from oracle import oracle as O


def tree_digest(sig_a, sig_b):
    """Digest of both players' tree signatures (records of 6 int64: label index, N, W / P / Q bits, n_children; A's tree first)."""
    a = np.ascontiguousarray(np.asarray(sig_a, dtype=np.int64).reshape(-1, 6))
    b = np.ascontiguousarray(np.asarray(sig_b, dtype=np.int64).reshape(-1, 6))
    return hashlib.sha256(np.int64(len(a)).tobytes() + a.tobytes() + b.tobytes()).hexdigest()[:16]


def f32_hex(x):
    return "%08x" % int(np.float32(x).view(np.uint32))


def _search(tree, side, rr, p):
    err = tree.search(side, rr, p["playouts"], p["net"]) if p["K"] <= 1 else tree.search_fifo(side, rr, p["playouts"], p["K"], p["net"])
    if err:
        raise RuntimeError("oracle tree error %d" % err)


def arena_game(a, b, a_red, seed, temperature=1):
    """One match.  a / b: dict(net=<stand-in net name>, playouts=..., K=<search_threads>).  Returns dict(winner, plies, ply) with one
    entry [mover 'a' / 'b', action, mover's visits, mover's Q(act) f32 hex, other's Q(act) f32 hex, tree digest (A, B)] per ply."""
    rs = np.random.RandomState(seed)
    trees = dict(a=O.Tree(), b=O.Tree())
    players = dict(a=a, b=b)
    red, black = ("a", "b") if a_red else ("b", "a")
    board = O.from_state(O.START)
    side, rr = 0, 0
    plies = []
    with np.errstate(divide="ignore"):
        while True:
            mover = red if side == 0 else black
            other = black if side == 0 else red
            tm, to = trees[mover], trees[other]
            _search(tm, side, rr, players[mover])                           # get_action: MCTS_tree.main on the reused tree
            mv, N, W, P, Q = tm.root_children()
            visits = [int(v) for v in N]
            probs = O.softmax(1.0 / temperature * np.log(visits))
            acts = [O.move_str(m) for m in mv]
            act = rs.choice(acts, p=probs)
            idx = acts.index(act)
            q_mover = Q[idx]
            tm.update(idx)
            if len(to.root_children()[0]) == 0:                             # human_move: root.child == {} -> search first
                _search(to, side, rr, players[other])
            omv = list(to.root_children()[0])
            if int(mv[idx]) not in omv:
                raise KeyError(act)                                         # update_tree's KeyError (main.py:275)
            oidx = omv.index(int(mv[idx]))
            q_other = to.root_children()[4][oidx]
            to.update(oidx)
            plies.append([mover, act, visits, f32_hex(q_mover), f32_hex(q_other), tree_digest(trees["a"].signature(), trees["b"].signature())])
            board, cap = O.apply_move(board, mv[idx])
            side ^= 1
            rr = rr + 1 if cap == 0 else 0
            hasK, hask = (board == 1).any(), (board == 8).any()
            if not hasK:
                return dict(winner="b", plies=len(plies), ply=plies)
            if not hask:
                return dict(winner="w", plies=len(plies), ply=plies)
            if rr >= 60:
                return dict(winner="t", plies=len(plies), ply=plies)
