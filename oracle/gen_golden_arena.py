"""TEST INFRASTRUCTURE ONLY -- golden arena matches of the UNMODIFIED reference: two play-mode cchess_main objects facing each other.

Each match is two reference cchess_main objects (ref_harness.make_cchess_main, exploration=False, the stand-in nets of
fakenets_np.py) driven through their own select_move('mcts') (main.py:1437-1470, get_action 1332-1358) and human_move(coord, 'mcts')
(main.py:1394-1430) until check_end (1380-1392) ends the game.  search_threads > 1 runs each tree on its own deterministic event loop
(detloop.DetLoop("busy")), as gen_golden_k16_selfplay.py does.  np.random.seed(seed) comes after both objects are built.  Recorded
per ply: the mover, the action, the mover's visit counts (read as update_tree is called), both Q(act) as float32 bits and a digest
of both trees' signatures (oracle_arena.tree_digest over ref_harness.tree_signature).

    python oracle/gen_golden_arena.py        ->  tests/golden/arena.json.gz
"""
import asyncio
import gzip
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle.oracle_arena import f32_hex, tree_digest   # noqa: E402  (before HERE goes on the path: `oracle` is the package)
sys.path.insert(0, HERE)
import detloop as D          # noqa: E402
import ref_harness as H      # noqa: E402

# (name, A, B, seeds); every pairing is played with A as red and with A as black
PAIRINGS = [
    ("different nets, K=1", dict(net="hash_pos", playouts=32, K=1), dict(net="hash_signed", playouts=32, K=1), [1, 2]),
    ("different nets, K=16", dict(net="hash_pos", playouts=32, K=16), dict(net="mod17", playouts=32, K=16), [3, 4]),
    ("same net, K=16 against K=4", dict(net="hash_signed", playouts=32, K=16), dict(net="hash_signed", playouts=32, K=4), [5, 6]),
    ("same net, 40 against 120 playouts", dict(net="hash_pos", playouts=40, K=16), dict(net="hash_pos", playouts=120, K=16), [7, 8]),
    ("K=1 against K=16", dict(net="mod17", playouts=32, K=1), dict(net="mod17", playouts=32, K=16), [9, 10]),
    ("same net and settings", dict(net="hash_signed", playouts=24, K=16), dict(net="hash_signed", playouts=24, K=16), [11, 12]),
]


def player(spec):
    m = H.make_cchess_main(H.FAKE_NETS[spec["net"]], spec["playouts"], spec["K"], exploration=False)
    if spec["K"] > 1:
        m.mcts.loop = D.DetLoop("busy")              # MCTS_tree.main runs self.loop.run_until_complete(...) (main.py:492)
    seen = []
    orig = m.mcts.update_tree

    def update_tree(act):                            # the root's visit counts as get_action / human_move leave them
        seen.append([int(n.N) for n in m.mcts.root.child.values()])
        return orig(act)
    m.mcts.update_tree = update_tree
    return m, seen


def play(a, b, a_red, seed):
    ref = H.load_reference()
    (ma, seen_a), (mb, seen_b) = player(a), player(b)
    np.random.seed(seed)
    names = {id(ma): "a", id(mb): "b"}
    red, black = (ma, mb) if a_red else (mb, ma)
    plies = []
    with H.quiet(), np.errstate(all="ignore"):
        while True:
            mover, other = (red, black) if red.game_borad.current_player == "w" else (black, red)
            asyncio.set_event_loop(mover.mcts.loop)
            (sx, sy, ddx, ddy), q_mover = mover.select_move("mcts")
            visits = (seen_a if mover is ma else seen_b)[-1]
            coord = (sx, sy, sx + ddx, sy + ddy)
            action = "abcdefghi"[coord[0]] + str(coord[1]) + "abcdefghi"[coord[2]] + str(coord[3])
            asyncio.set_event_loop(other.mcts.loop)
            q_other = other.human_move(coord, "mcts")
            assert mover.game_borad.state == other.game_borad.state
            plies.append([names[id(mover)], action, visits, f32_hex(q_mover), f32_hex(q_other),
                          tree_digest(H.tree_signature(ma.mcts.root, ref), H.tree_signature(mb.mcts.root, ref))])
            end, winner = mover.check_end()
            if end:
                break
    for m in (ma, mb):
        m.mcts.loop.close()
    return dict(a_red=a_red, seed=seed, winner=winner, plies=len(plies), ply=plies)


def main():
    H.load_reference()
    out = []
    for name, a, b, seeds in PAIRINGS:
        matches = []
        for seed in seeds:
            for a_red in (True, False):
                g = play(a, b, a_red, seed)
                matches.append(g)
                print(name, "seed", seed, "A red" if a_red else "A black", g["winner"], g["plies"], flush=True)
        out.append(dict(name=name, a=a, b=b, matches=matches))
    path = os.path.join(os.path.dirname(HERE), "tests", "golden", "arena.json.gz")
    with open(path, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", compresslevel=9, mtime=0) as f:
        f.write(json.dumps(dict(protocol="two play-mode cchess_main objects: select_move('mcts') / human_move(coord, 'mcts'), temperature 1",
                                pairings=out)).encode())
    print("wrote", path)


if __name__ == "__main__":
    main()
