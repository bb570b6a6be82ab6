"""TEST INFRASTRUCTURE ONLY -- golden searches of the UNMODIFIED reference's coroutines on oracle/detloop.py's deterministic loop.

    python oracle/gen_golden_detloop.py        ->  tests/golden/k16_detloop.json   (needs the reference, live or staged; ~15 s)

Two records, both at search_threads=16 in the canonical "busy" schedule, which tests/test_oracle_golden.py compares with the C
restatement of that schedule (co_tree_search_fifo):
  positions  : the root visit counts of the first 12 positions of tests/golden/k16_stats.json.gz, one fresh tree each;
  tree_reuse : five consecutive searches from the start position on ONE tree (MCTS_tree.update_tree with the most visited move
               in between, the self-play / play-mode pattern): every root child's (move, N, Q bits) after each search."""
import asyncio
import gzip
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import detloop as D          # noqa: E402
import ref_harness as H      # noqa: E402

GOLDEN = os.path.join(os.path.dirname(HERE), "tests", "golden")
OUT = os.path.join(GOLDEN, "k16_detloop.json")
START = "RNBAKABNR/9/1C5C1/P1P1P1P1P/9/9/p1p1p1p1p/1c5c1/9/rnbakabnr"
N_POS, REUSE_NET, REUSE_PLAYOUTS, REUSE_PLIES = 12, "hash_pos", 96, 5


def positions():
    with gzip.open(os.path.join(GOLDEN, "k16_stats.json.gz"), "rb") as f:
        d = json.loads(f.read().decode())
    out = []
    for r in d["records"][:N_POS]:
        ref, t, loop = D.make_tree(H, H.FAKE_NETS[d["net"]], 16, r["state"], "busy")
        with np.errstate(all="ignore"):
            D.run_reference_search(ref, t, r["state"], r["player"], r["rr"], d["playouts"], loop)
        loop.close()
        out.append(dict(state=r["state"], player=r["player"], rr=r["rr"], visits=[int(c.N) for c in t.root.child.values()]))
    return dict(net=d["net"], playouts=d["playouts"], records=out)


def tree_reuse():
    ref = H.load_reference()
    state, player, rr = START, "w", 0
    rtree = None
    plies = []
    for _ in range(REUSE_PLIES):
        loop = D.DetLoop("busy")
        asyncio.set_event_loop(loop)
        if rtree is None:
            rtree = ref.MCTS_tree_py312(state, H.FAKE_NETS[REUSE_NET], 16)
        rtree.loop = loop
        rtree.sem = asyncio.Semaphore(16)                 # fresh primitives for the fresh loop (main() builds new coroutines each call)
        rtree.queue = asyncio.Queue(16)
        rtree.running_simulation_num = 0
        with np.errstate(all="ignore"):
            D.run_reference_search(ref, rtree, state, player, rr, REUSE_PLAYOUTS, loop)
        loop.close()
        children = [[a, int(c.N), H.f32_bits(c.Q)] for a, c in rtree.root.child.items()]
        plies.append(dict(state=state, player=player, rr=rr, children=children))
        act = max(rtree.root.child.items(), key=lambda kv: kv[1].N)[0]     # first maximum, as np.argmax
        nxt = ref.GameBoard.sim_do_action(act, state)
        rr = rr + 1 if ref.is_kill_move(state, nxt) == 0 else 0
        rtree.update_tree(act)
        state, player = nxt, ("b" if player == "w" else "w")
    return dict(net=REUSE_NET, playouts=REUSE_PLAYOUTS, plies=plies)


def main():
    out = dict(schedule="detloop busy (canonical uvloop FIFO schedule), search_threads 16", positions=positions(), tree_reuse=tree_reuse())
    with open(OUT, "w") as f:
        json.dump(out, f)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
