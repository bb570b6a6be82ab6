"""Pins the CPU oracle (oracle/cchess_oracle.c) to golden vectors produced by the UNMODIFIED
reference (oracle/gen_golden.py).  CPU-only; runs everywhere."""
import hashlib

import numpy as np
import pytest

from conftest import load_golden
from oracle import oracle as O


def sha(b):
    return hashlib.sha256(b).hexdigest()[:16]


def bits(v):
    """float32 bit pattern with NaN canonicalised (see oracle/ref_harness.py:f32_bits)"""
    v = np.float32(v)
    return 0x7FC00000 if np.isnan(v) else int(v.view(np.uint32))


def test_labels():
    g = load_golden("labels.json")
    assert O.labels() == g["labels"]
    assert O.unflipped_index() == g["unflipped_index"]
    assert g["sha_labels"] == "c6e10a93f1d69164"  # SURVEY Appendix B
    assert g["sha_unflipped"] == "da24858f23137be3"
    lab = g["labels"]
    for i in (0, 223, 916, 1125, 1832, 2035, 2042, 2056):
        m = lab[i]
        assert O.label_index(O.move_from_str(m) & 127, O.move_from_str(m) >> 7) == i


def test_rules_against_reference_vectors():
    g = load_golden("movegen.json.gz")
    assert g["n"] == len(g["records"]) > 7000
    for r in g["records"]:
        b = O.from_state(r["state"])
        side = 0 if r["player"] == "w" else 1
        assert O.to_state(b) == r["state"]
        mv = O.legal_moves(b, side)
        assert " ".join(O.move_str(m) for m in mv) == r["moves"], r["state"]
        enc = O.encode(b, side)
        assert [int(i) for i in np.nonzero(enc.reshape(-1))[0]] == r["enc"]
        assert set(np.unique(enc)) <= {0.0, 1.0}
        fb = O.flip_board(b) if side == 1 else b
        assert O.to_state(fb) == r["flip"]
        if "move" in r:
            nb, cap = O.apply_move(b, O.move_from_str(r["move"]))
            assert O.to_state(nb) == r["next"]
            assert int(cap != 0) == r["kill"]


def test_appendix_b_known_answers():
    start = O.from_state(O.START)
    mv = [O.move_str(m) for m in O.legal_moves(start, 0)]
    assert len(mv) == 44 and mv[:5] == ["a0a1", "a0a2", "b0a2", "b0c2", "c0e2"] and mv[-1] == "i3i4"
    enc = O.encode(start, 0)
    assert enc.sum() == 26.0 and sha(enc.tobytes()) == "8ca9caf6c0b9416c"
    assert np.array_equal(enc, O.encode(start, 1))
    kk = O.from_state("4K4/9/9/9/9/9/9/9/9/4k4")
    assert [O.move_str(m) for m in O.legal_moves(kk, 0)] == ["e0d0", "e0f0", "e0e1", "e0e9"]


@pytest.mark.parametrize("i", range(13))
def test_tree_against_reference(i):
    g = load_golden("tree.json")
    if i >= len(g["cases"]):
        pytest.skip("no such case")
    c = g["cases"][i]
    t = O.Tree(O.from_state(c["state"]))
    t.search(0 if c["player"] == "w" else 1, c["rr"], c["playouts"], c["net"])
    sig = t.signature()
    assert sig.shape[0] == c["n_nodes"]
    assert sig[:40].tolist() == c["head"]
    assert sha(sig.tobytes()) == c["sha_sig"], c["note"]
    mv, N, W, P, Q = t.root_children()
    got = [[O.move_str(m), int(n), bits(w), bits(p), bits(q)]
           for m, n, w, p, q in zip(mv, N, W, P, Q)]
    assert got == c["root"]


@pytest.mark.parametrize("i", range(6))
def test_selfplay_tuples_against_reference(i):
    g = load_golden("selfplay.json")["games"][i]
    with np.errstate(all="ignore"):
        r = O.selfplay_game(g["net"], g["playouts"], np.random.RandomState(g["seed"]))
    assert len(r["states"]) == g["n"]
    assert r["states"] == g["states"]
    assert [float(v) for v in r["z"]] == g["z"]
    assert sha(np.asarray(r["pis"], dtype=np.float64).tobytes()) == g["sha_pi"]
    for p, sp in zip(r["pis"], g["pi_sparse"]):
        assert [[int(k), float(p[k]).hex()] for k in np.nonzero(p)[0]] == sp


def test_selfplay_full_game_at_1200_playouts_against_reference():
    """One complete game of the reference at the BASELINE playout count (search_threads=1), 77 plies."""
    g = load_golden("selfplay_1200.json")["games"][0]
    with np.errstate(all="ignore"):
        r = O.selfplay_game(g["net"], g["playouts"], np.random.RandomState(g["seed"]))
    assert len(r["states"]) == g["n"] and r["states"] == g["states"]
    assert [float(v) for v in r["z"]] == g["z"]
    assert sha(np.asarray(r["pis"], dtype=np.float64).tobytes()) == g["sha_pi"]


@pytest.mark.parametrize("i", range(6))
def test_selfplay_at_search_threads_16_against_reference_coroutines(i):
    """Whole self-play games of the unmodified reference at search_threads = 16 / 8 / 4 (its own coroutines on the canonical
    deterministic schedule, oracle/gen_golden_k16_selfplay.py) against the C restatement of that schedule."""
    g = load_golden("selfplay_k16.json")["games"][i]
    with np.errstate(all="ignore"):
        r = O.selfplay_game(g["net"], g["playouts"], np.random.RandomState(g["seed"]), search_threads=g["search_threads"])
    assert len(r["states"]) == g["n"] and r["states"] == g["states"]
    assert [float(v) for v in r["z"]] == g["z"]
    assert sha(np.asarray(r["pis"], dtype=np.float64).tobytes()) == g["sha_pi"]
    for p, sp in zip(r["pis"], g["pi_sparse"]):
        assert [[int(k), float(p[k]).hex()] for k in np.nonzero(p)[0]] == sp


def test_leaf_parallel_spec_with_one_slot_is_the_reference_search():
    """oracle co_tree_search_multi (the serial spec of the package's own K-leaves-per-wave schedule) must degenerate to the
    reference-pinned search for K = 1; for K > 1 it must conserve visits."""
    for net in ("hash_pos", "hash_signed", "mod17"):
        a, b = O.Tree(), O.Tree()
        a.search(0, 0, 300, net)
        assert b.search_multi(0, 0, 300, 1, net) == 0
        assert np.array_equal(a.signature(), b.signature())
    for K in (2, 4, 16, 64):
        t = O.Tree()
        assert t.search_multi(0, 0, 500, K, "hash_pos") == 0
        assert t.root_children()[1].sum() == 500 and t.stats()["n_playout"] == 500


def test_rules_are_symmetric_under_the_colour_flip():
    """Domain property (size independent): flipping the board (rows reversed, colours swapped, try_flip main.py:560-574) and the side
    to move maps the legal-move SET onto its rank mirror; captures and king-capture terminals map onto each other."""
    rng = np.random.RandomState(8)
    b, side = O.from_state(O.START), 0
    checked = 0
    for _ in range(3000):
        mv = O.legal_moves(b, side)
        fb = O.flip_board(b)
        fm = O.legal_moves(fb, side ^ 1)

        def mirror(m):
            s, d = int(m) & 127, int(m) >> 7
            return ((9 - s // 9) * 9 + s % 9) | (((9 - d // 9) * 9 + d % 9) << 7)
        assert sorted(mirror(m) for m in mv) == sorted(int(m) for m in fm)
        checked += 1
        if len(mv) == 0:
            b, side = O.from_state(O.START), 0
            continue
        m = mv[rng.randint(len(mv))]
        nb, cap = O.apply_move(b, m)
        nfb, fcap = O.apply_move(fb, mirror(m))
        assert np.array_equal(O.flip_board(nb), nfb) and (cap == 0) == (fcap == 0)
        b, side = nb, side ^ 1
        if cap in (1, 8):
            b, side = O.from_state(O.START), 0
    assert checked == 3000


def test_tree_extra_cases_against_reference():
    """72 more search trees of the reference (random-play positions from opening to bare endgames, both colours, rr up to 59)."""
    g = load_golden("tree_extra.json")
    assert len(g["cases"]) >= 60
    for c in g["cases"]:
        t = O.Tree(O.from_state(c["state"]))
        t.search(0 if c["player"] == "w" else 1, c["rr"], c["playouts"], c["net"])
        sig = t.signature()
        assert sig.shape[0] == c["n_nodes"] and sha(sig.tobytes()) == c["sha_sig"], (c["state"], c["player"], c["rr"])


def test_fifo_schedule_spec_reproduces_real_reference_runs_at_search_threads_16():
    """oracle co_tree_search_fifo (the canonical FIFO form of the reference's search_threads > 1 schedule) against REAL uvloop runs
    of the unmodified reference at search_threads=16 (tests/golden/k16_stats.json.gz; every position was searched twice by the
    reference, the second time with 2 ms of evaluator latency).  The reference differs from itself on a few per cent of the
    positions (timing-dependent spins); the specification must equal one of its two runs on every position."""
    from conftest import load_golden
    d = load_golden("k16_stats.json.gz")
    first = either = self_consistent = 0
    for r in d["records"]:
        side = 0 if r["player"] == "w" else 1
        t = O.Tree(O.from_state(r["state"]))
        assert t.search_fifo(side, r["rr"], d["playouts"], 16, d["net"]) == 0
        mv, N, W, P, Q = t.root_children()
        assert " ".join(O.move_str(m) for m in mv) == r["moves"]
        v = [int(x) for x in N]
        first += v == r["k16"]
        either += v == r["k16"] or v == r["k16_delay2ms"]
        self_consistent += r["k16"] == r["k16_delay2ms"]
        t1 = O.Tree(O.from_state(r["state"]))
        assert t1.search_fifo(side, r["rr"], d["playouts"], 1, d["net"]) == 0
        assert [int(x) for x in t1.root_children()[1]] == r["k1"]            # K = 1 degenerates to the search_threads=1 reference
    assert either == len(d["records"]) and first >= 0.95 * len(d["records"])
    assert self_consistent == d["reference_k16_identical_under_2ms_latency"]


def test_fifo_schedule_spec_with_playouts_that_end_in_their_first_step():
    """King capturable at the root / 60-move rule one ply away: real uvloop runs of the reference (three per position and evaluator,
    tests/golden/k16_terminal.json) against the C restatement of the schedule."""
    d = load_golden("k16_terminal.json")
    first = total = 0
    for r in d["records"]:
        for run in r["runs"]:
            o = O.Tree(O.from_state(r["state"]))
            assert o.search_fifo(0 if r["player"] == "w" else 1, r["rr"], d["playouts"], 16, run["net"]) == 0
            v = [int(x) for x in o.root_children()[1]]
            assert v in run["k16_runs"], (r["state"], run["net"])
            first += v == run["k16_runs"][0]
            total += 1
    assert first >= 0.9 * total


def test_deterministic_event_loop_runs_the_reference_coroutines_to_the_same_trees():
    """The UNMODIFIED coroutines of the reference (tree_search / start_tree_search / prediction_worker) on oracle/detloop.py's
    deterministic event loop (tests/golden/k16_detloop.json, oracle/gen_golden_detloop.py) give the visit counts of the real uvloop
    run AND of the C restatement."""
    d = load_golden("k16_detloop.json")["positions"]
    real = load_golden("k16_stats.json.gz")
    assert d["net"] == real["net"] and d["playouts"] == real["playouts"] and len(d["records"]) == 12
    for r, u in zip(d["records"], real["records"]):
        assert (r["state"], r["player"], r["rr"]) == (u["state"], u["player"], u["rr"])
        v = r["visits"]
        assert v == u["k16"] or v == u["k16_delay2ms"]
        o = O.Tree(O.from_state(r["state"]))
        o.search_fifo(0 if r["player"] == "w" else 1, r["rr"], d["playouts"], 16, d["net"])
        assert v == [int(x) for x in o.root_children()[1]]


def test_fifo_schedule_across_tree_reuse_matches_the_reference_coroutines():
    """Several consecutive searches at search_threads=16 with MCTS_tree.update_tree in between (the self-play / play-mode pattern):
    the stored Q, the left-over visit counts of the re-used subtree and the frozen root N must carry over exactly as in the
    reference's object tree.  Reference side: its own coroutines on the deterministic loop (tests/golden/k16_detloop.json);
    other side: the C restatement."""
    d = load_golden("k16_detloop.json")["tree_reuse"]
    net, P = d["net"], d["playouts"]
    board, player, rr = O.from_state(O.START), "w", 0
    ctree = O.Tree()
    assert len(d["plies"]) == 5
    for ply, g in enumerate(d["plies"]):
        assert (O.to_state(board), player, rr) == (g["state"], g["player"], g["rr"]), ply
        assert ctree.search_fifo(0 if player == "w" else 1, rr, P, 16, net) == 0
        mv, N, W, Pp, Q = ctree.root_children()
        got = [tuple(c) for c in g["children"]]
        want = [(O.move_str(m), int(n), bits(q)) for m, n, q in zip(mv, N, Q)]
        assert got == want, ply
        best = int(np.argmax(N))
        board, cap = O.apply_move(board, mv[best])
        rr = rr + 1 if cap == 0 else 0
        ctree.update(best)
        player = "b" if player == "w" else "w"
