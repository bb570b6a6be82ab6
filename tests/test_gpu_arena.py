"""The arena on the GPU: cz_engine_play_moves against cz_engine_play, Arena against the unmodified reference's own matches
(tests/golden/arena.json.gz), and matches of real networks."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden

pytestmark = pytest.mark.gpu


def _midgame_positions(B, plies, seed0):
    """Positions reached by seeded self-play (stand-in net, 24 playouts, K = 1): boards, sides, restrict_round."""
    from cchess_zero_b200.fakenet import FakeNet
    from cchess_zero_b200.selfplay import SelfPlay
    sp = SelfPlay(B, FakeNet("hash_pos"), 24, seeds=[seed0 + g for g in range(B)], auto_reset=False, keep_records=False)
    for _ in range(plies):
        sp.step()
    st = sp.engine.status()
    sp.engine.close()
    return st["boards"], st["side"], st["rr"]


def _searched_pair(K, boards, sides, rr, playouts):
    """Two identical engines searched identically from the same positions."""
    from cchess_zero_b200.engine import Engine
    from cchess_zero_b200.fakenet import FakeNet
    B = len(boards)
    fn = FakeNet("hash_signed")
    out = []
    for _ in range(2):
        e = Engine(B, 1 << 17, search_threads=K if K > 1 else None)
        e.reset(None, boards, sides, rr)
        nn_in = torch.zeros((e.rows, 9, 10, 14), device="cuda")
        logits = torch.zeros((e.rows, 2086), device="cuda")
        value = torch.zeros((e.rows,), device="cuda")

        def fwd(x, logits=logits, value=value):
            lo, v = fn(x)
            logits.copy_(lo); value.copy_(v)
        out.append((e, lambda e=e, fwd=fwd, nn_in=nn_in, logits=logits, value=value: e.search(fwd, playouts, nn_in, logits, value)))
    return out


def _records_equal(a, b):
    for k in a:
        assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), k


@pytest.mark.parametrize("K", [1, 16])
def test_play_moves_equals_play_by_index(K):
    """Engine X plays child indices (k_play), engine Y the same children by move code (k_play_moves): status records and whole
    tree signatures equal bit for bit, over two rounds of search + move, including children that were never expanded (N = 0)."""
    from cchess_zero_b200._lib import NOMOVE
    B = 24
    boards, sides, rr = _midgame_positions(B, 9, 300)
    (x, search_x), (y, search_y) = _searched_pair(K, boards, sides, rr, 40)
    unexpanded_played = 0
    for rnd in range(2):
        live = np.nonzero(x.status()["terminal"] == 0)[0]
        search_x(); search_y()
        rc = x.root_children()
        assert np.array_equal(rc["visits"], y.root_children()["visits"])
        ci = np.full(B, -1, dtype=np.int32)
        for g in live:
            n = int(rc["n"][g])
            zero = np.nonzero(rc["visits"][g, :n] == 0)[0]
            if g % 3 == 0 and len(zero):                # a child that was never expanded
                ci[g] = int(zero[len(zero) // 2])
                unexpanded_played += 1
            elif g % 3 == 1:
                ci[g] = int(np.argmax(rc["visits"][g, :n]))
            else:
                ci[g] = n - 1
        mv = np.full(B, NOMOVE, dtype=np.uint16)
        mv[ci >= 0] = rc["moves"][ci >= 0, ci[ci >= 0]]
        sx = x.play(ci)
        sy = y.play_moves(mv)
        _records_equal(sx, sy)
        for g in range(B):
            assert np.array_equal(x.tree_signature(g), y.tree_signature(g)), (rnd, g)
        x.raise_on_error(); y.raise_on_error()
    assert unexpanded_played >= 4
    x.close(); y.close()


@pytest.mark.parametrize("K", [1, 16])
def test_play_moves_rejects_a_move_that_is_not_a_child(K):
    """A move that is not a root child, or any move at an unexpanded root, sets CZ_ERR_NOCHILD and leaves the game unchanged;
    CZ_NOMOVE leaves the game unchanged and still writes its status."""
    from cchess_zero_b200._lib import NOMOVE, EngineError
    B = 8
    boards, sides, rr = _midgame_positions(B, 5, 900)
    (e, search), _ = _searched_pair(K, boards, sides, rr, 32)
    before = e.status()
    st = e.play_moves(np.full(B, NOMOVE, dtype=np.uint16))            # NOMOVE: unchanged, status written
    _records_equal(before, st)
    assert e.counters()["error"] == 0
    search()
    rc = e.root_children()
    sigs = [e.tree_signature(g) for g in range(B)]
    before = e.status()
    bad = np.full(B, NOMOVE, dtype=np.uint16)
    bad[1] = 0                                                         # a0 -> a0: never a move
    n1 = int(rc["n"][1])
    legal = set(int(m) for m in rc["moves"][1, :n1])
    bad[3] = next(s | (d << 7) for s in range(90) for d in range(90) if s != d and (s | (d << 7)) not in legal)
    e.play_moves(bad, want_status=False)
    _records_equal(before, e.status())
    for g in range(B):
        assert np.array_equal(e.tree_signature(g), sigs[g])
    c = e.counters()
    assert c["error"] == 32 and c["first_error_game"] == 1
    with pytest.raises(EngineError, match="NOCHILD"):
        e.play_moves(bad)
    e.close()

    # a root that was never expanded: every move is rejected
    (f, _), _ = _searched_pair(K, boards, sides, rr, 32)
    before = f.status()
    assert (f.root_children()["n"] == -1).all()
    legal = [int(rc["moves"][g, 0]) for g in range(B)]
    f.play_moves(np.array(legal, dtype=np.uint16), want_status=False)
    _records_equal(before, f.status())
    assert f.counters()["error"] == 32
    f.close()


def _play_golden(pairing, matches, M=None, slots=None, other_seed=1000):
    """Plays `matches` of a golden pairing through Arena with FakeNet evaluators and checks every ply; with M / slots the golden
    matches sit at `slots` of an M-match batch whose other matches are seeded differently."""
    from cchess_zero_b200 import rules
    from cchess_zero_b200.arena import Arena
    from cchess_zero_b200.fakenet import FakeNet
    from oracle.oracle_arena import f32_hex, tree_digest
    a, b = pairing["a"], pairing["b"]
    M = M or len(matches)
    slots = list(range(len(matches))) if slots is None else slots
    seeds = [other_seed + m for m in range(M)]
    a_red = [m % 3 != 0 for m in range(M)]
    for s, g in zip(slots, matches):
        seeds[s], a_red[s] = g["seed"], g["a_red"]
    ar = Arena(FakeNet(a["net"]), FakeNet(b["net"]), M, a["playouts"], b["playouts"], a["K"], b["K"], seeds=seeds, a_red=a_red,
               arena_words=1 << 18)
    A, B = ar.players
    ply = 0
    while ar.live[slots].any():
        live = ar.live.copy()
        r = ar.step()
        for s, g in zip(slots, matches):
            if not live[s]:
                continue
            mover, act, visits, qm, qo, dig = g["ply"][ply]
            assert ("a" if r["a_moves"][s] else "b") == mover, (pairing["name"], s, ply)
            assert rules.move_to_label(int(r["move"][s])) == act, (pairing["name"], s, ply)
            assert [int(v) for v in r["visits"][s, : r["n"][s]]] == visits, (pairing["name"], s, ply)
            q_mover, q_other = (r["q_a"][s], r["q_b"][s]) if mover == "a" else (r["q_b"][s], r["q_a"][s])
            assert (f32_hex(q_mover), f32_hex(q_other)) == (qm, qo), (pairing["name"], s, ply)
            assert tree_digest(A.engine.tree_signature(s), B.engine.tree_signature(s)) == dig, (pairing["name"], s, ply)
        ply += 1
    if M == len(matches):
        assert not ar.live.any()
    res = ar.result()
    for s, g in zip(slots, matches):
        assert (res.winner[s], int(res.plies[s])) == (g["winner"], g["plies"])
    for p in ar.players:
        p.engine.raise_on_error()
    return ar


@pytest.mark.parametrize("k", range(6))
def test_arena_reproduces_the_reference_matches(k):
    """Every pairing of arena.json.gz (both colour orders, two seeds each): moves, visits, Q bits, both trees' signature digests after
    every ply, and the results."""
    p = load_golden("arena.json.gz")["pairings"][k]
    _play_golden(p, p["matches"])


def test_batching_does_not_couple_matches():
    """The golden matches of one pairing (search_threads 16) placed among 60 other seeded matches in the same batch."""
    p = load_golden("arena.json.gz")["pairings"][1]
    _play_golden(p, p["matches"], M=64, slots=[3, 17, 40, 63])


def _nets(tmp_path):
    from cchess_zero_b200.net import policy_value_network
    return [policy_value_network(7, precision="fp16", seed=s, save_dir=str(tmp_path / ("net%d" % s))) for s in (1, 2)]


def test_real_networks(tmp_path):
    """Two seeded 7-block networks, 64 matches x 64 playouts, search_threads 16: every result agrees with the final board, two runs
    with the same seeds agree, and cchess_main.policy_evaluate gives the Arena's score."""
    from cchess_zero_b200.arena import Arena
    from cchess_zero_b200.selfplay import cchess_main
    net_a, net_b = _nets(tmp_path)
    runs = []
    for _ in range(2):
        ar = Arena(net_a, net_b, 64, 64, search_threads_a=16, arena_words=1 << 20)
        res = ar.play()
        st = ar.players[0].engine.status()
        assert np.array_equal(st["boards"], ar.players[1].engine.status()["boards"])
        for m in range(64):
            b = st["boards"][m]
            king_missing = not (b == 1).any() or not (b == 8).any()
            assert king_missing == (res.winner[m] in ("w", "b")), m
            assert (st["rr"][m] >= 60 and not king_missing) == (res.winner[m] == "t"), m
            if king_missing:
                assert res.winner[m] == ("b" if not (b == 1).any() else "w")
            assert len(res.moves[m]) == res.plies[m] == st["ply"][m]
        runs.append(res)
        for p in ar.players:
            p.engine.raise_on_error()
    r0, r1 = runs
    assert r0.winner == r1.winner and np.array_equal(r0.plies, r1.plies) and r0.moves == r1.moves
    assert all(np.array_equal(np.asarray(x, np.float32).view(np.uint32), np.asarray(y, np.float32).view(np.uint32))
               for x, y in zip(r0.q_a + r0.q_b, r1.q_a + r1.q_b))
    s = r0.summary()
    assert s["w"] + s["d"] + s["l"] == 64
    m = cchess_main(playout=64, in_search_threads=16, network=net_a, log_file=False)
    assert m.policy_evaluate(net_b, n_games=64) == s["win_ratio"]


def test_cli_prints_one_json_line(tmp_path):
    net_a, net_b = _nets(tmp_path)
    pa, pb = net_a.save(1), net_b.save(2)
    r = subprocess.run([sys.executable, "-m", "cchess_zero_b200.arena", "--a", pa, "--b", pb, "--matches", "4", "--playouts", "16",
                        "--search_threads", "4", "--playouts_b", "24", "--search_threads_b", "1", "--seed", "5", "--arena_words", str(1 << 18)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900, env=dict(os.environ, PYTHONNOUSERSITE="1"))
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [x for x in r.stdout.splitlines() if x.strip()]
    assert len(lines) == 1
    out = json.loads(lines[0])
    s = out["summary"]
    assert s["n"] == 4 and s["w"] + s["d"] + s["l"] == 4 and 0.0 <= s["score"] <= 1.0
    assert out["settings"]["playouts_b"] == 24 and out["settings"]["search_threads_b"] == 1 and out["device"]
