"""The arena without a GPU: its C specification against the unmodified reference's own matches (tests/golden/arena.json.gz), the
match statistics, and the command line's argument checks."""
import math

import pytest

from conftest import load_golden


def test_oracle_arena_reproduces_the_reference_matches_bit_for_bit():
    """Moves, visit counts, both Q(act) bits, both trees' signature digests after every ply, winners and ply counts."""
    from oracle.oracle_arena import arena_game
    d = load_golden("arena.json.gz")
    assert len(d["pairings"]) == 6
    n = 0
    for p in d["pairings"]:
        assert {m["a_red"] for m in p["matches"]} == {True, False}
        for m in p["matches"]:
            o = arena_game(p["a"], p["b"], m["a_red"], m["seed"])
            assert o["ply"] == m["ply"], (p["name"], m["seed"], m["a_red"])
            assert (o["winner"], o["plies"]) == (m["winner"], m["plies"])
            n += 1
    assert n >= 24


def test_summary_statistics():
    from cchess_zero_b200.arena import summarize
    # W=60 D=20 L=20, A red in even slots: score 0.7, Elo +147.2, 95 % interval [+86.2, +218.3], LOS 0.999996
    a_red = [m % 2 == 0 for m in range(100)]
    res = ["a"] * 60 + ["d"] * 20 + ["l"] * 20
    winners = [("w" if r else "b") if x == "a" else ("t" if x == "d" else ("b" if r else "w")) for r, x in zip(a_red, res)]
    s = summarize(a_red, winners)
    assert (s["w"], s["d"], s["l"], s["n"]) == (60, 20, 20, 100)
    assert s["score"] == pytest.approx(0.7) and s["win_ratio"] == s["score"]
    assert round(s["elo"], 1) == 147.2
    assert [round(x, 1) for x in s["elo_95"]] == [86.2, 218.3]
    assert round(s["los"], 6) == 0.999996
    for k in ("w", "d", "l"):                                   # per colour sums to the totals
        assert s["as_red"][k] + s["as_black"][k] == s[k]
    assert s["as_red"] == dict(w=30, d=10, l=10) and s["as_black"] == dict(w=30, d=10, l=10)
    assert s["red_score"] == pytest.approx((40 + 0.5 * 20) / 100)  # red won 30 (A as red) + 10 (B as red), 20 draws

    d = summarize([True, False] * 5, ["t"] * 10)
    assert d["elo"] == 0.0 and d["elo_95"] == [0.0, 0.0] and d["los"] == 0.5 and d["score"] == 0.5

    w = summarize([True, False] * 5, ["w", "b"] * 5)            # A wins every game
    assert w["score"] == 1.0 and w["elo"] == math.inf and w["elo_95"][1] == math.inf and math.isfinite(w["elo_95"][0])
    assert w["los"] > 0.999
    l = summarize([True, False] * 5, ["b", "w"] * 5)            # A loses every game
    assert l["score"] == 0.0 and l["elo"] == -math.inf and l["elo_95"][0] == -math.inf and math.isfinite(l["elo_95"][1])
    assert l["los"] < 0.001


def test_policy_evaluate_win_ratio_is_the_reference_formula():
    """main.py:1219: win_ratio = (win + 0.5 * tie) / n_games, from the evaluated network's side."""
    from cchess_zero_b200.arena import summarize
    a_red = [True, False, True, False, True, False, True]
    winners = ["w", "w", "t", "b", "b", "t", "w"]     # A: win, loss, draw, win, loss, draw, win
    s = summarize(a_red, winners)
    assert (s["w"], s["l"], s["d"]) == (3, 2, 2)
    assert s["win_ratio"] == 1.0 * (3 + 0.5 * 2) / 7


def test_cli_rejects_bad_arguments_before_any_device_work(tmp_path):
    from cchess_zero_b200.arena import parse_args
    a, b = tmp_path / "a.ckpt", tmp_path / "b.ckpt"
    a.write_bytes(b"x")
    b.write_bytes(b"x")
    ok = ["--a", str(a), "--b", str(b)]
    args = parse_args(ok + ["--playouts", "64", "--search_threads", "4"])
    assert (args.playouts_b, args.search_threads_b, args.res_block_nums_b) == (64, 4, 7)
    for bad in (["--a", str(tmp_path / "missing"), "--b", str(b)], ok + ["--matches", "0"], ok + ["--playouts", "0"],
                ok + ["--playouts_b", "-3"], ok + ["--search_threads", "33"], ok + ["--search_threads_b", "0"],
                ok + ["--res_block_nums_b", "0"], ok + ["--arena_words", "-1"], ok + ["--precision", "int3"], ok + ["--seed", "-1"],
                ["--a", str(a)]):
        with pytest.raises(SystemExit):
            parse_args(bad)
