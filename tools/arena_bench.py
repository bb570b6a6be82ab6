"""Arena throughput against self-play on one GPU, measured in the same process (alternating), plus one complete match set.

  leg 1: Arena(1024 matches, 400 playouts = the reference's play_playout, search_threads 16, 7 blocks, fp16, two seeded networks)
         and SelfPlay(1024 games, search_threads 16, 400 playouts) on the same networks, timed alternately (ROUNDS x PLIES plies
         each, after WARMUP plies of each): expansions/s from the engine counters, network rows evaluated per leaf, launches per ply.
  leg 2: a complete 400-match arena (the slowest match included): wall time and matches/hour.
Writes profiles/arena_<date>.json (or --out) with the card's name and power limit read in the same call.

    python tools/arena_bench.py [--matches 1024] [--playouts 400] [--full-matches 400] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch        # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() or q.stderr.strip())


class Meter:
    """Engine counters, network rows and launches of a set of SelfPlay search paths over a timed window."""

    def __init__(self, sps):
        self.sps = sps

    def snap(self):
        return [(sp.engine.counters()["n_expand"], getattr(sp, "rows_evaluated", 0), sp.engine.launches) for sp in self.sps]

    @staticmethod
    def diff(a, b):
        return dict(expansions=sum(y[0] - x[0] for x, y in zip(a, b)), rows=sum(y[1] - x[1] for x, y in zip(a, b)),
                    launches=sum(y[2] - x[2] for x, y in zip(a, b)))


def timed(fn, n, meter):
    torch.cuda.synchronize()
    s0 = meter.snap()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dt, Meter.diff(s0, meter.snap())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--matches", type=int, default=1024)
    ap.add_argument("--playouts", type=int, default=400)
    ap.add_argument("--search_threads", type=int, default=16)
    ap.add_argument("--res_blocks", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--plies", type=int, default=3, help="plies per timed round")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--full-matches", type=int, default=400)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("arena_bench needs a CUDA device")
    from cchess_zero_b200.arena import Arena
    from cchess_zero_b200.net import policy_value_network
    from cchess_zero_b200.selfplay import SelfPlay

    nets = [policy_value_network(a.res_blocks, precision="fp16", seed=s, save_dir=os.devnull) for s in (1, 2)]
    K, M = a.search_threads, a.matches
    ar = Arena(nets[0], nets[1], M, a.playouts, search_threads_a=K, arena_words=1 << 21)
    sp = SelfPlay(M, None, a.playouts, seeds=range(M), auto_reset=True, keep_records=False, search_threads=K, arena_words=1 << 21,
                  plan_factory=lambda n: nets[0].native_plan(n))
    sp.capture_graph()
    for _ in range(a.warmup):
        ar.step()
        sp.step()
    tot = dict(arena=dict(s=0.0, plies=0, expansions=0, rows=0, launches=0), selfplay=dict(s=0.0, plies=0, expansions=0, rows=0, launches=0))
    for _ in range(a.rounds):
        for name, fn, meter in (("arena", ar.step, Meter(ar.players)), ("selfplay", sp.step, Meter([sp]))):
            dt, d = timed(fn, a.plies, meter)
            t = tot[name]
            t["s"] += dt
            t["plies"] += a.plies
            for k in ("expansions", "rows", "launches"):
                t[k] += d[k]
    out = dict(card=card(), settings=dict(matches=M, playouts=a.playouts, search_threads=K, res_blocks=a.res_blocks, precision="fp16",
                                          warmup_plies=a.warmup, timed_plies_per_side=a.plies * a.rounds, alternation_rounds=a.rounds))
    for name, t in tot.items():
        out[name] = dict(expansions_per_s=t["expansions"] / t["s"], s_per_ply=t["s"] / t["plies"], rows_per_leaf=t["rows"] / max(1, t["expansions"]),
                         rows_evaluated=t["rows"], expansions=t["expansions"], launches_per_ply=t["launches"] / t["plies"])
    out["arena_over_selfplay_expansions_per_s"] = out["arena"]["expansions_per_s"] / out["selfplay"]["expansions_per_s"]
    del ar, sp
    torch.cuda.empty_cache()

    if a.full_matches > 0:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        full = Arena(nets[0], nets[1], a.full_matches, a.playouts, search_threads_a=K, arena_words=1 << 21)
        t1 = time.perf_counter()
        res = full.play()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        out["full"] = dict(matches=a.full_matches, setup_s=t1 - t0, play_s=t2 - t1, matches_per_hour=a.full_matches / (t2 - t1) * 3600,
                           plies_mean=float(np.mean(res.plies)), plies_max=int(np.max(res.plies)), summary=res.summary())
    path = a.out or os.path.join(ROOT, "profiles", "arena_%s.json" % time.strftime("%Y%m%d"))
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
