#!/usr/bin/env python
"""bench.py -- MCTS node-expansions/sec and self-play games/hour of batched self-play (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          our arm (one rank per GPU under torchrun)
  python bench.py --impl reference ...                    CPU arm: the UNMODIFIED reference's self-play on the host cores

A "step" is one ply of EVERY concurrent game: a full MCTS_tree.main of `--playouts` playouts per game
(select / encode / network / expand / backup waves), then get_action's host-side move choice and the
re-root.  Main workload = BASELINE.json configs[1]: 1024 concurrent games x 1200 playouts, res_block_nums=7,
per GPU (weak scaling).  Expansions are counted by the engine (calls of expand), not inferred.

value : expansions / device time of the search waves (CUDA events, state resident in HBM)
e2e   : expansions / time of the whole SelfPlay.step() loop through the public API, including the per-ply
        device->host read of root statistics / status, host->device write of the chosen moves, host move
        sampling, tuple recording and (N > 1) the NCCL gather of the finished games' tuples.

Further bounded legs, reported under `extra` of the same JSON line (each can be switched off with --legs):
  precision : the same workload in tf32, tf32x3 (fp32-accurate on the tensor cores) and fp32 (a few plies each)
                                                                             -> extra.by_precision      (N = 1)
  config3   : BASELINE configs[2] per-rank shape, 512 games x 1600 playouts -> extra.config3
  config4   : BASELINE configs[3], 19 residual blocks                       -> extra.config4           (N = 1)
  config5   : BASELINE configs[4], play-mode move latency p50/p95 through get_hint + select_move (ChessGame.py:153-181)
                                                                             -> extra.config5           (N = 1)
  threads16 : batched self-play with the reference's search_threads=16 schedule inside every game, 256 games and the full batch,
              row compaction of the K-rows-per-game network batch  -> extra.search_threads_16, extra.search_threads_16_full_batch (N = 1)
  dedup     : board hashing: share of the evaluated leaves of one ply that repeat a position            -> extra.eval_dedup        (N = 1)
  soak      : every game slot plays on for >= 3 mean game lengths; games/hour from plies/s and the measured
              game-length distribution (no short-game selection bias)       -> extra.games_per_hour
  cpu       : the reference's own CPU self-play beside it                    -> cpu_baseline             (N = 1)
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "mcts_node_expansions_per_sec"
FLOPS_PER_EVAL = {7: 375.4e6, 19: 1012.4e6}
ALL_LEGS = "precision,config3,config4,config5,threads16,dedup,soak,cpu"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--games", type=int, default=1024, help="concurrent games per GPU")
    ap.add_argument("--playouts", type=int, default=1200)
    ap.add_argument("--res-blocks", type=int, default=7)
    ap.add_argument("--precision", default=os.environ.get("CCHESS_NN_PRECISION", "fp16"))
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--first-conv", default=None, choices=["gather", "tc", "mma"], help="first-layer kernel: mma.sync with register-built one-hot operand (default), CUDA-core gather-add, or tcgen05/TMEM")
    ap.add_argument("--lanes", type=int, default=1, choices=[1, 2], help="2 = pipeline two half-batches (tree kernel under the other half's network)")
    ap.add_argument("--library-ends", action="store_true", help="use cuDNN/cuBLAS for the first conv and the heads instead of csrc/cz_net.cu")
    ap.add_argument("--legs", default=os.environ.get("CCHESS_BENCH_LEGS", ALL_LEGS), help="comma list of extra legs (%s) or 'none'" % ALL_LEGS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--soak-plies", type=int, default=170)
    ap.add_argument("--profile-waves", type=int, default=200, help="waves timed individually for the roofline line")
    ap.add_argument("--arena-words", type=int, default=0)
    ap.add_argument("--kwave-capture", action="store_true", help="ncu helper: play --warmup plies (deep trees), then run --profile-waves eager waves and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed plies, write what the last one returned (rank 0) as DIR/<name>.npy, float32 / float64, <= 64 MB")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be >= 1")
    return a


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    samples=len(sm), reasons=sorted(reasons))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", d
    return 6650.0, "fallback (B200_PROFILING.md)", {}


def algorithmic_bytes(c0, c1, enc_bytes):
    """SURVEY.md 8(d): per playout sum_l 12*c_l + 36*L; per expansion 90 + encode + 4C+4 + 14C."""
    d = {k: c1[k] - c0[k] for k in ("n_expand", "n_playout", "sum_L", "sum_c", "sum_C")}
    return 12 * d["sum_c"] + 36 * d["sum_L"] + d["n_expand"] * (90 + enc_bytes + 4) + 18 * d["sum_C"], d


# ---------------------------------------------------------------------------------------------
# CPU arms.  Both are test/baseline infrastructure under oracle/ (the only place bench.py may execute it).
#   reference : oracle/ref_cpu_arm.py -- the UNMODIFIED reference's cchess_main.selfplay(), search_threads=16, one process per core
#   port      : the C oracle port driving lock-step trees + torch CPU net (kept as a second, labelled figure)
# ---------------------------------------------------------------------------------------------
def host_cores():
    from oracle import ref_cpu_arm
    return ref_cpu_arm.usable_cores()


class PortArm:
    """The oracle C port (oracle/cchess_oracle.c) drives n_games trees in lock-step (one leaf per game per wave,
    search_threads=1 semantics) and the same seed-0 network is evaluated by PyTorch on the CPU, all host threads."""

    def __init__(self, n_games, playouts, res_blocks, threads=None):
        import ctypes as C
        from cchess_zero_b200.net import PolicyValueNet
        from oracle import oracle as O
        self.C, self.O, self.L = C, O, O.lib()
        torch.manual_seed(0)
        self.net = PolicyValueNet(res_blocks).eval().to(memory_format=torch.channels_last)
        self.B, self.playouts = n_games, playouts
        self.trees = [O.Tree() for _ in range(n_games)]
        self.arr = (C.c_void_p * n_games)(*[t.h for t in self.trees])
        self.side = np.zeros(n_games, dtype=np.int32)
        self.rr = np.zeros(n_games, dtype=np.int32)
        self.nn_in = np.zeros((n_games, 9, 10, 14), dtype=np.float32)
        self.pending = np.zeros(n_games, dtype=np.uint8)
        self.cores = host_cores()
        self.threads = threads or self.cores
        torch.set_num_threads(self.threads)

    def _p(self, a):
        return a.ctypes.data_as(self.C.c_void_p)

    def wave(self):
        L, p = self.L, self._p
        L.co_batch_select(self.arr, p(self.side), p(self.rr), self.B, self.playouts, p(self.nn_in), p(self.pending), self.threads)
        with torch.no_grad():
            lo, v = self.net(torch.from_numpy(self.nn_in))
        lo = np.ascontiguousarray(lo.numpy(), dtype=np.float32)
        v = np.ascontiguousarray(v.numpy().reshape(-1), dtype=np.float32)
        L.co_batch_finish(self.arr, self.B, p(lo), p(v), p(self.pending), self.threads)

    def expansions(self):
        return sum(t.stats()["n_expand"] for t in self.trees)

    def run(self, seconds):
        self.wave()                                            # warm-up wave (root expansions, allocator)
        e0, t0, n = self.expansions(), time.perf_counter(), 0
        while time.perf_counter() - t0 < seconds or n < 2:
            self.wave(); n += 1
        dt = time.perf_counter() - t0
        return dict(value=(self.expansions() - e0) / dt, seconds=dt, waves=n, games=self.B, threads=self.threads)


def port_figure(playouts, res_blocks, seconds):
    arm = PortArm(256, playouts, res_blocks)
    r = arm.run(seconds)
    return dict(value=r["value"], unit="expansions/s", kind="port", cores=arm.threads,
                sample="%d games x %d lock-step waves (%.1f s) from the start position, oracle C port (search_threads=1 schedule) + torch CPU fp32 net, %d threads"
                       % (r["games"], r["waves"], r["seconds"], arm.threads))


def reference_cpu(steps, warmup, playouts, res_blocks, budget_s, tree_only=True):
    """cpu_baseline dict measured with the unmodified reference; falls back to the port (labelled) when the staged reference is absent."""
    from oracle import ref_cpu_arm
    if ref_cpu_arm.available() is None:
        f = port_figure(playouts, res_blocks, min(budget_s, 15.0))
        f["note"] = "staged reference (oracle/_ref/reference) not found on this box: oracle port timed instead"
        return f, None
    r = ref_cpu_arm.run(steps, warmup, playouts, res_blocks, 16, budget_s)
    out = dict(value=r["value"], unit="expansions/s", cores=r["cores"], kind="reference", sample=r["sample"], search_threads=16,
               mean_nn_batch=r["mean_nn_batch"], usable_cores=r["usable_cores"], quota=r["quota"], timed_s=r["timed_s"])
    if tree_only:
        t = ref_cpu_arm.run(2, 1, playouts, res_blocks, 16, 8.0, net="zero")
        out["tree_only_value"] = t["value"]                     # zero-cost evaluator: shows the network substitution hides nothing
    return out, r


def run_reference(a, rank, world):
    """--impl reference: rank 0 times the reference's own CPU self-play on the host cores; other ranks exit 0."""
    if rank != 0:
        return
    budget = float(os.environ.get("CCHESS_REF_SECONDS", "150"))
    cpu, r = reference_cpu(a.steps, a.warmup, a.playouts, a.res_blocks, budget, tree_only=True)
    v = cpu["value"]
    ms = r["ms_per_step"] if r is not None else None
    try:
        cpu["port_value"] = port_figure(a.playouts, a.res_blocks, 8.0)
    except Exception as e:  # the labelled second figure must never break the arm
        cpu["port_value"] = dict(error=str(e))
    line = dict(metric=METRIC, value=v, unit="expansions/s", n_gpus=a.gpus, steps=a.steps, warmup=a.warmup,
                ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic (seed-0 xavier-initialised network, games from the start position)", impl="reference",
                config=dict(workload="%d concurrent self-play games x %d playouts per move, res_block_nums=%d, per GPU" % (a.games, a.playouts, a.res_blocks),
                            games_per_gpu=a.games, playouts=a.playouts, res_block_nums=a.res_blocks, search_threads=16,
                            note="the reference plays one game per process; a step is a bounded sample (a fixed quota of expansions per process) of that workload"),
                cpu_baseline=cpu,
                e2e=dict(value=v, unit="expansions/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
class Runner:
    """One SelfPlay instance + timing helpers; every leg of our arm goes through it."""

    def __init__(self, a, rank, world, local_rank, games, playouts, res_blocks, precision, pv=None, arena_words=None):
        from cchess_zero_b200.net import policy_value_network
        from cchess_zero_b200.selfplay import SelfPlay
        self.a, self.rank, self.world, self.dev = a, rank, world, torch.device("cuda", local_rank)
        self.B, self.playouts, self.res_blocks, self.precision = games, playouts, res_blocks, precision
        with contextlib.redirect_stdout(io.StringIO()):
            self.pv = pv or policy_value_network(res_blocks, precision=precision, device=local_rank, seed=0)
        native = precision == "fp16" and not a.library_ends
        pvx = self.pv
        if pv is not None and pv.precision != precision:        # same weights, another arithmetic
            from cchess_zero_b200.net import make_plan
            factory = lambda n: make_plan(pvx.net, precision)  # noqa: E731
        else:
            factory = (lambda n: pvx.native_plan(n, a.first_conv)) if native else (lambda n: pvx.plan())
        self.plan = factory(games // a.lanes)
        self.sp = SelfPlay(games, None, playouts, seeds=[rank * games + g for g in range(games)], device=local_rank,
                           auto_reset=True, keep_records=True, plan=self.plan if a.lanes == 1 else None, plan_factory=factory, lanes=a.lanes,
                           arena_words=a.arena_words if arena_words is None else arena_words)
        if not a.no_graph:
            self.sp.capture_graph()
        self.search_ms = []
        self._orig_search = self.sp.search

        def timed_search():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            w = self._orig_search()
            e1.record()
            self.search_ms.append((e0, e1))
            return w
        self.sp.search = timed_search
        self.gather = None
        if world > 1:
            from cchess_zero_b200.distributed import AsyncTupleGather
            self.gather = AsyncTupleGather(self.dev)
        self.tuples_gathered = 0

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def close(self):
        self.sp.search = self._orig_search
        eng = self.sp.engine
        for l in (self.sp.lanes or []):
            l.engine.close()
        if hasattr(eng, "close"):
            eng.close()
        self.sp = None
        torch.cuda.empty_cache()

    def plies(self, steps, warmup, clocks=None, on_step=None):
        """warmup untimed plies, then exactly `steps` timed plies bracketed by barrier + synchronize; max over ranks."""
        import torch.distributed as dist
        sp, e = self.sp, self.sp.engine
        for _ in range(warmup):
            out = sp.step()
            if on_step:
                on_step(out)
        self.barrier()
        if clocks is not None:
            clocks.start()
        self.search_ms.clear()
        c0, l0 = e.counters(), e.launches
        waves0, fin0 = sp.waves, len(sp.finished)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(steps):
            out = sp.step()
            if self.gather is not None:                         # counts of step s, payload of step s-1, landed tuples of step s-2: all asynchronous
                self.gather.start([r for _, r in out["finished"]])
                tb = self.gather.finish()
                if tb is not None:
                    self.tuples_gathered += len(tb)
            if on_step:
                on_step(out)
        if self.gather is not None:
            self.tuples_gathered += len(self.gather.drain())
        ev1.record()
        self.barrier()
        wall = time.perf_counter() - t0
        clk = clocks.stop() if clocks is not None else None
        c1 = e.raise_on_error()
        e2e_ms = ev0.elapsed_time(ev1)
        dev_ms = sum(x.elapsed_time(y) for x, y in self.search_ms)
        t = torch.tensor([dev_ms, e2e_ms, wall * 1e3], dtype=torch.float64, device=self.dev)
        n = torch.tensor([c1["n_expand"] - c0["n_expand"], e.launches - l0, len(sp.finished) - fin0,
                          sum(len(r) for _, r in sp.finished[fin0:])], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(n, op=dist.ReduceOp.SUM)
        dev_ms, e2e_ms, wall_ms = [float(x) for x in t]
        tot_exp, tot_launch, games_done, tuples_done = [float(x) for x in n]
        return dict(dev_ms=dev_ms, e2e_ms=e2e_ms, wall_ms=wall_ms, expansions=tot_exp, launches=tot_launch, games_done=games_done,
                    tuples_done=tuples_done, waves=sp.waves - waves0, steps=steps, c0=c0, c1=c1, clocks=clk,
                    value=tot_exp / (dev_ms * 1e-3), e2e=tot_exp / (e2e_ms * 1e-3), last=out)

    def kwave_roofline(self, n_waves):
        """k_wave timed per launch with CUDA events on the launching stream, in situ (the trees are those of the plies played so far)."""
        a, sp, e = self.a, self.sp, self.sp.engine
        hbm, peak_src, _ = measured_peaks()
        plan = self.plan
        enc_bytes = 96 if plan.dtype == torch.uint8 else 1260 * (4 if plan.dtype == torch.float32 else 2)
        timed, sp.search = sp.search, self._orig_search
        e.begin_search(self.playouts)
        k0 = e.counters()
        evs = []
        lanes = sp.lanes if sp.lanes is not None else [sp]       # a single-lane SelfPlay has the same attribute names
        for _ in range(n_waves):
            for ln in lanes:
                x, y = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                x.record(); ln.engine.wave(ln.nn_in, ln.logits, ln.value); y.record()
                evs.append((x, y))
                ln.forward(ln.nn_in)
        torch.cuda.synchronize()
        sp.search = timed
        k1 = e.counters()
        kms = [x.elapsed_time(y) for x, y in evs]
        ab, d = algorithmic_bytes(k0, k1, enc_bytes)
        per_launch = ab / len(kms)
        avg_ms = float(np.mean(kms))
        achieved = per_launch / (avg_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "kwave_traffic.json")
        if os.path.exists(tpath):        # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of an in-situ launch, per launch
            tj = json.load(open(tpath))
            traffic = (tj["dram_bytes_read_per_launch"] + tj["dram_bytes_write_per_launch"]) * (self.B // a.lanes) / tj["games_per_launch"]
            traffic_src = tj["source"]
        return dict(kernel="k_wave (expand+backup+select+encode, one warp per game; %d games per launch)" % (self.B // a.lanes), bound="hbm",
                    achieved=achieved, peak=hbm, unit="GB/s", frac=achieved / hbm, traffic=traffic, traffic_source=traffic_src, peak_source=peak_src,
                    avg_launch_ms=avg_ms, p50_launch_ms=float(np.median(kms)), max_launch_ms=float(np.max(kms)),
                    algorithmic_bytes_per_launch=per_launch, bytes_per_expansion=ab / max(1, d["n_expand"]), launches_timed=len(kms),
                    note="latency-bound pointer-chasing kernel: HBM fraction is reported as required, the binding limits are per-warp dependent loads and the network")


def leg_precision(a, rank, world, local_rank, pv):
    """The main workload in the other arithmetics, same weights: tf32, tf32x3 (fp32-accurate on the TF32 tensor cores: the mode that
    meets "within 1e-3 fp32" at trained-network magnitudes) and fp32 (the reference's own arithmetic).
    fp32 convolutions run ~57x slower than fp16 (no tensor cores), so that leg plays one ply of a 120-playout search: the rate per
    wave is what is measured (the network is > 99 % of such a wave), the line says which playout count was used."""
    out = {}
    for prec, steps, warm, playouts in (("tf32", 2, 1, a.playouts), ("tf32x3", 1, 1, a.playouts // 2), ("fp32", 1, 0, min(a.playouts, 120))):
        r = Runner(a, rank, world, local_rank, a.games, playouts, a.res_blocks, prec, pv=pv, arena_words=1 << 20)
        m = r.plies(steps, warm)
        out[prec] = dict(value=m["value"], e2e=m["e2e"], plies_timed=steps, playouts=playouts, ms_per_step=m["e2e_ms"] / steps,
                         nn_tflops=m["expansions"] * FLOPS_PER_EVAL.get(a.res_blocks, 0) / (m["dev_ms"] * 1e-3) / 1e12 / world)
        r.close()
    return out


def leg_config(a, rank, world, local_rank, games, playouts, res_blocks, steps, warmup, label, pv=None):
    r = Runner(a, rank, world, local_rank, games, playouts, res_blocks, a.precision, pv=pv, arena_words=1 << 20)
    m = r.plies(steps, warmup)
    out = dict(workload=label, value=m["value"], e2e=m["e2e"], unit="expansions/s", n_gpus=world, plies_timed=steps, ms_per_step=m["e2e_ms"] / steps,
               dtype=a.precision, nn_tflops_per_gpu=m["expansions"] * FLOPS_PER_EVAL.get(res_blocks, 0) / (m["dev_ms"] * 1e-3) / 1e12 / world)
    r.close()
    return out


def leg_config5(a, local_rank, pv):
    """BASELINE configs[4]: ai_count=2 play mode, mcts vs mcts, 1200 playouts.  One tree; per move the game_mode_2 sequence of
    ChessGame.change_player (ChessGame.py:153-181): get_hint('mcts') -- which runs a full search when the new root is not expanded
    (main.py:1281-1284) -- then perform_AI -> select_move('mcts') (another `playouts` playouts on the re-used root)."""
    from cchess_zero_b200.selfplay import cchess_main
    out = {}
    modes = (("search_threads_1", 1, 1, 12, "one playout at a time: bit-exact with the reference at search_threads=1"),
             ("search_threads_16", 16, 1, 24, "the reference's DEFAULT coroutine schedule (search_threads=16) in canonical FIFO form: "
                                              "identical visit counts wherever the reference reproduces itself; up to 16 leaves per network call"),
             ("leaf_parallel_8", 1, 8, 24, "the package's own virtual-loss batching of 8 leaves per network call (deterministic, not the reference's visit counts)"))
    for name, T, K, moves, sem in modes:
        with contextlib.redirect_stdout(io.StringIO()):
            m = cchess_main(playout=a.playouts, in_search_threads=T, network=pv, exploration=False, log_file=False, leaf_parallel=K)
        np.random.seed(0)
        lat, hint_s = [], []
        with contextlib.redirect_stdout(io.StringIO()):
            for i in range(moves + 2):
                t0 = time.perf_counter()
                m.get_hint("mcts", True, lambda: None)
                t1 = time.perf_counter()
                m.select_move("mcts")
                t2 = time.perf_counter()
                if i >= 2:
                    lat.append(t2 - t0); hint_s.append(t1 - t0)
                if m.check_end()[0]:
                    m.game_borad.reload(); m.mcts.reload()
        lat = np.array(lat)
        out[name] = dict(
            p50_s=float(np.median(lat)), p95_s=float(np.percentile(lat, 95)), mean_s=float(lat.mean()), max_s=float(lat.max()), moves=len(lat),
            get_hint_share=float(np.sum(hint_s) / np.sum(lat)), playouts_per_s=a.playouts / float(np.median(lat)), semantics=sem)
        m.mcts.engine.close()
    out["config"] = "1 game, mcts vs mcts, %d playouts, res_block_nums=%d, exploration off, per move get_hint('mcts') + select_move('mcts')" % (a.playouts, a.res_blocks)
    return out


def leg_threads16(a, rank, world, local_rank, pv, games=256):
    """`games` games x `playouts` playouts with search_threads = 16 inside every game (the reference's default schedule, exact): the
    network batch is games x 16 rows per wave, of which ~11 of 16 carry a leaf: only those are evaluated (row compaction,
    cz_engine_wave_compact; the network runs on bucketed batch sizes from lazily captured CUDA graphs)."""
    from cchess_zero_b200.selfplay import SelfPlay
    K = 16
    sp = SelfPlay(games, None, a.playouts, seeds=[rank * games + g for g in range(games)], device=local_rank, auto_reset=True, keep_records=False,
                  plan_factory=lambda n: pv.native_plan(n, a.first_conv), search_threads=K, arena_words=1 << 21)
    sp.capture_graph()
    e = sp.engine
    for _ in range(2):
        sp.step()
    torch.cuda.synchronize()
    c0, w0, r0 = e.counters(), sp.waves, getattr(sp, "rows_evaluated", 0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    steps = 4
    for _ in range(steps):
        sp.step()
    ev1.record()
    torch.cuda.synchronize()
    c1 = e.raise_on_error()
    ms = ev0.elapsed_time(ev1)
    n = c1["n_expand"] - c0["n_expand"]
    out = dict(workload="%d concurrent games x %d playouts, search_threads=%d inside every game (k_wave_fifo), res_block_nums=%d" % (games, a.playouts, K, a.res_blocks),
               e2e=n / (ms * 1e-3), unit="expansions/s", plies_timed=steps, ms_per_step=ms / steps, waves_per_step=(sp.waves - w0) / steps,
               network_rows_per_wave=games * K, leaves_per_wave=n / max(1, sp.waves - w0),
               row_compaction=bool(getattr(sp, "compact", False)),
               rows_evaluated_per_wave=((sp.rows_evaluated - r0) / max(1, sp.waves - w0)) if getattr(sp, "compact", False) else games * K,
               semantics="every game follows the reference's search_threads=16 coroutine schedule (canonical FIFO form, pinned to real uvloop runs)")
    e.close()
    return out


def leg_dedup(a, rank, world, local_rank, pv):
    """Board hashing (north_star): Zobrist keys of every evaluated leaf of one ply of the main workload.  Reports how many evaluations
    a position-keyed cache could have saved: repeats inside a game (transpositions in one tree) and identical positions in the same
    network batch (across games).  The keys never influence the search."""
    from cchess_zero_b200.selfplay import SelfPlay
    B = a.games
    sp = SelfPlay(B, None, a.playouts, seeds=[rank * B + g for g in range(B)], device=local_rank, auto_reset=True, keep_records=False,
                  plan=pv.native_plan(B, a.first_conv), hashing=True, arena_words=1 << 20)
    sp.capture_graph()
    for _ in range(6):                                          # six plies in: the games have diverged from the common start position
        sp.step()
    e = sp.engine
    e.begin_search(a.playouts)
    keys = []
    lk = e.leaf_hashes()
    for _ in range(a.playouts + 2):
        sp.graph.replay()
        keys.append(lk.clone())
    torch.cuda.synchronize()
    k = torch.stack(keys)                                        # [waves, B]; 0 = no leaf from that game in that wave
    live = k != 0
    total = int(live.sum())
    srt, _ = torch.sort(k, dim=0)
    per_game_unique = int(((srt[1:] != srt[:-1]) & (srt[1:] != 0)).sum() + (srt[0] != 0).sum())
    srt_w, _ = torch.sort(k, dim=1)
    per_wave_unique = int(((srt_w[:, 1:] != srt_w[:, :-1]) & (srt_w[:, 1:] != 0)).sum() + (srt_w[:, 0] != 0).sum())
    all_unique = int(torch.unique(k[live]).numel())
    e.close()
    return dict(evaluated_leaves=total, repeats_within_a_game=1.0 - per_game_unique / max(1, total),
                repeats_within_a_network_batch=1.0 - per_wave_unique / max(1, total), repeats_overall=1.0 - all_unique / max(1, total),
                note="one ply (ply 7) of the main workload; a repeat = a leaf whose Zobrist key (position + side to move) was already evaluated "
                     "in the same game's search / in the same wave's batch / anywhere in the ply")


def leg_soak(runner, plies):
    """games/hour without selection bias.  All slots restart from the start position at ply 0 of the soak; L = length of the
    FIRST game of every slot, observed exactly up to the window T (longer ones are censored at T), so
    E[min(L, T)] = sum_{t<T} S(t) is unbiased; with the censored share small it is the mean game length.
    games/hour = plies/s * 3600 / plies_per_game (renewal rate), plies/s measured end to end over the soak."""
    sp = runner.sp
    sp.engine.reset()
    st = sp.engine.status(boards=True)
    sp.boards, sp.sides = st["boards"], st["side"]
    from cchess_zero_b200.selfplay import GameRecord
    sp.records = [GameRecord(g, None, sp.temperature) for g in range(sp.B)]
    sp._span = [[] for _ in range(sp.B)]
    sp.keep_records = False                                    # lengths only: keeps the soak's host memory flat
    first_len = np.full(sp.B, -1, dtype=np.int64)
    all_len = []

    def on_step(out):
        for g, rec in out["finished"]:
            all_len.append(len(rec))
            if first_len[g] < 0:
                first_len[g] = len(rec)
        sp.pop_finished()
    gather, runner.gather = runner.gather, None               # the soak measures lengths only: no tuples to ship
    m = runner.plies(plies, 0, on_step=on_step)
    runner.gather = gather
    sp.keep_records = True
    T = plies
    obs = first_len[first_len >= 0]
    censored = int((first_len < 0).sum())
    lens = np.concatenate([obs, np.full(censored, T)])
    mean_trunc = float(lens.mean())                              # E[min(L, T)]
    plies_per_s = runner.world * sp.B * plies / (m["e2e_ms"] * 1e-3)
    ok = T >= 3 * mean_trunc and censored <= 0.05 * sp.B
    return dict(games_per_hour=(plies_per_s * 3600.0 / mean_trunc) if ok else None, plies_per_s=plies_per_s, window_plies=T,
                plies_per_game=mean_trunc, first_games_observed=int(len(obs)), first_games_censored_at_window=censored,
                length_percentiles={str(p): float(np.percentile(obs, p)) for p in (5, 25, 50, 75, 95)} if len(obs) else None,
                all_games_finished=len(all_len) * 1.0, value=m["value"], e2e=m["e2e"],
                valid=bool(ok), rule="reported only when the window is >= 3 x E[min(L,T)] and <= 5 % of the first games are censored",
                note="seed-0 (untrained) network: games end by king capture or the 60-ply no-capture rule (main.py:1532-1545)")


def dump_outputs(d, out, limit=63 << 20):
    """Writes what SelfPlay.step() returned (`out`) as d/<name>.npy: per game slot the chosen child, its win rate (mcts.Q) and the
    game status after the move; per game that ended in this ply its slot, length, z and dense pi rows (the (s, pi, z) tuples of
    selfplay(), game after game).  Integers are stored exactly as float64.  game_slots.npy names the slots written: all of them,
    or, when that would exceed `limit` bytes (64 MB less room for the .npy headers), a fixed seeded sample."""
    st = out["status"]
    per_game = dict(choice=out["choice"].astype(np.float64), win_rate=out["win_rate"].astype(np.float32),
                    boards=st["boards"].astype(np.float32), side=st["side"].astype(np.float64), terminal=st["terminal"].astype(np.float64),
                    winner=st["winner"].astype(np.float64), ply=st["ply"].astype(np.float64), rr=st["rr"].astype(np.float64),
                    q=st["q"].astype(np.float32), root_N=st["root_N"].astype(np.float64))
    B = len(out["choice"])
    fin = {g: (rec.z.astype(np.float64), rec.dense_pi()) for g, rec in out["finished"]}
    cost = np.full(B, sum(v[0].nbytes for v in per_game.values()), dtype=np.int64)
    for g, (z, pi) in fin.items():
        cost[g] += 16 + z.nbytes + pi.nbytes
    if cost.sum() <= limit:
        slots = np.arange(B)
    else:
        order = np.random.RandomState(0).permutation(B)
        slots = np.sort(order[:int(np.searchsorted(np.cumsum(cost[order]), limit, side="right"))])
    done = [g for g in slots if g in fin]
    arrays = {k: v[slots] for k, v in per_game.items()}
    arrays.update(game_slots=slots.astype(np.float64), finished_slot=np.array(done, dtype=np.float64),
                  finished_plies=np.array([len(fin[g][0]) for g in done], dtype=np.float64),
                  finished_z=np.concatenate([fin[g][0] for g in done] or [np.zeros(0)]),
                  finished_pi=np.concatenate([fin[g][1] for g in done] or [np.zeros((0, 2086))]))
    os.makedirs(d, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(d, k + ".npy"), v)


# ---------------------------------------------------------------------------------------------
def run_ours(a, rank, world, local_rank):
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    legs = set() if a.legs == "none" else set(x for x in a.legs.split(",") if x)
    if a.no_cpu_baseline:
        legs.discard("cpu")
    main = Runner(a, rank, world, local_rank, a.games, a.playouts, a.res_blocks, a.precision)
    sp, e, plan = main.sp, main.sp.engine, main.plan

    if a.kwave_capture:                                          # helper for ncu: deep trees first, then eager waves
        for _ in range(a.warmup):
            sp.step()
        main.kwave_roofline(a.profile_waves)
        return

    clocks = ClockSampler(local_rank) if rank == 0 else None
    m = main.plies(a.steps, a.warmup, clocks=clocks)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, m["last"])
    roof = main.kwave_roofline(a.profile_waves) if rank == 0 else None
    if world > 1:
        dist.barrier()
    c1 = m["c1"]
    extra = dict(expansions=m["expansions"], waves_per_step=m["waves"] / a.steps, games_finished_in_timed_region=m["games_done"],
                 tuples_all_gathered=main.tuples_gathered, tuple_gather_bytes=main.gather.bytes_gathered if main.gather else 0,
                 nn_tflops=m["expansions"] * FLOPS_PER_EVAL.get(a.res_blocks, 0) / (m["dev_ms"] * 1e-3) / 1e12 / world,
                 max_arena_words=c1["max_arena_words"], max_depth=c1["max_depth"],
                 mean_L=(c1["sum_L"] - m["c0"]["sum_L"]) / max(1, c1["n_playout"] - m["c0"]["n_playout"]),
                 mean_children=(c1["sum_C"] - m["c0"]["sum_C"]) / max(1, c1["n_expand"] - m["c0"]["n_expand"]))
    _, _, peaks = measured_peaks()
    tpeak = float(peaks.get("bf16_tflops_sustained", 0) or 0)
    # the kernels that DOMINATE a wave are the library tcgen05 convolutions of the residual tower: their share of the roofline over the
    # whole search (all other kernels, launch gaps and the tree kernel included in the time), against the measured sustained bf16 peak
    extra["tower_roofline"] = dict(bound="tensor", achieved=extra["nn_tflops"], unit="TFLOP/s", peak=tpeak or None,
                                   frac=(extra["nn_tflops"] / tpeak) if tpeak else None,
                                   peak_source="MEASURED_PEAKS.json bf16_tflops_sustained" if tpeak else None,
                                   note="network FLOPs of every evaluated leaf (%.1f MFLOP each) / device time of the whole search" % (FLOPS_PER_EVAL.get(a.res_blocks, 0) / 1e6))
    if "soak" in legs:
        s = leg_soak(main, a.soak_plies)
        extra["soak"] = s
        extra["games_per_hour"] = s["games_per_hour"]
        extra["plies_per_game"] = s["plies_per_game"]
    else:
        extra["games_per_hour"] = None                           # never extrapolated from the few games that end inside a short window
    pv = main.pv
    main.close()
    if "config3" in legs:
        extra["config3"] = leg_config(a, rank, world, local_rank, 512, 1600, 7, 3, 2,
                                      "BASELINE configs[2] per-rank shape: 512 concurrent games x 1600 playouts per GPU, res_block_nums=7 (4096 games at 8 GPUs)",
                                      pv=pv if a.res_blocks == 7 else None)
    if world == 1:
        if "precision" in legs:
            extra["by_precision"] = dict(fp16=dict(value=m["value"], e2e=m["e2e"], plies_timed=a.steps, playouts=a.playouts, ms_per_step=m["e2e_ms"] / a.steps)) \
                if a.precision == "fp16" else {}
            extra["by_precision"].update(leg_precision(a, rank, world, local_rank, pv))
            pp = os.path.join(ROOT, "profiles", "r02_nn_precision_scaled.json")
            if os.path.exists(pp):
                extra["by_precision"]["error_vs_fp64_at_realistic_logit_scale"] = json.load(open(pp))
        if "config4" in legs:
            extra["config4"] = leg_config(a, rank, world, local_rank, a.games, a.playouts, 19, 3, 2,
                                          "BASELINE configs[3]: %d games x %d playouts, res_block_nums=19" % (a.games, a.playouts))
        if "config5" in legs:
            extra["config5"] = leg_config5(a, local_rank, pv)
        if "threads16" in legs:
            extra["search_threads_16"] = leg_threads16(a, rank, world, local_rank, pv)
            extra["search_threads_16_full_batch"] = leg_threads16(a, rank, world, local_rank, pv, games=a.games)
        if "dedup" in legs:
            extra["eval_dedup"] = leg_dedup(a, rank, world, local_rank, pv)
    cpu = None
    if rank == 0 and world == 1 and "cpu" in legs:
        try:
            cpu, _ = reference_cpu(3, 1, a.playouts, a.res_blocks, a.cpu_seconds, tree_only=False)
        except Exception as ex:
            cpu = dict(error=str(ex)[-300:])

    if rank == 0:
        B = a.games
        h2d = B * 4 + B          # chosen child indices + search mask
        d2h = B * 4 + B * 128 * (2 + 4) + B * 112 + 4    # root n / moves / visits, packed status records, the unfinished count
        line = dict(metric=METRIC, value=m["value"], unit="expansions/s", n_gpus=world, steps=a.steps, warmup=a.warmup,
                    ms_per_step=m["e2e_ms"] / a.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype=a.precision, data="synthetic (seed-0 xavier-initialised network, all games from the start position)",
                    config=dict(workload="%d concurrent self-play games x %d playouts per move, res_block_nums=%d, per GPU" % (B, a.playouts, a.res_blocks),
                                games_per_gpu=B, playouts=a.playouts, res_block_nums=a.res_blocks, search_threads=1, exploration=True,
                                cuda_graph=not a.no_graph, lanes=a.lanes,
                                fused_conv_epilogue=plan.fused,
                                network_ends=("csrc/cz_net.cu (board-byte first conv [%s], fused heads)" % plan.first_conv) if plan.dtype == torch.uint8 else "library",
                                l2_policy="working set (trees %.1f GB + activations) exceeds the 126 MB L2" % (c1["max_arena_words"] * 4 * B / 1e9)),
                    e2e=dict(value=m["e2e"], unit="expansions/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, wall_ms=m["wall_ms"]),
                    gpu_launches=int(m["launches"]), clocks=m["clocks"], roofline=roof, cpu_baseline=cpu, extra=extra)
        print(json.dumps(line), flush=True)


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    run_ours(a, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
