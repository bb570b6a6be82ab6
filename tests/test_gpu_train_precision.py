"""GPU tests of rows a18 / f1: network precision at REALISTIC logit magnitudes, the training update rule on CUDA,
data-parallel training over NCCL, and the weights-version protocol that keeps captured CUDA graphs current."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _positions(n, seed=0):
    from oracle import oracle as O
    rng = np.random.RandomState(seed)
    xs, cb, b, side = [], [], O.from_state(O.START), 0
    while len(xs) < n:
        xs.append(O.encode(b, side))
        c = np.zeros(96, np.uint8)
        c[:90] = O.flip_board(b) if side == 1 else b
        cb.append(c)
        mv = O.legal_moves(b, side)
        b, cap = O.apply_move(b, mv[rng.randint(len(mv))]); side ^= 1
        if cap in (1, 8):
            b, side = O.from_state(O.START), 0
    return np.stack(xs), np.stack(cb)


def scaled_net(blocks, target_logit=8.0, target_value=0.5, seed=0):
    """The seed-0 network with its two output layers rescaled so that max |logit| ~ target_logit and median |value| ~
    target_value on random-play positions -- the magnitudes a trained policy produces (the raw xavier network gives
    |logit| <= 0.14, where every precision trivially passes an absolute tolerance)."""
    from cchess_zero_b200.net import PolicyValueNet
    torch.manual_seed(seed)
    net = PolicyValueNet(blocks).eval()
    x, _ = _positions(64, seed=1)
    with torch.no_grad():
        lo, _ = net.double()(torch.from_numpy(x).double())
        net.p_fc.weight.mul_(target_logit / lo.abs().max().item())
        # pre-tanh activation scaled to atanh(target_value) at the median
        v_pre = net.v_fc2(torch.relu(net.v_fc1(torch.relu(net.v_bn(net.v_conv(_tower(net, x)))).permute(0, 2, 3, 1).reshape(len(x), 90))))
        net.v_fc2.weight.mul_(float(np.arctanh(target_value)) / max(v_pre.abs().median().item(), 1e-12))
    return net.float()


def _tower(net, x):
    import torch.nn.functional as F
    t = torch.from_numpy(x).double().permute(0, 3, 1, 2)
    t = F.relu(net.bn_in(net.conv_in(t)))
    for b in net.blocks:
        t = b(t)
    return t


def precision_study(blocks, n=96):
    """max-abs and relative error of every inference precision against an fp64 evaluation of the same weights."""
    from cchess_zero_b200.net import NativePlan, make_plan
    net = scaled_net(blocks)
    x, canon = _positions(n, seed=2)
    with torch.no_grad():
        rl, rv = net.double()(torch.from_numpy(x).double())
    net = net.float().cuda().to(memory_format=torch.channels_last)
    scale_l, scale_v = rl.abs().max().item(), rv.abs().max().item()
    out = dict(logit_absmax=scale_l, value_absmax=scale_v, value_absmedian=rv.abs().median().item())
    for prec in ("fp32", "tf32x3", "tf32", "fp16", "bf16"):
        plan = make_plan(net, prec)
        l, v = plan(torch.from_numpy(x).cuda().to(plan.dtype))
        el = (l.double().cpu() - rl).abs().max().item()
        ev = (v.double().cpu().reshape(-1) - rv.reshape(-1)).abs().max().item()
        out[prec] = dict(logit_abs=el, value_abs=ev, logit_rel=el / scale_l, value_rel=ev / max(scale_v, 1e-12))
    nat = NativePlan(net, n)
    lo = torch.zeros((n, 2086), device="cuda"); vo = torch.zeros((n,), device="cuda")
    nat(torch.from_numpy(canon).cuda(), lo, vo)
    torch.cuda.synchronize()
    el = (lo.double().cpu() - rl).abs().max().item()
    ev = (vo.double().cpu() - rv.reshape(-1)).abs().max().item()
    out["fp16_native_ends"] = dict(logit_abs=el, value_abs=ev, logit_rel=el / scale_l, value_rel=ev / max(scale_v, 1e-12))
    return out


@pytest.mark.parametrize("blocks", [7, 19])
def test_precision_at_realistic_logit_scale(blocks):
    """north_star: "NN outputs match within 1e-3 fp32".  With max |logit| ~ 8 and |value| ~ 0.5 (a trained network's range;
    the raw seed-0 network has |logit| <= 0.14, where any arithmetic passes an absolute bound):
      * fp32 (the reference's own arithmetic, policy_value_network.py:202-214) meets 1e-3 ABSOLUTE with two decades of margin;
      * fp16 (default) and tf32 carry 10-11 bit mantissas through 15 (7 blocks) / 39 (19 blocks) convolutions: measured
        1.0e-3 .. 1.4e-3 of max |logit| at 7 blocks and 4.3e-3 .. 5.7e-3 at 19 blocks on the logits (1e-2 / 4.5e-2 absolute at
        |logit| = 8), 5e-4 .. 7e-4 / 1.2e-3 .. 1.8e-3 absolute on the tanh value.  They do NOT meet an absolute 1e-3 on logits of
        this size.  The tolerance this package states for them (DESIGN.md section 4) is relative to max |logit| -- priors are ratios of
        logits, main.py:176-187 -- 2e-3 (7 blocks) / 8e-3 (19 blocks), and 1e-3 / 3e-3 absolute on the value.  precision="fp32"
        is the 1e-3-absolute mode and what it costs is on the bench line (extra.by_precision);
      * tf32x3 (net.py: SplitTf32Plan -- hi/lo operand split, three TF32 products per term accumulated in f32 on the tensor cores)
        meets 1e-3 ABSOLUTE with the same margin as fp32 at a fraction of fp32's cost (extra.by_precision);
      * bf16 misses all of it by a decade and is not offered."""
    r = precision_study(blocks)
    print("precision study (%d blocks): %s" % (blocks, json.dumps(r)))
    assert 4.0 < r["logit_absmax"] < 16.0 and 0.2 < r["value_absmedian"] < 0.9
    assert r["fp32"]["logit_abs"] < 1e-3 / 5 and r["fp32"]["value_abs"] < 1e-4      # 1e-3 absolute, with margin
    assert r["tf32x3"]["logit_abs"] < 1e-3 / 2 and r["tf32x3"]["value_abs"] < 1e-4  # the tensor-core mode that meets it too (accumulator truncation is what is left)
    rel_tol, val_tol = (2e-3, 1e-3) if blocks <= 7 else (8e-3, 3e-3)
    for p in ("tf32", "fp16", "fp16_native_ends"):
        assert r[p]["logit_rel"] < rel_tol, (p, r[p])
        assert r[p]["value_abs"] < val_tol, (p, r[p])
    assert r["bf16"]["logit_rel"] > rel_tol                                          # why bf16 is rejected


def test_tf32_split_kernel_matches_its_torch_statement_and_search_runs_in_tf32x3():
    """csrc/cz_net.cu: k_split_tf32 == net.split_acts bit for bit (incl. negative values, zeros, denormal-sized residues), and a
    whole search with precision="tf32x3" (engine planes -> SplitTf32Plan -> tree) gives the visit counts of the fp32 evaluator on
    the same weights (both are ~1e-6 from the exact network, far below any PUCT decision margin of these positions)."""
    import ctypes as C
    from cchess_zero_b200._lib import lib
    from cchess_zero_b200.net import policy_value_network, split_acts
    from cchess_zero_b200.mcts import MCTS_tree
    torch.manual_seed(3)
    for n_pix in (1, 90, 90 * 37 + 5):
        y = torch.randn((n_pix, 128), device="cuda") * torch.logspace(-4, 3, 128, device="cuda")
        y[0, :4] = torch.tensor([0.0, -0.0, 1.0, -1.0], device="cuda")
        hi = torch.full((n_pix, 128), float("nan"), device="cuda")
        x2 = torch.full((n_pix, 256), float("nan"), device="cuda", dtype=torch.float16)
        assert lib().cz_net_split_tf32(y.data_ptr(), hi.data_ptr(), x2.data_ptr(), n_pix, C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        rh, r2 = split_acts(y.t().reshape(1, 128, n_pix, 1))
        assert torch.equal(hi.view(torch.int32), rh.reshape(128, n_pix).t().contiguous().view(torch.int32))
        assert torch.equal(x2.view(torch.int16), r2.reshape(256, n_pix).t().contiguous().view(torch.int16))
        assert int((hi.view(torch.int32) & 0x1FFF).abs().max()) == 0
        # the fused epilogue + split: v = relu(t + 2^-11 s + bias + skip) written in place of skip, and v's split
        t = torch.randn((n_pix, 128), device="cuda"); sc = (torch.randn((n_pix, 128), device="cuda") * 3).half()
        bias = torch.randn(128, device="cuda"); skip = torch.randn((n_pix, 128), device="cuda")
        want = torch.relu(((t + sc.float() * (1.0 / 2048.0)) + bias) + skip)
        xs = skip.clone(); hi.fill_(float("nan")); x2.fill_(float("nan"))
        assert lib().cz_net_epilogue_split(t.data_ptr(), sc.data_ptr(), bias.data_ptr(), xs.data_ptr(), xs.data_ptr(), hi.data_ptr(), x2.data_ptr(),
                                           n_pix, C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        assert torch.equal(xs, want)
        rh, r2 = split_acts(want.t().reshape(1, 128, n_pix, 1))
        assert torch.equal(hi, rh.reshape(128, n_pix).t()) and torch.equal(x2.view(torch.int16), r2.reshape(256, n_pix).t().contiguous().view(torch.int16))
        xo = torch.empty_like(t)                                                # no cross terms, no skip, no split (first layer / last layer shapes)
        assert lib().cz_net_epilogue_split(t.data_ptr(), None, bias.data_ptr(), None, xo.data_ptr(), None, None, n_pix,
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        assert torch.equal(xo, torch.relu(t + bias))
    visits = {}
    for prec in ("fp32", "tf32x3"):
        pv = policy_value_network(2, precision=prec, seed=5)
        with torch.no_grad():
            pv.net.p_fc.weight.mul_(40.0)
        pv.weights_version += 1
        from cchess_zero_b200 import rules
        t = MCTS_tree(rules.START_STATE, pv.forward, 1)
        t.main(rules.START_STATE, "w", 0, 200)
        visits[prec] = [[a, n.N] for a, n in t.root.child.items()]
    assert sum(n for _, n in visits["fp32"]) == 200 - 1 or sum(n for _, n in visits["fp32"]) == 200
    assert visits["fp32"] == visits["tf32x3"]


def test_train_step_on_cuda_matches_written_out_update_rule():
    """train_step_module ON THE GPU against the float64 restatement of policy_value_network.py:76-126 (the CPU tier pins the
    same rule on the host; this is the path the product runs)."""
    from cchess_zero_b200.net import PolicyValueNet, train_step_module
    torch.manual_seed(3)
    net = PolicyValueNet(1).cuda()
    ref = PolicyValueNet(1).double()
    ref.load_state_dict({k: v.double().cpu() for k, v in net.state_dict().items()})
    opt = torch.optim.SGD(net.parameters(), lr=1e-3, momentum=0.9, nesterov=True)
    g = torch.Generator().manual_seed(5)
    x = (torch.rand(10, 9, 10, 14, generator=g) < 0.03).float()
    pi = torch.softmax(torch.randn(10, 2086, generator=g) * 3, 1)
    z = torch.sign(torch.randn(10, 1, generator=g))
    lr, m, c = 0.02, 0.9, 1e-4
    accum = [torch.zeros_like(p) for p in ref.parameters()]
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False     # training runs in fp32 like the reference
    try:
        for step in range(3):
            acc, loss = train_step_module(net, opt, x.cuda(), pi.cuda(), z.cuda(), lr)
            ref.train()
            lo, v = ref(x.double())
            rloss = (-(pi.double() * torch.log_softmax(lo, 1)).sum(1)).mean() + ((v - z.double()) ** 2).mean() \
                + c * sum((p ** 2).sum() / 2 for p in ref.parameters())
            grads = torch.autograd.grad(rloss, list(ref.parameters()))
            gn = torch.sqrt(sum((gr ** 2).sum() for gr in grads))
            scale = min(1.0, 100.0 / float(gn))
            with torch.no_grad():
                for p, gr, a in zip(ref.parameters(), grads, accum):
                    gr = gr * scale
                    a.mul_(m).add_(gr)
                    p.sub_(lr * (gr + m * a))
            assert abs(loss - float(rloss)) < 2e-4 * max(1.0, abs(float(rloss)))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    for p, q in zip(net.parameters(), ref.parameters()):
        assert torch.allclose(p.double().cpu(), q, atol=5e-5, rtol=2e-4)


def test_search_uses_trained_weights_after_train_step_and_restore(tmp_path, monkeypatch):
    """ADVICE r1 (high): MCTS_tree / SelfPlay capture a plan with folded weight COPIES into a CUDA graph; train_step and
    restore must reach those copies.  Protocol: policy_value_network.weights_version + plan.refresh_if_stale()."""
    monkeypatch.chdir(tmp_path)
    from cchess_zero_b200 import rules
    from cchess_zero_b200.mcts import MCTS_tree
    from cchess_zero_b200.net import policy_value_network
    from cchess_zero_b200.selfplay import SelfPlay
    pv = policy_value_network(res_block_nums=2)
    t = MCTS_tree(rules.START_STATE, pv.forward, 1)
    sp = SelfPlay(8, None, 8, seeds=range(8), arena_words=1 << 16, plan=pv.native_plan(8), auto_reset=False)
    sp.capture_graph()

    def root_priors():
        t.reload()
        t.main(rules.START_STATE, "w", 0, 4)
        return np.array([n.P for n in t.root.child.values()])

    def batch_priors():
        sp.engine.reset()
        sp.search()
        return sp.engine.root_children()["p"][0, :44].copy()

    p0, b0 = root_priors(), batch_priors()
    assert np.array_equal(p0, root_priors())                           # deterministic while the weights stand still
    x, _ = _positions(16)
    pi = np.zeros((16, 2086), np.float32); pi[np.arange(16), np.arange(16) * 11] = 1
    z = np.ones((16, 1), np.float32)
    v0 = pv.weights_version
    for _ in range(3):
        pv.train_step(x, pi, z, 0.05)
    assert pv.weights_version == v0 + 3
    p1, b1 = root_priors(), batch_priors()
    assert not np.array_equal(p0, p1), "MCTS_tree searched with stale weights"
    assert not np.array_equal(b0, b1), "SelfPlay searched with stale weights"
    assert np.allclose(p1, b1, rtol=2e-2, atol=2e-3)                   # both paths now evaluate the same (new) network (cluster trunk vs cuDNN trunk: fp16 rounding apart)
    path = pv.save(3)
    for _ in range(2):
        pv.train_step(x, pi, z, 0.05)
    p2 = root_priors()
    pv.restore(path)                                                    # back to the step-3 weights
    p3 = root_priors()
    assert not np.array_equal(p2, p3) and np.array_equal(p1, p3)


def test_gpu_variant_restores_from_its_own_directory(tmp_path, monkeypatch):
    """ADVICE r1 (medium): policy_value_network_gpus saves to AND restores from ./gpu_models (policy_value_network_gpus.py:14)."""
    monkeypatch.chdir(tmp_path)
    from cchess_zero_b200.net import policy_value_network, policy_value_network_gpus
    a = policy_value_network_gpus(1, 2)
    x, _ = _positions(8)
    pi = np.zeros((8, 2086), np.float32); pi[:, 5] = 1
    a.train_step(x, pi, np.ones((8, 1), np.float32), 0.01)
    a.save(1)
    assert os.path.isfile(tmp_path / "gpu_models" / "checkpoint") and not os.path.exists(tmp_path / "models")
    b = policy_value_network_gpus(1, 2)
    assert b.global_step == 1
    assert np.array_equal(a.forward(x)[0], b.forward(x)[0])
    c = policy_value_network(2)                                          # the cpu variant does not pick the gpu checkpoint up
    assert c.global_step == 0


_NCCL_DP = r'''
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
from cchess_zero_b200.net import PolicyValueNet, train_step_module
lr_ = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr_)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr_))
rank, world = dist.get_rank(), dist.get_world_size()
torch.manual_seed(0)
net = PolicyValueNet(2).cuda()
opt = torch.optim.SGD(net.parameters(), lr=1e-2, momentum=0.9, nesterov=True)
g = torch.Generator().manual_seed(100 + rank)                    # one mini-batch ("tower") per rank
x = (torch.rand(8, 9, 10, 14, generator=g) < 0.03).float().cuda()
pi = torch.softmax(torch.randn(8, 2086, generator=g), 1).cuda()
z = torch.sign(torch.randn(8, 1, generator=g)).cuda()
before = torch.cat([p.detach().reshape(-1) for p in net.parameters()]).clone()
for _ in range(3):
    acc, loss = train_step_module(net, opt, x, pi, z, 1e-2)      # gradient all_reduce over NCCL inside
after = torch.cat([p.detach().reshape(-1) for p in net.parameters()])
allp = [torch.empty_like(after) for _ in range(world)]
dist.all_gather(allp, after)
assert torch.isfinite(after).all() and not torch.equal(before, after)
assert all(torch.equal(allp[0], q) for q in allp), "replicas diverged"
if rank == 0: print("NCCL_DP_OK", world, float(loss))
dist.barrier(); dist.destroy_process_group()
'''


def test_data_parallel_train_step_over_nccl(tmp_path):
    """f1 on the hardware it targets: the gradient all_reduce that replaces policy_value_network_gpus.average_gradients
    (policy_value_network_gpus.py:216-250), 2 ranks over NCCL.  Needs 2 GPUs (gpurun --gpus 2); skipped on a 1-GPU box."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "dp.py"
    script.write_text(_NCCL_DP % ROOT)
    env = dict(os.environ, CCHESS_NO_REBUILD="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29541", str(script)], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "NCCL_DP_OK 2" in r.stdout


@pytest.mark.parametrize("blocks,cluster,npos", [(2, 1, 1), (2, 8, 3), (7, 1, 2), (7, 2, 1), (7, 4, 5), (7, 8, 16), (19, 8, 1)])
def test_small_tower_cluster_kernel_matches_library_plan_and_fp64(blocks, cluster, npos):
    """csrc/cz_tower.cu (whole trunk in one launch: TMA-streamed weights, tcgen05.mma with tap-shifted A descriptors, TMEM epilogues
    exchanging channel slices through distributed shared memory) against the cuDNN plan and an fp64 evaluation, for every cluster size."""
    from cchess_zero_b200.net import NativePlan, PolicyValueNet, SmallTowerPlan
    torch.manual_seed(1)
    net = PolicyValueNet(blocks).eval()
    with torch.no_grad():   # non-trivial biases / BN statistics so that every folded term is exercised
        for m in net.modules():
            if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear)):
                m.bias.uniform_(-0.1, 0.1)
            if hasattr(m, "running_var"):
                m.running_var.uniform_(0.5, 1.5); m.running_mean.uniform_(-0.2, 0.2)
    x, canon = _positions(npos, seed=5 + npos)
    with torch.no_grad():
        rl, rv = net.double()(torch.from_numpy(x).double())
    net = net.float().cuda().to(memory_format=torch.channels_last)
    boards = torch.from_numpy(canon).cuda()
    lo = torch.zeros((npos, 2086), device="cuda"); vo = torch.zeros((npos,), device="cuda")
    lo2 = torch.zeros_like(lo); vo2 = torch.zeros_like(vo)
    small = SmallTowerPlan(net, 16, cluster)
    small(boards, lo, vo)
    NativePlan(net, 16)(boards, lo2, vo2)
    torch.cuda.synchronize()
    e_small = max((lo.double().cpu() - rl).abs().max().item(), (vo.double().cpu() - rv.reshape(-1)).abs().max().item())
    e_lib = max((lo2.double().cpu() - rl).abs().max().item(), (vo2.double().cpu() - rv.reshape(-1)).abs().max().item())
    print("max abs err vs fp64: cluster trunk (CL=%d) %.3g, library trunk %.3g" % (cluster, e_small, e_lib))
    assert e_small < max(1e-3, 1.25 * e_lib)              # as accurate as the library trunk (same fp16 arithmetic, fp32 accumulation)
    assert (lo - lo2).abs().max().item() < max(2e-3, 2 * e_lib) and (vo - vo2).abs().max().item() < max(2e-3, 2 * e_lib)
    small(boards, lo2, vo2)                               # run-to-run identical
    torch.cuda.synchronize()
    assert torch.equal(lo, lo2) and torch.equal(vo, vo2)


@pytest.mark.parametrize("B", [128, 203, 1024])
def test_tcgen05_policy_fc_and_mma_head_conv_match_the_simt_heads(B):
    """cz_net_heads_tc (mma.sync head conv writing UMMA-tiled features, tcgen05 policy FC, 8-position value MLP) against the round-1
    kernels (cz_net_heads with CCHESS_HEAD_CONV=simt semantics) and against fp64, on a random trunk output."""
    from cchess_zero_b200.net import NativePlan, PolicyValueNet
    torch.manual_seed(2)
    net = PolicyValueNet(2).eval()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, (torch.nn.Conv2d, torch.nn.Linear)):
                m.bias.uniform_(-0.2, 0.2)
    net = net.cuda().to(memory_format=torch.channels_last)
    x, canon = _positions(B, seed=11)
    boards = torch.from_numpy(canon).cuda()
    outs = {}
    for mode in ("tc", "mma"):
        plan = NativePlan(net, B)
        plan.heads = mode
        lo = torch.zeros((B, 2086), device="cuda"); vo = torch.zeros((B,), device="cuda")
        plan(boards, lo, vo)
        plan(boards, lo, vo)
        torch.cuda.synchronize()
        outs[mode] = (lo, vo)
    with torch.no_grad():
        rl, rv = net.double()(torch.from_numpy(x).double().cuda())
    d_l = (outs["tc"][0] - outs["mma"][0]).abs().max().item()
    d_v = (outs["tc"][1] - outs["mma"][1]).abs().max().item()
    e_tc = max((outs["tc"][0].double() - rl).abs().max().item(), (outs["tc"][1].double() - rv.reshape(-1)).abs().max().item())
    e_mma = max((outs["mma"][0].double() - rl).abs().max().item(), (outs["mma"][1].double() - rv.reshape(-1)).abs().max().item())
    print("B=%d: tc vs mma heads: logits %.3g value %.3g; vs fp64: tc %.3g, mma %.3g" % (B, d_l, d_v, e_tc, e_mma))
    assert d_l < 1e-4 and d_v < 1e-5          # same fp16 operands, fp32 accumulation: only the summation order differs
    assert e_tc < max(1e-3, 1.25 * e_mma)


def test_single_tree_graph_with_several_waves_per_replay_is_the_same_search(monkeypatch):
    """MCTS_tree over the package's network replays a CUDA graph that holds 8 (wave -> evaluation) pairs (mcts.py: _search_graph);
    waves issued after the search is complete must change nothing: same visit counts and Q as one pair per replay, for playout counts
    that are not multiples of 8, and the tree stays reusable (update_tree + a second search)."""
    from cchess_zero_b200 import rules
    from cchess_zero_b200.mcts import MCTS_tree
    from cchess_zero_b200.net import policy_value_network
    pv = policy_value_network(2, seed=7)
    with torch.no_grad():
        pv.net.p_fc.weight.mul_(30.0)
    pv.weights_version += 1
    out = {}
    for reps in ("1", "8"):
        monkeypatch.setenv("CCHESS_WAVES_PER_GRAPH", reps)
        t = MCTS_tree(rules.START_STATE, pv.forward, 1)
        assert t._plan is not None
        res = []
        for playouts in (51, 333):
            t.main(t._state, "w" if t._side == 0 else "b", t._rr, playouts)
            ch = [(a, n.N, float(n.Q)) for a, n in t.root.child.items()]
            res.append(ch)
            best = max(ch, key=lambda x: x[1])[0]
            t.update_tree(best)
        assert t._reps == int(reps)
        out[reps] = res
        t.engine.close()
    assert out["1"] == out["8"]
