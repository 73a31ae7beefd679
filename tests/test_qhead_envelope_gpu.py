"""GPU tests of the fused output-layer + envelope + Bellman kernel (csrc/qhead_envelope.cu; SURVEY 8(f)2: the envelope operator folded into
the last-layer epilogue, reference multi_policy/envelope/envelope.py:420-440 + :298).

The kernel must be BIT-IDENTICAL to the three-launch chain it replaces (morl_gemm_planes_f32 for each net, then morl_envelope_td_f32):
  * its Q tiles (optional fp32 copies) equal the unfused output-layer GEMM bit for bit (same MMA order in tensor memory, same epilogue fma);
  * targets / preference indices / action indices equal the standalone operator's on those Q tensors AND the CPU oracle's
    (integer outputs and fp32 targets: exact equality, no tolerance);
  * Envelope.update() with the fused head produces exactly the losses, priorities and parameters of the update without it.
Shapes: the north-star (B=1024, |W|=64, |A|=8, d=3, K=256: 512 tiles on 148 CTAs, every ring / accumulator phase wraps), BASELINE
configs[1] (minecart dims: |W|=32, |A|=6, N=18 -- ragged Q rows, four transitions per tile), small / odd ones, constant Q (every
candidate ties: first occurrence), both row orders, the three scalarisation arithmetics."""

import os
import sys

import numpy as np
import pytest
import torch as th

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _operands(dev, B, W, A, D, K, seed, zero_act=False):
    from morl_baselines_b200 import ops

    fmt = ops.FMT_F16X2
    g = th.Generator(device=dev).manual_seed(seed)
    M, N = B * W, A * D
    s_act, s_w_on, s_w_tg = ops.scale_tensor(2.0, dev), ops.scale_tensor(4096.0, dev), ops.scale_tensor(2048.0, dev)
    h_on = th.randn(M, K, device=dev, generator=g).relu_()
    h_tg = (h_on + 0.05 * th.randn(M, K, device=dev, generator=g)).relu_()
    if zero_act:
        h_on.zero_()
        h_tg.zero_()
    w_on = th.randn(N, K, device=dev, generator=g) / 16.0
    w_tg = w_on + 0.01 * th.randn(N, K, device=dev, generator=g)
    b_on, b_tg = th.randn(N, device=dev, generator=g) * 0.1, th.randn(N, device=dev, generator=g) * 0.1
    a_on = ops.split_planes(h_on, fmt, rows_pad=M, ldp=K, scale=s_act)
    a_tg = ops.split_planes(h_tg, fmt, rows_pad=M, ldp=K, scale=s_act)
    p_on = ops.split_planes(w_on, fmt, rows_pad=32, ldp=K, scale=s_w_on)
    p_tg = ops.split_planes(w_tg, fmt, rows_pad=32, ldp=K, scale=s_w_tg)
    wset = th.rand(W, D, device=dev, generator=g)
    wset = wset / wset.sum(1, keepdim=True)
    rew = th.randn(B, D, device=dev, generator=g)
    done = (th.rand(B, device=dev, generator=g) < 0.1).float()
    return dict(a_on=a_on, a_tg=a_tg, p_on=p_on, p_tg=p_tg, b_on=b_on, b_tg=b_tg, s_act=s_act, s_w_on=s_w_on, s_w_tg=s_w_tg, wset=wset, rew=rew, done=done)


SHAPES = [
    pytest.param(1024, 64, 8, 3, 256, id="north_star"),
    pytest.param(256, 32, 6, 3, 256, id="config2_minecart"),
    pytest.param(2, 64, 8, 3, 64, id="one_tile"),
    pytest.param(40, 16, 4, 2, 128, id="w16_d2"),
    pytest.param(6, 64, 8, 4, 192, id="d4_n32"),
    pytest.param(48, 8, 4, 3, 64, id="w8"),
]


@pytest.mark.parametrize("B,W,A,D,K", SHAPES)
@pytest.mark.parametrize("row_order", [0, 1])
def test_qhead_envelope_equals_three_launch_chain_and_oracle(cuda, B, W, A, D, K, row_order):
    from morl_baselines_b200 import ops
    from oracle import oracle as orc

    assert ops.qhead_envelope_supported(ops.FMT_F16X2, B, W, A, D, K)
    o = _operands(cuda, B, W, A, D, K, seed=B + W + K)
    M, N = B * W, A * D
    # the chain the kernel replaces
    q_on, _ = ops.gemm_planes(o["a_on"], o["p_on"], N, bias=o["b_on"], a_scale=o["s_act"], b_scale=o["s_w_on"])
    q_tg, _ = ops.gemm_planes(o["a_tg"], o["p_tg"], N, bias=o["b_tg"], a_scale=o["s_act"], b_scale=o["s_w_tg"])
    for mode in (ops.DOT_UNFUSED, ops.DOT_FMA, ops.DOT_PAIRFMA):
        t_ref, p_ref, a_ref = ops.envelope_td(q_on.view(B, W, A, D), q_tg.view(B, W, A, D), o["wset"], o["rew"], o["done"], 0.99, mode, row_order)
        qo, qt = th.full((M, N), float("nan"), device=cuda), th.full((M, N), float("nan"), device=cuda)
        t, p, a = ops.qhead_envelope_td(o["a_on"], o["a_tg"], o["p_on"], o["p_tg"], o["b_on"], o["b_tg"], o["wset"], o["rew"], o["done"], 0.99, B, W, A, D,
                                        mode, row_order, a_scale_on=o["s_act"], a_scale_tg=o["s_act"], w_scale_on=o["s_w_on"], w_scale_tg=o["s_w_tg"],
                                        want_indices=True, q_on_out=qo, q_tg_out=qt, reverse_tiles=bool(mode & 1))
        th.cuda.synchronize()
        assert th.equal(qo, q_on) and th.equal(qt, q_tg), "Q tiles differ from the unfused output-layer GEMM"
        assert th.equal(p, p_ref) and th.equal(a, a_ref), f"indices differ from the standalone operator (mode {mode})"
        assert th.equal(t, t_ref), f"targets differ from the standalone operator (mode {mode})"
    # ... and the CPU oracle on the same Q tensors (contract arithmetic)
    to, po, ao = orc.envelope_td(q_on.view(B, W, A, D).cpu().numpy(), q_tg.view(B, W, A, D).cpu().numpy(), o["wset"].cpu().numpy(), o["rew"].cpu().numpy(),
                                 o["done"].cpu().numpy(), 0.99, row_order=row_order)
    t, p, a = ops.qhead_envelope_td(o["a_on"], o["a_tg"], o["p_on"], o["p_tg"], o["b_on"], o["b_tg"], o["wset"], o["rew"], o["done"], 0.99, B, W, A, D,
                                    ops.DOT_UNFUSED, row_order, a_scale_on=o["s_act"], a_scale_tg=o["s_act"], w_scale_on=o["s_w_on"], w_scale_tg=o["s_w_tg"],
                                    want_indices=True)
    assert np.array_equal(t.cpu().numpy(), to) and np.array_equal(p.cpu().numpy(), po) and np.array_equal(a.cpu().numpy(), ao)


def test_qhead_envelope_constant_q_takes_first_occurrence(cuda):
    """Zero activations: Q[b, j, a, :] = bias[a, :] for every j -- every weight ties across all 64 preference rows; the near-tie path must
    return the FIRST (j, a) like th.max(dim=2) then th.argmax(dim=1)."""
    from morl_baselines_b200 import ops

    B, W, A, D, K = 4, 64, 8, 3, 64
    o = _operands(cuda, B, W, A, D, K, seed=3, zero_act=True)
    q_on, _ = ops.gemm_planes(o["a_on"], o["p_on"], A * D, bias=o["b_on"], a_scale=o["s_act"], b_scale=o["s_w_on"])
    q_tg, _ = ops.gemm_planes(o["a_tg"], o["p_tg"], A * D, bias=o["b_tg"], a_scale=o["s_act"], b_scale=o["s_w_tg"])
    t_ref, p_ref, a_ref = ops.envelope_td(q_on.view(B, W, A, D), q_tg.view(B, W, A, D), o["wset"], o["rew"], o["done"], 0.99, ops.DOT_UNFUSED, 1)
    t, p, a = ops.qhead_envelope_td(o["a_on"], o["a_tg"], o["p_on"], o["p_tg"], o["b_on"], o["b_tg"], o["wset"], o["rew"], o["done"], 0.99, B, W, A, D,
                                    ops.DOT_UNFUSED, 1, a_scale_on=o["s_act"], a_scale_tg=o["s_act"], w_scale_on=o["s_w_on"], w_scale_tg=o["s_w_tg"],
                                    want_indices=True)
    assert int(p.max()) == 0, "ties over j must resolve to the first preference row"
    assert th.equal(p, p_ref) and th.equal(a, a_ref) and th.equal(t, t_ref)


def test_qhead_envelope_rejects_what_it_does_not_cover(cuda):
    from morl_baselines_b200 import _lib, ops

    assert not ops.qhead_envelope_supported(ops.FMT_BF16X3, 1024, 64, 8, 3, 256)
    assert not ops.qhead_envelope_supported(ops.FMT_F16X2, 1024, 48, 8, 3, 256)   # |W| does not divide 128
    assert not ops.qhead_envelope_supported(ops.FMT_F16X2, 3, 64, 8, 3, 256)      # B*W not a multiple of 128
    assert not ops.qhead_envelope_supported(ops.FMT_F16X2, 1024, 64, 16, 3, 256)  # A*D > 32
    o = _operands(cuda, 3, 64, 8, 3, 64, seed=1)
    with pytest.raises(_lib.MorlB200Error):
        ops.qhead_envelope_td(o["a_on"], o["a_tg"], o["p_on"], o["p_tg"], o["b_on"], o["b_tg"], o["wset"], o["rew"], o["done"], 0.99, 3, 64, 8, 3)


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
def test_envelope_update_with_fused_head_equals_update_without(cuda, graph):
    """Envelope.update() through the fused head == Envelope.update() through the three-launch chain, bit for bit (indices, loss,
    priorities, every parameter after 4 updates incl. a target sync)."""
    from morl_baselines_b200.multi_policy.envelope import envelope as env_mod
    from morl_baselines_b200.testing import FakeEnv, synthetic_store

    OBS, A, D, B, W = 12, 4, 3, 64, 8
    results = []
    for fused in (True, False):
        env_mod._FUSED_HEAD = fused
        try:
            th.manual_seed(5)
            np.random.seed(5)
            agent = env_mod.Envelope(FakeEnv(obs_dim=OBS, n_actions=A, reward_dim=D), batch_size=B, num_sample_w=W, per=True, buffer_size=2048,
                                     net_arch=[64, 64, 64], log=False, seed=5, device=cuda, use_cuda_graph=graph, target_net_update_freq=3)
            st = synthetic_store(1024, OBS, A, D, seed=2)
            rb = agent.replay_buffer
            rb.obs[:1024], rb.next_obs[:1024], rb.actions[:1024], rb.rewards[:1024], rb.dones[:1024] = st["obs"], st["next_obs"], st["actions"], st["rewards"], st["dones"]
            rb.size, rb.ptr = 1024, 0
            rb.mark_all_dirty()
            rb.tree.batch_set(np.arange(1024), np.linspace(0.1, 1.0, 1024))
            losses, prios = [], []
            for step in range(4):
                np.random.seed(20 + step)
                agent.global_step = step + 1
                agent.update()
                losses.append(float(agent._last_loss))
                prios.append((agent._last_inds.copy(), np.asarray(agent._last_priority).copy()))
            th.cuda.synchronize()
            results.append((losses, prios, [p.detach().cpu().numpy().copy() for p in agent.q_net.parameters()]))
        finally:
            env_mod._FUSED_HEAD = True
    (l1, p1, w1), (l0, p0, w0) = results
    assert l1 == l0
    for (i1, x), (i0, y) in zip(p1, p0):
        assert np.array_equal(i1, i0) and np.array_equal(x, y)
    for x, y in zip(w1, w0):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("M,N,K", [(65536, 24, 256), (8192, 18, 256), (256, 32, 64), (640, 5, 128)])
def test_narrow_head_gemm_equals_general_gemm(cuda, M, N, K):
    """morl_qhead_gemm_f32 (output layer with resident weight planes; the training pass's last layer) == morl_gemm_planes_f32, bit for bit,
    both tile orders."""
    from morl_baselines_b200 import ops

    fmt = ops.FMT_F16X2
    g = th.Generator(device=cuda).manual_seed(M + N)
    s_a, s_w = ops.scale_tensor(2.0, cuda), ops.scale_tensor(4096.0, cuda)
    a = ops.split_planes(th.randn(M, K, device=cuda, generator=g).relu_(), fmt, rows_pad=M, ldp=K, scale=s_a)
    w = ops.split_planes(th.randn(N, K, device=cuda, generator=g) / 16.0, fmt, rows_pad=32, ldp=K, scale=s_w)
    bias = th.randn(N, device=cuda, generator=g)
    assert ops.qhead_gemm_supported(fmt, M, N, K)
    ref, _ = ops.gemm_planes(a, w, N, bias=bias, a_scale=s_a, b_scale=s_w)
    for rev in (False, True):
        out = th.full((M, N), float("nan"), device=cuda)
        ops.qhead_gemm(a, w, N, bias, out=out, a_scale=s_a, w_scale=s_w, reverse_tiles=rev)
        assert th.equal(out, ref)
    assert not ops.qhead_gemm_supported(fmt, 100, N, K) and not ops.qhead_gemm_supported(fmt, M, 40, K)


def test_chained_passes_equal_per_layer_passes(cuda):
    """TCPairMlp forward / backward with the hidden layers as chained launches (forward chain, dX chain) == the per-layer launches, bit for
    bit: Q, every gradient tensor."""
    _chained_equals_per_layer(cuda, n_hidden=4)


def test_chained_backward_of_a_deep_net_equals_per_layer_passes(cuda):
    """Six weight-gradient products: more than one multi-job launch takes them (MN_MAX_JOBS per launch), still bit-identical."""
    from morl_baselines_b200 import _lib

    assert 6 > _lib.MN_MAX_JOBS
    _chained_equals_per_layer(cuda, n_hidden=6)


def _chained_equals_per_layer(cuda, n_hidden):
    from torch import nn

    from morl_baselines_b200 import ops, tc_mlp

    th.manual_seed(3)
    B, W, F, D, H, OUT = 64, 8, 12, 3, 256, 12
    layers = [nn.Linear(F + D, H), nn.ReLU()]  # (built in this order: the seeded weights of every layer stay those of n_hidden = 4)
    for _ in range(n_hidden - 1):
        layers += [nn.Linear(H, H), nn.ReLU()]
    net = nn.Sequential(*layers, nn.Linear(H, OUT)).to(cuda)
    feats, wset = th.randn(B, F, device=cuda), th.rand(W, D, device=cuda)
    dq = th.randn(B * W, OUT, device=cuda) * 1e-3
    results = []
    saved = (tc_mlp._CHAIN, tc_mlp._CHAIN_BWD)
    try:
        for chain in (False, True):
            tc_mlp._CHAIN, tc_mlp._CHAIN_BWD = chain, chain
            plan = tc_mlp.TCPairMlp(net, F, B, W, trainable=True)
            assert plan.chain_supported() == chain
            plan.refresh_weights()
            q = plan.forward_pairs(feats, wset).clone()
            grads = [g.clone() for g in plan.backward(feats, wset, dq)]
            th.cuda.synchronize()
            results.append((q, grads))
    finally:
        tc_mlp._CHAIN, tc_mlp._CHAIN_BWD = saved
    (q0, g0), (q1, g1) = results
    assert th.equal(q0, q1)
    for a, b in zip(g0, g1):
        assert th.equal(a, b)
