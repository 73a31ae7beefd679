"""Small launches of EVERY kernel of libmorl_b200.so for compute-sanitizer (SURVEY.md section 5):

    compute-sanitizer --tool memcheck|racecheck|synccheck|initcheck python scripts/sanitize_all.py [group ...]

groups: envelope td gemm optim pareto replay layer1 qhead dyna chain mn_multi (default: all).  Shapes are small (sanitizer slows kernels 10-100x) but exercise
every code path: all envelope kernel families, both GEMM operand formats x CTA modes x accumulator modes, MN split-K GEMM with the fused
column sums, every split / reduction helper, the loss kernels, Adam, polyak, Pareto + front records, replay gather."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch as th

from morl_baselines_b200 import ops

dev = th.device("cuda:0")
g = th.Generator(device=dev).manual_seed(0)
if os.environ.get("SAN_ZERO_PLANES") == "1":
    # initcheck does not see the writes of TMA bulk tensor STORES (cp.async.bulk.tensor ... global.shared::cta): plane tensors produced
    # by the GEMM epilogue then look uninitialised to later readers.  Pre-zeroing every plane allocation separates that tool artefact
    # from a genuine read of memory nobody wrote (profiles/r02_sanitize_initcheck*.txt).
    _empty = ops.empty_planes
    ops.empty_planes = lambda *a, **k: _empty(*a, **k).zero_()
groups = set(sys.argv[1:]) or {"envelope", "td", "gemm", "optim", "pareto", "replay", "layer1", "qhead", "dyna", "chain", "mn_multi"}


def rn(*s, scale=1.0):
    return th.randn(*s, device=dev, generator=g) * scale


if "envelope" in groups:
    for (B, W, A, D) in [(40, 64, 8, 3), (9, 48, 4, 2)]:
        q_on, q_tg, wset, rew, done = rn(B, W, A, D), rn(B, W, A, D), th.rand(W, D, device=dev, generator=g), rn(B, D), th.zeros(B, device=dev)
        ref = None
        for path in ("v1", "v3", "wp"):
            if path == "wp" and W <= 32:
                continue
            os.environ["MORL_ENVELOPE_PATH"] = path
            out = ops.envelope_td(q_on, q_tg, wset, rew, done, 0.99)
            th.cuda.synchronize()
            ref = ref or out
            assert all(th.equal(a, b) for a, b in zip(ref, out)), path
        os.environ.pop("MORL_ENVELOPE_PATH", None)
    print("envelope ok")

if "td" in groups:
    B, W, A, D = 24, 8, 4, 3
    q = rn(B * W, A, D)
    ops.greedy_td(q, rn(B * W, A, D), th.rand(W, D, device=dev, generator=g), rn(B, D), th.zeros(B, device=dev), 0.99, ops.DOT_UNFUSED, ops.MAP_TILE, ops.MAP_BLOCK)
    act = th.randint(0, A, (B,), device=dev, generator=g, dtype=th.int32)
    lam = th.full((1,), 0.3, device=dev)
    ops.td_mse_priority(q, act, rn(B * W, D), th.rand(W, D, device=dev, generator=g), 0.0, B, W, ops.ROWS_BMAJOR, lambda_dev=lam)
    qn = rn(2, B, A, D)
    ops.critic_min_td(qn, th.rand(B, D, device=dev, generator=g), rn(B, D), th.zeros(B, device=dev), 0.99)
    ops.gpi_envelope(rn(2, B, 5, A, D), th.rand(B, D, device=dev, generator=g))
    act2 = th.randint(0, A, (B // 2,), device=dev, generator=g, dtype=th.int32)
    ops.td_huber_priority(rn(2, B, A, D, scale=0.02), act2, rn(B, D, scale=0.02), rn(B, D, scale=0.02), th.rand(B, D, device=dev, generator=g), 0.01, B // 2)
    ops.actor_critic_td(rn(2, B, D), th.rand(D, device=dev, generator=g), rn(B, D), th.zeros(B, 1, device=dev), rn(B, 1), 0.2, 0.99, ops.AC_SCALAR_MIN)
    th.cuda.synchronize()
    print("td ok")

if "gemm" in groups:
    for fmt in (ops.FMT_F16X2, ops.FMT_BF16X3):
        sa = ops.scale_tensor(8.0, dev) if fmt == ops.FMT_F16X2 else None
        sw = ops.scale_tensor(512.0, dev) if fmt == ops.FMT_F16X2 else None
        for M in (100, 700):  # 1-CTA kernel / CTA-pair kernel with a ragged last tile
            a, b, bias = rn(M, 128), rn(64, 128, scale=1 / 8), rn(64)
            ap, bp = ops.split_planes(a, fmt, scale=sa), ops.split_planes(b, fmt, scale=sw)
            for split in (True, False):
                bits = ops.empty_relu_bits(M, dev)
                c, cp = ops.gemm_planes(ap, bp, 64, bias=bias, relu=True, out_f32=True, out_planes=True, a_scale=sa, b_scale=sw, c_scale=sa, split_acc=split,
                                        relu_bits_out=bits)
                ops.gemm_planes(ap, bp, 64, relu_mask=cp, out_f32=True, a_scale=sa, b_scale=sw, split_acc=split, reverse_tiles=True)
                ops.gemm_planes(ap, bp, 64, relu_bits_in=bits, out_f32=True, a_scale=sa, b_scale=sw, split_acc=split)
                ref = (a.double() @ b.double().t() + bias.double()).clamp_min(0)
                assert float((c.double() - ref).abs().max()) < 1e-4
                # the planes the TMA bulk store wrote hold the same values as the fp32 output of the same call: they WERE written, whatever
                # initcheck reports about later reads of them (it does not track cp.async.bulk.tensor stores; see DESIGN 5b)
                back = sum(cp[i].double() for i in range(cp.shape[0])) / (8.0 if sa is not None else 1.0)
                assert float((back - c.double()).abs().max()) <= 2.0**-20 * float(c.abs().max())
                assert bool(th.equal(ops.unpack_relu_bits(bits, 64), c > 0))
        G, H = rn(600, 24, scale=1e-3), rn(600, 128).relu_()
        sg = ops.scale_tensor(2.0**16, dev) if fmt == ops.FMT_F16X2 else None
        Gp, Hp = ops.split_planes(G, fmt, ldp=64, scale=sg), ops.split_planes(H, fmt, scale=sa)
        cs = th.empty(24, device=dev)
        dW = ops.gemm_planes_mn(Gp, 24, Hp, 128, colsum=cs, g_scale=sg, h_scale=sa)
        assert float((dW.double() - G.double().t() @ H.double()).abs().max()) < 1e-4
        ops.colsum_planes(Gp, 24, scale=sg)
        ops.pairs_grad_reduce(ops.split_planes(rn(6 * 5, 64), fmt, scale=sa), 6, 5, scale=sa)
        ops.pairs_grad_reduce(ops.split_planes(rn(3 * 70, 64), fmt, scale=sa), 3, 70, scale=sa)
        ops.pairs_relu_split(rn(6, 64), rn(5, 64), fmt=fmt, scale=sa, relu_bits_out=ops.empty_relu_bits(30, dev))
        w1, w2 = rn(64, 64, scale=0.1), rn(24, 64)
        o = [ops.empty_planes(fmt, 64, 64, dev), ops.empty_planes(fmt, 64, 64, dev), ops.empty_planes(fmt, 32, 64, dev)]
        s1, s2 = ops.scale_tensor(1.0, dev), ops.scale_tensor(1.0, dev)
        te = 14 if fmt == ops.FMT_F16X2 else None
        ops.split_planes_multi([(w1, o[0], False, s1, te), (w1, o[1], True, s1, te), (w2, o[2], False, s2, te)], fmt)
        ops.split_planes(rn(50, 13), fmt, ldp=32, scale=sa)
    out, ws = th.zeros(1, device=dev), th.zeros(2, device=dev, dtype=th.int32)
    ops.amax_scale(rn(5000, scale=1e-5), 9, out, ws)
    th.cuda.synchronize()
    assert ops.plane_overflow_count() == 0
    print("gemm ok")

if "layer1" in groups:
    feats, wset, W1, b1 = rn(37, 11), th.rand(5, 2, device=dev, generator=g), rn(64, 13), rn(64)
    u, v = ops.pair_layer1_uv(feats, wset, W1, b1)
    ops.pair_layer1_grad(rn(37, 64), rn(5, 64), feats, wset)
    th.cuda.synchronize()
    print("layer1 ok")

if "optim" in groups:
    from morl_baselines_b200.common.fused_adam import FusedClipAdam

    ps = [th.nn.Parameter(rn(64, 35)), th.nn.Parameter(rn(64))]
    opt = FusedClipAdam(ps, lr=1e-3)
    for _ in range(2):
        for p in ps:
            p.grad = th.randn_like(p)
        opt.step_fused(1.0)
    ts = [rn(64, 35), rn(64)]
    ops.PolyakPlan([p.data for p in ps], ts).run(0.5)
    th.cuda.synchronize()
    print("optim ok")

if "pareto" in groups:
    pts = th.randn(700, 3, device=dev, generator=g, dtype=th.float64)
    keep = ops.pareto_mask(pts, True, raw=True)
    ops.pareto_mask(pts.float(), False)
    rec = th.empty(1 + 64 * 3 + 2, dtype=th.float64, device=dev)
    ops.front_pack(pts, keep, 64, rec, th.ones(2, dtype=th.float64, device=dev))
    gathered = th.stack([rec, rec]).contiguous()
    ops.front_unpack(gathered, 2, 3, 64, 2, th.empty(128, 3, dtype=th.float64, device=dev), th.empty(2, 3, dtype=th.float64, device=dev))
    th.cuda.synchronize()
    print("pareto ok")

if "replay" in groups:
    N, B = 300, 32
    obs, nobs = rn(N, 7), rn(N, 7)
    act = th.randint(0, 4, (N, 1), device=dev, generator=g, dtype=th.uint8)
    rew, done = rn(N, 3), th.zeros(N, 1, device=dev)
    idx = th.randint(0, N, (B,), device=dev, generator=g)
    ops.replay_gather(obs, nobs, act, rew, done, idx)
    th.cuda.synchronize()
    print("replay ok")
if "qhead" in groups:
    # fused output layers + envelope + Bellman (csrc/qhead_envelope.cu): several tiles per CTA are not needed for the protocol (ring and
    # accumulator phases wrap within 5 tiles of one CTA when the grid is capped) -- MORL has no grid cap switch, so a shape with more tiles
    # than SMs (B*W/128 = 160) exercises the wrap, and a W = 32 shape the four-transitions-per-tile path with ragged N = 18 rows
    for (B, W, A, D, K) in [(320, 64, 8, 3, 64), (24, 32, 6, 3, 128)]:
        M, N = B * W, A * D
        s_a, s_w = ops.scale_tensor(2.0, dev), ops.scale_tensor(1024.0, dev)
        a_on = ops.split_planes(rn(M, K).relu_(), ops.FMT_F16X2, rows_pad=M, ldp=K, scale=s_a)
        a_tg = ops.split_planes(rn(M, K).relu_(), ops.FMT_F16X2, rows_pad=M, ldp=K, scale=s_a)
        p_on = ops.split_planes(rn(N, K, scale=0.1), ops.FMT_F16X2, rows_pad=32, ldp=K, scale=s_w)
        p_tg = ops.split_planes(rn(N, K, scale=0.1), ops.FMT_F16X2, rows_pad=32, ldp=K, scale=s_w)
        b_on, b_tg, wset, rew, done = rn(N), rn(N), th.rand(W, D, device=dev, generator=g), rn(B, D), th.zeros(B, device=dev)
        q1, _ = ops.gemm_planes(a_on, p_on, N, bias=b_on, a_scale=s_a, b_scale=s_w)
        q2, _ = ops.gemm_planes(a_tg, p_tg, N, bias=b_tg, a_scale=s_a, b_scale=s_w)
        ref = ops.envelope_td(q1.view(B, W, A, D), q2.view(B, W, A, D), wset, rew, done, 0.99)
        qo, qt = th.zeros(M, N, device=dev), th.zeros(M, N, device=dev)
        out = ops.qhead_envelope_td(a_on, a_tg, p_on, p_tg, b_on, b_tg, wset, rew, done, 0.99, B, W, A, D, a_scale_on=s_a, a_scale_tg=s_a, w_scale_on=s_w,
                                    w_scale_tg=s_w, want_indices=True, q_on_out=qo, q_tg_out=qt)
        th.cuda.synchronize()
        assert th.equal(qo, q1) and th.equal(qt, q2) and all(th.equal(x, y) for x, y in zip(out, ref)), (B, W, A, D, K)
    print("qhead ok")

if "dyna" in groups:
    E, N, O = 5, 77, 35
    raw = rn(E, N, 2 * O, scale=3.0)
    idx = th.randint(0, E, (N,), device=dev, generator=g, dtype=th.int32)
    smp, var, unc = ops.ensemble_sample(raw, th.zeros(O, device=dev), th.full((O,), -5.0, device=dev), idx, rn(E, N, O), rn(N, O - 3), 3)
    th.cuda.synchronize()
    assert bool(th.isfinite(smp).all()) and bool((var > 0).all()) and bool((unc > 0).all())
    print("dyna ok")
if "chain" in groups:
    # chained hidden layers (gemm_chain_kernel): 2 chains x 2 layers on 5 tiles (groups of 2 + a ragged last group), then a 1-chain dX chain with masks
    M, H = 1200, 256
    sa, sw = ops.scale_tensor(2.0, dev), ops.scale_tensor(1024.0, dev)
    acts, ws, bs, sws, bits = [], [], [], [], []
    for c in range(2):
        acts.append([ops.split_planes(rn(M, H).relu_(), ops.FMT_F16X2, rows_pad=M, ldp=H, scale=sa)] + [ops.empty_planes(ops.FMT_F16X2, M, H, dev) for _ in range(2)])
        ws.append([ops.split_planes(rn(H, H, scale=0.06), ops.FMT_F16X2, rows_pad=H, ldp=H, scale=sw) for _ in range(2)])
        bs.append([rn(H, scale=0.1) for _ in range(2)])
        sws.append([sw, sw])
        bits.append([ops.empty_relu_bits(M, dev) for _ in range(2)])
    ops.GemmChain(acts, ws, bs, sws, bits, act_scale=sa)()
    for c in range(2):
        a = acts[c][0]
        for l in range(2):
            _, a = ops.gemm_planes(a, ws[c][l], H, bias=bs[c][l], relu=True, out_f32=False, out_planes=True, a_scale=sa, b_scale=sw, c_scale=sa)
            assert th.equal(a.view(th.int16), acts[c][l + 1].view(th.int16)), (c, l)
    gb = [acts[0][2]] + [ops.empty_planes(ops.FMT_F16X2, M, H, dev) for _ in range(2)]
    ops.GemmChain([gb], [ws[0]], None, [sws[0]], None, act_scale=sa, relu=False, bits_in=[bits[0]])()
    th.cuda.synchronize()
    print("chain ok")
if "mn_multi" in groups:
    # multi-job weight-gradient launch (gemm_planes_mn_multi_kernel + reduce_partials_vec4_multi_kernel): 220 units on at most 148 CTAs, so
    # CTAs take several units (ring and accumulator phases wrap across units of different jobs); a 24-wide job with trimmed partial rows
    M = 6000
    for fmt in (ops.FMT_F16X2, ops.FMT_BF16X3):
        sg = ops.scale_tensor(2.0**16, dev) if fmt == ops.FMT_F16X2 else None
        sa = ops.scale_tensor(2.0, dev) if fmt == ops.FMT_F16X2 else None
        jobs, ref = [], []
        for gc, hc, ldg, colsum in ((256, 128, 256, True), (24, 128, 64, True), (64, 64, 64, False)):
            Gp = ops.split_planes(rn(M, gc, scale=1e-3), fmt, ldp=ldg, scale=sg)
            Hp = ops.split_planes(rn(M, hc).relu_(), fmt, scale=sa)
            cs = th.empty(gc, device=dev) if colsum else None
            ref.append((ops.gemm_planes_mn(Gp, gc, Hp, hc, colsum=cs, g_scale=sg, h_scale=sa), cs))
            jobs.append((Gp, gc, Hp, hc, th.empty(gc, hc, device=dev), th.empty(gc, device=dev) if colsum else None, sg, sa))
        ops.GemmMnMulti(jobs)()
        th.cuda.synchronize()
        for (dW, cs), j in zip(ref, jobs):
            assert th.equal(j[4], dW) and (cs is None or th.equal(j[5], cs))
    print("mn_multi ok")
print("sanitize run ok")
