"""bench.py -- Envelope-Q gradient updates/sec on synthetic transitions (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one gradient update of Envelope Q-learning (reference envelope.py:269-334, gradient_updates=1) at
obs_dim=32, |A|=8, d_obj=3, |W|=64, batch=1024, net 4x256: replay gather -> Q on the B*|W| = 65,536 distinct rows (online +
target, no grad) -> fused envelope-TD target -> online forward on 65,536 rows -> fused TD loss/priorities -> backward ->
grad clip -> Adam (+ target sync every 200 steps).

  value  : updates/s of the FULL update (SURVEY 8(d): PER sample, targets, forward/backward, optimiser, priority write-back) through
           Envelope.update() with the replay store resident in HBM (per step 9 KB of indices + weights in, 4 KB of priorities + loss out).
  e2e    : updates/s through the same call with a HOST-resident replay buffer: per step the gathered minibatch (pinned, 283 KB) crosses
           host->device and the priorities + loss come back device->host; the loss is read as a python float every update.
  roofline     : the dominant kernel of the step -- the chained hidden-layer launch (layers 2..4 of both Q-networks, 6 f16x2 tcgen05 products in
                 one persistent kernel) -- against its binding roofline, the measured dense 16-bit tensor peak (HBM view inside);
                 roofline_gemm_layer: the per-layer kernel it replaces.
  roofline_envelope : the fused envelope-TD kernel north_star names, in the form the update runs it (output layers of both nets + envelope
                 operator + Bellman line in one kernel, Q never in HBM), against the measured HBM bandwidth, timed alone in a CUDA graph on
                 rotating buffer sets larger than L2; roofline_envelope_operator: the standalone operator on Q tensors in HBM.
  cpu_baseline : the reference's CPU implementation (oracle port, or the unmodified reference when mounted) at the SAME full config,
                 a bounded NUMBER of updates (not a bounded batch); cpu_dedup_restatement: the de-duplicated CPU restatement for context.
N > 1: every rank runs an independent update stream (weak scaling, no data-path collective); the ranks exchange their non-dominated
fronts with ONE NCCL all-gather per evaluation round, which is timed separately (config.ms_eval_round_*), not inside the updates.

--dump-outputs DIR (envelope workload): after the timed updates, rank 0 writes what the last update of each arm handed its caller -- loss,
sampled replay indices, written-back priorities and the updated online Q-network -- as DIR/<name>.npy (float32 / float64; `e2e.` prefix for
the host-replay arm).  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OBS, A, D, W, B, STORE = 32, 8, 3, 64, 1024, 65536
NET = [256, 256, 256, 256]
METRIC = "envelope_q_updates_per_sec"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index=0, period=0.1):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.stop_flag = [], set(), False
        self.max_mhz = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def _fill_store(rb, store):
    n = len(store["obs"])
    rb.obs[:n], rb.next_obs[:n], rb.actions[:n] = store["obs"], store["next_obs"], store["actions"]
    rb.rewards[:n], rb.dones[:n] = store["rewards"], store["dones"]
    rb.size, rb.ptr = n, 0
    rb.mark_all_dirty()
    if hasattr(rb, "tree"):
        rb.tree.batch_set(np.arange(n), np.full(n, rb.min_priority))


def _make_agent(dev, seed, on_device):
    from morl_baselines_b200.multi_policy.envelope.envelope import Envelope
    from morl_baselines_b200.testing import FakeEnv  # spaces-only stand-in for a mo-gymnasium env (rollouts are not part of the metric)

    env = FakeEnv(obs_dim=OBS, n_actions=A, reward_dim=D)
    return Envelope(env, batch_size=B, num_sample_w=W, per=True, buffer_size=STORE, net_arch=NET, log=False, seed=seed, device=dev,
                    replay_on_device=on_device)


def _last_update_outputs(agent, prefix=""):
    """What Envelope.update() hands its caller after its last gradient step, as host arrays: the critic loss, the replay indices it sampled
    (float64: exact), the priorities it wrote back and the updated online Q-network."""
    out = {prefix + "loss": np.array([agent.last_loss_host()], np.float32), prefix + "indices": np.asarray(agent._last_inds, np.float64),
           prefix + "priorities": np.asarray(agent._last_priority, np.float32)}
    for name, p in agent.q_net.named_parameters():
        out[f"{prefix}q_net.{name}"] = p.detach().float().cpu().numpy()
    return out


def _dump_outputs(path, arrays):
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "dumped outputs exceed 64 MB"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


def time_envelope_kernel(dev, replays=25):
    """Average launch duration of morl_envelope_td_f32 at the north-star shape: 16 launches on 16 rotating input sets
    (16 x 13.4 MB = 214 MB > 126 MB L2, so every launch streams its Q tensors from HBM) captured in ONE CUDA graph -- the way the
    update issues it -- and the graph replayed `replays` times between two CUDA events on the launching stream.  (A python launch
    loop measures the host's ctypes call, ~12 us, not the kernel.)"""
    import torch as th

    from morl_baselines_b200 import ops

    nsets = 16
    g = th.Generator(device=dev).manual_seed(1)
    sets = []
    for _ in range(nsets):
        q_on = th.randn(B, W, A, D, device=dev, generator=g)
        q_tg = q_on + 0.05 * th.randn(B, W, A, D, device=dev, generator=g)
        wset = th.rand(W, D, device=dev, generator=g)
        wset = wset / wset.sum(1, keepdim=True)
        sets.append((q_on, q_tg, wset, th.randn(B, D, device=dev, generator=g), (th.rand(B, device=dev, generator=g) < 0.02).float()))
    out = th.empty(W * B, D, device=dev)

    def sweep():
        for i in range(nsets):
            ops.envelope_td(*sets[i], 0.99, ops.DOT_UNFUSED, ops.ROWS_BMAJOR, want_indices=False, out=out)

    side = th.cuda.Stream()
    side.wait_stream(th.cuda.current_stream())
    with th.cuda.stream(side):
        sweep()
        sweep()
    th.cuda.current_stream().wait_stream(side)
    graph = th.cuda.CUDAGraph()
    with th.cuda.graph(graph):
        sweep()
    for _ in range(3):
        graph.replay()
    th.cuda.synchronize()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    th.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / (replays * nsets)


def time_qhead_kernel(dev, replays=12):
    """Average launch duration of morl_qhead_envelope_td_f32 -- output layers of both Q-nets + envelope operator + Bellman line in ONE
    kernel, the form the update uses -- at the north-star shape: 8 launches on 4 rotating pairs of activation-plane tensors
    (4 x 2 x 67 MB > L2) captured in one CUDA graph, CUDA events around the replays."""
    import torch as th

    from morl_baselines_b200 import ops

    fmt, K, M, N = ops.FMT_F16X2, NET[-1], B * W, A * D
    g = th.Generator(device=dev).manual_seed(3)
    s_act, s_w = ops.scale_tensor(2.0, dev), ops.scale_tensor(4096.0, dev)
    nsets = 4
    a_on = [ops.split_planes(th.randn(M, K, device=dev, generator=g).relu_(), fmt, rows_pad=M, ldp=K, scale=s_act) for _ in range(nsets)]
    a_tg = [ops.split_planes(th.randn(M, K, device=dev, generator=g).relu_(), fmt, rows_pad=M, ldp=K, scale=s_act) for _ in range(nsets)]
    p_on = ops.split_planes(th.randn(N, K, device=dev, generator=g) / 16, fmt, rows_pad=32, ldp=K, scale=s_w)
    p_tg = ops.split_planes(th.randn(N, K, device=dev, generator=g) / 16, fmt, rows_pad=32, ldp=K, scale=s_w)
    b_on, b_tg = th.randn(N, device=dev, generator=g), th.randn(N, device=dev, generator=g)
    wset = th.rand(W, D, device=dev, generator=g)
    wset = wset / wset.sum(1, keepdim=True)
    rew, done = th.randn(B, D, device=dev, generator=g), (th.rand(B, device=dev, generator=g) < 0.02).float()
    out = th.empty(W * B, D, device=dev)

    def sweep():
        for r in range(2):
            for i in range(nsets):
                ops.qhead_envelope_td(a_on[i], a_tg[i], p_on, p_tg, b_on, b_tg, wset, rew, done, 0.99, B, W, A, D, ops.DOT_UNFUSED, ops.ROWS_BMAJOR,
                                      a_scale_on=s_act, a_scale_tg=s_act, w_scale_on=s_w, w_scale_tg=s_w, out=out)

    side = th.cuda.Stream()
    side.wait_stream(th.cuda.current_stream())
    with th.cuda.stream(side):
        sweep()
    th.cuda.current_stream().wait_stream(side)
    graph = th.cuda.CUDAGraph()
    with th.cuda.graph(graph):
        sweep()
    for _ in range(3):
        graph.replay()
    th.cuda.synchronize()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    th.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / (replays * 2 * nsets)


def time_chain_kernel(dev, replays=10):
    """Average launch duration of the dominant kernel of the step, morl_gemm_chain_f32 in the form the two no-grad passes use it: hidden layers
    2..4 of BOTH networks (2 chains x 3 layers of 65,536 x 256 x 256, bias + ReLU + plane re-split epilogue) in ONE persistent launch.  4 launches
    on 2 rotating sets of activation buffers (2 x 8 x 67 MB, far above L2) captured in one CUDA graph, CUDA events around the replays."""
    import torch as th

    from morl_baselines_b200 import ops

    fmt, M, H, L = ops.FMT_F16X2, B * W, NET[0], len(NET) - 1
    g = th.Generator(device=dev).manual_seed(4)
    sa = ops.scale_tensor(2.0, dev)
    sets = []
    for _ in range(2):
        acts, ws, bs, sws = [], [], [], []
        for c in range(2):
            a0 = ops.split_planes(th.randn(M, H, device=dev, generator=g).relu_(), fmt, rows_pad=M, ldp=H, scale=sa)
            acts.append([a0] + [ops.empty_planes(fmt, M, H, dev) for _ in range(L)])
            sw = [ops.scale_tensor(2048.0, dev) for _ in range(L)]
            ws.append([ops.split_planes(th.randn(H, H, device=dev, generator=g) / 16.0, fmt, rows_pad=H, ldp=H, scale=sw[l]) for l in range(L)])
            bs.append([th.randn(H, device=dev, generator=g) * 0.1 for _ in range(L)])
            sws.append(sw)
        sets.append(ops.GemmChain(acts, ws, bs, sws, None, act_scale=sa))

    def sweep():
        for _ in range(2):
            for ch in sets:
                ch()

    side = th.cuda.Stream()
    side.wait_stream(th.cuda.current_stream())
    with th.cuda.stream(side):
        sweep()
    th.cuda.current_stream().wait_stream(side)
    graph = th.cuda.CUDAGraph()
    with th.cuda.graph(graph):
        sweep()
    for _ in range(2):
        graph.replay()
    th.cuda.synchronize()
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    th.cuda.synchronize()
    t = e0.elapsed_time(e1) * 1e-3 / (replays * 4)
    n_prod = 2 * L
    return t, n_prod, 3 * 2 * M * H * H * n_prod, (2 + n_prod) * 4 * M * H + n_prod * 4 * H * H  # s, layer products, MMA flops issued, algorithmic bytes


def time_gemm_kernel(dev, iters=200, fmt=None):
    """Average launch duration of the dominant kernel of the step, morl_gemm_planes_f32 on one hidden layer of the pair batch
    (65,536 x 256 x 256, bias + ReLU + plane re-split epilogue), CUDA events around graph replays, 4 rotating activation sets (> L2).  Returns
    (seconds per launch, tensor-core flops issued per launch, MMAs per fp32 product, bytes per element)."""
    import torch as th

    from morl_baselines_b200 import ops

    fmt = ops.FMT_F16X2 if fmt is None else fmt
    nprod, bpe = (3, 4) if fmt == ops.FMT_F16X2 else (6, 6)
    sa = ops.scale_tensor(8.0, dev) if fmt == ops.FMT_F16X2 else None
    sw = ops.scale_tensor(2048.0, dev) if fmt == ops.FMT_F16X2 else None
    M, H = B * W, NET[0]
    g = th.Generator(device=dev).manual_seed(2)
    wp = ops.split_planes(th.randn(H, H, device=dev, generator=g) / 16.0, fmt, rows_pad=H, ldp=H, scale=sw)
    bias = th.randn(H, device=dev, generator=g) * 0.1
    a_sets = [ops.split_planes(th.randn(M, H, device=dev, generator=g).relu_(), fmt, rows_pad=M, ldp=H, scale=sa) for _ in range(4)]
    c_sets = [th.empty_like(a_sets[0]) for _ in range(4)]

    def launch(i):
        ops.gemm_planes(a_sets[i % 4], wp, H, bias=bias, relu=True, out_f32=False, out_planes=True, c_planes=c_sets[i % 4], a_scale=sa, b_scale=sw,
                        c_scale=sa)

    # 16 launches captured in ONE CUDA graph -- the way the update issues them; a python launch loop measures the host (4 tensor-map
    # encodes + the ctypes call, ~30 us) once the kernel is faster than that
    per_graph = 16
    side = th.cuda.Stream()
    side.wait_stream(th.cuda.current_stream())
    with th.cuda.stream(side):
        for i in range(8):
            launch(i)
    th.cuda.current_stream().wait_stream(side)
    graph = th.cuda.CUDAGraph()
    with th.cuda.graph(graph):
        for i in range(per_graph):
            launch(i)
    for _ in range(3):
        graph.replay()
    th.cuda.synchronize()
    replays = max(1, iters // per_graph)
    iters = replays * per_graph
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        graph.replay()
    e1.record()
    th.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / iters, nprod * 2 * M * H * H, nprod, bpe


def _cpu_info():
    model = "unknown"
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:  # cgroup v2 CPU quota: the affinity mask can be wider than what the container may actually use
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = max(1, int(float(q) / float(per)))
    except (OSError, ValueError):
        pass
    return model, avail, quota


def _pick_cpu_threads():
    """Thread count for the CPU arm: probe {32, 64, all usable cores} once on the arm's dominant operation (a Linear + ReLU on 262,144
    rows, ~35 GFLOP per call) and keep the fastest.  `all` comes from the affinity mask / cgroup quota, not os.cpu_count()."""
    import torch as th

    model, avail, quota = _cpu_info()
    usable = min(avail, quota) if quota else avail
    cands = sorted({c for c in (32, 64, usable) if 1 <= c <= usable} or {usable})
    x = th.randn(262144, 256)
    lin = th.nn.Linear(256, 256)
    best, probe = None, {}
    with th.no_grad():
        for c in cands:
            th.set_num_threads(c)
            th.relu(lin(x))
            t0 = time.perf_counter()
            for _ in range(3):
                th.relu(lin(x))
            probe[c] = (time.perf_counter() - t0) / 3
            if best is None or probe[c] < probe[best]:
                best = c
    th.set_num_threads(best)
    return best, {"cpu_model": model, "cores_affinity": avail, "cores_cgroup_quota": quota, "cores_os": os.cpu_count(),
                  "thread_probe_s": {str(k): round(v, 4) for k, v in probe.items()}}


def cpu_reference_arm(max_steps, warmup, budget_s, dedup=False):
    """Time the reference's CPU update at the FULL metric configuration (B = 1024 transitions, |W| = 64, net 4x256, per=True: both Q-nets
    run on B*|W|^2 = 4,194,304 rows, ~3.6 TFLOP and ~11 GB per update) -- no batch sub-sampling, no scaling.  The unmodified reference
    when /root/reference is mounted (kind "reference"), else its PyTorch-CPU port (kind "port", oracle/envelope_update_port.py, pinned
    bit-for-bit to the reference by tests/test_port_vs_reference.py).  `dedup=True` times the de-duplicated restatement instead
    (B*|W| rows; NOT the reference's code path, reported for context only).  The number of timed steps is bounded by `budget_s`
    (at least 1); the per-step times are returned so the caller can report the median."""
    import torch as th

    from oracle import ref_harness as rh
    from oracle.envelope_update_port import EnvelopeUpdatePort
    from morl_baselines_b200.testing import synthetic_store

    threads, info = _pick_cpu_threads()
    n_store = 16384
    store = synthetic_store(n_store, OBS, A, D, seed=0)
    rng = np.random.default_rng(0)
    if rh.reference_available() and not dedup:
        kind = "reference"
        envm = rh.import_reference("morl_baselines.multi_policy.envelope.envelope")
        agent = envm.Envelope(rh.FakeEnv(obs_dim=OBS, n_actions=A, reward_dim=D), batch_size=B, num_sample_w=W, per=True,
                              buffer_size=n_store, net_arch=NET, log=False, seed=0, device="cpu")
        rb = agent.replay_buffer
        rb.obs[:n_store], rb.next_obs[:n_store], rb.actions[:n_store], rb.rewards[:n_store], rb.dones[:n_store] = (
            store[k] for k in ("obs", "next_obs", "actions", "rewards", "dones"))
        rb.size, rb.ptr = n_store, 0
        rb.tree.batch_set(np.arange(n_store), np.full(n_store, rb.min_priority))
        agent.global_step = 1
        step = agent.update
    else:
        kind = "dedup-restatement" if dedup else "port"
        port = EnvelopeUpdatePort(OBS, A, D, NET, seed=0)

        def step():
            idx = rng.integers(0, n_store, size=B)
            wset = np.abs(rng.standard_normal((W, D)))
            wset = th.from_numpy((wset / wset.sum(1, keepdims=True)).astype(np.float32))
            port.update(th.from_numpy(store["obs"][idx]), th.from_numpy(store["actions"][idx]), th.from_numpy(store["rewards"][idx]),
                        th.from_numpy(store["next_obs"][idx]), th.from_numpy(store["dones"][idx]), wset, dedup=dedup)

    t_begin = time.perf_counter()
    t_warm = []
    for _ in range(warmup):
        t0 = time.perf_counter()
        step()
        t_warm.append(time.perf_counter() - t0)
    est = min(t_warm) if t_warm else None
    times = []
    while len(times) < max_steps:
        if times or est is not None:
            nxt = np.median(times) if times else est
            if times and (time.perf_counter() - t_begin) + nxt > budget_s:
                break
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    return times, kind, threads, info


def run_reference_arm(args, rank):
    """`--impl reference`: the reference's own CPU implementation of the update on this box's host cores, SAME config as the B200 arm
    (full batch, full weight set).  Warm-up is capped at one full update and the number of timed updates by a wall-clock budget
    (MORL_CPU_BUDGET_S, default 240 s) -- `steps` in the line is the number actually timed, `steps_requested` what was asked for."""
    if rank != 0:
        return
    budget = float(os.environ.get("MORL_CPU_BUDGET_S", "240"))
    times, kind, threads, info = cpu_reference_arm(max_steps=args.steps, warmup=min(args.warmup, 1), budget_s=budget)
    t_med = float(np.median(times))
    value = 1.0 / t_med
    sample = (f"FULL config, no sub-sampling: batch {B} x |W|={W} (B*|W|^2 = {B * W * W} net rows per Q-net per update), "
              f"{len(times)} timed updates after 1 warm-up, median; {threads} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "updates/s", "n_gpus": args.gpus, "steps": len(times),
        "steps_requested": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": t_med * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"Envelope-Q gradient update obs={OBS} |A|={A} d={D} |W|={W} batch={B} net=4x256 per=True (CPU, full config)",
                   "step_seconds": [round(t, 3) for t in times], "host": info},
        "cpu_baseline": {"value": value, "unit": "updates/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_b200(args, rank, local_rank, world):
    import torch as th
    import torch.distributed as dist

    from morl_baselines_b200 import ops
    from morl_baselines_b200.parallel import allgather_fronts
    from morl_baselines_b200.testing import synthetic_store

    dev = th.device("cuda", local_rank)
    th.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, args.warmup
    store = synthetic_store(STORE, OBS, A, D, seed=0)
    np.random.seed(1000 + rank)
    th.manual_seed(rank)  # network initialisation: torch's default generator is not seeded reproducibly

    # ---------------- `value`: the full update of SURVEY 8(d) -- PER sample + targets + forward/backward + optimiser + priority write-back --
    # through the public API with the replay store RESIDENT IN HBM: per step the host walks the sum-tree, 9 KB of indices + weights go
    # host->device, one graph replay, 4 KB of priorities + loss come back and are written into the tree (overlapped with backward + Adam)
    agent = _make_agent(dev, seed=rank, on_device=True)
    _fill_store(agent.replay_buffer, store)
    agent.replay_buffer.flush()
    agent.global_step = 1
    s = agent._ensure_static()
    for _ in range(max(Wm, 3)):
        agent.update()
    launches_per_step = agent.launches_per_step

    # one evaluation round: local non-dominated front of this rank's policy set -> ONE all-gather -> global prune, all stream-ordered
    from morl_baselines_b200.tc_mlp import TCPairMlp

    ev_plan = TCPairMlp(agent.q_net.net, agent.q_net.feat_dim, 256, W, share_weights_with=agent._tc_on)
    ev_w = s["wset"].repeat(256, 1)
    ev_vals64 = th.empty((256 * W, D), dtype=th.float64, device=dev)

    def eval_round():
        with th.no_grad():
            ev = agent.replay_buffer.device_stores()[0][:256]
            q = ev_plan.forward_pairs(ev, s["wset"])  # [256 * W, A * D] on the tensor cores (weight planes of the last update)
            vals, _, _ = ops.gpi_envelope(q.view(1, 256 * W, 1, A, D), ev_w)
            ev_vals64.copy_(vals)
        return allgather_fronts(ev_vals64, cap=512)

    eval_round()  # untimed warm-up of the evaluation round
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ops.launch_count
    e0, em, e1 = (th.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    for _ in range(K):
        agent.update()
    em.record()
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    ms_steps = e0.elapsed_time(em)
    clocks = sampler.result()
    outputs = _last_update_outputs(agent) if args.dump_outputs and rank == 0 else None
    gpu_launches = (ops.launch_count - launches0) + launches_per_step * K
    # the evaluation round, timed on its own (it is NOT part of an update): 3 rounds, the last one reported
    for _ in range(3):
        em.record()
        global_front = eval_round()
        e1.record()
        th.cuda.synchronize()
    ms_eval = em.elapsed_time(e1)
    t_ms = th.tensor([ms_steps, ms_eval], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms, ms_eval_max = float(t_ms[0]), float(t_ms[1])
    value = world * K / (ms * 1e-3)
    loss_dev = agent.last_loss_host()
    h2d_value = B * 8 + 16 + W * D * 4
    del ev_plan

    # ---------------- end-to-end arm (`e2e`): public API, host replay + host PER tree ------------------------------
    agent_h = _make_agent(dev, seed=rank, on_device=False)
    _fill_store(agent_h.replay_buffer, store)
    agent_h.global_step = 1
    loss_host = 0.0
    for _ in range(max(Wm, 3)):
        agent_h.update()
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    e2, e3 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(K):
        agent_h.update()  # H2D minibatch + weights, graph replay, D2H priorities + loss (event sync) -> host sum-tree
        loss_host = agent_h.last_loss_host()  # the reference reads critic_loss.item() every update (envelope.py:327): a python float here too
    e3.record()
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    t2 = th.tensor([e2.elapsed_time(e3)], device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * K / (float(t2.item()) * 1e-3)
    h2d = B * (OBS * 4 * 2 + 4 + D * 4 + 4) + W * D * 4
    d2h = B * 4 + 4
    if args.dump_outputs and rank == 0:
        outputs.update(_last_update_outputs(agent_h, "e2e."))
        _dump_outputs(args.dump_outputs, outputs)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the fused envelope-TD kernel (rank 0) ------------------------------------------
    hbm_peak, bf16_peak, peak_src = _peaks()
    t_kernel = time_envelope_kernel(dev)
    t_gemm, gemm_flops, gemm_nprod, gemm_bpe = time_gemm_kernel(dev)
    alg_bytes = 2 * B * W * A * D * 4 + W * D * 4 + B * D * 4 + B * 4 + W * B * D * 4  # SURVEY.md 8(d): 13,386,496 B
    achieved = alg_bytes / t_kernel / 1e9
    traffic = gemm_traffic = None
    tpath = os.path.join(ROOT, "profiles", "envelope_td_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):
        gemm_traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    gemm_alg_bytes = 2 * gemm_bpe * B * W * NET[0] + gemm_bpe * NET[0] * NET[0]  # A planes read + C planes written + weight planes
    # fused output layers + envelope + Bellman (the form Envelope.update uses when the shape is inside the kernel): the last hidden
    # activation planes of both nets are its HBM input (the Q tensors never exist in HBM), plus the small operands and the targets
    fused = None
    from morl_baselines_b200 import ops as _ops

    if agent.tensor_core_format == "f16x2" and _ops.qhead_envelope_supported(_ops.FMT_F16X2, B, W, A, D, NET[-1]):
        t_fused = time_qhead_kernel(dev)
        fused_bytes = 2 * 4 * B * W * NET[-1] + 2 * 4 * 32 * NET[-1] + W * D * 4 + B * D * 4 + B * 4 + W * B * D * 4
        tf = os.path.join(ROOT, "profiles", "qhead_envelope_traffic.json")
        fused = {"bound": "hbm", "kernel": "qhead_envelope_kernel<f16x2, 3, UNFUSED> (output layers of both Q-nets 65536x24x256 on tcgen05 + envelope "
                                           "operator + Bellman line; Q tiles in tensor / shared memory only)",
                 "achieved": fused_bytes / t_fused / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": fused_bytes / t_fused / 1e9 / hbm_peak,
                 "traffic": json.load(open(tf)).get("dram_bytes_per_launch") if os.path.exists(tf) else None, "algorithmic_bytes": fused_bytes,
                 "us_per_launch": t_fused * 1e6, "peak_source": peak_src, "in_update": bool(getattr(agent, "fused_head_active", False)),
                 "replaces": "2 x morl_gemm_planes_f32 (N = 24) + morl_envelope_td_f32",
                 "timing": "8 launches on 4 rotating pairs of activation-plane tensors (4 x 2 x 67 MB > L2) in one CUDA graph, 12 replays, CUDA events"}
    mlp_flops = 5 * B * W * 211712 * 2  # SURVEY.md 8(d): 1.39e11 FLOP/update (2 no-grad fwd + fwd + 2x bwd)
    standalone_env = {"bound": "hbm", "kernel": "envelope_td_wp_kernel<3,UNFUSED> (morl_envelope_td_f32 alone: Q_on / Q_tg read from HBM)", "achieved": achieved,
                      "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic, "algorithmic_bytes": alg_bytes,
                      "us_per_launch": t_kernel * 1e6, "peak_source": peak_src,
                      "timing": "16 launches on rotating input sets (214 MB > L2) in one CUDA graph, 25 replays, CUDA events"}
    gemm_layer = {"kernel": "gemm_planes_kernel<pair, f16x2> (ONE hidden layer 65536x256x256 per launch: the per-layer form the chained launch replaces)",
                  "us_per_launch": t_gemm * 1e6, "hbm_frac": gemm_alg_bytes / t_gemm / 1e9 / hbm_peak, "tensor_frac": gemm_flops / t_gemm / 1e12 / bf16_peak}
    chain_roofline = None
    if agent.tensor_core_format == "f16x2" and _ops.gemm_chain_supported(_ops.FMT_F16X2, B * W, NET[0]) and os.environ.get("MORL_GEMM_CHAIN", "1") == "1":
        t_ch, n_prod, ch_flops, ch_bytes = time_chain_kernel(dev)
        # dominant kernel of the step: the chained hidden layers (3 launches per update, ~45 % of it).  Floors of the 6-product launch: tensor pipe
        # 6 x 3 x 8.6 GFLOP / 1687 TFLOP/s = 91.6 us, HBM (2 inputs read + 6 outputs written, intermediates re-read from L2) 537 MB / 6.48 TB/s
        # = 82.9 us -> the binding roofline is the tensor pipe; the HBM view is reported next to it
        chain_roofline = {"bound": "tensor", "kernel": f"gemm_chain_kernel<f16x2> (hidden layers 2..4 of both Q-networks, {n_prod} products 65536x256x256 in ONE persistent "
                                                       "launch, 3 fp16 tcgen05 MMAs per fp32 product, CTA pairs, bias + ReLU + re-split epilogue, intermediates re-read from L2)",
                          "achieved": ch_flops / t_ch / 1e12, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ch_flops / t_ch / 1e12 / bf16_peak,
                          "traffic": None, "algorithmic_flops": ch_flops // 3, "algorithmic_tflops": ch_flops / 3 / t_ch / 1e12,
                          "fp32_accurate_peak_tflops": bf16_peak / 3, "us_per_launch": t_ch * 1e6, "us_per_layer_product": t_ch * 1e6 / n_prod,
                          "peak_source": peak_src,
                          "hbm": {"algorithmic_bytes": ch_bytes, "achieved_gbs": ch_bytes / t_ch / 1e9, "peak": hbm_peak, "frac": ch_bytes / t_ch / 1e9 / hbm_peak},
                          "timing": "4 launches on 2 rotating sets of activation buffers (2 x 8 x 67 MB > L2) captured in one CUDA graph, 10 replays, CUDA events"}
        tf = os.path.join(ROOT, "profiles", "gemm_chain_traffic.json")
        if os.path.exists(tf):
            chain_roofline["traffic"] = json.load(open(tf)).get("dram_bytes_per_launch")
    line = {
        "metric": METRIC, "value": value, "unit": "updates/s", "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": f"Envelope-Q gradient update obs={OBS} |A|={A} d={D} |W|={W} batch={B} net=4x256 per=True, store {STORE} transitions",
            "parallelism": f"replicas x{world} + 1 front all-gather per evaluation round" if world > 1 else "single GPU",
            "l2": "no explicit flush: each step streams ~0.7 GB of activation planes (65,536 x 256 x 4 B per layer), far above the 126 MB L2",
            "value_definition": "Envelope.update() with the replay store resident in HBM: PER sum-tree walk, H2D of indices + weights "
                                f"({h2d_value} B), one CUDA-graph replay, D2H of priorities + loss ({B * 4 + 4} B), priority write-back -- all inside the timed region",
            "e2e_definition": "the same call with a HOST-resident replay buffer: the gathered minibatch crosses PCIe every update",
            "eval_round": "NOT inside the timed updates: local front -> one all-gather of fixed-shape records -> global prune, stream-ordered; "
                          "timed separately, max over ranks",
            "front_points_after_allgather": int(global_front.shape[0]),
            "ms_steps_rank0": ms_steps, "ms_eval_round_rank0": ms_eval, "ms_eval_round_max": ms_eval_max,
        },
        "e2e": {"value": e2e_value, "unit": "updates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(gpu_launches),
        "clocks": clocks,
        # dominant kernel of the step (58 % of it, profiles/r02_launches.txt): one hidden layer of the pair batch.  With the f16x2 operand
        # format its HBM floor (plane bytes in + out) is above its tensor floor, so the binding roofline is HBM: `achieved` = algorithmic
        # plane bytes / time against the measured bandwidth; the tensor-pipe view (MMA flops actually issued against the measured dense
        # 16-bit peak; SURVEY 8(d)'s "FP32-accurate peak actually used" = peak / products) is reported under "tensor".
        "roofline": chain_roofline if chain_roofline is not None else {"bound": "hbm", "kernel": f"gemm_planes_kernel<pair, {agent.tensor_core_format}> (65536x256x256: one hidden layer of the pair batch, "
                                                f"{gemm_nprod} 16-bit tcgen05 products per fp32 product, CTA pairs, bias + ReLU + re-split epilogue)",
                     "achieved": gemm_alg_bytes / t_gemm / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": gemm_alg_bytes / t_gemm / 1e9 / hbm_peak,
                     "traffic": gemm_traffic, "algorithmic_bytes": gemm_alg_bytes, "us_per_launch": t_gemm * 1e6, "peak_source": peak_src,
                     "why_hbm": "floors of this launch: HBM 134.5 MB / 6.48 TB/s = 20.7 us, tensor pipe 3 x 8.6 GFLOP / 1687 TFLOP/s = 15.3 us",
                     "tensor": {"issued_tflops": gemm_flops / t_gemm / 1e12, "peak": bf16_peak, "frac": gemm_flops / t_gemm / 1e12 / bf16_peak,
                                "algorithmic_flops": gemm_flops // gemm_nprod, "algorithmic_tflops": gemm_flops / gemm_nprod / t_gemm / 1e12,
                                "fp32_accurate_peak_tflops": bf16_peak / gemm_nprod},
                     "timing": "16 launches on 4 rotating activation sets (4 x 2 x 67 MB > L2) captured in one CUDA graph, 12 replays, CUDA events"},
        "roofline_gemm_layer": gemm_layer,
        # the kernel north_star names: fused envelope-max TD target against the HBM roofline
        # the kernel north_star names ("the envelope operator ... and the vector-reward Bellman target fused into one kernel"): the form the update
        # runs -- output layers of both nets + operator + Bellman line in one kernel, Q never in HBM -- when the shape is inside it, else the
        # standalone operator; the standalone operator (the C-ABI entry morl_envelope_td_f32, issue-bound: DESIGN 4.1) is always reported too
        "roofline_envelope": fused if (fused is not None and fused["in_update"]) else standalone_env,
        "roofline_envelope_operator": standalone_env,
        "mlp": {"flop_per_step": mlp_flops, "fp32_equivalent_tflops": mlp_flops / (ms / K * 1e-3) / 1e12,
                "path": "layer 1 separable (one fp32 kernel on B + |W| rows), layers 2.. tcgen05 split-operand GEMMs forward and backward",
                "note": "whole-step time used, so this is a lower bound on the dense-layer rate"},
        "loss": loss_dev, "loss_e2e_last": loss_host,
    }
    if world == 1 and os.environ.get("MORL_SKIP_CPU_BASELINE", "0") != "1":  # (development runs only: the driver's line always carries it)
        # the reference's CPU update at the SAME config (full batch, full weight set), bounded to ~1 minute of CPU work: 1 warm-up + up to 3
        # timed updates; next to it the de-duplicated CPU restatement (not reference code; BASELINE.md section 2) for context
        times, kind, threads, info = cpu_reference_arm(max_steps=3, warmup=1, budget_s=float(os.environ.get("MORL_CPU_BASELINE_BUDGET_S", "60")))
        t_med = float(np.median(times))
        line["cpu_baseline"] = {
            "value": 1.0 / t_med, "unit": "updates/s", "cores": threads, "kind": kind,
            "sample": f"FULL config (batch {B} x |W|={W}, B*|W|^2 = {B * W * W} rows per Q-net), {len(times)} timed update(s) after 1 warm-up, median",
            "step_seconds": [round(t, 3) for t in times], "host": info,
        }
        times_d, _, _, _ = cpu_reference_arm(max_steps=3, warmup=1, budget_s=15.0, dedup=True)
        line["cpu_dedup_restatement"] = {"value": 1.0 / float(np.median(times_d)), "unit": "updates/s", "cores": threads,
                                         "note": "same update with Q evaluated on the B*|W| distinct rows (NOT the reference's code path): the ratio "
                                                 "against it excludes the reference's own |W|-fold redundancy"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_morld(args, rank, local_rank, world):
    """`--workload morld` (BASELINE.json configs[4]): MORL/D with 64 MOSAC subproblems at mo-hopper-v4 dimensions (obs 11, 3 actions, 3
    objectives; 2 x 256 nets, batch 128), policy p owned by rank p % world.  A step = one improvement pass of ``__update_others``
    (reference morld.py:423-433: every policy but the current one gets one SAC update, strictly serially) over the rank's shard, replayed
    as ONE multi-branch CUDA graph per rank; no data-path collective.  Metric: policy updates / s, whole job.  One evaluation-round
    exchange (fronts + evaluations in ONE all-gather) is timed separately."""
    import torch as th
    import torch.distributed as dist

    from morl_baselines_b200 import ops
    from morl_baselines_b200.multi_policy.morld.morld import MORLD
    from morl_baselines_b200.testing import FakeEnv

    dev = th.device("cuda", local_rank)
    th.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    POP, OBS_H, ACT_H, D_H, N_BUF = 64, 11, 3, 3, 16384
    env = FakeEnv(obs_dim=OBS_H, continuous_action_dim=ACT_H, reward_dim=D_H)
    algo = MORLD(env, pop_size=POP, update_passes=1, log=False, device=dev, seed=0, weight_init_method="random", shared_buffer=True,
                 neighborhood_size=1, policy_args={"learning_starts": 0, "buffer_size": N_BUF})
    algo.population_graph = os.environ.get("MORL_POPULATION_GRAPH", "1") != "0"
    rng = np.random.default_rng(0)
    buf = algo.population[0].wrapped.get_buffer()
    buf.obs[:], buf.next_obs[:] = rng.standard_normal((N_BUF, OBS_H)).astype(np.float32), rng.standard_normal((N_BUF, OBS_H)).astype(np.float32)
    buf.actions[:] = rng.uniform(-1, 1, (N_BUF, ACT_H)).astype(np.float32)
    buf.rewards[:], buf.dones[:] = rng.standard_normal((N_BUF, D_H)).astype(np.float32), (rng.random((N_BUF, 1)) < 0.02).astype(np.float32)
    buf.size, buf.ptr = N_BUF, 0
    buf.mark_all_dirty()
    np.random.seed(1000 + rank)
    local = algo.local_policies()
    current = algo.population[0]
    n_upd = len([p for p in local if p != current])
    K, Wm = args.steps, max(args.warmup, 3)

    def one_pass(t):
        for p in algo.population:
            p.wrapped.global_step = 2 * t  # actor + target updates every pass (policy_freq = 2, target_net_freq = 1)
        algo._update_others(current)

    for t in range(Wm):
        one_pass(t)
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ops.launch_count
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(K):
        one_pass(Wm + t)
    e1.record()
    if world > 1:
        dist.barrier()
    th.cuda.synchronize()
    clocks = sampler.result()
    # evaluation round exchange (stub evaluations: the rollouts are host work and not part of this measurement)
    evs = {p.id: rng.standard_normal(D_H) for p in algo.population}
    algo._eval_policy = lambda agent, eval_env, n: evs[agent.id]
    algo.archive.individuals, algo.archive.evaluations = [], []
    algo._eval_all_policies(None, 1, 5, np.zeros(D_H))
    th.cuda.synchronize()
    t0 = time.perf_counter()
    algo._eval_all_policies(None, 1, 5, np.zeros(D_H))
    ms_eval = (time.perf_counter() - t0) * 1e3
    t_ms = th.tensor([e0.elapsed_time(e1)], device=dev)
    n_all = th.tensor([float(n_upd)], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_all, op=dist.ReduceOp.SUM)
    if rank == 0:
        ms = float(t_ms.item())
        line = {"metric": "morld_policy_updates_per_sec", "value": float(n_all.item()) * K / (ms * 1e-3), "unit": "policy updates/s", "n_gpus": world,
                "steps": K, "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"MORL/D __update_others pass: {POP} MOSAC subproblems (obs {OBS_H}, act {ACT_H}, d {D_H}, 2x256, batch 128), "
                                       f"policy p on rank p % {world}, shared replay buffer of {N_BUF} transitions",
                           "parallelism": f"population sharded over {world} rank(s), one multi-branch CUDA graph per rank"
                                          if algo.population_graph else "one graph replay per policy (serial)",
                           "policies_updated_per_pass": int(n_all.item()), "ms_eval_exchange_rank0": ms_eval,
                           "front_points": int(algo.global_front.shape[0]),
                           "note": "dense layers of the 2x256 actor / critics are library (cuBLAS) kernels inside the graph; the TD target, Adam, "
                                   "polyak and replay gather are repo kernels"},
                "gpu_launches": int(ops.launch_count - l0), "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_envelope_dp(args, rank, local_rank, world):
    """DP-Envelope (SURVEY 8(e), reported separately from the replica headline): ONE update stream over `world` GPUs -- the scalarising weight
    set of every update is sharded over the ranks, ONE gradient all-reduce per update keeps the network identical -- strong scaling:
    value = updates/s of that single stream (max over ranks of the device time)."""
    import torch as th
    import torch.distributed as dist

    from morl_baselines_b200 import ops
    from morl_baselines_b200.multi_policy.envelope.envelope import Envelope
    from morl_baselines_b200.testing import FakeEnv, synthetic_store

    dev = th.device("cuda", local_rank)
    th.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, args.warmup
    np.random.seed(1000)  # identical on every rank: the ranks of one learner sample the same minibatches and weight sets
    th.manual_seed(0)
    agent = Envelope(FakeEnv(obs_dim=OBS, n_actions=A, reward_dim=D), batch_size=B, num_sample_w=W, per=True, buffer_size=STORE, net_arch=NET, log=False, seed=0,
                     device=dev, replay_on_device=True, dp_group=True if world > 1 else None)
    _fill_store(agent.replay_buffer, synthetic_store(STORE, OBS, A, D, seed=0))
    agent.replay_buffer.flush()
    agent.global_step = 1
    for _ in range(max(Wm, 3)):
        agent.update()
    th.cuda.synchronize()
    if world > 1:
        dist.barrier()
    mon = ClockSampler(local_rank)
    mon.start()
    l0 = ops.launch_count
    e0, e1 = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        agent.update()
    e1.record()
    th.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = mon.result()
    t_ms = th.tensor([e0.elapsed_time(e1)], device=dev)
    psum = th.stack([p.detach().double().sum() for p in agent.q_net.parameters()]).sum().reshape(1)
    pmin, pmax = psum.clone(), psum.clone()
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        dist.all_reduce(pmax, op=dist.ReduceOp.MAX)
    if rank == 0:
        ms = float(t_ms.item())
        line = {"metric": "envelope_q_dp_updates_per_sec", "value": K / (ms * 1e-3), "unit": "updates/s", "n_gpus": world, "steps": K, "warmup": Wm,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"DP-Envelope: ONE Envelope-Q update stream obs={OBS} |A|={A} d={D} |W|={W} batch={B} net=4x256 per=True over {world} GPU(s)",
                           "parallelism": f"weight set sharded {W}/{world} per rank for the training pass (targets for all weights recomputed per rank), "
                                          "ONE all-reduce per update (gradients 851 KB + priorities + loss)" if world > 1 else "single GPU (same code path, no collective)",
                           "replicas_identical": bool(float(pmin.item()) == float(pmax.item())), "loss": float(agent._last_loss)},
                "gpu_launches": int(ops.launch_count - l0), "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="envelope", choices=["envelope", "morld", "envelope_dp"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed update as DIR/<name>.npy (envelope workload, rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "envelope"):
        ap.error("--dump-outputs is available for --impl b200 --workload envelope")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
    elif args.workload == "morld":
        run_morld(args, rank, local_rank, world)
    elif args.workload == "envelope_dp":
        run_envelope_dp(args, rank, local_rank, world)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
