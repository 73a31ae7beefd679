"""Thin PyTorch-facing wrappers over the C-ABI (include/morl_b200.h).

PyTorch is plumbing here: it owns the device buffers and the stream; every operator below is one (or two) launches of a
hand-written sm_100a kernel from libmorl_b200.so.  All wrappers require CUDA tensors and raise otherwise -- there is
no CPU / eager fallback (the CPU restatement lives in oracle/ and is test-only).
"""

from __future__ import annotations

from typing import Optional, Tuple

import torch as th

from . import _lib
from ._lib import (  # noqa: F401  (re-exported constants)
    AC_ARGMIN_GATHER,
    AC_ELEMENTWISE_MIN,
    AC_SCALAR_MIN,
    DOT_FMA,
    DOT_PAIRFMA,
    DOT_UNFUSED,
    MAP_BLOCK,
    MAP_TILE,
    ROWS_BMAJOR,
    ROWS_REFERENCE,
)

# number of kernels launched through this module (bench.py reports it as `gpu_launches`)
launch_count = 0


def _count(n=1):
    global launch_count
    launch_count += n


def _dev(t: th.Tensor, name: str, dtype=th.float32) -> th.Tensor:
    if not isinstance(t, th.Tensor) or not t.is_cuda:
        raise _lib.MorlB200Error(f"{name} must be a CUDA tensor (morl_baselines_b200 has no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.MorlB200Error(f"{name} must have dtype {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _ptr(t: Optional[th.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return th.cuda.current_stream().cuda_stream


def envelope_td(q_online, q_target, wset, reward, done, gamma: float, dot_mode: int = DOT_UNFUSED, row_order: int = ROWS_REFERENCE,
                want_indices: bool = True, out: Optional[th.Tensor] = None, pref_out=None, act_out=None):
    """Fused envelope-max TD target (reference envelope.py:404-440 + :298).  q_*: [B, W, A, D]; returns
    (target [W*B, D], pref [W*B] int32, act [W*B] int32)."""
    q_online, q_target = _dev(q_online, "q_online"), _dev(q_target, "q_target")
    B, W, A, D = q_online.shape
    if q_target.shape != q_online.shape:
        raise _lib.MorlB200Error("q_online / q_target shape mismatch")
    wset, reward, done = _dev(wset, "wset"), _dev(reward, "reward"), _dev(done, "done")
    if wset.shape != (W, D) or reward.shape != (B, D) or done.numel() != B:
        raise _lib.MorlB200Error(f"bad shapes: wset {tuple(wset.shape)}, reward {tuple(reward.shape)}, done {tuple(done.shape)}")
    if out is None:
        out = th.empty((W * B, D), device=q_online.device, dtype=th.float32)
    if want_indices:
        pref_out = th.empty(W * B, device=q_online.device, dtype=th.int32) if pref_out is None else pref_out
        act_out = th.empty(W * B, device=q_online.device, dtype=th.int32) if act_out is None else act_out
    rc = _lib.load().morl_envelope_td_f32(_ptr(q_online), _ptr(q_target), _ptr(wset), _ptr(reward), _ptr(done), float(gamma), B, W, A, D,
                                          dot_mode, row_order, _ptr(out), _ptr(pref_out), _ptr(act_out), _stream())
    _lib.check(rc, "morl_envelope_td_f32")
    _count()
    return out, pref_out, act_out


def _rows(t, D, name):
    t = _dev(t, name)
    return t.reshape(-1, D)


def greedy_td(q_select, q_eval, w, reward=None, done=None, gamma: float = 0.0, dot_mode: int = DOT_UNFUSED, w_map: int = MAP_BLOCK,
              r_map: int = MAP_TILE):
    """Double-DQN target with per-row weights (reference envelope.py:442-463).  q_*: [N, A, D]."""
    q_select, q_eval = _dev(q_select, "q_select"), _dev(q_eval, "q_eval")
    N, A, D = q_select.shape
    w = _rows(w, D, "w")
    if reward is not None:
        reward, done = _rows(reward, D, "reward"), _dev(done, "done").reshape(-1)
    out = th.empty((N, D), device=q_select.device, dtype=th.float32)
    act = th.empty(N, device=q_select.device, dtype=th.int32)
    rc = _lib.load().morl_greedy_td_f32(_ptr(q_select), _ptr(q_eval), _ptr(w), w.shape[0], w_map, _ptr(reward), _ptr(done),
                                        N if reward is None else reward.shape[0], r_map, float(gamma), N, A, D, dot_mode, _ptr(out),
                                        _ptr(act), _stream())
    _lib.check(rc, "morl_greedy_td_f32")
    _count()
    return out, act


def critic_min_td(q_nets, w, reward=None, done=None, gamma: float = 0.0, dot_mode: int = DOT_UNFUSED, w_map: int = MAP_BLOCK,
                  r_map: int = MAP_TILE):
    """GPI-PD critic-min greedy target (reference gpi_pd.py:445-463).  q_nets: [n_nets, N, A, D]."""
    q_nets = _dev(q_nets, "q_nets")
    n_nets, N, A, D = q_nets.shape
    w = _rows(w, D, "w")
    if reward is not None:
        reward, done = _rows(reward, D, "reward"), _dev(done, "done").reshape(-1)
    out = th.empty((N, D), device=q_nets.device, dtype=th.float32)
    act = th.empty(N, device=q_nets.device, dtype=th.int32)
    rc = _lib.load().morl_critic_min_td_f32(_ptr(q_nets), n_nets, _ptr(w), w.shape[0], w_map, _ptr(reward), _ptr(done),
                                            N if reward is None else reward.shape[0], r_map, float(gamma), N, A, D, dot_mode, _ptr(out),
                                            _ptr(act), _stream())
    _lib.check(rc, "morl_critic_min_td_f32")
    _count()
    return out, act


def gpi_envelope(q_nets, w, reward=None, done=None, gamma: float = 0.0, dot_mode: int = DOT_UNFUSED, w_map: int = MAP_BLOCK,
                 r_map: int = MAP_TILE):
    """GPI envelope / policy-set evaluation (reference gpi_pd.py:662-690, 564-582).  q_nets: [n_nets, B, P, A, D];
    returns (out [B, D], policy [B] int32, action [B] int32)."""
    q_nets = _dev(q_nets, "q_nets")
    n_nets, B, P, A, D = q_nets.shape
    w = _rows(w, D, "w")
    if reward is not None:
        reward, done = _rows(reward, D, "reward"), _dev(done, "done").reshape(-1)
    out = th.empty((B, D), device=q_nets.device, dtype=th.float32)
    pol = th.empty(B, device=q_nets.device, dtype=th.int32)
    act = th.empty(B, device=q_nets.device, dtype=th.int32)
    rc = _lib.load().morl_gpi_envelope_f32(_ptr(q_nets), n_nets, _ptr(w), w.shape[0], w_map, _ptr(reward), _ptr(done),
                                           B if reward is None else reward.shape[0], r_map, float(gamma), B, P, A, D, dot_mode, _ptr(out),
                                           _ptr(pol), _ptr(act), _stream())
    _lib.check(rc, "morl_gpi_envelope_f32")
    _count()
    return out, pol, act


def actor_critic_td(q_nets, w, reward, done, logp, alpha: float, gamma: float, variant: int, w_map: int = MAP_BLOCK):
    """Continuous-action vector targets (CAPQL / MOSAC / TD3-style GPI-PD; SURVEY Appendix A.4).  q_nets: [n_nets, N, D]."""
    q_nets = _dev(q_nets, "q_nets")
    n_nets, N, D = q_nets.shape
    reward, done = _dev(reward, "reward").reshape(N, D), _dev(done, "done").reshape(-1)
    if w is not None:
        w = _rows(w, D, "w")
    if logp is not None:
        logp = _dev(logp, "logp").reshape(-1)
    out = th.empty((N,) if variant == AC_SCALAR_MIN else (N, D), device=q_nets.device, dtype=th.float32)
    rc = _lib.load().morl_actor_critic_td_f32(_ptr(q_nets), n_nets, _ptr(w), 0 if w is None else w.shape[0], w_map, _ptr(reward), _ptr(done),
                                              _ptr(logp), float(alpha), float(gamma), N, D, variant, _ptr(out), _stream())
    _lib.check(rc, "morl_actor_critic_td_f32")
    _count()
    return out


def td_workspace(n_rows: int, device) -> th.Tensor:
    nbytes = _lib.load().morl_td_workspace_bytes(int(n_rows))
    return th.empty((nbytes + 3) // 4, device=device, dtype=th.float32)


def td_mse_priority(q_values, action, target_q, wset, homotopy_lambda: float, B: int, W: int, row_order: int = ROWS_REFERENCE,
                    want_grad: bool = True, want_prio: bool = True, workspace: Optional[th.Tensor] = None, loss_out=None, grad_out=None,
                    prio_out=None, q_taken_out=None, lambda_dev=None):
    """Fused Envelope TD loss + d loss / d q_values + priorities (reference envelope.py:301-313, 329-331).  ``lambda_dev`` (device f32 [1])
    overrides ``homotopy_lambda`` and is read by the kernels at run time (graph-replay safe)."""
    q_values = _dev(q_values, "q_values")
    N, A, D = q_values.shape
    if N != B * W:
        raise _lib.MorlB200Error(f"q_values has {N} rows, expected B*W = {B * W}")
    action = _dev(action, "action", th.int32).reshape(-1)
    target_q, wset = _dev(target_q, "target_q"), _dev(wset, "wset")
    dev = q_values.device
    loss = th.empty(1, device=dev, dtype=th.float32) if loss_out is None else loss_out
    grad = (th.empty_like(q_values) if grad_out is None else grad_out) if want_grad else None
    prio = (th.empty(B, device=dev, dtype=th.float32) if prio_out is None else prio_out) if want_prio else None
    ws = td_workspace(N, dev) if workspace is None else workspace
    rc = _lib.load().morl_td_mse_priority_f32(_ptr(q_values), _ptr(action), _ptr(target_q), _ptr(wset), float(homotopy_lambda), _ptr(lambda_dev), B, W, A, D,
                                              row_order, _ptr(loss), _ptr(grad), _ptr(q_taken_out), _ptr(prio), _ptr(ws), _stream())
    _lib.check(rc, "morl_td_mse_priority_f32")
    _count(2)
    return loss, grad, prio


def td_huber_priority(q_values, action, target_q, target_q_gpi, w, min_priority: float, p_rows: int, w_map: int = MAP_BLOCK,
                      want_grad: bool = True, workspace: Optional[th.Tensor] = None):
    """GPI-PD Huber-style loss, gradient seed and raw priorities (reference gpi_pd.py:469-487, 507-520)."""
    q_values = _dev(q_values, "q_values")
    n_nets, N, A, D = q_values.shape
    action = _dev(action, "action", th.int32).reshape(-1)
    target_q = _dev(target_q, "target_q")
    if target_q_gpi is not None:
        target_q_gpi = _dev(target_q_gpi, "target_q_gpi")
    w = _rows(w, D, "w")
    dev = q_values.device
    loss = th.empty(1, device=dev, dtype=th.float32)
    grad = th.empty_like(q_values) if want_grad else None
    prio = th.empty(p_rows, device=dev, dtype=th.float32) if p_rows > 0 else None
    ws = td_workspace(N, dev) if workspace is None else workspace
    rc = _lib.load().morl_td_huber_priority_f32(_ptr(q_values), n_nets, _ptr(action), action.shape[0], _ptr(target_q), _ptr(target_q_gpi),
                                                _ptr(w), w.shape[0], w_map, float(min_priority), N, A, D, p_rows, _ptr(loss), _ptr(grad),
                                                _ptr(prio), _ptr(ws), _stream())
    _lib.check(rc, "morl_td_huber_priority_f32")
    _count(2)
    return loss, grad, prio


def replay_gather(obs_store, next_obs_store, act_store, rew_store, done_store, idx, outs=None):
    """Gather a minibatch from device-resident stores (reference buffer.py:82-94).  Returns
    (obs, actions, rewards, next_obs, dones); uint8 actions come back as int32."""
    obs_store, next_obs_store = _dev(obs_store, "obs_store"), _dev(next_obs_store, "next_obs_store")
    rew_store, done_store = _dev(rew_store, "rew_store"), _dev(done_store, "done_store")
    idx = _dev(idx, "idx", th.int64).reshape(-1)
    cap, obs_dim = obs_store.shape[0], obs_store[0].numel()
    is_u8 = act_store.dtype == th.uint8
    act_store = _dev(act_store, "act_store", th.uint8 if is_u8 else th.float32)
    act_dim, rew_dim = act_store[0].numel(), rew_store[0].numel()
    B = idx.shape[0]
    dev = obs_store.device
    if outs is None:
        obs = th.empty((B,) + tuple(obs_store.shape[1:]), device=dev, dtype=th.float32)
        nobs = th.empty_like(obs)
        act = th.empty((B, act_dim), device=dev, dtype=th.int32 if is_u8 else th.float32)
        rew = th.empty((B, rew_dim), device=dev, dtype=th.float32)
        done = th.empty((B, 1), device=dev, dtype=th.float32)
    else:
        obs, act, rew, nobs, done = outs
    rc = _lib.load().morl_replay_gather(_ptr(obs_store), _ptr(next_obs_store), _ptr(act_store), _ptr(rew_store), _ptr(done_store), _ptr(idx),
                                        B, obs_dim, act_dim, rew_dim, int(is_u8), cap, _ptr(obs), _ptr(nobs), _ptr(act), _ptr(rew), _ptr(done),
                                        _stream())
    _lib.check(rc, "morl_replay_gather")
    _count()
    return obs, act, rew, nobs, done


def pareto_mask(points: th.Tensor, remove_duplicates: bool = True, raw: bool = False, out: Optional[th.Tensor] = None) -> th.Tensor:
    """Non-dominated mask (reference pareto.py:34-57) of an [N, D] fp32 / fp64 CUDA tensor -> bool [N] (``raw``: the kernel's uint8 [N],
    optionally written into ``out``: no further launch)."""
    if not points.is_cuda:
        raise _lib.MorlB200Error("points must be a CUDA tensor (morl_baselines_b200 has no CPU fallback)")
    if points.dtype not in (th.float32, th.float64):
        raise _lib.MorlB200Error(f"points must be float32 or float64, got {points.dtype}")
    points = points.contiguous()
    N, D = points.shape
    keep = th.empty(N, device=points.device, dtype=th.uint8) if out is None else out
    if N == 0:
        return keep if raw else keep.bool()
    fn = _lib.load().morl_pareto_mask_f32 if points.dtype == th.float32 else _lib.load().morl_pareto_mask_f64
    rc = fn(_ptr(points), N, D, int(bool(remove_duplicates)), _ptr(keep), _stream())
    _lib.check(rc, "morl_pareto_mask")
    _count(2)
    return keep if raw else keep.bool()


def front_pack(points: th.Tensor, keep: Optional[th.Tensor], cap: int, rec: th.Tensor, extras: Optional[th.Tensor] = None) -> th.Tensor:
    """rec (float64 [1 + cap*d + n_extra]) = [count | first cap kept rows of points [n, d] (float64), -inf padded | extras]; one launch,
    no host sync (the count stays on the device)."""
    n, d = points.shape
    n_extra = 0 if extras is None else extras.numel()
    if points.dtype != th.float64 or not points.is_contiguous() or rec.numel() != 1 + cap * d + n_extra:
        raise _lib.MorlB200Error("front_pack: points must be contiguous float64 [n, d] and rec float64 [1 + cap*d + n_extra]")
    rc = _lib.load().morl_front_pack_f64(_ptr(points), _ptr(keep), n, d, cap, _ptr(extras), n_extra, _ptr(rec), _stream())
    _lib.check(rc, "morl_front_pack_f64")
    _count()
    return rec


def front_unpack(gathered: th.Tensor, world: int, d: int, cap: int, n_extra: int, pts_out: th.Tensor, meta_out: th.Tensor):
    """gathered records [world, 1 + cap*d + n_extra] -> pts_out [world*cap, d], meta_out [world, 1 + n_extra] (count, extras); one launch."""
    rc = _lib.load().morl_front_unpack_f64(_ptr(gathered), world, d, cap, n_extra, _ptr(pts_out), _ptr(meta_out), _stream())
    _lib.check(rc, "morl_front_unpack_f64")
    _count()
    return pts_out, meta_out


def hypervolume(points: th.Tensor, ref_point: th.Tensor, keep: Optional[th.Tensor] = None, out: Optional[th.Tensor] = None) -> th.Tensor:
    """Exact hypervolume (maximisation, d <= 3, n <= 2048) of float64 CUDA points [n, d] above ``ref_point`` [d]; returns a device float64
    scalar tensor [1] (no host sync).  ``keep`` (uint8 [n]) restricts the set, e.g. to the output of ``pareto_mask(..., raw=True)``."""
    if not points.is_cuda or points.dtype != th.float64 or not points.is_contiguous():
        raise _lib.MorlB200Error("hypervolume: points must be a contiguous float64 CUDA tensor [n, d]")
    n, d = points.shape
    ref_point = ref_point.to(device=points.device, dtype=th.float64).contiguous()
    out = th.empty(1, dtype=th.float64, device=points.device) if out is None else out
    rc = _lib.load().morl_hypervolume_f64(_ptr(points), _ptr(keep), n, d, _ptr(ref_point), _ptr(out), _stream())
    _lib.check(rc, "morl_hypervolume_f64")
    _count()
    return out


class PolyakPlan:
    """Device-side (param, target, size) table for morl_polyak_f32; build once per pair of networks."""

    def __init__(self, params, targets):
        params, targets = list(params), list(targets)
        assert len(params) == len(targets) and len(params) > 0
        for p, t in zip(params, targets):
            if not (p.is_cuda and t.is_cuda and p.dtype == th.float32 and t.dtype == th.float32 and p.is_contiguous() and t.is_contiguous()):
                raise _lib.MorlB200Error("polyak: parameters must be contiguous float32 CUDA tensors")
            assert p.numel() == t.numel()
        dev = params[0].device
        self.keepalive = (params, targets)
        self.p_tab = th.tensor([p.data_ptr() for p in params], dtype=th.int64, device=dev)
        self.t_tab = th.tensor([t.data_ptr() for t in targets], dtype=th.int64, device=dev)
        self.sizes = th.tensor([p.numel() for p in params], dtype=th.int64, device=dev)
        self.n = len(params)
        self.max_size = max(p.numel() for p in params)

    def run(self, tau: float):
        rc = _lib.load().morl_polyak_f32(_ptr(self.p_tab), _ptr(self.t_tab), _ptr(self.sizes), self.n, self.max_size, float(tau), _stream())
        _lib.check(rc, "morl_polyak_f32")
        _count()


def sm_count() -> int:
    n = _lib.load().morl_device_sm_count()
    if n < 0:
        _lib.check(n, "morl_device_sm_count")
    return n


# ------------------------------------------------------------------------------------------------ tcgen05 dense layers
def _pad(n: int, m: int) -> int:
    return (n + m - 1) // m * m


FMT_BF16X3, FMT_F16X2 = _lib.FMT_BF16X3, _lib.FMT_F16X2
_FMT_DTYPE = {FMT_BF16X3: th.bfloat16, FMT_F16X2: th.float16}
_FMT_PLANES = {FMT_BF16X3: 3, FMT_F16X2: 2}


def fmt_of(planes: th.Tensor) -> int:
    """Plane format of a plane tensor: bf16 [3, rows, ld] = bf16x3, fp16 [2, rows, ld] = f16x2."""
    if planes.dtype == th.bfloat16 and planes.shape[0] == 3:
        return FMT_BF16X3
    if planes.dtype == th.float16 and planes.shape[0] == 2:
        return FMT_F16X2
    raise _lib.MorlB200Error(f"not a plane tensor: dtype {planes.dtype}, leading dimension {planes.shape[0]}")


def empty_planes(fmt: int, rows: int, ld: int, device) -> th.Tensor:
    return th.empty((_FMT_PLANES[fmt], rows, ld), device=device, dtype=_FMT_DTYPE[fmt])


def scale_tensor(value: float, device) -> th.Tensor:
    """A device-resident power-of-two scale (float32 [1])."""
    return th.full((1,), float(value), device=device, dtype=th.float32)


def plane_overflow_count(reset: bool = False) -> int:
    """Number of f16x2 range violations (|scale * x| > 65504) the plane-producing kernels saw since the last reset (synchronises)."""
    n = _lib.load().morl_plane_overflow_count(int(reset))
    if n < 0:
        _lib.check(n, "morl_plane_overflow_count")
    return n


def amax_scale(x: th.Tensor, target_exp: int, scale_out: th.Tensor, workspace: th.Tensor) -> th.Tensor:
    """scale_out[0] = 2^(target_exp - e) with max|x| < 2^e (one launch; workspace: 2 zeroed int32, left zeroed)."""
    x = _dev(x, "x")
    rc = _lib.load().morl_amax_scale_f32(_ptr(x), x.numel(), int(target_exp), _ptr(scale_out), _ptr(workspace), _stream())
    _lib.check(rc, "morl_amax_scale_f32")
    _count()
    return scale_out


def split_planes(x: th.Tensor, fmt: int = FMT_F16X2, rows_pad: Optional[int] = None, ldp: Optional[int] = None, transpose: bool = False,
                 out: Optional[th.Tensor] = None, scale: Optional[th.Tensor] = None) -> th.Tensor:
    """fp32 [rows, cols] -> planes [P, rows_pad, ldp] of scale * x (zero padded); with ``transpose`` the planes hold x^T."""
    x = _dev(x, "x")
    r, c = (x.shape[1], x.shape[0]) if transpose else (x.shape[0], x.shape[1])
    rows_pad = r if rows_pad is None else rows_pad
    ldp = _pad(c, 64 if fmt == FMT_F16X2 else 32) if ldp is None else ldp
    if out is None:
        out = empty_planes(fmt, rows_pad, ldp, x.device)
    rc = _lib.load().morl_split_planes(fmt, _ptr(x), r, c, x.shape[1], int(transpose), _ptr(out), rows_pad, ldp, out.stride(0), _ptr(scale), _stream())
    _lib.check(rc, "morl_split_planes")
    _count()
    return out


def split_planes_multi(jobs, fmt: int = FMT_F16X2) -> None:
    """One launch for several splits.  jobs: iterable of (src [rows, cols] fp32 CUDA, out planes [P, rows_pad, ldp], transpose, scale, target_exp):
    ``scale`` is a device float [1] or None; ``target_exp`` None = use the scale as given, an int = derive it from the matrix's amax and store it."""
    jobs = list(jobs)
    if not jobs:
        return
    if len(jobs) > _lib.SPLIT_MAX_JOBS:
        raise _lib.MorlB200Error(f"split_planes_multi: at most {_lib.SPLIT_MAX_JOBS} jobs per call")
    arr = (_lib.SplitJob * len(jobs))()
    for k, job in enumerate(jobs):
        src, out, transpose = job[0], job[1], job[2]
        scale = job[3] if len(job) > 3 else None
        target_exp = job[4] if len(job) > 4 else None
        src = _dev(src, "src")
        rows, cols = (src.shape[1], src.shape[0]) if transpose else (src.shape[0], src.shape[1])
        arr[k].src, arr[k].dst_planes, arr[k].plane_stride = src.data_ptr(), out.data_ptr(), out.stride(0)
        arr[k].scale = None if scale is None else scale.data_ptr()
        arr[k].rows, arr[k].cols, arr[k].ld_src, arr[k].transpose = rows, cols, src.stride(0), int(bool(transpose))
        arr[k].rows_pad, arr[k].ldp = out.shape[1], out.shape[2]
        arr[k].auto_scale, arr[k].target_exp = (0, 0) if target_exp is None else (1, int(target_exp))
    rc = _lib.load().morl_split_planes_multi(fmt, arr, len(jobs), _stream())
    _lib.check(rc, "morl_split_planes_multi")
    _count(2 if any(a.auto_scale for a in arr) else 1)


def gemm_planes(a_planes: th.Tensor, b_planes: th.Tensor, n_out: int, bias: Optional[th.Tensor] = None, relu: bool = False,
                relu_mask: Optional[th.Tensor] = None, out_f32: bool = True, out_planes: bool = False, c_f32: Optional[th.Tensor] = None,
                c_planes: Optional[th.Tensor] = None, reverse_tiles: bool = False, a_scale: Optional[th.Tensor] = None,
                b_scale: Optional[th.Tensor] = None, c_scale: Optional[th.Tensor] = None, split_acc: bool = False,
                relu_bits_in: Optional[th.Tensor] = None, relu_bits_out: Optional[th.Tensor] = None):
    """C = act(A . B^T + bias) on the tcgen05 tensor cores with split operands (fp32-accurate).
    a_planes [P, M, K], b_planes [P, N_pad, K]; the scales are device floats the planes were multiplied by (None = 1);
    ``split_acc``: leading and correction products in separate accumulators (the tensor cores truncate their fp32 accumulation; ~2.5x
    smaller systematic error, ~20 % slower per launch); False (default): one double-buffered accumulator.
    ``relu_bits_out`` / ``relu_bits_in`` (:func:`empty_relu_bits`): the forward call records [C > 0] as one bit per column, the backward
    call zeroes the outputs whose bit is clear (ReLU backward from 32 bytes per row instead of the activation planes; ``relu_mask`` is the
    plane-based form of the same mask).
    returns (c_f32 [M, n_out] or None, c_planes [P, M, ldp] holding c_scale * C, or None)."""
    fmt = fmt_of(a_planes)
    if fmt_of(b_planes) != fmt or not a_planes.is_cuda:
        raise _lib.MorlB200Error("gemm_planes: operands must be CUDA plane tensors of the same format")
    _, M, K = a_planes.shape
    _, n_pad, Kb = b_planes.shape
    if Kb != K or a_planes.stride(1) != K or b_planes.stride(1) != K:
        raise _lib.MorlB200Error("gemm_planes: operand planes must be K-major with equal K")
    dev = a_planes.device
    if out_f32 and c_f32 is None:
        c_f32 = th.empty((M, n_out), device=dev, dtype=th.float32)
    if out_planes and c_planes is None:
        c_planes = empty_planes(fmt, M, _pad(n_out, 32), dev)
    mask0 = None if relu_mask is None else relu_mask[0]
    for bits in (relu_bits_in, relu_bits_out):
        if bits is not None and (bits.dtype != th.int32 or tuple(bits.shape) != (M, 8) or not bits.is_contiguous() or bits.device != dev):
            raise _lib.MorlB200Error(f"gemm_planes: ReLU bit masks must be contiguous int32 [{M}, 8] on {dev}")
    rc = _lib.load().morl_gemm_planes_f32(fmt, _ptr(a_planes), a_planes.stride(0), _ptr(a_scale), _ptr(b_planes), b_planes.stride(0), _ptr(b_scale), M,
                                          n_out, n_pad, K, _ptr(bias), int(relu), _ptr(mask0), 0 if mask0 is None else mask0.stride(0), _ptr(c_f32),
                                          0 if c_f32 is None else c_f32.stride(0), _ptr(c_planes), 0 if c_planes is None else c_planes.shape[2],
                                          0 if c_planes is None else c_planes.stride(0), _ptr(c_scale), int(reverse_tiles), int(bool(split_acc)),
                                          _ptr(relu_bits_in), _ptr(relu_bits_out), _stream())
    _lib.check(rc, "morl_gemm_planes_f32")
    _count()
    return c_f32, c_planes


def ensemble_sample(out: th.Tensor, max_logvar: th.Tensor, min_logvar: th.Tensor, model_idx: th.Tensor, noise: Optional[th.Tensor] = None,
                    obs: Optional[th.Tensor] = None, rew_dim: int = 0):
    """Probabilistic-ensemble sampling + ensemble uncertainty in one pass (reference probabilistic_ensemble.py:115-154, utils.py:165).
    out [E, N, 2*O] raw last-layer output, model_idx [N] int32, noise [E, N, O] or None (deterministic), obs [N, O - rew_dim] or None.
    Returns (sample [N, O], var [N, O], uncertainty [N])."""
    out = _dev(out, "out")
    E, N, O2 = out.shape
    O = O2 // 2
    max_logvar, min_logvar = _dev(max_logvar, "max_logvar").reshape(-1), _dev(min_logvar, "min_logvar").reshape(-1)
    model_idx = _dev(model_idx, "model_idx", th.int32)
    if O2 != 2 * O or max_logvar.numel() != O or min_logvar.numel() != O or model_idx.numel() != N:
        raise _lib.MorlB200Error(f"ensemble_sample: bad shapes out {tuple(out.shape)}, logvar bounds {max_logvar.numel()}, model_idx {tuple(model_idx.shape)} {model_idx.dtype}")
    if noise is not None:
        noise = _dev(noise, "noise")
        if tuple(noise.shape) != (E, N, O):
            raise _lib.MorlB200Error(f"ensemble_sample: noise must be [{E}, {N}, {O}]")
    if obs is not None:
        obs = _dev(obs, "obs")
        if tuple(obs.shape) != (N, O - rew_dim):
            raise _lib.MorlB200Error(f"ensemble_sample: obs must be [{N}, {O - rew_dim}]")
    sample = th.empty((N, O), device=out.device, dtype=th.float32)
    var = th.empty((N, O), device=out.device, dtype=th.float32)
    unc = th.empty(N, device=out.device, dtype=th.float32)
    rc = _lib.load().morl_ensemble_sample_f32(_ptr(out), _ptr(max_logvar), _ptr(min_logvar), _ptr(model_idx), _ptr(noise), _ptr(obs), int(rew_dim), E, N, O,
                                              _ptr(sample), _ptr(var), _ptr(unc), _stream())
    _lib.check(rc, "morl_ensemble_sample_f32")
    _count()
    return sample, var, unc


def qhead_envelope_supported(fmt: int, B: int, W: int, A: int, D: int, K: int) -> bool:
    """True if :func:`qhead_envelope_td` covers the configuration (else use gemm_planes x 2 + envelope_td)."""
    return bool(_lib.load().morl_qhead_envelope_supported(int(fmt), int(B), int(W), int(A), int(D), int(K)))


def qhead_envelope_td(a_on: th.Tensor, a_tg: th.Tensor, w_on: th.Tensor, w_tg: th.Tensor, bias_on: th.Tensor, bias_tg: th.Tensor, wset, reward,
                      done, gamma: float, B: int, W: int, A: int, D: int, dot_mode: int = DOT_UNFUSED, row_order: int = ROWS_REFERENCE,
                      a_scale_on=None, a_scale_tg=None, w_scale_on=None, w_scale_tg=None, want_indices: bool = False, out=None, pref_out=None,
                      act_out=None, q_on_out=None, q_tg_out=None, reverse_tiles: bool = False):
    """Output layer of both Q-networks + envelope operator + Bellman line in ONE kernel (reference envelope.py:420-440, :298): the Q
    tensors never reach HBM.  a_on / a_tg: last hidden activation planes [2, B*W, K] (row b*W + j) of the online / target net on s';
    w_on / w_tg: output-layer weight planes [2, 32, K]; the rest as :func:`envelope_td`.  ``q_on_out`` / ``q_tg_out`` ([B*W, A*D] fp32)
    optionally receive the Q tiles (validation).  Returns (target [W*B, D], pref, act)."""
    fmt = fmt_of(a_on)
    if fmt_of(a_tg) != fmt or fmt_of(w_on) != fmt or fmt_of(w_tg) != fmt or not a_on.is_cuda:
        raise _lib.MorlB200Error("qhead_envelope_td: operands must be CUDA plane tensors of one format")
    _, M, K = a_on.shape
    if M != B * W or tuple(a_tg.shape) != tuple(a_on.shape) or a_on.stride(1) != K or a_tg.stride(1) != K or a_tg.stride(0) != a_on.stride(0):
        raise _lib.MorlB200Error(f"qhead_envelope_td: activation planes must both be [P, {B * W}, K], K-major, equal plane strides")
    if tuple(w_on.shape) != tuple(w_tg.shape) or w_on.shape[1] != 32 or w_on.shape[2] != K or w_on.stride(1) != K or w_tg.stride(0) != w_on.stride(0):
        raise _lib.MorlB200Error(f"qhead_envelope_td: weight planes must both be [P, 32, {K}], K-major")
    wset, reward, done = _dev(wset, "wset"), _dev(reward, "reward"), _dev(done, "done")
    if wset.shape != (W, D) or reward.shape != (B, D) or done.numel() != B or bias_on.numel() != A * D or bias_tg.numel() != A * D:
        raise _lib.MorlB200Error(f"bad shapes: wset {tuple(wset.shape)}, reward {tuple(reward.shape)}, done {tuple(done.shape)}, bias {tuple(bias_on.shape)}")
    dev = a_on.device
    if out is None:
        out = th.empty((W * B, D), device=dev, dtype=th.float32)
    if want_indices:
        pref_out = th.empty(W * B, device=dev, dtype=th.int32) if pref_out is None else pref_out
        act_out = th.empty(W * B, device=dev, dtype=th.int32) if act_out is None else act_out
    rc = _lib.load().morl_qhead_envelope_td_f32(fmt, _ptr(a_on), _ptr(a_tg), a_on.stride(0), _ptr(a_scale_on), _ptr(a_scale_tg), _ptr(w_on), _ptr(w_tg),
                                                w_on.stride(0), _ptr(w_scale_on), _ptr(w_scale_tg), _ptr(bias_on), _ptr(bias_tg), K, _ptr(wset),
                                                _ptr(reward), _ptr(done), float(gamma), B, W, A, D, dot_mode, row_order, int(reverse_tiles), _ptr(out),
                                                _ptr(pref_out), _ptr(act_out), _ptr(q_on_out), _ptr(q_tg_out), _stream())
    _lib.check(rc, "morl_qhead_envelope_td_f32")
    _count()
    return out, pref_out, act_out


def gemm_chain_supported(fmt: int, M: int, K: int) -> bool:
    return bool(_lib.load().morl_gemm_chain_supported(int(fmt), int(M), int(K)))


class GemmChain:
    """Static plan of a chained launch (:func:`gemm_chain`): the pointer tables are built once, a call is one launch.
    ``acts[c]``: the n_layers + 1 plane tensors [P, M, 256] of chain c (input, then every layer's output); ``weights[c]`` / ``w_scales[c]`` /
    ``biases[c]`` / ``bits[c]`` (ReLU masks recorded) / ``bits_in[c]`` (ReLU-backward masks applied): per layer, all optional.  ``relu``: ReLU on every
    output (forward chains); False for the dX chains of the backward pass."""

    def __init__(self, acts, weights, biases=None, w_scales=None, bits=None, act_scale=None, relu: bool = True, bits_in=None, k_first: int = 0):
        import ctypes as C

        self.n_chains, self.n_layers = len(acts), len(weights[0])
        a0 = acts[0][1]  # (the first OUTPUT: the chain's input may be narrower, see k_first)
        self.fmt = fmt_of(a0)
        _, self.M, self.K = a0.shape
        self.k_first = int(k_first) if k_first else self.K
        flat_a = [t for ch in acts for t in ch]
        flat_w = [t for ch in weights for t in ch]
        flat_b = [None] * len(flat_w) if biases is None else [t.detach() for ch in biases for t in ch]
        flat_i = [None] * len(flat_w) if bits_in is None else [t for ch in bits_in for t in ch]
        flat_s = [None] * len(flat_w) if w_scales is None else [t for ch in w_scales for t in ch]
        flat_m = [None] * len(flat_w) if bits is None else [t for ch in bits for t in ch]
        if len(flat_a) != self.n_chains * (self.n_layers + 1) or any(len(w) != self.n_layers for w in weights):
            raise _lib.MorlB200Error("GemmChain: every chain needs n_layers + 1 activation tensors and n_layers weight tensors")
        for i, t in enumerate(flat_a):
            kk = self.k_first if i % (self.n_layers + 1) == 0 else self.K
            if fmt_of(t) != self.fmt or tuple(t.shape[1:]) != (self.M, kk) or not t.is_contiguous() or not t.is_cuda:
                raise _lib.MorlB200Error(f"GemmChain: activation planes must be contiguous CUDA plane tensors [P, {self.M}, {kk}] (input {self.k_first} wide, outputs 256)")
        for i, t in enumerate(flat_w):
            kk = self.k_first if i % self.n_layers == 0 else self.K
            if fmt_of(t) != self.fmt or tuple(t.shape[1:]) != (256, kk) or not t.is_contiguous():
                raise _lib.MorlB200Error(f"GemmChain: weight planes must be contiguous [P, 256, {kk}]")
        for t in flat_m + flat_i:
            if t is not None and (t.dtype != th.int32 or tuple(t.shape) != (self.M, 8) or not t.is_contiguous()):
                raise _lib.MorlB200Error(f"GemmChain: ReLU bit masks must be contiguous int32 [{self.M}, 8]")
        self._keep = (flat_a, flat_w, flat_b, flat_s, flat_m, flat_i, act_scale)
        self.relu = bool(relu)
        arr = lambda ts: (C.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])  # noqa: E731
        self._pa, self._pw, self._pb, self._ps, self._pm, self._pi = arr(flat_a), arr(flat_w), arr(flat_b), arr(flat_s), arr(flat_m), arr(flat_i)
        self._a_stride, self._w_stride, self._act_scale = a0.stride(0), 256 * self.K, act_scale

    def __call__(self):
        rc = _lib.load().morl_gemm_chain_f32(self.fmt, self.n_chains, self.n_layers, self._pa, self._a_stride, _ptr(self._act_scale), self._pw, self._w_stride,
                                             self._ps, self._pb, int(self.relu), self._pi, self._pm, self.M, self.K, self.k_first, _stream())
        _lib.check(rc, "morl_gemm_chain_f32")
        _count()


def qhead_gemm_supported(fmt: int, M: int, N: int, K: int) -> bool:
    return bool(_lib.load().morl_qhead_gemm_supported(int(fmt), int(M), int(N), int(K)))


def qhead_gemm(a_planes: th.Tensor, w_planes: th.Tensor, n_out: int, bias: th.Tensor, out: Optional[th.Tensor] = None, a_scale=None, w_scale=None,
               reverse_tiles: bool = False) -> th.Tensor:
    """Output layer Q = A . W^T + bias (n_out <= 32) as fp32 [M, n_out]: the narrow form of :func:`gemm_planes` (bit-identical) with the weight
    planes resident in shared memory (csrc/qhead_envelope.cu without its operator half)."""
    fmt = fmt_of(a_planes)
    _, M, K = a_planes.shape
    if fmt_of(w_planes) != fmt or tuple(w_planes.shape[1:]) != (32, K) or a_planes.stride(1) != K or w_planes.stride(1) != K:
        raise _lib.MorlB200Error(f"qhead_gemm: need K-major planes A [P, M, K] and W [P, 32, K] of one format (got {tuple(a_planes.shape)}, {tuple(w_planes.shape)})")
    if out is None:
        out = th.empty((M, n_out), device=a_planes.device, dtype=th.float32)
    rc = _lib.load().morl_qhead_gemm_f32(fmt, _ptr(a_planes), a_planes.stride(0), _ptr(a_scale), _ptr(w_planes), w_planes.stride(0), _ptr(w_scale), _ptr(bias), M,
                                         n_out, K, int(reverse_tiles), _ptr(out), _stream())
    _lib.check(rc, "morl_qhead_gemm_f32")
    _count()
    return out


def empty_relu_bits(rows: int, device) -> th.Tensor:
    """ReLU bit-mask tensor [rows, 8] int32 (layout: include/morl_b200.h, morl_gemm_planes_f32)."""
    return th.empty((rows, 8), device=device, dtype=th.int32)


def unpack_relu_bits(bits: th.Tensor, n_cols: int) -> th.Tensor:
    """[rows, n_cols] bool from a ReLU bit-mask tensor (tests / diagnostics)."""
    c = th.arange((n_cols + 31) // 32, device=bits.device)
    words = bits[:, (c & 1) * 4 + (c >> 1)].to(th.int64) & 0xFFFFFFFF  # [rows, chunks]
    j = th.arange(32, device=bits.device)
    return (((words[:, :, None] >> j) & 1) != 0).reshape(bits.shape[0], -1)[:, :n_cols]


def pairs_relu_split(u: th.Tensor, v: th.Tensor, out: Optional[th.Tensor] = None, fmt: int = FMT_F16X2, scale: Optional[th.Tensor] = None,
                     relu_bits_out: Optional[th.Tensor] = None) -> th.Tensor:
    """relu(u[b] + v[j]) for every pair, written as planes [P, B*W, H] of scale * h (row b*W + j); ``relu_bits_out`` [B*W, 8] int32
    additionally receives [h > 0] as bits (the ReLU-backward mask of :func:`gemm_planes`)."""
    u, v = _dev(u, "u"), _dev(v, "v")
    B, H = u.shape
    W = v.shape[0]
    if out is None:
        out = empty_planes(fmt, B * W, H, u.device)
    else:
        fmt = fmt_of(out)
    rc = _lib.load().morl_pairs_relu_split_planes(fmt, _ptr(u), _ptr(v), B, W, H, _ptr(out), out.stride(0), _ptr(scale), _ptr(relu_bits_out), _stream())
    _lib.check(rc, "morl_pairs_relu_split_planes")
    _count()
    return out


def pair_layer1_uv(feats: th.Tensor, wset: th.Tensor, weight: th.Tensor, bias: th.Tensor, u: Optional[th.Tensor] = None,
                   v: Optional[th.Tensor] = None):
    """u = feats @ W1[:, :F]^T [B, H] and v = wset @ W1[:, F:]^T + b1 [W, H] in one launch (separable first layer of the pair batch)."""
    feats, wset, weight, bias = _dev(feats, "feats"), _dev(wset, "wset"), _dev(weight, "weight"), _dev(bias, "bias")
    B, F = feats.shape
    W, D = wset.shape
    H = weight.shape[0]
    if weight.shape[1] != F + D or bias.numel() != H:
        raise _lib.MorlB200Error(f"pair_layer1_uv: weight {tuple(weight.shape)} does not match F={F}, D={D}")
    u = th.empty((B, H), device=feats.device, dtype=th.float32) if u is None else u
    v = th.empty((W, H), device=feats.device, dtype=th.float32) if v is None else v
    rc = _lib.load().morl_pair_layer1_uv_f32(_ptr(feats), _ptr(wset), _ptr(weight), _ptr(bias), B, W, F, D, H, _ptr(u), _ptr(v), _stream())
    _lib.check(rc, "morl_pair_layer1_uv_f32")
    _count()
    return u, v


def pair_layer1_grad_workspace(F: int, D: int, H: int, device) -> th.Tensor:
    nbytes = _lib.load().morl_pair_layer1_grad_workspace_bytes(int(F), int(D), int(H))
    return th.zeros((nbytes + 3) // 4, device=device, dtype=th.float32)  # arrival counters start at zero (self-resetting afterwards)


def pair_layer1_grad(dU: th.Tensor, dV: th.Tensor, feats: th.Tensor, wset: th.Tensor, dW1: Optional[th.Tensor] = None, db1: Optional[th.Tensor] = None,
                     workspace: Optional[th.Tensor] = None):
    """dW1 [H, F + D] = [dU^T feats | dV^T wset] and db1 [H] = colsum(dV) in one launch (backward of the separable first layer)."""
    dU, dV, feats, wset = _dev(dU, "dU"), _dev(dV, "dV"), _dev(feats, "feats"), _dev(wset, "wset")
    B, H = dU.shape
    W, D = wset.shape
    F = feats.shape[1]
    if dV.shape != (W, H) or feats.shape[0] != B:
        raise _lib.MorlB200Error(f"pair_layer1_grad: dU {tuple(dU.shape)}, dV {tuple(dV.shape)}, feats {tuple(feats.shape)}, wset {tuple(wset.shape)} disagree")
    dW1 = th.empty((H, F + D), device=dU.device, dtype=th.float32) if dW1 is None else dW1
    db1 = th.empty(H, device=dU.device, dtype=th.float32) if db1 is None else db1
    ws = pair_layer1_grad_workspace(F, D, H, dU.device) if workspace is None else workspace
    rc = _lib.load().morl_pair_layer1_grad_f32(_ptr(dU), _ptr(dV), _ptr(feats), _ptr(wset), B, W, F, D, H, _ptr(dW1), _ptr(db1), _ptr(ws), _stream())
    _lib.check(rc, "morl_pair_layer1_grad_f32")
    _count()
    return dW1, db1


def gemm_mn_workspace(M: int, g_cols: int, h_cols: int, device) -> th.Tensor:
    nbytes = _lib.load().morl_gemm_mn_workspace_bytes(int(M), int(g_cols), int(h_cols))
    return th.empty((nbytes + 3) // 4, device=device, dtype=th.float32)


def gemm_planes_mn(g_planes: th.Tensor, g_cols: int, h_planes: th.Tensor, h_cols: int, transpose_out: bool = False,
                   out: Optional[th.Tensor] = None, workspace: Optional[th.Tensor] = None, colsum: Optional[th.Tensor] = None,
                   g_scale: Optional[th.Tensor] = None, h_scale: Optional[th.Tensor] = None) -> th.Tensor:
    """out[n, k] = sum_m G[m, n] H[m, k] (weight gradient; reduction over the rows) from plane tensors [P, M, ld] (scales removed), as a
    one-job launch of the :class:`GemmMnMulti` kernel.  ``colsum`` ([g_cols] fp32, optional) also receives sum_m G[m, n] (the bias gradient)."""
    fmt = fmt_of(g_planes)
    _, M, ldg = g_planes.shape
    _, M2, ldh = h_planes.shape
    if M != M2 or fmt_of(h_planes) != fmt:
        raise _lib.MorlB200Error("gemm_planes_mn: plane tensors must share format and number of rows")
    dev = g_planes.device
    if out is None:
        out = th.empty((h_cols, g_cols) if transpose_out else (g_cols, h_cols), device=dev, dtype=th.float32)
    ws = gemm_mn_workspace(M, g_cols, h_cols, dev) if workspace is None else workspace
    rc = _lib.load().morl_gemm_planes_mn_f32(fmt, _ptr(g_planes), g_planes.stride(0), ldg, g_cols, _ptr(g_scale), _ptr(h_planes), h_planes.stride(0), ldh,
                                             h_cols, _ptr(h_scale), M, int(transpose_out), _ptr(out), out.stride(0), _ptr(colsum), _ptr(ws), _stream())
    _lib.check(rc, "morl_gemm_planes_mn_f32")
    _count(2)
    return out


class GemmMnMulti:
    """Static plan of several weight-gradient products over the same rows in ONE persistent launch plus one reduction
    (morl_gemm_planes_mn_multi_f32): each entry of ``jobs`` is ``(g_planes, g_cols, h_planes, h_cols, out, colsum, g_scale, h_scale)``
    with the meaning of :func:`gemm_planes_mn` (``colsum`` and the scales may be None; ``out`` is [g_cols, h_cols], not transposed).  No output
    depends on the other jobs: each is bit-identical to :func:`gemm_planes_mn` of that job alone.  Table and workspace are built once; a call is two launches."""

    def __init__(self, jobs):
        if not 1 <= len(jobs) <= _lib.MN_MAX_JOBS:
            raise _lib.MorlB200Error(f"GemmMnMulti: 1 to {_lib.MN_MAX_JOBS} products per launch (got {len(jobs)})")
        self.fmt = fmt_of(jobs[0][0])
        self.M = jobs[0][0].shape[1]
        arr = (_lib.MnJob * len(jobs))()
        for i, (g, gc, h, hc, out, colsum, sg, sh) in enumerate(jobs):
            if fmt_of(g) != self.fmt or fmt_of(h) != self.fmt or g.shape[1] != self.M or h.shape[1] != self.M:
                raise _lib.MorlB200Error("GemmMnMulti: plane tensors must share format and number of rows")
            if tuple(out.shape) != (gc, hc) or out.stride(1) != 1 or out.dtype != th.float32:
                raise _lib.MorlB200Error(f"GemmMnMulti: job {i}: out must be fp32 [{gc}, {hc}] with unit column stride")
            if colsum is not None and (colsum.numel() < gc or colsum.dtype != th.float32 or not colsum.is_contiguous()):
                raise _lib.MorlB200Error(f"GemmMnMulti: job {i}: colsum must be a contiguous fp32 tensor of {gc} elements")
            arr[i] = _lib.MnJob(_ptr(g), g.stride(0), _ptr(sg), _ptr(h), h.stride(0), _ptr(sh), _ptr(out), _ptr(colsum), g.shape[2], int(gc), h.shape[2],
                                int(hc), out.stride(0))
        self._jobs, self._n = arr, len(jobs)
        self._keep = jobs
        nbytes = _lib.load().morl_gemm_mn_multi_workspace_bytes(arr, self._n, self.M)
        if nbytes == 0:
            raise _lib.MorlB200Error("GemmMnMulti: bad job shapes")
        self.workspace = th.empty((nbytes + 3) // 4, device=jobs[0][0].device, dtype=th.float32)

    def __call__(self):
        rc = _lib.load().morl_gemm_planes_mn_multi_f32(self.fmt, self._jobs, self._n, self.M, _ptr(self.workspace), _stream())
        _lib.check(rc, "morl_gemm_planes_mn_multi_f32")
        _count(2)


def colsum_planes(planes: th.Tensor, n_cols: int, out: Optional[th.Tensor] = None, workspace: Optional[th.Tensor] = None,
                  scale: Optional[th.Tensor] = None) -> th.Tensor:
    """Column sums over the rows and the planes, scale removed (bias gradients)."""
    fmt = fmt_of(planes)
    _, M, ld = planes.shape
    dev = planes.device
    out = th.empty(n_cols, device=dev, dtype=th.float32) if out is None else out
    ws = th.empty(296 * n_cols, device=dev, dtype=th.float32) if workspace is None else workspace
    rc = _lib.load().morl_colsum_planes(fmt, _ptr(planes), planes.stride(0), _ptr(scale), M, ld, n_cols, _ptr(out), _ptr(ws), _stream())
    _lib.check(rc, "morl_colsum_planes")
    _count(2)
    return out


def pairs_grad_reduce(planes: th.Tensor, B: int, W: int, workspace: Optional[th.Tensor] = None, dU: Optional[th.Tensor] = None,
                      dV: Optional[th.Tensor] = None, scale: Optional[th.Tensor] = None):
    """dU [B, H] and dV [W, H] from the planes of dL/dh1 [P, B*W, H] (gradient of relu(u[b] + v[j]) w.r.t. u and v), scale removed."""
    fmt = fmt_of(planes)
    _, M, H = planes.shape
    dev = planes.device
    dU = th.empty((B, H), device=dev, dtype=th.float32) if dU is None else dU
    dV = th.empty((W, H), device=dev, dtype=th.float32) if dV is None else dV
    ws = th.empty(296 * W * H, device=dev, dtype=th.float32) if workspace is None else workspace
    rc = _lib.load().morl_pairs_grad_reduce_planes(fmt, _ptr(planes), planes.stride(0), _ptr(scale), B, W, H, _ptr(dU), _ptr(dV), _ptr(ws), _stream())
    _lib.check(rc, "morl_pairs_grad_reduce_planes")
    _count(2)
    return dU, dV
