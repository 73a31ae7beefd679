"""Dense layers of the weight-conditioned Q-network on the tcgen05 tensor cores (csrc/gemm_planes.cu).

``TCPairMlp`` runs the reference's ``mlp`` stack (common/networks.py:10-48: Linear -> ReLU ... -> Linear) for every
(observation b, weight vector j) pair of a minibatch without ever materialising fp32 activations in HBM:

    layer 1   : u = feats @ W1[:, :F]^T (B rows), v = wset @ W1[:, F:]^T + b1 (W rows)  -- one launch (morl_pair_layer1_uv_f32) --
                 h1[b*W + j] = relu(u[b] + v[j]) written straight into operand planes (morl_pairs_relu_split_planes);
    layers 2..: the 256-wide hidden layers of a pass as ONE chained launch (morl_gemm_chain_f32: a CTA pair takes its row tiles through
                 all layers, intermediate activations re-read from L2; both no-grad nets together) -- or, for other widths, one
                 morl_gemm_planes_f32 launch per layer (TMA -> tcgen05.mma -> TMEM -> epilogue, activation re-split fused in the epilogue);
                 the last layer writes fp32 Q-values (morl_qhead_gemm_f32 when it is <= 32 wide) or is consumed, together with the other
                 network's, by the fused head (morl_qhead_envelope_td_f32: Q never reaches HBM).

Operand formats (``fmt``): ``ops.FMT_F16X2`` (default; two fp16 planes of a power-of-two-scaled operand, three MMAs per product, 4 B per
element) or ``ops.FMT_BF16X3`` (three bf16 planes, six MMAs, 6 B per element, fp32 exponent range).  Scales of the f16x2 format, all
device-resident so a captured CUDA graph survives their changes:
    activations : fixed 2^1   (|h| < 32,752 representable; absolute resolution 2^-26)
    weights     : per matrix, from its own largest magnitude at every refresh (amax * s in [2^13, 2^14))
    gradients   : one per update, from the largest magnitude of dL/dQ (amax * s in [2, 4)).  dL/dh grows through the backward chain by
                  up to the gain of the network (a Q-function with returns of ~25 from unit inputs has a gain of that order per
                  layer product): the seed scale leaves 2^13 of head-room (a first choice of 2^7 overflowed 2,500 updates into the
                  hypervolume-parity run); elements below 2^-14 / s keep an ABSOLUTE accuracy of 2^-26 of the largest seed element,
                  far below the accumulation noise of the 65,536-row reductions they enter.
A value outside the fp16 range becomes Inf/NaN in the planes -- ReLU and the masks propagate NaN like torch's, so it reaches the loss and
the priorities, where ``Envelope.update`` checks for it -- and raises ``ops.plane_overflow_count()``.

The weight planes are refreshed with ``refresh_weights()`` after every optimiser step (one small launch per 16 matrices).

Hand-written backward for the training pass:
    G_L = dL/dQ;  dW_l = G_l^T H_{l-1} (MN-major split-K GEMM);  db_l = colsum(G_l);
    G_{l-1} = (G_l W_l) * [H_{l-1} > 0] (K-major GEMM with the ReLU mask fused in the epilogue; all layers as one chained launch);
    layer 1: dU = sum_j G_1, dV = sum_b G_1 (morl_pairs_grad_reduce_planes), dW1 = [dU^T feats | dV^T wset], db1 = sum_j dV
             (morl_pair_layer1_grad_f32).
No library (ATen / cuBLAS) kernel runs anywhere in forward or backward.
"""

from __future__ import annotations

import os
from typing import List, Optional

import torch as th
from torch import nn

from . import ops

_SNAKE = os.environ.get("MORL_TC_SNAKE", "1") == "1"          # alternate the GEMM tile order between chained layers
_CHAIN = os.environ.get("MORL_GEMM_CHAIN", "1") == "1"        # hidden layers 2.. of a pass as ONE chained launch (+10 % on the update; =0: one launch per layer)
_CHAIN_BWD = os.environ.get("MORL_GEMM_CHAIN_BWD", "1") == "1"  # ... and the 256-wide dX products of the backward pass (+2.7 %; =0: per-layer launches)
_NARROW_HEAD = os.environ.get("MORL_NARROW_HEAD", "1") == "1"  # output layer through morl_qhead_gemm_f32 (19.7 us against 26 us in the update; =0: general kernel)
_DEFAULT_FMT = ops.FMT_BF16X3 if os.environ.get("MORL_TC_FMT", "f16x2") == "bf16x3" else ops.FMT_F16X2

ACT_SCALE = 2.0        # f16x2 activations: |h| < 32,752 representable
W_TARGET_EXP = 14      # f16x2 weights: amax * scale in [2^13, 2^14) (the matrix is known when it is split: it cannot overflow)
G_TARGET_EXP = 2       # f16x2 gradients: amax(dL/dQ) * scale in [2, 4): 2^13 of growth head-room through the backward chain


def _pad(n: int, m: int) -> int:
    return (n + m - 1) // m * m


class TCPairMlp:
    """Static plan (buffers + weight planes) for one nn.Sequential MLP and a fixed number of pair rows."""

    @staticmethod
    def supported(net: nn.Sequential, fmt: int = _DEFAULT_FMT) -> bool:
        mods = list(net)
        lin = [m for m in mods if isinstance(m, nn.Linear)]
        if len(lin) < 2 or any(not isinstance(m, (nn.Linear, nn.ReLU)) for m in mods):
            return False
        if not all(isinstance(mods[2 * i], nn.Linear) for i in range(len(lin))):
            return False
        hidden = [l.out_features for l in lin[:-1]]
        kmul = 64 if fmt == ops.FMT_F16X2 else 32  # K extent of one pipeline stage
        return all(h % kmul == 0 and h <= 256 for h in hidden) and lin[-1].out_features <= 256

    @staticmethod
    def trainable_supported(net: nn.Sequential, n_w: int, fmt: int = _DEFAULT_FMT) -> bool:
        """The hand-written backward additionally needs equal hidden widths (multiples of 64) and at most 64 weight vectors."""
        if not TCPairMlp.supported(net, fmt):
            return False
        hidden = {m.out_features for m in list(net)[:-1] if isinstance(m, nn.Linear)}
        return len(hidden) == 1 and next(iter(hidden)) % 64 == 0 and n_w <= 64

    def __init__(self, net: nn.Sequential, feat_dim: int, n_obs: int, n_w: int, share_weights_with: Optional["TCPairMlp"] = None,
                 trainable: bool = False, fmt: Optional[int] = None, split_acc: bool = False):
        self.net = net
        # forward GEMMs: one double-buffered accumulator (default) or split leading / correction accumulators (2.5x smaller systematic
        # error of the truncating tensor-core accumulation, ~20 % slower per layer); the backward dX GEMMs always use one accumulator
        self.split_acc = bool(split_acc)
        self.lin: List[nn.Linear] = [m for m in net if isinstance(m, nn.Linear)]
        self.feat_dim = feat_dim
        self.B, self.W = n_obs, n_w
        self.fmt = fmt = (share_weights_with.fmt if share_weights_with is not None else _DEFAULT_FMT) if fmt is None else fmt
        if not TCPairMlp.supported(net, fmt):
            raise ops._lib.MorlB200Error("TCPairMlp: unsupported network (Linear/ReLU stack with hidden widths that are multiples of 64 (f16x2) or "
                                         "32 (bf16x3) and <= 256)")
        dev = self.lin[0].weight.device
        M = n_obs * n_w
        scaled = fmt == ops.FMT_F16X2
        self.h = [ops.empty_planes(fmt, M, l.out_features, dev) for l in self.lin[:-1]]
        self.s_act = ops.scale_tensor(ACT_SCALE, dev) if scaled else None
        if share_weights_with is not None:
            if share_weights_with.fmt != fmt:
                raise ops._lib.MorlB200Error("TCPairMlp: plans sharing weight planes must use the same operand format")
            self.wp, self.s_w = share_weights_with.wp, share_weights_with.s_w  # same network: one set of weight planes, refreshed once per step
        else:
            self.wp = [ops.empty_planes(fmt, _pad(l.out_features, 32), l.in_features, dev) for l in self.lin[1:]]
            self.s_w = [ops.scale_tensor(1.0, dev) if scaled else None for _ in self.lin[1:]]
        self.q = th.empty((M, self.lin[-1].out_features), device=dev, dtype=th.float32)
        self._chain = self._gchain = self._gbufs = self._mn_multi = None
        self.trainable = trainable
        if trainable:
            if n_w > 64:
                raise ops._lib.MorlB200Error("TCPairMlp backward supports at most 64 weight vectors per minibatch")
            out = self.lin[-1].out_features
            self.ld_last = _pad(out, 64)
            hid = max(l.out_features for l in self.lin[:-1])
            self.g_last = ops.empty_planes(fmt, M, self.ld_last, dev)
            self.g = [ops.empty_planes(fmt, M, hid, dev) for _ in range(2)]
            # relu'(H_k) as bits (32 B per row), written by the forward pass, read by the dX GEMMs instead of the 512-B activation rows
            self.hbits = [ops.empty_relu_bits(M, dev) for _ in self.lin[:-1]]
            self.s_g = ops.scale_tensor(1.0, dev) if scaled else None
            self.ws_amax = th.zeros(2, device=dev, dtype=th.int32)
            # transposed weight planes W_l^T [P, in_l, K = padded out_l] for the dX products
            self.wtp = []
            for k, l in enumerate(self.lin[1:], start=1):
                kdim = self.ld_last if k == len(self.lin) - 1 else l.out_features
                self.wtp.append(ops.empty_planes(fmt, _pad(l.in_features, 32), kdim, dev))
            self.ws_mn = ops.gemm_mn_workspace(M, 256, 256, dev)
            self.ws_red = th.empty(296 * max(n_w * hid, 256), device=dev, dtype=th.float32)
            first = self.lin[0]
            self.ws_l1 = ops.pair_layer1_grad_workspace(feat_dim, first.in_features - feat_dim, first.out_features, dev)
            self.dU = th.empty((n_obs, first.out_features), device=dev, dtype=th.float32)
            self.dV = th.empty((n_w, first.out_features), device=dev, dtype=th.float32)

    # ------------------------------------------------------------------------------------------------ weight planes
    def _texp(self):
        return W_TARGET_EXP if self.fmt == ops.FMT_F16X2 else None

    def _weight_jobs(self):
        return [(l.weight.detach(), wp, False, s, self._texp()) for l, wp, s in zip(self.lin[1:], self.wp, self.s_w)]

    def _transposed_jobs(self):
        # same matrix, same amax, same scale: the transposed job re-derives (and re-publishes) the value of the plain one
        return [(l.weight.detach(), wt, True, s, self._texp()) for l, wt, s in zip(self.lin[1:], self.wtp, self.s_w)]

    def refresh_weights(self):
        """Re-split the (fp32) weights of layers 2.. into operand planes; call after every optimiser step / target sync."""
        ops.split_planes_multi(self._weight_jobs(), self.fmt)

    def refresh_transposed_weights(self):
        ops.split_planes_multi(self._transposed_jobs(), self.fmt)

    @staticmethod
    def refresh_many(plans, transposed_of=()):
        """All weight planes of several plans (and the transposed planes of the trainable ones) in a single launch per 16 matrices.
        Plans sharing their planes (``share_weights_with``) are split once."""
        jobs, seen = [], set()
        fmt = plans[0].fmt
        for p in plans:
            if p.fmt != fmt:
                raise ops._lib.MorlB200Error("TCPairMlp.refresh_many: mixed operand formats")
            if id(p.wp) not in seen:
                seen.add(id(p.wp))
                jobs += p._weight_jobs()
        for p in transposed_of:
            jobs += p._transposed_jobs()
            p._wt_fresh = True
        for i in range(0, len(jobs), 16):
            ops.split_planes_multi(jobs[i:i + 16], fmt)

    # ------------------------------------------------------------------------------------------------ forward / backward
    @th.no_grad()
    def forward_pairs(self, feats: th.Tensor, wset: th.Tensor) -> th.Tensor:
        """feats [B, F], wset [W, D] -> Q [B*W, out] (fp32, row b*W + j).  Uses the planes of the last refresh_weights()."""
        first = self.lin[0]
        if feats.shape[1] != self.feat_dim or first.in_features != self.feat_dim + wset.shape[1]:
            raise ops._lib.MorlB200Error(f"TCPairMlp: feats {tuple(feats.shape)} / wset {tuple(wset.shape)} do not match the first layer ({first.in_features} inputs)")
        a = self.forward_hidden(feats, wset, _checked=True)
        n = len(self.lin)
        last = self.lin[-1]
        wp_last = self.wp[n - 2]
        if _NARROW_HEAD and not self.split_acc and wp_last.shape[1] == 32 and ops.qhead_gemm_supported(self.fmt, a.shape[1], last.out_features, a.shape[2]):
            # narrow output layer: weight planes resident in shared memory, deep activation ring (bit-identical to the general kernel)
            return ops.qhead_gemm(a, wp_last, last.out_features, last.bias.detach(), out=self.q, a_scale=self.s_act, w_scale=self.s_w[n - 2],
                                  reverse_tiles=_SNAKE and bool((n - 1) & 1))
        q, _ = ops.gemm_planes(a, wp_last, last.out_features, bias=last.bias, relu=False, out_f32=True, c_f32=self.q,
                               reverse_tiles=_SNAKE and bool((n - 1) & 1), a_scale=self.s_act, b_scale=self.s_w[n - 2], split_acc=self.split_acc)
        return q

    @th.no_grad()
    def forward_hidden(self, feats: th.Tensor, wset: th.Tensor, _checked: bool = False) -> th.Tensor:
        """Layers 1 .. n-1: returns the planes of the LAST hidden activation [P, B*W, H] (the operand of the output layer, which
        :func:`ops.qhead_envelope_td` consumes together with the other network's)."""
        first = self.lin[0]
        if not _checked and (feats.shape[1] != self.feat_dim or first.in_features != self.feat_dim + wset.shape[1]):
            raise ops._lib.MorlB200Error(f"TCPairMlp: feats {tuple(feats.shape)} / wset {tuple(wset.shape)} do not match the first layer ({first.in_features} inputs)")
        u, v = ops.pair_layer1_uv(feats, wset, first.weight.detach(), first.bias.detach())  # one launch (csrc/pair_layer1.cu)
        hb = self.hbits if self.trainable else [None] * len(self.h)
        a = ops.pairs_relu_split(u, v, out=self.h[0], scale=self.s_act, relu_bits_out=hb[0])
        n = len(self.lin)
        if self.chain_supported():
            if self._chain is None:
                self._chain = TCPairMlp.make_chain([self])
            self._chain()  # hidden layers 2.. in one persistent launch (intermediate activations re-read from L2)
            return self.h[-1]
        for k in range(1, n - 1):
            l = self.lin[k]
            # alternate the tile order: a layer starts on the rows its producer wrote last (L2-resident)
            _, a = ops.gemm_planes(a, self.wp[k - 1], l.out_features, bias=l.bias, relu=True, out_f32=False, out_planes=True, c_planes=self.h[k],
                                   reverse_tiles=_SNAKE and bool(k & 1), a_scale=self.s_act, b_scale=self.s_w[k - 1], c_scale=self.s_act,
                                   split_acc=self.split_acc, relu_bits_out=hb[k])
        return a

    # ------------------------------------------------------------------------------------------------ chained hidden layers
    def chain_supported(self) -> bool:
        """Hidden layers 2.. as ONE launch (ops.GemmChain): 256-wide square layers, single accumulator, at least two 128-row tiles."""
        hid = [l.out_features for l in self.lin[:-1]]
        return (_CHAIN and not self.split_acc and len(hid) >= 2 and all(h == 256 for h in hid)
                and ops.gemm_chain_supported(self.fmt, self.B * self.W, 256))

    def layer1(self, feats: th.Tensor, wset: th.Tensor) -> th.Tensor:
        """Layer 1 only (separable first layer): h1 planes (+ ReLU bits when trainable)."""
        first = self.lin[0]
        u, v = ops.pair_layer1_uv(feats, wset, first.weight.detach(), first.bias.detach())
        hb = self.hbits if self.trainable else [None] * len(self.h)
        return ops.pairs_relu_split(u, v, out=self.h[0], scale=self.s_act, relu_bits_out=hb[0])

    def chain_spec(self):
        """(activations, weight planes, biases, weight scales, ReLU bit tensors) of the hidden layers 2.. for ops.GemmChain."""
        n = len(self.lin)
        hb = self.hbits if self.trainable else [None] * len(self.h)
        return (list(self.h), [self.wp[k - 1] for k in range(1, n - 1)], [self.lin[k].bias for k in range(1, n - 1)],
                [self.s_w[k - 1] for k in range(1, n - 1)], [hb[k] for k in range(1, n - 1)])

    @staticmethod
    def make_chain(plans):
        """One chained launch for the hidden layers 2.. of one plan, or of two plans of equal shape (the two no-grad passes)."""
        specs = [p.chain_spec() for p in plans]
        return ops.GemmChain([sp[0] for sp in specs], [sp[1] for sp in specs], [sp[2] for sp in specs], [sp[3] for sp in specs],
                             [sp[4] for sp in specs], act_scale=plans[0].s_act)

    def head_operands(self):
        """(weight planes [P, 32, K], weight scale, bias) of the output layer, or None if it is wider than 32 columns."""
        last = self.lin[-1]
        wp = self.wp[len(self.lin) - 2]
        if wp.shape[1] != 32:
            return None
        return wp, self.s_w[len(self.lin) - 2], last.bias

    @th.no_grad()
    def backward(self, feats: th.Tensor, wset: th.Tensor, dq: th.Tensor, grads_out: Optional[List[th.Tensor]] = None, after_gemms=None):
        """Gradients of all Linear parameters given dL/dQ [B*W, out]; uses the activations of the last forward_pairs().
        ``grads_out`` (weight, bias per Linear, in order) receives them in place -- the persistent ``.grad`` buffers of the update.
        ``after_gemms`` (callable, optional) is invoked once the last persistent tensor-core GEMM has been enqueued: the place to fork side
        work that must not take an SM away from those one-CTA-per-SM kernels (the layer-1 reductions that follow are ordinary grids)."""
        n = len(self.lin)
        grads = [None] * (2 * n) if grads_out is None else list(grads_out)
        if getattr(self, "_wt_fresh", False):
            self._wt_fresh = False  # refreshed together with the forward planes of this step (refresh_many)
        else:
            self.refresh_transposed_weights()
        if self.s_g is not None:
            ops.amax_scale(dq, G_TARGET_EXP, self.s_g, self.ws_amax)  # this update's gradient scale
        G = ops.split_planes(dq, self.fmt, rows_pad=dq.shape[0], ldp=self.ld_last, out=self.g_last, scale=self.s_g)
        if _CHAIN_BWD and self.chain_supported() and n >= 4:
            return self._backward_chained(feats, wset, G, grads, after_gemms)
        for k in range(n - 1, 0, -1):
            l = self.lin[k]
            # dW_k = G_k^T H_{k-1} and db_k = colsum(G_k) in one pass over the G planes
            if grads[2 * k + 1] is None:
                grads[2 * k + 1] = th.empty(l.out_features, device=dq.device, dtype=th.float32)
            grads[2 * k] = ops.gemm_planes_mn(G, l.out_features, self.h[k - 1], l.in_features, out=grads[2 * k], workspace=self.ws_mn,
                                              colsum=grads[2 * k + 1], g_scale=self.s_g, h_scale=self.s_act)
            # G_{k-1} = (G_k . W_k) masked by relu'(H_{k-1}), kept at the gradient scale
            _, G = ops.gemm_planes(G, self.wtp[k - 1], l.in_features, relu_bits_in=self.hbits[k - 1], out_f32=False, out_planes=True,
                                   c_planes=self.g[k & 1], reverse_tiles=_SNAKE and bool(k & 1), a_scale=self.s_g, b_scale=self.s_w[k - 1],
                                   c_scale=self.s_g, split_acc=False)  # gradients: Adam is invariant to the ~2e-6 uniform shrinkage
        if after_gemms is not None:
            after_gemms()
        dU, dV = ops.pairs_grad_reduce(G, self.B, self.W, workspace=self.ws_red, dU=self.dU, dV=self.dV, scale=self.s_g)
        grads[0], grads[1] = ops.pair_layer1_grad(dU, dV, feats, wset, dW1=grads[0], db1=grads[1], workspace=self.ws_l1)
        return grads

    def _backward_chained(self, feats, wset, G, grads, after_gemms):
        """Backward with the 256-wide dX products as ONE chained launch: G_{n-2} from the (narrow) output layer as before, then
        G_{k-1} = (G_k . W_k) * relu'(H_{k-1}) for k = n-2 .. 1 in one persistent kernel (each G_k in its own buffer: the weight-gradient
        products read them afterwards), then the n-1 weight-gradient products as multi-job launches (ops.GemmMnMulti), at most
        MN_MAX_JOBS products per launch."""
        n = len(self.lin)
        dev = G.device
        if self._gchain is None:
            M, hid = self.B * self.W, self.lin[1].in_features
            self._gbufs = [ops.empty_planes(self.fmt, M, hid, dev) for _ in range(n - 1)]  # dL/d(output of lin[n-2]), ..., dL/d(output of lin[0])
            # chain input = the planes of dL/dQ (ld_last wide: the first job reduces over ld_last columns only), outputs the n - 1 hidden gradients
            ks = list(range(n - 1, 0, -1))  # layers whose dX product is in the chain: the narrow output layer first
            self._gchain = ops.GemmChain([[self.g_last] + self._gbufs], [[self.wtp[k - 1] for k in ks]], None, [[self.s_w[k - 1] for k in ks]], None,
                                         act_scale=self.s_g, relu=False, bits_in=[[self.hbits[k - 1] for k in ks]], k_first=self.ld_last)
        for k in range(1, n):
            if grads[2 * k] is None:
                grads[2 * k] = th.empty((self.lin[k].out_features, self.lin[k].in_features), device=dev, dtype=th.float32)
            if grads[2 * k + 1] is None:
                grads[2 * k + 1] = th.empty(self.lin[k].out_features, device=dev, dtype=th.float32)
        self._gchain()  # all n - 1 dX products (the narrow one of the output layer included) in one launch
        key = tuple(grads[i].data_ptr() for i in range(2, 2 * n))
        if self._mn_multi is None or self._mn_multi[0] != key:
            # dL/dh_k is _gbufs[n - 2 - k]; the chain writes _gbufs[n - 3] (dW of lin[1]) last, so that product goes first (part of its G may
            # still be in L2), the narrow output layer last
            jobs = [(self._gbufs[n - 2 - k], self.lin[k].out_features, self.h[k - 1], self.lin[k].in_features, grads[2 * k], grads[2 * k + 1], self.s_g,
                     self.s_act) for k in range(1, n - 1)]
            jobs.append((G, self.lin[n - 1].out_features, self.h[n - 2], self.lin[n - 1].in_features, grads[2 * (n - 1)], grads[2 * (n - 1) + 1], self.s_g,
                         self.s_act))
            per = ops._lib.MN_MAX_JOBS
            self._mn_multi = (key, [ops.GemmMnMulti(jobs[i:i + per]) for i in range(0, len(jobs), per)])
        for plan in self._mn_multi[1]:
            plan()
        return self._backward_tail(feats, wset, grads, after_gemms)

    def _backward_tail(self, feats, wset, grads, after_gemms):
        """After the last tensor-core GEMM of the chained backward: fork the side work, then the layer-1 gradients."""
        if after_gemms is not None:
            after_gemms()
        dU, dV = ops.pairs_grad_reduce(self._gbufs[len(self.lin) - 2], self.B, self.W, workspace=self.ws_red, dU=self.dU, dV=self.dV, scale=self.s_g)
        grads[0], grads[1] = ops.pair_layer1_grad(dU, dV, feats, wset, dW1=grads[0], db1=grads[1], workspace=self.ws_l1)
        return grads


class TCPairMlpFn(th.autograd.Function):
    """Q = mlp(pairs(feats, wset)) with the dense layers on the tcgen05 tensor cores, forward and backward."""

    @staticmethod
    def forward(ctx, plan: TCPairMlp, feats: th.Tensor, wset: th.Tensor, *params):
        q = plan.forward_pairs(feats, wset)
        ctx.plan = plan
        ctx.save_for_backward(feats, wset)
        return q

    @staticmethod
    def backward(ctx, dq):
        feats, wset = ctx.saved_tensors
        grads = ctx.plan.backward(feats, wset, dq.contiguous())
        return (None, None, None, *grads)
