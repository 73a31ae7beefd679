"""Recorded outputs of the per-layer weight-gradient kernel, as SHA-256 digests:
    python tests/golden/make_golden_mn_digests.py   ->  tests/golden/mn_per_layer_digests.json
(needs a CUDA device and the built library)

The cases are the seeded inputs of tests/test_gemm_gpu.py::test_gemm_mn_weight_gradient (plain, transposed and with the fused column
sums) and every job of every case of tests/test_gemm_mn_multi_gpu.py.  For each case the file holds the digests of the input planes and
of the bytes of every dW and db that ``ops.gemm_planes_mn`` returned.  The recorded digests were written by the per-layer split-K
kernel that a one-job launch of the multi-job kernel has since replaced; tests/test_gemm_mn_golden_gpu.py recomputes every case and
demands the same bytes, so the replacement stays bit-identical to it."""

import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

PATH = os.path.join(HERE, "mn_per_layer_digests.json")
FMT_NAMES = {0: "bf16x3", 1: "f16x2"}

# tests/test_gemm_gpu.py::test_gemm_mn_weight_gradient: (M, g_cols, h_cols)
GEMM_SHAPES = [(65536, 256, 256), (5000, 256, 256), (4096, 24, 256), (1000, 128, 64), (333, 256, 192)]
# tests/test_gemm_mn_multi_gpu.py: (name, M, [(g_cols, h_cols, ldg) per job], seed, colsum)
MULTI_CASES = [
    ("update", 65536, [(256, 256, 256), (256, 256, 256), (256, 256, 256), (24, 256, 64)], 1, True),
    ("single", 5000, [(256, 256, 256)], 2, True),
    ("mixed333", 333, [(256, 192, 256), (24, 256, 64)], 333, True),
    ("mixed1000", 1000, [(128, 64, 128), (256, 192, 256), (24, 256, 64), (64, 128, 64)], 1000, True),
    ("mixed4097", 4097, [(200, 256, 256), (24, 64, 64), (256, 128, 256)], 4097, True),
    ("nocolsum", 2048, [(256, 256, 256), (24, 256, 64)], 3, False),
]


def case_ids():
    ids = [f"gemm-{FMT_NAMES[f]}-{M}x{gc}x{hc}" for f in (1, 0) for M, gc, hc in GEMM_SHAPES]
    return ids + [f"multi-{FMT_NAMES[f]}-{c[0]}" for f in (1, 0) for c in MULTI_CASES]


def _sha(t):
    import torch as th

    return hashlib.sha256(t.contiguous().cpu().view(-1).view(th.uint8).numpy().tobytes()).hexdigest()  # (bf16 has no numpy type)


def _gemm_case(fmt, M, gc, hc):
    """The inputs and calls of test_gemm_mn_weight_gradient."""
    import torch as th

    from morl_baselines_b200 import ops

    dev = th.device("cuda:0")
    g_ = th.Generator(device=dev).manual_seed(M + gc)
    G = th.randn(M, gc, device=dev, generator=g_) * 1e-4
    H = th.randn(M, hc, device=dev, generator=g_).clamp_min(0)
    scaled = fmt == ops.FMT_F16X2
    sg, sh = (ops.scale_tensor(2.0**20, dev), ops.scale_tensor(8.0, dev)) if scaled else (None, None)
    Gp = ops.split_planes(G, fmt, ldp=(gc + 63) // 64 * 64, scale=sg)
    Hp = ops.split_planes(H, fmt, ldp=(hc + 63) // 64 * 64, scale=sh)
    inputs = {"G": _sha(Gp), "H": _sha(Hp)}
    dW = ops.gemm_planes_mn(Gp, gc, Hp, hc, g_scale=sg, h_scale=sh)
    dWt = ops.gemm_planes_mn(Gp, gc, Hp, hc, transpose_out=True, g_scale=sg, h_scale=sh)
    cs = th.full((gc,), float("nan"), device=dev)
    dW2 = ops.gemm_planes_mn(Gp, gc, Hp, hc, colsum=cs, g_scale=sg, h_scale=sh)
    return inputs, {"dW": _sha(dW), "dWt": _sha(dWt), "dW_colsum": _sha(dW2), "db": _sha(cs)}


def _multi_case(fmt, M, shapes, seed, colsum):
    """The operands of tests/test_gemm_mn_multi_gpu.py::_operands and the per-product calls of its _check."""
    import torch as th

    from morl_baselines_b200 import ops

    dev = th.device("cuda")
    g = th.Generator(device=dev).manual_seed(seed)
    sg = ops.scale_tensor(2.0**20, dev) if fmt == ops.FMT_F16X2 else None
    sh = ops.scale_tensor(2.0, dev) if fmt == ops.FMT_F16X2 else None
    inputs, outputs = {}, {}
    for i, (gc, hc, ldg) in enumerate(shapes):
        G = th.randn(M, gc, device=dev, generator=g) * 1e-4
        H = th.randn(M, hc, device=dev, generator=g).clamp_min(0)
        Gp = ops.split_planes(G, fmt, ldp=ldg, scale=sg)
        Hp = ops.split_planes(H, fmt, ldp=(hc + 63) // 64 * 64, scale=sh)
        inputs[f"G{i}"], inputs[f"H{i}"] = _sha(Gp), _sha(Hp)
        cs = th.empty(gc, device=dev) if colsum else None
        outputs[f"dW{i}"] = _sha(ops.gemm_planes_mn(Gp, gc, Hp, hc, colsum=cs, g_scale=sg, h_scale=sh))
        if colsum:
            outputs[f"db{i}"] = _sha(cs)
    return inputs, outputs


def compute(case_id):
    """(input digests, output digests) of one case, computed by the current ops.gemm_planes_mn."""
    kind, fmt_name, rest = case_id.split("-", 2)
    fmt = {v: k for k, v in FMT_NAMES.items()}[fmt_name]
    if kind == "gemm":
        M, gc, hc = (int(x) for x in rest.split("x"))
        return _gemm_case(fmt, M, gc, hc)
    _, M, shapes, seed, colsum = next(c for c in MULTI_CASES if c[0] == rest)
    return _multi_case(fmt, M, shapes, seed, colsum)


def main():
    out = {}
    for cid in case_ids():
        inputs, outputs = compute(cid)
        assert compute(cid) == (inputs, outputs), f"{cid}: two runs gave different bytes"
        out[cid] = {"inputs": inputs, "outputs": outputs}
    with open(PATH, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(f"wrote {PATH}: {len(out)} cases")


if __name__ == "__main__":
    main()
