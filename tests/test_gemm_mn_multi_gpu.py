"""GPU tests of the multi-job weight-gradient launch (ops.GemmMnMulti, csrc/gemm_planes.cu: gemm_planes_mn_multi_kernel): every dW and
db must be BIT-identical to the one-job ops.gemm_planes_mn call on that product alone, i.e. dealing the units of several jobs together
changes no bit.  tests/test_gemm_mn_golden_gpu.py pins the one-job results to the recorded outputs of the former per-layer kernel."""

import pytest
import torch as th

pytestmark = pytest.mark.gpu

FMTS = [pytest.param(1, id="f16x2"), pytest.param(0, id="bf16x3")]


def _operands(fmt, M, shapes, seed):
    """Plane tensors of G [M, gc] (ld a multiple of 64) and H [M, hc] per (gc, hc, ldg) job, with the update's scales."""
    from morl_baselines_b200 import ops

    dev = th.device("cuda")
    g = th.Generator(device=dev).manual_seed(seed)
    sg = ops.scale_tensor(2.0**20, dev) if fmt == ops.FMT_F16X2 else None
    sh = ops.scale_tensor(2.0, dev) if fmt == ops.FMT_F16X2 else None
    ops_ = []
    for gc, hc, ldg in shapes:
        G = th.randn(M, gc, device=dev, generator=g) * 1e-4
        H = th.randn(M, hc, device=dev, generator=g).clamp_min(0)
        ops_.append((ops.split_planes(G, fmt, ldp=ldg, scale=sg), gc, ops.split_planes(H, fmt, ldp=(hc + 63) // 64 * 64, scale=sh), hc))
    return ops_, sg, sh


def _check(fmt, M, shapes, seed, colsum=True):
    from morl_baselines_b200 import ops

    jobs_in, sg, sh = _operands(fmt, M, shapes, seed)
    ref, jobs = [], []
    for Gp, gc, Hp, hc in jobs_in:
        cs = th.empty(gc, device="cuda") if colsum else None
        ref.append((ops.gemm_planes_mn(Gp, gc, Hp, hc, colsum=cs, g_scale=sg, h_scale=sh), cs))
        out = th.full((gc, hc), float("nan"), device="cuda")
        cs2 = th.full((gc,), float("nan"), device="cuda") if colsum else None
        jobs.append((Gp, gc, Hp, hc, out, cs2, sg, sh))
    plan = ops.GemmMnMulti(jobs)
    for _ in range(2):  # a second call on the same workspace gives the same result
        plan()
        th.cuda.synchronize()
        for (dW, cs), job in zip(ref, jobs):
            assert th.equal(job[4], dW)
            if colsum:
                assert th.equal(job[5], cs)


@pytest.mark.parametrize("fmt", FMTS)
def test_update_job_list_is_bit_identical(fmt):
    """The backward pass of an update: three 256 x 256 hidden layers and the 24-wide output layer (G planes 64 wide) over 65,536 rows."""
    _check(fmt, 65536, [(256, 256, 256), (256, 256, 256), (256, 256, 256), (24, 256, 64)], seed=1)


@pytest.mark.parametrize("fmt", FMTS)
def test_single_job_is_bit_identical(fmt):
    _check(fmt, 5000, [(256, 256, 256)], seed=2)


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("M,shapes", [
    (333, [(256, 192, 256), (24, 256, 64)]),                               # M not a multiple of 32 or of the split size
    (1000, [(128, 64, 128), (256, 192, 256), (24, 256, 64), (64, 128, 64)]),  # four jobs of mixed widths
    (4097, [(200, 256, 256), (24, 64, 64), (256, 128, 256)]),              # partial column tile, narrow H
])
def test_mixed_jobs_are_bit_identical(fmt, M, shapes):
    _check(fmt, M, shapes, seed=M)


@pytest.mark.parametrize("fmt", FMTS)
def test_without_column_sums(fmt):
    _check(fmt, 2048, [(256, 256, 256), (24, 256, 64)], seed=3, colsum=False)


def test_unsupported_arguments_raise():
    from morl_baselines_b200 import _lib, ops

    (Gp, gc, Hp, hc), = _operands(ops.FMT_F16X2, 512, [(256, 256, 256)], seed=4)[0]
    out = th.empty(gc, hc, device="cuda")
    with pytest.raises(_lib.MorlB200Error):  # transposed output
        ops.GemmMnMulti([(Gp, gc, Hp, hc, th.empty(hc, gc, device="cuda").t(), None, None, None)])
    with pytest.raises(_lib.MorlB200Error):  # more than MORL_MN_MAX_JOBS products
        ops.GemmMnMulti([(Gp, gc, Hp, hc, out, None, None, None)] * (_lib.MN_MAX_JOBS + 1))
    with pytest.raises(_lib.MorlB200Error):  # the reduction stores four columns at a time
        ops.GemmMnMulti([(Gp, gc, Hp, 62, th.empty(gc, 62, device="cuda"), None, None, None)])()
