"""The weight-gradient products (ops.gemm_planes_mn) against the recorded bytes of the per-layer kernel they replaced
(tests/golden/mn_per_layer_digests.json, written by tests/golden/make_golden_mn_digests.py): every dW and db of every case must be
bit-identical.  tests/test_gemm_mn_multi_gpu.py checks the multi-job launch against the one-job call, so both stay pinned to the old kernel."""

import json

import pytest

from tests.golden import make_golden_mn_digests as mk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def recorded():
    with open(mk.PATH) as f:
        return json.load(f)


def test_every_case_is_recorded(recorded):
    assert sorted(recorded) == sorted(mk.case_ids())


@pytest.mark.parametrize("case_id", mk.case_ids())
def test_outputs_equal_the_per_layer_kernel(cuda, recorded, case_id):
    inputs, outputs = mk.compute(case_id)
    want = recorded[case_id]
    assert inputs == want["inputs"], f"{case_id}: the input planes differ from the recorded ones (input generation drifted, not the kernel)"
    assert outputs == want["outputs"], f"{case_id}: outputs differ from the per-layer kernel's recorded bytes"
