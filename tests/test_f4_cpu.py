"""f4 variants (gumbel sampling, affine re-parametrisation, orthogonal regularisation, materialised similarities): the
product's host logic -- `Codebook._run` with the variants on, the VectorQuantize / ResidualVQ glue -- on CPU with the
plain-torch statements of the C entry points (tests/cpu_kernels.py), against the fixtures recorded from the live
reference (tests/golden/make_golden_f4.py).  The kernels behind the entry points are tested on the GPU (test_gpu_f4.py)."""
import pytest
import torch

import f4_util as F
from test_orchestration_cpu import cpu_dense_ops, cpu_ops  # noqa: F401  (fixtures)


@pytest.mark.parametrize("name", F.names())
def test_f4_host_logic_matches_reference_fixture(name, cpu_dense_ops, monkeypatch):  # noqa: F811
    F.run_and_check(F.load(name), torch.device("cpu"), monkeypatch)
