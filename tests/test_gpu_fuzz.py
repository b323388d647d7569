"""The CUDA path (through the C ABI) on the seeded random configurations of tests/fuzz.py, in FP64 and in FP32."""
import pytest

from fiveeqscm_b200 import _abi
from tests import fuzz
from tests.util import to_dev, to_np

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    from fiveeqscm_b200 import concentrations as c
    _abi.lib()
    return c


def _run(api):
    import torch

    def run(*a, **kw):
        r = api.run_ensemble(*a, **kw)
        torch.cuda.synchronize()
        return r
    return run


@pytest.mark.parametrize("seed", range(fuzz.N_CASES))
def test_random_configuration_matches_oracle(api, seed):
    fuzz.check_case(seed, _run(api), api.HistSpec, to_dev, to_np)


@pytest.mark.parametrize("seed", range(fuzz.N_CASES))
def test_random_configuration_fp32_matches_oracle(api, seed):
    """The same configurations on the FP32 instantiations: T within 1e-4 K, each gas's C within 2e-5."""
    fuzz.check_case(seed, _run(api), api.HistSpec, to_dev, to_np, precision="f32")
