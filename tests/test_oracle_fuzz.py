"""The numpy oracle against the C oracle on the same seeded random configurations the GPU fuzz test
uses (tests/fuzz.py): the two independent restatements must agree on every layout / mode /
concentration-driven combination, gas by gas and state row by state row, and the harness itself is exercised
on CPU."""
from dataclasses import dataclass
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import c_oracle as co
from oracle import ufair_oracle as o
from tests import fuzz


@dataclass
class _Spec:
    lo: float
    hi: float
    bins: int
    copies: int = 1


def _numpy_oracle_as_api(E, gp, tp, *, dt, stats, outputs, alpha_mode, t_mode, precision, conc_driven=None, **kw):
    assert precision == "f64"
    mask = sum(1 << g for g, f in enumerate(conc_driven or []) if f)
    out = o.oxfair(E, gp, tp, dt=dt, alpha_mode=fuzz._AM[alpha_mode], t_mode=o.T_END if t_mode == "end" else o.T_MID,
                   want_alpha=True, conc_driven=mask, **kw)
    if stats is not None:
        hist, mom = o.temperature_stats(out["T"], stats.lo, stats.hi, stats.bins)
        out["hist"], out["moments"] = hist.astype(np.int64), mom
    return SimpleNamespace(**out)


@pytest.mark.parametrize("seed", range(0, fuzz.N_CASES, 2))
def test_numpy_oracle_matches_c_oracle(seed):
    fuzz.check_case(seed, _numpy_oracle_as_api, _Spec, lambda x: x, np.asarray)
