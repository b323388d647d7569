"""Tabular front-end (SURVEY.md 8f-4, "DataFrame/CSV front-end"): emission scenarios in from CSV /
DataFrames, ensemble summaries out as DataFrames.  Pure host convenience around
:func:`fiveeqscm_b200.concentrations.run_ensemble`; nothing here touches the GPU.

Scenario table layout (long format), one row per (scenario, year):

    year, scenario, co2, ch4, n2o          # `scenario` optional (one scenario if absent)

Years must be equally spaced and identical across scenarios; units are the gas's own emission
units per year (GtC, MtCH4, MtN2O-N for the illustrative defaults in :mod:`.params`).
"""
from __future__ import annotations

from typing import Sequence

import numpy as np

from . import stats as _stats
from .params import GASES


def scenarios_from_frame(df, gases: Sequence[str] = GASES, year_col: str = "year", scenario_col: str = "scenario"):
    """(years [n_t], names [S], emissions [G][n_t][S] float64, dt) from a long-format table."""
    missing = [c for c in (year_col, *gases) if c not in df.columns]
    if missing:
        raise ValueError(f"scenario table lacks column(s) {missing}")
    if scenario_col in df.columns:
        names = list(dict.fromkeys(df[scenario_col].tolist()))
        groups = [df[df[scenario_col] == n] for n in names]
    else:
        names, groups = ["scenario"], [df]
    years = None
    cols = []
    for name, g in zip(names, groups):
        g = g.sort_values(year_col)
        y = g[year_col].to_numpy(dtype=np.float64)
        if years is None:
            years = y
        elif y.shape != years.shape or not np.array_equal(y, years):
            raise ValueError(f"scenario {name!r} does not cover the same years as {names[0]!r}")
        cols.append(np.stack([g[gas].to_numpy(dtype=np.float64) for gas in gases]))      # [G][n_t]
    if years.size == 0:
        raise ValueError("scenario table is empty")
    dt = 1.0
    if years.size > 1:
        steps = np.diff(years)
        dt = float(steps[0])
        if dt <= 0 or not np.allclose(steps, dt, rtol=0, atol=1e-9 * max(1.0, abs(dt))):
            raise ValueError("years must be strictly increasing and equally spaced")
    E = np.ascontiguousarray(np.stack(cols, axis=2))                                          # [G][n_t][S]
    if not np.all(np.isfinite(E)):
        raise ValueError("scenario table contains non-finite emissions")
    return years, names, E, dt


def scenarios_from_csv(path, gases: Sequence[str] = GASES, **kw):
    """:func:`scenarios_from_frame` on ``pandas.read_csv(path)``."""
    import pandas as pd
    return scenarios_from_frame(pd.read_csv(path), gases, **kw)


def summary_frame(result, years, pcts: Sequence[float] = (5.0, 17.0, 50.0, 83.0, 95.0), group_names=None):
    """Per-year ensemble summary of temperature from a result computed with ``stats=HistSpec(...)``
    (after the cross-GPU all-reduce, if any): mean, std, min, max and percentiles off the histogram.
    Grouped statistics (``stat_group=``) give a long frame, one block of years per group, led by a
    ``scenario`` column (grouped by scenario) or a ``group`` column (by labels) holding ``group_names[g]``
    (default: the group index).  A group's member count is its histogram row sum.  For a weighted run
    (``stat_weight=``) that row sum is the weight total: the ``members`` column then holds the weight total, and
    mean, std and percentiles are the weighted ones."""
    import pandas as pd
    if result.hist is None or result.moments is None or result.spec is None:
        raise ValueError("summary_frame needs a result computed with stats=HistSpec(...)")
    mom = _stats._np(result.moments)
    hist = _stats._np(result.hist)
    grouped = hist.ndim == 3
    if not grouped:
        hist, mom = hist[None], mom[None]
    n = hist.sum(axis=-1)                                                                    # [groups][n_t]
    if not np.all(n == n[:, :1]):
        raise ValueError("histogram rows count different numbers of members")
    with np.errstate(invalid="ignore", divide="ignore"):   # an empty group has no mean
        mean, std = _stats.mean_std(mom, n)
    p = _stats.percentiles(hist, result.spec.lo, result.spec.hi, pcts)
    n_grp, n_t = n.shape
    data = {"year": np.tile(np.asarray(years), n_grp), "members": n.ravel(), "T_mean": mean.ravel(),
            "T_std": std.ravel(), "T_min": mom[..., 2].ravel(), "T_max": mom[..., 3].ravel()}
    for j, q in enumerate(pcts):
        data[f"T_p{q:g}"] = p[..., j].ravel()
    if grouped:
        names = list(range(n_grp)) if group_names is None else list(group_names)
        if len(names) != n_grp:
            raise ValueError(f"group_names has {len(names)} entries for {n_grp} groups")
        col = "scenario" if getattr(result, "stat_group", None) == "scenario" else "group"
        data = {col: np.repeat(np.asarray(names, dtype=object), n_t), **data}
    return pd.DataFrame(data)


def member_frame(result, years, member: int = 0, gases: Sequence[str] = GASES):
    """One member's trajectory as a table: C_<gas>, RF_<gas>, (E_<gas>,) T per year."""
    import pandas as pd
    data = {"year": np.asarray(years)}
    for field, prefix in (("C", "C_"), ("RF", "RF_"), ("E", "E_"), ("alpha", "alpha_")):
        arr = getattr(result, field, None)
        if arr is not None:
            a = _stats._np(arr[:, :, member])
            for g, gas in enumerate(gases):
                data[prefix + gas] = a[g]
    if result.T is not None:
        data["T"] = _stats._np(result.T[:, member])
    return pd.DataFrame(data)
