"""-m gpu: the rebalancer kernel against the CPU oracle where its fast paths end (inputs from
tests/rebalance_cases.py): hosts past 64 items, decisions with more than 64 victims or victims of more
than 63 users, preempted synthetic tasks, gpu / disk / lifetime constraints, more than four groups or
more than 64 distinct attribute values, spare-only hosts, exact eligibility edges.  Every case also runs
off the exact grid, where the re-folds take their serial forms."""
import os

import numpy as np
import pytest

from cook_b200 import abi, traces
from rebalance_cases import all_cases, crowded_hosts, mass_preemption

pytestmark = pytest.mark.gpu

CASES = all_cases()


def _bits(x):
    return np.array(x, np.float64).view(np.int64).tolist()


def _same_decisions(got, want):
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert (g["pending_idx"], g["host"]) == (w["pending_idx"], w["host"]), k
        assert g["victims"] == w["victims"], k
        assert _bits([g[f] for f in ("dru", "mem", "cpus", "gpus")]) == _bits([w[f] for f in ("dru", "mem", "cpus", "gpus")]), k


def _same_trace(tg, to):
    _same_decisions(tg["decisions"], to["decisions"])
    assert tg["below_quota"] == to["below_quota"]
    assert _bits(np.nan_to_num(tg["pending_dru"], nan=-1.0)) == _bits(np.nan_to_num(to["pending_dru"], nan=-1.0))
    assert tg["order"] == to["order"]
    assert _bits(tg["order_dru"]) == _bits(to["order_dru"])
    assert tg["spare"].keys() == to["spare"].keys()
    assert all(_bits(tg["spare"][h]) == _bits(to["spare"][h]) for h in to["spare"])


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_rebalance_paths(gpu, oracle, case):
    want = oracle.rebalance(*case["args"], groups=case["groups"])
    assert want
    _same_decisions(gpu.rebalance(*case["args"], groups=case["groups"]), want)


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_rebalance_paths_trace(gpu, oracle, case):
    """K18/K21 state after the walk: order_dru checks every re-fold, not only the ones that decided."""
    _same_trace(gpu.rebalance_trace(*case["args"], groups=case["groups"]),
                oracle.rebalance_trace(*case["args"], groups=case["groups"]))


@pytest.mark.parametrize("make", [crowded_hosts, mass_preemption], ids=lambda m: m.__name__)
def test_ctas_per_sm_does_not_change_decisions(gpu, oracle, make):
    """Equal-DRU ties go to the greatest hostname whichever CTA owns the host: the walk under
    COOK_REB_CTAS_PER_SM = 1 and = 4 (the library clamps it to the kernel's occupancy) is the oracle's."""
    case = make()
    saved = os.environ.get("COOK_REB_CTAS_PER_SM")
    out = []
    try:
        for v in ("1", "4"):
            os.environ["COOK_REB_CTAS_PER_SM"] = v
            out.append(gpu.rebalance_trace(*case["args"], groups=case["groups"]))
    finally:
        if saved is None:
            os.environ.pop("COOK_REB_CTAS_PER_SM", None)
        else:
            os.environ["COOK_REB_CTAS_PER_SM"] = saved
    to = oracle.rebalance_trace(*case["args"], groups=case["groups"])
    for tg in out:
        _same_trace(tg, to)


def test_gpu_dru_mode_rejects_rebalance():
    """cook_rebalance on a GPU-DRU-mode handle: COOK_E_UNSUPPORTED_CONSTRAINT, and the handle still ranks."""
    from cook_b200.engine import CookError, GpuEngine
    from oracle.pyoracle import OracleEngine
    case = mass_preemption()
    eng = GpuEngine(pool_name="gpu-mode-reb", dru_mode=1)
    try:
        with pytest.raises(CookError) as e:
            eng.rebalance(*case["args"], groups=case["groups"])
        assert e.value.code == abi.COOK_E_UNSUPPORTED_CONSTRAINT
        t = traces.gen_pool(961, 3000, 16, 40, 800)
        rg = eng.rank(t["running"], t["pending"], t["users"])
        ro = OracleEngine(dru_mode=1).rank(t["running"], t["pending"], t["users"])
        assert np.array_equal(rg["ranked"], ro["ranked"])
        assert np.array_equal(rg["order"], ro["order"])
        assert np.array_equal(np.nan_to_num(rg["dru"], nan=-1.0), np.nan_to_num(ro["dru"], nan=-1.0))
    finally:
        eng.close()
