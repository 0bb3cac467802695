"""-m gpu: CUDA path vs the CPU oracle, bit for bit, where rounding decides the answer (inputs from
tests/exactness_cases.py): off-grid Mesos-like amounts, fitness denominators that are adjacent
doubles, running sums on the boundaries of the exact-grid flag, sort and scan tile edges, and GPU
DRU mode at scale, where equal DRUs are the normal case."""
import os

import numpy as np
import pytest

from cook_b200 import abi, traces
from exactness_cases import (OFFGRID_CPUS, OFFGRID_MATCH, ULP_SEEDS, boundary_considerable_inputs,
                             boundary_exchange_inputs, boundary_rank_inputs, boundary_rebalance_inputs,
                             gen_gpu_mode_pool, gen_offgrid_pool, gen_ulp_close_pool, grid_boundary_cases,
                             greedy_reference)

pytestmark = pytest.mark.gpu

THREADS = 8


def _same_dru(a, b):
    return np.array_equal(np.nan_to_num(a, nan=-1.0), np.nan_to_num(b, nan=-1.0))


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def _rank_parity(gpu, oracle, *args, **kw):
    rg = gpu.rank(*args, **kw)
    ro = oracle.rank(*args, **kw)
    assert np.array_equal(rg["order"], ro["order"])
    assert np.array_equal(rg["ranked"], ro["ranked"])
    assert _same_dru(rg["dru"], ro["dru"])
    return ro


def _match_parity(gpu, oracle, t, ranked, constraints, reference=True):
    prm = traces.match_params(len(ranked), host_lifetime_mins=t.get("host_lifetime_mins", 0))
    kw = dict(groups=t["groups"], max_ports=2) if constraints else {}
    mg = gpu.match(ranked, t["jobs"], t["offers"], t["users"], prm, **kw)
    mo = oracle.match(ranked, t["jobs"], t["offers"], t["users"], prm, threads=THREADS, **kw)
    assert np.array_equal(mg["considerable"], mo["considerable"])
    assert np.array_equal(mg["assign"], mo["assign"])
    assert np.array_equal(mg["ports"], mo["ports"])
    assert np.array_equal(mg["fail"] == 0, mo["fail"] == 0)
    for k in ("n_considerable", "n_matched", "head_matched", "n_offers_used", "evals"):
        assert mg["stats"][k] == mo["stats"][k], k
    assert mo["stats"]["n_matched"] > 0
    if reference and not constraints:
        assert np.array_equal(greedy_reference(mo["considerable"], t["jobs"], t["offers"]), mo["assign"])
    return prm, mo


@pytest.mark.parametrize("constraints", [False, True], ids=["cpumem", "constraints"])
@pytest.mark.parametrize("seed,nj,no", OFFGRID_MATCH)
def test_off_grid_pools(gpu, oracle, seed, nj, no, constraints):
    """Mesos-like off-grid amounts through rank and both match kernels, at offer counts that reach every
    storage path of the matcher; then the per-reason failure counts, whose device side rebuilds each
    VM's state by a left fold over off-grid job sizes."""
    t = gen_offgrid_pool(seed, nj, no, constraints=constraints)
    ranked = _rank_parity(gpu, oracle, t["running"], t["pending"], t["users"])["ranked"]
    prm, mo = _match_parity(gpu, oracle, t, ranked, constraints)
    unplaced, placed = np.nonzero(mo["assign"] < 0)[0], np.nonzero(mo["assign"] >= 0)[0]
    ks = np.unique(np.concatenate([unplaced[:20], unplaced[-5:], placed[:10], placed[-10:],
                                   placed[len(placed) // 2:len(placed) // 2 + 5]])).astype(np.int32)
    fg = gpu.match_failures(ks)
    fo = oracle.match_failures(ranked, t["jobs"], t["offers"], t["users"], prm, ks, groups=t["groups"])
    assert fg == fo


@pytest.mark.parametrize("knobs", [{}, {"COOK_KMIN": "6", "COOK_LOOKAHEAD": "8"}], ids=["default", "kmin6-la8"])
@pytest.mark.parametrize("constraints", [False, True], ids=["cpumem", "constraints"])
@pytest.mark.parametrize("seed", ULP_SEEDS)
def test_ulp_close_fitness(gpu, oracle, seed, constraints, knobs):
    """Fitness denominators one ulp apart, all-ones significands (plain division) next to their
    neighbours (reciprocal), tie sets wider than TOPK, 1e100 denominators: every placement as the oracle
    and the plain-numpy restatement make it, with the candidate bound moved by the pipeline knobs."""
    t = gen_ulp_close_pool(seed)
    if constraints:
        traces.add_constraints(t, seed + 1000, frac_gpu_nodes=0.0, frac_gpu_jobs=0.0, frac_attr=0.1,
                               frac_group_jobs=0.02, frac_novel=0.05)
    ranked = _rank_parity(gpu, oracle, t["running"], t["pending"], t["users"])["ranked"]
    saved = {k: os.environ.get(k) for k in ("COOK_KMIN", "COOK_LOOKAHEAD")}
    try:
        for k in saved:
            os.environ.pop(k, None)
        os.environ.update(knobs)
        _match_parity(gpu, oracle, t, ranked, constraints)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


BOUNDARY = grid_boundary_cases()


@pytest.mark.parametrize("case", BOUNDARY, ids=lambda c: c["name"])
def test_grid_boundary_rank(gpu, oracle, case):
    """The per-user DRU folds and the pool, group and offensive filters of the rank."""
    inp = boundary_rank_inputs(case)
    ro = _rank_parity(gpu, oracle, inp["running"], inp["pending"], inp["users"], pool_quota=inp["pool_quota"],
                      group_quota=inp["group_quota"], group_usage=inp["group_usage"], params=inp["params"])
    assert 0 < len(ro["ranked"]) < inp["pending"].n


@pytest.mark.parametrize("case", BOUNDARY, ids=lambda c: c["name"])
def test_grid_boundary_considerable(gpu, oracle, case):
    """The user-quota fold of the considerable set, from the user's running usage."""
    ranked, jobs, offers, users, n = boundary_considerable_inputs(case)
    prm = traces.match_params(n)
    mg = gpu.match(ranked, jobs, offers, users, prm)
    mo = oracle.match(ranked, jobs, offers, users, prm, threads=THREADS)
    assert np.array_equal(mg["considerable"], mo["considerable"])
    assert np.array_equal(mg["assign"], mo["assign"])
    assert 0 < len(mo["considerable"]) <= n


@pytest.mark.parametrize("case", BOUNDARY, ids=lambda c: c["name"])
def test_grid_boundary_exchange(gpu, oracle, case):
    """The usage delta of a match round against an explicit left fold in considerable order."""
    ranked, jobs, offers, users, nu = boundary_exchange_inputs(case)
    prm = traces.match_params(len(ranked))
    mg = gpu.match(ranked, jobs, offers, users, prm)
    mo = oracle.match(ranked, jobs, offers, users, prm, threads=THREADS)
    assert np.array_equal(mg["assign"], mo["assign"])
    want = np.zeros((nu, 4))
    jc, jm, ju = jobs.col("cpus"), jobs.col("mem"), jobs.col("user")
    for k, j in enumerate(mo["considerable"]):
        if mo["assign"][k] < 0:
            continue
        u = ju[j]
        want[u, 0] = want[u, 0] + 1.0
        want[u, 1] = want[u, 1] + jc[j]
        want[u, 2] = want[u, 2] + jm[j]
    got = gpu.exchange_usage(nu)[0]
    assert want[0, 0] > 0
    assert np.array_equal(_bits(got), _bits(want))


@pytest.mark.parametrize("case", BOUNDARY, ids=lambda c: c["name"])
def test_grid_boundary_rebalance(gpu, oracle, case):
    """job-below-quota from the pending job's amounts, the per-user refolds after each preemption and
    the host phase from off-grid spare resources: decisions and the K18/K21 trace state."""
    inp = boundary_rebalance_inputs(case)
    args = (inp["running"], inp["pending"], inp["pending_job_id"], inp["pending_priority"], inp["hosts"],
            inp["users"], inp["params"])
    assert gpu.rebalance(*args) == oracle.rebalance(*args)
    tg, to = gpu.rebalance_trace(*args), oracle.rebalance_trace(*args)
    assert tg["decisions"] == to["decisions"]
    assert tg["below_quota"] == to["below_quota"]
    assert _same_dru(tg["pending_dru"], to["pending_dru"])
    assert tg["order"] == to["order"]
    assert np.array_equal(_bits(tg["order_dru"]), _bits(to["order_dru"]))
    assert tg["spare"] == to["spare"]


@pytest.mark.parametrize("grid", [True, False], ids=["grid", "offgrid"])
@pytest.mark.parametrize("n", [2047, 2048, 2049, 4095, 4097])
def test_sort_and_scan_edges(gpu, oracle, n, grid):
    """pending + running at the edges of the 2048-wide sort and scan tiles; three users of about equal
    size, so the middle user's segment straddles a tile boundary and a 1024-entry filter chunk."""
    nr = n // 5
    kw = {} if grid else dict(cpus_choices=OFFGRID_CPUS, mem_fn=lambda r, k: r.integers(300, 30000, size=k) / 3.0)
    t = traces.gen_pool(900 + n, n - nr, 64, 3, nr, zipf=None, **kw)
    tot = float(np.sum(t["pending"].col("cpus"))) + float(np.sum(t["running"].col("cpus")))
    q = lambda f: abi.make_pool_quota(dict(count=1e12, cpus=f * tot, mem=1e15, gpus=1e12))
    ro = _rank_parity(gpu, oracle, t["running"], t["pending"], t["users"], pool_quota=q(0.7), group_quota=q(0.5),
                      group_usage=np.array([3.0, 7.5 if grid else 7.3, 4096.0, 0.0]),
                      params=abi.RankParams(100, 0, 0.0, 0.0))
    assert 0 < len(ro["ranked"]) < n - nr
    _rank_parity(gpu, oracle, t["running"], t["pending"], t["users"])


@pytest.fixture(scope="module")
def gpu_mode():
    from cook_b200.engine import GpuEngine
    from oracle.pyoracle import OracleEngine
    eng = GpuEngine(pool_name="gpu-mode", dru_mode=1)
    yield eng, OracleEngine(dru_mode=1)
    eng.close()


def _gpu_mode_parity(gpu_mode, t, label, **kw):
    eng, ora = gpu_mode
    ro = _rank_parity(eng, ora, t["running"], t["pending"], t["users"], **kw)
    ms = eng.last_stats(abi.PHASE_RANK)["ms_device"]
    print(f"\n[gpu-mode rank] {label}: {t['pending'].n} pending + {t['running'].n} running, "
          f"device {ms:.3f} ms (last_stats PHASE_RANK)")
    return ro


def test_gpu_mode_gpu_pool(gpu_mode):
    """(a) every job asks for 1, 2, 4 or 8 gpus, users' gpu shares vary: 20k tasks."""
    t = gen_gpu_mode_pool(951, 16_000, 4_000, 200, 1.0)
    _gpu_mode_parity(gpu_mode, t, "gpu pool")


def test_gpu_mode_mostly_zero_dru_at_c2_size(gpu_mode):
    """(b) C2 size, Zipf users, 90 % of jobs without gpus: nearly the whole queue is one run of DRU 0.0,
    ordered by the merge's arrival rule across many sort tiles."""
    t = gen_gpu_mode_pool(952, 100_000, 20_000, 1_000, 0.1)
    ro = _gpu_mode_parity(gpu_mode, t, "mixed, C2 size")
    assert np.count_nonzero(ro["dru"] == 0.0) > 90_000


def test_gpu_mode_quotas_bind_at_c2_size(gpu_mode):
    """(c) case (b) with the pool and quota-group filters binding."""
    t = gen_gpu_mode_pool(952, 100_000, 20_000, 1_000, 0.1)
    tot_c = float(np.sum(t["pending"].col("cpus")))
    pool = abi.make_pool_quota(dict(count=80_000 + 20_000, cpus=1e15, mem=1e15, gpus=1e12))
    group = abi.make_pool_quota(dict(count=1e12, cpus=0.5 * tot_c, mem=1e15, gpus=1e12))
    ro = _gpu_mode_parity(gpu_mode, t, "mixed, C2 size, quotas", pool_quota=pool, group_quota=group,
                          group_usage=np.array([0.0, 1000.5, 0.0, 0.0]))
    assert 0 < len(ro["ranked"]) < 80_000
