"""CPU checks that the rebalancer path tests (test_gpu_rebalance_paths.py) can fail: each case of
tests/rebalance_cases.py reaches its regime in the oracle's walk, each constraint of a constraint case
changes the oracle's decisions when it is removed, and the eligibility edges are exact."""
from fractions import Fraction

import numpy as np
import pytest

from rebalance_cases import (CASES, MIN_DIFF, SAFE, crowded_hosts, eligibility_edges, gpu_disk_lifetime,
                             many_groups, mass_preemption, off_grid_twin, pack, regimes, spare_only_hosts,
                             synthetic_victims, variant)


def _walk(oracle, case):
    return oracle.rebalance(*case["args"], groups=case["groups"])


def _owners(case, decisions):
    c = case["cols"]
    return list(c["run"]["user"]) + [int(c["pend"]["user"][d["pending_idx"]]) for d in decisions]


def test_crowded_hosts_leave_the_fast_path(oracle):
    case = crowded_hosts()
    r = regimes(case, _walk(oracle, case))
    real = np.bincount(case["cols"]["run"]["host"])
    for n in (63, 64, 65, 150, 400):
        assert n in real
    assert r["most_items"] > 64
    assert r["crossed_by_syn"]           # a host with <= 64 real tasks passes 64 items through synthetic ones
    assert r["most_victims"] > 64


def test_mass_preemption_victim_counts(oracle):
    case = mass_preemption()
    dec = _walk(oracle, case)
    own = _owners(case, dec)
    counts = [(len(d["victims"]), len({own[i] for i in d["victims"]})) for d in dec]
    assert any(nv > 64 and nu == 1 for nv, nu in counts)          # one user, more than 64 victims
    assert any(nu > 63 and nv > 64 for nv, nu in counts)          # 150 victims of 150 users
    assert any(nu > 63 and nv <= 64 for nv, nu in counts)         # 64 victims of 64 users: the user list overflows
    # the victims' users have later tasks whose DRU the re-fold moves
    run = case["cols"]["run"]
    assert all(np.count_nonzero(run["user"] == own[i]) > 1 for d in dec for i in d["victims"])


def test_synthetic_tasks_are_preempted_on_both_paths(oracle):
    case = synthetic_victims()
    dec = _walk(oracle, case)
    R = len(case["cols"]["run"]["user"])
    real = np.bincount(case["cols"]["run"]["host"], minlength=len(case["cols"]["host"]["name_rank"]))
    paths = set()
    for k, d in enumerate(dec):
        if any(i >= R for i in d["victims"]):
            items = real[d["host"]] + sum(1 for e in dec[:k] if e["host"] == d["host"])
            paths.add("general" if items > 64 else "fast")
    assert paths == {"fast", "general"}
    # a host whose synthetic victim died is decided again later
    hit = [d["host"] for d in dec if any(i >= R for i in d["victims"])]
    assert any(d["host"] in hit for k, d in enumerate(dec) if k > 0 and any(
        e["host"] == d["host"] and any(i >= R for i in e["victims"]) for e in dec[:k]))


def test_gpu_jobs_are_decided(oracle):
    case = gpu_disk_lifetime()
    dec = _walk(oracle, case)
    pg = case["cols"]["pend"]["gpus"]
    gd = [d for d in dec if pg[d["pending_idx"]] > 0]
    assert len(gd) >= 4 and all(d["gpus"] >= pg[d["pending_idx"]] > 0 for d in gd)
    assert {pg[d["pending_idx"]] for d in gd} >= {1.0, 2.0, 4.0, 8.0}
    # the gpu term lengthens a prefix: some decision has more victims than its cpus and mem need
    run = case["cols"]["run"]
    assert any(d["victims"] and run["gpus"][d["victims"][0]] > 0 for d in gd)


def test_group_jobs_leave_the_tables(oracle):
    case = many_groups()
    r = regimes(case, _walk(oracle, case))
    assert r["most_groups"] > 4
    assert r["most_distinct_values"] > 64
    distinct = [len(set(g["cot_attrs"])) for g in case["cols"]["groups"]]
    assert {32, 33, 64, 65} <= set(distinct)


@pytest.mark.parametrize("make,flags", [(gpu_disk_lifetime, dict(gpu_tables=False)),
                                        (gpu_disk_lifetime, dict(disk_tables=False)),
                                        (gpu_disk_lifetime, dict(host_start=False)),
                                        (many_groups, dict(with_groups=False)),
                                        (spare_only_hosts, dict(with_groups=False))],
                         ids=["gpu_tables", "disk_tables", "host_start", "groups", "spare_only_groups"])
def test_each_constraint_matters(oracle, make, flags):
    case = make()
    assert _walk(oracle, case) != _walk(oracle, variant(case, **flags))


def test_spare_only_attributes_matter(oracle):
    """The spare-only hosts' attributes and location, removed: decisions change."""
    case = spare_only_hosts()
    c = dict(case["cols"])
    host = dict(c["host"])
    empty = (host["has_spare"] == 1) & (np.bincount(c["run"]["host"], minlength=len(host["has_spare"])) == 0)
    assert np.count_nonzero(empty) >= 4
    attr, loc = host["attr"].copy(), host["location"].copy()
    attr[:, empty] = 0
    loc[empty] = -1
    host.update(attr=attr, location=loc)
    c["host"] = host
    base = _walk(oracle, case)
    assert base != _walk(oracle, pack("spare_only_hosts~noattr", c))
    # a spare-only host is decided before and after it has a task
    assert any(empty[d["host"]] and d["victims"] == [] for d in base)


def _dru0(case, task):
    """Exact DRU of a running task before the walk: its user's tasks in (-priority, start) order."""
    run, usr = case["cols"]["run"], case["cols"]["user"]
    u = run["user"][task]
    mine = sorted(np.nonzero(run["user"] == u)[0], key=lambda i: (-run["prio"][i], run["start"][i]))
    cm = cc = Fraction(0)
    for i in mine:
        cm += Fraction(float(run["mem"][i]))
        cc += Fraction(float(run["cpus"][i]))
        if i == task:
            return max(cm / Fraction(float(usr["div_mem"][u])), cc / Fraction(float(usr["div_cpus"][u])))
    raise AssertionError


def test_eligibility_edges_are_exact(oracle):
    case = eligibility_edges()
    e = case["cols"]["edges"]
    tr = oracle.rebalance_trace(*case["args"], groups=case["groups"])
    dec = tr["decisions"]
    # the first decision needs the task at exactly safe_dru_threshold
    d0 = [d for d in dec if d["pending_idx"] == e["safe_job"]]
    assert d0 and d0[0]["victims"] == [e["safe_task"]]
    assert _dru0(case, e["safe_task"]) == Fraction(SAFE)
    assert d0[0]["dru"] == SAFE
    # the task exactly min_dru_diff above the job's pending DRU is not eligible: the job finds no host
    pd = Fraction(float(tr["pending_dru"][e["diff_job"]]))
    assert _dru0(case, e["diff_task"]) - pd == Fraction(MIN_DIFF)
    assert not any(d["pending_idx"] == e["diff_job"] for d in dec)
    # max_preemption stops the walk in the middle; jobs between decisions find no host
    mp = case["args"][6].max_preemption
    assert len(dec) == mp
    assert tr["below_quota"][-1] is None and tr["below_quota"][dec[-1]["pending_idx"]] is not None
    decided = {d["pending_idx"] for d in dec}
    assert any(p not in decided for p in range(dec[-1]["pending_idx"]))


def test_off_grid_twins_decide(oracle):
    for make in CASES:
        twin = off_grid_twin(make())
        run = twin["cols"]["run"]
        assert np.all(run["cpus"] * 1024.0 != np.rint(run["cpus"] * 1024.0))
        assert _walk(oracle, twin)


def test_generators_are_deterministic(oracle):
    for make in CASES:
        a, b = make(), make()
        for side in ("run", "pend", "host", "user"):
            for k, v in a["cols"][side].items():
                w = b["cols"][side][k]
                assert (np.array_equal(v, w) if isinstance(v, np.ndarray) else v == w), (a["name"], side, k)
        assert a["cols"]["groups"] == b["cols"]["groups"]
        assert _walk(oracle, a) == _walk(oracle, b)
