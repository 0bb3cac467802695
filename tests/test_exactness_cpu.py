"""CPU checks that the rounding-sensitive GPU tests (test_gpu_exactness.py) can fail: the independent
matcher restatement agrees with the oracle off the grid, the reciprocal division without its correction
step gives different assignments, the ulp-close trace really has near-ties, and every grid-boundary
case separates the left fold from the scan association."""
from fractions import Fraction

import numpy as np
import pytest

from cook_b200 import traces
from exactness_cases import (OFFGRID_MATCH, ULP_SEEDS, flip_quota, gen_offgrid_pool, gen_ulp_close_pool,
                             grid_boundary_cases, grid_flag_allows, greedy_reference, greedy_steps, left_fold,
                             pick, scan_assoc)


def _match(oracle, t):
    ranked = oracle.rank(t["running"], t["pending"], t["users"])["ranked"]
    return oracle.match(ranked, t["jobs"], t["offers"], t["users"], traces.match_params(len(ranked)), threads=4)


@pytest.mark.parametrize("seed,nj,no", OFFGRID_MATCH)
def test_reference_matches_oracle_off_grid(oracle, seed, nj, no):
    t = gen_offgrid_pool(seed, nj, no)
    m = _match(oracle, t)
    assert m["stats"]["n_matched"] > 0
    assert np.array_equal(greedy_reference(m["considerable"], t["jobs"], t["offers"]), m["assign"])


@pytest.mark.parametrize("seed", ULP_SEEDS)
def test_reference_matches_oracle_ulp_close(oracle, seed):
    t = gen_ulp_close_pool(seed)
    m = _match(oracle, t)
    assert np.array_equal(greedy_reference(m["considerable"], t["jobs"], t["offers"]), m["assign"])


@pytest.mark.parametrize("seed", ULP_SEEDS)
def test_uncorrected_reciprocal_changes_assignments(oracle, seed):
    """x * RN(1/den) without the correction step is what the device would compute if the correction
    were lost: on the ulp-close pool it must place some job elsewhere."""
    t = gen_ulp_close_pool(seed)
    cons = _match(oracle, t)["considerable"]
    good = greedy_reference(cons, t["jobs"], t["offers"])
    bad = greedy_reference(cons, t["jobs"], t["offers"], div="uncorrected")
    assert np.count_nonzero(good != bad) > 0


def _exact_fitness(t, j, v, ac, am):
    jb, of = t["jobs"], t["offers"]
    num_c = (jb.col("cpus")[j] + ac[v]) + of.col("run_cpus")[v]
    num_m = (jb.col("mem")[j] + am[v]) + of.col("run_mem")[v]
    den_c = of.col("cpus")[v] + of.col("run_cpus")[v]
    den_m = of.col("mem")[v] + of.col("run_mem")[v]
    return (Fraction(num_c) / Fraction(den_c) + Fraction(num_m) / Fraction(den_m)) / 2


@pytest.mark.parametrize("seed", ULP_SEEDS)
def test_ulp_close_trace_has_near_ties(oracle, seed):
    """Among the first 300 placements, at least 12 have a runner-up whose exact rational fitness is
    within one f64 ulp of the winner's (and not equal): correct rounding decides them."""
    t = gen_ulp_close_pool(seed)
    cons = _match(oracle, t)["considerable"]
    by_name = np.argsort(t["offers"].col("name_rank"), kind="stable")
    g = greedy_steps(cons, t["jobs"], t["offers"])
    near = 0
    step = next(g)
    for _ in range(300):
        k, j, f, ac, am = step
        v = pick(f, by_name)
        top = np.argsort(-f, kind="stable")[:48]
        ex = sorted((_exact_fitness(t, j, int(w), ac, am) for w in top if f[w] > 0), reverse=True)
        if len(ex) >= 2:
            ulp = Fraction(float(np.spacing(f[v])))
            gaps = [ex[0] - e for e in ex[1:] if e != ex[0]]
            if gaps and min(gaps) < ulp:
                near += 1
        step = g.send(v)
    assert near >= 12, near


@pytest.mark.parametrize("case", grid_boundary_cases(), ids=lambda c: c["name"])
def test_boundary_cases_separate_associations(case):
    x, s = case["x"], case["start"][1]
    lf, sc = left_fold(x, s), scan_assoc(x, s)
    if case["same"]:
        assert grid_flag_allows(x, s)
        assert np.array_equal(lf, sc)
        return
    assert not grid_flag_allows(x, s)
    assert not np.array_equal(lf, sc)
    q = flip_quota(case)
    assert q is not None
    quota, k = q
    assert (lf[k] <= quota) != (sc[k] <= quota)      # one quota decision differs at the flip point


def test_generators_are_deterministic():
    def cols(t):
        out = [t[s].col(c) for s in ("pending", "running") for c in ("user", "cpus", "mem", "gpus")]
        out += [t["offers"].col(c) for c in ("name_rank", "cpus", "mem", "run_cpus", "run_mem")]
        return out + [t["jobs"].col("mem")]
    for make in (lambda: gen_offgrid_pool(611, 300, 50, constraints=True), lambda: gen_ulp_close_pool(5)):
        a, b = cols(make()), cols(make())
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    a, b = grid_boundary_cases(), grid_boundary_cases()
    assert [c["name"] for c in a] == [c["name"] for c in b]
    assert all(np.array_equal(c["x"], d["x"]) and c["start"] == d["start"] for c, d in zip(a, b))
