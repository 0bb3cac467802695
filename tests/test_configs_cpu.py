"""CPU side of BASELINE configs #3-#5: the generators' shapes, the pool -> GPU plan bench.py uses,
and the oracle running a miniature of every config (the -m gpu suite runs them at stated size)."""
import numpy as np
import pytest

from cook_b200 import abi, sharding, traces


def test_config_shapes():
    for cfg, (nj, no, pools) in {"c3": (1_000_000, 20_000, 4), "c4": (1_000_000, 20_000, 4),
                                 "c5": (10_000_000, 100_000, 16)}.items():
        s = traces.pool_sizes(cfg)
        assert len(s) == pools and sum(x[0] for x in s) == nj
        assert abs(sum(x[1] for x in s) - no) <= pools          # rounding of the node split
    assert sum(x[3] for x in traces.pool_sizes("c4")) == 400_000
    assert sum(x[3] for x in traces.pool_sizes("c5")) == 2_000_000


def test_lpt_plan_covers_every_pool_once():
    import bench
    for cfg in ("c3", "c4", "c5"):
        for world in (1, 2, 4, 8):
            plan = bench.pool_plan(cfg, world)
            assert sorted(p for p, _ in plan) == list(range(len(traces.pool_sizes(cfg))))
            assert all(0 <= r < world for _, r in plan)
            load = [0] * world
            for p, r in plan:
                j, o, _, _ = traces.pool_sizes(cfg)[p]
                load[r] += j * o
            if world <= len(plan):
                assert min(load) > 0                             # nobody idles while pools remain
    assert bench.pool_plan("c2", 4) == [(0, 0), (1, 1), (2, 2), (3, 3)]
    a = bench.config_dict("c5", 8, bench.pool_plan("c5", 8))
    assert a["n_pools"] == 16 and a["jobs"] == 10_000_000 and sum(a["pools_per_gpu"]) == 16
    assert a["pools_per_gpu"][0] == 1            # the largest pool gets a GPU to itself


@pytest.mark.parametrize("cfg,p", [("c3", 0), ("c4", 3), ("c5", 7)])
def test_config_miniature_through_oracle(oracle, cfg, p):
    t = traces.gen_config_pool(cfg, p, scale=0.01)
    r = oracle.rank(t["running"], t["pending"], t["users"])
    assert 0 < len(r["ranked"]) <= t["jobs"].n
    prm = traces.match_params(t["jobs"].n, host_lifetime_mins=t["host_lifetime_mins"])
    m = oracle.match(r["ranked"], t["jobs"], t["offers"], t["users"], prm, groups=t["groups"], max_ports=2)
    assert m["stats"]["n_matched"] > 0
    # threaded = single-threaded (the reference arm of bench.py uses the threaded form)
    m2 = oracle.match(r["ranked"], t["jobs"], t["offers"], t["users"], prm, groups=t["groups"], max_ports=2, threads=4)
    assert np.array_equal(m["assign"], m2["assign"]) and np.array_equal(m["ports"], m2["ports"])
    if cfg != "c3":
        rb = t["rebalance"]
        d = oracle.rebalance(rb["running"], rb["pending"], rb["pending_job_id"], rb["pending_priority"], rb["hosts"],
                             rb["users"], rb["params"], groups=rb["groups"])
        assert isinstance(d, list)


def test_fast_constraint_generator_invariants():
    t = traces.gen_config_pool("c3", 1, scale=0.05)
    j, o = t["jobs"], t["offers"]
    ao, ac = j.col("attr_off"), j.col("attr_col")
    two = np.where(np.diff(ao) == 2)[0]
    assert len(two) and (ac[ao[two]] != ac[ao[two] + 1]).all()           # distinct columns per job
    no, nh = j.col("novel_off"), j.col("novel_host")
    for k in np.where(np.diff(no) >= 2)[0][:500]:
        hs = nh[no[k]:no[k + 1]]
        assert len(set(hs.tolist())) == len(hs)                          # distinct previous hosts
    g = t["groups"]
    assert g is not None and g.n_groups > 0
    assert j.col("group_idx").max() < g.n_groups
    assert (o.col("gpu_off")[1:] - o.col("gpu_off")[:-1]).max() <= 1


def test_nonsaturating_c2_variant_places_everything(oracle):
    t = traces.gen_c2(seed=2, n_jobs=4000, n_offers=200, n_users=50, n_running=800, offer_scale=6)
    r = oracle.rank(t["running"], t["pending"], t["users"])["ranked"]
    m = oracle.match(r, t["jobs"], t["offers"], t["users"], traces.match_params(4000))
    assert m["stats"]["n_matched"] == 4000


def test_dump_outputs_fits_its_budget_and_samples_the_same_rows(oracle, tmp_path):
    """bench.py --dump-outputs: float64 files of the cycle's results; over budget, a fixed sample of
    rows whose numbers are stored beside it, the same in every run."""
    import bench
    t = traces.gen_config_pool("c4", 3, scale=0.01)
    r = oracle.rank(t["running"], t["pending"], t["users"])
    m = oracle.match(r["ranked"], t["jobs"], t["offers"], t["users"],
                     traces.match_params(t["jobs"].n, host_lifetime_mins=t["host_lifetime_mins"]),
                     groups=t["groups"], max_ports=2)
    rb = t["rebalance"]
    d = oracle.rebalance(rb["running"], rb["pending"], rb["pending_job_id"], rb["pending_priority"], rb["hosts"],
                         rb["users"], rb["params"], groups=rb["groups"])
    assert len(d) > 0
    arrays = bench.output_arrays({3: (r, m, d)}, np.arange(2 * 8 * 4.0).reshape(1, 2, 8, 4))
    assert all(a.dtype == np.float64 for a in arrays.values())
    assert np.array_equal(arrays["pool03_match_assign"], m["assign"])
    assert arrays["pool03_rebalance_decisions"].shape == (len(d), 7)
    assert arrays["exchange_usage"].shape == (16, 4)
    full = sum(a.nbytes for a in arrays.values())
    bench.dump_outputs(str(tmp_path / "all"), arrays, 2 * full)
    for k, a in arrays.items():
        assert np.array_equal(np.load(tmp_path / "all" / (k + ".npy")), a, equal_nan=True), k
    budget = full // 4
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, budget)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= budget
    for k, a in arrays.items():
        got = np.load(tmp_path / "a" / (k + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got, np.load(tmp_path / "b" / (k + ".npy")), equal_nan=True)
        if len(a) > 1:
            rows = np.load(tmp_path / "a" / (k + ".rows.npy")).astype(np.int64)
            assert 0 < len(rows) < len(a) and np.array_equal(got, a[rows], equal_nan=True), k


def test_reference_arm_prints_one_json_line():
    """The driver's contract: `bench.py --impl reference` runs on the host cores alone and prints exactly ONE
    line on stdout - the JSON with the arm's own cpu_baseline and e2e blocks (everything else, including what
    libraries write to fd 1 behind Python's back, goes to stderr)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = p.stdout.splitlines()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    import bench
    assert d["config"] == bench.config_dict("c2", 1, bench.pool_plan("c2", 1))
