"""-m gpu: BASELINE configs #3, #4, #5 at their STATED sizes through the CUDA path, bit-identical to
the oracle (assignments, ports, considerable sets, rank order, preemption decisions and victims);
the device-side usage exchange; pools of different size sharing one GPU; a repeated-cycle stress
test of the matcher's lock-free pipeline."""
import os
import threading

import numpy as np
import pytest

from cook_b200 import abi, sharding, traces

pytestmark = pytest.mark.gpu


def _same_dru(a, b):
    return np.array_equal(np.nan_to_num(a, nan=-1.0), np.nan_to_num(b, nan=-1.0))


def _cycle_parity(gpu, oracle, t, threads=0, rebalance=False):
    rg = gpu.rank(t["running"], t["pending"], t["users"])
    ro = oracle.rank(t["running"], t["pending"], t["users"])
    assert np.array_equal(rg["ranked"], ro["ranked"])
    assert _same_dru(rg["dru"], ro["dru"])
    prm = traces.match_params(t["jobs"].n, host_lifetime_mins=t["host_lifetime_mins"])
    mg = gpu.match(rg["ranked"], t["jobs"], t["offers"], t["users"], prm, groups=t["groups"], max_ports=2)
    mo = oracle.match(ro["ranked"], t["jobs"], t["offers"], t["users"], prm, groups=t["groups"], max_ports=2,
                      threads=threads or min(64, os.cpu_count() or 1))
    assert np.array_equal(mg["considerable"], mo["considerable"])
    assert np.array_equal(mg["assign"], mo["assign"])
    assert np.array_equal(mg["ports"], mo["ports"])
    assert mg["stats"]["n_matched"] == mo["stats"]["n_matched"] > 0
    assert mg["stats"]["evals"] == mo["stats"]["evals"]
    if rebalance:
        r = t["rebalance"]
        dg = gpu.rebalance(r["running"], r["pending"], r["pending_job_id"], r["pending_priority"], r["hosts"],
                           r["users"], r["params"], groups=r["groups"])
        do = oracle.rebalance(r["running"], r["pending"], r["pending_job_id"], r["pending_priority"], r["hosts"],
                              r["users"], r["params"], groups=r["groups"])
        assert len(dg) == len(do) > 0
        for a, b in zip(dg, do):
            assert (a["pending_idx"], a["host"], a["victims"]) == (b["pending_idx"], b["host"], b["victims"])
            assert (a["dru"], a["mem"], a["cpus"], a["gpus"]) == (b["dru"], b["mem"], b["cpus"], b["gpus"])
    return mg


@pytest.mark.parametrize("p", [0, 1, 2, 3])
def test_c3_full_size_pools(gpu, oracle, p):
    """BASELINE config #3 at stated size: 1M jobs x 20k nodes in 4 pools (400k x 8k, 300k x 6k,
    200k x 4k, 100k x 2k), every constraint kind, user quotas binding for ~10 % of the users."""
    t = traces.gen_config_pool("c3", p)
    assert (t["jobs"].n, t["offers"].n) == traces.pool_sizes("c3")[p][:2]
    _cycle_parity(gpu, oracle, t)


@pytest.mark.parametrize("p", [0, 3])
def test_c4_full_size_pools_with_rebalancer(gpu, oracle, p):
    """BASELINE config #4: config #3's pools with 400k running tasks in total (160k / 40k in these
    two pools) + the rebalancer sweep, max-preemption 128: decisions and victims identical."""
    t = traces.gen_config_pool("c4", p)
    _cycle_parity(gpu, oracle, t, rebalance=True)


def test_c5_one_full_size_pool(gpu, oracle):
    """BASELINE config #5: one of the 16 pools at stated size (pool 5: ~614k jobs x ~6.1k nodes,
    ~123k running tasks): rank + match + rebalance, bit-identical."""
    sizes = traces.pool_sizes("c5")
    assert sum(s[0] for s in sizes) == 10_000_000 and len(sizes) == 16
    t = traces.gen_config_pool("c5", 5)
    assert t["jobs"].n > 500_000
    _cycle_parity(gpu, oracle, t, rebalance=True)


def test_usage_exchange_device_delta(gpu, oracle):
    """cook_exchange_usage (world 1): the per-user usage delta computed on the device equals the host
    restatement (sharding.usage_delta) of generate-user-usage-map over the placed jobs."""
    t = traces.gen_pool(71, 20000, 800, 150, 3000)
    ranked = gpu.rank(t["running"], t["pending"], t["users"])["ranked"]
    m = gpu.match(ranked, t["jobs"], t["offers"], t["users"], traces.match_params(20000))
    got = gpu.exchange_usage(160)            # padded to 160 users
    assert got.shape == (1, 160, 4)
    j = t["jobs"]
    want = sharding.usage_delta(m["considerable"], m["assign"], j.col("user"), j.col("cpus"), j.col("mem"),
                                j.col("gpus"), 150)
    assert np.array_equal(got[0, :150], want)
    assert not got[0, 150:].any()
    assert want[:, 0].sum() == m["stats"]["n_matched"]
    s = gpu.last_stats(abi.PHASE_EXCHANGE)
    assert s["n_launches"] == 3 and s["ms_device"] > 0.0


def test_usage_exchange_batch_of_pools(gpu, oracle):
    """cook_exchange_usage_batch (world 1): the deltas of several handles of one GPU in one call, slot i =
    handle i, spare slots zero - the same numbers the per-pool call returns for each of them."""
    from cook_b200.engine import GpuEngine, exchange_usage_batch
    ta = traces.gen_pool(83, 9000, 400, 70, 1000)
    tb = traces.gen_pool(84, 5000, 250, 40, 600)
    eb = GpuEngine(pool_name="batch-b")
    try:
        for eng, t in ((gpu, ta), (eb, tb)):
            r = eng.rank(t["running"], t["pending"], t["users"])["ranked"]
            eng.match(r, t["jobs"], t["offers"], t["users"], traces.match_params(t["jobs"].n))
        one_a, one_b = gpu.exchange_usage(80)[0], eb.exchange_usage(80)[0]
        assert one_a[:, 0].sum() > 0 and one_b[:, 0].sum() > 0
        got = exchange_usage_batch([gpu, eb], 80, n_slots=3)
        assert got.shape == (1, 3, 80, 4)
        assert np.array_equal(got[0, 0], one_a) and np.array_equal(got[0, 1], one_b)
        assert not got[0, 2].any()
        s = gpu.last_stats(abi.PHASE_EXCHANGE)
        assert s["n_launches"] == 6 and s["d2h_bytes"] == 8 * 3 * 320
        with pytest.raises(Exception):
            exchange_usage_batch([gpu, eb], 80, n_slots=1)     # fewer slots than handles
    finally:
        eb.close()


def test_exchange_feeds_next_rank(gpu, oracle):
    """The exchange's result is CONSUMED: two pools of one quota group; the usage gathered after pool
    A's match round is pool B's group_usage in the next rank cycle, and decides how deep B's queue
    survives the quota-group filter (scheduler.clj:2125-2157) - identical to the oracle fed with the
    host-side delta."""
    from cook_b200.engine import GpuEngine
    ta = traces.gen_pool(81, 8000, 400, 60, 1000)
    tb = traces.gen_pool(82, 6000, 300, 60, 800)
    eb = GpuEngine(pool_name="group-b")
    try:
        ra = gpu.rank(ta["running"], ta["pending"], ta["users"])["ranked"]
        ma = gpu.match(ra, ta["jobs"], ta["offers"], ta["users"], traces.match_params(8000))
        g = gpu.exchange_usage(60)[0]                      # [60, 4]
        tot = g.sum(axis=0)
        j = ta["jobs"]
        want = sharding.usage_delta(ma["considerable"], ma["assign"], j.col("user"), j.col("cpus"), j.col("mem"),
                                    j.col("gpus"), 60).sum(axis=0)
        assert np.array_equal(tot, want) and tot[0] > 0
        gq = abi.make_pool_quota({"count": tot[0] + 500, "cpus": tot[1] + 1500, "mem": tot[2] + 6.0e6, "gpus": 1e9})
        rb_g = eb.rank(tb["running"], tb["pending"], tb["users"], group_quota=gq, group_usage=tot)
        rb_o = oracle.rank(tb["running"], tb["pending"], tb["users"], group_quota=gq, group_usage=want)
        assert np.array_equal(rb_g["ranked"], rb_o["ranked"])
        rb_0 = oracle.rank(tb["running"], tb["pending"], tb["users"], group_quota=gq, group_usage=np.zeros(4))
        assert 0 < len(rb_g["ranked"]) < len(rb_0["ranked"])   # the gathered usage really cut the queue
    finally:
        eb.close()


def test_pools_of_different_size_side_by_side(oracle):
    """Handles of one GPU may run concurrently (cook_gpu.h): pools with DIFFERENT offer counts (hence
    different dynamic shared-memory needs) matched from two host threads, many times, stay correct -
    the kernel attribute is raised monotonically, never lowered under another pool's launch."""
    from cook_b200.engine import GpuEngine
    shapes = [(91, 6000, 300, 40, 500), (92, 9000, 2400, 60, 900)]
    ts = [traces.gen_pool(*s) for s in shapes]
    want = []
    for t in ts:
        r = oracle.rank(t["running"], t["pending"], t["users"])["ranked"]
        want.append((r, oracle.match(r, t["jobs"], t["offers"], t["users"], traces.match_params(t["jobs"].n))["assign"]))
    engs = [GpuEngine(pool_name=f"side-{i}") for i in range(2)]
    errs = []

    def work(i):
        try:
            for _ in range(12):
                m = engs[i].match(want[i][0], ts[i]["jobs"], ts[i]["offers"], ts[i]["users"],
                                  traces.match_params(ts[i]["jobs"].n, max_ctas=60))
                if not np.array_equal(m["assign"], want[i][1]):
                    errs.append((i, "assignments differ"))
        except Exception as e:   # noqa: BLE001
            errs.append((i, repr(e)))
    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    for e in engs:
        e.close()
    assert not errs, errs


def test_matcher_stress_repeated_cycles(oracle):
    """A lock-free pipeline needs more than one green run: 200 C2-shaped cycles with the
    pipeline's knobs varied (queue depth, candidates per result, spec CTAs, grid size), every one
    bit-identical to the oracle."""
    from cook_b200.engine import GpuEngine
    t = traces.gen_c2(seed=5, n_jobs=30_000, n_offers=1_500, n_users=300, n_running=5_000)
    ranked = oracle.rank(t["running"], t["pending"], t["users"])["ranked"]
    want = oracle.match(ranked, t["jobs"], t["offers"], t["users"], traces.match_params(30_000))["assign"]
    knobs = [{}, {"COOK_LOOKAHEAD": "8"}, {"COOK_LOOKAHEAD": "31"}, {"COOK_KMIN": "6"}, {"COOK_KMIN": "16"},
             {"COOK_NSPEC": "1"}, {"COOK_NSPEC": "6"}, {"COOK_MATCH_B": "16", "COOK_MATCH_BMIN": "16"},
             {"COOK_MATCH_TARGET": "8"}, {"COOK_POLL_NS": "20"}]
    eng = GpuEngine(pool_name="stress")
    saved = {k: os.environ.get(k) for kn in knobs for k in kn}
    try:
        n = 0
        for rep in range(20):
            for i, kn in enumerate(knobs):
                for k in saved:
                    os.environ.pop(k, None)
                os.environ.update(kn)
                ctas = [0, 0, 37, 9, 148, 3][(rep + i) % 6]
                m = eng.match(ranked, t["jobs"], t["offers"], t["users"], traces.match_params(30_000, max_ctas=ctas))
                assert np.array_equal(m["assign"], want), (rep, kn, ctas)
                n += 1
        assert n == 200
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        eng.close()


def test_off_grid_amounts_keep_the_left_fold(gpu, oracle):
    """Amounts that are NOT on the binary grid (cpus 0.1, 0.3, ...): the association-free scan fast
    path must not trigger; DRU scores, quota filters and rebalancer decisions stay bit-identical to
    the oracle's left folds."""
    rng = np.random.default_rng(123)
    t = traces.gen_pool(61, 6000, 300, 25, 1500, cpus_choices=(0.1, 0.3, 0.7, 1.1, 2.9),
                        mem_fn=lambda r, n: r.integers(1, 4000, size=n) / 7.0)
    nu = 25
    quota = {"count": rng.integers(50, 400, nu).astype(float), "cpus": rng.integers(20, 300, nu) + 0.1,
             "mem": rng.integers(20000, 400000, nu) / 3.0, "gpus": np.full(nu, 1e9)}
    usage = {k: t["users"].col("usage_" + k) for k in ("count", "cpus", "mem", "gpus")}
    users = abi.make_users(nu, name_rank=t["users"].col("name_rank"), div_mem=t["users"].col("div_mem") / 3.0,
                           div_cpus=t["users"].col("div_cpus") / 7.0, quota=quota, usage=usage)
    pq = abi.make_pool_quota({"count": 3000, "cpus": 2500.3, "mem": 2.0e6 / 3.0, "gpus": 1e9})
    prm_r = abi.RankParams(7, 0, 0.0, 0.0)
    rg = gpu.rank(t["running"], t["pending"], users, pool_quota=pq, group_quota=pq, group_usage=np.array([3.0, 0.7, 11.0 / 7.0, 0.0]),
                  params=prm_r)
    ro = oracle.rank(t["running"], t["pending"], users, pool_quota=pq, group_quota=pq, group_usage=np.array([3.0, 0.7, 11.0 / 7.0, 0.0]),
                     params=prm_r)
    assert np.array_equal(rg["ranked"], ro["ranked"]) and _same_dru(rg["dru"], ro["dru"])
    assert 0 < len(ro["ranked"]) < 6000
    mg = gpu.match(ro["ranked"], t["jobs"], t["offers"], users, traces.match_params(6000), pool_quota=pq)
    mo = oracle.match(ro["ranked"], t["jobs"], t["offers"], users, traces.match_params(6000), pool_quota=pq)
    assert np.array_equal(mg["considerable"], mo["considerable"]) and np.array_equal(mg["assign"], mo["assign"])
    r = traces.gen_rebalance(62, 8000, 60, 400, 80, max_preemption=20)
    # knock the running tasks off the grid
    rt = r["running"].col("t")
    run2 = abi.RunningSoA(t=abi.make_tasks(user=rt.col("user"), priority=rt.col("priority"), start_time=rt.col("start_time"),
                                           task_id=rt.col("task_id"), job_id=rt.col("job_id"),
                                           cpus=rt.col("cpus") + 0.1, mem=rt.col("mem") / 3.0), host=r["running"].col("host"))
    args = (run2, r["pending"], r["pending_job_id"], r["pending_priority"], r["hosts"], r["users"], r["params"])
    dg = gpu.rebalance(*args, groups=r["groups"])
    do = oracle.rebalance(*args, groups=r["groups"])
    assert dg == do and len(do) > 0


def test_row_pretest_borderline_requests(gpu, oracle):
    """The evaluators skip a row whose request exceeds the most room left on any usable VM by more than a
    guard margin (1e-9 x scale).  Requests that differ from each other - and so from the room left as
    the cluster fills - by 1 ulp .. 1e-8 relative sit INSIDE that margin or just outside it: whatever
    the pre-test decides, placements stay bit-identical to the oracle's exact `assigned + request >
    limit` (cpu+mem kernel and constraint kernel, saturated clusters)."""
    eps = (0.0, 2.3e-16, 1e-13, 3e-10, 0.9e-9, 1.1e-9, 2e-9, 1e-8, 1e-6)
    cpus = tuple(b * (1.0 + e) for b in (0.5, 1.0, 2.0, 4.0) for e in eps)

    def mem_fn(r, n):
        base = 512.0 * r.integers(1, 33, size=n)
        return base * (1.0 + r.choice(np.array(eps), size=n))
    for constraints, seed in ((False, 301), (True, 302), (False, 303)):
        t = traces.gen_pool(seed, 9000, 160, 30, 600, cpus_choices=cpus, mem_fn=mem_fn,
                            constraints=constraints, n_attr_cols=4 if constraints else 0)
        ro = oracle.rank(t["running"], t["pending"], t["users"])
        rg = gpu.rank(t["running"], t["pending"], t["users"])
        assert np.array_equal(rg["ranked"], ro["ranked"])
        prm = traces.match_params(9000)
        kw = dict(groups=t.get("groups"), max_ports=2) if constraints else {}
        mg = gpu.match(ro["ranked"], t["jobs"], t["offers"], t["users"], prm, **kw)
        mo = oracle.match(ro["ranked"], t["jobs"], t["offers"], t["users"], prm, **kw)
        assert np.array_equal(mg["considerable"], mo["considerable"])
        assert np.array_equal(mg["assign"], mo["assign"])
        assert 0 < mo["stats"]["n_matched"] < 0.5 * mo["stats"]["n_considerable"]   # saturated: most rows are hopeless


def test_placement_failure_summaries(gpu, oracle):
    """SURVEY §8f-3: per-reason host counts of unplaced (and a few placed) jobs AT THEIR TURN, through
    the CUDA path, equal the oracle's counts from replaying the match; the summary has the
    fenzo_utils.clj:45-57 shape."""
    from cook_b200.cycle import CONSTRAINT_NAMES, summarize_failures
    t = traces.gen_c3_pool(77, 6000, 400, 60, 1200, frac_group_jobs=0.25, group_size=(3, 12), frac_gpu_jobs=0.1,
                           frac_gpu_nodes=0.3, frac_port_jobs=0.2)
    ranked = oracle.rank(t["running"], t["pending"], t["users"])["ranked"]
    prm = traces.match_params(6000, host_lifetime_mins=t["host_lifetime_mins"])
    mg = gpu.match(ranked, t["jobs"], t["offers"], t["users"], prm, groups=t["groups"], max_ports=2)
    unplaced = np.where(mg["assign"] < 0)[0]
    placed = np.where(mg["assign"] >= 0)[0]
    ks = np.concatenate([unplaced[:40], unplaced[-10:], placed[:5], placed[-5:]]).astype(np.int32)
    fg = gpu.match_failures(ks)
    fo = oracle.match_failures(ranked, t["jobs"], t["offers"], t["users"], prm, ks, groups=t["groups"])
    assert fg == fo
    seen = set()
    for k, f in zip(ks, fg):
        assert f["n_vms"] == 400
        assert sum(f["counts"][2:]) + f["n_passed"] <= 400
        if mg["assign"][k] < 0:
            assert f["n_passed"] == 0               # an unplaced job failed on every VM
        s = summarize_failures(f["counts"])
        seen |= set(s.get("constraints", {}))
        assert set(s) <= {"resources", "constraints"} and set(s.get("resources", {})) <= {"cpus", "mem"}
    assert len(seen & set(CONSTRAINT_NAMES)) >= 3   # several kinds of constraint failure occur in the trace


def test_bench_dumps_what_its_last_timed_step_computed(oracle, tmp_path):
    """bench.py --steps 2 --dump-outputs on C2: one JSON line reporting the 2 timed steps, and the dumped
    queue, considerable set and assignments are the oracle's on the same seeded inputs."""
    import json
    import subprocess
    import sys
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--no-nonsat", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=root)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = p.stdout.splitlines()
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    t = bench.gen_pool_inputs("c2", 0)
    ro = oracle.rank(t["running"], t["pending"], t["users"])
    mo = oracle.match(ro["ranked"], t["jobs"], t["offers"], t["users"], traces.match_params(t["jobs"].n),
                      threads=min(64, os.cpu_count() or 1))
    for name, want in (("rank_ranked", ro["ranked"]), ("rank_dru", ro["dru"]), ("match_considerable", mo["considerable"]),
                       ("match_assign", mo["assign"])):
        got = np.load(tmp_path / f"pool00_{name}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, want, equal_nan=True), name
    assert np.load(tmp_path / "exchange_usage.npy")[:, 0].sum() == mo["stats"]["n_matched"] > 0


def test_bad_index_columns_are_rejected_not_faulted(gpu):
    """A bad index from the shim comes back as COOK_E_BADARG (-1); the context stays usable."""
    from cook_b200.engine import CookError
    t = traces.gen_pool(95, 500, 40, 9, 100)
    ranked = gpu.rank(t["running"], t["pending"], t["users"])["ranked"]
    bad = ranked.copy()
    bad[3] = 10_000
    with pytest.raises(CookError) as e:
        gpu.match(bad, t["jobs"], t["offers"], t["users"], traces.match_params(500))
    assert e.value.code == abi.COOK_E_BADARG
    ju = t["jobs"].col("user").copy()
    ju[7] = 99
    jb = abi.JobsSoA(n=500, user=ju, cpus=t["jobs"].col("cpus"), mem=t["jobs"].col("mem"), gpus=t["jobs"].col("gpus"),
                     ports=t["jobs"].col("ports"), allowed=t["jobs"].col("allowed"), plugin_accept=t["jobs"].col("plugin_accept"))
    with pytest.raises(CookError) as e:
        gpu.match(ranked, jb, t["offers"], t["users"], traces.match_params(500))
    assert e.value.code == abi.COOK_E_BADARG
    m = gpu.match(ranked, t["jobs"], t["offers"], t["users"], traces.match_params(500))   # still works
    assert m["stats"]["n_considerable"] == len(ranked)
