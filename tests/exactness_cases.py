"""Inputs where f64 rounding decides the answer, and an independent reference to judge them by.

`cook_b200.traces` keeps every amount on a binary grid (cpus in halves, mem in whole MiB, four offer
types), so sums are exact in any order and every fitness denominator is 2^k or 3*2^k.  That makes
divisions exact and parallel scans legal, which is exactly what leaves three fast paths untested:
the reciprocal division of the matcher (match.cu div_y), the exact-grid flag that licenses parallel
scans (common.cuh grid_exact / grid_value_ok), and the equal-DRU merge walk-back of gpu mode
(rank.cu LessMerge).  The generators here produce Mesos-like off-grid amounts, fitness
denominators that are adjacent doubles, and running sums that sit exactly on the grid flag's
boundaries.  Every generator is seeded and deterministic.

`greedy_reference` restates the cpu+mem matcher (FENZO 3a + 4, oracle eval_pair) in numpy, one
job at a time, vectorised over the VMs.  `left_fold` / `scan_assoc` are the two associations of a
running sum (the reference's left fold and the 32-lane scan with a carry that the fast paths use);
the CPU tests use them to show that each boundary case separates the two.
"""
import numpy as np

from cook_b200 import abi, traces

OFFGRID_CPUS = (0.1, 0.3, 0.7, 1.1, 2.9, 0.45, 3.3)
TWO43 = 2.0 ** 43
# (seed, jobs, offers) of the off-grid match pools: tile edges (31-33 VMs), shared-memory tables (100,
# 1000), the static table read from L2 (7000) and the newest-log-entry table in global memory (45000)
OFFGRID_MATCH = [(601, 400, 31), (602, 400, 32), (603, 400, 33), (604, 2000, 100), (605, 4000, 1000),
                 (606, 3000, 7000), (607, 1500, 45000)]
ULP_SEEDS = (5, 6)


# ---------------------------------------------------------------------------------- reference
def greedy_steps(considerable, jobs, offers, div="ieee"):
    """Yields (k, j, fitness over all VMs, assigned cpus, assigned mem) before each placement and
    applies the placement after the consumer resumes.  div="uncorrected" divides as x * RN(1/den)
    (the reciprocal path without its correction step)."""
    jc, jm = jobs.col("cpus"), jobs.col("mem")
    lc, lm = offers.col("cpus"), offers.col("mem")
    O = offers.n
    rc = offers.col("run_cpus") if offers.col("run_cpus") is not None else np.zeros(O)
    rm = offers.col("run_mem") if offers.col("run_mem") is not None else np.zeros(O)
    den_c, den_m = lc + rc, lm + rm
    with np.errstate(divide="ignore", over="ignore", invalid="ignore", under="ignore"):
        yc, ym = 1.0 / den_c, 1.0 / den_m
    by_name = np.argsort(offers.col("name_rank"), kind="stable")   # equal fitness -> lowest name_rank
    ac, am = np.zeros(O), np.zeros(O)
    for k, j in enumerate(np.asarray(considerable)):
        fits = ~((ac + jc[j] > lc) | (am + jm[j] > lm))
        num_c, num_m = (jc[j] + ac) + rc, (jm[j] + am) + rm
        with np.errstate(divide="ignore", over="ignore", invalid="ignore", under="ignore"):
            if div == "ieee":
                fc, fm = num_c / den_c, num_m / den_m
            elif div == "uncorrected":
                fc, fm = num_c * yc, num_m * ym
            else:
                raise ValueError(div)
            f = np.where(fits, (fc + fm) / 2.0, 0.0)
        v = yield k, j, f, ac, am
        if v is not None and v >= 0:
            ac[v] = ac[v] + jc[j]
            am[v] = am[v] + jm[j]


def pick(f, by_name):
    """Argmax of the fitness, ties to the lowest name_rank; -1 when nothing fits (fitness 0)."""
    fs = f[by_name]
    i = int(np.argmax(fs))
    return int(by_name[i]) if fs[i] > 0.0 else -1


def greedy_reference(considerable, jobs, offers, div="ieee"):
    """Assignment (VM index or -1) of every considerable job, as the oracle's cpu+mem matcher makes it."""
    by_name = np.argsort(offers.col("name_rank"), kind="stable")
    out = np.full(len(considerable), -1, np.int32)
    g = greedy_steps(considerable, jobs, offers, div)
    step = next(g, None)
    while step is not None:
        k, _, f, _, _ = step
        out[k] = pick(f, by_name)
        step = _send(g, out[k])
    return out


def _send(g, v):
    try:
        return g.send(int(v))
    except StopIteration:
        return None


# ------------------------------------------------------------------------- associations
def left_fold(x, start=0.0):
    """Prefix sums ((start + x0) + x1) + ...: the reference's association."""
    out = np.empty(len(x))
    acc = float(start)
    for i, v in enumerate(np.asarray(x, np.float64)):
        acc = acc + float(v)
        out[i] = acc
    return out


def scan_assoc(x, start=0.0):
    """Prefix sums in the fast paths' association: an inclusive Hillis-Steele scan over each chunk of
    32 lanes, added to the carry of the chunks before it (start is the first carry)."""
    x = np.asarray(x, np.float64)
    out = np.empty(len(x))
    carry = float(start)
    for b in range(0, len(x), 32):
        s = x[b:b + 32].copy()
        o = 1
        while o < 32:
            prev = s.copy()
            s[o:] = prev[o:] + prev[:-o]
            o <<= 1
        out[b:b + len(s)] = carry + s
        carry = float(out[b + len(s) - 1])
    return out


def on_grid(x):
    x = np.asarray(x, np.float64)
    return bool(np.all((x >= 0) & (x <= 2.0 ** 40) & (x * 1024.0 == np.rint(x * 1024.0))))


def grid_flag_allows(x, start=0.0):
    """What common.cuh grid_exact decides for addends x and one start value."""
    m = max(float(np.max(x)), 1.0)
    return on_grid(x) and on_grid([start]) and (len(x) + 1) * m + start < TWO43


# --------------------------------------------------------------------------- generators
def _offers(hostname_id, name_rank, lc, lm, rc, rm, run_count):
    return abi.OffersSoA(n=len(lc), hostname_id=hostname_id, name_rank=name_rank, cpus=lc, mem=lm,
                         run_cpus=rc, run_mem=rm, run_count=run_count, n_attr_cols=0)


def gen_offgrid_pool(seed, n_jobs, n_offers, n_users=40, n_running=None, constraints=False, **ckw):
    """traces.gen_pool shape with Mesos-like amounts: offer cpus in 0.1 steps (31.9 after executor
    overhead), offer mem in tenths and sevenths of a MiB, running amounts likewise; job cpus from
    OFFGRID_CPUS and job mem in thirds of a MiB.  constraints=True adds traces.add_constraints."""
    n_running = n_jobs // 4 if n_running is None else n_running
    t = traces.gen_pool(seed, n_jobs, n_offers, n_users, n_running, cpus_choices=OFFGRID_CPUS,
                        mem_fn=lambda r, n: r.integers(300, 30000, size=n) / 3.0)
    rng = np.random.Generator(np.random.PCG64(seed + 7))
    O = n_offers
    lc = rng.integers(5, 960, O) / 10.0
    busy = rng.random(O) < 0.6
    rc = np.where(busy, rng.integers(1, 400, O) / 10.0, 0.0)
    dv = np.where(rng.random(O) < 0.5, 10.0, 7.0)
    lm = rng.integers(20_000, 4_000_000, O) / dv
    rm = np.where(busy, rng.integers(1_000, 2_000_000, O) / dv, 0.0)
    rcount = np.where(busy, rng.integers(1, 9, O), 0).astype(np.int32)
    of = t["offers"]
    t["offers"] = _offers(of.col("hostname_id"), of.col("name_rank"), lc, lm, rc, rm, rcount)
    t["groups"] = None
    t["host_lifetime_mins"] = 0
    if constraints:
        traces.add_constraints(t, seed + 1000, **ckw)
    return t


def _adjacent(base, n):
    out = [float(base)]
    for _ in range(n - 1):
        out.append(float(np.nextafter(out[-1], np.inf)))
    return out


def ulp_close_denominators():
    """(cpu denominator, cpu run) of the VMs of gen_ulp_close_pool, grouped in blocks that share a
    name-rank range.  The runs are chosen so that lease + run gives the denominator back exactly."""
    blocks = []
    for base, run in ((16.0, 4.0), (24.0, 4.0), (20.0, 0.0), (48.0, 16.0), (2.0 ** 20, 2.0 ** 18)):
        blocks.append([(d, run) for d in _adjacent(base, 16)])              # adjacent doubles
    ones16 = 16.0 - 2.0 ** -49                                              # all-ones significands
    ones32 = 32.0 - 2.0 ** -48
    ones20 = 2.0 ** 20 - 2.0 ** -33
    blocks.append([(ones16, 4.0), (float(np.nextafter(ones16, 0)), 4.0), (16.0, 4.0), (ones16, 0.0),
                   (ones32, 4.0), (float(np.nextafter(ones32, 0)), 4.0), (32.0, 0.0), (24.0, 0.0),
                   (float(np.nextafter(16.0, np.inf)), 4.0), (ones20, 2.0 ** 18), (2.0 ** 20, 0.0),
                   (float(np.nextafter(ones20, 0)), 2.0 ** 18), (3.0 * 2.0 ** 18, 0.0)])
    blocks.append([(16.0, 4.0)] * 12 + [(ones16, 4.0)] * 12)                 # tie sets wider than TOPK
    blocks.append([(1e100, 0.0), (float(np.nextafter(1e100, 0)), 0.0), (1e100, 0.0),
                   (float(np.nextafter(1e100, 0)), 0.0)])
    return blocks


def gen_ulp_close_pool(seed, n_jobs=1200, n_users=12, n_running=300, copies=2):
    """VMs whose cpu fitness denominators are adjacent doubles (base * (1 + k 2^-52), k = 0..15 for
    bases 16, 24, 20, 48, 2^20), all-ones significands (16 - 2^-49, 32 - 2^-48, 2^20 - 2^-33) and the
    double below them, powers of two, 3 * 2^k, tie sets of 12 identical VMs, cpu denominators at 1e100
    and one ulp inside, and mem denominators at 1e-100 and one ulp inside.  All VMs but the tiny-mem
    ones share one mem lease, so early placements are decided by the last bit of the cpu quotient:
    by correct rounding or by the hostname tie-break.  Both branches of div_y (reciprocal and plain
    division) compete for the same jobs."""
    t = traces.gen_pool(seed, n_jobs, 8, n_users, n_running, cpus_choices=(0.1, 0.3, 1.1, 2.9),
                        mem_fn=lambda r, n: r.integers(30, 3000, size=n) / 3.0)
    rng = np.random.Generator(np.random.PCG64(seed + 11))
    blocks = ulp_close_denominators() * copies
    tiny = float(np.nextafter(1e-100, np.inf))
    blocks.append([(64.0, 0.0)] * 2 + [(48.0, 0.0)] * 2)                   # carry the tiny mem leases
    lc, rc, lm, rm, nrank = [], [], [], [], []
    order = rng.permutation(len(blocks))                                    # blocks in shuffled name order
    rank0 = np.zeros(len(blocks), np.int64)
    rank0[order] = np.cumsum([0] + [len(blocks[b]) for b in order])[:-1]
    for b, blk in enumerate(blocks):
        last = b == len(blocks) - 1
        for i, (den, run) in enumerate(blk):
            lease = den - run
            assert lease + run == den, (den, run)
            lc.append(lease); rc.append(run)
            if last:
                lm.append([1e-100, tiny][i % 2]); rm.append(0.0)
            else:
                lm.append(196608.0); rm.append(0.0)
            nrank.append(rank0[b] + i)
    O = len(lc)
    lc, rc, lm, rm = (np.array(a, np.float64) for a in (lc, rc, lm, rm))
    t["offers"] = _offers(np.arange(O, dtype=np.int32), np.array(nrank, np.int32), lc, lm, rc, rm,
                          np.where(rc > 0, 3, 0).astype(np.int32))
    # a few jobs without memory, which fit the tiny-mem VMs
    jobs = t["jobs"]
    mem = jobs.col("mem").copy()
    mem[rng.random(jobs.n) < 0.05] = 0.0
    t["jobs"] = abi.JobsSoA(n=jobs.n, user=jobs.col("user"), cpus=jobs.col("cpus"), mem=mem,
                            gpus=jobs.col("gpus"), ports=jobs.col("ports"), allowed=jobs.col("allowed"),
                            plugin_accept=jobs.col("plugin_accept"))
    t["groups"] = None
    t["host_lifetime_mins"] = 0
    return t


def _fine_grid(rng, n, scale=1.0):
    """Multiples of 2^-10 that are not multiples of 2^-1, times a power-of-two scale."""
    k = rng.integers(1, 4096, n)
    k = np.where(k % 512 == 0, k + 1, k)
    return k * 2.0 ** -10 * scale


def grid_boundary_cases():
    """One running-sum input per boundary of the exact-grid flag.  Each case: name, addends `x` (the
    cpus of one user's tasks in queue order), `start` (count, cpus, mem, gpus) the fold starts from,
    `role` of the start value (None, "user_usage", "group_usage", "pending_job") and `same`: True when
    the flag must allow the fast path and every association agrees."""
    rng = np.random.Generator(np.random.PCG64(4242))
    z = (0.0, 0.0, 0.0, 0.0)
    cases = []
    cases.append(dict(name="fine_grid", x=_fine_grid(rng, 3000), start=z, role=None, same=True))
    # One 2^-11 among on-grid addends whose total crosses 2^42 (ulp 2^-10) while (n+1) * max stays below
    # 2^43: the addend alone must send the sums to the serial path.  (A lone 0.1 or 1/3 among on-grid
    # addends below 2^43 is only ever rounded at binade crossings, where both associations round alike.)
    n = 1500
    m = 2.0 ** 43 / (n + 2)
    x = rng.integers(int(0.6 * m * 1024), int(m * 1024), n) * 2.0 ** -10
    x[700] = 2.0 ** -11
    cases.append(dict(name="one_addend_2^-11", x=x, start=z, role=None, same=False))
    x = np.concatenate([[2.0 ** 40], _fine_grid(rng, 5)])      # the largest addend the flag accepts
    cases.append(dict(name="addend_2^40", x=x, start=z, role=None, same=True))
    # just above it, off the grid: 2^40 + 2^-12, in pairs that share a 32-lane chunk once the total is past
    # 2^42, so the chunk's sum carries a 2^-11 that the left fold drops one 2^-12 at a time
    x = rng.integers(2 ** 20, 2 ** 31, 3000) * 2.0 ** -10
    x[[5, 2100, 2101, 2600, 2611, 2800, 2803]] = 2.0 ** 40 + 2.0 ** -12
    cases.append(dict(name="addend_2^40+2^-12", x=x, start=z, role=None, same=False))
    x = np.full(200, 2.0 ** 36 + 2.0 ** -10)                    # on the grid, totals cross 2^43
    cases.append(dict(name="totals_cross_2^43", x=x, start=z, role=None, same=False))
    # on-grid addends, off-grid start value that is not the largest of the four (cpus 1/3 next to mem
    # 4096): only the explicit per-value checks see it.  1/3 rather than 0.1: the bits of 0.1 never
    # make a double rounding differ, so with it the fast path would be wrong without the suite noticing.
    for role in ("user_usage", "group_usage", "pending_job"):
        x = rng.integers(1, 64, 2500) * 0.25
        cases.append(dict(name="start_" + role, x=x, start=(3.0, 1.0 / 3.0, 4096.0, 0.0), role=role, same=False))
    return cases


def flip_quota(case):
    """A cpus quota at which the left fold and the scan association decide some prefix differently:
    the left-fold value of the first prefix where the scan lands above it (or, failing that, the scan's
    value where it lands below).  None when the two associations agree everywhere."""
    x, s = case["x"], case["start"][1]
    lf, sc = left_fold(x, s), scan_assoc(x, s)
    up = np.nonzero(sc > lf)[0]
    if len(up):
        return float(lf[up[0]]), int(up[0])
    dn = np.nonzero(sc < lf)[0]
    if len(dn):
        return float(sc[dn[0]]), int(dn[0])
    return None


def _user_tasks(x, user, id_base, running=False, mem=1.0):
    n = len(x)
    job_id = (id_base + np.arange(n)).astype(np.int64) * 2
    return abi.make_tasks(user=np.full(n, user, np.int32), priority=np.full(n, 50, np.int32),
                          start_time=(1_600_000_000_000 + np.arange(n)).astype(np.int64) if running
                          else np.full(n, abi.INT64_MAX, np.int64),
                          task_id=job_id + 1 if running else np.full(n, -1, np.int64), job_id=job_id,
                          cpus=np.asarray(x, np.float64), mem=np.full(n, mem))


def boundary_rank_inputs(case):
    """One user whose pending jobs carry the case's addends as cpus (DRU = cumulative cpus / 1.0), a
    second user with a few small jobs, pool and group quotas at flip points of the queue-order sums
    (group usage = the case's start for the group_usage role) and an offensive-job cap."""
    x = case["x"]
    other = np.full(40, 0.5)
    cpus = np.concatenate([x, other])
    user = np.concatenate([np.zeros(len(x), np.int32), np.ones(40, np.int32)])
    n = len(cpus)
    job_id = (1_000_000 + np.arange(n)).astype(np.int64) * 2
    pending = abi.make_tasks(user=user, priority=np.full(n, 50, np.int32), start_time=np.full(n, abi.INT64_MAX, np.int64),
                             task_id=np.full(n, -1, np.int64), job_id=job_id, cpus=cpus, mem=np.full(n, 1.0))
    big = np.finfo(np.float64).max
    # the second user's DRU is far above: the merged queue is user 0's jobs first, in their order
    users = abi.make_users(2, name_rank=np.array([1, 0], np.int32), div_mem=np.array([1e300, 1e300]),
                           div_cpus=np.array([1.0, 2.0 ** -60]), div_gpus=np.ones(2))
    gs = case["start"] if case["role"] == "group_usage" else (0.0, 0.0, 0.0, 0.0)
    fq = flip_quota(dict(case, start=gs))
    pool_cpus = float(left_fold(x)[-1]) + 1.0
    group_cpus = big
    if fq is not None:
        group_cpus = fq[0]
        pq = flip_quota(dict(case, start=(0.0,) * 4))
        if pq is not None and pq[1] > fq[1]:
            pool_cpus = pq[0]
    pool = abi.make_pool_quota(dict(count=1e12, cpus=pool_cpus, mem=1e15, gpus=1e12))
    group = abi.make_pool_quota(dict(count=1e12, cpus=group_cpus, mem=1e15, gpus=1e12))
    params = abi.RankParams(100, 1, 1e15, float(np.max(x)) if len(x) > 8 else 1e15)
    return dict(running=None, pending=pending, users=users, pool_quota=pool, group_quota=group,
                group_usage=np.array(gs, np.float64), params=params)


def boundary_considerable_inputs(case):
    """The case's addends as the cpus of one user's queued jobs, the user's running usage = the case's
    start for the user_usage role, and a user cpus quota at a flip point.  Returns (ranked, jobs,
    offers, users, num_considerable)."""
    x = case["x"]
    n = len(x)
    us = case["start"] if case["role"] == "user_usage" else (0.0, 0.0, 0.0, 0.0)
    fq = flip_quota(dict(case, start=us))
    qc = fq[0] if fq is not None else float(left_fold(x, us[1])[-1])
    users = abi.make_users(1, div_mem=np.array([1e300]), div_cpus=np.array([1.0]), div_gpus=np.ones(1),
                           quota=dict(count=np.array([1e12]), cpus=np.array([qc]), mem=np.array([1e15]),
                                      gpus=np.array([1e12])),
                           usage=dict(count=np.array([us[0]]), cpus=np.array([us[1]]), mem=np.array([us[2]]),
                                      gpus=np.array([us[3]])))
    jobs = _jobs(x, np.zeros(n, np.int32))
    return np.arange(n, dtype=np.int32), jobs, _big_offers(x), users, n


def _jobs(cpus, user, mem=1.0):
    n = len(cpus)
    return abi.JobsSoA(n=n, user=user, cpus=np.asarray(cpus, np.float64), mem=np.full(n, mem), gpus=np.zeros(n),
                       ports=np.zeros(n, np.int32), allowed=np.ones(n, np.uint8), plugin_accept=np.ones(n, np.uint8))


def _big_offers(x, n=8):
    cap = max(2.0 ** 46, 4.0 * float(np.sum(x)))
    return _offers(np.arange(n, dtype=np.int32), np.arange(n, dtype=np.int32)[::-1].copy(), np.full(n, cap),
                   np.full(n, 2.0 ** 40), np.zeros(n), np.zeros(n), np.zeros(n, np.int32))


def boundary_exchange_inputs(case):
    """Two users' jobs interleaved (user 0 carries the case's addends), offers large enough for all of
    them.  Returns (ranked, jobs, offers, users, n_users)."""
    x = case["x"]
    other = np.full(len(x) // 4 + 1, 0.75)
    cpus = np.concatenate([x, other])
    user = np.concatenate([np.zeros(len(x), np.int32), np.ones(len(other), np.int32)])
    perm = np.argsort(np.concatenate([np.arange(len(x)) * 4.0, np.arange(len(other)) * 16.0 + 1.5]), kind="stable")
    jobs = _jobs(cpus, user)
    users = abi.make_users(2, div_mem=np.full(2, 1e300), div_cpus=np.ones(2), div_gpus=np.ones(2))
    return perm.astype(np.int32), jobs, _big_offers(cpus), users, 2


def boundary_rebalance_inputs(case):
    """A rebalancer state in the K18/K21 shape: user 0 runs the case's addends as cpus on host 0, user 1
    runs large tasks on host 1, user 2 waits with nothing running.  User 0 also has a pending job (for
    the pending_job role: cpus 0.1, mem 4096, the fold's start) and a cpus quota at the flip point of
    job-below-quota; host 0 has off-grid spare resources."""
    x = np.asarray(case["x"], np.float64)
    n = len(x)
    big_n = 64
    cpus = np.concatenate([x, np.full(big_n, 6.5)])
    mem = np.concatenate([np.full(n, 1.0), np.full(big_n, 20480.0)])
    user = np.concatenate([np.zeros(n, np.int32), np.ones(big_n, np.int32)])
    R = n + big_n
    job_id = (1 + np.arange(R)).astype(np.int64) * 2
    t = abi.make_tasks(user=user, priority=np.full(R, 50, np.int32),
                       start_time=(1_600_000_000_000 + np.arange(R)).astype(np.int64), task_id=job_id + 1,
                       job_id=job_id, cpus=cpus, mem=mem)
    running = abi.RunningSoA(t=t, host=np.concatenate([np.zeros(n, np.int32), np.ones(big_n, np.int32)]))
    if case["role"] == "pending_job":
        pc, pm = case["start"][1], case["start"][2]
    else:
        pc, pm = 1.0, 1.0
    p_cpus = np.array([pc, 3.3, 0.7])
    p_mem = np.array([pm, 8000.0, 1000.3])
    p_user = np.array([0, 2, 2], np.int32)
    pending = abi.JobsSoA(n=3, user=p_user, cpus=p_cpus, mem=p_mem, gpus=np.zeros(3))
    tot = left_fold(x, pc)[-1]
    sc = scan_assoc(x, pc)[-1]
    qc = float(tot if sc > tot else (sc if sc < tot else tot))
    big = np.finfo(np.float64).max
    share_c = max(8.0, float(np.sum(x)) / 4.0)
    users = abi.make_users(3, name_rank=np.array([2, 0, 1], np.int32), div_mem=np.full(3, 65536.0),
                           div_cpus=np.full(3, share_c), div_gpus=np.ones(3),
                           quota=dict(count=np.full(3, big), cpus=np.array([qc, big, big]), mem=np.full(3, big),
                                      gpus=np.full(3, big)))
    hosts = abi.HostTable(n=2, hostname_id=np.arange(2, dtype=np.int32), name_rank=np.array([1, 0], np.int32),
                          has_spare=np.array([1, 0], np.uint8), spare_cpus=np.array([0.7, 0.0]),
                          spare_mem=np.array([1000.3, 0.0]), spare_gpus=np.zeros(2), n_attr_cols=0)
    return dict(running=running, pending=pending, pending_job_id=(10_000_000 + np.arange(3)).astype(np.int64) * 2,
                pending_priority=np.full(3, 50, np.int32), hosts=hosts, users=users,
                params=abi.RebalanceParams(8, 0.05, 0.0, 0))


def gen_gpu_mode_pool(seed, n_jobs, n_running, n_users, frac_gpu_jobs, offers=16):
    """A pool for GPU-mode ranking (DRU = cumulative gpus / gpu share): the tasks of a random set of
    users holding about frac_gpu_jobs of all tasks ask for gpus from {1, 2, 4, 8}, everyone else's for
    none; users' gpu shares vary.  With most tasks at 0 gpus nearly the whole queue is one run of DRU
    0.0 (a user's DRU is cumulative, so one gpu job early in a list would lift all that follow)."""
    t = traces.gen_pool(seed, n_jobs, offers, n_users, n_running)
    rng = np.random.Generator(np.random.PCG64(seed + 5))
    c = t["cols"]
    per_user = np.bincount(np.concatenate([c["pending"]["user"], c["running"]["user"]]), minlength=n_users)
    order = rng.permutation(n_users)
    gpu_user = np.zeros(n_users, bool)
    gpu_user[order[np.cumsum(per_user[order]) <= frac_gpu_jobs * per_user.sum()]] = True
    for side, n in (("pending", n_jobs), ("running", n_running)):
        d = dict(c[side])
        d["gpus"] = np.where(gpu_user[d["user"]], rng.choice(np.array([1.0, 2.0, 4.0, 8.0]), n), 0.0)
        c[side] = d
        t[side] = abi.make_tasks(**d)
    run = c["running"]
    usage = {k: np.zeros(n_users) for k in ("count", "cpus", "mem", "gpus")}
    np.add.at(usage["count"], run["user"], 1.0)
    for k in ("cpus", "mem", "gpus"):
        np.add.at(usage[k], run["user"], run[k])
    t["users"] = abi.make_users(n_users, name_rank=c["name_rank"], div_mem=c["div_mem"], div_cpus=c["div_cpus"],
                                div_gpus=rng.choice(np.array([1.0, 2.0, 3.0, 4.0, 8.0, 10.0]), n_users), usage=usage)
    return t
