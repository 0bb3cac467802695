"""Rebalancer inputs that reach the paths `traces.gen_rebalance` never does.

`gen_rebalance` always builds the same kind of pool: Zipf owners, tasks spread uniformly over hosts, no
gpus and at most one group per job.  Each generator here targets one regime of
`cook_b200/csrc/rebalance.cu` instead:

* `crowded_hosts`: hosts with 63 ... 400 running tasks, and hosts with 60-64 tasks that synthetic tasks
  push past 64 items, so `host_select` leaves its register fast path for the general one;
* `mass_preemption`: decisions with more than 64 victims, or victims from more than 63 users, so the
  re-fold after the decision folds every user (`Refold::all`);
* `synthetic_victims`: a later job preempts a task that an earlier decision of the same walk created;
* `gpu_disk_lifetime`: gpu models and counts, disk tables and host lifetimes on Kubernetes and Mesos hosts;
* `many_groups`: more than `GP_MAXG` groups on a job, and 32 / 33 / 64 / 65 / 100+ distinct attribute
  values over [preempted hosts ; cotasks], so the group tables fill both halves or fall back to the
  scalar walk;
* `spare_only_hosts`: hosts with spare resources and no task, whose attributes read as nil until a
  synthetic task lands there;
* `eligibility_edges`: task DRUs exactly at `safe_dru_threshold` and exactly `min_dru_diff` above the
  pending DRU, `max_preemption` reached in the middle of the walk.

Every case keeps its amounts on a binary grid, so the device takes its exact-scan forms; `off_grid_twin`
moves them off it (running cpus + 0.1, mem / 3, pending mem / 3), so the serial left folds run instead.
A case is a dict: `name`, `args` (the argument tuple of `rebalance` / `rebalance_trace`), `groups`, and
the plain columns it was built from (`cols`).  Every generator is seeded and deterministic.
"""
import numpy as np

from cook_b200 import abi

BIG = float(np.finfo(np.float64).max)
T0 = 1_600_000_000_000


class _Pool:
    """Accumulates hosts, users, running tasks, pending jobs and groups; `cols` returns plain columns for `pack`."""

    def __init__(self, seed):
        self.rng = np.random.Generator(np.random.PCG64(seed))
        self.h = []      # host dicts
        self.u = []      # user dicts
        self.t = []      # running task dicts
        self.p = []      # pending job dicts
        self.g = []      # group dicts
        self.n_attr = 3

    def user(self, cpus=1.0, mem=1024.0, count_quota=BIG):
        self.u.append(dict(div_cpus=float(cpus), div_mem=float(mem), quota_count=float(count_quota)))
        return len(self.u) - 1

    def host(self, spare=None, k8s=0, location=0, gpus=None, disk=None, start=-1, attr=None, key=None):
        """spare: (cpus, mem, gpus) or None; gpus / disk: {model or type: count or space}; key orders the
        hostnames (greater key = greater name; None draws one below every explicit key)."""
        a = list(attr) if attr is not None else [int(x) for x in self.rng.integers(1, 5, self.n_attr)]
        self.h.append(dict(spare=spare, k8s=int(k8s), location=int(location), gpus=dict(gpus or {}),
                           disk=dict(disk or {}), start=int(start), attr=a,
                           key=float(key) if key is not None else float(self.rng.random())))
        return len(self.h) - 1

    def task(self, user, host, cpus, mem, gpus=0.0, prio=50):
        k = len(self.t)
        self.t.append(dict(user=user, host=host, cpus=float(cpus), mem=float(mem), gpus=float(gpus), prio=int(prio),
                           start=T0 + 1000 * k, tid=2 * k + 1, jid=2 * k))
        return k

    def job(self, user, cpus, mem, gpus=0.0, prio=50, gpu_model=-1, disk=(-1.0, -1), est_end=-1, ckpt=-1,
            attrs=(), novel=(), groups=()):
        self.p.append(dict(user=user, cpus=float(cpus), mem=float(mem), gpus=float(gpus), prio=int(prio),
                           gpu_model=int(gpu_model), disk_request=float(disk[0]), disk_type=int(disk[1]),
                           est_end=int(est_end), ckpt=int(ckpt), attrs=list(attrs), novel=list(novel),
                           groups=list(groups)))
        return len(self.p) - 1

    def group(self, kind, attr_col=-1, minimum=1, cot_hosts=(), cot_attrs=None):
        """cot_attrs defaults to the cotask hosts' values in `attr_col`."""
        ch = [int(x) for x in cot_hosts]
        if cot_attrs is None:
            cot_attrs = [self.h[x]["attr"][attr_col] if 0 <= attr_col < self.n_attr else 0 for x in ch]
        self.g.append(dict(kind=kind, attr_col=attr_col, minimum=minimum, cot_hosts=ch,
                           cot_attrs=[int(x) for x in cot_attrs]))
        return len(self.g) - 1

    def cols(self, max_preemption, min_dru_diff, safe_dru_threshold, host_lifetime_mins=0):
        H, U = len(self.h), len(self.u)
        keys = np.array([x["key"] for x in self.h])
        host_rank = np.empty(H, np.int32)
        host_rank[np.argsort(keys, kind="stable")] = np.arange(H, dtype=np.int32)
        f = lambda rows, k, dt: np.array([r[k] for r in rows], dt)
        return dict(
            host=dict(name_rank=host_rank, has_spare=np.array([x["spare"] is not None for x in self.h], np.uint8),
                      spare=np.array([x["spare"] or (0.0, 0.0, 0.0) for x in self.h], np.float64).reshape(H, 3),
                      k8s=f(self.h, "k8s", np.uint8), location=f(self.h, "location", np.int32),
                      gpus=[x["gpus"] for x in self.h], disk=[x["disk"] for x in self.h],
                      start=f(self.h, "start", np.int64),
                      attr=np.array([x["attr"] for x in self.h], np.int32).reshape(H, self.n_attr).T.copy()),
            user=dict(name_rank=self.rng.permutation(U).astype(np.int32), div_cpus=f(self.u, "div_cpus", np.float64),
                      div_mem=f(self.u, "div_mem", np.float64), quota_count=f(self.u, "quota_count", np.float64)),
            run={k: f(self.t, k, dt) for k, dt in (("user", np.int32), ("host", np.int32), ("cpus", np.float64),
                                                  ("mem", np.float64), ("gpus", np.float64), ("prio", np.int32),
                                                  ("start", np.int64), ("tid", np.int64), ("jid", np.int64))},
            pend=dict({k: f(self.p, k, dt) for k, dt in (("user", np.int32), ("cpus", np.float64), ("mem", np.float64),
                                                         ("gpus", np.float64), ("prio", np.int32),
                                                         ("gpu_model", np.int32), ("disk_request", np.float64),
                                                         ("disk_type", np.int32), ("est_end", np.int64),
                                                         ("ckpt", np.int32))},
                      jid=(10_000_000 + 2 * np.arange(len(self.p))).astype(np.int64),
                      attrs=[x["attrs"] for x in self.p], novel=[x["novel"] for x in self.p],
                      groups=[x["groups"] for x in self.p]),
            groups=[dict(x) for x in self.g],
            params=(int(max_preemption), float(min_dru_diff), float(safe_dru_threshold), int(host_lifetime_mins)))


def pack(name, c):
    """ABI structs from the plain columns of a case."""
    hc, uc, rc, pc = c["host"], c["user"], c["run"], c["pend"]
    H, U, P = len(hc["name_rank"]), len(uc["name_rank"]), len(pc["user"])
    gpu_off, gpu_model = abi.csr([sorted(d) for d in hc["gpus"]])
    _, gpu_count = abi.csr([[d[k] for k in sorted(d)] for d in hc["gpus"]], np.float64)
    disk_off, disk_type = abi.csr([sorted(d) for d in hc["disk"]])
    _, disk_space = abi.csr([[d[k] for k in sorted(d)] for d in hc["disk"]], np.float64)
    hosts = abi.HostTable(n=H, hostname_id=np.arange(H, dtype=np.int32), name_rank=hc["name_rank"],
                          has_spare=hc["has_spare"], spare_cpus=hc["spare"][:, 0], spare_mem=hc["spare"][:, 1],
                          spare_gpus=hc["spare"][:, 2], is_k8s=hc["k8s"], location=hc["location"],
                          gpu_off=gpu_off if c.get("gpu_tables", True) else None, gpu_model=gpu_model, gpu_count=gpu_count,
                          disk_off=disk_off if c.get("disk_tables", True) else None, disk_type=disk_type,
                          disk_space=disk_space,
                          host_start_time=hc["start"] if c.get("host_start", True) else None,
                          n_attr_cols=hc["attr"].shape[0], attr=hc["attr"].reshape(-1))
    users = abi.make_users(U, name_rank=uc["name_rank"], div_mem=uc["div_mem"], div_cpus=uc["div_cpus"],
                           div_gpus=np.ones(U), quota=dict(count=uc["quota_count"]))
    t = abi.make_tasks(user=rc["user"], priority=rc["prio"], start_time=rc["start"], task_id=rc["tid"],
                       job_id=rc["jid"], cpus=rc["cpus"], mem=rc["mem"], gpus=rc["gpus"])
    running = abi.RunningSoA(t=t, host=rc["host"])
    attr_off, attr_col = abi.csr([[a for a, _ in x] for x in pc["attrs"]])
    _, attr_val = abi.csr([[v for _, v in x] for x in pc["attrs"]])
    novel_off, novel_host = abi.csr(pc["novel"])
    groups = None
    jkw = {}
    gl = c["groups"] if c.get("with_groups", True) else []
    if gl:
        group_off, group_idx = abi.csr(pc["groups"])
        cot_off, cot_host = abi.csr([g["cot_hosts"] for g in gl])
        _, cot_attr = abi.csr([g["cot_attrs"] for g in gl])
        groups = abi.Groups(n_groups=len(gl), kind=np.array([g["kind"] for g in gl], np.int32),
                            attr_col=np.array([g["attr_col"] for g in gl], np.int32),
                            minimum=np.array([g["minimum"] for g in gl], np.int32), cot_off=cot_off,
                            cot_hostname_id=cot_host, cot_attr_val=cot_attr)
        jkw = dict(group_off=group_off, group_idx=group_idx)
    pending = abi.JobsSoA(n=P, user=pc["user"], cpus=pc["cpus"], mem=pc["mem"], gpus=pc["gpus"],
                          gpu_model=pc["gpu_model"], disk_request=pc["disk_request"], disk_type=pc["disk_type"],
                          est_end_ms=pc["est_end"], ckpt_location=pc["ckpt"], attr_off=attr_off, attr_col=attr_col,
                          attr_val=attr_val, novel_off=novel_off, novel_host=novel_host, **jkw)
    params = abi.RebalanceParams(*c["params"])
    return dict(name=name, cols=c, groups=groups,
                args=(running, pending, pc["jid"], pc["prio"], hosts, users, params))


def off_grid_twin(case):
    """The same case with running cpus + 0.1, running, pending and spare mem / 3: every re-fold, quota fold
    and prefix sum leaves the exact grid and takes its serial, left-fold form."""
    c = dict(case["cols"])
    run = dict(c["run"]); run["cpus"] = run["cpus"] + 0.1; run["mem"] = run["mem"] / 3.0
    pend = dict(c["pend"]); pend["mem"] = pend["mem"] / 3.0
    host = dict(c["host"]); spare = host["spare"].copy(); spare[:, 1] /= 3.0; host["spare"] = spare
    c.update(run=run, pend=pend, host=host)
    return pack(case["name"] + "~offgrid", c)


def variant(case, **flags):
    """The case with parts of it removed: gpu_tables / disk_tables / host_start / with_groups = False."""
    c = dict(case["cols"], **flags)
    return pack(case["name"] + "~" + "-".join(sorted(flags)), c)


# ------------------------------------------------------------------------------------------ cases
def _background(pool, n_hosts, n_users, tasks_per_host, spare_frac=0.05, share=(2.0, 2048.0)):
    """Ordinary hosts with a few whole-cpu tasks of Zipf-distributed users; a few hosts with spare."""
    rng = pool.rng
    users = [pool.user(*share) for _ in range(n_users)]
    w = 1.0 / np.arange(1, n_users + 1) ** 1.1
    w /= w.sum()
    hosts = []
    for _ in range(n_hosts):
        sp = (float(rng.integers(1, 5)), 1024.0 * float(rng.integers(1, 5)), 0.0) if rng.random() < spare_frac else None
        h = pool.host(spare=sp)
        hosts.append(h)
        for _ in range(int(rng.integers(*tasks_per_host))):
            pool.task(users[int(rng.choice(n_users, p=w))], h, float(rng.choice([0.5, 1.0, 2.0])),
                      512.0 * float(rng.integers(1, 5)))
    return users, hosts


def crowded_hosts(seed=71):
    """Hosts with 63, 64, 65, 150 and 400 tasks of 0.25 cpus among 3000 ordinary hosts (enough hosts for the
    grid size to change which CTA owns which host), hosts with 60-64 tasks and spare that small jobs fill
    with synthetic tasks past 64 items, then jobs that need long victim prefixes on all of them."""
    pool = _Pool(seed)
    rng = pool.rng
    _background(pool, 3000, 200, (2, 7))
    crowd = [pool.user(0.25, 256.0) for _ in range(40)]
    k = 0
    for n in (63, 64, 65, 150, 400):
        h = pool.host(key=1.5 + 0.01 * n)
        for _ in range(n):
            z = rng.random() < 0.1          # zero-size tasks: equal DRUs inside a user
            pool.task(crowd[k % len(crowd)], h, 0.0 if z else 0.25, 0.0 if z else 256.0)
            k += 1
    small = [pool.user(0.5, 512.0) for _ in range(30)]
    fill = []
    for n in (60, 61, 62, 63, 64):
        h = pool.host(spare=(3.0, 3072.0, 0.0), key=2.0 + 0.01 * n)
        fill.append(h)
        for i in range(n):
            pool.task(small[(i + n) % len(small)], h, 0.25, 256.0)
    pend = [pool.user(1000.0, 1e6) for _ in range(6)]
    for q in range(4):                      # long prefixes on the crowd hosts
        pool.job(pend[q], float(10 + 8 * q), 10240.0 + 8192.0 * q)
    for q in range(30):                     # small jobs pile onto the fill hosts through their spare
        pool.job(pend[4 + q % 2], 0.5, 512.0)
    for q in range(40):                     # then need victims there (general path, synthetic items)
        pool.job(pend[q % 6], float(rng.choice([1.0, 1.5, 2.0, 3.0])), 256.0 * float(rng.integers(2, 12)))
    for q in range(6):
        pool.job(pend[q], float(20 + 4 * q), 16384.0)
    return pack("crowded_hosts", pool.cols(128, 0.5, 1.0))


def mass_preemption(seed=72):
    """Two crowd hosts of 150 one-task-per-user tasks at DRU 2.0, each user with a second task elsewhere;
    a host where one user owns 100 tasks (some of zero size) with 30 more on another host; a host of 64
    tasks of 64 users.  Decisions preempt 150 victims from 150 users, 80 victims of one user, and
    exactly 64 victims of 64 users (the last large decision: no later re-fold of every user hides a user
    it missed)."""
    pool = _Pool(seed)
    rng = pool.rng
    _, ordinary = _background(pool, 3000, 150, (1, 5))
    crowd_hosts = [pool.host(key=3.0), pool.host(key=3.1)]
    for h in crowd_hosts:
        us = [pool.user(0.125, 128.0) for _ in range(150)]
        for u in us:
            pool.task(u, h, 0.25, 256.0)
        for u in us:                        # a later task elsewhere: its DRU moves when the first one dies
            pool.task(u, ordinary[int(rng.integers(len(ordinary)))], 0.25, 256.0)
    w = pool.user(0.25, 256.0)
    hz, hz2 = pool.host(key=2.5), pool.host(key=2.6)
    for i in range(100):
        z = i % 10 == 9
        pool.task(w, hz, 0.0 if z else 0.25, 0.0 if z else 256.0)
    for i in range(30):
        pool.task(w, hz2, 0.25, 256.0)
    hv = pool.host(key=3.5)
    vs = [pool.user(0.25, 256.0) for _ in range(64)]
    for u in vs:
        pool.task(u, hv, 0.5, 512.0)
    for u in vs:
        pool.task(u, ordinary[int(rng.integers(len(ordinary)))], 0.5, 512.0)
    pend = [pool.user(1000.0, 1e6) for _ in range(4)]
    pool.job(pend[0], 35.0, 35000.0)        # 150 victims, 150 users
    pool.job(pend[1], 20.0, 18432.0)        # 80 victims, one user
    pool.job(pend[3], 35.0, 35000.0)        # the other crowd host
    pool.job(pend[2], 32.0, 32768.0)        # 64 victims, 64 users, and no re-fold of every user after it
    for q in range(20):
        pool.job(pend[q % 4], float(rng.choice([0.5, 1.0, 2.0])), 512.0 * float(rng.integers(1, 4)))
    return pack("mass_preemption", pool.cols(32, 0.5, 1.0))


def synthetic_victims(seed=73):
    """User Q is over its count quota, so only its own tasks are eligible for its jobs.  Low-priority jobs
    of Q land on spare hosts S (62 real tasks: past 64 items after three of them) and S2 (5 real tasks,
    the greater name); high-priority jobs of Q then sort before those synthetic tasks and preempt them,
    on S2 through the register fast path and on S through the general path; later jobs look at S2 again
    after its synthetic victim died."""
    pool = _Pool(seed)
    rng = pool.rng
    bg, _ = _background(pool, 60, 20, (3, 9), spare_frac=0.0)
    q = pool.user(1.0, 1024.0, count_quota=5.0)
    ha, hg = pool.host(key=1.2), pool.host(key=1.3)
    for i in range(20):
        pool.task(q, ha if i < 10 else hg, 0.5, 512.0)
    s = pool.host(spare=(4.0, 4096.0, 0.0), key=4.0)
    s2 = pool.host(spare=(4.0, 4096.0, 0.0), key=5.0)
    for i in range(62):
        pool.task(bg[i % len(bg)], s, 0.25, 256.0)
    for i in range(5):
        pool.task(bg[i], s2, 0.25, 256.0)
    for _ in range(3):
        pool.job(q, 1.0, 1024.0, prio=10, novel=[s2])   # onto S through its spare
    pool.job(q, 2.0, 2048.0, prio=10)       # S's spare is short: onto S2
    pool.job(q, 3.0, 3072.0, prio=90)       # preempts the synthetic task on S2 (fast path)
    pool.job(q, 1.5, 1536.0, prio=90)       # preempts a synthetic task on S (general path)
    for i in range(8):                      # S2 again, with its synthetic victim dead
        pool.job(q, float(rng.choice([0.5, 1.0, 1.5, 2.0])), 512.0 * float(rng.integers(1, 4)),
                 prio=int(rng.choice([10, 90, 95])))
    other = [pool.user(100.0, 102400.0) for _ in range(3)]
    for i in range(12):                     # below-quota jobs that may take anyone's tasks, synthetic ones too
        pool.job(other[i % 3] if i % 2 else q, float(rng.choice([0.5, 1.0, 2.0])), 512.0 * float(rng.integers(1, 5)),
                 prio=int(rng.choice([10, 50, 90])))
    return pack("synthetic_victims", pool.cols(40, 0.25, 1.0))


LIFETIME_MINS = 60
L_START = (1_700_000_000, 1_700_000_100)


def death_ms(start):
    return 1000 * start + 60_000 * LIFETIME_MINS


def gpu_disk_lifetime(seed=74):
    """Kubernetes hosts with 1 / 2 / 4 / 8 gpus of two models, gpu tasks below higher-DRU cpu tasks (so the
    gpu term decides how long a prefix is), spare gpus; disk tables with a request exactly equal to the
    space; host lifetimes with est-completion exactly at death (fails) and one ms before (passes);
    Mesos hosts mixed in."""
    pool = _Pool(seed)
    rng = pool.rng
    bg, _ = _background(pool, 40, 12, (2, 8))
    gu = [pool.user(1.0, 1024.0) for _ in range(8)]
    for u in gu:                            # earliest in their users' order: every later task is eligible
        pool.task(u, int(rng.integers(0, 40)), 1.5, 1536.0)
    gh = {}
    for m, n, key in ((0, 1, 6.0), (0, 2, 6.1), (1, 4, 6.2), (1, 4, 6.25), (1, 8, 6.3), (0, 8, 6.35)):
        spare = (1.0, 1024.0, 2.0) if n == 8 and m == 1 else None
        h = pool.host(spare=spare, k8s=1, gpus={m: float(n)}, key=key)
        gh[(m, n, key)] = h
        n_gpu_tasks = n - (2 if spare else 0)
        for i in range(n_gpu_tasks):        # gpu tasks first in their users' order: low DRU
            pool.task(gu[i % 4], h, 0.5, 512.0, gpus=1.0)
        for i in range(4):                  # cpu tasks later in order: higher DRU, preempted first
            pool.task(gu[(i + 1) % 4], h, 1.0, 1024.0)
    for _ in range(6):                      # Kubernetes hosts without gpus, Mesos hosts with gpu-less tasks
        h = pool.host(k8s=1)
        for i in range(5):
            pool.task(gu[4 + i % 4], h, 1.0, 1024.0)
    d1 = pool.host(spare=(2.0, 2048.0, 0.0), k8s=1, disk={0: 100.0, 1: 50.0}, key=7.0)
    d2 = pool.host(spare=(2.0, 2048.0, 0.0), k8s=1, disk={0: 200.0}, key=6.9)
    for h in (d1, d2):
        pool.task(bg[0], h, 0.5, 512.0)
    l1 = pool.host(spare=(2.0, 2048.0, 0.0), start=L_START[0], key=8.0)
    l2 = pool.host(spare=(2.0, 2048.0, 0.0), start=L_START[1], key=7.9)
    for h in (l1, l2):
        pool.task(bg[1], h, 0.5, 512.0)
    pu = [pool.user(100.0, 102400.0) for _ in range(6)]
    for g, m in ((1, 0), (2, 0), (4, 1), (8, 1), (4, 0), (8, 0), (2, 1), (1, 0), (4, 1)):
        pool.job(pu[g % 6], 1.0, 1024.0, gpus=float(g), gpu_model=m)
    pool.job(pu[0], 1.0, 1024.0, disk=(100.0, 0), est_end=death_ms(L_START[1]))   # d1: space == request
    pool.job(pu[1], 1.0, 1024.0, disk=(150.0, 0), est_end=death_ms(L_START[1]))   # d2 only
    pool.job(pu[2], 1.0, 1024.0, disk=(60.0, 1))                                  # no disk host has it
    pool.job(pu[3], 0.5, 512.0, est_end=death_ms(L_START[0]))                     # l1 fails: exactly at death
    pool.job(pu[4], 0.5, 512.0, est_end=death_ms(L_START[1]) - 1)                 # l2 passes: one ms before
    pool.job(pu[5], 0.5, 512.0, est_end=death_ms(L_START[0]) - 1)
    for i in range(16):
        g = float(rng.choice([0.0, 0.0, 1.0, 2.0, 4.0, 8.0]))
        pool.job(pu[i % 6], float(rng.choice([0.5, 1.0])), 512.0, gpus=g, gpu_model=int(rng.integers(0, 2)),
                 disk=(100.0, 0) if rng.random() < 0.3 else (-1.0, -1),
                 est_end=death_ms(L_START[int(rng.integers(0, 2))]) - int(rng.integers(0, 2)) if rng.random() < 0.3 else -1)
    return pack("gpu_disk_lifetime", pool.cols(40, 0.25, 1.0, LIFETIME_MINS))


def many_groups(seed=75):
    """Attribute column 0 has a distinct value per host (130 hosts).  Jobs first, before anything is
    preempted: attribute-equals and balanced groups whose cotasks hold exactly 32 / 33 / 64 / 65 / 100
    distinct values, the target host's value last, minimum above and below the distinct count; jobs with
    5-8 groups.  Later, after decisions with 40+ victims, unique groups whose excluded host sits past
    entry 32 of the preempted-host list."""
    pool = _Pool(seed)
    rng = pool.rng
    pool.n_attr = 2
    H = 130
    us = [pool.user(2.0, 2048.0) for _ in range(30)]
    hosts = []
    for i in range(H):
        h = pool.host(attr=[i + 1, int(rng.integers(1, 4))], key=float(i))
        hosts.append(h)
        for _ in range(int(rng.integers(2, 8))):
            pool.task(us[int(rng.integers(len(us)))], h, float(rng.choice([0.5, 1.0])), 512.0 * float(rng.integers(1, 3)))
    big_user = pool.user(0.25, 256.0)
    hb1, hb2 = pool.host(attr=[200, 1], key=-2.0), pool.host(attr=[201, 2], key=-1.0)
    for h in (hb1, hb2):
        for _ in range(48):
            pool.task(big_user, h, 0.25, 256.0)
    # target hosts: spare, greatest names, values 300+
    targets = [pool.host(spare=(4.0, 4096.0, 0.0), attr=[300 + k, 1], key=1000.0 + k) for k in range(8)]
    for h in targets:                       # a task, or the host's attributes read as nil
        pool.task(us[0], h, 0.5, 512.0)
    pu = [pool.user(100.0, 102400.0) for _ in range(4)]
    others = [h for h in hosts]
    rng.shuffle(others)

    def cot(n_distinct, target, repeat=0):
        hs = others[:n_distinct - 1] + [target] + others[:repeat]
        return hs

    AE, BAL, UNI = abi.GROUP_ATTR_EQUALS, abi.GROUP_BALANCED, abi.GROUP_UNIQUE
    for k, n in enumerate((32, 33, 64, 65, 100)):
        g = pool.group(AE, 0, 1, cot(n, targets[k]))
        pool.job(pu[k % 4], 1.0, 1024.0, groups=[g])
    # balanced, every value once: minimum above the distinct count makes the target's value too frequent
    for k, (n, mn) in enumerate(((33, 40), (64, 65), (70, 100), (70, 3), (64, 2))):
        g = pool.group(BAL, 0, mn, cot(n, targets[5 + k % 3]))
        pool.job(pu[k % 4], 1.0, 1024.0, groups=[g])
    # balanced with one value twice (max frequency 2): hosts with that value fail
    g = pool.group(BAL, 0, 1, cot(80, targets[7], repeat=1))
    pool.job(pu[0], 1.0, 1024.0, groups=[g])
    # 5-8 groups per job: the scalar walk
    for ng in (5, 6, 7, 8):
        gs = [pool.group(AE, 1, 1, others[:3]) for _ in range(ng - 2)]
        gs.append(pool.group(UNI, -1, 1, [targets[(ng + 1) % 8]]))
        gs.append(pool.group(BAL, 0, 50 if ng % 2 else 1, cot(20, targets[ng % 8])))
        pool.job(pu[ng % 4], 1.0, 1024.0, groups=gs)
    # mass preemptions on hb1 then hb2, then unique groups (preempted entries past 32)
    pool.job(pu[0], 10.0, 10240.0)
    pool.job(pu[1], 2.0, 2048.0)
    pool.job(pu[2], 6.0, 6144.0)
    for i in range(6):
        g = pool.group(UNI, -1, 1, others[i:i + 2])
        pool.job(pu[i % 4], 0.5, 512.0, groups=[g])
    for i in range(20):
        kind = int(rng.choice([AE, BAL, UNI]))
        gs = [pool.group(kind, int(rng.integers(0, 2)), int(rng.integers(1, 80)),
                         [others[int(x)] for x in rng.integers(0, H, int(rng.integers(0, 90)))])
              for _ in range(int(rng.integers(1, 7)))]
        pool.job(pu[i % 4], float(rng.choice([0.5, 1.0, 2.0])), 512.0 * float(rng.integers(1, 5)), groups=gs)
    return pack("many_groups", pool.cols(64, 0.5, 1.0))


def spare_only_hosts(seed=76):
    """Hosts with spare and no task (attribute 7 in column 0, location 1, the greatest names) next to
    ordinary hosts; jobs with attribute, novel-host, unique-group, attribute-group and checkpoint-location
    constraints before and after the first synthetic task lands on a spare-only host."""
    pool = _Pool(seed)
    rng = pool.rng
    bg, hosts = _background(pool, 50, 15, (3, 9), spare_frac=0.0)
    for h in hosts[::7]:
        pool.h[h]["location"] = 1
    z = [pool.host(spare=(4.0, 4096.0, 0.0), location=1, attr=[7, 7, 7], key=10.0 + k) for k in range(4)]
    pu = [pool.user(100.0, 102400.0) for _ in range(4)]
    AE, BAL, UNI = abi.GROUP_ATTR_EQUALS, abi.GROUP_BALANCED, abi.GROUP_UNIQUE
    pool.job(pu[0], 1.0, 1024.0, attrs=[(0, 7)])               # nil attributes: no host
    pool.job(pu[1], 1.0, 1024.0, ckpt=1)                        # spare-only hosts have no location yet
    pool.job(pu[2], 1.0, 1024.0, groups=[pool.group(UNI, -1, 1, [])])
    pool.job(pu[3], 1.0, 1024.0, groups=[pool.group(AE, 0, 1, [], [7])])
    pool.job(pu[0], 1.0, 1024.0, novel=[z[3]])                  # novel passes on a host without tasks
    pool.job(pu[1], 1.0, 1024.0, attrs=[(0, 7)])                # now z[3] has a task
    pool.job(pu[2], 1.0, 1024.0, novel=[z[3]])
    pool.job(pu[3], 1.0, 1024.0, ckpt=1)
    pool.job(pu[0], 1.0, 1024.0, groups=[pool.group(AE, 0, 1, [], [7])])
    pool.job(pu[1], 1.0, 1024.0, groups=[pool.group(UNI, -1, 1, [z[3]])])
    pool.job(pu[2], 1.0, 1024.0, groups=[pool.group(BAL, 1, 3, [z[3], z[2], hosts[0]])])
    for i in range(16):
        kind = rng.integers(0, 5)
        kw = [dict(attrs=[(int(rng.integers(0, 3)), 7)]), dict(ckpt=int(rng.integers(0, 2))),
              dict(novel=[z[int(rng.integers(0, 4))]]), dict(groups=[pool.group(UNI, -1, 1, [])]),
              dict(groups=[pool.group(AE, int(rng.integers(0, 3)), 1, [], [7])])][kind]
        pool.job(pu[i % 4], float(rng.choice([0.5, 1.0, 2.0])), 512.0 * float(rng.integers(1, 5)), **kw)
    return pack("spare_only_hosts", pool.cols(40, 0.5, 1.0))


SAFE, MIN_DIFF = 1.0, 0.25


def eligibility_edges(seed=77):
    """DRUs on a power-of-two grid.  Users A and B are over their count quota, so only their own tasks are
    eligible for their jobs: A's first job needs A's task at DRU exactly `safe_dru_threshold`, B's first job
    could only use B's task exactly `min_dru_diff` above the job's pending DRU (and finds no host), B's second
    job takes B's task above that.  Then jobs that find no host between decisions, and more decidable jobs
    than `max_preemption`."""
    pool = _Pool(seed)
    rng = pool.rng
    bg = [pool.user(64.0, 65536.0) for _ in range(10)]         # background DRUs stay far below SAFE
    hosts = []
    for _ in range(30):
        h = pool.host()
        hosts.append(h)
        for _ in range(int(rng.integers(2, 6))):
            pool.task(bg[int(rng.integers(len(bg)))], h, 0.5, 512.0)
    a = pool.user(1.0, 1024.0, count_quota=1.0)
    e1, e2, e3 = pool.host(key=5.0), pool.host(key=6.0), pool.host(key=4.0)
    pool.task(a, e1, 0.5, 512.0)                               # DRU 0.5
    safe_task = pool.task(a, e1, 0.5, 512.0)                   # DRU 1.0 == SAFE
    b = pool.user(1.0, 1024.0, count_quota=1.0)
    pool.task(b, hosts[0], 0.5, 512.0, prio=90)                # DRU 0.5, sorts before B's jobs (prio 70)
    diff_task = pool.task(b, e2, 0.75, 768.0)                  # DRU 1.25 = pending DRU 1.0 + MIN_DIFF
    pool.task(b, e3, 0.25, 256.0)                              # DRU 1.5
    safe_job = pool.job(a, 0.5, 512.0, prio=90)                # pending DRU 0.5: only the SAFE task qualifies
    diff_job = pool.job(b, 0.5, 512.0, prio=70)                # pending DRU 1.0: e2 alone is large enough
    pool.job(b, 0.25, 256.0, prio=70)                          # pending DRU 0.75: e3's 1.5 (and e2's 1.25)
    mid = pool.user(1.0, 1024.0)            # victims for the later jobs, too little memory for the first ones
    for i in range(60):
        pool.task(mid, hosts[i % len(hosts)], 0.25, 1.0)
    pu = [pool.user(64.0, 65536.0) for _ in range(4)]
    for i in range(30):
        if i % 4 == 3:
            pool.job(pu[i % 4], 1000.0, 16.0)                 # no host is large enough
        else:
            pool.job(pu[i % 4], float(rng.choice([0.25, 0.5, 1.0])), float(rng.integers(1, 4)))
    c = pool.cols(12, MIN_DIFF, SAFE)
    c["edges"] = dict(safe_task=safe_task, safe_job=safe_job, diff_task=diff_task, diff_job=diff_job)
    return pack("eligibility_edges", c)


CASES = [crowded_hosts, mass_preemption, synthetic_victims, gpu_disk_lifetime, many_groups, spare_only_hosts,
         eligibility_edges]


def all_cases():
    """Every case and its off-grid twin."""
    out = []
    for make in CASES:
        c = make()
        out += [c, off_grid_twin(c)]
    return out


# ------------------------------------------------------------------------------------ what a run reached
def regimes(case, decisions):
    """What a walk's decisions reached, from the inputs and the decisions alone (the columns of the table
    in the commit message that introduced these cases)."""
    c = case["cols"]
    run, pend = c["run"], c["pend"]
    R = len(run["user"])
    H = len(c["host"]["name_rank"])
    real = np.bincount(run["host"], minlength=H)
    syn = np.zeros(H, np.int64)
    max_items = int(real.max()) if R else 0
    crossed_by_syn = False
    owner = list(run["user"])
    preempted = []
    most_v = most_vu = 0
    syn_victims = 0
    gpu_dec = 0
    max_groups = 0
    max_distinct = 0
    for d in decisions:
        p = d["pending_idx"]
        # the walk step that made this decision saw the synthetic tasks of the decisions before it
        items = real + syn
        max_items = max(max_items, int(items.max()))
        crossed_by_syn |= bool(np.any((real <= 64) & (items > 64)))
        gl = pend["groups"][p]
        max_groups = max(max_groups, len(gl))
        for gi in gl:
            g = c["groups"][gi]
            if g["kind"] == abi.GROUP_UNIQUE:
                continue
            col = g["attr_col"]
            vals = [int(c["host"]["attr"][col][h]) if 0 <= col < c["host"]["attr"].shape[0] else 0 for h in preempted]
            max_distinct = max(max_distinct, len(set(vals + g["cot_attrs"])))
        vs = d["victims"]
        most_v = max(most_v, len(vs))
        most_vu = max(most_vu, len({owner[i] for i in vs}))
        syn_victims += sum(1 for i in vs if i >= R)
        if pend["gpus"][p] > 0 and d["gpus"] > 0:
            gpu_dec += 1
        preempted += [run["host"][i] if i < R else decisions[i - R]["host"] for i in vs]
        syn[d["host"]] += 1
        owner.append(int(pend["user"][p]))
    return dict(most_real_tasks=int(real.max()) if R else 0, most_items=max_items, crossed_by_syn=crossed_by_syn,
                decisions=len(decisions), most_victims=most_v, most_victim_users=most_vu,
                synthetic_victims=syn_victims, gpu_decisions=gpu_dec, most_groups=max_groups,
                most_distinct_values=max_distinct)
