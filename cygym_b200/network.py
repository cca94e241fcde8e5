"""Networks for the batched step path: the flattened, struct-of-arrays form of the reference's
Device / App / OperatingSystem / Vulnerability / Exploit / Subnet object graph.

A `Network` is what every env of a VectorCyberDefenseEnv shares (the base graph in CSR with
ascending neighbour lists and pair multiplicities == the `_outnbrs` cache of
volt_typhoon_env.py:456-473, per-device statics, the device x exploit applicability bits) plus
the template dynamic state a reset() copies into every env (canonical layout of
include/cygym_b200.h).

`synthetic_network()` builds one directly, without igraph / pymetis, following what
initialize_environment() (volt_typhoon_env.py:1485-1900) produces: directed Barabasi-Albert
(m=2) clusters joined by router edges, DomainControllers = highest-degree devices
(:1583, :1634, :1655), attacker-owned sample (:1584, :1700-1725) with its star
(CDSimulatorComponents.py:722-748; sparse for M >= 500, volt:1399-1429), one reachable
neighbour per owned device (:1738-1838), Bernoulli(0.4) initial compromise (:45, :1846-1851),
bootstrap workloads (:1853-1864), and vulnerability bits drawn from a synthetic CVE table with
attach probability exploitabilityScore/10 (:1664-1667, :1697-1700).
"""
import math

import numpy as np

from . import cve as CVE
from ._capi import (DEV_COMP, DEV_HASWL, DEV_KNOWN, DEV_NYA, DEV_OWNED, DEV_PT_SHIFT, NSCAL, S_PREV_X, ST_DC, ST_NAPPS_SHIFT,
                    ST_REACH, ST_SERVER, ST_VULN_SHIFT)

DEFAULT_CFG = dict(
    X=6, n_exploits=2, Min_network_size=2, work_scale=1.0, comp_scale=30.0, def_scale=1.0, gamma=0.99,
    default_high=3, lambda_events=0.7, p_add=0.1, p_attacker=0.0, evolve_period=2,
    workload_period_base=50, workload_period_max=200, workload_cap=-1, scaling_vulnerability=1, turbo=0,
    zero_day=0, zero_day_mask=0, def_space_n=14,
    turbo_fraction_clients=0.05, turbo_fraction_servers=0.02, turbo_max_clients=200, turbo_max_servers=40, turbo_ramp_steps=200,
)


class Network:
    def __init__(self, row_ptr, col, mult, dev_static, os_val, ver_val, cfg, template=None, cve_table=None):
        self.row_ptr = np.ascontiguousarray(row_ptr, np.int32)
        self.col = np.ascontiguousarray(col, np.int32)
        self.mult = np.ascontiguousarray(mult, np.uint8)
        self.dev_static = np.ascontiguousarray(dev_static, np.uint32)
        self.os_val = np.ascontiguousarray(os_val, np.float32)
        self.ver_val = np.ascontiguousarray(ver_val, np.float32)
        self.cfg = dict(cfg)
        self.M = int(self.cfg["M"])
        self.E = int(len(self.col))
        self.W = (self.M + 31) // 32
        self.EW = max(1, (self.E + 31) // 32)
        self.X = int(self.cfg["X"])
        self.cve_table = cve_table
        self.template = template if template is not None else self.blank_template()
        assert len(self.row_ptr) == self.M + 1 and self.row_ptr[-1] == self.E

    def blank_template(self, xcap=16):
        scal = np.zeros(NSCAL, np.uint32)
        scal[S_PREV_X] = 0xFFFF  # _prev_att_potential is None
        return dict(dev=np.zeros(self.M, np.uint32), ckpt=np.zeros(self.M, np.uint32),
                    blocked=np.zeros(self.EW, np.uint32), extra=np.zeros(0, np.uint32), scal=scal)

    @property
    def obs_dims(self):
        """(defender, attacker, full) observation widths (CyberDefenseEnv.py:241/194/146)."""
        return 6 * self.M, 4 * self.M + self.X, 6 * self.M

    def algorithmic_bytes_per_step(self, obs=False):
        """SURVEY.md section 8(d): bytes one env-step must move."""
        M, E = self.M, self.E
        b = 2 * 4 * M + (E + 7) // 8 + 2 * 64 + (4 + (M + 7) // 8) + 12
        if obs:
            b += 4 * (5 * M + 3)
        return b

    @classmethod
    def from_arrays(cls, d, cfg, template=None):
        return cls(d["row_ptr"], d["col"], d["mult"], d["dev_static"], d["os_val"], d["ver_val"], cfg, template)


def _directed_ba(n, m, rng):
    """Edges (new -> old) of a directed Barabasi-Albert graph on nodes 0..n-1 (igraph Graph.Barabasi
    semantics as used at CDSimulatorComponents.py:629: each new node attaches m out-edges to earlier
    nodes with probability proportional to in-degree + 1; repeats allowed => multi-edges)."""
    edges = []
    weight = np.ones(n, np.float64)
    for i in range(1, n):
        k = min(m, i) if i >= m else i
        p = weight[:i] / weight[:i].sum()
        targets = rng.choice(i, size=k, replace=True, p=p)
        for t in targets:
            edges.append((i, int(t)))
            weight[t] += 1.0
    return edges


def synthetic_network(M=100, num_of_device=None, n_subnets=8, seed=0, n_cve_rows=256, init_ratio_compromise=0.4,
                      vulns_per_exploit=24, **overrides):
    """One shared network + template state of the named shape (BASELINE.json configs C2-C4)."""
    rng = np.random.default_rng(seed)
    if num_of_device is None:
        num_of_device = max(1, M - 10)  # Max_network_size = numOfDevice + 10 (volt_typhoon_do.py:1473)
    cfg = dict(DEFAULT_CFG)
    cfg.update(overrides)
    cfg["M"] = M
    cfg["numOfDevice"] = num_of_device
    X, n_exploits = cfg["X"], cfg["n_exploits"]
    cfg["att_space_n"] = n_exploits + 3

    # --- topology: per-subnet BA clusters + router ring --------------------------------------------
    n_subnets = max(1, min(n_subnets, M))
    pair = {}

    def add_edge(u, v):
        if u != v:
            pair[(u, v)] = pair.get((u, v), 0) + 1

    bounds = np.linspace(0, M, n_subnets + 1).astype(int)
    routers = []
    for s in range(n_subnets):
        lo, hi = int(bounds[s]), int(bounds[s + 1])
        if hi <= lo:
            continue
        routers.append(lo)
        for (a, b) in _directed_ba(hi - lo, 2, rng):
            add_edge(lo + a, lo + b)
    for i in range(len(routers)):
        if len(routers) > 1:
            a, b = routers[i], routers[(i + 1) % len(routers)]
            add_edge(a, b)
            add_edge(b, a)
    deg = np.zeros(M, np.int64)
    for (u, v), c in pair.items():
        deg[u] += c
        deg[v] += c

    # --- roles -------------------------------------------------------------------------------------
    n_dc = max(1, int(math.ceil(num_of_device / 50.0)))
    n_owned = max(1, int(round(num_of_device * 0.05)))
    by_degree = sorted(range(M), key=lambda d: (-deg[d], d))
    forced_active = set(by_degree[:max(3, n_dc)])
    dcs = set(by_degree[:n_dc])
    owned = set(int(x) for x in rng.choice(M, size=min(n_owned, M), replace=False))
    active = set(range(num_of_device)) | forced_active | owned
    if M < 500:  # dense star: owned -> every other device (CDSimulatorComponents.py:735-737)
        for o in sorted(owned):
            for v in range(M):
                add_edge(o, v)
    else:        # sparse: every DC + a few random others (volt:1399-1429)
        k_extra = max(1, int(round(math.log2(M) / 2)))
        for o in sorted(owned):
            for v in sorted(dcs):
                add_edge(o, v)
            for v in rng.choice(M, size=k_extra, replace=False):
                add_edge(o, int(v))
        # ... and the bidirectional hub-star among the active owned devices (hub = lowest id) that the reference's FIRST
        # evolve_network() adds to the graph (CyberDefenseEnv.py:738-774): generated as base edges, i.e. the network as it
        # stands after that first call and the cache rebuild that follows it (volt:1329 -> :456).  Without it every env
        # would carry 2 (n_owned - 1) extra edges in its per-env list from the second step on.
        oa = sorted(o for o in owned if o in active)
        for i in oa[1:]:
            if (oa[0], i) not in pair:
                add_edge(oa[0], i)
            if (i, oa[0]) not in pair:
                add_edge(i, oa[0])
    for (u, v) in list(pair):
        pair[(u, v)] = min(pair[(u, v)], 4)

    rows = [[] for _ in range(M)]
    for (u, v), c in pair.items():
        rows[u].append((v, c))
    row_ptr, col, mult = [0], [], []
    for u in range(M):
        for (v, c) in sorted(rows[u]):
            col.append(v)
            mult.append(c)
        row_ptr.append(len(col))

    reach = set()
    for o in sorted(owned):
        nb = [v for (v, _) in sorted(rows[o])]
        if nb:
            reach.add(int(nb[int(rng.integers(len(nb)))]))

    # --- applicability bits from the synthetic CVE table -------------------------------------------
    table = CVE.synthetic_cve_table(n_cve_rows, seed=seed + 7)
    score = np.asarray(table["exploitabilityScore"], np.float64)
    targets = []
    for e in range(n_exploits):
        t = set(int(x) for x in rng.choice(n_cve_rows, size=min(vulns_per_exploit, n_cve_rows), replace=False))
        t.add(e % n_cve_rows)  # rows 0/1 are the two hard-coded Volt Typhoon ids
        targets.append(t)
    dev_static = np.zeros(M, np.uint32)
    n_app_ids = 3
    for d in range(M):
        w = 0
        is_dc = d in dcs
        napps = 3 + (2 if is_dc else 4)
        n_app_ids += napps - 3
        if is_dc:
            w |= ST_DC
        else:
            w |= ST_SERVER  # every non-DC device ends up wtype='server' (volt:1680-1683)
        if d in reach:
            w |= ST_REACH
        w |= napps << ST_NAPPS_SHIFT
        attached = set()
        for _ in range(napps):
            r = int(rng.integers(n_cve_rows))
            if rng.random() < score[r] / 10.0:
                attached.add(r)
        for e in range(n_exploits):
            if attached & targets[e]:
                w |= 1 << (ST_VULN_SHIFT + e)
        dev_static[d] = w
    cfg["n_app_ids"] = n_app_ids
    os_val = np.arange(M, dtype=np.float32)  # OS.id == device index (CDSimulatorComponents.py:663)
    ver_val = rng.integers(1, 4, size=M).astype(np.float32)

    # --- template dynamic state --------------------------------------------------------------------
    dev = np.zeros(M, np.uint32)
    for d in range(M):
        w = 0
        if d not in active:
            w |= DEV_NYA
        if d in owned:
            w |= DEV_COMP | DEV_OWNED | DEV_KNOWN
        if d in active and rng.random() < init_ratio_compromise:
            w |= DEV_COMP | DEV_KNOWN
        dev[d] = w
    # bootstrap workloads (volt:1853-1864 -> _scaled_numloads): servers ~ round(10 * n_active/50)
    n_active = len(active)
    servers = [d for d in sorted(active) if not (dev_static[d] & ST_DC)]
    clients = [d for d in sorted(active) if (dev_static[d] & ST_DC)]
    n_s = min(len(servers), max(1, int(round(10 * n_active / 50.0))))
    n_c = min(len(clients), max(1, int(round(100 * n_active / 50.0))))
    for pool, k in ((clients, n_c), (servers, n_s)):
        if not pool:
            continue
        for d in rng.choice(pool, size=k, replace=False):
            pt = int(math.ceil(rng.triangular(0, 2, 5)))
            pt = min(5, max(1, pt))
            dev[int(d)] |= DEV_HASWL | (pt << DEV_PT_SHIFT)
    scal = np.zeros(NSCAL, np.uint32)
    scal[S_PREV_X] = 0xFFFF
    E = len(col)
    template = dict(dev=dev, ckpt=np.zeros(M, np.uint32), blocked=np.zeros(max(1, (E + 31) // 32), np.uint32),
                    extra=np.zeros(0, np.uint32), scal=scal)
    net = Network(row_ptr, col, mult, dev_static, os_val, ver_val, cfg, template, cve_table=table)
    net.n_dc, net.n_owned, net.n_subnets = n_dc, n_owned, n_subnets
    return net


def network_from_golden(g):
    """Network + template from a tests/golden/*.npz trajectory (recorded from the live reference)."""
    import json
    meta = json.loads(str(g["meta"]))
    d = {k: np.array(g["net_" + k]) for k in ("row_ptr", "col", "mult", "dev_static", "os_val", "ver_val")}
    template = {k: np.array(g["init_" + k]) for k in ("dev", "ckpt", "blocked", "extra", "scal")}
    return Network.from_arrays(d, meta["cfg"], template), meta
