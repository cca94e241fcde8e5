"""Snapshots: networks + env state in and out of the struct-of-arrays form.

The reference persists experiments as pickled env objects (`initial_net_DO_its<N>.pkl`, init_experiments.py:53-62,
volt_typhoon_env.py:1877-1895, reloaded by reset(from_init=True), :1904-1925).  Two entry points:

 * `from_reference_env(env)`  -- flatten a LIVE reference env object (e.g. one just unpickled in a process that
   can import the reference) into a `Network` whose template is the env's current state.  Duck-typed: it only
   reads the attributes listed in SURVEY.md section 8(a)/(b) and never imports the reference.
 * `save_npz / load_npz`      -- our own portable snapshot (numpy .npz) of a Network + template, so that the same
   experiment can be re-run where the reference is not installed (the GPU box).
"""
import json

import numpy as np

from . import _capi as K
from ._capi import (CK_COMP, CK_HASWL, CK_KNOWN, CK_NYA, CK_REACH, CK_VALID, DEV_ACTSET, DEV_BUSY_MASK, DEV_BUSY_SHIFT,
                    DEV_BUSYSET, DEV_CBY_MASK, DEV_CBY_SHIFT, DEV_COMP, DEV_HASWL, DEV_KNOWN, DEV_NYA, DEV_OWNED, DEV_PT_MASK,
                    DEV_PT_SHIFT, DEV_REMOVED, NSCAL, ST_DC, ST_NAPPS_SHIFT, ST_REACH, ST_SERVER, ST_VULN_SHIFT)
from .network import Network


def save_npz(path, net: Network):
    t = net.template
    np.savez_compressed(path, row_ptr=net.row_ptr, col=net.col, mult=net.mult, dev_static=net.dev_static,
                        os_val=net.os_val, ver_val=net.ver_val, cfg=np.asarray(json.dumps(net.cfg)),
                        **{"t_" + k: np.asarray(v, np.uint32) for k, v in t.items()})
    return path


def load_npz(path):
    g = np.load(path)
    template = {k[2:]: np.array(g[k]) for k in g.files if k.startswith("t_")}
    d = {k: np.array(g[k]) for k in ("row_ptr", "col", "mult", "dev_static", "os_val", "ver_val")}
    return Network.from_arrays(d, json.loads(str(g["cfg"])), template)


def from_reference_env(env):
    """Flatten a live reference Volt_Typhoon_CyberDefenseEnv (its graph cache must be current: call
    env._rebuild_graph_cache() first, as DoubleOracle.restore does, do_agent.py:891-895)."""
    net = env.simulator.subnet.net
    M = len(net)
    if sorted(net.keys()) != list(range(M)):
        raise ValueError("device ids must be 0..M-1")
    row_ptr, col, mult = [0], [], []
    for u in range(M):  # _outnbrs: ascending neighbour ids, multi-edges as repeats (volt:456-473)
        prev = None
        for v in env._outnbrs.get(u, []):
            v = int(v)
            if prev is not None and v < prev:
                raise ValueError("neighbour list not ascending")
            if v == prev:
                mult[-1] += 1
            else:
                col.append(v)
                mult.append(1)
            prev = v
        row_ptr.append(len(col))
    exploits = list(env.simulator.exploits)
    eid_of = {exp.id: i for i, exp in enumerate(exploits)}
    X = int(env.MaxExploits)
    dev_static = np.zeros(M, np.uint32)
    os_val = np.zeros(M, np.float32)
    ver_val = np.zeros(M, np.float32)
    dev = np.zeros(M, np.uint32)
    ckpt = np.zeros(M, np.uint32)
    busyset = {d.id for d in (getattr(env, "_busy_devices", None) or ())}
    has_sets = hasattr(env, "_active_ids") and hasattr(env, "_inactive_ids")
    for i in range(M):
        d = net[i]
        w = 0
        if d.device_type == "DomainController":
            w |= ST_DC
        if d.wtype == "server":
            w |= ST_SERVER
        if d.reachable_by_attacker:
            w |= ST_REACH
        w |= min(255, len(d.apps)) << ST_NAPPS_SHIFT
        for e, exp in enumerate(exploits):
            if any(vul.id in exp.target for app in d.apps.values() for vul in app.vulnerabilities.values()):
                w |= 1 << (ST_VULN_SHIFT + e)
        dev_static[i] = w
        os_val[i] = env.os_to_float(d.OS)
        try:
            ver_val[i] = float(d.version)
        except Exception:
            ver_val[i] = -1.0
        s = 0
        s |= DEV_COMP if d.isCompromised else 0
        s |= DEV_KNOWN if d.Known_to_attacker else 0
        s |= DEV_NYA if d.Not_yet_added else 0
        s |= DEV_OWNED if d.attacker_owned else 0
        s |= DEV_REMOVED if d.removed_before else 0
        if d.workload is not None:
            s |= DEV_HASWL | (int(d.workload.processing_time) << DEV_PT_SHIFT)
        s |= int(d.busy_time) << DEV_BUSY_SHIFT
        for x in d.compromised_by:
            s |= (1 << eid_of[x]) << DEV_CBY_SHIFT
        if i in busyset:
            s |= DEV_BUSYSET
        if has_sets and i in env._active_ids:
            s |= DEV_ACTSET
        dev[i] = s
        c = getattr(env, "_device_ckpts", {}).get(i)
        if c is not None:
            k = CK_VALID
            k |= CK_COMP if c["isCompromised"] else 0
            k |= CK_KNOWN if c["Known_to_attacker"] else 0
            k |= CK_NYA if c["Not_yet_added"] else 0
            k |= CK_REACH if c["reachable_by_attacker"] else 0
            if c["workload"]:
                k |= CK_HASWL | (int(c["workload"]["processing_time"]) << DEV_PT_SHIFT)
            k |= int(c["busy_time"]) << DEV_BUSY_SHIFT
            for x in c["compromised_by"]:
                k |= (1 << eid_of[x]) << DEV_CBY_SHIFT
            ckpt[i] = k
    E = len(col)
    eidx = {}
    for u in range(M):
        for e in range(row_ptr[u], row_ptr[u + 1]):
            eidx[(u, col[e])] = e
    blocked = np.zeros(max(1, (E + 31) // 32), np.uint32)
    for (u, v) in getattr(env, "_blocked", ()):  # blocked pairs outside the cache cannot occur after a rebuild
        e = eidx.get((int(u), int(v)))
        if e is not None:
            blocked[e >> 5] |= np.uint32(1 << (e & 31))
    scal = np.zeros(NSCAL, np.uint32)
    scal[K.S_STEP] = env.step_num
    fl = (K.FL_HAS_CKPT if env.checkpoint is not None else 0) | (K.FL_SETS_INIT if has_sets else 0)
    if getattr(env.simulator.detector, "trained", False):
        fl |= K.FL_DET_TRAINED
    for i, exp in enumerate(exploits):
        if exp.discovered:
            fl |= 1 << (K.FL_DISC_SHIFT + i)
    scal[K.S_FLAGS] = fl
    prev = getattr(env, "_prev_att_potential", None)
    scal[K.S_PREV_X] = 0xFFFF if prev is None else int(round(prev * M / env.γ))
    scal[K.S_DEF_STEP], scal[K.S_ATT_STEP] = env.defender_step, env.attacker_step
    scal[K.S_LOGS] = len(env.simulator.logger.logs)
    scal[K.S_COMPCNT], scal[K.S_WORK] = env.compromised_devices_cnt, env.work_done
    f32 = np.array([env.defensive_cost, env.clearning_cost], np.float32).view(np.uint32)
    scal[K.S_DEFCOST], scal[K.S_CLEANCOST] = f32[0], f32[1]
    scal[K.S_SCAN], scal[K.S_REVERT], scal[K.S_CKPT] = env.scan_cnt, env.revert_count, env.checkpoint_count
    scal[K.S_EBLK], scal[K.S_EADD] = env.edges_blocked, env.edges_added
    zd = 0
    if env.zero_day:
        for i in (set(env.common_exploit_indices) | set(env.private_exploit_indices)):
            zd |= 1 << int(i)
    cfg = dict(
        M=M, X=X, n_exploits=len(exploits), numOfDevice=int(env.numOfDevice), Min_network_size=int(env.Min_network_size),
        work_scale=float(env.work_scale), comp_scale=float(env.comp_scale), def_scale=float(env.def_scale),
        gamma=float(env.γ), default_high=int(env.default_high), lambda_events=float(env.lambda_events),
        p_add=float(env.p_add), p_attacker=float(env.p_attacker), evolve_period=int(env._evolve_period),
        workload_period_base=int(env.workload_period_base), workload_period_max=int(env.workload_period_max),
        workload_cap=(-1 if env.workload_cap is None else int(env.workload_cap)),
        scaling_vulnerability=int(bool(env.scaling_vulnerability)), turbo=int(bool(env.turbo)),
        zero_day=int(bool(env.zero_day)), zero_day_mask=zd, att_space_n=int(env.attacker_action_space.n),
        def_space_n=int(env.defender_action_space.n), n_app_ids=int(env.get_num_app_indices()),
        turbo_fraction_clients=float(env.turbo_fraction_clients), turbo_fraction_servers=float(env.turbo_fraction_servers),
        turbo_max_clients=int(env.turbo_max_clients), turbo_max_servers=int(env.turbo_max_servers),
        turbo_ramp_steps=int(env.turbo_ramp_steps))
    template = dict(dev=dev, ckpt=ckpt, blocked=blocked, extra=np.zeros(0, np.uint32), scal=scal)
    return Network(row_ptr, col, mult, dev_static, os_val, ver_val, cfg, template)


# ---- the reference's own on-disk format: a pickled env object (init_experiments.py:53-62, volt_typhoon_env.py:1904-1925) ----
def load_reference_pickle(path):
    """`initial_net_DO_its<N>.pkl` -> Network (template = the pickled env's state).  Unpickling needs the reference's
    classes importable in this process (the file stores objects of volt_typhoon_env / CDSimulatorComponents); this
    module itself never imports them.  Returns (network, env_object)."""
    import pickle
    with open(path, "rb") as f:
        env = pickle.load(f)
    if isinstance(env, dict):
        raise ValueError("old dict snapshot {'simulator', 'state'} (volt:1884-1888): load it through a reference env's reset()")
    env._rebuild_graph_cache()  # what reset(from_init=True) does right after loading (volt:1933-1936)
    return from_reference_env(env), env


def apply_state_to_reference_env(env, net, state):
    """The inverse of from_reference_env for the DYNAMIC state: write a canonical state (dict of numpy arrays dev / ckpt
    / blocked / extra / scal for ONE env, layout of include/cygym_b200.h) stepped on `net` into the live reference env
    object it was flattened from, so that the reference can go on from where the kernels stopped -- or be pickled back
    to disk.  Duck-typed: classes (Workload) are taken from the objects already in the graph."""
    import sys
    sim = env.simulator
    devs = sim.subnet.net
    M = net.M
    dev = np.asarray(state["dev"], np.uint32)
    ck = np.asarray(state["ckpt"], np.uint32)
    sc = np.asarray(state["scal"], np.uint32)
    exploits = list(sim.exploits)
    Workload = getattr(sys.modules[type(devs[0]).__module__], "Workload")
    for i in range(M):
        d, w = devs[i], int(dev[i])
        d.isCompromised = bool(w & DEV_COMP)
        d.Known_to_attacker = bool(w & DEV_KNOWN)
        d.Not_yet_added = bool(w & DEV_NYA)
        d.attacker_owned = bool(w & DEV_OWNED)
        d.removed_before = 1 if w & DEV_REMOVED else 0
        d.busy_time = float((w >> DEV_BUSY_SHIFT) & DEV_BUSY_MASK)
        if w & DEV_HASWL:
            wl = Workload()
            wl.processing_time = (w >> DEV_PT_SHIFT) & DEV_PT_MASK
            wl.adversarial, wl.assigned, wl.wtype = False, True, d.wtype
            d.workload = wl
        else:
            d.workload = None
        cb = (w >> DEV_CBY_SHIFT) & DEV_CBY_MASK
        d.compromised_by = type(d.compromised_by)(exploits[e].id for e in range(len(exploits)) if (cb >> e) & 1)
    env._device_ckpts = {}
    for i in range(M):
        k = int(ck[i])
        if k & CK_VALID:
            cb = (k >> DEV_CBY_SHIFT) & DEV_CBY_MASK
            env._device_ckpts[i] = dict(
                isCompromised=bool(k & CK_COMP), Known_to_attacker=bool(k & CK_KNOWN), Not_yet_added=bool(k & CK_NYA),
                reachable_by_attacker=bool(k & CK_REACH),
                workload=({"processing_time": (k >> DEV_PT_SHIFT) & DEV_PT_MASK, "adversarial": False} if k & CK_HASWL else None),
                busy_time=float((k >> DEV_BUSY_SHIFT) & DEV_BUSY_MASK),
                compromised_by=[exploits[e].id for e in range(len(exploits)) if (cb >> e) & 1])
    # extra (hub-star) edges go into the graph; the cache rebuild makes them visible and forgets the blocks (volt:476) ...
    g = sim.subnet.graph
    n_extra = int(sc[K.S_PREV_X]) >> 16
    have = set(g.get_edgelist())
    new_edges = [(u, v) for u, v, _ in K.extra_edges(np.asarray(state["extra"], np.uint32)[:n_extra])]
    add = [e for e in new_edges if e not in have]
    if add:
        g.add_edges(add)
    env._rebuild_graph_cache()
    # ... so the blocked set is put back after it
    blocked = set()
    bl = np.asarray(state["blocked"], np.uint32)
    for u in range(M):
        for e in range(int(net.row_ptr[u]), int(net.row_ptr[u + 1])):
            if (int(bl[e >> 5]) >> (e & 31)) & 1:
                blocked.add((u, int(net.col[e])))
    for u, v, is_blocked in K.extra_edges(np.asarray(state["extra"], np.uint32)[:n_extra]):
        if is_blocked:
            blocked.add((u, v))
    env._blocked = blocked
    env._busy_devices = {devs[i] for i in range(M) if int(dev[i]) & DEV_BUSYSET}
    if int(sc[K.S_FLAGS]) & K.FL_SETS_INIT:
        env._active_ids = {i for i in range(M) if int(dev[i]) & DEV_ACTSET}
        env._inactive_ids = {i for i in range(M) if not int(dev[i]) & DEV_ACTSET}
    else:
        for a in ("_active_ids", "_inactive_ids"):
            if hasattr(env, a):
                delattr(env, a)
    env.checkpoint = {"simulator": sim, "state": env.state} if int(sc[K.S_FLAGS]) & K.FL_HAS_CKPT else None  # an alias, as checkpoint_variables stores it
    for e, exp in enumerate(exploits):
        exp.discovered = bool((int(sc[K.S_FLAGS]) >> (K.FL_DISC_SHIFT + e)) & 1)
    pn = int(sc[K.S_PREV_X]) & 0xFFFF
    env._prev_att_potential = None if pn == 0xFFFF else env.γ * (pn / M)
    env.step_num, env.defender_step, env.attacker_step = int(sc[K.S_STEP]), int(sc[K.S_DEF_STEP]), int(sc[K.S_ATT_STEP])
    env.compromised_devices_cnt, env.work_done = int(sc[K.S_COMPCNT]), int(sc[K.S_WORK])
    env.defensive_cost = float(sc[K.S_DEFCOST:K.S_DEFCOST + 1].view(np.float32)[0])
    env.clearning_cost = float(sc[K.S_CLEANCOST:K.S_CLEANCOST + 1].view(np.float32)[0])
    env.scan_cnt, env.revert_count, env.checkpoint_count = int(sc[K.S_SCAN]), int(sc[K.S_REVERT]), int(sc[K.S_CKPT])
    env.edges_blocked, env.edges_added = int(sc[K.S_EBLK]), int(sc[K.S_EADD])
    # the hop log: the kernels keep its length; records beyond what is known are neutral placeholders
    logs = sim.logger.logs
    n = int(sc[K.S_LOGS])
    if len(logs) > n:
        del logs[n:]
    while len(logs) < n:
        logs.append({"time_step": 0, "from_device": 0, "to_device": 0, "kind": "D"})
    env.state = env._get_state()
    return env


def write_reference_pickle(path, env, net=None, state=None):
    """Write a reference-format snapshot (init_experiments.py:60-61: pickle.dump(env)) -- of `env` as it is, or, with
    (net, state), after the kernels' canonical state has been written into it."""
    import pickle
    if state is not None:
        apply_state_to_reference_env(env, net, state)
    with open(path, "wb") as f:
        pickle.dump(env, f)
    return path
