"""Drop-in single-env front end: the reset()/step() Gym surface of the reference's
Volt_Typhoon_CyberDefenseEnv (volt_typhoon_env.py:30) on top of the batched CUDA path (a batch of 1).

Callers in the reference (do_agent.py, IPPO.py, MAPPO.py, HMARL.py, meta_hierarchical_br.py ...) touch the env through
the members listed in SURVEY.md section 8(b); those are what this class provides, with the same names, argument
meaning, return shapes and error behaviour -- enough for the reference's UNMODIFIED DoubleOracle to be constructed
on it, checkpoint / restore it and roll games out on it (tests/test_dropin_reference_caller.py).

The Device / App / ... object graph itself is not rebuilt: state lives on the GPU as bit-planes.  What callers read
from it -- `env.simulator.subnet.net[id]` device attributes (IPPO.py:74-96, HMARL.py:126-159), `simulator.exploits`,
`simulator.logger.logs`, `simulator.subnet.graph.get_edgelist()` (meta_hierarchical_br.py:74-119),
`_get_ordered_devices()` -- are read-only VIEWS over one cached device-to-host copy of the canonical state per step.
"""
import numpy as np
import torch

from . import _capi as K
from ._capi import (DEV_BUSY_MASK, DEV_BUSY_SHIFT, DEV_CBY_MASK, DEV_CBY_SHIFT, DEV_COMP, DEV_HASWL, DEV_KNOWN, DEV_NYA,
                    DEV_OWNED, DEV_PT_MASK, DEV_PT_SHIFT, DEV_REMOVED, ST_DC, ST_NAPPS_SHIFT, ST_REACH, ST_SERVER)
from .network import Network, synthetic_network
from .vector_env import ActionBatch, VectorCyberDefenseEnv, decode_header

_COUNTER_SLOTS = {attr: (slot, is_float) for attr, _, slot, is_float in K.COUNTERS}


def _counter(scal, slot, is_float):
    """One counter from a host copy of an env's scalars."""
    return float(scal[slot: slot + 1].view(np.float32)[0]) if is_float else int(scal[slot])


# ---- read-only views of the object graph (CDSimulatorComponents.py:18-26, :219-242, :491-499; CDSimulator.py:663-679) ----
class _Workload:
    def __init__(self, processing_time, wtype):
        self.processing_time, self.wtype, self.adversarial, self.assigned = int(processing_time), wtype, False, True


class _OS:
    def __init__(self, ident, value):
        self.id, self._value = ident, value


class DeviceView:
    """`Device` attributes of one slot, decoded from the canonical device word (include/cygym_b200.h)."""

    def __init__(self, env, d):
        self._env, self.id = env, int(d)

    def _w(self):
        return int(self._env._snap()["dev"][self.id])

    def _st(self):
        return int(self._env._net.dev_static[self.id])

    isCompromised = property(lambda s: bool(s._w() & DEV_COMP))
    Known_to_attacker = property(lambda s: bool(s._w() & DEV_KNOWN))
    Not_yet_added = property(lambda s: bool(s._w() & DEV_NYA))
    attacker_owned = property(lambda s: bool(s._w() & DEV_OWNED))
    removed_before = property(lambda s: 1 if s._w() & DEV_REMOVED else 0)
    reachable_by_attacker = property(lambda s: bool(s._st() & ST_REACH))
    busy_time = property(lambda s: (s._w() >> DEV_BUSY_SHIFT) & DEV_BUSY_MASK)
    anomaly_score = 0.0  # stays 0 under fast_scan (volt_typhoon_env.py:46)
    device_type = property(lambda s: "DomainController" if s._st() & ST_DC else "Workstation")
    wtype = property(lambda s: "server" if s._st() & ST_SERVER else "client")
    version = property(lambda s: float(s._env._net.ver_val[s.id]))
    OS = property(lambda s: _OS(s.id, float(s._env._net.os_val[s.id])))
    n_apps = property(lambda s: (s._st() >> ST_NAPPS_SHIFT) & 0xFF)

    @property
    def workload(self):
        w = self._w()
        return _Workload((w >> DEV_PT_SHIFT) & DEV_PT_MASK, self.wtype) if w & DEV_HASWL else None

    @property
    def compromised_by(self):
        m = (self._w() >> DEV_CBY_SHIFT) & DEV_CBY_MASK
        return {self._env.simulator.exploits[e].id for e in range(len(self._env.simulator.exploits)) if (m >> e) & 1}

    def __setattr__(self, name, value):
        if name in ("_env", "id"):
            object.__setattr__(self, name, value)
        else:
            raise AttributeError(f"DeviceView.{name} is read-only: the device state lives on the GPU (step() changes it)")


class _NetView(dict):
    """`subnet.net`: id -> DeviceView (a real dict of views, so keys() / values() / items() / len() behave)."""


class _GraphView:
    """`subnet.graph`: the directed multigraph as callers read it (get_edgelist, vcount, ecount, neighbors)."""

    def __init__(self, env):
        self._env = env

    def get_edgelist(self):
        n, out = self._env._net, []
        for u in range(n.M):
            for e in range(int(n.row_ptr[u]), int(n.row_ptr[u + 1])):
                out.extend([(u, int(n.col[e]))] * int(n.mult[e]))
        out.extend((u, v) for u, v, _ in K.extra_edges(self._env._snap()["extra"][: self._env._n_extra()]))
        return out

    def vcount(self):
        return self._env._net.M

    def ecount(self):
        return int(self._env._net.mult.sum()) + self._env._n_extra()

    def neighbors(self, u, mode="out"):
        return sorted(v for (a, v) in self.get_edgelist() if a == int(u))


class _SubnetView:
    def __init__(self, env):
        self.net = _NetView((d, DeviceView(env, d)) for d in range(env._net.M))
        self.graph = _GraphView(env)
        self.partitions = None


class _ExploitView:
    def __init__(self, env, e):
        self._env, self._e, self.id = env, e, f"exploit-{e}"

    @property
    def discovered(self):
        return bool((int(self._env._snap()["scal"][K.S_FLAGS]) >> (K.FL_DISC_SHIFT + self._e)) & 1)


class _LoggerView:
    """`simulator.logger`: the hop log (CDSimulator.py:663-679).  The kernels keep its length (CYG_S_LOGS) and a ring of
    the last `log_cap` records; get_logs() returns a list of the full length whose last log_cap entries are the records
    ({"time_step", "from_device", "to_device", "kind"}; time_step is not tracked: the step path never reads it) and
    whose older entries are None -- callers take len() and tail slices (do_agent.py:51-62 keeps the last 2000)."""

    def __init__(self, env):
        self._env = env

    def _n(self):
        return int(self._env._snap()["scal"][K.S_LOGS])

    def get_logs(self):
        n = self._n()
        ring = self._env._snap().get("logs")
        if ring is None or len(ring) == 0:
            return [None] * n
        k = min(n, len(ring))
        return [None] * (n - k) + [{"time_step": None, "from_device": int(a), "to_device": int(b), "kind": "A"}
                                   for a, b in K.log_records(ring, n, k)]

    logs = property(lambda s: s.get_logs())

    def set_logs(self, logs):  # DoubleOracle.restore puts its snapshot back (do_agent.py:824-848): the log is env state here
        pass


class _DetectorView:
    def __init__(self, env):
        self._env = env

    trained = property(lambda s: bool(int(s._env._snap()["scal"][K.S_FLAGS]) & K.FL_DET_TRAINED))
    random_detection = False


class SimulatorView:
    def __init__(self, env):
        self.subnet = _SubnetView(env)
        self.exploits = [_ExploitView(env, e) for e in range(int(env._net.cfg["n_exploits"]))]
        self.logger = _LoggerView(env)
        self.detector = _DetectorView(env)
        self.system_time = 0


class Volt_Typhoon_CyberDefenseEnv:
    """reset(from_init) / step(action, agent_cnt) / step_grouped(groups) with the reference's 6-tuple return
    (state, raw_reward, shaped_reward, done, info, logs) (volt_typhoon_env.py:1333)."""

    MaxExploits = 6

    def __init__(self, network: Network = None, device="cuda:0", seed=0, env_id=0, xcap=32, venv_cls=None, log_cap=2048):
        """venv_cls: the batched backend (default and only product backend: VectorCyberDefenseEnv on CUDA; the CPU test
        suite injects a stand-in built on the host compile of the device source, tests/emu/emu_venv.py)."""
        d = self.__dict__
        d["_venv_cls"] = venv_cls or VectorCyberDefenseEnv
        d["_pending"] = {}               # counters assigned before the env is built (constructor-then-configure callers)
        d["_venv"] = None
        self.numOfDevice = 10            # init_experiments.py:41-42 defaults
        self.Max_network_size = 20
        self.mode = "defender"
        self.tech = "DO"
        self.debug = False
        self.zero_day = False
        self.snapshot_path = None
        self.time_budget_deadline = None
        self.time_budget_exceeded = False
        self.its = 1
        self.k_known, self.j_private = 1, 1
        self.private_exploit_id, self.private_exploit_ids, self.common_exploit_ids, self.unknown_pool_ids = None, [], [], []
        self.prior_pi = None
        self.alpha, self.khop, self.preknown = 0.5, 1, 0
        self._device, self._seed, self._env_id, self._xcap, self._log_cap = device, seed, env_id, xcap, int(log_cap)
        self.detector_fit_seed = None    # parity runs: seed of numpy's global stream before every detector fit
        self._net = network
        self._base_line = "Nash"
        self._scales = {}
        self._host = None   # cached canonical state on the host (one device->host copy per step)
        self._sim = None
        self.state = None
        if network is not None:
            self.numOfDevice, self.Max_network_size = network.cfg["numOfDevice"], network.M
            self._build()

    # ---- configuration attributes the callers set ----
    @property
    def base_line(self):
        return self._base_line

    @base_line.setter
    def base_line(self, name):
        if name != self._base_line and self._venv is not None:
            self._venv.set_base_line(name)
        self._base_line = name

    def _cfg_get(self, k):
        return self._scales.get(k, None if self._net is None else self._net.cfg[k])

    def _cfg_set(self, k, v):
        self._scales[k] = float(v)
        if self._venv is not None:  # kernel constants: rebuild the handle, keep the state
            st = self._venv.export_state()
            self._net.cfg[k] = float(v)
            self._venv.close()
            self.__dict__["_venv"] = self._venv_cls(self._net, 1, device=self._device, seed=self._seed, env_id0=self._env_id,
                                                    base_line=self._base_line, xcap=self._xcap, log_cap=self._log_cap, detector_slots=1)
            self._venv.import_state(st)

    work_scale = property(lambda s: s._cfg_get("work_scale"), lambda s, v: s._cfg_set("work_scale", v))
    comp_scale = property(lambda s: s._cfg_get("comp_scale"), lambda s, v: s._cfg_set("comp_scale", v))
    def_scale = property(lambda s: s._cfg_get("def_scale"), lambda s, v: s._cfg_set("def_scale", v))
    lambda_events = property(lambda s: s._cfg_get("lambda_events"), lambda s, v: s._cfg_set("lambda_events", v))
    p_add = property(lambda s: s._cfg_get("p_add"), lambda s, v: s._cfg_set("p_add", v))
    p_attacker = property(lambda s: s._cfg_get("p_attacker"), lambda s, v: s._cfg_set("p_attacker", v))

    def _build(self):
        for k, v in self._scales.items():
            self._net.cfg[k] = v
        if self._venv is not None:
            self._venv.close()
        self.__dict__["_venv"] = self._venv_cls(self._net, 1, device=self._device, seed=self._seed, env_id0=self._env_id,
                                                base_line=self._base_line, xcap=self._xcap, log_cap=self._log_cap, detector_slots=1)
        self._sim = SimulatorView(self)
        self._host = None
        for name, value in list(self._pending.items()):  # counters a caller set before initialize_environment()
            setattr(self, name, value)
        self._pending.clear()
        self.state = self._get_state()

    # ---- setup (volt_typhoon_env.py:1485-1900, :1904-2107) ----
    def initialize_environment(self, seed=None, n_subnets=None):
        """Builds a synthetic network of the configured size (numOfDevice, Max_network_size) and resets to it."""
        M = int(self.Max_network_size)
        self._net = synthetic_network(M, num_of_device=int(self.numOfDevice),
                                      n_subnets=n_subnets or max(1, M // 12), seed=self._seed if seed is None else seed)
        self._build()
        return self.state

    def reset(self, from_init=True):
        if self._venv is None:
            return self.initialize_environment()
        self._venv.reset()
        self._host = None
        self.state = self._get_state()
        return self.state

    def seed(self, seed=None):
        self._seed = 0 if seed is None else int(seed)
        return [self._seed]

    @property
    def simulator(self):
        return self._sim

    def _get_ordered_devices(self):
        """Devices sorted by id, trimmed to Max_network_size (CyberDefenseEnv.py:95-102)."""
        return [self._sim.subnet.net[i] for i in range(self._net.M)][: int(self.Max_network_size)]

    # ---- pickling: the reference ships env copies to worker processes (do_agent.py:642-705, volt_typhoon_do.py:346) ----
    def __getstate__(self):
        d = {k: v for k, v in self.__dict__.items() if k not in ("_venv", "_sim", "_host")}
        d["_pickled_state"] = None if self._venv is None else {k: np.array(v) for k, v in self._snap().items()}
        return d

    def __setstate__(self, d):
        st = d.pop("_pickled_state", None)
        self.__dict__.update(d)
        self.__dict__.update(_venv=None, _sim=None, _host=None)
        if self._net is not None:
            state = self.__dict__.get("state")
            self._build()
            if st is not None:
                self._venv.import_state({k: np.asarray(v, np.uint32)[None] for k, v in st.items()})
                self._host = None
            self.state = state

    # ---- sizes ----
    def get_num_action_types(self, mode=None):
        if mode == "defender":
            return 14
        if mode == "attacker":
            return 3
        raise ValueError("Invalid mode: must be either 'defender' or 'attacker'")

    def get_device_indices(self):
        return list(range(self._net.M))

    def get_num_exploit_indices(self):
        return int(self._net.cfg["n_exploits"])

    def get_num_app_indices(self):
        return int(self._net.cfg.get("n_app_ids", 0))

    # ---- host copy of the canonical state: ONE device->host transfer per step, shared by every view and counter ----
    def _snap(self):
        if self._host is None:
            c = self._venv.export_state()
            self._host = {k: v[0].cpu().numpy().view(np.uint32) for k, v in c.items()}  # .cpu() synchronises
        return self._host

    def _n_extra(self):
        return int(self._snap()["scal"][K.S_PREV_X]) >> 16

    # ---- counters: views of the env's scalars; callers zero them between rollouts (do_agent.py:192-196) ----
    def __getattr__(self, name):
        if name in _COUNTER_SLOTS:
            d = self.__dict__
            if d.get("_venv") is None:
                if name in d.get("_pending", {}):
                    return d["_pending"][name]
                raise AttributeError(name)
            return _counter(self._snap()["scal"], *_COUNTER_SLOTS[name])
        raise AttributeError(name)

    def __setattr__(self, name, value):
        if name in _COUNTER_SLOTS:
            if self.__dict__.get("_venv") is None:
                self._pending[name] = value  # replayed into the scalars by _build()
                return
            slot, is_float = _COUNTER_SLOTS[name]
            self._venv.scalars[0, slot] = int(np.float32(value).view(np.int32)) if is_float else int(value)
            self.__dict__["_host"] = None
        else:
            object.__setattr__(self, name, value)

    # ---- observations (CyberDefenseEnv.py:146/241/194) ----
    def _obs(self, mode, dtype):
        o = self._venv.observe(mode)
        return o[0].cpu().numpy().astype(dtype)

    def _get_state(self):
        return self._obs(3, np.float64)

    def _get_defender_state(self):
        return self._obs(1, np.float64)

    def _get_attacker_state(self):
        return self._obs(2, np.float32)

    def os_to_float(self, os_obj):
        return float(getattr(os_obj, "_value", 0.0))

    # ---- actions ----
    def _mode_id(self):
        if self.mode not in ("defender", "attacker"):
            raise ValueError("Invalid mode")
        return 1 if self.mode == "attacker" else 0

    def sample_action(self):
        """(action_type, exploit_indices, device_indices, app_index) with device_indices in random.sample's draw order
        (CyberDefenseEnv.py:555-578)."""
        ab = self._venv.sample_actions(self._mode_id(), want_order=True)
        f = decode_header(ab.hdr.cpu())
        devs = [int(x) for x in ab.order[0, :int(f.n_dev[0])].cpu().numpy().view(np.uint16)]
        self._host = None  # the draw epoch moved
        return (int(f.atype[0]), np.array([int(f.ex[0, 0])], dtype=int), devs, int(f.app[0]))

    def randomize_compromise_and_ownership(self):
        self._venv.randomize_compromise_and_ownership()
        self._host = None

    def _rebuild_graph_cache(self):
        """The kernels read the network tables directly; what a rebuild changes for the step path is that the new
        cache forgets every blocked edge (volt_typhoon_env.py:476)."""
        if self._venv is not None:
            self._venv.rebuild_graph_cache()
            self._host = None

    def _pack(self, action, mode):
        if action is not None:
            atype, ex, devs, app = action
            devs = [int(d) for d in devs]
            if int(atype) in (11, 12, 13) and mode == 0 and len(devs) == 0 and self._base_line == "Nash":
                raise ValueError("device_indices[0] is required")  # volt:965-966, :1103-1104, :1112-1113
            order_form = devs != sorted(set(devs))
            action = (atype, ex, devs, app)
        else:
            order_form = False
        return ActionBatch.pack([action], mode, self._net.M, order_form=order_form)

    def _finish(self, raw, shaped, done, action, grouped, executed):
        v = self._venv
        # one device->host copy: rewards, done and the pre-evolve masks; the counters come from the cached state copy
        out = torch.cat([raw.view(torch.int32).reshape(-1), shaped.view(torch.int32).reshape(-1), done.view(torch.int32).reshape(-1),
                         v.pre_masks().reshape(-1)]).cpu().numpy()
        self._host = None
        if int(self._snap()["scal"][K.S_FLAGS]) & K.FL_DET_PENDING:  # defender action 10 trained the detector (volt:945-962)
            seed = self.detector_fit_seed
            self._venv.service_detectors(None if seed is None else (lambda b: seed))
            self._host = None
        M, W = self._net.M, self._net.W
        pre = out[3:].view(np.uint32).reshape(3, W)
        bits = lambda row: ((pre[row, np.arange(M) >> 5] >> (np.arange(M) & 31)) & 1).astype(np.float64)
        st = np.zeros((M, 6), np.float64)  # the pre-evolve `state` step() returns (volt:1306)
        st[:, 0], st[:, 1] = self._net.os_val, self._net.ver_val
        st[:, 2], st[:, 4], st[:, 5] = bits(0), bits(1), bits(2)
        self.state = st.reshape(-1)
        s = self._snap()["scal"]
        c = [(key, _counter(s, slot, is_float)) for _, key, slot, is_float in K.COUNTERS]
        # the reference's info dict: its first six counters, action_taken, four more; no defender_step / attacker_step
        info = dict([("mode", self.mode)] + c[:6] + [("action_taken", action)] + c[6:10])
        # step() builds info BEFORE step_num increments (volt:1272-1285), step_grouped() after (volt:746-755)
        if executed and not grouped:
            info["step_count"] -= 1
        return (self.state, float(out[0:1].view(np.float32)[0]), float(out[1:2].view(np.float32)[0]), bool(out[2]), info,
                self._sim.logger.get_logs())

    def step(self, action, agent_cnt=None):
        if isinstance(action, (list, tuple)) and action and isinstance(action[0], (list, tuple)):
            return self.step_grouped(action)
        mode = self._mode_id()
        hdr, mask, order = self._pack(action, mode)
        flags = 0
        if agent_cnt is not None and agent_cnt != self._net.M:
            flags |= K.STEP_SKIP_WORK  # volt:1207, :1307
        raw, shaped, done = self._venv.step(self._venv.to_device(hdr, mask, order), flags=flags, want_pre=True)
        return self._finish(raw, shaped, done, action, grouped=False, executed=not flags)

    def step_grouped(self, groups):
        mode = self._mode_id()
        batches = []
        any_order = any(list(map(int, g[2])) != sorted(set(map(int, g[2]))) for g in groups)
        for g in groups:
            h, m, o = ActionBatch.pack([(g[0], g[1], [int(d) for d in g[2]], g[3])], mode, self._net.M, order_form=any_order)
            batches.append(self._venv.to_device(h, m, o))
        raw, shaped, done = self._venv.step_grouped(batches, want_pre=True)
        return self._finish(raw, shaped, done, list(groups), grouped=True, executed=True)


CyberDefenseEnv = Volt_Typhoon_CyberDefenseEnv
