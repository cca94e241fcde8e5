"""The drop-in Gym class driven by the reference's own, UNMODIFIED caller: DoubleOracle (do_agent.py:498) is
constructed on it, checkpoints / restores it and rolls games out on it with _simulate_game_serial
(do_agent.py:1957-2089); the 10-tuple must equal what the same code returns on the reference env under replayed draws.

Build container only: /root/reference does not exist on the GPU box, and this container has no GPU -- so the drop-in
runs on the host compile of the device source (tests/emu/emu_venv.py) here; the CUDA-backed class replays the recorded
reference trajectories on the GPU box (tests/test_gpu_dropin.py)."""
import warnings

import numpy as np
import pytest

from oracle import ref_harness as H

needs_reference = pytest.mark.skipif(not H.available(), reason="reference checkout not present")


class ReplayedRef:
    """The reference env with every draw-consuming call inside one replay window (== one draw epoch), as the kernels
    count them.  Everything else is the reference object itself."""

    def __init__(self, env):
        object.__setattr__(self, "_env", env)

    def __getattr__(self, name):
        return getattr(self._env, name)

    def __setattr__(self, name, value):
        setattr(self._env, name, value)

    def step(self, action, agent_cnt=None):
        with H.context().window():
            return self._env.step(action) if agent_cnt is None else self._env.step(action, agent_cnt)

    def sample_action(self):
        with H.context().window():
            return self._env.sample_action()

    def randomize_compromise_and_ownership(self):
        with H.context().window():
            return self._env.randomize_compromise_and_ownership()


def _pair(numOfDevice, M, seed, draw_seed=77, env_id=5):
    from cygym_b200 import snapshot
    from cygym_b200.volt_typhoon_env import Volt_Typhoon_CyberDefenseEnv
    from tests.emu.emu_venv import EmuVectorEnv
    ref = H.build_env(numOfDevice=numOfDevice, Max_network_size=M, seed=seed)
    ctx = H.context()
    ctx.seed, ctx.env_id, ctx.epoch = draw_seed, env_id, 0
    net = snapshot.from_reference_env(ref)
    ours = Volt_Typhoon_CyberDefenseEnv(net, seed=draw_seed, env_id=env_id, xcap=64, venv_cls=EmuVectorEnv)
    return ReplayedRef(ref), ours


@needs_reference
@pytest.mark.parametrize("numOfDevice,M,seed", [(10, 20, 21), (40, 50, 22)])
def test_unmodified_double_oracle_runs_on_the_dropin(numOfDevice, M, seed):
    warnings.filterwarnings("ignore")
    import importlib
    import torch
    H.load_reference()
    do_agent = importlib.import_module("do_agent")
    Strategy = importlib.import_module("strategy").Strategy
    ref, ours = _pair(numOfDevice, M, seed)
    steps = 24
    dos = []
    for env in (ref, ours):
        torch.manual_seed(0)
        H.context().epoch = 0 if env is ref else H.context().epoch
        dos.append(do_agent.DoubleOracle(env, num_episodes=1, steps_per_episode=steps, seed=0, baseline="Nash",
                                         dynamic_neighbor_search=False, BR_type="ddpg", zero_day=False))
    do_ref, do_ours = dos
    # the constructor sampled 2 x steps actions on either env (defense_strategy / init_attack_strategy, do_agent.py:1001-1013)
    for a, b in zip(do_ref.defender_strategies[0].actions + do_ref.attacker_strategies[0].actions,
                    do_ours.defender_strategies[0].actions + do_ours.attacker_strategies[0].actions):
        assert int(a[0]) == int(b[0]) and list(map(int, a[1])) == list(map(int, b[1])) and list(map(int, a[2])) == list(map(int, b[2])) \
            and int(a[3]) == int(b[3])
    assert do_ref.D_init == do_ours.D_init and do_ref.E_init == do_ours.E_init and do_ref.A_init == do_ours.A_init
    assert do_ref.env._get_defender_state().shape == do_ours.env._get_defender_state().shape

    def typed(acts):  # the sampled lists with real action types (sklearn's branch, defender 10, stays out)
        return [a for a in acts]

    # a fixed sequence with every action type the policies sample (real sample_action() draws, in draw order)
    seqs = []
    for env in (ref, ours):
        ep0 = H.context().epoch if env is ref else None
        d_acts, a_acts = [], []
        for t in range(steps):
            env.mode = "defender"
            a = env.sample_action()
            d_acts.append((8 if int(a[0]) == 10 else int(a[0]), a[1], a[2], a[3]))
            env.mode = "attacker"
            a_acts.append(env.sample_action())
        seqs.append((d_acts, a_acts))
    pairs = [
        (lambda D: D.defender_strategies[0], lambda D: D.attacker_strategies[0]),          # the constructor's fixed sequences
        (lambda D: Strategy(baseline_name="No Defense"), lambda D: Strategy(baseline_name="No Attack")),
        (lambda D: Strategy(baseline_name="Preset"), lambda D: D.attacker_strategies[0]),
        (None, None),                                                                       # the sampled typed sequences
    ]
    for do_, seq in ((do_ref, seqs[0]), (do_ours, seqs[1])):
        do_.checkpoint_now()
    for i, (fd, fa) in enumerate(pairs):
        outs = []
        for do_, seq in ((do_ref, seqs[0]), (do_ours, seqs[1])):
            sd = Strategy(actions=seq[0]) if fd is None else fd(do_)
            sa = Strategy(actions=seq[1]) if fa is None else fa(do_)
            outs.append(do_._simulate_game_serial(sd, sa, 2, [None], [1.0]))
        r, o = np.asarray(outs[0], np.float64), np.asarray(outs[1], np.float64)
        assert np.allclose(o, r, rtol=1e-5, atol=1e-6), (i, r.tolist(), o.tolist())
    # the views IPPO / HMARL read (IPPO.py:74-96, HMARL.py:126-159) agree with the reference objects after all that
    for d_ref, d_our in zip(ref._get_ordered_devices(), ours._get_ordered_devices()):
        for attr in ("isCompromised", "Known_to_attacker", "Not_yet_added", "attacker_owned", "reachable_by_attacker", "wtype"):
            assert getattr(d_ref, attr) == getattr(d_our, attr), (d_ref.id, attr)
        assert (d_ref.device_type == "DomainController") == (d_our.device_type == "DomainController")  # the one type the step path reads
        assert int(d_ref.busy_time) == int(d_our.busy_time) and (d_ref.workload is None) == (d_our.workload is None)
    assert sorted(ref.simulator.subnet.graph.get_edgelist()) == sorted(ours.simulator.subnet.graph.get_edgelist())
    la, lb = ref.simulator.logger.get_logs(), ours.simulator.logger.get_logs()
    assert len(la) == len(lb)
    assert [(l["from_device"], l["to_device"]) for l in la[-2000:]] == [(l["from_device"], l["to_device"]) for l in lb[-2000:]]
    assert [e.discovered for e in ref.simulator.exploits] == [e.discovered for e in ours.simulator.exploits]


def test_dropin_pickles_and_info_counters():
    """Workers get pickled env copies (do_agent.py:642-705); info['step_count'] is pre-increment for step() and
    post-increment for step_grouped() (volt:1272-1285 / :746-755); counters set before the env exists survive."""
    import pickle
    from cygym_b200 import synthetic_network
    from cygym_b200.volt_typhoon_env import Volt_Typhoon_CyberDefenseEnv
    from tests.emu.emu_venv import EmuVectorEnv
    env = Volt_Typhoon_CyberDefenseEnv(venv_cls=EmuVectorEnv, seed=3)
    env.step_num = 7          # constructor-then-configure (init_experiments.py pattern)
    env.numOfDevice, env.Max_network_size = 20, 30
    env.initialize_environment()
    assert env.step_num == 7
    env.mode = "defender"
    _, _, _, _, info, _ = env.step((8, [0], [], 0))
    assert info["step_count"] == 7 and env.step_num == 8
    _, _, _, _, info, _ = env.step([(1, [0], [1, 2], 0), (2, [0], [3], 0)])
    assert info["step_count"] == 9 and env.step_num == 9
    for t in range(6):
        env.mode = "attacker" if t & 1 else "defender"
        a = env.sample_action()
        env.step((8 if env.mode == "defender" and a[0] == 10 else a[0], a[1], a[2], a[3]))
    clone = pickle.loads(pickle.dumps(env))
    assert clone.step_num == env.step_num and np.array_equal(clone._get_state(), env._get_state())
    for e in (env, clone):
        e.mode = "attacker"
    ra, rb = env.step((1, [0], [], 0)), clone.step((1, [0], [], 0))
    assert ra[1] == rb[1] and ra[3] == rb[3] and np.array_equal(ra[0], rb[0]) and ra[4]["Compromised_devices"] == rb[4]["Compromised_devices"]
    with pytest.raises(AttributeError):
        env.simulator.subnet.net[0].isCompromised = True


@pytest.mark.parametrize("name", ["c2_m50_detector", "c1_m30_detector_busy_log"])
def test_dropin_replays_the_references_detector_trajectories(name):
    """The reference's recorded detector trajectories (defender 10 fits the IsolationForest on the hop log, scans consult
    it) fed to the drop-in on the host compile of the device source: the drop-in must fit where the reference did, with
    numpy's stream seeded alike, and reach the same 6-tuples, device state and hop log after every step."""
    from cygym_b200 import network_from_golden
    from cygym_b200.volt_typhoon_env import Volt_Typhoon_CyberDefenseEnv
    from tests.common import GOLDEN, load_golden, replay_golden_on_gym
    from tests.emu.emu_venv import EmuVectorEnv
    warnings.filterwarnings("ignore")
    g = load_golden([p for p in GOLDEN if name in p][0])
    net, meta = network_from_golden(g)
    env = Volt_Typhoon_CyberDefenseEnv(net, seed=meta["draw_seed"], env_id=meta["env_id"], xcap=meta["xcap"], venv_cls=EmuVectorEnv)
    replay_golden_on_gym(env, g)
    assert env.simulator.detector.trained and int((g["train_seed"] >= 0).sum()) >= 10


@needs_reference
def test_dropin_trains_and_consults_the_detector_like_the_reference():
    """Defender action 10 fits the IsolationForest on the hop log (scikit-learn, on the host, from the ring the kernels
    keep) and later scans (action 5) consult it on the device (volt:945-962, :1020-1069): same 6-tuples, same device
    state, same log as the reference, step by step, with numpy's global stream seeded alike before every fit."""
    warnings.filterwarnings("ignore")
    ref, ours = _pair(20, 30, 41)
    rng = np.random.default_rng(5)
    trained = scans_that_cleaned = 0
    for t in range(260):
        mode = "defender" if t % 2 == 0 else "attacker"
        ref.mode = ours.mode = mode
        a, b = ref.sample_action(), ours.sample_action()
        assert int(a[0]) == int(b[0]) and list(map(int, a[2])) == list(map(int, b[2]))
        at = int(rng.choice([5, 5, 5, 10, 8, 6])) if mode == "defender" else int(rng.choice([1, 1, 2]))
        act = (at, a[1], a[2], a[3])
        if at == 10 and len(ref.simulator.logger.get_logs()) > 0:
            H.seed_numpy_global(9000 + t)
            ours.detector_fit_seed = 9000 + t
            trained += 1
        before = sum(d.isCompromised for d in ref._get_ordered_devices())
        ra, rb = ref.step(act), ours.step(act)
        if at == 5 and sum(d.isCompromised for d in ref._get_ordered_devices()) < before:
            scans_that_cleaned += 1
        assert abs(ra[1] - rb[1]) <= 1e-5 * max(1.0, abs(ra[1])) and ra[3] == rb[3], t
        assert np.array_equal(np.asarray(ra[0]), rb[0]), t
        for x, y in zip(ref._get_ordered_devices(), ours._get_ordered_devices()):
            assert x.isCompromised == y.isCompromised and int(x.busy_time) == int(y.busy_time), (t, x.id)
    la, lb = ref.simulator.logger.get_logs(), ours.simulator.logger.get_logs()
    assert [(l["from_device"], l["to_device"]) for l in la[-2000:]] == [(l["from_device"], l["to_device"]) for l in lb[-2000:]]
    assert ours.simulator.detector.trained and trained >= 5 and scans_that_cleaned >= 1, (trained, scans_that_cleaned)
