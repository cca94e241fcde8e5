"""The drop-in Gym surface (Volt_Typhoon_CyberDefenseEnv.reset()/step()) against golden trajectories of the
reference: same action tuples in, same rewards / done / observations / counters out."""
import numpy as np
import pytest

from tests.common import GOLDEN, load_golden, replay_golden_on_gym

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", ["c1_m20_plain", "c1_m20_order", "c1_m20_baselines", "c2_m50_plain",
                                  "c2_m50_detector", "c1_m30_detector_busy_log"])
def test_gym_surface_replays_golden(name):
    from cygym_b200 import network_from_golden
    from cygym_b200.volt_typhoon_env import Volt_Typhoon_CyberDefenseEnv
    g = load_golden([p for p in GOLDEN if name in p][0])
    net, meta = network_from_golden(g)
    env = Volt_Typhoon_CyberDefenseEnv(net, seed=meta["draw_seed"], env_id=meta["env_id"], xcap=meta["xcap"])
    assert env.get_num_action_types("defender") == 14 and env.get_num_action_types("attacker") == 3
    assert env.Max_network_size == meta["M"] and env.MaxExploits == 6
    replay_golden_on_gym(env, g)


def test_gym_surface_errors_and_counters():
    from cygym_b200.volt_typhoon_env import Volt_Typhoon_CyberDefenseEnv
    env = Volt_Typhoon_CyberDefenseEnv()
    env.numOfDevice, env.Max_network_size = 10, 20
    s0 = env.initialize_environment()
    assert s0.shape == (120,)
    env.mode = "defender"
    for at in (11, 12, 13):
        with pytest.raises(ValueError):
            env.step((at, [0], [], 0))
    with pytest.raises(ValueError):
        env.get_num_action_types("nobody")
    env.mode = "attacker"
    a = env.sample_action()
    assert 0 <= a[0] < 5 and len(a[2]) >= 1 and len(a[1]) == 1
    env.step(a)
    assert env.step_num == 1 and env.attacker_step == 1
    env.step_num = 0          # callers zero counters between rollouts (do_agent.py:192-196)
    env.defensive_cost = 0
    assert env.step_num == 0 and env.defensive_cost == 0.0
    s1 = env.reset(from_init=True)
    assert np.array_equal(s0, s1)


def test_gym_surface_pickle_rebuild_and_views():
    """Pickled copies step like the original (workers: do_agent.py:642-705); _rebuild_graph_cache() from outside a step
    forgets the blocked edges (volt:476); the simulator views read the live state."""
    import pickle
    from cygym_b200.volt_typhoon_env import Volt_Typhoon_CyberDefenseEnv
    env = Volt_Typhoon_CyberDefenseEnv(seed=5)
    env.step_num = 3          # set before the env exists: replayed into the scalars by initialize_environment()
    env.numOfDevice, env.Max_network_size = 30, 40
    env.initialize_environment()
    assert env.step_num == 3
    env.mode = "defender"
    env.step((6, [0], list(range(0, 40, 2)), 0))  # block one edge per listed active device
    assert env.edges_blocked > 0
    blocked = int(np.unpackbits(env._snap()["blocked"].view(np.uint8)).sum())
    assert blocked == env.edges_blocked
    clone = pickle.loads(pickle.dumps(env))
    for e in (env, clone):
        e.mode = "attacker"
    ra, rb = env.step((1, [0], [], 0)), clone.step((1, [0], [], 0))
    assert ra[1] == rb[1] and np.array_equal(ra[0], rb[0]) and ra[4] == rb[4]
    assert [d.isCompromised for d in env.simulator.subnet.net.values()] == [d.isCompromised for d in clone.simulator.subnet.net.values()]
    env._rebuild_graph_cache()
    assert int(np.unpackbits(env._snap()["blocked"].view(np.uint8)).sum()) == 0 and env.edges_blocked > 0
    assert len(env.simulator.subnet.graph.get_edgelist()) == env.simulator.subnet.graph.ecount()
    a = env.sample_action()
    assert len(a[2]) == len(set(a[2])) and a[2] != sorted(a[2]) or len(a[2]) < 3  # draw order, not ascending
