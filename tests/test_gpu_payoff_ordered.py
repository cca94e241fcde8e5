"""Payoff evaluation of strategies whose defender device lists are in draw order (the sequences DoubleOracle samples with
sample_action, do_agent.py:1001-1013): the order-form rollout kernel (cyg_rollout_ordered) against single steps with
order arrays, and both evaluators against the oracle and each other."""
import numpy as np
import pytest

from tests.common import oracle_for, oracle_state_from_template

pytestmark = pytest.mark.gpu


def _sampled_sequences(net, mode, n_seq, length, seed, map10=True):
    """n_seq fixed sequences of `length` actions drawn by the oracle's sample_action (device lists in draw order)."""
    from cygym_b200.vector_env import ActionBatch
    out = []
    for k in range(n_seq):
        orc, _ = oracle_for(net, seed=seed + k, xcap=32, env_id0=1000 * k)
        st = oracle_state_from_template(orc, net, length)
        orc.randomize(st)
        h, m, o = orc.sample_actions(st, mode, want_order=True)
        acts = ActionBatch.unpack(h, m, o)
        if map10:
            acts = [a if a is None or a[0] != 10 else (8,) + tuple(a[1:]) for a in acts]
        out.append(acts)
    return out


def _unsorted(a):
    return a is not None and [int(d) for d in a[2]] != sorted(set(int(d) for d in a[2]))


def _oracle_payoff(net, defs, atts, N, T, seed, xcap):
    """The pair-by-pair loop on the oracle, packing a list that is not ascending and duplicate-free in order form."""
    from cygym_b200.vector_env import ActionBatch
    out = np.zeros((len(defs), len(atts), 10))
    for i, ds in enumerate(defs):
        for j, as_ in enumerate(atts):
            orc, _ = oracle_for(net, seed=seed, xcap=xcap, env_id0=(i * len(atts) + j) * N)
            st = oracle_state_from_template(orc, net, N)
            orc.randomize(st)
            for slot in (0, 4, 5, 8, 13, 9, 10, 12, 11):
                st.scal[:, slot] = 0
            bl = "Nash"
            dr, ar = np.zeros(N), np.zeros(N)
            for t in range(T):
                mode = t & 1
                action, nb = (ds if mode == 0 else as_).decide(t)
                if nb is not None and nb != bl:
                    bl = nb
                    orc.set_base_line(bl)
                h, m, o = ActionBatch.pack([action], mode, net.M, order_form=_unsorted(action))
                r = orc.step(st, np.repeat(h, N, 0), np.repeat(m, N, 0), None if o is None else np.repeat(o, N, 0), n_threads=8)
                (dr if mode == 0 else ar).__iadd__(r["raw"])
            sc = st.scal
            cols = [dr, ar, sc[:, 7], sc[:, 8], sc[:, 11], sc[:, 9].copy().view(np.float32), sc[:, 13], sc[:, 12], sc[:, 14], sc[:, 15]]
            out[i, j] = [np.asarray(c, np.float64).sum() / N for c in cols]
            out[i, j, 2] /= max(1.0, T)
    return out


def _tables(M, R, T, rng):
    """Rollout tables [T, R] mixing ordered defender rows of types 1/4/5/6/9/12/13, set-form defender rows, baseline
    rows and attacker rows: hdr, mask, order (int16, -1 = ORDER_NONE), base_line."""
    from cygym_b200.vector_env import ActionBatch
    hdr = np.zeros((T, R, 4), np.uint32)
    mask = np.zeros((T, R, (M + 31) // 32), np.uint32)
    order = np.full((T, R, M), -1, np.int16)
    bl = np.zeros((T, R), np.uint8)
    types = (1, 4, 5, 6, 9, 12, 13)
    for t in range(T):
        mode = t & 1
        for r in range(R):
            kind = (r + t) % 4
            k = int(rng.integers(2, min(M, 24)))
            devs = [int(d) for d in rng.permutation(M)[:k]]
            if mode == 0:
                if kind <= 1:
                    act, ordered = (types[(r + t // 2) % len(types)], [0], devs, int(rng.integers(0, 3))), True
                elif kind == 2:
                    act, ordered = (int(rng.choice([1, 3, 4, 6, 7, 9, 11, 12])), [0], sorted(devs), 0), False
                else:
                    act, ordered = None, False
                    bl[t, r] = rng.choice([0, 1, 2])
            else:
                act = None if kind == 3 else (int(rng.integers(0, 3)), [int(rng.integers(0, 4))], devs, 0)
                ordered = False
                if act is None:
                    bl[t, r] = rng.choice([0, 3])
            h, m, o = ActionBatch.pack([act], mode, M, order_form=True)
            hdr[t, r], mask[t, r] = h[0], m[0]
            if ordered:
                order[t, r] = o[0].view(np.int16)
    return hdr, mask, order, bl


@pytest.mark.parametrize("M", [20, 50, 100, 128])
@pytest.mark.parametrize("log_cap", [0, 16])
def test_rollout_ordered_equals_single_steps(M, log_cap):
    """cyg_rollout_ordered against T cyg_step calls with per-env order arrays (the set rows carry their ascending list)
    and per-env base_line: returns, the canonical state and the hop-log rings bit-identical."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import ActionBatch, VectorCyberDefenseEnv
    net = synthetic_network(M, n_subnets=3, seed=M)
    R, epr, T = 12, 8, 10
    B = R * epr
    hdr, mask, order, bl = _tables(M, R, T, np.random.default_rng(M + log_cap))
    assert (order[0::2, :, 0] != -1).any()
    envs = [VectorCyberDefenseEnv(net, B, seed=7, env_id0=300, xcap=32, log_cap=log_cap) for _ in range(2)]
    for e in envs:
        e.randomize_compromise_and_ownership()
    a, b = envs
    dev = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x).view(dt)).cuda()
    ret_a = a.rollout(dev(hdr, np.int32), dev(mask, np.int32), dev(bl, np.uint8), epr, 0, order=dev(order, np.int16))
    row = np.arange(B) // epr
    ret_b = torch.zeros(2, B, dtype=torch.float64, device="cuda")
    for t in range(T):
        h, m, o = hdr[t][row], mask[t][row], order[t][row].copy()
        for e_ in range(B):  # set rows: the ascending list of the mask
            if o[e_, 0] == -1:
                bits = np.unpackbits(m[e_].view(np.uint8), bitorder="little")[:M]
                lst = np.nonzero(bits)[0]
                o[e_] = 0
                o[e_, :len(lst)] = lst
        b.set_base_line_per_env(dev(bl[t][row], np.uint8))
        raw, _, _ = b.step(ActionBatch(dev(h, np.int32), dev(m, np.int32), dev(o, np.int16)))
        ret_b[t & 1] += raw.double()
    torch.cuda.synchronize()
    assert torch.equal(ret_a, ret_b)
    sa, sb = a.export_state(), b.export_state()
    assert set(sa) == set(sb) and ("logs" in sa) == (log_cap > 0)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    if log_cap:
        assert int(sa["scal"][:, 6].max()) > 0  # the rings saw hops


def _ordered_setup(net, seed=11):
    from cygym_b200.payoff import Strategy
    dseq = _sampled_sequences(net, 0, 3, 8, seed)
    aseq = _sampled_sequences(net, 1, 2, 6, seed + 50)
    assert sum(_unsorted(x) for s in dseq for x in s) >= 6
    defs = [Strategy(actions=s) for s in dseq] + [Strategy(baseline_name="No Defense"), Strategy(baseline_name="Nash")]
    atts = [Strategy(actions=s) for s in aseq] + [Strategy(baseline_name="No Attack")]
    return defs, atts, dseq, aseq


def test_ordered_sequences_in_both_evaluators():
    """DoubleOracle-style sampled sequences: the pair-by-pair evaluator matches the oracle with order-form packing, the
    batched evaluator equals it for any sharding and launch cut, and a sorted copy of the sequences gives another matrix."""
    from cygym_b200 import synthetic_network
    from cygym_b200.payoff import Strategy, evaluate_payoff_matrix, evaluate_payoff_matrix_batched, reduce_payoff
    net = synthetic_network(50, n_subnets=3, seed=21)
    defs, atts, dseq, aseq = _ordered_setup(net)
    N, T, seed, xcap = 32, 24, 5, 32
    per_pair = evaluate_payoff_matrix(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    exp = _oracle_payoff(net, defs, atts, N, T, seed, xcap)
    assert np.allclose(per_pair, exp, rtol=1e-5, atol=1e-6), np.abs(per_pair - exp).max()
    one = evaluate_payoff_matrix_batched(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    assert np.allclose(one, per_pair, rtol=1e-12, atol=1e-9), np.abs(one - per_pair).max()
    for world in (2, 3):  # 2: strided env ids, 3: contiguous slices
        parts = [evaluate_payoff_matrix_batched(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap, rank=r, world=world,
                                                reduce=False) for r in range(world)]
        both = reduce_payoff(sum(parts[1:], parts[0]), N, T).cpu().numpy()
        assert np.allclose(both, per_pair, rtol=1e-12, atol=1e-9), world
    for spl in (7, 1):
        alt = evaluate_payoff_matrix_batched(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap, steps_per_launch=spl).cpu().numpy()
        assert np.allclose(alt, per_pair, rtol=1e-12, atol=1e-9), spl
    # the order is honoured, not sorted away: the unsorted actions retyped to 13 / 6 / 1 / 4 with the largest listed id
    # first (13 acts on device_indices[0]; 6, 1 and 4 take their draws per listed device in list order)
    def force(s):
        out = []
        for k, a in enumerate(s):
            if _unsorted(a):
                d = [int(x) for x in a[2]]
                top = max(d)
                d.remove(top)
                a = ((13, 6, 1, 4)[k % 4], a[1], [top] + d, a[3])
            out.append(a)
        return out
    srt = lambda s: [a if a is None else (a[0], a[1], sorted(set(a[2])), a[3]) for a in s]
    forced = [Strategy(actions=force(s)) for s in dseq]
    as_drawn = evaluate_payoff_matrix_batched(net, forced, atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    ref = evaluate_payoff_matrix(net, forced, atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    assert np.allclose(as_drawn, ref, rtol=1e-12, atol=1e-9), np.abs(as_drawn - ref).max()
    other = evaluate_payoff_matrix_batched(net, [Strategy(actions=srt(force(s))) for s in dseq], atts, N, steps_per_episode=T,
                                           seed=seed, xcap=xcap).cpu().numpy()
    assert not np.allclose(other, as_drawn, rtol=1e-9, atol=1e-9)


def test_ordered_sequences_that_train_the_detector():
    """train_detectors=True with sampled type-10 actions kept: the batched evaluator equals the pair-by-pair one."""
    from cygym_b200 import synthetic_network
    from cygym_b200.payoff import Strategy, evaluate_payoff_matrix, evaluate_payoff_matrix_batched
    net = synthetic_network(50, n_subnets=3, seed=21)
    dseq = _sampled_sequences(net, 0, 3, 8, 11, map10=False)
    dseq[0][1] = (10, [0], dseq[0][1][2] if dseq[0][1] is not None else [3, 1], 0)  # at least one sequence trains
    dseq[0][3] = (5, [0], [4, 9, 2, 30], 0)
    aseq = _sampled_sequences(net, 1, 2, 6, 61)
    defs = [Strategy(actions=s) for s in dseq] + [Strategy(baseline_name="Nash")]
    atts = [Strategy(actions=s) for s in aseq] + [Strategy(baseline_name="No Attack")]
    assert defs[0].can_train()
    N, T, seed, xcap = 16, 20, 5, 32
    ref = evaluate_payoff_matrix(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap, train_detectors=True).cpu().numpy()
    for spl in (None, 7):
        got = evaluate_payoff_matrix_batched(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap, steps_per_launch=spl,
                                             train_detectors=True).cpu().numpy()
        assert np.allclose(got, ref, rtol=1e-12, atol=1e-9), (spl, np.abs(got - ref).max())


def test_attacker_lists_travel_as_sets():
    """attacker_act reads exploits and sources, never device_indices: an attacker sequence with draw-order lists gives the
    same matrix through the pair-by-pair evaluator (order form) and the batched one (set form)."""
    from cygym_b200 import synthetic_network
    from cygym_b200.payoff import Strategy, evaluate_payoff_matrix, evaluate_payoff_matrix_batched
    net = synthetic_network(50, n_subnets=3, seed=21)
    aseq = _sampled_sequences(net, 1, 3, 6, 77)
    assert any(_unsorted(a) for s in aseq for a in s)
    defs = [Strategy(baseline_name="Nash"), Strategy(actions=[(1, [0], [0, 3, 7, 20], 0), (6, [0], [1, 2, 3], 0)])]
    atts = [Strategy(actions=s) for s in aseq]
    N, T, seed, xcap = 32, 16, 3, 32
    a = evaluate_payoff_matrix(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    b = evaluate_payoff_matrix_batched(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    assert np.allclose(a, b, rtol=1e-12, atol=1e-9), np.abs(a - b).max()


def test_closed_loop_with_ordered_sequences():
    """The closed-loop path: an actor strategy next to ordered sequences (the ordered turns pass an order array to every
    env, the actor's envs the ascending list of their decoded mask), and a network beyond 128 device slots.  The pairs of
    sequences and baselines equal the pair-by-pair evaluator."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.payoff import Strategy, evaluate_payoff_matrix, evaluate_payoff_matrix_batched
    net = synthetic_network(50, n_subnets=3, seed=21)
    M, X, A = net.M, net.X, int(net.cfg.get("n_app_ids", 0))
    torch.manual_seed(3)
    actor = torch.nn.Sequential(torch.nn.Linear(6 * M, 64), torch.nn.ReLU(), torch.nn.Linear(64, 14 + M + X + A), torch.nn.Tanh())
    actor = actor.double().cuda().eval()
    defs, atts, _, _ = _ordered_setup(net)
    N, T, seed, xcap = 16, 16, 5, 32
    wrapped = lambda x: actor(x.double())
    got = evaluate_payoff_matrix_batched(net, defs + [Strategy(actor=wrapped)], atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    ref = evaluate_payoff_matrix(net, defs, atts, N, steps_per_episode=T, seed=seed, xcap=xcap).cpu().numpy()
    assert np.allclose(got[:len(defs)], ref, rtol=1e-12, atol=1e-9), np.abs(got[:len(defs)] - ref).max()
    assert np.isfinite(got[len(defs)]).all()
    big = synthetic_network(150, n_subnets=4, seed=5)
    assert big.W > 4
    defs_b, atts_b, _, _ = _ordered_setup(big, seed=31)
    got_b = evaluate_payoff_matrix_batched(big, defs_b, atts_b, 8, steps_per_episode=12, seed=seed, xcap=xcap).cpu().numpy()
    ref_b = evaluate_payoff_matrix(big, defs_b, atts_b, 8, steps_per_episode=12, seed=seed, xcap=xcap).cpu().numpy()
    assert np.allclose(got_b, ref_b, rtol=1e-12, atol=1e-9), np.abs(got_b - ref_b).max()


def test_rollout_ordered_refuses_bad_arguments():
    """CYG_E_INVAL for a NULL order table, order_stride < M and CYG_STEP_GROUPED, before anything is launched."""
    import ctypes as C
    import torch
    from cygym_b200 import _capi as K
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    net = synthetic_network(50, n_subnets=3, seed=21)
    env = VectorCyberDefenseEnv(net, 64, seed=1)
    T, R, M = 2, 4, net.M
    hdr = torch.zeros(T, R, 4, dtype=torch.int32, device="cuda")
    mask = torch.zeros(T, R, net.W, dtype=torch.int32, device="cuda")
    order = torch.full((T, R, M), -1, dtype=torch.int16, device="cuda")
    ret = torch.zeros(2, 64, dtype=torch.float64, device="cuda")
    a = K.CygRolloutArgs(hdr.data_ptr(), mask.data_ptr(), None, T, R, 0, 16, 0, ret.data_ptr(), None)
    n0 = env.launch_count
    for ptr, stride, flags in ((None, M, 0), (order.data_ptr(), M - 1, 0), (order.data_ptr(), M, K.STEP_GROUPED)):
        assert env.L.cyg_rollout_ordered(env.h, C.byref(a), ptr, stride, flags, None) == K.E_INVAL
    assert env.launch_count == n0
    assert env.L.cyg_rollout_ordered(env.h, C.byref(a), order.data_ptr(), M, 0, None) == 0
    torch.cuda.synchronize()
    assert env.launch_count == n0 + 1
