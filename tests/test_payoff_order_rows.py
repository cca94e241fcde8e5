"""The order rows of the batched payoff evaluator's strategy tables (payoff._strategy_rows), on the host."""
import numpy as np


def test_strategy_rows_carry_draw_order_lists():
    """Sequences drawn by the oracle's sample_action: a defender row whose list is not ascending and duplicate-free
    carries it in its order row, every other row (and every attacker row) starts with ORDER_NONE; unpacking the rows
    gives back the strategies' actions."""
    from cygym_b200 import _capi as K
    from cygym_b200 import synthetic_network
    from cygym_b200.payoff import Strategy, _strategy_rows
    from cygym_b200.vector_env import ActionBatch
    from tests.common import oracle_for, oracle_state_from_template
    net = synthetic_network(50, n_subnets=3, seed=21)
    M, L, T = net.M, 10, 7
    seqs = {}
    for mode in (0, 1):
        orc, _ = oracle_for(net, seed=3 + mode, xcap=32)
        st = oracle_state_from_template(orc, net, L)
        orc.randomize(st)
        seqs[mode] = ActionBatch.unpack(*orc.sample_actions(st, mode, want_order=True))
    is_set = lambda a: a is None or list(a[2]) == sorted(set(a[2]))
    assert sum(not is_set(a) for a in seqs[0]) >= 3 and sum(not is_set(a) for a in seqs[1]) >= 1
    defs = [Strategy(actions=seqs[0]), Strategy(baseline_name="Nash")]
    atts = [Strategy(baseline_name="No Attack"), Strategy(actions=seqs[1])]
    (hd, md, rd, bd, od), (ha, ma, ra, ba, oa) = _strategy_rows(defs, atts, T, M)
    assert od.shape == (L + 1, M) and od.dtype == np.uint16 and oa.shape == (1 + L, M)
    assert rd.shape == (T, 2) and list(rd[:, 0]) == [t % L for t in range(T)] and list(bd) == [255, K.BASE_LINES["Nash"]]
    for k, a in enumerate(seqs[0]):
        if is_set(a):
            assert od[k, 0] == K.ORDER_NONE
        else:
            assert list(od[k, :len(a[2])]) == [int(d) for d in a[2]]
    assert od[L, 0] == K.ORDER_NONE and (oa[:, 0] == K.ORDER_NONE).all()
    # unpacking: the defender rows in order form where ordered, as the set otherwise
    back = [ActionBatch.unpack(hd[k:k + 1].view(np.uint32), md[k:k + 1].view(np.uint32),
                               None if od[k, 0] == K.ORDER_NONE else od[k:k + 1])[0] for k in range(L)]
    for a, b in zip(seqs[0], back):
        if a is None:
            assert b is None
        else:
            assert (int(b[0]), [int(x) for x in b[1]], int(b[3])) == (int(a[0]), [int(x) for x in a[1]], int(a[3]))
            assert [int(d) for d in b[2]] == ([int(d) for d in a[2]] if not is_set(a) else sorted(int(d) for d in a[2]))
    # attacker rows hold the SET of their list in the mask
    for k, a in enumerate(seqs[1]):
        b = ActionBatch.unpack(ha[1 + k:2 + k].view(np.uint32), ma[1 + k:2 + k].view(np.uint32))[0]
        assert (a is None) == (b is None)
        if a is not None:
            assert [int(d) for d in b[2]] == sorted(set(int(d) for d in a[2]))
