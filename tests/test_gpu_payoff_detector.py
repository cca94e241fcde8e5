"""Payoff evaluation of defender strategies that train the detector (action 10, then trained scans with action 5):
evaluate_payoff_matrix_batched / evaluate_payoff_matrix with train_detectors=True against the oracle with scikit-learn
fits between the turns, invariance over launch cuts and sharding, the rollout kernel with a hop-log ring against single
steps, and the grid-wide slot assignment of cyg_fit_detectors."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
pytest.importorskip("sklearn")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.common import oracle_state_from_template  # noqa: E402

SEED, XCAP = 5, 32
N, T = 32, 60


def _net():
    from cygym_b200 import synthetic_network
    return synthetic_network(50, n_subnets=3, seed=21)


def _strategies(train=True):
    """Defender: trains every third defender turn (turns 0, 6, 12, ...) and scans a device list in between, Nash, No
    Defense.  Attacker: an exploit-heavy sequence (the hop logs fill), Nash.  train=False: type 10 -> the no-op 8."""
    from cygym_b200.payoff import Strategy
    scan = list(range(0, 50, 2))
    defs = [Strategy(actions=[(10 if train else 8, [0], [], 0), (5, [0], scan, 0), (5, [0], scan[:12], 0)]),
            Strategy(baseline_name="Nash"), Strategy(baseline_name="No Defense")]
    atts = [Strategy(actions=[(1, [0], [], 0), (1, [1], [], 0), (2, [0], [], 0)]), Strategy(baseline_name="Nash")]
    return defs, atts


def _oracle_for(net, env_id0):
    from oracle import cyg_oracle as O
    from cygym_b200.payoff import DETECTOR_LOG_CAP
    cfg = O.make_config(net.cfg, net.E, seed=SEED, xcap=XCAP, log_cap=DETECTOR_LOG_CAP)
    d = dict(row_ptr=net.row_ptr, col=net.col, mult=net.mult, dev_static=net.dev_static, os_val=net.os_val, ver_val=net.ver_val)
    return O.Oracle(d, cfg, env_id0=env_id0)


def _decode(raw_a, nt, M, X, A):
    """decode_action (do_agent.py:972-998, epsilon-free) of actor outputs, env by env."""
    acts = []
    for v in raw_a:
        acts.append((int(np.argmax(v[:nt])), [int(np.argmax(v[nt + M:nt + M + X]))], [int(d) for d in np.where(v[nt:nt + M] > 0)[0]],
                     int(np.argmax(v[nt + M + X:nt + M + X + A])) if A > 0 else 0))
    return acts


def _oracle_payoff(net, defs, atts, n, steps, fit=True):
    """The payoff loop of tests/test_gpu_payoff.py on the oracle, with hop-log rings and detector slots: after every
    defender turn the pending envs are fitted by scikit-learn, seeded with detector_fit_seeds().  Actors run on the GPU
    in float64 on the oracle's observations.  Returns ([n_def, n_att, 10] averages, number of fits)."""
    import torch
    from cygym_b200.payoff import detector_fit_seeds
    from cygym_b200.vector_env import ActionBatch
    M, X, A = net.M, net.X, int(net.cfg.get("n_app_ids", 0))
    out = np.zeros((len(defs), len(atts), 10))
    n_fits = 0
    for i, ds in enumerate(defs):
        for j, as_ in enumerate(atts):
            g0 = (i * len(atts) + j) * n
            orc = _oracle_for(net, g0)
            st = oracle_state_from_template(orc, net, n)
            orc.randomize(st)
            for slot in (0, 4, 5, 8, 13, 9, 10, 12, 11):
                st.scal[:, slot] = 0
            bl = "Nash"
            dr, ar = np.zeros(n), np.zeros(n)
            for t in range(steps):
                mode = t & 1
                strat = ds if mode == 0 else as_
                if strat.actor is not None:
                    obs = torch.from_numpy(orc.observe(st, 1 + mode)).cuda()
                    with torch.no_grad():
                        raw_a = strat.actor(obs).cpu().numpy()
                    h, m, _ = ActionBatch.pack(_decode(raw_a, 14 if mode == 0 else 3, M, X, A), mode, M)
                else:
                    action, nb = strat.decide(t)
                    if nb is not None and nb != bl:
                        bl = nb
                        orc.set_base_line(bl)
                    h1, m1, _ = ActionBatch.pack([action], mode, M)
                    h, m = np.repeat(h1, n, 0), np.repeat(m1, n, 0)
                r = orc.step(st, h, m, n_threads=8)
                if mode == 0:
                    dr += r["raw"]
                    if fit:
                        seeds = detector_fit_seeds(SEED, torch.arange(g0, g0 + n), t).numpy()
                        n_fits += orc.service_detectors(st, lambda b: int(seeds[b]))
                else:
                    ar += r["raw"]
            assert not (st.scal[:, 2] & 0xF0).any(), "the oracle run raised an error bit"
            sc = st.scal
            cols = [dr, ar, sc[:, 7], sc[:, 8], sc[:, 11], sc[:, 9].copy().view(np.float32), sc[:, 13], sc[:, 12], sc[:, 14], sc[:, 15]]
            out[i, j] = [np.asarray(c, np.float64).sum() / n for c in cols]
            out[i, j, 2] /= max(1.0, steps)
    return out, n_fits


@pytest.fixture(scope="module")
def batched():
    from cygym_b200.payoff import evaluate_payoff_matrix_batched
    defs, atts = _strategies()
    return evaluate_payoff_matrix_batched(_net(), defs, atts, N, steps_per_episode=T, seed=SEED, xcap=XCAP,
                                          train_detectors=True).cpu().numpy()


def test_detector_fit_seeds():
    import torch
    from cygym_b200.payoff import detector_fit_seeds
    g = torch.arange(0, 5000, dtype=torch.int64)
    a = detector_fit_seeds(3, g, 4)
    assert a.dtype == torch.int64 and bool(((a >= 0) & (a < 2 ** 32)).all())
    assert torch.equal(a, detector_fit_seeds(3, g.cuda(), 4).cpu())  # the same on either device
    assert torch.equal(a[1234:1240], detector_fit_seeds(3, g[1234:1240], 4))  # per env: no dependence on the batch
    assert len(set(a.tolist())) > 4990
    assert not torch.equal(a, detector_fit_seeds(4, g, 4)) and not torch.equal(a, detector_fit_seeds(3, g, 6))


def test_batched_matches_oracle_with_fits(batched):
    defs, atts = _strategies()
    exp, n_fits = _oracle_payoff(_net(), defs, atts, N, T)
    assert n_fits > 100
    assert batched.shape == (3, 2, 10)
    assert np.allclose(batched, exp, rtol=1e-5, atol=1e-6), np.abs(batched - exp).max()
    # the scans consulted a model: the same oracle run without training differs
    defs0, _ = _strategies(train=False)
    plain, _ = _oracle_payoff(_net(), defs0[:1], atts, N, T, fit=False)
    assert not np.allclose(plain[0], exp[0], rtol=1e-5, atol=1e-6)


def test_invariance(batched):
    from cygym_b200.payoff import evaluate_payoff_matrix, evaluate_payoff_matrix_batched, reduce_payoff
    net = _net()
    defs, atts = _strategies()
    kw = dict(steps_per_episode=T, seed=SEED, xcap=XCAP, train_detectors=True)
    for spl in (7, 1):
        alt = evaluate_payoff_matrix_batched(net, defs, atts, N, steps_per_launch=spl, **kw).cpu().numpy()
        assert np.allclose(alt, batched, rtol=1e-12, atol=1e-9), (spl, np.abs(alt - batched).max())
    for world in (3, 2):  # world 3: contiguous slices of the (pair, rollout) index; world 2 divides N: strided env ids
        parts = [evaluate_payoff_matrix_batched(net, defs, atts, N, rank=r, world=world, reduce=False, **kw) for r in range(world)]
        got = reduce_payoff(sum(parts), N, T).cpu().numpy()
        assert np.allclose(got, batched, rtol=1e-12, atol=1e-9), (world, np.abs(got - batched).max())
    pairwise = evaluate_payoff_matrix(net, defs, atts, N, **kw).cpu().numpy()
    assert np.allclose(pairwise, batched, rtol=1e-12, atol=1e-9), np.abs(pairwise - batched).max()


def test_default_path_leaves_the_error_bit():
    """Without train_detectors the evaluation runs as before: the stub scans leave CYG_FL_ERR_DETECTOR, nothing raises,
    and the result differs from the one with fits."""
    from cygym_b200 import _capi as K
    from cygym_b200.payoff import _ENV_CACHE, evaluate_payoff_matrix_batched
    net = _net()
    defs, atts = _strategies()
    got = evaluate_payoff_matrix_batched(net, defs[:1], atts[:1], 8, steps_per_episode=T, seed=SEED, xcap=XCAP).cpu().numpy()
    (env,) = _ENV_CACHE.values()
    assert env.log_cap == 0
    assert bool(((env.error_flags() & K.FL_ERR_DETECTOR) != 0).any())
    fit = evaluate_payoff_matrix_batched(net, defs[:1], atts[:1], 8, steps_per_episode=T, seed=SEED, xcap=XCAP,
                                         train_detectors=True).cpu().numpy()
    (env2,) = _ENV_CACHE.values()
    assert env2 is not env and env2.log_cap > 0
    assert not np.allclose(got, fit)


class _TrainOrScan:
    """A fixed actor (float64, exact: no matmul whose reduction order could flip a decision): the type slice's argmax is
    10 (train) when the observed known / not-yet-added bits sum to an even number and 5 (scan) otherwise; the device
    slice lists every visible device; exploit and app slices argmax to 0."""

    def __new__(cls, M, X, A):
        import torch

        class Actor(torch.nn.Module):
            def forward(self, x):
                x = x.double()
                s = x[:, 4::6].sum(1) + x[:, 5::6].sum(1)
                y = torch.full((x.shape[0], 14 + M + X + A), -1.0, dtype=torch.float64, device=x.device)
                train = torch.remainder(s, 2) == 0
                y[:, 10] = torch.where(train, 1.0, 0.0)
                y[:, 5] = torch.where(train, 0.0, 1.0)
                y[:, 14:14 + M] = torch.where(x[:, 0::6] != -1, 1.0, -1.0)
                y[:, 14 + M] = 0.0
                if A:
                    y[:, 14 + M + X] = 0.0
                return y
        return Actor().cuda().eval()


def test_actor_strategies_with_fits():
    from cygym_b200.payoff import Strategy, evaluate_payoff_matrix_batched
    net = _net()
    M, X, A = net.M, net.X, int(net.cfg.get("n_app_ids", 0))
    defs = [Strategy(actor=_TrainOrScan(M, X, A)), Strategy(baseline_name="Nash")]
    atts = [Strategy(actions=[(1, [0], [], 0), (1, [1], [], 0), (2, [0], [], 0)])]
    n, steps = 16, 30
    got = evaluate_payoff_matrix_batched(net, defs, atts, n, steps_per_episode=steps, seed=SEED, xcap=XCAP,
                                         train_detectors=True).cpu().numpy()
    exp, n_fits = _oracle_payoff(net, defs, atts, n, steps)
    assert n_fits > 20
    assert np.allclose(got, exp, rtol=1e-5, atol=1e-6), np.abs(got - exp).max()


# ---- the rollout kernel with a ring (cyg_step_kernel<W, true, true>) ----

def _tables(M, T, R, rng):
    """Per-row action tables [T, R, 4] / [T, R, W] (int32, device): defender rows train (type 10) on some turns and scan
    (type 5) on others, attacker rows attack (types 1 / 2).  Returns (hdr, mask, the turns at which some row trains)."""
    import torch
    from cygym_b200.vector_env import ActionBatch
    hs, ms, train_turns = [], [], []
    for t in range(T):
        acts = []
        for r in range(R):
            if t & 1:
                acts.append((int(rng.integers(1, 3)), [int(rng.integers(0, 2))], [], 0))
            else:
                at = 10 if (t % 8 == 4 and r % 3 != 2) else int(rng.choice([5, 5, 7, 1, 6]))
                devs = sorted(int(d) for d in rng.choice(M, size=int(rng.integers(1, M)), replace=False))
                acts.append((at, [0], devs, 0))
        if any(a[0] == 10 for a in acts) and not (t & 1):
            train_turns.append(t)
        h, m, _ = ActionBatch.pack(acts, t & 1, M)
        hs.append(h.view(np.int32))
        ms.append(m.view(np.int32))
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(np.stack(a))).cuda()
    return tt(hs), tt(ms), train_turns


def _state_words(env):
    c = env.export_state()
    return {**c, "det_slots": env._det_slots.clone(), "det_of_env": env._det_of_env.clone(), "next_slot": env._next_slot.clone()}


@pytest.mark.parametrize("M", [20, 50, 100])
def test_rollout_with_ring_matches_single_steps(M):
    import torch
    from cygym_b200 import _capi as K, synthetic_network
    from cygym_b200.vector_env import ActionBatch, VectorCyberDefenseEnv
    B, R, T_ = 2048, 16, 40
    net = synthetic_network(M, n_subnets=max(1, M // 16), seed=M)
    assert net.W == {20: 1, 50: 2, 100: 4}[M]
    mk = lambda: VectorCyberDefenseEnv(net, B, seed=7, env_id0=11, xcap=XCAP, log_cap=2000, detector_slots=B)
    roll, single = mk(), mk()
    for e in (roll, single):
        e.randomize_compromise_and_ownership()
    hdr, mask, train_turns = _tables(M, T_, R, np.random.default_rng(M))
    assert len(train_turns) >= 4
    epr = B // R
    row = torch.arange(B, device="cuda") // epr
    seeds = torch.from_numpy(np.random.default_rng(1).integers(0, 2 ** 32, size=B, dtype=np.int64)).cuda()
    bounds = [0] + [t + 1 for t in train_turns if t < T_ - 1] + [T_]
    n_fitted = 0
    for t0, t1 in zip(bounds[:-1], bounds[1:]):
        roll.rollout(hdr[t0:t1], mask[t0:t1], None, epr, 0)
        for t in range(t0, t1):
            single.step(ActionBatch(hdr[t][row].contiguous(), mask[t][row].contiguous()))
        torch.cuda.synchronize()
        n_fitted += len(roll.pending_detectors())
        for e in (roll, single):
            e.fit_detectors(seeds)
        a, b = _state_words(roll), _state_words(single)
        for k in a:
            assert torch.equal(a[k], b[k]), f"M={M}, turns [{t0}, {t1}): {k}"
    assert n_fitted > B
    flags = roll.scalars[:, K.S_FLAGS]
    assert not bool(((flags & K.FL_ERR_DETECTOR) != 0).any())
    assert bool(((flags & K.FL_DET_TRAINED) != 0).any())
    assert int(roll.scalars[:, K.S_SCAN].sum()) > 0


def test_train_then_scan_in_one_launch_sets_the_error_bit():
    """No fit inside a launch: an env that trains and scans later in the SAME rollout launch gets CYG_FL_ERR_DETECTOR
    (as in cyg_step_multi); the envs that did not train get none."""
    import torch
    from cygym_b200 import _capi as K
    from cygym_b200.vector_env import ActionBatch, VectorCyberDefenseEnv
    net = _net()
    M, B, R = net.M, 2048, 8
    env = VectorCyberDefenseEnv(net, B, seed=3, xcap=XCAP, log_cap=2000, detector_slots=B)
    env.randomize_compromise_and_ownership()
    attack = [(1, [0], [], 0)] * R
    every = list(range(M))
    turns = [([(8, [0], [], 0)] * R, 0), (attack, 1)] * 6 + \
            [([(10, [0], [], 0) if r % 2 == 0 else (8, [0], [], 0) for r in range(R)], 0), (attack, 1), ([(5, [0], every, 0)] * R, 0)]
    packed = [ActionBatch.pack(a, mode, M) for a, mode in turns]
    hdr = torch.from_numpy(np.stack([h.view(np.int32) for h, _, _ in packed])).cuda().contiguous()
    mask = torch.from_numpy(np.stack([m.view(np.int32) for _, m, _ in packed])).cuda().contiguous()
    env.rollout(hdr, mask, None, B // R, 0)
    torch.cuda.synchronize()
    flags = env.scalars[:, K.S_FLAGS]
    trained = (torch.arange(B, device="cuda") // (B // R)) % 2 == 0
    pending = (flags & K.FL_DET_PENDING) != 0
    err = (flags & K.FL_ERR_DETECTOR) != 0
    assert bool(pending[trained].float().mean() > 0.5)  # almost every env attacked (a non-empty log) before it trained
    assert not bool(pending[~trained].any())
    assert torch.equal(err, pending)


# ---- cyg_fit_detectors: grid-wide slot assignment ----

def _sparse_pending(B, rng):
    """An irregular, sparse set of envs: the ends, both sides of assignment-chunk boundaries, a dense run, scattered."""
    idx = {0, 1, B - 1, 2047, 2048, 2049, 4095, 4096, 131071, 131072}
    idx |= set(range(70000, 70000 + 300))
    idx |= set(rng.choice(B, 1500, replace=False).tolist())
    return np.array(sorted(idx))


def _make_pending(env, envs, rng, n_logs=None):
    """Env b of `envs` trained: CYG_FL_DET_TRAINED | PENDING, a hop log of n_logs (default: 40..399) records written into
    its ring over the network's device ids."""
    import torch
    from cygym_b200 import _capi as K
    envs_t = torch.from_numpy(envs).cuda()
    n = torch.from_numpy(rng.integers(40, 400, size=len(envs)).astype(np.int32)).cuda() if n_logs is None else \
        torch.full((len(envs),), n_logs, dtype=torch.int32, device="cuda")
    base = env.B * (env.S + env.M + env.xcap)
    ring = env._state[base:base + env.B * env.log_cap].view(env.B, env.log_cap)
    words = torch.from_numpy((rng.integers(0, env.M, size=(len(envs), 400)) | (rng.integers(0, env.M, size=(len(envs), 400)) << 16)).astype(np.int32)).cuda()
    ring[envs_t, :400] = words
    env.scalars[envs_t, K.S_LOGS] = n
    env.scalars[envs_t, K.S_FLAGS] |= K.FL_DET_TRAINED | K.FL_DET_PENDING


def _host_slot(env, b, seed):
    from cygym_b200 import detector as DET
    return DET.pack_detector(DET.fit_detector(env.log_records(b), int(seed))).view(np.int32)


def test_grid_wide_slot_assignment():
    import torch
    from cygym_b200 import _capi as K, synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    B = 262144
    rng = np.random.default_rng(11)
    net = synthetic_network(50, n_subnets=3, seed=2)
    seeds = torch.from_numpy(rng.integers(0, 2 ** 32, size=B, dtype=np.int64)).cuda()
    env = VectorCyberDefenseEnv(net, B, seed=1, log_cap=2000, detector_slots=8192)
    first = _sparse_pending(B, rng)
    _make_pending(env, first, rng)
    env.fit_detectors(seeds)
    torch.cuda.synchronize()
    slots = env._det_of_env.cpu().numpy()
    assert np.array_equal(slots[first], np.arange(len(first)))  # env order from slot 0
    assert (np.delete(slots, first) == -1).all()
    assert int(env._next_slot.item()) == len(first)
    assert not bool((env.error_flags() != 0).any()) and env.pending_detectors() == []
    # a second round: some envs retrain (they keep their slots), new ones take the next slots in env order, and pending
    # envs whose log is empty cannot be fitted (error bit, no slot)
    again = np.sort(rng.choice(first, 200, replace=False))
    new = np.setdiff1d(_sparse_pending(B, np.random.default_rng(12)), first)
    empty = np.setdiff1d(np.array([5, 3000, 200001]), np.concatenate([first, new]))
    _make_pending(env, np.concatenate([again, new]), rng)
    _make_pending(env, empty, rng, n_logs=0)
    env.fit_detectors(seeds)
    torch.cuda.synchronize()
    slots2 = env._det_of_env.cpu().numpy()
    assert np.array_equal(slots2[first], slots[first])
    assert np.array_equal(slots2[new], len(first) + np.arange(len(new)))
    assert (slots2[empty] == -1).all()
    assert int(env._next_slot.item()) == len(first) + len(new)
    flags = env.scalars[:, K.S_FLAGS].cpu().numpy()
    err = np.nonzero(flags & K.FL_ERR_DETECTOR)[0]
    assert np.array_equal(err, empty) and np.array_equal(np.nonzero(flags & K.FL_DET_PENDING)[0], empty)
    for b in list(rng.choice(new, 6, replace=False)) + list(rng.choice(again, 4, replace=False)) + [new[0], new[-1]]:
        assert np.array_equal(env._det_slots[slots2[b]].cpu().numpy(), _host_slot(env, b, seeds[b])), f"env {b}"
    del env
    torch.cuda.empty_cache()

    # fewer slots than pending envs: the first n in env order get them, the rest stay pending with the error bit
    n_slots = 700
    small = VectorCyberDefenseEnv(net, B, seed=1, log_cap=2000, detector_slots=n_slots)
    _make_pending(small, first, np.random.default_rng(13))
    small.fit_detectors(seeds)
    torch.cuda.synchronize()
    slots = small._det_of_env.cpu().numpy()
    flags = small.scalars[:, K.S_FLAGS].cpu().numpy()
    got, over = first[:n_slots], first[n_slots:]
    assert np.array_equal(slots[got], np.arange(n_slots)) and (slots[over] == -1).all()
    assert ((flags[over] & K.FL_DET_PENDING) != 0).all() and ((flags[over] & K.FL_ERR_DETECTOR) != 0).all()
    assert ((flags[got] & (K.FL_DET_PENDING | K.FL_ERR_DETECTOR)) == 0).all()
    assert int(small._next_slot.item()) == n_slots
    for b in [got[0], got[n_slots // 2], got[-1]]:
        assert np.array_equal(small._det_slots[slots[b]].cpu().numpy(), _host_slot(small, b, seeds[b])), f"env {b}"
