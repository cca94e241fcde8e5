"""Parity of the CUDA path with the oracle, through the C-ABI (run on the B200 box: -m gpu).

 * golden trajectories recorded from the unmodified reference, replayed on the GPU (B = 1);
 * batched random rollouts at the BASELINE.json shapes vs the C oracle on the same seeded inputs:
   integer / boolean state bit-exact, rewards within 1e-5 relative (fp32 outputs vs float64);
 * at the full 65 536 x 100 size: size-independent properties (shard invariance, determinism,
   export/import round trip) plus an oracle check of a contiguous slice of the big batch.
"""
import numpy as np
import pytest

from oracle import trajectory as TR
from tests.common import (GOLDEN, GOLDEN_IDS, CudaImpl, compare_rewards, compare_states, load_golden, oracle_for,
                          oracle_state_from_template, sanitize_actions)

pytestmark = pytest.mark.gpu
RTOL = 1e-5  # north_star: rewards / payoffs within 1e-5 relative


def _np(c):
    return {k: v.cpu().numpy().view(np.uint32) for k, v in c.items()}


def test_library_loaded_is_the_cuda_one():
    import torch
    from cygym_b200 import _capi
    assert torch.cuda.is_available()
    assert _capi.lib().cyg_version() == 3
    assert "sm_100" in " ".join(torch.cuda.get_arch_list()) or torch.cuda.get_device_capability()[0] >= 10


@pytest.mark.parametrize("path", GOLDEN, ids=GOLDEN_IDS)
def test_cuda_replays_golden(path):
    g = load_golden(path)
    n = TR.replay(g, CudaImpl(g), rtol=RTOL, label="cuda")
    assert n == len(g["kind"])


def _rollout_vs_oracle(M, subnets, B, T, seed=5, env_id0=3, obs_every=7, xcap=64, dense_multi=False, base_line="Nash", net=None, **kw):
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv, ActionBatch
    if net is None:
        net = synthetic_network(M, n_subnets=subnets, seed=seed, **kw)
    if dense_multi:  # ~10 % of the pairs become multi-edges of multiplicity 2..4 (> 2 per list -> the general routines)
        rng = np.random.default_rng(M)
        m = net.mult.copy()
        idx = rng.choice(len(m), size=max(1, len(m) // 10), replace=False)
        m[idx] = rng.integers(2, 5, size=len(idx))
        net.mult = m
    orc, cfg = oracle_for(net, seed=1234, xcap=xcap, env_id0=env_id0, base_line=base_line)
    env = VectorCyberDefenseEnv(net, B, seed=1234, env_id0=env_id0, xcap=xcap, base_line=base_line)
    so = oracle_state_from_template(orc, net, B)
    for t in range(T):
        mode = t & 1
        if t % 29 == 28:
            orc.randomize(so)
            env.randomize_compromise_and_ownership()
        ho, mo = orc.sample_actions(so, mode)
        ab = env.sample_actions(mode)
        torch.cuda.synchronize()
        assert np.array_equal(ab.hdr.cpu().numpy().view(np.uint32), ho), f"sample_action hdr t={t}"
        assert np.array_equal(ab.mask.cpu().numpy().view(np.uint32), mo), f"sample_action mask t={t}"
        ho = sanitize_actions(ho, so.scal[:, 6], mode)
        if t % 11 == 10:
            ho[::3, 0] = 0x80 | (mode << 8)
        oo = orc.step(so, ho, mo, n_threads=8)
        om = 1 + (t % 3) if t % obs_every == 0 else 0
        raw, shaped, done = env.step(env.to_device(ho, mo), obs_mode=om)
        torch.cuda.synchronize()
        og = dict(raw=raw.cpu().numpy(), shaped=shaped.cpu().numpy(), done=done.cpu().numpy())
        compare_rewards(og, oo, f"t={t}", RTOL)
        if t % 5 == 0 or t == T - 1:
            compare_states(_np(env.export_state()), dict(dev=so.dev, ckpt=so.ckpt, blocked=so.blocked, extra=so.extra, scal=so.scal), f"t={t}", RTOL)
        if om:
            assert np.array_equal(env.last_obs(om).cpu().numpy(), orc.observe(so, om)), f"fused obs mode {om} t={t}"
            assert np.array_equal(env.observe(om).cpu().numpy(), orc.observe(so, om)), f"observe mode {om} t={t}"
    assert int(env.error_flags().max().item()) == 0
    assert env.launch_count > T


def test_snapshot_of_a_reference_env_steps_like_the_oracle():
    """f2: tests/golden/snapshots/ref_m30_step30.npz is a reference env 30 steps into an episode, flattened by
    cygym_b200.snapshot.from_reference_env and saved by save_npz (oracle/gen_snapshot.py; the flattening itself is checked
    against the harness in tests/test_oracle_vs_reference.py).  Loaded here without the reference, its state (compromised
    devices, workloads in flight, busy timers, counters) is the template of 512 envs that then step bit-exactly with the
    oracle from that state."""
    import os
    from cygym_b200 import snapshot
    from tests.common import ROOT
    net = snapshot.load_npz(os.path.join(ROOT, "tests", "golden", "snapshots", "ref_m30_step30.npz"))
    assert net.M == 30 and int((net.template["dev"] & 1).sum()) > 0 and int(net.template["scal"][0]) == 30
    _rollout_vs_oracle(net.M, 1, 512, 120, net=net)


def test_c1_default_network_rollout():
    _rollout_vs_oracle(20, 1, 64, 300, num_of_device=10)


def test_c2_4096_envs_50_devices():
    _rollout_vs_oracle(50, 3, 4096, 60)


def test_c3_shape_8192_envs_100_devices():
    _rollout_vs_oracle(100, 8, 8192, 50)


def test_ragged_batch_and_odd_sizes():
    _rollout_vs_oracle(33, 2, 1001, 40)      # B not a multiple of the CTA block; M not a multiple of 32
    _rollout_vs_oracle(128, 4, 257, 30)      # maximum M of the bit-matrix kernels
    _rollout_vs_oracle(1, 1, 5, 20, num_of_device=1)


def test_c4_large_network_2000_devices_64_subnets():
    """BASELINE.json config C4: the adjacency bit matrix exceeds shared memory -> generic global-memory kernel."""
    _rollout_vs_oracle(2000, 64, 1024, 12, obs_every=5, xcap=256)  # ~100 attacker-owned devices: up to 198 hub-star edges
    _rollout_vs_oracle(300, 8, 200, 30)


def test_evolving_topology_with_attacker_arrivals():
    _rollout_vs_oracle(60, 3, 512, 80, xcap=160, p_add=0.5, p_attacker=0.4, lambda_events=1.5)


def test_dense_multi_edges_and_other_attributes():
    """Dense multi-edges (general block/unblock and attack routines inside the warp-per-env phase), workload caps,
    frequent arrivals, odd evolve periods, every base line."""
    _rollout_vs_oracle(100, 8, 1024, 50, dense_multi=True)
    _rollout_vs_oracle(64, 4, 600, 50, dense_multi=True, xcap=200, zero_day=1, zero_day_mask=0b11, p_attacker=0.5, p_add=0.5, lambda_events=1.2)
    _rollout_vs_oracle(100, 8, 900, 40, workload_period_base=3, workload_period_max=12, workload_cap=5)
    _rollout_vs_oracle(40, 1, 500, 40, scaling_vulnerability=0, evolve_period=3, default_high=5)
    for bl in ("No Defense", "Preset", "No Attack"):
        _rollout_vs_oracle(50, 3, 300, 16, base_line=bl)


def test_zero_day_remap():
    _rollout_vs_oracle(40, 2, 256, 60, zero_day=1, zero_day_mask=0b10)


def test_grouped_and_order_form_steps():
    """step_grouped (volt:694-779) and explicit device_indices order, vs the oracle."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    rng = np.random.default_rng(0)
    M, B, G = 50, 300, 4
    net = synthetic_network(M, n_subnets=3, seed=11)
    orc, cfg = oracle_for(net, seed=77, xcap=32)
    env = VectorCyberDefenseEnv(net, B, seed=77, xcap=32)
    so = oracle_state_from_template(orc, net, B)
    W = net.W
    for t in range(40):
        mode = t & 1
        hdr = np.zeros((G, B, 4), np.uint32); mask = np.zeros((G, B, W), np.uint32); order = np.zeros((G, B, M), np.uint16)
        for g in range(G):
            for b in range(B):
                n = int(rng.integers(0, M))
                devs = rng.permutation(M)[:n]
                at = int(rng.choice([0, 1, 1, 2, 3, 8, 11, 1, 5, 7])) if n > 0 else 8
                if t % 4 == 3:
                    at = int(rng.integers(0, 14 if mode == 0 else 5))
                    if at == 10 and so.scal[b, 6] > 0:
                        at = 8
                    if at in (11, 12, 13) and n == 0:
                        at = 8
                hdr[g, b] = [(at & 0xFF) | (mode << 8) | (1 << 16), int(rng.integers(0, 6)), n, int(rng.integers(0, 9))]
                order[g, b, :n] = devs
                for d in devs:
                    mask[g, b, d >> 5] |= np.uint32(1 << (d & 31))
        from cygym_b200.vector_env import ActionBatch
        if t % 4 == 3:   # plain step with an explicit order
            oo = orc.step(so, hdr[0], mask[0], order[0])
            raw, shaped, done = env.step(env.to_device(hdr[0], mask[0], order[0]))
        else:
            oo = orc.step(so, hdr, mask, order, flags=1)
            raw, shaped, done = env.step_grouped([env.to_device(hdr[g], mask[g], order[g]) for g in range(G)])
        torch.cuda.synchronize()
        compare_rewards(dict(raw=raw.cpu().numpy(), shaped=shaped.cpu().numpy(), done=done.cpu().numpy()), oo, f"t={t}", RTOL)
        compare_states(_np(env.export_state()), dict(dev=so.dev, ckpt=so.ckpt, blocked=so.blocked, extra=so.extra, scal=so.scal), f"t={t}", RTOL)


def test_full_size_properties_65536_x_100():
    """BASELINE.json C3 at full size: shard invariance + determinism + round trip + oracle slice."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    net = synthetic_network(100, n_subnets=8, seed=0)
    B, T, xcap = 65536, 24, 16
    whole = VectorCyberDefenseEnv(net, B, seed=42, xcap=xcap)
    halves = [VectorCyberDefenseEnv(net, B // 2, seed=42, env_id0=i * (B // 2), xcap=xcap) for i in range(2)]
    k0, kn = 40000, 768
    orc, cfg = oracle_for(net, seed=42, xcap=xcap, env_id0=k0)
    so = oracle_state_from_template(orc, net, kn)
    for t in range(T):
        mode = t & 1
        ab = whole.sample_actions(mode)
        hs = [h.sample_actions(mode) for h in halves]
        torch.cuda.synchronize()
        assert torch.equal(torch.cat([x.hdr for x in hs]), ab.hdr) and torch.equal(torch.cat([x.mask for x in hs]), ab.mask)
        # the trained-detector branch is out of scope: rewrite defender 10 -> 8 on the device
        if mode == 0:
            for a, e in [(ab, whole)] + list(zip(hs, halves)):
                bad = ((a.hdr[:, 0] & 0xFF) == 10) & (e.scalars[:, 6] > 0)
                a.hdr[:, 0] = torch.where(bad, (a.hdr[:, 0] & ~0xFF) | 8, a.hdr[:, 0])
        r = [x.clone() for x in whole.step(ab)]
        rh = [[x.clone() for x in h.step(a)] for h, a in zip(halves, hs)]
        torch.cuda.synchronize()
        for i in range(3):
            assert torch.equal(torch.cat([rh[0][i], rh[1][i]]), r[i]), f"shard invariance, output {i}, t={t}"
        ho = ab.hdr[k0:k0 + kn].cpu().numpy().view(np.uint32)
        mo = ab.mask[k0:k0 + kn].cpu().numpy().view(np.uint32)
        so.scal[:, 1] += 1  # the sample_action epoch
        oo = orc.step(so, ho, mo, n_threads=8)
        compare_rewards(dict(raw=r[0][k0:k0 + kn].cpu().numpy(), shaped=r[1][k0:k0 + kn].cpu().numpy(),
                             done=r[2][k0:k0 + kn].cpu().numpy()), oo, f"slice t={t}", RTOL)
    cw = _np(whole.export_state())
    ch = [_np(h.export_state()) for h in halves]
    for k in cw:
        assert np.array_equal(np.concatenate([ch[0][k], ch[1][k]]), cw[k]), f"shard invariance of {k}"
    compare_states({k: v[k0:k0 + kn] for k, v in cw.items()},
                   dict(dev=so.dev, ckpt=so.ckpt, blocked=so.blocked, extra=so.extra, scal=so.scal), "slice", RTOL)
    # export -> import -> export is the identity
    again = VectorCyberDefenseEnv(net, B, seed=42, xcap=xcap)
    again.import_state(whole.export_state())
    ca = _np(again.export_state())
    for k in cw:
        assert np.array_equal(ca[k], cw[k]), f"round trip of {k}"
    # conservation: every env advanced exactly T steps; counters are consistent
    s = cw["scal"]
    assert (s[:, 0] == T).all() and (s[:, 4] + s[:, 5] == T).all()
    assert int(whole.error_flags().max().item()) == 0


def test_errors_are_loud():
    import ctypes as C
    from cygym_b200 import _capi as K, synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    net = synthetic_network(20, n_subnets=1, seed=1)
    env = VectorCyberDefenseEnv(net, 4)
    a = K.CygActions(None, None, None, 0, 1)
    o = K.CygStepOut(None, None, None, None, None, 0)
    rc = env.L.cyg_step(env.h, C.byref(a), 0, C.byref(o), None)
    assert rc == K.E_INVAL and b"null" in env.L.cyg_last_error()
    with pytest.raises(K.CygError):
        net.cfg["evolve_period"] = 0
        VectorCyberDefenseEnv(net, 4)


def test_step_host_matches_device_step():
    """The host-buffer call (pinned H2D + kernel + D2H, CUDA-graph replayed) gives the same transition as step()."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    net = synthetic_network(100, n_subnets=8, seed=2)
    B = 3000
    a = VectorCyberDefenseEnv(net, B, seed=9)
    b = VectorCyberDefenseEnv(net, B, seed=9)
    hdr_h, mask_h, out_h = b.host_buffers()
    for t in range(12):
        ab = a.sample_actions(t & 1)
        b.sample_actions(t & 1)          # keeps the draw epochs of the two envs aligned
        torch.cuda.synchronize()
        r = [x.clone() for x in a.step(ab)]
        hdr_h.copy_(ab.hdr.cpu()); mask_h.copy_(ab.mask.cpu())
        raw, shaped, done = b.step_host(use_graph=(t >= 2))   # eager first, then captured + replayed
        assert torch.equal(raw, r[0].cpu()) and torch.equal(shaped, r[1].cpu()) and torch.equal(done, r[2].cpu()), t
    # combined [B, 4 + W] rows in the caller's own pinned buffer (one host->device copy)
    ab = a.sample_actions(0)
    b.sample_actions(0)
    torch.cuda.synchronize()
    r = [x.clone() for x in a.step(ab)]
    rows = torch.cat([ab.hdr, ab.mask], dim=1).cpu().pin_memory()
    for _ in range(1):
        raw, shaped, done = b.step_host(act=rows)
    assert torch.equal(raw, r[0].cpu()) and torch.equal(done, r[2].cpu())
    # compact [B, 2 + W] rows (24 bytes per env over PCIe instead of 32), expanded on the device by cyg_unpack_actions
    from cygym_b200.vector_env import compact_action_rows, expand_action_rows
    rows_c = torch.empty(B, 2 + a.W, dtype=torch.int32).pin_memory()  # ONE staging buffer, kept: the replayed graph holds its address
    for t in range(4):
        ab = a.sample_actions(t & 1)
        b.sample_actions(t & 1)
        torch.cuda.synchronize()
        r = [x.clone() for x in a.step(ab)]
        rows_c.copy_(torch.from_numpy(compact_action_rows(ab.hdr.cpu(), ab.mask.cpu())))
        raw, shaped, bits = b.step_host(act=rows_c, packed_done=(t >= 2))   # t >= 2: done comes back as one bit per env
        done = bits if t < 2 else torch.from_numpy(((bits.numpy().view(np.uint32)[np.arange(B) >> 5] >> (np.arange(B) & 31)) & 1).astype(np.int32))
        assert torch.equal(raw, r[0].cpu()) and torch.equal(shaped, r[1].cpu()) and torch.equal(done, r[2].cpu()), t
        assert b.host_result_bytes(True) == 4 * (2 * B + (B + 31) // 32)
        h2, m2 = expand_action_rows(rows_c.numpy())
        assert np.array_equal(b._host["d_hdr"].cpu().numpy().view(np.uint32), h2) and np.array_equal(b._host["d_mask"].cpu().numpy().view(np.uint32), m2)
    ca, cb = a.export_state(), b.export_state()
    for k in ca:
        assert torch.equal(ca[k], cb[k]), k
    assert b.launch_count >= 13


def test_step_host_follows_base_line_changes():
    """A captured step_host() graph holds the kernel parameters by value: set_base_line() / set_base_line_per_env()
    between two replays must reach the next step (the captures are dropped), as they do for step()."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    net = synthetic_network(100, n_subnets=8, seed=2)
    B = 1500
    a = VectorCyberDefenseEnv(net, B, seed=9)
    b = VectorCyberDefenseEnv(net, B, seed=9)
    hdr_h, mask_h, _ = b.host_buffers()

    def both(t):
        ab = a.sample_actions(t & 1)
        b.sample_actions(t & 1)
        torch.cuda.synchronize()
        r = [x.clone().cpu() for x in a.step(ab)]
        hdr_h.copy_(ab.hdr.cpu()); mask_h.copy_(ab.mask.cpu())
        raw, shaped, done = b.step_host()
        assert torch.equal(raw, r[0]) and torch.equal(shaped, r[1]) and torch.equal(done, r[2]), t

    for t in range(4):
        both(t)                     # captured at t = 0, replayed afterwards
    for e in (a, b):
        e.set_base_line("No Defense")
    for t in range(4, 8):
        both(t)
    codes = (torch.arange(B, device="cuda") % 4).to(torch.uint8)
    for e in (a, b):
        e.set_base_line_per_env(codes)
    for t in range(8, 12):
        both(t)
    for e in (a, b):
        e.set_base_line_per_env(None)
        e.set_base_line("Nash")
    for t in range(12, 14):
        both(t)
    ca, cb = a.export_state(), b.export_state()
    for k in ca:
        assert torch.equal(ca[k], cb[k]), k


def test_step_host_two_groups_async():
    """Two env groups on two streams driven through step_host(sync=False) / wait_host() (the double-buffered rollout
    loop of bench.py's e2e leg) give the same rewards and states as the synchronous device steps."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    net = synthetic_network(100, n_subnets=8, seed=3)
    B = 2048
    ref = [VectorCyberDefenseEnv(net, B, seed=4, env_id0=g * B) for g in range(2)]
    rows, want = {}, {}
    for t in range(6):
        for g in range(2):
            ab = ref[g].sample_actions(t & 1)
            torch.cuda.synchronize()
            want[g, t] = [x.clone().cpu() for x in ref[g].step(ab)]
            rows[g, t] = torch.cat([ab.hdr, ab.mask], dim=1).cpu().pin_memory()
    torch.cuda.synchronize()
    # the same six turns of both groups, interleaved, a group only ever waiting for its own previous step
    grp = [VectorCyberDefenseEnv(net, B, seed=4, env_id0=g * B, stream=torch.cuda.Stream()) for g in range(2)]
    torch.cuda.synchronize()
    for t in range(6):
        for g in range(2):
            if t > 0:
                raw, shaped, done = grp[g].wait_host()
                w = want[g, t - 1]
                assert torch.equal(raw, w[0]) and torch.equal(shaped, w[1]) and torch.equal(done, w[2]), (g, t)
            grp[g].sample_actions(t & 1)  # keeps the draw epochs aligned with the reference envs
            grp[g].step_host(act=rows[g, t], sync=False)
    for g in range(2):
        raw, shaped, done = grp[g].wait_host()
        assert torch.equal(raw, want[g, 5][0]) and torch.equal(done, want[g, 5][2])
        ca, cb = ref[g].export_state(), grp[g].export_state()
        torch.cuda.synchronize()
        for k in ca:
            assert torch.equal(ca[k].cpu(), cb[k].cpu()), (g, k)


def test_step_many_equals_single_steps():
    """cyg_step_multi: T plain steps fused into one launch (records resident in shared memory) == T cyg_step calls,
    rewards and states bit for bit; C3 shape with a ragged last CTA, and a one-word network."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    for M, subnets, B, T in ((100, 8, 5000, 7), (30, 2, 777, 5)):
        net = synthetic_network(M, n_subnets=subnets, seed=5)
        a = VectorCyberDefenseEnv(net, B, seed=11)  # only here to generate T valid action batches
        hdrs, masks = [], []
        for t in range(T):
            ab = a.sample_actions(t & 1)
            if (t & 1) == 0:  # detector training is out of scope: defender 10 -> 8
                ab.hdr[:, 0] = torch.where((ab.hdr[:, 0] & 0xFF) == 10, (ab.hdr[:, 0] & ~0xFF) | 8, ab.hdr[:, 0])
            hdrs.append(ab.hdr.clone()); masks.append(ab.mask.clone())
            a.step(ab)
        b = VectorCyberDefenseEnv(net, B, seed=11)
        c = VectorCyberDefenseEnv(net, B, seed=11)
        hdr = torch.stack(hdrs).contiguous(); mask = torch.stack(masks).contiguous()
        for t in range(T):
            c.step(type(ab)(hdr[t], mask[t]))
        raw, shaped, done = b.step_many(hdr, mask)
        torch.cuda.synchronize()
        cw = [x.clone() for x in (c.raw, c.shaped, c.done)]
        assert torch.equal(raw[T - 1], cw[0]) and torch.equal(shaped[T - 1], cw[1]) and torch.equal(done[T - 1], cw[2])
        sb, sc = b.export_state(), c.export_state()
        for k in sb:
            assert torch.equal(sb[k], sc[k]), (M, k)
        # and every intermediate reward row
        d = VectorCyberDefenseEnv(net, B, seed=11)
        for t in range(T):
            r = d.step(type(ab)(hdr[t], mask[t]))
            assert torch.equal(raw[t], r[0]) and torch.equal(shaped[t], r[1]) and torch.equal(done[t], r[2]), (M, t)
        assert b.error_flags().max().item() == d.error_flags().max().item()
