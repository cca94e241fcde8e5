"""cyg_fit_detectors / VectorCyberDefenseEnv.fit_detectors on the GPU: the device fit against the host fit
(scikit-learn, service_detectors) slot for slot and step for step."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
pytest.importorskip("sklearn")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.common import GOLDEN, CudaImpl  # noqa: E402


def _env(B, log_cap=2048, detector_slots=None, M=100, seed=3):
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import VectorCyberDefenseEnv
    net = synthetic_network(M, n_subnets=8, seed=seed)
    return VectorCyberDefenseEnv(net, B, seed=seed, log_cap=log_cap, detector_slots=B if detector_slots is None else detector_slots)


def _force(ab, atype, envs=None):
    """Defender action type `atype` for the envs in the bool mask `envs` (all when None)."""
    import torch
    sel = torch.ones_like(ab.hdr[:, 0], dtype=torch.bool) if envs is None else envs
    ab.hdr[:, 0] = torch.where(sel, (ab.hdr[:, 0] & ~0xFF) | atype, ab.hdr[:, 0])


def _no_training(ab):
    import torch
    ab.hdr[:, 0] = torch.where((ab.hdr[:, 0] & 0xFF) == 10, (ab.hdr[:, 0] & ~0xFF) | 8, ab.hdr[:, 0])


def _fill_logs(env, turns):
    """Sampled attack-heavy play: every attacker turn attacks, defender turns never train (10 -> 8)."""
    for t in range(turns):
        ab = env.sample_actions(t & 1)
        if (t & 1) == 0:
            _no_training(ab)
        env.step(ab)


def _train(env, envs=None):
    """One defender step of sampled actions with action 10 forced on `envs`."""
    ab = env.sample_actions(0)
    _no_training(ab)
    _force(ab, 10, envs)
    env.step(ab)


def _host_slot(env, b, seed):
    from cygym_b200 import detector as DET
    return DET.pack_detector(DET.fit_detector(env.log_records(b), int(seed))).view(np.int32)


def _seeds(B, seed=0):
    import torch
    return torch.from_numpy(np.random.default_rng(seed).integers(0, 2 ** 32, size=B, dtype=np.int64))


def test_batch_fit_matches_host():
    import torch
    from cygym_b200 import _capi as K
    env = _env(4096)
    _fill_logs(env, 41)
    _train(env)
    torch.cuda.synchronize()
    pend = env.pending_detectors()
    assert len(pend) > 2000
    before = {k: v.clone() for k, v in env.export_state().items()}
    seeds = _seeds(env.B, 1)
    env.fit_detectors(seeds)
    torch.cuda.synchronize()
    after = env.export_state()
    flags_b, flags_a = before["scal"][:, K.S_FLAGS], after["scal"][:, K.S_FLAGS]
    assert not bool((flags_a & K.FL_DET_PENDING).any())
    assert bool(((flags_a & K.FL_DET_TRAINED) == (flags_b & K.FL_DET_TRAINED)).all())
    assert torch.equal(flags_a, flags_b & ~K.FL_DET_PENDING)
    for k in before:
        if k != "scal":
            assert torch.equal(before[k], after[k]), k
    keep = [i for i in range(K.NSCAL) if i != K.S_FLAGS]
    assert torch.equal(before["scal"][:, keep], after["scal"][:, keep])
    slots = env._det_of_env.cpu().numpy()
    assert np.array_equal(slots[pend], np.arange(len(pend)))  # env order, unique
    assert int(env._next_slot.item()) == len(pend)
    rng = np.random.default_rng(2)
    for b in list(rng.choice(pend, 24, replace=False)) + [pend[0], pend[-1]]:
        got = env._det_slots[slots[b]].cpu().numpy()
        assert np.array_equal(got, _host_slot(env, b, seeds[b])), f"env {b}"


def test_lockstep_with_host_fit():
    import torch
    from cygym_b200 import _capi as K
    B = 512
    a, d = _env(B), _env(B)
    seeds = _seeds(B, 7)
    seed_list = seeds.tolist()
    n_fit = 0
    for t in range(300):
        ab = a.sample_actions(t & 1)
        d.sample_actions(t & 1)  # keeps the draw epochs of the two batches aligned
        ra = [x.clone() for x in a.step(ab)]
        rd = [x.clone() for x in d.step(ab)]
        if (t & 1) == 0:
            n_fit += a.service_detectors(lambda b: seed_list[b])
            d.fit_detectors(seeds)
        torch.cuda.synchronize()
        for i in range(3):
            assert torch.equal(ra[i], rd[i]), f"output {i}, t={t}"
        ca, cd = a.export_state(), d.export_state()
        for k in ca:
            assert torch.equal(ca[k], cd[k]), f"{k}, t={t}"
        assert torch.equal(a.error_flags(), d.error_flags())
        assert not bool(((a.error_flags() & K.FL_ERR_DETECTOR) != 0).any())
    assert n_fit > 100
    used = a._det_of_env >= 0
    assert torch.equal(used, d._det_of_env >= 0)
    # the same slots hold the same models (both paths assign slots in env order within a step)
    assert torch.equal(a._det_of_env, d._det_of_env)
    assert torch.equal(a._det_slots, d._det_slots)
    ns = int(a._next_slot.item())
    assert ns == int(d._next_slot.item()) == int(used.sum().item())
    assert bool(((a.scalars[:, K.S_FLAGS] & K.FL_DET_TRAINED) != 0).any())


class DeviceFitImpl(CudaImpl):
    """The CUDA replay, with the detector fitted on the device from the recorded seed."""

    def service_detector(self, seed):
        import torch
        if seed < 0:
            return super().service_detector(seed)
        self.env.fit_detectors(torch.tensor([seed], dtype=torch.int64))


@pytest.mark.parametrize("name", ["c2_m50_detector", "c1_m30_detector_busy_log"])
def test_goldens_with_device_fit(name):
    from oracle import trajectory as TR
    path = [f for f in GOLDEN if os.path.basename(f) == name + ".npz"]
    assert path, name
    g = dict(np.load(path[0]))
    assert TR.replay(g, DeviceFitImpl(g), rtol=1e-5, label="cuda-devfit") > 0


def test_slot_exhaustion():
    import torch
    from cygym_b200 import _capi as K
    env = _env(64, detector_slots=8)
    _fill_logs(env, 11)
    _train(env)
    seeds = _seeds(64, 3)
    env.fit_detectors(seeds)
    torch.cuda.synchronize()
    pend = np.nonzero(env.export_state()["scal"][:, K.S_FLAGS].cpu().numpy() & K.FL_DET_TRAINED)[0]
    assert len(pend) > 8
    slots = env._det_of_env.cpu().numpy()
    flags = env.scalars[:, K.S_FLAGS].cpu().numpy()
    got, over = pend[:8], pend[8:]
    assert np.array_equal(slots[got], np.arange(8))
    assert (slots[over] == -1).all()
    assert ((flags[over] & K.FL_DET_PENDING) != 0).all() and ((flags[over] & K.FL_ERR_DETECTOR) != 0).all()
    assert ((flags[got] & (K.FL_DET_PENDING | K.FL_ERR_DETECTOR)) == 0).all()
    assert int(env._next_slot.item()) == 8
    env.fit_detectors(seeds)  # nothing left to give: the same envs stay pending, no slot is written twice
    torch.cuda.synchronize()
    assert np.array_equal(env._det_of_env.cpu().numpy(), slots)
    for b in got:
        assert np.array_equal(env._det_slots[slots[b]].cpu().numpy(), _host_slot(env, b, seeds[b]))


def test_mixed_paths_share_the_slot_counter():
    import torch
    from cygym_b200 import _capi as K
    env = _env(64, detector_slots=64)
    _fill_logs(env, 11)
    even = torch.arange(64, device=env.device) % 2 == 0
    _train(env, even)
    torch.cuda.synchronize()
    n_host = env.service_detectors(lambda b: 1000 + b)
    _train(env, ~even)
    seeds = _seeds(64, 4)
    env.fit_detectors(seeds)
    _train(env, even)  # retrain: envs keep their slots, on the device this time
    env.fit_detectors(seeds)
    torch.cuda.synchronize()
    slots = env._det_of_env.cpu().numpy()
    used = slots[slots >= 0]
    assert len(used) == len(set(used.tolist())) == int(env._next_slot.item()) > n_host
    assert not bool(((env.error_flags() & K.FL_ERR_DETECTOR) != 0).any())
    for b in range(0, 64, 4):  # the even envs: fitted last, on the device
        if slots[b] >= 0:
            assert np.array_equal(env._det_slots[slots[b]].cpu().numpy(), _host_slot(env, b, seeds[b]))


def test_refusals():
    import torch
    from cygym_b200 import _capi as K
    short = _env(16, log_cap=30)
    _fill_logs(short, 11)
    _train(short)
    torch.cuda.synchronize()
    assert (short.scalars[:, K.S_LOGS] > 30).any()
    short.fit_detectors(_seeds(16))
    torch.cuda.synchronize()
    flags = short.scalars[:, K.S_FLAGS]
    long = (short.scalars[:, K.S_LOGS] > 30) & ((flags & K.FL_DET_TRAINED) != 0)
    assert bool(((flags[long] & K.FL_DET_PENDING) != 0).all()) and bool(((flags[long] & K.FL_ERR_DETECTOR) != 0).all())
    assert bool((short._det_of_env[long] == -1).all())
    with pytest.raises(ValueError):
        short.service_detectors(lambda b: b)
    bare = _env(4, detector_slots=0)
    with pytest.raises(K.CygError) as e:
        bare.fit_detectors(_seeds(4))
    assert e.value.code == K.E_INVAL
