"""bench.py: --steps is the number of timed headline steps (also when it is not a multiple of the steps fused per launch),
and --dump-outputs writes what the last timed step returned, the same arrays from run to run, so that two builds can be
compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.common import ROOT

pytestmark = pytest.mark.gpu

NAMES = ("raw_reward", "shaped_reward", "done", "obs")


def _bench(out_dir, args):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--warmup", "3", "--no-legs", "--no-e2e", "--no-cpu-baseline",
           "--dump-outputs", str(out_dir)] + list(args)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def _last_step_by_single_steps(B, K, obs):
    """The headline schedule of bench.py (default network, 3 env sets, a ring of 8 action batches per turn, 64 pre-heat
    launches, warm-up 3) redone with one VectorCyberDefenseEnv.step() per step: what its last timed step returns."""
    import torch
    from cygym_b200 import synthetic_network
    from cygym_b200.vector_env import ActionBatch, VectorCyberDefenseEnv
    n_sets, n_ring, warm, preheat = 3, 8, 3, 64
    F = 1 if obs else 4
    net = synthetic_network(100, n_subnets=8, seed=0)
    sets = [VectorCyberDefenseEnv(net, B, device="cuda:0", seed=0, env_id0=s * B, xcap=16) for s in range(n_sets)]
    ring = {0: [], 1: []}
    for mode in (0, 1):
        for r in range(n_ring):
            ab = sets[r % n_sets].sample_actions(mode)
            if mode == 0:  # detector untrained: defender 10 -> no-op 8
                ab.hdr[:, 0] = torch.where((ab.hdr[:, 0] & 0xFF) == 10, (ab.hdr[:, 0] & ~0xFF) | 8, ab.hdr[:, 0])
            ring[mode].append(ActionBatch(ab.hdr.clone(), ab.mask.clone()))
    if F == 1:
        for i in range(max(warm, preheat) + K):
            env, turn = sets[i % n_sets], (i // n_sets) & 1
            out = list(env.step(ring[turn][(i // (2 * n_sets)) % n_ring], obs_mode=1 + turn if obs else 0))
        if obs:
            out.append(env.last_obs(1 + turn))
    else:
        p0 = max((warm + F - 1) // F, preheat)
        launches = [F] * p0 + [min(F, K - k * F) for k in range((K + F - 1) // F)]
        for j, T in enumerate(launches):  # launch j: env set j % 3, batch variant (j // 3) & 1, T steps
            s_i, v = j % n_sets, (j // n_sets) & 1
            for t in range(T):
                out = list(sets[s_i].step(ring[t & 1][(s_i + v * 3 + t // 2) % n_ring]))
    return {k: x.float().cpu().numpy() for k, x in zip(NAMES, out)}


@pytest.mark.parametrize("args,names,launches", [
    (["--envs", "2048", "--steps", "7"], ["done", "raw_reward", "shaped_reward"], 2),  # 4 steps per launch: 4 + 3
    (["--steps", "5", "--obs", "1"], ["done", "env_index", "obs", "raw_reward", "shaped_reward"], None),  # 65 536 x 600 obs: sampled
], ids=["fused", "obs_sampled"])
def test_bench_steps_and_dumped_outputs(tmp_path, args, names, launches):
    a, da = _bench(tmp_path / "a", args)
    b, db = _bench(tmp_path / "b", args)
    K = int(args[args.index("--steps") + 1])
    assert a["steps"] == b["steps"] == K
    if launches is not None:
        assert a["gpu_launches"] == launches
    assert sorted(da) == sorted(db) == names
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in names) <= 64_000_000
    B = a["config"]["envs_per_gpu"]
    for k in names:
        assert da[k].dtype in (np.float32, np.float64), k
        assert len(da[k]) == len(da["raw_reward"]) <= B, k
        assert np.array_equal(da[k], db[k]), k
    idx = np.arange(B)
    if "env_index" in da:
        idx = da["env_index"]
        assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < B
        idx = idx.astype(np.int64)
    ref = _last_step_by_single_steps(B, K, "--obs" in args)
    for k in names:
        if k != "env_index":
            assert np.array_equal(da[k], ref[k][idx]), k
