"""Detector fits on the device (cyg_fit_detectors) at config-C3 shape: 65 536 envs x 100 device slots, log_cap 2048,
65 536 detector slots.  Writes profiles/detector_fit_leg.json (or the path given as argv[1]):

  fit_launch_ms          CUDA-event time of one fit_detectors() call (warmed, median of 5) with 4 096 / 65 536 envs
                         pending, every ring holding >= 2000 records (the fit reads the last 2000)
  closed_loop            200 alternating turns of sampled actions, action 10 kept, fit_detectors() after every defender
                         step: step time of the hop-log (LOG) step kernel, pending envs and fit time per defender step,
                         and whether any env raised an error flag
  host_fit_ms_per_env    pack_detector(fit_detector(...)) (scikit-learn) for 32 of the same envs, per fit
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cygym_b200 import _capi as K, detector as DET, synthetic_network  # noqa: E402
from cygym_b200.vector_env import VectorCyberDefenseEnv  # noqa: E402

B, M, LOG_CAP = 65536, 100, 2048


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the query is informational only
        out = f"unavailable: {e}"
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": out}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def main(out_path):
    net = synthetic_network(M, n_subnets=8, seed=0)
    res = {"card": card(), "shape": dict(B=B, M=M, log_cap=LOG_CAP, detector_slots=B)}
    seeds = torch.from_numpy(np.random.default_rng(0).integers(0, 2 ** 32, size=B, dtype=np.int64)).cuda()

    # 1. launch time: every ring full (2000+ records drawn over the network's device ids), envs pending
    env = VectorCyberDefenseEnv(net, B, seed=1, log_cap=LOG_CAP, detector_slots=B)
    c = env.export_state()
    g = torch.Generator(device="cuda").manual_seed(5)
    frm = torch.randint(0, M, (B, LOG_CAP), device="cuda", generator=g, dtype=torch.int32)
    to = torch.randint(0, M, (B, LOG_CAP), device="cuda", generator=g, dtype=torch.int32)
    c["logs"] = frm | (to << 16)
    c["scal"][:, K.S_LOGS] = 2000 + torch.randint(0, 3000, (B,), device="cuda", generator=g, dtype=torch.int32)
    c["scal"][:, K.S_FLAGS] |= K.FL_DET_TRAINED
    env.import_state(c)
    res["fit_launch_ms"] = {}
    for n in (4096, 65536):
        ts = []
        for rep in range(6):
            env.scalars[:n, K.S_FLAGS] |= K.FL_DET_PENDING
            ts.append(timed(lambda: env.fit_detectors(seeds)))
            assert env.pending_detectors() == []
        res["fit_launch_ms"][str(n)] = {"median": float(np.median(ts[1:])), "all": ts}
    res["error_flags_any_launch_leg"] = bool(env.error_flags().any())
    # host comparison on 32 of the same envs
    t0 = time.perf_counter()
    for b in range(32):
        slot = DET.pack_detector(DET.fit_detector(env.log_records(b), int(seeds[b])))
        assert np.array_equal(slot.view(np.int32), env._det_slots[int(env._det_of_env[b])].cpu().numpy())
    res["host_fit_ms_per_env"] = (time.perf_counter() - t0) * 1000 / 32
    del env
    torch.cuda.empty_cache()

    # 2. closed loop with action 10 kept
    env = VectorCyberDefenseEnv(net, B, seed=2, log_cap=LOG_CAP, detector_slots=B)
    step_ms, fit_ms, pending = [], [], []
    for t in range(200):
        ab = env.sample_actions(t & 1)
        step_ms.append(timed(lambda: env.step(ab)))
        if (t & 1) == 0:
            pending.append(int(((env.scalars[:, K.S_FLAGS] & K.FL_DET_PENDING) != 0).sum().item()))
            fit_ms.append(timed(lambda: env.fit_detectors(seeds)))
    torch.cuda.synchronize()
    res["closed_loop"] = {
        "turns": 200, "log_step_ms_median": float(np.median(step_ms[10:])),
        "log_step_ms_defender_median": float(np.median(step_ms[10::2])), "log_step_ms_attacker_median": float(np.median(step_ms[11::2])),
        "pending_per_defender_step": pending, "pending_mean": float(np.mean(pending)),
        "fit_ms_per_defender_step": fit_ms, "fit_ms_median": float(np.median(fit_ms[5:])),
        "mean_logs_at_end": float(env.scalars[:, K.S_LOGS].double().mean().item()),
        "detectors_fitted": int(env._next_slot.item()),
        "error_flags_any": bool(env.error_flags().any()),
        "error_detector_any": bool(((env.error_flags() & K.FL_ERR_DETECTOR) != 0).any()),
    }
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "closed_loop"} | {"closed_loop": {
        k: v for k, v in res["closed_loop"].items() if not isinstance(v, list)}}, indent=1))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "detector_fit_leg.json"))
