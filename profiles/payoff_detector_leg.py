"""Payoff evaluation with defender strategies that train the detector (train_detectors=True), at config-C5 shape: 32 x 32
strategy pairs x 1024 rollouts x 100 turns on one GPU (2^20 envs).  Writes profiles/payoff_detector_leg.json (or the
path given as the last argument):

  c5_plain          bench.py's C5 strategy set (same generator, same seed), train_detectors=False: seconds (CUDA events
                    around the whole call, warmed, best and median of 3) and the checksum, which must equal bench.py's
  c5_training       the same set with 4 of the 29 defender sequences rewritten to train (type 10) on one turn of their
                    cycle and scan (type 5) on two others, train_detectors=True: seconds, launches of the library,
                    fit_detectors() calls, CUDA-event time inside those calls, envs that end with an error bit
  fit_walk_ms       one fit_detectors() call with NO pending env (slot assignment walk + an empty fit launch), at
                    B = 2^20 and B = 4096, median of 20 after warm-up

--walk-only runs the last part alone with whatever cygym_b200 sits next to this file's directory, so the same file
copied into a built checkout of an older commit times that commit's assignment walk.  --parent DIR does that in the same
process run (DIR = such a checkout, with this file at DIR/profiles/) and records it as fit_walk_ms_parent.
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cygym_b200 import synthetic_network  # noqa: E402
from cygym_b200.vector_env import VectorCyberDefenseEnv  # noqa: E402

BENCH_C5_CHECKSUM = 245130.44076141246  # bench.py --gpus 1, legs.c5.checksum (profiles/r02_bench_line.json)
N_TRAINING = 4


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
    r = fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b), r


def fit_walk():
    """fit_detectors() with no env pending: what every training turn of an evaluation pays for the envs that did not train."""
    net = synthetic_network(100, n_subnets=8, seed=0)
    res = {}
    for B in (1 << 20, 4096):
        env = VectorCyberDefenseEnv(net, B, seed=1, detector_slots=1)
        seeds = torch.zeros(B, dtype=torch.int64, device="cuda")
        for _ in range(3):
            env.fit_detectors(seeds)
        ts = [timed(lambda: env.fit_detectors(seeds))[0] for _ in range(20)]
        assert env.pending_detectors() == [] and int(env._next_slot.item()) == 0
        res[str(B)] = {"median_ms": float(np.median(ts)), "min_ms": float(min(ts)), "all_ms": ts}
        del env
        torch.cuda.empty_cache()
    return res


def c5_strategies(training):
    """bench.py's C5 set: the same generator, seed and draw order.  training: the first N_TRAINING defender sequences
    train on action 0 of their 5-action cycle and scan on actions 2 and 4 (their device lists are kept)."""
    from cygym_b200.payoff import Strategy
    rng5 = np.random.default_rng(0)
    devices = 100

    def seq(mode, L):
        out = []
        for _ in range(L):
            n = int(rng5.integers(1, 40))
            devs = sorted(int(d) for d in rng5.choice(devices, size=n, replace=False))
            at = int(rng5.choice([1, 2, 3, 4, 5, 6, 7, 9, 11, 12, 13])) if mode == 0 else int(rng5.integers(1, 3))
            out.append((at, [int(rng5.integers(0, 2))], devs, int(rng5.integers(0, 7))))
        return out

    nS = 32
    def_seqs = [seq(0, 5) for _ in range(nS - 3)]
    att_seqs = [seq(1, 4) for _ in range(nS - 2)]
    if training:
        for s in def_seqs[:N_TRAINING]:
            s[0] = (10,) + tuple(s[0][1:])
            s[2] = (5,) + tuple(s[2][1:])
            s[4] = (5,) + tuple(s[4][1:])
    defs = [Strategy(baseline_name="No Defense"), Strategy(baseline_name="Preset"), Strategy(baseline_name="Nash")] + \
           [Strategy(actions=s) for s in def_seqs]
    atts = [Strategy(baseline_name="No Attack"), Strategy(baseline_name="Nash")] + [Strategy(actions=s) for s in att_seqs]
    return defs, atts


def c5_leg(net, training):
    from cygym_b200 import payoff
    from cygym_b200.payoff import evaluate_payoff_matrix_batched
    defs, atts = c5_strategies(training)
    N5, T5 = 1024, 100
    fit_events = []
    orig_fit = VectorCyberDefenseEnv.fit_detectors

    def counted_fit(self, seeds):  # CUDA events around every fit_detectors() call of the evaluator
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        orig_fit(self, seeds)
        b.record()
        fit_events.append((a, b))

    VectorCyberDefenseEnv.fit_detectors = counted_fit
    try:
        run = lambda: evaluate_payoff_matrix_batched(net, defs, atts, N5, steps_per_episode=T5, seed=1, device="cuda:0",
                                                     train_detectors=training)
        run()  # the first evaluation of the shape: allocation, module load
        samples, launches, fits, fit_ms = [], [], [], []
        for _ in range(3):
            fit_events.clear()
            (env,) = payoff._ENV_CACHE.values()
            l0 = env.launch_count
            ms, out = timed(run)
            (env,) = payoff._ENV_CACHE.values()
            samples.append(ms * 1e-3)
            launches.append(env.launch_count - l0)
            fits.append(len(fit_events))
            fit_ms.append(sum(a.elapsed_time(b) for a, b in fit_events))
        err = env.error_flags()
        res = {"seconds_best": min(samples), "seconds_median": float(np.median(samples)), "samples_seconds": samples,
               "checksum": float(out.sum().item()), "library_launches": launches[-1], "fit_detectors_calls": fits[-1],
               "fit_detectors_ms_total": float(np.median(fit_ms)), "fit_detectors_ms_samples": fit_ms,
               "envs_with_error_bit": int((err != 0).sum().item()), "log_cap": env.log_cap,
               "detector_slots": 0 if env._det_slots is None else int(env._det_slots.shape[0]),
               "detectors_fitted": 0 if env._next_slot is None else int(env._next_slot.item())}
        del env
    finally:
        VectorCyberDefenseEnv.fit_detectors = orig_fit
        for k in list(payoff._ENV_CACHE):
            payoff._ENV_CACHE.pop(k).close()
        torch.cuda.empty_cache()
    return res


def parent_walk(parent_dir):
    """fit_walk() of the checkout at parent_dir, in a process of its own (its own cygym_b200 and library)."""
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "walk.json")
        subprocess.run([sys.executable, os.path.join(parent_dir, "profiles", "payoff_detector_leg.py"), "--walk-only", out], check=True)
        with open(out) as f:
            return json.load(f)["fit_walk_ms"]


def main(argv):
    walk_only = "--walk-only" in argv
    parent = argv[argv.index("--parent") + 1] if "--parent" in argv else None
    args = [a for i, a in enumerate(argv) if not a.startswith("--") and not (i > 0 and argv[i - 1] == "--parent")]
    out_path = args[0] if args else os.path.join(ROOT, "profiles", "payoff_detector_leg.json")
    res = {"card": card()}
    if not walk_only:
        net = synthetic_network(100, n_subnets=8, seed=0)
        res["c5_plain"] = c5_leg(net, False)
        res["c5_plain"]["checksum_equals_bench"] = res["c5_plain"]["checksum"] == BENCH_C5_CHECKSUM
        res["c5_training"] = c5_leg(net, True)
        res["c5_training"]["training_defender_sequences"] = N_TRAINING
    res["fit_walk_ms"] = fit_walk()
    if parent:
        res["fit_walk_ms_parent"] = parent_walk(parent)
        res["fit_walk_ms_parent"]["what"] = "the same measurement with the parent commit's library: one CTA walks every env"
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main(sys.argv[1:])
