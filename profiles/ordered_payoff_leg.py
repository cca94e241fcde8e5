"""Payoff evaluation of DoubleOracle-style strategies -- fixed sequences drawn by sample_action with their device lists in
draw order (do_agent.py:1001-1013) -- at config-C5 shape: 32 x 32 strategy pairs x 1024 rollouts x 100 turns on one GPU
(2^20 envs).  Writes profiles/ordered_payoff_leg.json (or the path given as the last argument).

Strategies: 29 defender and 30 attacker sequences of 10 actions from VectorCyberDefenseEnv.sample_actions(want_order=True)
on the C3/C5 network, plus bench.py's baselines (No Defense, Preset, Nash / No Attack, Nash).  Two variants:
  train    the sampled defender type-10 actions kept, train_detectors=True
  map10    type 10 mapped to 8 (no-op), train_detectors=False
Per variant:
  a  evaluate_payoff_matrix_batched on the sequences as drawn (order-form rows: cyg_rollout_ordered)
  a_no_block_order   the same with the rollout's block_order left out (CTAs in index order): is _block_order's estimate,
                     which prices every row as the warp-per-env set form, worse than no ordering at all?
  b  the same sequences with every device list sorted, through the set-form path (cyg_rollout)
  c  evaluate_payoff_matrix, pair by pair, on SUBSET x SUBSET of the pairs (the full shape takes too long), and a on the
     same subset; c_full_estimate_seconds scales c by pairs
Timing: CUDA events around the whole call, after one warm-up call of the same shape; best and median of the samples.
"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cygym_b200 import payoff, synthetic_network  # noqa: E402
from cygym_b200.payoff import Strategy, evaluate_payoff_matrix, evaluate_payoff_matrix_batched  # noqa: E402
from cygym_b200.vector_env import ActionBatch, VectorCyberDefenseEnv  # noqa: E402

N5, T5, L, SUBSET, SAMPLES = 1024, 100, 10, 4, 3


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
    return a.elapsed_time(b) * 1e-3, r


def sampled(net, mode, n_seq, seed):
    """n_seq sequences of L actions, one env per action, as sample_action draws them (lists in draw order)."""
    env = VectorCyberDefenseEnv(net, n_seq * L, seed=seed)
    env.randomize_compromise_and_ownership()
    ab = env.sample_actions(mode, want_order=True)
    acts = ActionBatch.unpack(ab.hdr.cpu().numpy().view(np.uint32), ab.mask.cpu().numpy().view(np.uint32),
                              ab.order.cpu().numpy().view(np.uint16))
    env.close()
    return [acts[k * L:(k + 1) * L] for k in range(n_seq)]


def strategies(def_seqs, att_seqs, map10, sort):
    fix = lambda a: a if a is None else ((8 if (map10 and a[0] == 10) else a[0]), a[1], sorted(set(a[2])) if sort else a[2], a[3])
    defs = [Strategy(baseline_name="No Defense"), Strategy(baseline_name="Preset"), Strategy(baseline_name="Nash")] + \
           [Strategy(actions=[fix(a) for a in s]) for s in def_seqs]
    atts = [Strategy(baseline_name="No Attack"), Strategy(baseline_name="Nash")] + [Strategy(actions=[fix(a) for a in s]) for s in att_seqs]
    return defs, atts


def samples_of(fn, n=SAMPLES):
    fn()  # warm-up: allocation, module load
    ts, out = [], None
    for _ in range(n):
        t, out = timed(fn)
        ts.append(t)
    return {"seconds_best": min(ts), "seconds_median": float(np.median(ts)), "samples_seconds": ts}, out


def clear_cache():
    for k in list(payoff._ENV_CACHE):
        payoff._ENV_CACHE.pop(k).close()
    torch.cuda.empty_cache()


def variant(net, def_seqs, att_seqs, map10):
    train = not map10
    res = {}
    defs, atts = strategies(def_seqs, att_seqs, map10, sort=False)
    res["ordered_defender_rows"] = int(sum(a is not None and list(a[2]) != sorted(set(a[2])) for s in defs for a in (s.actions or ())))
    res["defender_rows"] = int(sum(len(s.actions or ()) for s in defs))
    res["training_defender_sequences"] = int(sum(s.can_train() for s in defs))
    batched = lambda d, a: evaluate_payoff_matrix_batched(net, d, a, N5, steps_per_episode=T5, seed=1, train_detectors=train)
    res["a"], out_a = samples_of(lambda: batched(defs, atts))
    (env,) = payoff._ENV_CACHE.values()
    l0 = env.launch_count
    batched(defs, atts)
    torch.cuda.synchronize()
    res["a"]["library_launches"] = env.launch_count - l0
    res["a"]["checksum"] = float(out_a.sum().item())
    del env
    orig = payoff._block_order
    payoff._block_order = lambda *args, **kw: None
    try:
        res["a_no_block_order"], out_n = samples_of(lambda: batched(defs, atts))
        res["a_no_block_order"]["equal_to_a"] = bool(torch.equal(out_n, out_a))
    finally:
        payoff._block_order = orig
    sdefs, satts = strategies(def_seqs, att_seqs, map10, sort=True)
    res["b"], out_b = samples_of(lambda: batched(sdefs, satts))
    res["b"]["checksum"] = float(out_b.sum().item())
    res["ratio_a_over_b"] = res["a"]["seconds_median"] / res["b"]["seconds_median"]
    clear_cache()
    # c: the pair-by-pair evaluator on a subset of pairs, and a on the same subset
    sd, sa = defs[3:3 + SUBSET], atts[2:2 + SUBSET]
    res["subset"] = f"defender sequences 0..{SUBSET - 1} x attacker sequences 0..{SUBSET - 1} ({SUBSET * SUBSET} pairs x {N5} rollouts x {T5} turns)"
    res["c_subset"], out_c = samples_of(lambda: evaluate_payoff_matrix(net, sd, sa, N5, steps_per_episode=T5, seed=1,
                                                                       train_detectors=train), n=2)
    res["a_subset"], out_as = samples_of(lambda: batched(sd, sa))
    res["a_subset"]["max_abs_diff_to_c"] = float((out_as - out_c).abs().max().item())
    res["speedup_c_over_a_subset"] = res["c_subset"]["seconds_median"] / res["a_subset"]["seconds_median"]
    res["c_full_estimate_seconds"] = res["c_subset"]["seconds_median"] * (len(defs) * len(atts)) / (SUBSET * SUBSET)
    res["speedup_c_full_estimate_over_a"] = res["c_full_estimate_seconds"] / res["a"]["seconds_median"]
    clear_cache()
    return res


def main(argv):
    out_path = argv[0] if argv else os.path.join(ROOT, "profiles", "ordered_payoff_leg.json")
    res = {"card": card(), "shape": f"32 x 32 strategies x {N5} rollouts x {T5} turns, sequences of {L} sampled actions"}
    net = synthetic_network(100, n_subnets=8, seed=0)
    def_seqs, att_seqs = sampled(net, 0, 29, 5), sampled(net, 1, 30, 6)
    res["map10"] = variant(net, def_seqs, att_seqs, map10=True)
    res["train"] = variant(net, def_seqs, att_seqs, map10=False)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main(sys.argv[1:])
