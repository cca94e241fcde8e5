#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused CyGym step kernel on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun)
    python bench.py --impl reference --steps K --warmup W    # the CPU arm (oracle port on the host cores)

Workload (config.workload "C3"): 65 536 envs x 100 device slots / 8 subnets per GPU, synthetic network
(cygym_b200.network.synthetic_network), uniformly random sample_action()-style defender / attacker
actions on alternating turns, detector untrained (defender action 10 rewritten to the no-op 8).
A "step" is ONE pass of cyg_step over one batch of B envs.  Envs shard across GPUs with no
data-path collective (weak scaling: B envs per GPU); NCCL only carries the timing reduction.

L2 policy: the C3 legs rotate over `--sets` independent env sets (default 3 x 59 MB of state
> 126 MB L2) and a ring of pre-generated action batches, so a launch never finds its records
in L2 from the previous launch.  The small-state legs (C2, C4) write a 256 MB buffer between
launches and are timed per launch with CUDA events.

One JSON line.  Besides the contract keys it carries `single_step_launch` (the same workload at
one launch per step) and `legs`: the same kernel on the other shapes callers use --
`randomized` (after randomize_compromise_and_ownership: every Double-Oracle rollout), `obs_on`
(observation rows materialised every step), `grouped` (13-group step_grouped: the IPPO / MAPPO
rollout shape), `c2` (4096 x 50) and `c4` (1024 x 2000) -- each with its own roofline fraction
(at N = 1 only: they are diagnostics of the kernel, not scaling points).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec at 64K envs x 100 devices"
UNIT = "env-steps/s"
PREHEAT = 64  # untimed launches before every timed region, whatever --warmup says: allocator, clocks, L2 and the env states (an episode a few hundred steps in steps differently from a fresh one) are then those of a long run


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000, help="timed steps of the headline workload (a fused run's last launch takes the remainder)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--devices", type=int, default=100)
    ap.add_argument("--subnets", type=int, default=8)
    ap.add_argument("--sets", type=int, default=3, help="independent env sets rotated to defeat L2 residency")
    ap.add_argument("--ring", type=int, default=8, help="pre-generated action batches per mode")
    ap.add_argument("--fuse", type=int, default=4, help="plain steps fused per launch (VectorCyberDefenseEnv.step_many / cyg_step_multi); 1 = one launch per step")
    ap.add_argument("--randomize", action="store_true", help="headline on envs after randomize_compromise_and_ownership() (the `randomized` leg as the main line)")
    ap.add_argument("--obs", type=int, default=0, help="fused observation mode inside the step (0 none, 1 defender, 2 attacker)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--e2e-groups", type=int, default=5, help="env groups (of --envs envs each, one stream each, every one closed-loop) the e2e leg keeps in flight")
    ap.add_argument("--e2e-steps", type=int, default=240, help="host-buffer steps of the e2e leg (fixed: the leg is host / PCIe paced and noisy when short)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-legs", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed headline step returned as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


def workload_name(a):
    return f"C3: {a.envs} envs x {a.devices} device slots / {a.subnets} subnets per GPU, random sample_action defender/attacker turns"


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons DURING the timed region.  The timed region is tens of milliseconds, so the
    sampler polls NVML in-process every ~2 ms (nvidia-smi, the B200_PROFILING.md clocks line, is the fallback)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.sm, self.max_sm, self.reasons, self.how = [], 0.0, set(), "nvml"
        self._stop_evt = threading.Event()
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[gpu_index])
                                                        if os.environ.get("CUDA_VISIBLE_DEVICES") else gpu_index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None
            self.how = "nvidia-smi"

    def _poll_nvml(self):
        n = self._nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)

    def _poll_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            s = [x.strip() for x in out.split(",")]
            self.sm.append(float(s[1]))
            self.max_sm = max(self.max_sm, float(s[2]))
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def run(self):
        while not self._stop_evt.is_set():
            try:
                self._poll_nvml() if self._nvml else self._poll_smi()
            except Exception:
                pass
            self._stop_evt.wait(0.002 if self._nvml else 0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm or None, "reasons": sorted(self.reasons),
                "samples": len(sm), "how": self.how}


def cpu_arm(a, seconds, threads=None):
    """The oracle port (oracle/cyg_oracle.c, OpenMP over envs) timed on the host cores on a bounded
    sample of the same workload.  The thread count is passed explicitly (the `num_threads` clause of cyo_step), so
    torchrun's OMP_NUM_THREADS=1 does not collapse the arm.  Returns (env-steps/s, cores, description)."""
    import numpy as np
    from cygym_b200 import synthetic_network
    from tests.common import oracle_for, oracle_state_from_template, sanitize_actions
    net = synthetic_network(a.devices, n_subnets=a.subnets, seed=a.seed)
    cores = max(1, int(threads or host_cores()))
    Bc = max(cores * 256, 1024)
    orc, _ = oracle_for(net, seed=a.seed, xcap=16)
    st = oracle_state_from_template(orc, net, Bc)
    acts = []
    for mode in (0, 1):
        h, m = orc.sample_actions(st, mode)
        h = sanitize_actions(h, np.ones(Bc, np.uint32), mode)
        acts.append((h, m))
    for t in range(4):
        orc.step(st, *acts[t & 1], n_threads=cores)
    n, t0 = 0, time.perf_counter()
    while True:
        orc.step(st, *acts[n & 1], n_threads=cores)
        n += 1
        el = time.perf_counter() - t0
        if el >= seconds or n >= 100000:
            break
    return Bc * n / el, cores, f"{Bc} envs x {n} steps of the same workload, {cores} OpenMP threads (explicit), {el:.1f}s", net


def reference_python_record():
    """The unmodified reference's own Python step() timed in the BUILD container (oracle/time_reference.py): the
    reference cannot travel to the GPU box, so this is a committed record with its host stated, not a live number."""
    try:
        with open(os.path.join(ROOT, "profiles", "reference_python_steps.json")) as f:
            r = json.load(f)
        r["note"] = "measured in the build container by oracle/time_reference.py, not on this box"
        return r
    except Exception:
        return None


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    per_step = max(0.5, min(20.0, 120.0 / max(1, a.steps + a.warmup)))
    # each "step" of this arm is one bounded CPU sample
    vals = []
    for i in range(a.warmup + a.steps):
        v, cores, sample, net = cpu_arm(a, per_step)
        if i >= a.warmup:
            vals.append(v)
    val = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": workload_name(a), "envs_per_gpu": a.envs, "device_slots": a.devices, "edges": int(net.E),
                   "l2_policy": "n/a (CPU arm)", "sampled_envs": int(sample.split()[0])},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample + f" per step, {a.steps} steps",
                         "reference_python": reference_python_record()},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def latest_profile(pattern):
    """Newest committed profiles/rNN_<pattern> (the ncu-derived per-launch DRAM traffic of the current kernels)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r[0-9][0-9]_" + pattern)))
    return files[-1] if files else None


DUMP_BYTES = 60 << 20  # --dump-outputs stays below 64 MB, .npy headers included


def dump_outputs(out_dir, arrays):
    """Write every [B, ...] device tensor of `arrays` as out_dir/<name>.npy in float32.  Above DUMP_BYTES in all, the
    same fixed, seeded sample of envs is taken from every array and its env indices go to env_index.npy (float64)."""
    import numpy as np
    arrays = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    B = len(next(iter(arrays.values())))
    per_env = sum(v[0].nbytes for v in arrays.values())
    if B * per_env > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // (per_env + 8), replace=False))
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    import numpy as np
    import torch
    import torch.distributed as dist
    from cygym_b200 import marl, synthetic_network
    from cygym_b200.vector_env import ActionBatch, VectorCyberDefenseEnv

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, Wm = a.envs, a.steps, max(3, a.warmup)

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, warm, counters=()):
        """W warm-up calls (+ the fixed pre-heat), then n calls between two CUDA events on the current stream."""
        for i in range(max(warm, PREHEAT)):
            fn(i)
        barrier()
        l0 = sum(s.launch_count for s in counters)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for i in range(n):
            fn(max(warm, PREHEAT) + i)
        ev1.record()
        barrier()
        return ev0.elapsed_time(ev1), sum(s.launch_count for s in counters) - l0

    flush_buf = None

    def timed_flushed(fn, n, warm):
        """Small-state legs: a 256 MB write between launches evicts the state from L2; every launch has its own pair of
        CUDA events (the flush is outside them).  Returns the summed launch time in ms."""
        nonlocal flush_buf
        if flush_buf is None:
            flush_buf = torch.empty(64 * 1024 * 1024, dtype=torch.int32, device=dev)
        for i in range(max(warm, PREHEAT)):
            fn(i)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        torch.cuda.synchronize()
        for i in range(n):
            flush_buf.fill_(i)
            evs[i][0].record()
            fn(max(warm, PREHEAT) + i)
            evs[i][1].record()
        torch.cuda.synchronize()
        return sum(e0.elapsed_time(e1) for e0, e1 in evs)

    def make_sets(net, nB, n_sets, randomize, id_base=0, xcap=16):
        sets = [VectorCyberDefenseEnv(net, nB, device=dev, seed=a.seed, env_id0=id_base + (rank * n_sets + s) * nB, xcap=xcap)
                for s in range(n_sets)]
        if randomize:
            for s_ in sets:
                s_.randomize_compromise_and_ownership()
        return sets

    def make_ring(sets, n_ring):
        """Pre-generated sample_action batches (inputs resident in HBM before any timed region)."""
        ring = {0: [], 1: []}
        for mode in (0, 1):
            for r in range(n_ring):
                ab = sets[r % len(sets)].sample_actions(mode)
                if mode == 0:  # detector untrained: defender 10 -> no-op 8
                    ab.hdr[:, 0] = torch.where((ab.hdr[:, 0] & 0xFF) == 10, (ab.hdr[:, 0] & ~0xFF) | 8, ab.hdr[:, 0])
                for spec in filter(None, os.environ.get('CYG_BENCH_EXCLUDE', '').split(',')):  # diagnostics only
                    m_, t_ = spec.split(':')
                    if int(m_) == mode:
                        ab.hdr[:, 0] = torch.where((ab.hdr[:, 0] & 0xFF) == int(t_), (ab.hdr[:, 0] & ~0xFF) | (8 if mode == 0 else 3), ab.hdr[:, 0])
                ring[mode].append(ActionBatch(ab.hdr.clone(), ab.mask.clone()))
        torch.cuda.synchronize()
        return ring

    def plain_legs(net, sets, ring, n_steps, fuse, obs=0, flushed=False, keep_last=False):
        """Fused (`fuse` plain steps per launch) and one-launch-per-step timings of alternating defender / attacker turns
        over the rotating env sets, n_steps steps each.  Returns dict(ms_fused, steps_fused, launches, ms_single, steps_single);
        keep_last adds `last`: copies of what the last step of the first timed region (fused if fuse > 1) returned."""
        nB, n_sets, n_ring = sets[0].B, len(sets), len(ring[0])

        def one_step(i):
            env = sets[i % n_sets]
            turn = (i // n_sets) & 1  # every set alternates defender / attacker turns
            om = 0 if not obs else (1 + turn)  # the view the turn's player reads (defender 6M / attacker 4M+X)
            env.step(ring[turn][(i // (2 * n_sets)) % n_ring], obs_mode=om)

        out = {}
        F = max(1, fuse) if not obs else 1
        if F > 1:
            n_launch = (n_steps + F - 1) // F  # the last launch of a timed region fuses the remaining n_steps - (n_launch - 1) * F
            w_f = (Wm + F - 1) // F
            p0 = max(w_f, PREHEAT)  # index of the first timed launch: timed() and timed_flushed() pre-heat with launches 0 .. p0 - 1
            fused = []
            for s_i in range(n_sets):
                per_set = []
                for v in range(2):  # two variants per set so that consecutive launches of a set read different batches
                    hs = [ring[t & 1][(s_i + v * 3 + t // 2) % n_ring].hdr for t in range(F)]
                    mk = [ring[t & 1][(s_i + v * 3 + t // 2) % n_ring].mask for t in range(F)]
                    per_set.append((torch.stack(hs).contiguous(), torch.stack(mk).contiguous()))
                fused.append(per_set)
            outs = [(torch.empty(F, nB, dtype=torch.float32, device=dev), torch.empty(F, nB, dtype=torch.float32, device=dev),
                     torch.empty(F, nB, dtype=torch.int32, device=dev)) for _ in range(n_sets)]
            torch.cuda.synchronize()

            def one_launch(j, T=F):
                s_i = j % n_sets
                h_, m_ = fused[s_i][(j // n_sets) & 1]
                o_ = outs[s_i]
                if T < F:
                    h_, m_, o_ = h_[:T], m_[:T], tuple(x[:T] for x in o_)
                sets[s_i].step_many(h_, m_, out=o_)

            def timed_launch(j):
                one_launch(j, min(F, n_steps - (j - p0) * F))

            if flushed:
                out["ms_fused"], out["launches"] = timed_flushed(timed_launch, n_launch, w_f), n_launch
            else:
                out["ms_fused"], out["launches"] = timed(timed_launch, n_launch, w_f, sets)
            out["steps_fused"] = n_steps
            if keep_last:
                T_last = n_steps - (n_launch - 1) * F
                out["last"] = [x[T_last - 1].clone() for x in outs[(p0 + n_launch - 1) % n_sets]]
        K1 = n_steps
        if flushed:
            out["ms_single"] = timed_flushed(one_step, K1, Wm)
        else:
            out["ms_single"], l1 = timed(one_step, K1, Wm, sets)
            if F == 1:
                out["launches"] = l1
        out["steps_single"] = K1
        if keep_last and F == 1:
            i = max(Wm, PREHEAT) + K1 - 1  # the last timed step (see one_step)
            env = sets[i % n_sets]
            out["last"] = [x.clone() for x in (env.raw, env.shaped, env.done)]
            if obs:
                out["last"].append(env.last_obs(1 + ((i // n_sets) & 1)).clone())
        if not flushed and not obs and n_sets > 1:
            # the same one-launch-per-step workload with every env set on its OWN stream (each set still steps in order:
            # closed loop per set): a launch's CTAs move onto SMs as the previous launch's CTAs leave them, so the
            # slowest-CTA tail and the load / store phases of one set overlap the compute of another
            streams = [torch.cuda.Stream(dev) for _ in range(n_sets)]
            cur = torch.cuda.current_stream(dev)

            def one_step_streams(i):
                s_i = i % n_sets
                streams[s_i].wait_stream(cur) if i < n_sets else None
                with torch.cuda.stream(streams[s_i]):
                    one_step(i)

            def run(n):
                for i in range(n):
                    one_step_streams(i)
                for st_ in streams:
                    cur.wait_stream(st_)

            run(max(Wm, PREHEAT))
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(K1)
            e1.record()
            barrier()
            out["ms_single_streams"] = e0.elapsed_time(e1)
            if F > 1:  # and the fused launches the same way (each set's launches in order on its own stream)
                def run_f(n, total=None):  # n launches; with `total`, exactly `total` steps
                    for j in range(n):
                        s_i = j % n_sets
                        if j < n_sets:
                            streams[s_i].wait_stream(cur)
                        with torch.cuda.stream(streams[s_i]):
                            one_launch(j, F if total is None else min(F, total - j * F))
                    for st_ in streams:
                        cur.wait_stream(st_)
                run_f(p0)
                barrier()
                e0.record()
                run_f(n_launch, n_steps)
                e1.record()
                barrier()
                out["ms_fused_streams"] = e0.elapsed_time(e1)
        return out

    def leg_record(net, nB, r, fuse, obs=False, extra=None):
        alg = net.algorithmic_bytes_per_step(obs=obs)
        d = {"envs": nB, "device_slots": net.M, "edges": int(net.E), "algorithmic_bytes_per_env_step": alg}
        if "ms_fused" in r:
            us = r["ms_fused"] * 1e3 / r["steps_fused"]
            d["fused"] = {"steps_per_launch": fuse, "us_per_step": us, "value": world * nB / (us * 1e-6), "unit": UNIT,
                          "roofline": {"bound": "hbm", "achieved": alg * nB / (us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                                       "frac": alg * nB / (us * 1e-6) / 1e9 / peak}}
        if "ms_fused_streams" in r:
            usf = r["ms_fused_streams"] * 1e3 / r["steps_fused"]
            d["fused_on_streams"] = {"us_per_step": usf, "value": world * nB / (usf * 1e-6), "unit": UNIT, "streams": "one per env set",
                                     "roofline": {"bound": "hbm", "achieved": alg * nB / (usf * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                                                  "frac": alg * nB / (usf * 1e-6) / 1e9 / peak}}
        us1 = r["ms_single"] * 1e3 / r["steps_single"]
        if "ms_single_streams" in r:
            uss = r["ms_single_streams"] * 1e3 / r["steps_single"]
            d["single_on_streams"] = {"us_per_step": uss, "value": world * nB / (uss * 1e-6), "unit": UNIT, "streams": "one per env set",
                                      "roofline": {"bound": "hbm", "achieved": alg * nB / (uss * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                                                   "frac": alg * nB / (uss * 1e-6) / 1e9 / peak}}
        d["single"] = {"launch_us": us1, "value": world * nB / (us1 * 1e-6), "unit": UNIT,
                       "roofline": {"bound": "hbm", "achieved": alg * nB / (us1 * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": alg * nB / (us1 * 1e-6) / 1e9 / peak}}
        if extra:
            d.update(extra)
        return d

    # ================= the headline: C3 =================
    net = synthetic_network(a.devices, n_subnets=a.subnets, seed=a.seed)
    sets = make_sets(net, B, a.sets, a.randomize)
    ring = make_ring(sets, a.ring)
    F = max(1, a.fuse) if not a.obs else 1
    sampler = ClockSampler(local)
    sampler.start()
    head = plain_legs(net, sets, ring, K, F, obs=a.obs, keep_last=bool(a.dump_outputs))
    clocks = sampler.stop()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, dict(zip(("raw_reward", "shaped_reward", "done", "obs"), head.pop("last"))))
    if F > 1:
        ms, Kh, launches = head["ms_fused"], head["steps_fused"], head["launches"]
    else:
        ms, Kh, launches = head["ms_single"], head["steps_single"], head["launches"]
    ms1, K1 = head["ms_single"], head["steps_single"]
    errs = int(max(int(s.error_flags().max().item()) for s in sets))
    rec_words, n_env_sets_bytes = sets[0].S, a.sets * B * (sets[0].S + net.M) * 4

    # ---- e2e: the public host-buffer call VectorCyberDefenseEnv.step_host(): every step copies that step's actions
    #      from pinned host memory, launches the kernel, reads (raw, shaped, done) back and synchronises ----
    e2e = None
    if not a.no_e2e:
        from cygym_b200.vector_env import compact_action_rows
        Ke = max(200, a.e2e_steps)
        # env groups in flight: the env sets of the rotation plus extra ones, every group closed-loop on its own stream.  One
        # group's step is a ~130 us chain (H2D, expand, kernel, D2H, the host's wake-up and next launch); three groups leave
        # the copy engines and the SMs idle part of the time, five keep them busy (profiles/NOTES_r02.md)
        n_groups = max(1, a.e2e_groups)
        groups = list(sets[:n_groups])
        if len(groups) < n_groups:
            groups += make_sets(net, B, n_groups - len(groups), a.randomize, id_base=(world * a.sets + 7) * B)
        host_actions = {}
        for gi, env in enumerate(groups):
            env._stream = torch.cuda.Stream(dev)  # one stream per env group
            env.host_buffers()
            for mode in (0, 1):
                ab = ring[mode][gi % len(ring[mode])]
                # [B, 2 + W] compact rows (include/cygym_b200.h: a 2-word header + the device mask, 24 bytes per env at W = 4)
                host_actions[gi, mode] = torch.from_numpy(compact_action_rows(ab.hdr.cpu(), ab.mask.cpu())).pin_memory()
        torch.cuda.synchronize()

        def run_e2e(n_groups, steps):
            """steps host-buffer steps over n_groups env groups (round robin).  Every step: wait for that group's
            previous results (the caller reads them before it chooses the group's next action), then enqueue H2D of the
            step's actions, the kernel and the D2H of (raw, shaped, done)."""
            turn = [0] * n_groups
            for g in range(n_groups):
                groups[g].wait_host()
            barrier()
            t0 = torch.cuda.Event(enable_timing=True)
            t1 = torch.cuda.Event(enable_timing=True)
            t0.record()
            for i in range(steps):
                g = i % n_groups
                env = groups[g]
                env.wait_host()
                env.step_host(act=host_actions[g, turn[g] & 1], sync=False, packed_done=True)
                turn[g] += 1
            for g in range(n_groups):
                groups[g].wait_host()
            t1.record()
            barrier()
            return t0.elapsed_time(t1)

        # the loop is host-driven (one graph launch + one event wait per step): the collector is kept out of the timed
        # regions, and the leg is sampled five times -- the MEDIAN is reported, all samples are listed
        import gc
        gc.collect()
        gc.disable()
        try:
            run_e2e(len(groups), max(len(groups) * PREHEAT, 120))
            e2e_samples = [run_e2e(len(groups), Ke) for _ in range(5)]
            run_e2e(1, PREHEAT)
            ems1 = run_e2e(1, Ke // 2)
        finally:
            gc.enable()
        if world > 1:  # every rank must pick the same sample: max over ranks per sample, then the median
            t_s = torch.tensor(e2e_samples, dtype=torch.float64, device=dev)
            dist.all_reduce(t_s, op=dist.ReduceOp.MAX)
            e2e_samples = [float(x) for x in t_s]
        ems = sorted(e2e_samples)[len(e2e_samples) // 2]
        e2e = (ems, Ke, host_actions[0, 0].numel() * 4, groups[0].host_result_bytes(True), ems1, Ke // 2, len(groups), e2e_samples)
        for env in groups:
            env._stream = None
        torch.cuda.synchronize()
        for env in groups[len(sets):]:
            env.close()
        del groups[len(sets):]

    # ================= the other shapes (N = 1: kernel diagnostics, not scaling points) =================
    legs = {}
    if world == 1 and not a.no_legs and not a.obs:
        Kl = min(K, 240)
        # (1) randomized ownership: what every Double-Oracle rollout steps (do_agent.py:2032: randomize first)
        if not a.randomize:
            rsets = make_sets(net, B, a.sets, True, id_base=10 * B * a.sets)
            rring = make_ring(rsets, a.ring)
            legs["randomized"] = leg_record(net, B, plain_legs(net, rsets, rring, Kl, F), F, extra={
                "what": "the headline workload after randomize_compromise_and_ownership() on every env (the owned set moves, "
                        "evolve_network adds extra hub-star edges): the state every Double-Oracle rollout steps"})
            del rsets, rring
        # (2) observations materialised every step (the view the turn's player reads)
        legs["obs_on"] = leg_record(net, B, plain_legs(net, sets, ring, Kl, 1, obs=1), 1, obs=True, extra={
            "what": "one launch per step with the fused observation epilogue: _get_defender_state (6M fp32) on defender turns, "
                    "_get_attacker_state (4M+X) on attacker turns; algorithmic bytes = SURVEY 8(d) with OBS"})
        # (3) the IPPO / MAPPO rollout shape: per-device action types -> 13 groups -> step_grouped (IPPO.py:559-573)
        genv = sets[0]
        gen = torch.Generator(device=dev)
        gen.manual_seed(1234 + a.seed)
        types = [torch.randint(0, 14, (B, net.M), device=dev, generator=gen, dtype=torch.int32) for _ in range(4)]
        exp_idx = torch.zeros(B, dtype=torch.int32, device=dev)
        app_idx = torch.zeros(B, dtype=torch.int32, device=dev)
        for t_ in types:  # sklearn's branch stays out: per-device type 10 (train detector) -> 8
            t_[t_ == 10] = 8
        pre = [marl.grouped_actions_from_types(genv, t_, marl.visibility_mask(genv, "defender"), exp_idx, app_idx, "defender", 14, 8)
               for t_ in types]
        ms_g = timed(lambda i: sets[i % a.sets].step_grouped(pre[i % 4]), Kl, Wm, sets)[0]

        gouts = [None] * a.sets

        def glue_and_step(i):
            env = sets[i % a.sets]
            gouts[i % a.sets] = marl.grouped_actions(env, types[i % 4], "defender", exp_idx, app_idx, "defender", 14, 8, out=gouts[i % a.sets])
            env.step_grouped(gouts[i % a.sets])

        ms_gg = timed(glue_and_step, Kl, Wm, sets)[0]
        alg_g = net.algorithmic_bytes_per_step() + 12 * (4 + (net.M + 7) // 8)  # 13 action groups instead of one
        us_g, us_gg = ms_g * 1e3 / Kl, ms_gg * 1e3 / Kl
        legs["grouped"] = {
            "what": "step_grouped with the 13 per-type groups of IPPO.py:559-570 (every device draws a type, the VISIBLE devices -- build_visibility_mask, "
                    "IPPO.py:74-96 -- are grouped by type), "
                    "defender turns; `single` = the grouped step alone on pre-built groups, `with_glue` = + visibility mask and "
                    "group encoding (cygym_b200.marl) as torch ops per step",
            "envs": B, "device_slots": net.M, "groups": 13, "algorithmic_bytes_per_env_step": alg_g,
            "single": {"launch_us": us_g, "value": B / (us_g * 1e-6), "unit": UNIT,
                       "roofline": {"bound": "hbm", "achieved": alg_g * B / (us_g * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": alg_g * B / (us_g * 1e-6) / 1e9 / peak}},
            "with_glue": {"us_per_step": us_gg, "value": B / (us_gg * 1e-6), "unit": UNIT}}
        del pre, types
        # (4) C2: 4096 envs x 50 device slots / 3 subnets (BASELINE.json configs[1])
        net2 = synthetic_network(50, n_subnets=3, seed=a.seed)
        s2 = make_sets(net2, 4096, 2, False, id_base=20 * B * a.sets)
        legs["c2"] = leg_record(net2, 4096, plain_legs(net2, s2, make_ring(s2, 4), Kl, F, flushed=True), F, extra={
            "what": "C2: 4096 envs x 50 device slots / 3 subnets; 2 MB of state: a 256 MB write between launches evicts it from L2, "
                    "per-launch CUDA events; 4096 envs fill 128 of the 148 SMs with one 32-env CTA each"})
        del s2
        # (5) C4: 1024 envs x 2000 device slots / 64 subnets (BASELINE.json configs[3])
        net4 = synthetic_network(2000, n_subnets=64, seed=a.seed)
        s4 = make_sets(net4, 1024, 1, False, id_base=30 * B * a.sets, xcap=512)  # a hub change re-stars ~100 owned devices
        legs["c4"] = leg_record(net4, 1024, plain_legs(net4, s4, make_ring(s4, 2), min(Kl, 60), 1, flushed=True), 1, extra={
            "what": "C4: 1024 envs x 2000 device slots / 64 subnets (the adjacency matrix exceeds shared memory); 256 MB write "
                    "between launches, per-launch CUDA events"})
        legs["c4"]["error_flags"] = int(s4[0].error_flags().max().item())
        errs = max(errs, legs["c4"]["error_flags"])
        del s4

    if world == 1 and not a.no_legs and not a.obs:
        # (6) C1: ONE env behind the reference's Gym surface (init_experiments.py defaults: numOfDevice 10, Max_network_size 20),
        #     sample_action() + step() on alternating turns: host-side latency per step, wall clock
        from cygym_b200.volt_typhoon_env import Volt_Typhoon_CyberDefenseEnv
        genv1 = Volt_Typhoon_CyberDefenseEnv(device=dev, seed=a.seed)
        genv1.numOfDevice, genv1.Max_network_size = 10, 20
        genv1.initialize_environment()

        def gym_steps(n, policy):
            for t in range(n):
                genv1.mode = "defender" if t % 2 == 0 else "attacker"
                if policy == "sample":
                    act = genv1.sample_action()
                    act = (8 if genv1.mode == "defender" and act[0] == 10 else act[0], act[1], act[2], act[3])
                else:
                    act = None
                genv1.step(act)

        res = {}
        for policy in ("sample", "none"):
            gym_steps(30, policy)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            gym_steps(300, policy)
            torch.cuda.synchronize()
            res[policy] = 300 / (time.perf_counter() - t0)
        refpy = (reference_python_record() or {}).get("sizes", {}).get("20", {})
        legs["c1"] = {"what": "C1: one env through the drop-in Volt_Typhoon_CyberDefenseEnv (batch of 1; every step = action packing, "
                              "H2D, one kernel, one D2H of rewards + pre-evolve masks + the 6-tuple), wall clock on the host",
                      "steps_per_s_sample_action_plus_step": res["sample"], "steps_per_s_step_only_none_action": res["none"],
                      "reference_python_steps_per_s_1_core": refpy.get("steps_per_s_1_core"),
                      "note": "a single 20-device env is launch- and PCIe-latency bound on a GPU; the reference's pure-Python step is "
                              "the faster one at this size -- the batched VectorCyberDefenseEnv is the product"}

    # ================= C5: the payoff-matrix evaluation, sharded over the ranks + ONE all-reduce =================
    c5 = None
    if not a.no_legs and not a.obs:
        from cygym_b200.payoff import Strategy, evaluate_payoff_matrix_batched
        rng5 = np.random.default_rng(0)

        def seq(mode, L):
            out = []
            for _ in range(L):
                n = int(rng5.integers(1, 40))
                devs = sorted(int(d) for d in rng5.choice(a.devices, size=n, replace=False))
                at = int(rng5.choice([1, 2, 3, 4, 5, 6, 7, 9, 11, 12, 13])) if mode == 0 else int(rng5.integers(1, 3))
                out.append((at, [int(rng5.integers(0, 2))], devs, int(rng5.integers(0, 7))))
            return out

        nS, N5, T5 = 32, 1024, 100
        defs = [Strategy(baseline_name="No Defense"), Strategy(baseline_name="Preset"), Strategy(baseline_name="Nash")] + \
               [Strategy(actions=seq(0, 5)) for _ in range(nS - 3)]
        atts = [Strategy(baseline_name="No Attack"), Strategy(baseline_name="Nash")] + [Strategy(actions=seq(1, 4)) for _ in range(nS - 2)]
        del sets, ring  # the evaluation allocates its own envs (1 M at N = 1)
        torch.cuda.empty_cache()
        # one untimed evaluation of the full size first: CUDA module load, allocator growth, NCCL's first all-reduce
        evaluate_payoff_matrix_batched(net, defs, atts, N5, steps_per_episode=T5, seed=1, device=dev, rank=rank, world=world)
        barrier()
        samples = []
        for _ in range(3):  # the evaluation is host-driven (a dozen launches and copies): three samples, the best one is reported
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            t0 = time.perf_counter()
            ev0.record()
            out5 = evaluate_payoff_matrix_batched(net, defs, atts, N5, steps_per_episode=T5, seed=1, device=dev, rank=rank, world=world)
            ev1.record()
            barrier()
            wall = time.perf_counter() - t0
            t5 = torch.tensor([ev0.elapsed_time(ev1), wall * 1e3], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t5, op=dist.ReduceOp.MAX)
            samples.append((float(t5[0]), float(t5[1])))
        t5 = min(samples)
        c5 = {"what": f"C5: DOAR payoff-matrix evaluation, {nS}x{nS} strategy pairs x {N5} rollouts x {T5} turns (baseline names + fixed "
                      "sequences), the (pair, rollout) index sharded over the ranks, per-pair action tables gathered inside ONE cyg_rollout "
                      "launch per rank, then ONE all-reduce(SUM) of the [32, 32, 10] sums (NCCL)",
              "n_gpus": world, "seconds": float(t5[0]) * 1e-3, "wall_seconds": float(t5[1]) * 1e-3, "samples_seconds": [x[0] * 1e-3 for x in samples],
              "env_steps_per_s": nS * nS * N5 * T5 / (float(t5[0]) * 1e-3), "checksum": float(out5.sum().item()),
              "collective": "all_reduce(SUM) of 10 240 float64 (NCCL)" if world > 1 else "none (1 rank)"}

    # ---- max over ranks ----
    t = torch.tensor([ms, e2e[0] if e2e else 0.0, e2e[4] if e2e else 0.0, ms1], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ems, ems1, ms1 = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    if rank == 0:
        alg = net.algorithmic_bytes_per_step(obs=bool(a.obs))

        def traffic_of(pattern, **match):
            p_ = latest_profile(pattern)
            try:
                with open(p_) as f:
                    tj = json.load(f)
                if all(tj.get(k) == v for k, v in match.items()) and not a.obs and not a.randomize:
                    return tj["dram_bytes_per_launch"], os.path.basename(p_)
            except Exception:
                pass
            return None, None
        traffic, traffic_src = traffic_of("step_kernel_traffic.json", envs_per_launch=B, device_slots=a.devices)
        traffic_f, traffic_f_src = traffic_of("step_kernel_fused_traffic.json", envs_per_launch=B, device_slots=a.devices, steps_per_launch=F)
        launch_s = ms * 1e-3 * F / Kh         # average duration of F steps (one launch)
        achieved = alg * B * F / launch_s / 1e9
        value = world * B * Kh / (ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": Kh, "warmup": Wm,
            "ms_per_step": ms / Kh, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(a), "envs_per_gpu": B, "device_slots": a.devices, "edges": net.E,
                       "obs_mode": a.obs, "env_sets": a.sets, "record_bytes": rec_words * 4, "actions": "pre-generated ring of sample_action batches resident in HBM; defender 10 (detector training) -> no-op",
                       "randomized_ownership": bool(a.randomize), "steps_per_launch": F, "preheat_launches": max(PREHEAT, (Wm + F - 1) // F),
                       "fusion": (f"{F} plain steps per launch (step_many / cyg_step_multi): open-loop action batches resident in HBM, records stay in "
                                  "shared memory between the steps of a launch, so per-step HBM traffic is actions in + rewards out; "
                                  "single_step_launch below is the same workload at one launch per step") if F > 1 else "one launch per step",
                       "l2_policy": f"rotating {a.sets} env sets ({n_env_sets_bytes / 1e6:.0f} MB of state > 126 MB L2) and {2 * a.ring} action batches",
                       "parallelism": f"env-sharded x{world}, no per-step collective", "error_flags": errs},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic if F == 1 else traffic_f, "traffic_source": traffic_src if F == 1 else traffic_f_src,
                         "algorithmic_bytes_per_env_step": alg, "envs_per_launch": B,
                         "env_steps_per_launch": B * F, "launch_us": launch_s * 1e6, "peak_source": peak_src,
                         "actual_bytes_per_env_step": (2 * rec_words * 4) / F + 4 * (4 + net.W) + 12,
                         "note": ("algorithmic bytes are SURVEY 8(d)'s per-step figure x env-steps per launch; a fused launch moves less than that "
                                  "(state in/out once per launch), which 8(d) allows for") if F > 1 else None},
            "single_step_launch": {"value": world * B * K1 / (ms1 * 1e-3), "unit": UNIT, "launch_us": ms1 * 1e3 / K1, "steps": K1,
                                   "roofline_frac": alg * B / (ms1 * 1e-3 / K1) / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src},
            "clocks": clocks, "gpu_launches": int(launches),
        }
        if "ms_single_streams" in head:
            uss = head["ms_single_streams"] * 1e3 / K1
            line["single_step_launch"]["on_streams"] = {
                "us_per_step": uss, "value": world * B * 1e6 / uss, "unit": UNIT, "roofline_frac": alg * B / (uss * 1e-6) / 1e9 / peak,
                "how": f"the same one-launch-per-step workload with each of the {a.sets} env sets on its own stream (every set steps in order); "
                       "launch_us above stays the duration of ONE launch on one stream"}
        if "ms_fused_streams" in head:
            usf = head["ms_fused_streams"] * 1e3 / head["steps_fused"]
            line["fused_on_streams"] = {
                "us_per_step": usf, "value": world * B * 1e6 / usf, "unit": UNIT, "roofline_frac": alg * B / (usf * 1e-6) / 1e9 / peak,
                "how": f"the headline workload ({F} steps per launch) with each of the {a.sets} env sets on its own stream; `value` above "
                       "stays the one-stream figure"}
        if c5:
            legs["c5"] = c5
        if legs:
            line["legs"] = legs
        if e2e:
            line["e2e"] = {"value": world * B * e2e[1] / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": e2e[2],
                           "d2h_bytes_per_step": e2e[3], "steps": e2e[1], "ms_per_step": ems / e2e[1], "preheat_steps": max(e2e[6] * PREHEAT, 120),
                           "samples_ms_per_step": [x / e2e[1] for x in e2e[7]], "reported": "median of the five samples",
                           "how": f"VectorCyberDefenseEnv.step_host(act=pinned compact rows [B, 2 + W], sync=False, packed_done=True) / wait_host() (results: raw f32, shaped f32, one done bit per env) over {e2e[6]} env groups of "
                                  f"{B} envs on {e2e[6]} streams: each group waits for its own previous (raw, shaped, done) before its next "
                                  "step; the copies of one group overlap the kernel of the other",
                           "one_group_synchronous": {"value": world * B * e2e[5] / (ems1 * 1e-3), "unit": UNIT,
                                                     "ms_per_step": ems1 / e2e[5], "steps": e2e[5]}}
        if not a.no_cpu_baseline and world == 1:
            v, cores, sample, _ = cpu_arm(a, a.cpu_seconds)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "reference_python": reference_python_record()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
