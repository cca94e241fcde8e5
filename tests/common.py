"""Shared helpers for the parity tests (TEST INFRASTRUCTURE)."""
import glob
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz")))
GOLDEN_IDS = [os.path.basename(f)[:-4] for f in GOLDEN]


def load_golden(path):
    return dict(np.load(path))


class CudaImpl:
    """oracle.trajectory.replay() protocol on top of the CUDA library (B = 1), through the C-ABI."""

    def __init__(self, g):
        import torch
        from cygym_b200 import network_from_golden
        from cygym_b200.vector_env import VectorCyberDefenseEnv
        self.torch = torch
        net, meta = network_from_golden(g)
        self.meta = meta
        self.env = VectorCyberDefenseEnv(net, 1, seed=meta["draw_seed"], env_id0=meta["env_id"], xcap=meta["xcap"],
                                         log_cap=meta.get("log_cap", 0), detector_slots=1 if meta.get("log_cap", 0) else 0)

    def load(self, init):
        self.env.import_state({k: np.asarray(v, np.uint32)[None] for k, v in init.items()})

    def bump_epoch(self, n):
        if n:
            self.env.scalars[:, 1] += int(n)

    def sample_action(self, mode):
        ab = self.env.sample_actions(mode, want_order=True)
        self.torch.cuda.synchronize()
        return (ab.hdr.cpu().numpy().view(np.uint32)[0], ab.mask.cpu().numpy().view(np.uint32)[0],
                ab.order.cpu().numpy().view(np.uint16)[0])

    def step(self, hdr, mask, order, flags):
        env = self.env
        G = hdr.shape[0]
        from cygym_b200.vector_env import ActionBatch
        groups = []
        for g in range(G):
            groups.append(env.to_device(hdr[g], mask[g], None if order is None else order[g]))
        if flags & 1:
            raw, shaped, done = env.step_grouped(groups, want_pre=True)
        else:
            raw, shaped, done = env.step(groups[0], flags=flags, want_pre=True)
        self.torch.cuda.synchronize()
        return dict(raw=raw.cpu().numpy().astype(np.float64), shaped=shaped.cpu().numpy().astype(np.float64),
                    done=done.cpu().numpy(), pre_masks=env.pre_masks().cpu().numpy().view(np.uint32))

    def randomize(self):
        self.env.randomize_compromise_and_ownership()

    def set_base_line(self, name):
        self.env.set_base_line(name)

    def state(self):
        c = self.env.export_state()
        self.torch.cuda.synchronize()
        d = {k: v.cpu().numpy().view(np.uint32)[0] for k, v in c.items()}
        if "logs" in d:
            from oracle.trajectory import log_tail_of_ring
            d["logs_tail"] = log_tail_of_ring(d["logs"], int(d["scal"][6]), self.env.log_cap)
        return d

    def service_detector(self, seed):
        self.env.service_detectors(lambda b: seed)

    def observe(self, mode):
        o = self.env.observe(mode)
        self.torch.cuda.synchronize()
        return o.cpu().numpy()[0]


def gym_action(hdr, mask, order, M, order_form):
    """A recorded action row (include/cygym_b200.h packing) as the reference's (type, exploits, devices, app) tuple."""
    at = int(np.int8(hdr[0] & 0xFF))
    if (int(hdr[0]) & 0xFF) == 0x80:
        return None
    n_ex = (int(hdr[0]) >> 16) & 0xFF
    ex = [int(np.int8((int(hdr[1]) >> (8 * i)) & 0xFF)) for i in range(n_ex)]
    n = int(hdr[2]) & 0xFFFF
    devs = [int(x) for x in order[:n]] if order_form else [d for d in range(M) if (int(mask[d >> 5]) >> (d & 31)) & 1]
    return (at, ex, devs, int(np.int32(hdr[3])))


def replay_golden_on_gym(env, g):
    """Feed golden trajectory `g` (recorded from the reference) to the drop-in Volt_Typhoon_CyberDefenseEnv `env` as the
    reference's action tuples, and compare after every op: the 6-tuple, observations, counters, the canonical state and,
    where the recording keeps it, the hop log.  Where the reference trained its detector, numpy's stream was seeded
    with `train_seed`; the drop-in gets the same seed and must fit (and later consult) the detector on its own."""
    from oracle import trajectory as TR
    meta = json.loads(str(g["meta"]))
    M = meta["M"]
    for t in range(len(g["kind"])):
        kind = int(g["kind"][t])
        if kind == TR.OP_RANDOMIZE:
            env.randomize_compromise_and_ownership()
        elif kind == TR.OP_BASELINE:
            env.base_line = TR.BASELINES[int(g["baseline"][t])]
        else:
            G = int(g["n_groups"][t])
            env.mode = "attacker" if int(g["mode"][t]) else "defender"
            acts = [gym_action(g["hdr"][t][k], g["mask"][t][k], g["order"][t][k], M, meta["order_form"]) for k in range(G)]
            # the reference drew every non-None action with sample_action(): one draw epoch each
            env._venv.scalars[:, 1] += sum(1 for a in acts if a is not None)
            env._host = None
            seed = int(g["train_seed"][t]) if "train_seed" in g else -1
            env.detector_fit_seed = seed if seed >= 0 else None
            out = env.step(acts if kind == TR.OP_GROUPED else acts[0])
            assert len(out) == 6
            state, raw, shaped, done, info, logs = out
            tol = 1e-5 * max(1.0, abs(float(g["raw"][t])))
            assert abs(raw - float(g["raw"][t])) <= tol and abs(shaped - float(g["shaped"][t])) <= tol, f"op {t}"
            assert done == bool(g["done"][t])
            assert state.shape == (6 * M,) and state.dtype == np.float64
            s6 = state.reshape(M, 6)
            for row, col in enumerate((2, 4, 5)):
                exp = np.array([(int(g["pre"][t][row, d >> 5]) >> (d & 31)) & 1 for d in range(M)], np.float64)
                assert np.array_equal(s6[:, col], exp), f"op {t}: returned state column {col}"
            assert np.array_equal(env._get_defender_state().astype(np.float32), g["obs_def"][t]), f"op {t}"
            a_obs = env._get_attacker_state()
            assert a_obs.dtype == np.float32 and a_obs.shape == (4 * M + 6,) and np.array_equal(a_obs, g["obs_att"][t])
            sc = g["scal"][t]
            assert env.step_num == int(sc[0]) and env.work_done == int(sc[8]) and env.scan_cnt == int(sc[11])
            assert env.compromised_devices_cnt == int(sc[7]) and env.edges_blocked == int(sc[14])
            assert info["Compromised_devices"] == int(sc[7]) and info["mode"] == env.mode
            # info is built before step_num moves in step(), after it in step_grouped() (volt:1272-1285 / :746-755)
            assert info["step_count"] == (int(sc[0]) if kind == TR.OP_GROUPED else int(sc[0]) - 1), f"op {t}"
            assert len(logs) == int(sc[6])
            nya = np.array([(int(g["dev"][t][d]) >> 2) & 1 for d in range(M)])
            assert [int(d.Not_yet_added) for d in env._get_ordered_devices()] == nya.tolist()
        st = env._snap()
        for k in ("dev", "ckpt", "blocked"):
            assert np.array_equal(st[k], g[k][t]), f"op {t}: {k}"
        a, r = np.array(st["scal"], np.uint32), np.array(g["scal"][t], np.uint32)
        assert np.allclose(a[9:11].view(np.float32), r[9:11].view(np.float32), rtol=1e-5, atol=1e-6), f"op {t}: cost counters"
        a[9:11] = r[9:11] = 0
        assert np.array_equal(a, r), f"op {t}: scalars {a} != {r}"  # includes the detector's trained / pending flags
        nx = int(g["n_extra"][t])
        assert sorted(int(x) & 0x1FFFFFF for x in st["extra"][:nx]) == sorted(int(x) for x in g["extra"][t][:nx]), f"op {t}: extra edges"
        if meta.get("log_cap", 0):
            tail = np.zeros(TR.LOG_TAIL, np.uint32)
            recs = [l for l in env.simulator.logger.get_logs()[-TR.LOG_TAIL:] if l is not None]
            tail[TR.LOG_TAIL - len(recs):] = [l["from_device"] | (l["to_device"] << 16) for l in recs]
            assert np.array_equal(tail, g["logs_tail"][t]), f"op {t}: hop-log records"


def oracle_for(net, seed, xcap, env_id0=0, base_line="Nash"):
    from oracle import cyg_oracle as O
    cfg = O.make_config(net.cfg, net.E, seed=seed, xcap=xcap, base_line=base_line)
    d = dict(row_ptr=net.row_ptr, col=net.col, mult=net.mult, dev_static=net.dev_static, os_val=net.os_val, ver_val=net.ver_val)
    return O.Oracle(d, cfg, env_id0=env_id0), cfg


def oracle_state_from_template(orc, net, B):
    st = orc.new_state(B)
    t = net.template
    st.dev[:] = np.asarray(t["dev"], np.uint32)[None]
    st.ckpt[:] = np.asarray(t["ckpt"], np.uint32)[None]
    st.blocked[:] = 0
    st.blocked[:, :len(t["blocked"])] = np.asarray(t["blocked"], np.uint32)[None]
    st.extra[:] = 0
    if len(t["extra"]):
        st.extra[:, :len(t["extra"])] = np.asarray(t["extra"], np.uint32)[None]
    st.scal[:] = np.asarray(t["scal"], np.uint32)[None]
    return st


def sanitize_actions(hdr, scal_logs, mode):
    """Drop the trained-IsolationForest branch (defender action 10 with a non-empty log): out of the
    kernel's scope (SURVEY.md section 8c).  Replaced by the no-op 8, in place."""
    if mode == 0:
        at = hdr[:, 0] & 0xFF
        bad = (at == 10) & (scal_logs > 0)
        hdr[bad, 0] = (hdr[bad, 0] & ~np.uint32(0xFF)) | np.uint32(8)
    return hdr


def compare_states(a, b, label, rtol=1e-5):
    """a, b: dicts of canonical numpy arrays [B, *]; raises AssertionError on the first mismatch."""
    for k in ("dev", "ckpt", "blocked", "extra"):
        x, y = np.asarray(a[k]).view(np.uint32), np.asarray(b[k]).view(np.uint32)
        w = min(x.shape[1], y.shape[1])
        if not np.array_equal(x[:, :w], y[:, :w]):
            bad = np.argwhere(x[:, :w] != y[:, :w])[:5]
            raise AssertionError(f"{label}: {k} differs at (env, idx) {bad.tolist()}: "
                                 f"{[hex(int(x[i, j])) for i, j in bad]} vs {[hex(int(y[i, j])) for i, j in bad]}")
    sa, sb = np.array(a["scal"]).view(np.uint32).copy(), np.array(b["scal"]).view(np.uint32).copy()
    fa, fb = sa[:, 9:11].copy().view(np.float32), sb[:, 9:11].copy().view(np.float32)
    if not np.allclose(fa, fb, rtol=rtol, atol=1e-6):
        raise AssertionError(f"{label}: cost counters differ")
    sa[:, 9:11] = 0
    sb[:, 9:11] = 0
    if not np.array_equal(sa, sb):
        bad = np.argwhere(sa != sb)[:5]
        raise AssertionError(f"{label}: scalars differ at (env, slot) {bad.tolist()}: "
                             f"{[int(sa[i, j]) for i, j in bad]} vs {[int(sb[i, j]) for i, j in bad]}")


def compare_rewards(out_a, out_b, label, rtol=1e-5):
    for k in ("raw", "shaped"):
        x, y = np.asarray(out_a[k], np.float64), np.asarray(out_b[k], np.float64)
        tol = rtol * np.maximum(1.0, np.abs(y))
        if np.any(np.abs(x - y) > tol):
            i = int(np.argmax(np.abs(x - y) - tol))
            raise AssertionError(f"{label}: {k} reward env {i}: {x[i]} vs {y[i]}")
    if not np.array_equal(np.asarray(out_a["done"]), np.asarray(out_b["done"])):
        raise AssertionError(f"{label}: done flags differ")
