"""VectorCyberDefenseEnv: B independent CyGym envs stepped by one fused CUDA launch.

The batched counterpart of Volt_Typhoon_CyberDefenseEnv (volt_typhoon_env.py:30): same
transition, same reset()/step() vocabulary, tensors instead of Python objects.  torch provides
device memory and streams only; every state transition is a kernel of libcygym_b200.so reached
through the C-ABI of include/cygym_b200.h.  There is no CPU path.
"""
import ctypes as C
from collections import namedtuple

import numpy as np
import torch

from . import _capi as K
from .network import Network


class ActionBatch:
    """One action per env: (action_type, exploit_indices, device_indices, app_index)
    (volt_typhoon_env.py:876) packed as hdr[B,4] + device mask[B,W] (+ optional explicit order)."""

    def __init__(self, hdr, mask, order=None):
        self.hdr, self.mask, self.order = hdr, mask, order

    @staticmethod
    def pack(actions, mode, M, order_form=False):
        """Host-side packing of a list of reference-style action tuples (or None) -> numpy arrays."""
        W = (M + 31) // 32
        B = len(actions)
        hdr = np.zeros((B, 4), np.uint32)
        mask = np.zeros((B, W), np.uint32)
        order = np.zeros((B, M), np.uint16) if order_form else None
        modes = mode if isinstance(mode, (list, tuple, np.ndarray)) else [mode] * B
        for b, a in enumerate(actions):
            m = 1 if modes[b] in (1, "attacker") else 0
            if a is None:
                hdr[b, 0] = K.ATYPE_NONE | (m << 8)
                continue
            atype, ex, devs, app = a
            ex = [int(x) for x in np.atleast_1d(ex)][:4]
            devs = [int(d) for d in devs]
            at = max(-127, min(127, int(atype)))
            hdr[b, 0] = (at & 0xFF) | (m << 8) | (len(ex) << 16)
            w1 = 0
            for i, x in enumerate(ex):
                w1 |= (max(-128, min(127, x)) & 0xFF) << (8 * i)
            hdr[b, 1] = w1
            hdr[b, 2] = len(devs)
            hdr[b, 3] = np.uint32(int(app) & 0xFFFFFFFF)
            for d in devs:
                if not 0 <= d < M:
                    raise IndexError(f"device index {d} out of range")
                mask[b, d >> 5] |= np.uint32(1 << (d & 31))
            if order_form:
                if len(devs) > M:
                    raise ValueError("more device indices than device slots")
                order[b, :len(devs)] = devs
            elif devs != sorted(set(devs)):
                raise ValueError("mask form needs an ascending duplicate-free device list; use order_form=True")
        return hdr, mask, order

    @staticmethod
    def unpack(hdr, mask, order=None):
        """The inverse of pack: hdr [B, 4] + mask [B, W] (+ order [B, >= n_dev] for the order form) -> the list of B
        reference-style action tuples, None where the header holds ATYPE_NONE."""
        f = decode_header(hdr)
        bits = np.unpackbits(np.ascontiguousarray(mask).view(np.uint8).reshape(len(f.atype), -1), axis=1, bitorder="little")
        devs = lambda b: [int(d) for d in order[b][:f.n_dev[b]]] if order is not None else np.nonzero(bits[b])[0].tolist()
        return [None if (f.atype[b] & 0xFF) == K.ATYPE_NONE else (int(f.atype[b]), f.ex[b, :f.n_ex[b]].tolist(), devs(b), int(f.app[b]))
                for b in range(len(f.atype))]


ActionHeader = namedtuple("ActionHeader", "atype mode n_ex ex n_dev first app")


def decode_header(hdr):
    """Action headers [B, 4] (numpy or CPU torch; include/cygym_b200.h) -> ActionHeader of [B] arrays: atype (the
    signed type byte; ATYPE_NONE reads as -128), mode, n_ex, ex [B, 4] (signed exploit bytes), n_dev, first
    (device_indices[0], -1 when not given) and app."""
    h = np.ascontiguousarray(hdr.numpy() if hasattr(hdr, "numpy") else hdr).view(np.uint32).reshape(-1, 4)
    i8 = lambda a: (a & 0xFF).astype(np.uint8).view(np.int8).astype(np.int32)
    return ActionHeader(atype=i8(h[:, 0]), mode=(h[:, 0] >> 8) & 1, n_ex=(h[:, 0] >> 16) & 0xFF,
                        ex=i8(h[:, 1][:, None] >> (8 * np.arange(4, dtype=np.uint32))), n_dev=h[:, 2] & 0xFFFF,
                        first=(h[:, 2] >> 16).astype(np.int64) - 1, app=h[:, 3].view(np.int32))


def header_rows(atype, mode, exploit, n_dev, app):
    """torch: single-exploit action headers [N, 4] int32 from int [N] tensors (mode: 0 defender, 1 attacker)."""
    i32 = lambda t: t.to(torch.int32)
    return torch.stack([(i32(atype) & 0xFF) | (mode << 8) | (1 << 16), i32(exploit) & 0xFF, i32(n_dev), i32(app)], dim=1)


def pack_device_mask(m, W):
    """torch: bool [B, M] -> int32 [B, W] device masks."""
    B, M = m.shape
    pad = W * 32 - M
    if pad:
        m = torch.nn.functional.pad(m, (0, pad))
    weights = (1 << torch.arange(32, device=m.device, dtype=torch.int64))
    words = (m.view(B, W, 32).to(torch.int64) * weights).sum(-1)
    return torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)


def compact_action_rows(hdr, mask):
    """hdr [B, 4] + mask [B, W] (numpy or CPU torch, the arrays of ActionBatch.pack) -> compact rows [B, 2 + W] int32
    (include/cygym_b200.h, cyg_unpack_actions): what a host-buffer step copies over PCIe.  Raises ValueError when an
    action does not fit the compact ranges (exploit indices -8..7, app_index -32768..32767, device_indices[0] < 255)."""
    h = np.ascontiguousarray(hdr.numpy() if hasattr(hdr, "numpy") else hdr).view(np.uint32)
    m = np.ascontiguousarray(mask.numpy() if hasattr(mask, "numpy") else mask).view(np.uint32)
    f = decode_header(h)
    n_ex, n_dev, first1, app, ex = f.n_ex, f.n_dev, (f.first + 1).astype(np.uint32), f.app, f.ex
    if (h[:, 0] >> 24).any() or ((h[:, 0] >> 9) & 0x7F).any() or (n_ex > 4).any() or (n_dev > 4095).any() or (first1 > 255).any() \
            or (app < -32768).any() or (app > 32767).any() or (ex < -8).any() or (ex > 7).any():
        raise ValueError("action outside the compact row ranges: use the full hdr / mask arrays")
    rows = np.empty((h.shape[0], 2 + m.shape[1]), np.uint32)
    rows[:, 0] = (h[:, 0] & 0x1FF) | (n_ex << 9) | (n_dev << 12) | (first1 << 24)
    rows[:, 1] = ((ex & 15).astype(np.uint32) << (4 * np.arange(4, dtype=np.uint32))).sum(1, dtype=np.uint32) | ((app & 0xFFFF).astype(np.uint32) << 16)
    rows[:, 2:] = m
    return rows.view(np.int32)


def expand_action_rows(rows):
    """The inverse of compact_action_rows on the host (what cyg_unpack_actions does on the device): (hdr, mask) uint32."""
    r = np.ascontiguousarray(rows).view(np.uint32)
    w0, w1 = r[:, 0], r[:, 1]
    x = ((w1[:, None] >> (4 * np.arange(4, dtype=np.uint32))) & 15).astype(np.int32)
    x = np.where(x >= 8, x - 16, x)
    hdr = np.empty((r.shape[0], 4), np.uint32)
    hdr[:, 0] = (w0 & 0x1FF) | (((w0 >> 9) & 7) << 16)
    hdr[:, 1] = ((x & 0xFF).astype(np.uint32) << (8 * np.arange(4, dtype=np.uint32))).sum(1, dtype=np.uint32)
    hdr[:, 2] = ((w0 >> 12) & 0xFFF) | ((w0 >> 24) << 16)
    hdr[:, 3] = (w1 >> 16).astype(np.uint16).view(np.int16).astype(np.int32).view(np.uint32)
    return hdr, r[:, 2:].copy()


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class VectorCyberDefenseEnv:
    def __init__(self, network: Network, num_envs, device="cuda:0", seed=0, env_id0=0, base_line="Nash", xcap=16,
                 stream=None, log_cap=0, detector_slots=0):
        """log_cap: records of every env's hop log kept in a ring (simulator.logger.logs, CDSimulator.py:663-679): 0 = only
        its length; >= 30 serves scans with a trained detector, 2000 what detector training reads.  detector_slots: how
        many envs can hold a trained detector (IsolationForest fitted by fit_detectors() on the device or by
        service_detectors() on the host)."""
        if not torch.cuda.is_available():
            raise RuntimeError("VectorCyberDefenseEnv needs a CUDA device (no CPU fallback)")
        self.L = K.lib()
        self.net = network
        self.B = int(num_envs)
        self.M, self.W, self.E, self.EW, self.X = network.M, network.W, network.E, network.EW, network.X
        self.device = torch.device(device)
        self.dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.xcap = max(int(xcap), len(network.template.get("extra", ())))
        self.env_id0 = int(env_id0)
        self.base_line = base_line
        self.log_cap = int(log_cap)
        self.cfg = K.make_config(network.cfg, network.E, seed=seed, xcap=self.xcap, base_line=base_line, log_cap=self.log_cap)
        hn = K.CygNetwork(network.row_ptr.ctypes.data, network.col.ctypes.data, network.mult.ctypes.data,
                          network.dev_static.ctypes.data, network.os_val.ctypes.data, network.ver_val.ctypes.data)
        self.h = C.c_void_p()
        K.check(self.L.cyg_create(C.byref(self.h), C.byref(self.cfg), C.byref(hn), self.B, self.env_id0, self.dev_index))
        words = C.c_int64()
        K.check(self.L.cyg_internal_words(self.h, C.byref(words)))
        self.S = int(words.value) - self.M - self.xcap - self.log_cap
        i32 = dict(dtype=torch.int32, device=self.device)
        self._state = torch.zeros(self.B * int(words.value), **i32)
        K.check(self.L.cyg_bind(self.h, _ptr(self._state)))
        self.records = self._state[: self.B * self.S].view(self.B, self.S)
        self.scalars = self.records[:, : K.NSCAL]  # live view of the 16 CYG_S_* scalars of every env
        # raw | shaped | done bits | done share one buffer so that a host caller reads the results with ONE device->host
        # copy: all of it, or (packed_done) the first 2 B + ceil(B / 32) words
        B, nbw = self.B, (self.B + 31) // 32
        self._nbw = nbw
        self._out = torch.zeros(3 * B + nbw, dtype=torch.float32, device=self.device)
        self.raw, self.shaped = self._out[:B], self._out[B:2 * B]
        self._done_bits = self._out[2 * B:2 * B + nbw].view(torch.int32)
        self.done = self._out[2 * B + nbw:].view(torch.int32)
        self._host = None
        self._host_evt = None
        self._graphs = {}
        self._graph_launches = 0  # step kernels launched through replayed CUDA graphs (not seen by cyg_launch_count)
        self._stream = stream
        self._obs = {}
        self._pre = None
        self._det_slots = self._det_of_env = self._next_slot = None
        if detector_slots:
            self._det_slots = torch.zeros(int(detector_slots), K.DET_WORDS, dtype=torch.int32, device=self.device)
            self._det_of_env = torch.full((self.B,), -1, dtype=torch.int32, device=self.device)
            # the first free slot: both fit paths take slots from this one device counter
            self._next_slot = torch.zeros(1, dtype=torch.int32, device=self.device)
            K.check(self.L.cyg_set_detectors(self.h, _ptr(self._det_slots), int(detector_slots), _ptr(self._det_of_env)))
        self.reset()

    # ---- plumbing ----
    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.L.cyg_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _s(self):
        s = self._stream if self._stream is not None else torch.cuda.current_stream(self.device)
        return C.c_void_p(s.cuda_stream)

    @property
    def launch_count(self):
        return int(self.L.cyg_launch_count(self.h)) + self._graph_launches

    def _drop_graphs(self):
        """A captured step_host() graph holds the kernel parameters BY VALUE (base_line, the per-env base_line
        pointer and stride, the debug buffer): whatever changes one of them must drop the captures."""
        if self._graphs:
            torch.cuda.synchronize(self.device)
            self._graphs = {}

    def set_base_line(self, name):
        self.base_line = name
        self._drop_graphs()
        K.check(self.L.cyg_set_base_line(self.h, K.BASE_LINES.get(name, K.BL_OTHER)))

    def set_base_line_per_env(self, codes):
        """codes: uint8 device tensor [B] of CYG_BL_* (see _capi.BASE_LINES), or [T, B] with one row per step of the
        next step_many() launches, or None to go back to the handle-wide value."""
        if codes is not None:
            codes = codes.to(self.device, torch.uint8).contiguous()
        self._bl_env = codes
        self._drop_graphs()
        if codes is not None and codes.dim() == 2:
            assert codes.shape[1] == self.B
            K.check(self.L.cyg_set_base_line_per_env_steps(self.h, _ptr(codes), int(codes.shape[0])))
        else:
            K.check(self.L.cyg_set_base_line_per_env(self.h, _ptr(codes)))

    def _canon_alloc(self):
        u = dict(dtype=torch.int32, device=self.device)
        d = dict(dev=torch.zeros(self.B, self.M, **u), ckpt=torch.zeros(self.B, self.M, **u),
                 blocked=torch.zeros(self.B, self.EW, **u), extra=torch.zeros(self.B, max(1, self.xcap), **u),
                 scal=torch.zeros(self.B, K.NSCAL, **u))
        if self.log_cap:
            d["logs"] = torch.zeros(self.B, self.log_cap, **u)
        return d

    def _cstate(self, c):
        return K.CygState(*[c[k].data_ptr() for k in ("dev", "ckpt", "blocked", "extra", "scal")],
                          c["logs"].data_ptr() if c.get("logs") is not None else None)

    # ---- state in / out (reset(from_init=True) / snapshot load, volt:1904-1925) ----
    def import_state(self, canon):
        """canon: dict of [B,*] int32/uint32 tensors or numpy arrays in the canonical layout."""
        c = {}
        for k, width in (("dev", self.M), ("ckpt", self.M), ("blocked", self.EW), ("extra", max(1, self.xcap)), ("scal", K.NSCAL)):
            a = canon[k]
            if isinstance(a, np.ndarray):
                a = torch.from_numpy(np.ascontiguousarray(a).view(np.int32).reshape(self.B, -1))
            a = a.to(self.device, torch.int32)
            if a.shape[1] < width:
                a = torch.nn.functional.pad(a, (0, width - a.shape[1]))
            c[k] = a.contiguous()
        if self.log_cap and canon.get("logs") is not None:  # the hop-log ring travels with the state when the caller has one
            a = canon["logs"]
            if isinstance(a, np.ndarray):
                a = torch.from_numpy(np.ascontiguousarray(a).view(np.int32).reshape(self.B, -1))
            a = a.to(self.device, torch.int32)
            if a.shape[1] < self.log_cap:
                a = torch.nn.functional.pad(a, (0, self.log_cap - a.shape[1]))
            c["logs"] = a[:, : self.log_cap].contiguous()
        cs = self._cstate(c)
        K.check(self.L.cyg_import_state(self.h, C.byref(cs), self._s()))
        self._keep = c
        return self

    def export_state(self):
        c = self._canon_alloc()
        cs = self._cstate(c)
        K.check(self.L.cyg_export_state(self.h, C.byref(cs), self._s()))
        return c

    def reset(self, env_epoch0=0):
        """Every env <- the network's template state (what reset(from_init=True) reloads)."""
        t = self.net.template
        canon = {}
        for k, width in (("dev", self.M), ("ckpt", self.M), ("blocked", self.EW), ("extra", max(1, self.xcap)), ("scal", K.NSCAL)):
            row = np.zeros(width, np.uint32)
            src = np.asarray(t[k], np.uint32)
            row[: len(src)] = src
            # one row to the device, broadcast there (B x width words never cross PCIe)
            canon[k] = torch.from_numpy(row.view(np.int32)).to(self.device).unsqueeze(0).expand(self.B, width).contiguous()
        return self.import_state(canon)

    # ---- the hot path ----
    def step(self, actions: ActionBatch, flags=0, obs_mode=0, want_pre=False):
        """One step() of every env (volt_typhoon_env.py:818).  Returns (raw, shaped, done) device tensors
        that are overwritten by the next call."""
        return self._step([actions], flags, obs_mode, want_pre)

    def step_grouped(self, groups, obs_mode=0, want_pre=False):
        """step_grouped() of every env (volt_typhoon_env.py:694): groups = list of ActionBatch."""
        return self._step(groups if hasattr(groups, "hdr") else list(groups), K.STEP_GROUPED, obs_mode, want_pre)

    def _step(self, groups, flags, obs_mode, want_pre):
        G = len(groups)
        if hasattr(groups, "hdr"):  # already stacked [G, B, ..] (marl.GroupedBatch): no per-step torch.stack
            hdr, mask, order = groups.hdr, groups.mask, None
        elif G == 1:
            hdr, mask, order = groups[0].hdr, groups[0].mask, groups[0].order
        else:
            hdr = torch.stack([g.hdr for g in groups]).contiguous()
            mask = torch.stack([g.mask for g in groups]).contiguous()
            order = torch.stack([g.order for g in groups]).contiguous() if groups[0].order is not None else None
        a = K.CygActions(hdr.data_ptr(), mask.data_ptr(), order.data_ptr() if order is not None else None,
                         order.shape[-1] if order is not None else 0, G)
        obs = None
        if obs_mode:
            obs = self._obs_buf(obs_mode)
        pre = None
        if want_pre:
            if self._pre is None:
                self._pre = torch.zeros(self.B, 3, self.W, dtype=torch.int32, device=self.device)
            pre = self._pre
        o = K.CygStepOut(self.raw.data_ptr(), self.shaped.data_ptr(), self.done.data_ptr(),
                         pre.data_ptr() if pre is not None else None, obs.data_ptr() if obs is not None else None, obs_mode)
        K.check(self.L.cyg_step(self.h, C.byref(a), flags, C.byref(o), self._s()))
        self._hold = (hdr, mask, order)
        return self.raw, self.shaped, self.done

    def step_many(self, hdr, mask, flags=0, out=None):
        """T consecutive plain steps in ONE launch (cyg_step_multi): hdr [T, B, 4], mask [T, B, W] int32 device tensors
        holding the T action batches (open-loop: fixed sequences, scripted or pre-sampled random policies -- the loop
        body of simulate_game, do_agent.py:1875-2089).  Returns (raw [T, B], shaped [T, B], done [T, B]); the records
        never leave shared memory between the steps.  Bit-identical to T step() calls."""
        T = int(hdr.shape[0])
        assert hdr.shape == (T, self.B, 4) and mask.shape == (T, self.B, self.W) and hdr.is_contiguous() and mask.is_contiguous()
        if out is None:
            out = (torch.empty(T, self.B, dtype=torch.float32, device=self.device),
                   torch.empty(T, self.B, dtype=torch.float32, device=self.device),
                   torch.empty(T, self.B, dtype=torch.int32, device=self.device))
        a = K.CygActions(hdr.data_ptr(), mask.data_ptr(), None, 0, 1)
        o = K.CygStepOut(out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), None, None, 0)
        K.check(self.L.cyg_step_multi(self.h, C.byref(a), T, flags, C.byref(o), self._s()))
        self._hold = (hdr, mask, out)
        return out

    def block_envs(self):
        """Slots per CTA of this handle's rollout launches (cyg_block_envs): what rollout(block_order=...) indexes."""
        nb = C.c_int32(0)
        K.check(self.L.cyg_block_envs(self.h, C.byref(nb)))
        return int(nb.value)

    def rollout(self, hdr, mask, base_line, envs_per_row, row_base, returns=None, flags=0, block_order=None):
        """n_steps plain steps of every env in ONE launch from per-ROW action tables (cyg_rollout): hdr [T, R, 4],
        mask [T, R, W] int32, base_line [T, R] uint8 or None; slot b reads row (row_base + env_index_of_slot()[b]) // envs_per_row.
        `returns` [2, B] float64 accumulates the raw rewards of defender / attacker turns.  The loop body of
        DoubleOracle.simulate_game (do_agent.py:1875-2089) for the strategies that need no observation."""
        T, R = int(hdr.shape[0]), int(hdr.shape[1])
        assert hdr.shape == (T, R, 4) and mask.shape == (T, R, self.W) and hdr.is_contiguous() and mask.is_contiguous()
        if returns is None:
            returns = torch.zeros(2, self.B, dtype=torch.float64, device=self.device)
        if base_line is not None:
            base_line = base_line.to(self.device, torch.uint8).contiguous()
            assert base_line.shape == (T, R)
        if block_order is not None:  # a permutation of the CTA indices: expensive blocks first
            block_order = block_order.to(self.device, torch.int32).contiguous()
            assert block_order.numel() == (self.B + self.block_envs() - 1) // self.block_envs()
        a = K.CygRolloutArgs(hdr.data_ptr(), mask.data_ptr(), None if base_line is None else base_line.data_ptr(), T, R,
                             int(row_base), int(envs_per_row), 0, returns.data_ptr(), None if block_order is None else block_order.data_ptr())
        K.check(self.L.cyg_rollout(self.h, C.byref(a), flags, self._s()))
        self._hold = (hdr, mask, base_line, returns, block_order)
        return returns

    def set_env_id_stride(self, run, stride):
        """Slot s holds env env_id0 + (s // run) * stride + s % run (cyg_set_env_id_stride; run divides B; run <= 0: the
        default, env_id0 + s).  For rollout(): a rank takes the same slice of rollouts of every strategy pair."""
        K.check(self.L.cyg_set_env_id_stride(self.h, int(run), int(stride)))
        self._id_stride = (int(run), int(stride)) if run > 0 else None

    def env_index_of_slot(self):
        """int64 [B] on the device: env id minus env_id0 of every slot."""
        s = torch.arange(self.B, device=self.device)
        st = getattr(self, "_id_stride", None)
        return s if st is None else (s // st[0]) * st[1] + s % st[0]

    # ---- host-buffer front end: what a CPU-side caller (the reference's rollout loops) uses ----
    def host_buffers(self):
        """Pinned host staging, allocated once: action headers [B, 4] and device masks [B, W] (int32) in, results
        [3, B] float32 (raw | shaped | done bits) out."""
        if self._host is None:
            self._host = dict(
                hdr=torch.empty(self.B, 4, dtype=torch.int32).pin_memory(),
                mask=torch.empty(self.B, self.W, dtype=torch.int32).pin_memory(),
                out=torch.empty(3 * self.B + self._nbw, dtype=torch.float32).pin_memory(),
                d_act=torch.empty(self.B, 4 + self.W, dtype=torch.int32, device=self.device),
                d_rows=torch.empty(self.B, 2 + self.W, dtype=torch.int32, device=self.device),
                d_hdr=torch.empty(self.B, 4, dtype=torch.int32, device=self.device),
                d_mask=torch.empty(self.B, self.W, dtype=torch.int32, device=self.device))
        return self._host["hdr"], self._host["mask"], self._host["out"]

    def _host_ops(self, hdr, mask, flags, packed_done=False):
        h = self._host
        if mask is None and hdr.shape[1] == 2 + self.W:  # compact rows (compact_action_rows): the smallest copy, expanded on the device
            h["d_rows"].copy_(hdr, non_blocking=True)
            K.check(self.L.cyg_unpack_actions(self.h, _ptr(h["d_rows"]), _ptr(h["d_hdr"]), _ptr(h["d_mask"]), self._s()))
        elif mask is None:  # combined [B, 4 + W] rows: ONE host->device copy, split on the device
            h["d_act"].copy_(hdr, non_blocking=True)
            h["d_hdr"].copy_(h["d_act"][:, :4])
            h["d_mask"].copy_(h["d_act"][:, 4:])
        else:
            h["d_hdr"].copy_(hdr, non_blocking=True)
            h["d_mask"].copy_(mask, non_blocking=True)
        self._step([ActionBatch(h["d_hdr"], h["d_mask"])], flags, 0, False)
        if packed_done:  # raw | shaped | one done bit per env: 8.1 bytes per env over PCIe instead of 12
            K.check(self.L.cyg_pack_done(self.h, _ptr(self.done), _ptr(self._done_bits), self._s()))
            n = 2 * self.B + self._nbw
            h["out"][:n].copy_(self._out[:n], non_blocking=True)
        else:
            h["out"].copy_(self._out, non_blocking=True)

    def _host_views(self, packed_done):
        o, B, nbw = self._host["out"], self.B, self._nbw
        done = o[2 * B:2 * B + nbw].view(torch.int32) if packed_done else o[2 * B + nbw:].view(torch.int32)
        return o[:B], o[B:2 * B], done

    def host_result_bytes(self, packed_done=False):
        """Bytes one step_host() copies device -> host."""
        return 4 * (2 * self.B + self._nbw) if packed_done else 4 * (3 * self.B + self._nbw)

    def step_host(self, hdr=None, mask=None, flags=0, use_graph=True, act=None, sync=True, packed_done=False):
        """step() with HOST buffers: two pinned host->device copies of the actions (`hdr`, `mask`: pinned tensors of
        the caller's, default the staging buffers of host_buffers()), the kernel, one device->host copy of
        (raw, shaped, done) into host_buffers()[2], then a stream synchronise (the caller reads the rewards before
        choosing the next action).  The four operations are captured once per (hdr, mask) buffer pair into a CUDA
        graph and replayed, so a step costs one graph launch on the host.  Returns (raw, shaped, done) host views.
        The graph holds the ADDRESS of the caller's pinned buffer: keep one staging buffer per env group alive and
        refill it (a pinned tensor freed after it was captured leaves the host allocator waiting on a captured event).

        sync=False returns right after the enqueue (the host views are valid after wait_host()): a caller that drives
        two env groups on two streams (`stream=` of the constructor) chooses the actions of one group while the other
        group's copies and kernel are in flight -- each group stays closed-loop, the PCIe copies of one overlap the
        kernel of the other."""
        if self._host is None:
            self.host_buffers()
        h = self._host
        if act is not None:  # pinned int32 rows, [B, 4 + W] (hdr | mask) or [B, 2 + W] (compact_action_rows): ONE copy
            assert act.shape[1] in (4 + self.W, 2 + self.W)
            hdr, mask = act, None
        else:
            hdr = h["hdr"] if hdr is None else hdr
            mask = h["mask"] if mask is None else mask
        stream = self._stream if self._stream is not None else torch.cuda.current_stream(self.device)
        key = (hdr.data_ptr(), 0 if mask is None else mask.data_ptr(), int(flags), bool(packed_done))
        self._host_packed = bool(packed_done)
        graph = self._graphs.get(key) if use_graph else None
        if use_graph and graph is None and key not in self._graphs:
            try:
                g = torch.cuda.CUDAGraph()
                side = torch.cuda.Stream(self.device)
                side.wait_stream(stream)
                saved, self._stream = self._stream, None  # launches go to the capturing (current) stream
                try:
                    with torch.cuda.graph(g, stream=side):
                        self._host_ops(hdr, mask, flags, packed_done)
                finally:
                    self._stream = saved
                stream.wait_stream(side)
                self._graphs[key] = graph = g
            except Exception:
                self._graphs[key] = None  # capture not possible here: stay on the eager path for this buffer pair
                torch.cuda.synchronize(self.device)
        if graph is not None:
            with torch.cuda.stream(stream):
                graph.replay()
            self._graph_launches += 1
        else:
            with torch.cuda.stream(stream):
                self._host_ops(hdr, mask, flags, packed_done)
        if sync:
            stream.synchronize()
        else:
            if self._host_evt is None:
                self._host_evt = torch.cuda.Event()
            self._host_evt.record(stream)
        return self._host_views(packed_done)

    def wait_host(self):
        """Block until the last step_host(sync=False) of this env group has delivered its results; returns the host views."""
        if self._host_evt is not None:
            self._host_evt.synchronize()
        return self._host_views(getattr(self, "_host_packed", False))

    def _obs_buf(self, mode):
        if mode not in self._obs:
            dim = 4 * self.M + self.X if mode == 2 else 6 * self.M
            self._obs[mode] = torch.zeros(self.B, dim, dtype=torch.float32, device=self.device)
        return self._obs[mode]

    def last_obs(self, mode):
        return self._obs[mode]

    def pre_masks(self):
        return self._pre

    def observe(self, mode):
        """1: _get_defender_state, 2: _get_attacker_state, 3: _get_state (CyberDefenseEnv.py:241/194/146)."""
        obs = self._obs_buf(mode)
        K.check(self.L.cyg_observe(self.h, mode, _ptr(obs), self._s()))
        return obs

    def randomize_compromise_and_ownership(self, env_mask=None):
        if env_mask is not None:
            env_mask = env_mask.to(self.device, torch.uint8).contiguous()
            self._hold_mask = env_mask
        K.check(self.L.cyg_randomize(self.h, _ptr(env_mask), self._s()))

    # ---- trained detectors (defender actions 10 / 5; fitted on the device from per-env seeds, or by scikit-learn) ----
    def log_records(self, b, last=2000):
        """The last `last` hop-log records of env b in log order: int array [n, 2] of (from_device, to_device)."""
        n = int(self.scalars[b, K.S_LOGS].item())
        k = min(n, last)
        if k > self.log_cap:
            raise ValueError(f"the hop-log ring keeps {self.log_cap} records per env, {k} are needed (log_cap=)")
        base = self.B * (self.S + self.M + self.xcap)
        return K.log_records(self._state[base + b * self.log_cap: base + (b + 1) * self.log_cap].cpu().numpy(), n, k)

    def pending_detectors(self):
        """Envs whose defender trained the detector (action 10 on a non-empty log) since the last service."""
        return torch.nonzero(self.scalars[:, K.S_FLAGS] & K.FL_DET_PENDING).flatten().tolist()

    def service_detectors(self, seed_of_env=None):
        """Fit (scikit-learn IsolationForest on the env's last <= 2000 hop-log records: Detector.train,
        CDSimulator.py:687-695) and upload the detector of every pending env; the next scan of that env consults it.
        Call after a step that may have trained (the Gym drop-in does it itself).  seed_of_env(b) -> seed for numpy's
        global stream before env b's fit (the reference's forest has random_state=None), or None: the fit then draws
        from numpy's stream as it stands, which only this host path can do.  With a seed per env, fit_detectors() does
        the same fits on the device in one launch."""
        from . import detector as DET
        pend = self.pending_detectors()
        for b in pend:
            if self._det_slots is None:
                raise RuntimeError("no detector slots: construct the env with detector_slots=")
            slot = int(self._det_of_env[b].item())
            if slot < 0:
                slot = int(self._next_slot.item())
                if slot >= self._det_slots.shape[0]:
                    raise RuntimeError(f"all {self._det_slots.shape[0]} detector slots are taken (detector_slots=)")
                self._next_slot.fill_(slot + 1)
                self._det_of_env[b] = slot
            model = DET.fit_detector(self.log_records(b), None if seed_of_env is None else seed_of_env(b))
            self._det_slots[slot] = torch.from_numpy(DET.pack_detector(model).view(np.int32)).to(self.device)
            self.scalars[b, K.S_FLAGS] &= ~K.FL_DET_PENDING
        return len(pend)

    def fit_detectors(self, seeds):
        """Fit the detector of every pending env on the device, in one launch and without a host synchronisation
        (cyg_fit_detectors): env b's slot becomes exactly what service_detectors(lambda b: seeds[b]) uploads, i.e.
        numpy's global stream seeded with seeds[b], then scikit-learn's IsolationForest on the env's last <= 2000 hop-log
        records.  seeds: integer tensor [B] with values in [0, 2**32).  An env that cannot be fitted (every slot taken,
        or a hop-log ring shorter than the records the fit reads) stays pending and gets CYG_FL_ERR_DETECTOR
        (error_flags()).  Envs without a slot take the next free ones in env order, from the counter service_detectors()
        uses as well."""
        s = torch.as_tensor(seeds).to(self.device, torch.int64, non_blocking=True).reshape(-1)
        assert s.numel() == self.B, "one seed per env"
        s = s & 0xFFFFFFFF
        s = torch.where(s >= 2 ** 31, s - 2 ** 32, s).to(torch.int32).contiguous()
        self._hold_seeds = s
        K.check(self.L.cyg_fit_detectors(self.h, _ptr(s), _ptr(self._next_slot), self._s()))

    def rebuild_graph_cache(self, env_mask=None):
        """_rebuild_graph_cache() from outside a step (volt_typhoon_env.py:456-483): every blocked edge is forgotten (:476)."""
        if env_mask is not None:
            env_mask = env_mask.to(self.device, torch.uint8).contiguous()
            self._hold_mask = env_mask
        K.check(self.L.cyg_rebuild_graph_cache(self.h, _ptr(env_mask), self._s()))

    def sample_actions(self, mode, out: ActionBatch = None, want_order=False):
        """sample_action() of every env (CyberDefenseEnv.py:555-578) as an ActionBatch on the device.  The set form
        (hdr + mask) carries device_indices[0] of the draw in hdr[:, 2] >> 16; want_order=True also fills `order`
        [B, M] int16 with the whole list in random.sample's draw order (stepping with it takes the order-form kernel)."""
        m = 1 if mode in (1, "attacker") else 0
        if out is None:
            out = ActionBatch(torch.zeros(self.B, 4, dtype=torch.int32, device=self.device),
                              torch.zeros(self.B, self.W, dtype=torch.int32, device=self.device))
        if want_order:
            if out.order is None:
                out.order = torch.zeros(self.B, self.M, dtype=torch.int16, device=self.device)
            K.check(self.L.cyg_sample_actions_ordered(self.h, m, _ptr(out.hdr), _ptr(out.mask), _ptr(out.order),
                                                      int(out.order.shape[1]), self._s()))
        else:
            K.check(self.L.cyg_sample_actions(self.h, m, _ptr(out.hdr), _ptr(out.mask), self._s()))
        return out

    def to_device(self, hdr, mask, order=None):
        f = lambda a, dt: None if a is None else torch.from_numpy(np.ascontiguousarray(a).view(dt)).to(self.device)
        return ActionBatch(f(hdr, np.int32), f(mask, np.int32), f(order, np.int16))

    # ---- counters (the `info` dict of volt:1272-1285, per env) ----
    def info(self):
        s = self.scalars
        return {key: s[:, slot].contiguous().view(torch.float32) if is_float else s[:, slot]
                for _, key, slot, is_float in K.COUNTERS}

    def error_flags(self):
        """Sticky per-env CYG_FL_ERR_* bits (0 everywhere on a healthy run)."""
        return self.scalars[:, K.S_FLAGS] & K.FL_ERR_MASK
