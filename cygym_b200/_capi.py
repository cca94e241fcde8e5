"""ctypes binding of libcygym_b200.so (the C-ABI of include/cygym_b200.h).

There is no CPU path: importing this module without the compiled CUDA library raises, and every
entry point needs a CUDA device.  `build()` compiles the library in-tree with nvcc for sm_100a.
"""
import ctypes as C
import os
import subprocess

from . import draw_tables as DT

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CYGYM_B200_LIB") or os.path.join(_HERE, "libcygym_b200.so")  # override: profiling builds only
_SRC = os.path.join(_HERE, "csrc", "cyg_kernels.cu")
_DEPS = [_SRC, os.path.join(_HERE, "csrc", "cyg_core.cuh"), os.path.join(_HERE, "csrc", "cyg_coop.cuh"),
         os.path.join(_HERE, "csrc", "cyg_tables.h"), os.path.join(_HERE, "csrc", "cyg_iforest.cuh"),
         os.path.join(os.path.dirname(_HERE), "include", "cygym_b200.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
PLANE_WIDTHS = (1, 2, 3, 4, 64)  # one translation unit of cyg_kernels.cu per plane width W (+ one for the C-ABI)

# The constants of include/cygym_b200.h, named as there without the CYG_ prefix (tests/test_abi_formats.py checks them).
ABI_VERSION = 2
NSCAL = 16
ATYPE_NONE = 0x80
MODE_DEFENDER, MODE_ATTACKER = 0, 1
STEP_GROUPED, STEP_SKIP_WORK = 1, 2
BL_NASH, BL_NO_DEFENSE, BL_PRESET, BL_NO_ATTACK, BL_OTHER = range(5)
BASE_LINES = {"Nash": BL_NASH, "No Defense": BL_NO_DEFENSE, "Preset": BL_PRESET, "No Attack": BL_NO_ATTACK}
E_INVAL, E_NOMEM, E_CUDA, E_STATE = -22, -12, -5, -71

# canonical per-device word dev[B][M] (CYG_DEV_*)
DEV_COMP, DEV_KNOWN, DEV_NYA, DEV_OWNED = 1 << 0, 1 << 1, 1 << 2, 1 << 3
DEV_REMOVED, DEV_HASWL, DEV_BUSYSET, DEV_ACTSET = 1 << 4, 1 << 5, 1 << 6, 1 << 7
DEV_PT_SHIFT, DEV_BUSY_SHIFT, DEV_CBY_SHIFT = 8, 12, 20
DEV_PT_MASK, DEV_BUSY_MASK, DEV_CBY_MASK = 0x7, 0xFF, 0x3F
# per-device checkpoint word ckpt[B][M] (CYG_CK_*); processing time, busy time and compromised_by use the DEV_* fields
CK_COMP, CK_KNOWN, CK_NYA, CK_REACH, CK_HASWL, CK_VALID = 1 << 0, 1 << 1, 1 << 2, 1 << 3, 1 << 5, 1 << 31
# static per-device word dev_static[M] (CYG_ST_*)
ST_DC, ST_SERVER, ST_REACH = 1 << 0, 1 << 1, 1 << 2
ST_NAPPS_SHIFT, ST_VULN_SHIFT = 8, 16

# scalar slots (CYG_S_*)
(S_STEP, S_EPOCH, S_FLAGS, S_PREV_X, S_DEF_STEP, S_ATT_STEP, S_LOGS, S_COMPCNT, S_WORK, S_DEFCOST,
 S_CLEANCOST, S_SCAN, S_REVERT, S_CKPT, S_EBLK, S_EADD) = range(16)
# flag bits of scal[S_FLAGS] (CYG_FL_*); bit FL_DISC_SHIFT + e: exploits[e].discovered
FL_HAS_CKPT, FL_SETS_INIT, FL_DET_TRAINED, FL_DET_PENDING = 0x1, 0x2, 0x4, 0x8
FL_ERR_BUSY, FL_ERR_XCAP, FL_ERR_DETECTOR, FL_ERR_MASK = 0x10, 0x20, 0x40, 0xF0
FL_DISC_SHIFT = 8

# The reference env's counters held in scalar slots: (attribute name, info-dict key, slot, slot holds float32 bits),
# in the key order of VectorCyberDefenseEnv.info() and of the reference's info dict (volt_typhoon_env.py:1272-1285).
COUNTERS = (
    ("step_num", "step_count", S_STEP, False), ("revert_count", "revert_count", S_REVERT, False),
    ("checkpoint_count", "checkpoint_count", S_CKPT, False), ("defensive_cost", "defensive_cost", S_DEFCOST, True),
    ("clearning_cost", "clearning_cost", S_CLEANCOST, True), ("scan_cnt", "Scan_count", S_SCAN, False),
    ("work_done", "work_done", S_WORK, False), ("compromised_devices_cnt", "Compromised_devices", S_COMPCNT, False),
    ("edges_blocked", "Edges Blocked", S_EBLK, False), ("edges_added", "Edges Added", S_EADD, False),
    ("defender_step", "defender_step", S_DEF_STEP, False), ("attacker_step", "attacker_step", S_ATT_STEP, False),
)

# extra (per-env) edge word extra[B][xcap] (CYG_X_*)
X_V_SHIFT, X_BLOCKED, X_IDMASK = 12, 1 << 24, 0xFFF

# trained-detector slot (CYG_DET_*)
DET_WORDS, DET_TREE0, DET_TREE_STRIDE, DET_TABLE, DET_WINDOW = 6160, 4, 2048, 4100, 2000


def extra_edges(words):
    """Extra-edge words -> [(from_device, to_device, blocked)]."""
    return [(int(w) & X_IDMASK, (int(w) >> X_V_SHIFT) & X_IDMASK, bool(int(w) & X_BLOCKED)) for w in words]


def log_records(ring, n, k):
    """The last k of the n records of an env's hop-log ring (record i at i % len(ring), from_device | to_device << 16),
    in log order: int64 array [k, 2] of (from_device, to_device)."""
    import numpy as np
    r = np.asarray(ring, np.uint32)[np.arange(n - k, n) % max(1, len(ring))]
    return np.stack([r & 0xFFFF, r >> 16], axis=1).astype(np.int64)


class CygConfig(C.Structure):
    """struct cyg_config"""
    _fields_ = [
        ("M", C.c_int32), ("E", C.c_int32), ("X", C.c_int32), ("n_exploits", C.c_int32), ("xcap", C.c_int32),
        ("num_of_device", C.c_int32), ("min_network_size", C.c_int32), ("evolve_period", C.c_int32),
        ("wl_period_base", C.c_int32), ("wl_period_max", C.c_int32), ("wl_cap", C.c_int32),
        ("scaling_vulnerability", C.c_int32), ("turbo", C.c_int32), ("zero_day", C.c_int32),
        ("zero_day_mask", C.c_uint32), ("att_space_n", C.c_int32), ("def_space_n", C.c_int32),
        ("default_high", C.c_int32), ("n_app_ids", C.c_int32), ("base_line", C.c_int32), ("tri_high", C.c_int32),
        ("log_cap", C.c_int32),
        ("work_scale", C.c_float), ("comp_scale", C.c_float), ("def_scale", C.c_float), ("gamma", C.c_float),
        ("thr_p_add", C.c_uint64), ("thr_p_attacker", C.c_uint64),
        ("poisson_tab", C.c_uint32 * 16), ("tri_tab", C.c_uint32 * 8), ("seed", C.c_uint64),
        ("turbo_frac_clients", C.c_double), ("turbo_frac_servers", C.c_double), ("turbo_max_clients", C.c_int32),
        ("turbo_max_servers", C.c_int32), ("turbo_ramp_steps", C.c_int32), ("reserved1", C.c_int32),
    ]


class CygNetwork(C.Structure):
    """struct cyg_network (host pointers)"""
    _fields_ = [("row_ptr", C.c_void_p), ("col", C.c_void_p), ("mult", C.c_void_p), ("dev_static", C.c_void_p),
                ("os_val", C.c_void_p), ("ver_val", C.c_void_p)]


class CygState(C.Structure):
    """struct cyg_state (device pointers, canonical layout)"""
    _fields_ = [("dev", C.c_void_p), ("ckpt", C.c_void_p), ("blocked", C.c_void_p), ("extra", C.c_void_p),
                ("scal", C.c_void_p), ("logs", C.c_void_p)]


class CygActions(C.Structure):
    """struct cyg_actions"""
    _fields_ = [("hdr", C.c_void_p), ("mask", C.c_void_p), ("order", C.c_void_p), ("order_stride", C.c_int32),
                ("n_groups", C.c_int32)]


class CygStepOut(C.Structure):
    """struct cyg_step_out"""
    _fields_ = [("raw_reward", C.c_void_p), ("shaped_reward", C.c_void_p), ("done", C.c_void_p),
                ("pre_masks", C.c_void_p), ("obs", C.c_void_p), ("obs_mode", C.c_int32)]


class CygRolloutArgs(C.Structure):
    """struct cyg_rollout_args"""
    _fields_ = [("hdr", C.c_void_p), ("mask", C.c_void_p), ("base_line", C.c_void_p), ("n_steps", C.c_int32), ("n_rows", C.c_int32),
                ("row_base", C.c_int64), ("envs_per_row", C.c_int32), ("reserved", C.c_int32), ("returns", C.c_void_p), ("block_order", C.c_void_p)]


EXPORTS = ["cyg_version", "cyg_last_error", "cyg_create", "cyg_destroy", "cyg_set_base_line", "cyg_set_base_line_per_env", "cyg_set_base_line_per_env_steps", "cyg_internal_words",
           "cyg_bind", "cyg_set_detectors", "cyg_fit_detectors", "cyg_import_state", "cyg_export_state", "cyg_step", "cyg_step_multi", "cyg_rollout", "cyg_unpack_actions", "cyg_pack_done", "cyg_block_envs", "cyg_set_env_id_stride", "cyg_randomize", "cyg_rebuild_graph_cache", "cyg_sample_actions", "cyg_sample_actions_ordered",
           "cyg_observe", "cyg_group_actions", "cyg_launch_count", "cyg_set_debug_cycles"]


class CygError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cygym_b200 error {code}: {msg}")
        self.code = code


SPILL_LIMIT = 256   # bytes of spill stores tolerated in the config-C3 step kernel (cyg_step_kernel<4, true>)
THREAD_CAPS = (640, 512)  # threads per CTA -> 93 / 127 registers per thread at one CTA per SM (640 measured fastest)


def _step_kernel_spill(ptxas_log, mangled="_Z15cyg_step_kernelILi4ELb1ELb0ELb0EEv10StepParams"):
    """Bytes of spill stores ptxas reports for the plain-step W = 4 kernel (None when the log has no such entry)."""
    import re
    m = re.search(r"Function properties for " + re.escape(mangled) + r"\s+\d+ bytes stack frame, (\d+) bytes spill stores", ptxas_log)
    return int(m.group(1)) if m else None


def compile_units(out_path, widths=PLANE_WIDTHS, extra=(), obj_dir=None, verbose=False):
    """nvcc -c one object per plane width (in parallel, each without --split-compile: the register allocation of a
    kernel then does not depend on what else is being compiled) plus the C-ABI unit, then link them into `out_path`.
    Returns the ptxas -v log of the W = 4 unit."""
    nvcc = os.environ.get("NVCC", "nvcc")
    obj_dir = obj_dir or os.path.join(_HERE, "_build")
    os.makedirs(obj_dir, exist_ok=True)
    tag = os.path.splitext(os.path.basename(out_path))[0]
    jobs = []
    for w in list(widths) + [None]:
        obj = os.path.join(obj_dir, f"{tag}_{'api' if w is None else 'w%d' % w}.o")
        cmd = [nvcc] + NVCC_FLAGS + list(extra) + ["-Xptxas", "-v", "-c", "-o", obj, _SRC]
        if w is not None:
            cmd.insert(-4, f"-DCYG_TU_W={w}")
            if w > 4:
                cmd[-4:-4] = ["--split-compile", "0"]  # the generic kernel: compile time matters, its registers do not
        jobs.append((w, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    logs, objs = {}, []
    for w, obj, pr in jobs:
        out, err = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed (unit {w}):\n" + out + err)
        logs[w] = err
        objs.append(obj)
    r = subprocess.run([nvcc, "-shared", "-o", out_path] + objs, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    if verbose:
        for w in logs:
            print(f"---- unit {w}\n{logs[w]}")
    return logs.get(4, "")


def build(force=False, verbose=False):
    """Compile cygym_b200/csrc/cyg_kernels.cu for sm_100a into cygym_b200/libcygym_b200.so.

    The step kernel runs one CTA per SM; 640 threads (93 registers per thread, no spills) measured fastest on B200
    (896 threads / 72 registers sat next to a ptxas cliff: ~90 bytes vs ~2 KB of spills in the warp-per-env routines).
    The recipe checks `-Xptxas -v` and, should the config-C3 kernel spill more than SPILL_LIMIT bytes, rebuilds with
    the next lower thread cap (more registers per thread)."""
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(d) for d in _DEPS):
        return LIB_PATH
    log = ""
    for cap in THREAD_CAPS:
        w4 = compile_units(LIB_PATH, extra=[f"-DCYG_MAX_BLOCK_THREADS={cap}"], verbose=verbose)
        spill = _step_kernel_spill(w4)
        log += f"[cygym_b200 build] {cap} threads per CTA: cyg_step_kernel<4, plain> spills {spill} bytes\n"
        if spill is None or spill <= SPILL_LIMIT:
            break
    with open(LIB_PATH + ".buildlog", "w") as f:
        f.write(log)
    if verbose:
        print(log)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(cygym_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.cyg_version.restype = C.c_int
        L.cyg_last_error.restype = C.c_char_p
        L.cyg_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(CygConfig), C.POINTER(CygNetwork), C.c_int32, C.c_int32, C.c_int32]
        L.cyg_destroy.argtypes = [C.c_void_p]
        L.cyg_set_base_line.argtypes = [C.c_void_p, C.c_int32]
        L.cyg_set_base_line_per_env.argtypes = [C.c_void_p, C.c_void_p]
        L.cyg_set_base_line_per_env_steps.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
        L.cyg_internal_words.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.cyg_bind.argtypes = [C.c_void_p, C.c_void_p]
        L.cyg_set_detectors.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.cyg_fit_detectors.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.cyg_import_state.argtypes = [C.c_void_p, C.POINTER(CygState), C.c_void_p]
        L.cyg_export_state.argtypes = [C.c_void_p, C.POINTER(CygState), C.c_void_p]
        L.cyg_step.argtypes = [C.c_void_p, C.POINTER(CygActions), C.c_uint32, C.POINTER(CygStepOut), C.c_void_p]
        L.cyg_step_multi.argtypes = [C.c_void_p, C.POINTER(CygActions), C.c_int32, C.c_uint32, C.POINTER(CygStepOut), C.c_void_p]
        L.cyg_rollout.argtypes = [C.c_void_p, C.POINTER(CygRolloutArgs), C.c_uint32, C.c_void_p]
        L.cyg_set_env_id_stride.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
        L.cyg_block_envs.argtypes = [C.c_void_p, C.POINTER(C.c_int32)]
        L.cyg_unpack_actions.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.cyg_pack_done.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.cyg_randomize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.cyg_rebuild_graph_cache.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.cyg_sample_actions.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.cyg_sample_actions_ordered.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.cyg_observe.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.cyg_group_actions.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
        L.cyg_launch_count.argtypes = [C.c_void_p]
        L.cyg_launch_count.restype = C.c_int64
        L.cyg_set_debug_cycles.argtypes = [C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise CygError(rc, lib().cyg_last_error().decode(errors="replace"))


def make_config(cfg, E, seed=0, xcap=16, base_line="Nash", tri_mode=2, tri_high=5, log_cap=0):
    """cfg: the attribute dict of a Network (network.py) -> struct cyg_config."""
    c = CygConfig()
    c.M, c.E, c.X, c.n_exploits, c.xcap = cfg["M"], E, cfg["X"], cfg["n_exploits"], xcap
    c.num_of_device, c.min_network_size = cfg["numOfDevice"], cfg["Min_network_size"]
    c.evolve_period = cfg["evolve_period"]
    c.wl_period_base, c.wl_period_max, c.wl_cap = cfg["workload_period_base"], cfg["workload_period_max"], cfg["workload_cap"]
    c.scaling_vulnerability, c.turbo, c.zero_day = cfg["scaling_vulnerability"], cfg["turbo"], cfg["zero_day"]
    c.zero_day_mask = cfg["zero_day_mask"]
    c.att_space_n, c.def_space_n, c.default_high = cfg["att_space_n"], cfg["def_space_n"], cfg["default_high"]
    c.n_app_ids = cfg.get("n_app_ids", 0)
    c.base_line = BASE_LINES.get(base_line, BL_OTHER)
    c.tri_high = tri_high
    c.log_cap = int(log_cap)
    c.work_scale, c.comp_scale, c.def_scale, c.gamma = cfg["work_scale"], cfg["comp_scale"], cfg["def_scale"], cfg["gamma"]
    c.thr_p_add = DT.bernoulli_threshold(cfg["p_add"])
    c.thr_p_attacker = DT.bernoulli_threshold(cfg["p_attacker"])
    for i, t in enumerate(DT.poisson_table(cfg["lambda_events"])):
        c.poisson_tab[i] = t
    for i, t in enumerate(DT.triangular_ceil_table(tri_mode, tri_high)):
        c.tri_tab[i] = t
    c.seed = seed
    c.turbo_frac_clients = cfg.get("turbo_fraction_clients", 0.05)
    c.turbo_frac_servers = cfg.get("turbo_fraction_servers", 0.02)
    c.turbo_max_clients = cfg.get("turbo_max_clients", 200)
    c.turbo_max_servers = cfg.get("turbo_max_servers", 40)
    c.turbo_ramp_steps = cfg.get("turbo_ramp_steps", 200)
    return c
