"""Device-side glue for the reference's IPPO / MAPPO style rollouts (IPPO.py:433-805, MAPPO.py same lines):
role visibility masks (IPPO.py:74-96) and the per-device-type -> grouped-action encoding (IPPO.py:559-570), for B
envs at once, as torch ops on the env's own device buffers.  The grouped step itself is
VectorCyberDefenseEnv.step_grouped (volt_typhoon_env.py:694-779)."""
import torch

from .vector_env import ActionBatch, VectorCyberDefenseEnv, header_rows, pack_device_mask

P_COMP, P_KNOWN, P_NYA, P_OWNED = 0, 1, 2, 3   # bit-plane ids of the internal record (cyg_core.cuh)
REC_PLANES = 16
SINGLE_DEVICE_TYPES = (11, 12)                  # IPPO.py:27


def plane_bits(env: VectorCyberDefenseEnv, plane):
    """bool [B, M]: one bit-plane of every env, unpacked on the device."""
    Wi = env.W if env.M <= 128 else 64           # plane width of the internal record (padded for large networks)
    words = env.records[:, REC_PLANES + plane * Wi: REC_PLANES + (plane + 1) * Wi]
    shifts = torch.arange(32, device=words.device, dtype=torch.int32)
    bits = (words.unsqueeze(-1) >> shifts) & 1
    return bits.reshape(env.B, Wi * 32)[:, : env.M].bool()


def visibility_mask(env: VectorCyberDefenseEnv, role):
    """float32 [B, M] in {0, 1} (build_visibility_mask, IPPO.py:74-96)."""
    nya, owned = plane_bits(env, P_NYA), plane_bits(env, P_OWNED)
    v = ~nya & owned
    if role == "attacker":
        v = v & plane_bits(env, P_KNOWN)
    return v.float()


class GroupedBatch:
    """The action groups of one grouped step, stacked: hdr [G, B, 4], mask [G, B, W] int32 device tensors (what
    cyg_step(CYG_STEP_GROUPED) reads); iterating yields the per-group ActionBatch views."""

    def __init__(self, hdr, mask):
        self.hdr, self.mask, self.order = hdr, mask, None

    def __len__(self):
        return int(self.hdr.shape[0])

    def __getitem__(self, g):
        return ActionBatch(self.hdr[g], self.mask[g])

    def __iter__(self):
        return (self[g] for g in range(len(self)))


_ROLES = {None: 0, "all": 0, "defender": 1, "attacker": 2}


def grouped_actions(env: VectorCyberDefenseEnv, per_dev_types, role, exp_idx, app_idx, mode, n_types, noop, visible=None,
                    single_choice=None, out: GroupedBatch = None):
    """The grouped action of IPPO.py:559-570 for B envs in ONE kernel (cyg_group_actions): every device drew a type
    (per_dev_types int [B, M]); the devices the role sees (build_visibility_mask, IPPO.py:74-96, read from the env's
    bit-planes; role None = all) and, when given, the caller's own `visible` [B, M] mask are grouped by type into the
    n_types - 1 groups of one step_grouped() call.  Returns a GroupedBatch (pass it to env.step_grouped)."""
    import ctypes as C
    from . import _capi as K
    m = 1 if mode in (1, "attacker") else 0
    G = n_types - 1
    dev = env.device
    if out is None:
        out = GroupedBatch(torch.empty(G, env.B, 4, dtype=torch.int32, device=dev), torch.empty(G, env.B, env.W, dtype=torch.int32, device=dev))
    t = per_dev_types.to(dev, torch.int32).contiguous()
    e = exp_idx.to(dev, torch.int32).contiguous()
    a = app_idx.to(dev, torch.int32).contiguous()
    v = None if visible is None else (visible > 0.5 if visible.dtype.is_floating_point else visible != 0).to(dev, torch.uint8).contiguous()
    sc = None if single_choice is None else single_choice.to(dev, torch.int32).contiguous()
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())
    K.check(env.L.cyg_group_actions(env.h, m, _ROLES[role], p(t), p(v), p(e), p(a), p(sc), int(n_types), int(noop), p(out.hdr), p(out.mask), env._s()))
    out._hold = (t, e, a, v, sc)
    return out


def grouped_actions_from_types(env: VectorCyberDefenseEnv, per_dev_types, visible, exp_idx, app_idx, mode, n_types, noop,
                               single_choice=None):
    """per_dev_types: int [B, M] sampled action type per device; visible: [B, M] (>0.5 = counts);
    exp_idx, app_idx: int [B].  Returns the list of n_types - 1 ActionBatch groups of IPPO.py:559-570 in ascending
    type order; a type with no device in an env becomes that env's no-op group (what the reference skips).
    single_choice: optional int [B, len(SINGLE_DEVICE_TYPES)] device to keep for the single-device types (the
    reference picks with random.choice); default = the lowest listed device."""
    B, M, W = env.B, env.M, env.W
    m = 1 if mode in (1, "attacker") else 0
    vis = visible > 0.5
    groups = []
    for t in range(n_types):
        if t == noop:
            continue
        sel = vis & (per_dev_types == t)
        if t in SINGLE_DEVICE_TYPES:
            if single_choice is not None:
                pick = single_choice[:, SINGLE_DEVICE_TYPES.index(t)].long().clamp(0, M - 1)
                keep = torch.zeros_like(sel)
                keep[torch.arange(B, device=sel.device), pick] = True
                sel = sel & keep
            else:
                first = torch.cumsum(sel.int(), dim=1) == 1
                sel = sel & first
        n_dev = sel.sum(1).to(torch.int32)
        atype = torch.where(n_dev > 0, torch.full_like(n_dev, t), torch.full_like(n_dev, noop))
        groups.append(ActionBatch(header_rows(atype, m, exp_idx, n_dev, app_idx), pack_device_mask(sel, W).contiguous()))
    return groups
