"""Batched payoff-matrix evaluation: the GPU counterpart of DoubleOracle.build_payoff_matrices /
simulate_game (do_agent.py:1666-1870, :1875-2089) for the non-neural Strategy flavours
(strategy.py:25-60): a baseline name, a fixed action sequence, or the no-op.

Every (defender strategy i, attacker strategy j) pair is rolled out `n_rollouts` times for
`steps_per_episode` alternating turns (defender on even t, do_agent.py:2053).  Rollouts are
independent, so they shard over ranks with no per-step collective: rank r runs rollouts
[r*N/world, (r+1)*N/world) of every pair and holds a partial [n_def, n_att, 10] sum; ONE
all-reduce(sum) of that tensor (NCCL over NVLink on GPUs, gloo in the CPU tests) finishes the
evaluation.  The 10 columns are simulate_game's return tuple (do_agent.py:2078-2089).

Defender action 10 trains the env's IsolationForest and a later action 5 scans with it (volt:945-962, :1020-1069).  Both
evaluators serve strategies that train only with train_detectors=True: the envs then keep a hop-log ring and detector
slots, and every pending env is fitted on the device between turns (VectorCyberDefenseEnv.fit_detectors, seeded by
detector_fit_seeds()).  Without it, a strategy that trains gets the stub scan -- no un-compromise, no stall -- and a
sticky CYG_FL_ERR_DETECTOR bit on the env, which the default path does not read.
"""
import numpy as np

from . import _capi as K

COLUMNS = ("defender_return", "attacker_return", "compromised_fraction", "jobs_completed", "scan_count",
           "defensive_cost", "checkpoint_count", "revert_count", "edges_blocked", "edges_added")
_INFO_OF_COLUMN = ("Compromised_devices", "work_done", "Scan_count", "defensive_cost", "checkpoint_count", "revert_count",
                   "Edges Blocked", "Edges Added")  # env.info() keys of COLUMNS[2:]
# the counters the reference zeroes before a rollout (do_agent.py:2038-2045)
_ROLLOUT_RESET = (K.S_STEP, K.S_DEF_STEP, K.S_ATT_STEP, K.S_WORK, K.S_CKPT, K.S_DEFCOST, K.S_CLEANCOST, K.S_REVERT, K.S_SCAN)
DETECTOR_LOG_CAP = K.DET_WINDOW  # hop-log records per env with train_detectors=True: the most a fit or a scan reads
_ERR_NAMES = ((K.FL_ERR_BUSY, "CYG_FL_ERR_BUSY"), (K.FL_ERR_XCAP, "CYG_FL_ERR_XCAP"), (K.FL_ERR_DETECTOR, "CYG_FL_ERR_DETECTOR"),
              (0x80, "error bit 0x80"))


def _columns(def_r, att_r, info):
    """The 10 COLUMNS of every env as float64 [B] tensors: the defender / attacker returns and env.info() counters."""
    return [def_r, att_r] + [info[k].double() for k in _INFO_OF_COLUMN]


class Strategy:
    """The flavours of strategy.Strategy the evaluators serve: baseline_name | actions (fixed sequence) | actor (a torch
    module: the parametric DDPG best responses, Actor of do_agent.py:357-371; evaluate_payoff_matrix_batched only) |
    none of them (no-op).  A defender sequence with a type-10 action, and any defender actor (its type slice may pick
    10), trains the detector: evaluate such strategies with train_detectors=True, or their scans run the stub and leave
    CYG_FL_ERR_DETECTOR on the env."""

    def __init__(self, baseline_name=None, actions=None, actor=None):
        self.baseline_name = baseline_name
        self.actions = list(actions) if actions is not None else None
        self.actor = actor

    def can_train(self):
        """Whether this strategy, as the defender, may execute action 10 (train the detector).  A baseline never does."""
        if self.actor is not None:
            return True
        return self.baseline_name is None and any(a is not None and int(a[0]) == 10 for a in (self.actions or ()))

    def decide(self, t_step):
        """(action, base_line to set or None) -- _strategy_decide_action (do_agent.py:707-764)."""
        if self.actor is not None:
            raise NotImplementedError("parametric strategies act on observations: evaluate_payoff_matrix_batched()")
        if self.baseline_name is not None:
            return None, self.baseline_name
        if self.actions:
            return self.actions[t_step % len(self.actions)], None
        return None, "Nash"


def shard_range(total, rank, world):
    """Contiguous split of `total` items over `world` ranks (the first total % world ranks get one more)."""
    base, extra = divmod(int(total), int(world))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def detector_fit_seeds(seed, env_ids, turn):
    """The seed of the detector fit of every env after turn `turn`: int64 tensor [n] of uint32 values (what
    fit_detectors() takes), on env_ids' device.  env_ids: int64 tensor of evaluation env ids g = pair * n_rollouts +
    rollout.  The reference fits with random_state=None, i.e. from numpy's global stream as it stands, so any fixed rule
    is a valid sample of its behaviour; this one depends on (seed, g, turn) alone -- not on the rank, the number of
    ranks, steps_per_launch or the evaluator -- so that every layout of an evaluation gives the same result."""
    import torch
    M = 0xFFFFFFFF

    def mul32(h, c):  # (h * c) mod 2^32 with every product below 2^48 (no int64 overflow)
        return ((h & 0xFFFF) * c + ((((h >> 16) * c) & 0xFFFF) << 16)) & M

    def fmix(h):  # MurmurHash3's 32-bit finaliser
        h = h ^ (h >> 16)
        h = mul32(h, 0x85EBCA6B)
        h = h ^ (h >> 13)
        h = mul32(h, 0xC2B2AE35)
        return h ^ (h >> 16)

    g = torch.as_tensor(env_ids).to(torch.int64)
    h = fmix(torch.full_like(g, (int(seed) + 0x9E3779B9) & M))
    h = fmix(h ^ (g & M))
    h = fmix(h ^ ((g >> 32) & M))
    return fmix(h ^ ((int(turn) + 0x7F4A7C15) & M))


def _check_error_bits(flags_of_envs):
    """train_detectors=True: raise when an env ended with a sticky CYG_FL_ERR_* bit (a scan without a fitted detector,
    a full busy set or extra-edge list), naming the bits and how many envs carry each."""
    import torch
    err = torch.cat([f.reshape(-1) & K.FL_ERR_MASK for f in flags_of_envs]) if flags_of_envs else None
    if err is None or not bool(err.any()):
        return
    found = [f"{name} on {int(((err & bit) != 0).sum())} envs" for bit, name in _ERR_NAMES if bool(((err & bit) != 0).any())]
    raise RuntimeError("payoff evaluation with train_detectors=True: envs ended with sticky error bits: " + ", ".join(found))


def reduce_payoff(partial_sums, n_rollouts, steps_per_episode, group=None):
    """All-reduce the per-rank [n_def, n_att, 10] sums and turn them into simulate_game's averages."""
    import torch
    import torch.distributed as dist
    t = partial_sums.clone()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    out = t / float(n_rollouts)
    out[..., 2] = out[..., 2] / max(1.0, float(steps_per_episode))  # avg_compromised_fraction (do_agent.py:2076)
    return out


def evaluate_payoff_matrix(network, def_strategies, att_strategies, n_rollouts, steps_per_episode=100, seed=0,
                           device="cuda:0", rank=0, world=1, xcap=16, group=None, reduce=True, train_detectors=False):
    """Returns a float64 tensor [n_def, n_att, 10] (averages) on `device`.

    train_detectors=True: every env keeps a hop-log ring of DETECTOR_LOG_CAP records (8 KB per env) and, where the
    defender strategy can train (Strategy.can_train), a detector slot (24.6 KB per env); after every defender turn the
    pending envs are fitted on the device with detector_fit_seeds(seed, env ids, turn), and the call raises RuntimeError
    when an env ends with a sticky CYG_FL_ERR_* bit.  Without it, a strategy that trains gets the stub scan and a sticky
    CYG_FL_ERR_DETECTOR bit, and the result does not say so."""
    import torch
    from .vector_env import ActionBatch, VectorCyberDefenseEnv
    lo, hi = shard_range(n_rollouts, rank, world)
    nloc = hi - lo
    nd, na = len(def_strategies), len(att_strategies)
    sums = torch.zeros(nd, na, len(COLUMNS), dtype=torch.float64, device=device)
    flags = []
    if nloc > 0:
        M = network.M
        for i, ds in enumerate(def_strategies):
            fits = train_detectors and ds.can_train()
            for j, as_ in enumerate(att_strategies):
                # env ids are unique per (pair, rollout) so that every rollout has its own draw stream
                id0 = (i * na + j) * n_rollouts + lo
                env = VectorCyberDefenseEnv(network, nloc, device=device, seed=seed, env_id0=id0, xcap=xcap,
                                            log_cap=DETECTOR_LOG_CAP if train_detectors else 0, detector_slots=nloc if fits else 0)
                g = id0 + torch.arange(nloc, device=env.device) if fits else None
                env.randomize_compromise_and_ownership()
                for slot in _ROLLOUT_RESET:
                    env.scalars[:, slot] = 0
                def_r = torch.zeros(nloc, dtype=torch.float64, device=device)
                att_r = torch.zeros(nloc, dtype=torch.float64, device=device)
                for t in range(steps_per_episode):
                    mode = t & 1
                    action, bl = (ds if mode == 0 else as_).decide(t)
                    if bl is not None and bl != env.base_line:
                        env.set_base_line(bl)
                    hdr, mask, order = ActionBatch.pack([action], mode, M, order_form=False) if (
                        action is None or list(action[2]) == sorted(set(action[2]))) else ActionBatch.pack([action], mode, M, order_form=True)
                    ab = env.to_device(np.repeat(hdr, nloc, 0), np.repeat(mask, nloc, 0),
                                       None if order is None else np.repeat(order, nloc, 0))
                    raw, _, _ = env.step(ab)
                    if mode == 0:
                        def_r += raw.double()
                        if fits and t < steps_per_episode - 1:
                            env.fit_detectors(detector_fit_seeds(seed, g, t))
                    else:
                        att_r += raw.double()
                sums[i, j] = torch.stack([c.sum() for c in _columns(def_r, att_r, env.info())])
                if train_detectors:
                    flags.append(env.scalars[:, K.S_FLAGS].clone())
                env.close()
    if train_detectors:
        _check_error_bits(flags)
    if not reduce:
        return sums
    return reduce_payoff(sums, n_rollouts, steps_per_episode, group=group)


def decode_actions(raw, mode, n_types, M, X, n_app, W):
    """DoubleOracle.decode_action (do_agent.py:935-998, the epsilon-free branch: evaluation) for a batch of actor outputs
    raw [N, n_types + M + X + n_app] on the device -> (hdr [N, 4], mask [N, W]) int32.  action_type = argmax of the type
    slice, device_indices = where(slice > 0) (ascending: the set form), exploit and app index = argmax of their slices."""
    import torch
    from .vector_env import header_rows, pack_device_mask
    m = 1 if mode in (1, "attacker") else 0
    at = raw[:, :n_types].argmax(1).to(torch.int32)
    dev = raw[:, n_types:n_types + M] > 0
    ex = raw[:, n_types + M:n_types + M + X].argmax(1).to(torch.int32)
    app = raw[:, n_types + M + X:n_types + M + X + n_app].argmax(1).to(torch.int32) if n_app > 0 else torch.zeros_like(at)
    return header_rows(at, m, ex, dev.sum(1), app), pack_device_mask(dev, W).contiguous()


def _is_set_form(action):
    """Whether an action's device_indices can travel as a set: None, or an ascending duplicate-free list."""
    return action is None or [int(d) for d in action[2]] == sorted(set(int(d) for d in action[2]))


def _strategy_rows(def_strategies, att_strategies, T, M):
    """The distinct action rows of every strategy, packed once on the host, and which row each strategy plays on each
    turn: per side (hdr rows [R, 4], mask rows [R, W], row index [T, S], base_line code [S] (255 = the strategy does not
    touch env.base_line), order rows [R, M] uint16).  A fixed sequence of L actions is L rows indexed by t % L.

    A defender row whose list is not ascending and duplicate-free (the draw order of the sequences DoubleOracle samples,
    do_agent.py:1001-1013) is ORDERED: its order row holds the list, and the kernel visits the devices in that order.
    Every other row is a set: its order row starts with ORDER_NONE.  Attacker rows are sets whatever their list
    (attacker_act reads the exploits and the sources, never device_indices)."""
    from .vector_env import ActionBatch
    out = []
    for mode, sts in ((0, def_strategies), (1, att_strategies)):
        hs, ms, os_, first, length, bls, n_rows = [], [], [], [], [], [], 0
        for st in sts:
            key = (mode, M)
            cached = st.__dict__.setdefault("_packed_rows", {}).get(key)  # a strategy is evaluated again and again as the matrices grow
            if cached is None:
                if st.actor is not None:
                    acts, bl = [None], 255
                elif st.baseline_name is not None:
                    acts, bl = [None], K.BASE_LINES.get(st.baseline_name, K.BL_OTHER)
                elif st.actions:
                    acts, bl = list(st.actions), 255
                else:
                    acts, bl = [None], K.BASE_LINES["Nash"]
                h, m, o = ActionBatch.pack(acts, mode, M, order_form=True)  # the mask holds the set of any list
                ordered = np.array([mode == K.MODE_DEFENDER and not _is_set_form(a) for a in acts], bool)
                o[~ordered] = K.ORDER_NONE
                cached = st._packed_rows[key] = (h.view(np.int32), m.view(np.int32), bl, o)
            h, m, bl, o = cached
            first.append(n_rows); length.append(len(h)); bls.append(bl)
            n_rows += len(h)
            hs.append(h); ms.append(m); os_.append(o)
        t = np.arange(T)[:, None]
        ridx = np.asarray(first)[None, :] + t % np.asarray(length)[None, :]
        out.append((np.concatenate(hs), np.concatenate(ms), ridx.astype(np.int64), np.asarray(bls, np.uint8), np.concatenate(os_)))
    return out


_ORDER_NONE_I16 = K.ORDER_NONE - 0x10000  # ORDER_NONE as the int16 the device tables hold


def _order_arrays(hdr, mask, ord_rows):
    """The order array of a closed-loop step whose batch has ordered rows (cyg_step applies an order array to every env):
    ord_rows [N, M] int16 where the env's row is ordered, the ascending list of its mask where the row is a set (the
    set read in order).  Width = the longest list of the batch.  int16 [N, width] on the device."""
    import torch
    N, M = ord_rows.shape
    width = max(1, int((hdr[:, 2] & 0xFFFF).max()))
    bits = (mask.to(torch.int32)[:, :, None] >> torch.arange(32, device=mask.device, dtype=torch.int32)) & 1  # [N, W, 32]
    ids = torch.arange(bits.shape[1] * 32, device=mask.device, dtype=torch.int32)
    asc = torch.where(bits.view(N, -1).bool(), ids, 0x7FFF).sort(dim=1).values[:, :M]  # set devices first, ascending
    out = torch.where((ord_rows[:, :1] != _ORDER_NONE_I16), ord_rows.to(torch.int32), asc)
    pad = max(0, width - M)
    return torch.nn.functional.pad(out, (0, pad))[:, :width].to(torch.int16).contiguous()


_ENV_CACHE = {}


def _cached_env(network, nloc, lo, device, seed, xcap, log_cap=0, detector_slots=0):
    """The evaluation's env batch, kept between calls (a Double-Oracle run evaluates the same network again and again:
    build_payoff_matrices, do_agent.py:1666-1870): re-creating 1 M envs costs ~15 ms of allocation and table upload per
    call, a reset() of the kept ones ~2 ms.  The hop-log ring and the detector slots are part of the key (a kept handle
    without a ring never serves an evaluation that trains); a kept handle's envs give their slots back."""
    from .vector_env import VectorCyberDefenseEnv
    key = (id(network), int(nloc), int(lo), str(device), int(seed), int(xcap), int(log_cap), int(detector_slots))
    env = _ENV_CACHE.get(key)
    if env is None:
        for k in list(_ENV_CACHE):
            _ENV_CACHE.pop(k).close()
        env = _ENV_CACHE[key] = VectorCyberDefenseEnv(network, nloc, device=device, seed=seed, env_id0=lo, xcap=xcap,
                                                      log_cap=log_cap, detector_slots=detector_slots)
    else:
        env.reset()
        env.set_base_line_per_env(None)
        env.release_detectors()
    return env


# rough SM cycles per env of one turn by executed action type (measured on a B200 with a per-env cycle counter the step
# kernel no longer has, see git history: warp-per-env tasks shared by the 20 warps of a CTA, thread-per-env types by
# 14 warps of 32 lanes); only the ORDER of the blocks depends on them
_DEF_PER_DEVICE = {6: 11.0, 9: 9.0, 1: 3.75, 3: 2.75, 4: 2.25}
_TURN_BASE, _ATTACK_COST, _BASELINE_COST = 25.0, 185.0, 60.0


def _block_order(env, sides, i_of_pair, j_of_pair, pair_of_env, T):
    """CTA indices of the rollout launch, most expensive first (longest processing time first): the blocks of a launch
    hold one to four strategy pairs each and the pairs differ by an order of magnitude in cost (a sequence of block /
    unblock actions over 40 devices against the no-op), so the launch used to end with whichever expensive blocks
    started last.  The estimate needs no measurement: action types and list lengths of the strategies' rows."""
    import torch
    from .vector_env import decode_header
    cost_side = []
    for mode, (h, _, ridx, bls, _) in enumerate(sides):
        f = decode_header(h)
        t = (f.atype & 0xFF).astype(np.int64)
        n = f.n_dev.astype(np.float64)
        if mode == 0:
            c = _TURN_BASE + np.array([_DEF_PER_DEVICE.get(int(x), 0.0) for x in t]) * n
        else:
            c = _TURN_BASE + np.where(t == 1, _ATTACK_COST, 0.0)
        c = c + np.where(t == K.ATYPE_NONE, _BASELINE_COST, 0.0)  # a baseline acts by itself (volt:836-853)
        turns = np.arange(mode, T, 2)
        cs = c[ridx[turns]].mean(axis=0) if len(turns) else np.zeros(ridx.shape[1])  # [n strategies]
        idle = np.isin(bls, [K.BASE_LINES["No Defense"], K.BASE_LINES["No Attack"]])
        cost_side.append(np.where(idle, _TURN_BASE, cs))
    pair_cost = torch.from_numpy(cost_side[0][i_of_pair] + cost_side[1][j_of_pair]).to(pair_of_env.device)
    nb = env.block_envs()
    n_blocks = (env.B + nb - 1) // nb
    per_slot = pair_cost[pair_of_env]
    pad = n_blocks * nb - env.B
    if pad:
        per_slot = torch.cat([per_slot, per_slot.new_zeros(pad)])
    return torch.argsort(per_slot.view(n_blocks, nb).sum(1), descending=True, stable=True).to(torch.int32)


def evaluate_payoff_matrix_batched(network, def_strategies, att_strategies, n_rollouts, steps_per_episode=100, seed=0,
                                   device="cuda:0", rank=0, world=1, xcap=16, group=None, reduce=True, steps_per_launch=None,
                                   train_detectors=False):
    """Same result as evaluate_payoff_matrix(), with ALL (pair, rollout) combinations in one batch: the flattened
    index g = pair * n_rollouts + rollout is split over the ranks (env id == g, so the draw streams do not depend on the
    number of ranks): every rank takes the same slice of rollouts of every pair when n_rollouts divides evenly (balanced
    work), a contiguous slice of g otherwise.

    Strategies that need no observation (baseline names, fixed sequences, the no-op) become per-PAIR tables of action
    rows and base_line codes for all turns, uploaded ONCE and gathered inside the kernel (cyg_rollout): the whole
    100-turn evaluation is `ceil(T / steps_per_launch)` launches (default: one) with no host work in between, the
    records staying in shared memory between the turns of a launch and the returns summed per env on the device.

    With a parametric strategy (Strategy(actor=...): the DDPG best responses) on either side the rollout is closed
    loop: per turn one observation launch, one batched actor forward per parametric strategy on the rows of its envs,
    decode_actions() on the device, one step launch.

    Fixed sequences whose defender actions list their devices in draw order (DoubleOracle's sampled strategies,
    do_agent.py:1001-1013) are evaluated as they are: those rows carry their list in an order table (_strategy_rows),
    the table-driven path launches cyg_rollout_ordered (an ordered row's env runs its action with one thread, in list
    order), and the closed-loop path passes an order array to the defender turns that have ordered rows.  An evaluation
    without such a row takes exactly the launches it took before.

    train_detectors=True serves defender strategies that train the detector (action 10; Strategy.can_train): the envs
    keep a hop-log ring of DETECTOR_LOG_CAP records, and this rank's envs whose defender can train get a detector slot
    each.  Memory at C5 shape (2^20 envs on one GPU): the ring is handle-wide, 2000 x 4 B x 2^20 = 8.4 GB; a slot is
    24.6 KB per env that can train.  A detector cannot be fitted inside a launch, so the table-driven path also ends a
    launch after every turn t < T - 1 at which some pair's defender row executes type 10 (its base_line is Nash), and
    fits every pending env on the device (fit_detectors, seeds detector_fit_seeds(seed, g, t)) before the next launch;
    the closed-loop path fits after every defender turn.  The result equals the same rollouts with those host fits, for
    any steps_per_launch and sharding.  After the last turn the call raises RuntimeError when an env carries a sticky
    CYG_FL_ERR_* bit.  Without the flag, a strategy that trains gets the stub scan and a sticky CYG_FL_ERR_DETECTOR bit,
    and the result does not say so."""
    import torch
    from .vector_env import ActionBatch, VectorCyberDefenseEnv
    nd, na = len(def_strategies), len(att_strategies)
    P, T = nd * na, int(steps_per_episode)
    M, W = network.M, network.W
    any_nn = any(st.actor is not None for st in list(def_strategies) + list(att_strategies))
    # Sharding.  Table-driven rollouts with n_rollouts divisible by the ranks: rank r takes rollouts [r * run, (r + 1) *
    # run) of EVERY pair (strided env ids, cyg_set_env_id_stride) -- every rank steps the same mix of cheap and expensive
    # pairs.  Otherwise a contiguous slice of the flattened (pair, rollout) index.  Env ids, hence all sums, are the same.
    strided = world > 1 and not any_nn and W <= 4 and n_rollouts % world == 0
    if strided:
        run = n_rollouts // world
        lo, nloc = rank * run, P * run
    else:
        lo, hi = shard_range(P * n_rollouts, rank, world)
        nloc = hi - lo
    sums = torch.zeros(P, len(COLUMNS), dtype=torch.float64, device=device)
    if nloc > 0:
        i_of_pair = np.arange(P) // na
        j_of_pair = np.arange(P) % na
        n_slots = 0
        if train_detectors:  # this rank's envs whose defender strategy can train
            trains = np.array([st.can_train() for st in def_strategies], bool)[i_of_pair]
            if strided:
                n_slots = run * int(trains.sum())
            else:
                n_slots = int(np.bincount(np.arange(lo, lo + nloc) // n_rollouts, minlength=P)[trains].sum())
        env = _cached_env(network, nloc, lo, device, seed, xcap, DETECTOR_LOG_CAP if train_detectors else 0, n_slots)
        env.set_env_id_stride(run if strided else 0, n_rollouts)
        g_of_env = lo + env.env_index_of_slot()
        pair_of_env = g_of_env // n_rollouts
        env.randomize_compromise_and_ownership()
        for slot in _ROLLOUT_RESET:
            env.scalars[:, slot] = 0
        # per-pair tables, assembled on the device from the strategies' packed rows: the moving side's row of every turn,
        # and the base_line each pair's env carries on that turn (a strategy that sets no base_line leaves it as the
        # other player's last baseline left it, do_agent.py:716-719)
        sides = _strategy_rows(def_strategies, att_strategies, T, M)
        tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
        of_pair = (tt(i_of_pair), tt(j_of_pair))
        hdr_side = [tt(h)[tt(r)][:, of_pair[m_]] for m_, (h, _, r, _, _) in enumerate(sides)]    # [T, P, 4] per side
        mask_side = [tt(m)[tt(r)][:, of_pair[m_]] for m_, (_, m, r, _, _) in enumerate(sides)]  # [T, P, W]
        even = (torch.arange(T, device=device) % 2 == 0)[:, None, None]
        hdr_d = torch.where(even, hdr_side[0], hdr_side[1]).contiguous()
        mask_d = torch.where(even, mask_side[0], mask_side[1]).contiguous()
        ord_d = None  # [T, P, M] int16 order rows, only when some defender row is ordered (attacker rows are sets)
        if (sides[0][4][:, 0] != K.ORDER_NONE).any():
            o_def = tt(sides[0][4].view(np.int16))[tt(sides[0][2])][:, of_pair[0]]
            ord_d = torch.where(even, o_def, o_def.new_full((), _ORDER_NONE_I16)).contiguous()
        bl_def, bl_att = tt(sides[0][3])[of_pair[0]], tt(sides[1][3])[of_pair[1]]                # [P] code each side sets (255: none)
        nash = torch.full((P,), K.BASE_LINES["Nash"], dtype=torch.uint8, device=device)
        # base_line after the defender's turn / after the attacker's turn, in the steady state of the alternation
        after_def0 = torch.where(bl_def == 255, nash, bl_def)                      # turn 0: nothing was set before
        after_att = torch.where(bl_att == 255, after_def0, bl_att)                 # turn 1
        after_def = torch.where(bl_def == 255, after_att, bl_def)                  # turns 2, 4, ...: the attacker's value may persist
        after_att2 = torch.where(bl_att == 255, after_def, bl_att)                 # turns 3, 5, ...
        bl_d = torch.empty(T, P, dtype=torch.uint8, device=device)
        bl_d[0::2] = after_def
        bl_d[1::2] = after_att2
        bl_d[0] = after_def0
        if T > 1:
            bl_d[1] = after_att
        bl_d = bl_d.contiguous()
        ret = torch.zeros(2, nloc, dtype=torch.float64, device=device)
        if not any_nn and W <= 4:
            spl = T if not steps_per_launch else max(1, int(steps_per_launch))
            order = _block_order(env, sides, i_of_pair, j_of_pair, pair_of_env, T)
            cuts = set(range(spl, T, spl))
            fit_after = set()
            if n_slots:  # the turns after which a fit must run: some pair's defender row executes type 10 (one read of [T, P])
                h0 = hdr_d[:, :, 0]
                trains_t = (((h0 & 0xFF) == 10) & (((h0 >> 8) & 1) == K.MODE_DEFENDER) & (bl_d == K.BASE_LINES["Nash"])).any(1)
                fit_after = {int(t) for t in torch.nonzero(trains_t).flatten().tolist() if t < T - 1}
                cuts |= {t + 1 for t in fit_after}
            bounds = [0] + sorted(cuts) + [T]
            for t0, t1 in zip(bounds[:-1], bounds[1:]):
                env.rollout(hdr_d[t0:t1], mask_d[t0:t1], bl_d[t0:t1], n_rollouts, lo, returns=ret, block_order=order,
                            order=None if ord_d is None else ord_d[t0:t1])  # the mode of a turn is in its headers
                if t1 - 1 in fit_after:
                    env.fit_detectors(detector_fit_seeds(seed, g_of_env, t1 - 1))
        else:
            X, n_app = network.X, int(network.cfg.get("n_app_ids", 0))
            side_of_env = [torch.from_numpy(i_of_pair).to(device)[pair_of_env], torch.from_numpy(j_of_pair).to(device)[pair_of_env]]
            nn_rows = [[(k, st, (side_of_env[m_] == k).nonzero(as_tuple=True)[0]) for k, st in enumerate(sts) if st.actor is not None]
                       for m_, sts in enumerate((def_strategies, att_strategies))]
            for t in range(T):
                mode = t & 1
                hdr_e = hdr_d[t][pair_of_env].contiguous()
                mask_e = mask_d[t][pair_of_env].contiguous()
                if nn_rows[mode]:
                    obs = env.observe(1 + mode)  # _get_defender_state / _get_attacker_state of every env (do_agent.py:748)
                    n_types = 14 if mode == 0 else 3  # get_num_action_types (volt:514-520): the actors' type slice
                    for k, st, idx in nn_rows[mode]:
                        if idx.numel() == 0:
                            continue
                        with torch.no_grad():
                            raw_a = st.actor(obs[idx])
                        h_k, m_k = decode_actions(raw_a, mode, n_types, M, X, n_app, W)
                        hdr_e[idx] = h_k
                        mask_e[idx] = m_k
                order_e = None
                if ord_d is not None and bool((ord_d[t, :, 0] != _ORDER_NONE_I16).any()):  # a defender turn with ordered rows
                    order_e = _order_arrays(hdr_e, mask_e, ord_d[t][pair_of_env])
                env.set_base_line_per_env(bl_d[t][pair_of_env])
                raw, _, _ = env.step(ActionBatch(hdr_e, mask_e, order_e))
                ret[mode] += raw.double()
                if n_slots and mode == 0 and t < T - 1:
                    env.fit_detectors(detector_fit_seeds(seed, g_of_env, t))
        sums.index_add_(0, pair_of_env, torch.stack(_columns(ret[0], ret[1], env.info()), dim=1))
        if train_detectors:
            _check_error_bits([env.scalars[:, K.S_FLAGS]])
    sums = sums.view(nd, na, len(COLUMNS))
    if not reduce:
        return sums
    return reduce_payoff(sums, n_rollouts, steps_per_episode, group=group)
