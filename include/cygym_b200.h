/*
 * cygym_b200.h -- C-ABI of the B200-native CyGym step path.
 *
 * The reference (Lan131/CyGym) has no FFI: its boundary is the Python attribute
 * surface of Volt_Typhoon_CyberDefenseEnv (SURVEY.md section 8b).  This header
 * is the C-ABI a maintainer would bind from Python (ctypes; see INTEGRATION.md)
 * to replace that path.  Each entry point cites the reference member it
 * replaces.  Plain pointers and sizes only; no torch types.  Device memory is
 * owned by the caller (torch tensors on the Python side); the library only
 * launches kernels on the caller's stream.
 *
 * Conventions: every function returns 0 on success and a negative CYG_E_* code
 * otherwise; cyg_last_error() returns a thread-local message.  All launches are
 * asynchronous on the given stream.  One host thread per handle.
 */
#ifndef CYGYM_B200_H
#define CYGYM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CYG_ABI_VERSION 3

/* ---- error codes ------------------------------------------------------- */
#define CYG_OK 0
#define CYG_E_INVAL (-22)   /* bad argument / unsupported configuration */
#define CYG_E_NOMEM (-12)
#define CYG_E_CUDA (-5)     /* a CUDA runtime call failed; see cyg_last_error() */
#define CYG_E_STATE (-71)   /* sticky per-env error flag raised by a kernel */

/* ---- canonical per-device word: dev[B][M] uint32 ------------------------
 * Flattening of the dynamic Device fields (CDSimulatorComponents.py:219-242)
 * and Workload (CDSimulatorComponents.py:18-26).                            */
#define CYG_DEV_COMP 0x00000001u      /* isCompromised */
#define CYG_DEV_KNOWN 0x00000002u     /* Known_to_attacker */
#define CYG_DEV_NYA 0x00000004u       /* Not_yet_added */
#define CYG_DEV_OWNED 0x00000008u     /* attacker_owned */
#define CYG_DEV_REMOVED 0x00000010u   /* removed_before */
#define CYG_DEV_HASWL 0x00000020u     /* workload is not None */
#define CYG_DEV_BUSYSET 0x00000040u   /* member of env._busy_devices (volt_typhoon_env.py:1330) */
#define CYG_DEV_ACTSET 0x00000080u    /* member of env._active_ids (CyberDefenseEnv.py:654-659) */
#define CYG_DEV_PT_SHIFT 8            /* workload.processing_time, 3 bits */
#define CYG_DEV_PT_MASK 0x7u
#define CYG_DEV_BUSY_SHIFT 12         /* busy_time, 8 bits canonical (kernels keep 4: 0..15) */
#define CYG_DEV_BUSY_MASK 0xFFu
#define CYG_DEV_CBY_SHIFT 20          /* compromised_by as a mask over exploit slots, 6 bits */
#define CYG_DEV_CBY_MASK 0x3Fu
#define CYG_BUSY_MAX 15

/* ---- per-device checkpoint word: ckpt[B][M] uint32 ----------------------
 * The 7 fields of _device_state (volt_typhoon_env.py:419-428).              */
#define CYG_CK_COMP 0x00000001u
#define CYG_CK_KNOWN 0x00000002u
#define CYG_CK_NYA 0x00000004u
#define CYG_CK_REACH 0x00000008u
#define CYG_CK_HASWL 0x00000020u
#define CYG_CK_VALID 0x80000000u
/* pt / busy / cby use the CYG_DEV_* shifts */

/* ---- static per-device word: dev_static[M] uint32 (shared by all envs) -- */
#define CYG_ST_DC 0x00000001u         /* device_type == "DomainController" */
#define CYG_ST_SERVER 0x00000002u     /* wtype == 'server' */
#define CYG_ST_REACH 0x00000004u      /* reachable_by_attacker (set once at init) */
#define CYG_ST_NAPPS_SHIFT 8          /* len(device.apps), 8 bits */
#define CYG_ST_VULN_SHIFT 16          /* bit e: an app vulnerability id is in exploits[e].target */

/* ---- per-env scalars: scal[B][16] uint32 -------------------------------- */
enum {
  CYG_S_STEP = 0,       /* step_num */
  CYG_S_EPOCH = 1,      /* draw epoch (bumped by every step / randomize / sample_action) */
  CYG_S_FLAGS = 2,      /* CYG_FL_* */
  CYG_S_PREV_X = 3,     /* low16: n_comp behind _prev_att_potential (0xFFFF = None); high16: #extra edges */
  CYG_S_DEF_STEP = 4,   /* defender_step */
  CYG_S_ATT_STEP = 5,   /* attacker_step */
  CYG_S_LOGS = 6,       /* len(simulator.logger.logs) */
  CYG_S_COMPCNT = 7,    /* compromised_devices_cnt */
  CYG_S_WORK = 8,       /* work_done */
  CYG_S_DEFCOST = 9,    /* defensive_cost (float bits) */
  CYG_S_CLEANCOST = 10, /* clearning_cost (float bits) */
  CYG_S_SCAN = 11,      /* scan_cnt */
  CYG_S_REVERT = 12,    /* revert_count */
  CYG_S_CKPT = 13,      /* checkpoint_count */
  CYG_S_EBLK = 14,      /* edges_blocked */
  CYG_S_EADD = 15,      /* edges_added */
  CYG_NSCAL = 16
};
#define CYG_FL_HAS_CKPT 0x00000001u     /* env.checkpoint is not None */
#define CYG_FL_SETS_INIT 0x00000002u    /* env._active_ids exists */
#define CYG_FL_DET_TRAINED 0x00000004u  /* action 10 ran with a non-empty log: simulator.detector.trained (CDSimulator.py:693-694) */
#define CYG_FL_DET_PENDING 0x00000008u  /* ... and that model is not yet fitted into the env's detector slot: either the host
                                           fits it with scikit-learn and uploads it (cyg_set_detectors), or cyg_fit_detectors
                                           fits every pending env on the device; the step kernels only PREDICT (tree walks).
                                           A scan that finds it set raises CYG_FL_ERR_DETECTOR.  Never part of a
                                           reference-side state: cleared by whichever fit ran. */
#define CYG_FL_ERR_BUSY 0x00000010u     /* busy_time exceeded CYG_BUSY_MAX (kernel saturated it) */
#define CYG_FL_ERR_XCAP 0x00000020u     /* more attacker-star edges than xcap */
#define CYG_FL_ERR_DETECTOR 0x00000040u /* a scan needed the trained detector and the env had none uploaded (no slot, model
                                           pending, or a hop-log ring shorter than the 30-record scan window); or
                                           cyg_fit_detectors could not fit a pending env (no free slot, or a ring shorter
                                           than the CYG_DET_WINDOW records the fit reads): the env stays pending */
#define CYG_FL_ERR_MASK 0x000000F0u
#define CYG_FL_DISC_SHIFT 8             /* bit e: exploits[e].discovered */

/* ---- extra (per-env) edges: extra[B][xcap] uint32 -----------------------
 * Attacker hub-star edges added by evolve_network (CyberDefenseEnv.py:738-774). */
#define CYG_X_V_SHIFT 12
#define CYG_X_BLOCKED 0x01000000u
#define CYG_X_IDMASK 0xFFFu

/* ---- actions -------------------------------------------------------------
 * One action = (action_type, exploit_indices, device_indices, app_index)
 * (volt_typhoon_env.py:876).  hdr[B][4] uint32 + dev_mask[B][W] uint32,
 * W = ceil(M/32).  device_indices is the ascending list of the mask's bits
 * unless an explicit order array is given (then order[b][0..n_dev) is used).  */
#define CYG_ATYPE_NONE 0x80u  /* action is None: filled from base_line (volt_typhoon_env.py:847-874) */
/* hdr[0]: atype (bits 0-7, signed) | mode<<8 (0 defender, 1 attacker) | n_ex<<16 (0..4) */
/* hdr[1]: exploit_indices[0..3], one signed byte each */
/* hdr[2]: n_dev (len(device_indices), bits 0-15) | (device_indices[0] + 1) << 16 -- the high half is optional: 0 means
 *         "the lowest listed id".  cyg_sample_actions fills it with the first device random.sample drew
 *         (CyberDefenseEnv.py:565), so that the actions that act on device_indices[0] (10, 11, 12, 13) hit a uniformly
 *         random device as in the reference; the remaining devices of a set-form list are visited in ascending order */
/* hdr[3]: app_index (int32) */
#define CYG_MODE_DEFENDER 0
#define CYG_MODE_ATTACKER 1

/* step flags */
#define CYG_STEP_GROUPED 0x1u   /* step_grouped semantics (volt_typhoon_env.py:694-779) */
#define CYG_STEP_SKIP_WORK 0x2u /* step(action, agent_cnt != len(net)) (volt_typhoon_env.py:1207,1307) */

/* base_line (volt_typhoon_env.py:849-873, :913, :1130, :1187) */
enum { CYG_BL_NASH = 0, CYG_BL_NO_DEFENSE = 1, CYG_BL_PRESET = 2, CYG_BL_NO_ATTACK = 3, CYG_BL_OTHER = 4 };

/* ---- configuration (attributes of the env; volt_typhoon_env.py:32-120,
 * CyberDefenseEnv.py:19-62) ------------------------------------------------ */
typedef struct cyg_config {
  int32_t M;                 /* Max_network_size == len(subnet.net) (device slots) */
  int32_t E;                 /* unique directed pairs in the base graph */
  int32_t X;                 /* MaxExploits */
  int32_t n_exploits;        /* len(simulator.exploits) */
  int32_t xcap;              /* capacity of the per-env extra-edge list */
  int32_t num_of_device;     /* numOfDevice */
  int32_t min_network_size;  /* Min_network_size */
  int32_t evolve_period;     /* _evolve_period (volt_typhoon_env.py:66) */
  int32_t wl_period_base;    /* workload_period_base */
  int32_t wl_period_max;     /* workload_period_max */
  int32_t wl_cap;            /* workload_cap, -1 = None */
  int32_t scaling_vulnerability;
  int32_t turbo;
  int32_t zero_day;
  uint32_t zero_day_mask;    /* common_exploit_indices | private_exploit_indices */
  int32_t att_space_n;       /* attacker_action_space.n = n_exploits + 3 */
  int32_t def_space_n;       /* defender_action_space.n = 14 */
  int32_t default_high;      /* default_high = 3 */
  int32_t n_app_ids;         /* get_num_app_indices() */
  int32_t base_line;         /* CYG_BL_* */
  int32_t tri_high;          /* `high` of np.random.triangular(0, mode, high) (CDSimulator.py:308) */
  int32_t log_cap;           /* hop-log ring per env: the last log_cap records of simulator.logger.logs (CDSimulator.py:663-679);
                                0 = only the length is kept (CYG_S_LOGS).  30 serves the scan window (volt:1052), 2000 what
                                detector training reads (volt:955-961) */
  float work_scale, comp_scale, def_scale, gamma;
  uint64_t thr_p_add;        /* random() < p_add      <=> x < thr (CyberDefenseEnv.py:679) */
  uint64_t thr_p_attacker;   /* random() < p_attacker <=> x < thr (CyberDefenseEnv.py:690) */
  uint32_t poisson_tab[16];  /* np.random.poisson(lambda_events): #{j: x >= tab[j]} (CyberDefenseEnv.py:668) */
  uint32_t tri_tab[8];       /* ceil(triangular): min(tri_high, 1 + #{v: x >= tab[v]}) */
  uint64_t seed;             /* Philox key */
  /* turbo workload throttle (volt_typhoon_env.py:219-231), used when `turbo` != 0 */
  double turbo_frac_clients; /* turbo_fraction_clients */
  double turbo_frac_servers; /* turbo_fraction_servers */
  int32_t turbo_max_clients; /* turbo_max_clients */
  int32_t turbo_max_servers; /* turbo_max_servers */
  int32_t turbo_ramp_steps;  /* turbo_ramp_steps */
  int32_t reserved1;
} cyg_config;

/* ---- shared network tables (device pointers for the CUDA library) ------- */
typedef struct cyg_network {
  const int32_t* row_ptr;      /* [M+1] CSR over unique out-pairs, ascending neighbour id (_outnbrs, volt:456-473) */
  const int32_t* col;          /* [E] */
  const uint8_t* mult;         /* [E] multiplicity of the pair in the igraph multigraph */
  const uint32_t* dev_static;  /* [M] CYG_ST_* */
  const float* os_val;         /* [M] os_to_float(d.OS) (CyberDefenseEnv.py:125-144) */
  const float* ver_val;        /* [M] float(d.version) */
} cyg_network;

/* ---- per-env state buffers (device pointers, canonical layout) ---------- */
typedef struct cyg_state {
  uint32_t* dev;      /* [B][M] */
  uint32_t* ckpt;     /* [B][M] */
  uint32_t* blocked;  /* [B][ceil(E/32)] bit e: base pair e is in env._blocked (volt:73) */
  uint32_t* extra;    /* [B][xcap] */
  uint32_t* scal;     /* [B][16] */
  uint32_t* logs;     /* optional [B][log_cap]: hop-log ring, record k of the env's log (k = 0 .. CYG_S_LOGS - 1) sits at
                         k % log_cap as from_device | to_device << 16; NULL = not transferred */
} cyg_state;

typedef struct cyg_actions {
  const uint32_t* hdr;    /* [G][B][4] */
  const uint32_t* mask;   /* [G][B][W] */
  const uint16_t* order;  /* optional [G][B][order_stride] explicit device_indices order, or NULL */
  int32_t order_stride;
  int32_t n_groups;       /* G: 1 for step(), len(groups) for step_grouped() */
} cyg_actions;

typedef struct cyg_step_out {
  float* raw_reward;     /* [B]   (volt_typhoon_env.py:1291,1303) */
  float* shaped_reward;  /* [B]   (volt_typhoon_env.py:1292,1304) */
  int32_t* done;         /* [B]   _check_done: step_num > 1000 (CyberDefenseEnv.py:547-552) */
  uint32_t* pre_masks;   /* optional [B][3][W]: compromised / known / not_yet_added BEFORE evolve_network,
                            i.e. the content of the `state` step() returns (volt_typhoon_env.py:1306) */
  float* obs;            /* optional [B][obs_dim] post-evolve view of `obs_mode` */
  int32_t obs_mode;      /* 0 none, 1 _get_defender_state (6M), 2 _get_attacker_state (4M+X), 3 _get_state (6M) */
} cyg_step_out;

typedef struct cyg_env_s* cyg_handle;

int cyg_version(void);
const char* cyg_last_error(void);

/* Replaces Volt_Typhoon_CyberDefenseEnv.__init__ + attribute configuration. The
 * network tables are copied to the device by the library (they are tiny). All
 * pointers in `net` are HOST pointers here. `device` is the CUDA ordinal.      */
int cyg_create(cyg_handle* out, const cyg_config* cfg, const cyg_network* host_net, int32_t B,
               int32_t env_id0, int32_t device);
int cyg_destroy(cyg_handle h);
int cyg_set_base_line(cyg_handle h, int32_t base_line);
/* Optional base_line PER ENV (device array [B] of CYG_BL_*, read by every following cyg_step; NULL = back to the
 * handle-wide value).  Lets one batch hold rollouts of different (defender, attacker) strategy pairs, whose
 * baselines set env.base_line on every turn (do_agent.py:716-719). */
int cyg_set_base_line_per_env(cyg_handle h, const uint8_t* base_line);
/* The same with one row per fused step: base_line[n_rows][B]; step t of a cyg_step_multi launch reads row t (the
 * baselines of the two players set env.base_line on alternating turns), cyg_step reads row 0. */
int cyg_set_base_line_per_env_steps(cyg_handle h, const uint8_t* base_line, int32_t n_rows);

/* uint32 words PER ENV the caller must allocate for the kernels' internal state.  The buffer holds, in this
 * order: B records of S words (16 scalars + bit-planes + the blocked-edge bitset in incidence-unit order;
 * what a CTA bulk-copies into shared memory), then B*M per-device checkpoint words (actions 11/12,
 * volt_typhoon_env.py:419-453), then B*xcap extra-edge words, then B*log_cap hop-log ring words.
 * words_per_env = S + M + xcap + log_cap. */
int cyg_internal_words(cyg_handle h, int64_t* words_per_env);

/* Bind the internal state buffer (device pointer, B * words_per_env uint32, 16-byte aligned). */
int cyg_bind(cyg_handle h, uint32_t* internal_state);

/* canonical <-> internal conversion (import = reset()/snapshot load, volt_typhoon_env.py:1904-1925). */
int cyg_import_state(cyg_handle h, const cyg_state* canonical, void* stream);
int cyg_export_state(cyg_handle h, const cyg_state* canonical, void* stream);

/* Replaces step() / step_grouped() (volt_typhoon_env.py:818-1333, :694-779). */
int cyg_step(cyg_handle h, const cyg_actions* actions, uint32_t step_flags, const cyg_step_out* out,
             void* stream);

/* n_steps consecutive plain step() calls in ONE launch: the loop body of the rollouts that replay fixed action
 * sequences or scripted / random policies (simulate_game, do_agent.py:1875-2089; Strategy, strategy.py:25-60), where
 * step t+1's action does not wait for a host-side policy.  actions->hdr / mask hold n_steps consecutive batches
 * ([n_steps][B][4], [n_steps][B][W]); out->raw_reward / shaped_reward / done receive n_steps consecutive [B] rows.
 * Every env's record stays in shared memory between the steps.  Plain steps only: no CYG_STEP_GROUPED, no order
 * array, no obs / pre_masks, networks of at most 128 device slots (CYG_E_INVAL otherwise).  The result is
 * bit-identical to n_steps cyg_step() calls. */
int cyg_step_multi(cyg_handle h, const cyg_actions* actions, int32_t n_steps, uint32_t step_flags,
                   const cyg_step_out* out, void* stream);

/* Whole rollouts of the payoff-matrix evaluation (DoubleOracle.simulate_game, do_agent.py:1875-2089, under
 * build_payoff_matrices, :1666-1870) in ONE launch: n_steps consecutive plain steps of every env, the records staying
 * in shared memory between them.  The strategies that need no observation (baseline names, fixed action sequences,
 * the no-op; strategy.py:25-60) are TABLES shared by runs of envs: env b reads action row (row_base + b) / envs_per_row
 * of the n_rows rows of a step -- with rows = (defender, attacker) strategy pairs and envs_per_row = rollouts per pair,
 * the per-pair tables are uploaded once per evaluation and gathered inside the kernel.  base_line (optional) has the
 * same row layout: what the two players' baselines set env.base_line to on their turns (do_agent.py:716-719).
 * returns[2][B] (float64) receives += the raw reward of every step, row 0 on defender turns, row 1 on attacker turns
 * (def_r / att_r of do_agent.py:2060-2062); the counters of the info dict are read from the scalars afterwards.
 * A handle with a hop-log ring (log_cap > 0) and detector slots keeps its rings and consults its detectors here as in
 * cyg_step.  No detector is fitted inside a launch: an env whose defender trains (action 10) stays CYG_FL_DET_PENDING
 * until cyg_fit_detectors runs, and a trained scan (action 5) of that env later in the SAME launch sets
 * CYG_FL_ERR_DETECTOR, exactly as in cyg_step_multi.  A caller whose strategies may train ends the launch after every
 * turn that may train and calls cyg_fit_detectors before the next one (cygym_b200/payoff.py, train_detectors=True). */
typedef struct cyg_rollout_args {
  const uint32_t* hdr;      /* [n_steps][n_rows][4] */
  const uint32_t* mask;     /* [n_steps][n_rows][W] */
  const uint8_t* base_line; /* optional [n_steps][n_rows] CYG_BL_* */
  int32_t n_steps, n_rows;
  int64_t row_base;
  int32_t envs_per_row;
  int32_t reserved;
  double* returns;          /* [2][B] */
  const int32_t* block_order; /* optional [ceil(B / cyg_block_envs)], a PERMUTATION of the block indices: the launch's
                                 i-th CTA steps slots [block_order[i] * block_envs, +block_envs).  CTAs start in index
                                 order, so listing the expensive blocks first (longest processing time first) shortens
                                 the tail of a launch whose blocks differ a lot in cost -- strategy pairs do */
} cyg_rollout_args;
/* Slots per CTA of this handle's step / rollout launches (what block_order indexes). */
int cyg_block_envs(cyg_handle h, int32_t* block_envs);
int cyg_rollout(cyg_handle h, const cyg_rollout_args* a, uint32_t step_flags, void* stream);

/* cyg_rollout with device_indices in a given ORDER: the sequences DoubleOracle draws with sample_action (do_agent.py:
 * 1001-1013) list their devices in random.sample draw order (CyberDefenseEnv.py:565), and for defender types 1, 4, 5, 6,
 * 9, 12 and 13 that order changes the result (the _stall draws are taken per listed device in list order; block /
 * unblock pick one edge per listed device, each pick seeing the flips before it, volt:485-511).
 * order[n_steps][n_rows][order_stride] (uint16) has the row layout of a->hdr.  A row whose first entry is
 * CYG_ORDER_NONE is a set-form row and steps exactly as in cyg_rollout; any other row lists its n_dev devices in order
 * in its first n_dev entries (as cyg_actions.order does for cyg_step; the mask still holds their set) and its env runs
 * the action with one thread, as cyg_step does with an order array.  A header whose n_dev exceeds order_stride is read
 * as order_stride: the kernel never reads past order_stride entries of a row.  Everything else -- base_line rows,
 * returns, block_order, strided env ids, hop-log rings and detectors -- is as in cyg_rollout, and the result of every
 * env is bit-identical to n_steps cyg_step() calls with the same order rows.  CYG_E_INVAL on a NULL order,
 * order_stride < M, networks beyond 128 device slots and CYG_STEP_GROUPED. */
#define CYG_ORDER_NONE 0xFFFFu
int cyg_rollout_ordered(cyg_handle h, const cyg_rollout_args* a, const uint16_t* order, int32_t order_stride,
                        uint32_t step_flags, void* stream);

/* Which env a slot of the handle holds.  Default: slot s is env env_id0 + s.  With run > 0 (run divides B, stride >= run)
 * slot s is env env_id0 + (s / run) * stride + s % run: runs of `run` consecutive env ids, `stride` ids apart.  The payoff
 * evaluation numbers its envs (strategy pair, rollout) row-major; a rank that takes rollouts [r * run, (r + 1) * run) of
 * EVERY pair (run = rollouts per pair / ranks, stride = rollouts per pair, env_id0 = r * run) gets the same mix of cheap
 * and expensive pairs as every other rank, where a contiguous slice of the id range would hand whole defender strategies
 * to single ranks (the imbalance of the reference's pool workers, do_agent.py:1737-1753).  The env id keys the draw
 * streams and, in cyg_rollout, the action row ((row_base + id - env_id0) / envs_per_row), so per-env results do not depend
 * on the layout.  Honoured by cyg_rollout, cyg_randomize, cyg_rebuild_graph_cache and cyg_sample_actions; cyg_step /
 * cyg_step_multi refuse a handle with strided ids.  run <= 0 restores the default. */
int cyg_set_env_id_stride(cyg_handle h, int32_t run, int32_t stride);

/* Compact action rows for callers that keep their actions in HOST memory: the copy over PCIe is what bounds a host-buffer
 * step (DESIGN.md), so the header of a set-form action travels in two words instead of four.  Row of env b =
 * [w0, w1, mask[0..Wm)] (2 + Wm words):
 *   w0 = action_type (bits 0-7, CYG_ATYPE_NONE as in hdr[0]) | mode << 8 | n_exploits << 9 (0..4) | n_devices << 12 (0..4095)
 *        | (device_indices[0] + 1) << 24 (0: none given)
 *   w1 = exploit index i as a signed 4-bit field at bit 4 i (-8..7) | app_index as a signed 16-bit field << 16
 * Actions outside those ranges (and networks above 254 device slots) use the full hdr / mask arrays.
 * cyg_unpack_actions expands B rows (device memory) into hdr [B][4] + mask [B][Wm] for cyg_step; it is one small launch
 * on `stream` and replaces nothing of the reference -- it is the decode of what volt_typhoon_env.py:876 unpacks. */
int cyg_unpack_actions(cyg_handle h, const uint32_t* rows, uint32_t* hdr, uint32_t* mask, void* stream);
/* The way back: the `done` flags of a step (cyg_step_out.done, [B] int32) as one bit per env -- bit b % 32 of word b / 32,
 * ceil(B / 32) words -- so that a host-buffer step reads 8.1 bytes per env (raw, shaped, done bit) instead of 12. */
int cyg_pack_done(cyg_handle h, const int32_t* done, uint32_t* bits, void* stream);

/* Replaces randomize_compromise_and_ownership() (volt_typhoon_env.py:330-383); env_mask may be NULL. */
int cyg_randomize(cyg_handle h, const uint8_t* env_mask, void* stream);

/* Replaces a _rebuild_graph_cache() call made from OUTSIDE a step (volt_typhoon_env.py:456-483; DoubleOracle.restore,
 * do_agent.py:891-895; reset(from_init), volt:1933-1936): the rebuilt cache forgets every blocked edge (volt:476).
 * env_mask may be NULL. */
int cyg_rebuild_graph_cache(cyg_handle h, const uint8_t* env_mask, void* stream);

/* ---- trained detector (defender action 5 after action 10; volt_typhoon_env.py:1020-1069, CDSimulator.py:681-723) -----
 * Detector = IsolationForest(n_estimators=2, max_samples=256).  The host fits it (scikit-learn, from the env's hop log)
 * and uploads the two trees plus the forest's verdict for every pair of leaves, or cyg_fit_detectors fits it on the
 * device into the same format; the kernels walk the trees.  One slot =
 * CYG_DET_WORDS uint32:
 *   [0]            L1 = leaves of tree 1 (row length of the verdict table)
 *   [4 + t*2048 + 4*n .. +4), t = 0, 1, node n < 512:  threshold (float64, lo / hi word), left | right << 16,
 *                  feature | leaf_index << 16   (feature 0 = from_device, 1 = to_device, 2 = leaf)
 *   [4100 + (l0*L1 + l1) / 32]  bit (l0*L1 + l1) % 32: model.predict == -1 ("A") for a point in leaves (l0, l1)
 * det_of_env[b] = slot of env b, -1 = none.  Both arrays are device memory owned by the caller; NULL switches it off. */
#define CYG_DET_WORDS 6160
#define CYG_DET_TREE0 4
#define CYG_DET_TREE_STRIDE 2048
#define CYG_DET_TABLE 4100
#define CYG_DET_WINDOW 2000 /* records a fit reads: the last min(CYG_S_LOGS, 2000) of the log (CDSimulator.py:691-692) */
int cyg_set_detectors(cyg_handle h, const uint32_t* slots, int32_t n_slots, const int32_t* det_of_env);
/* Detector.train (CDSimulator.py:687-695) of every env with CYG_FL_DET_PENDING, on the device: numpy's global stream
 * seeded with seeds[b] (uint32), then IsolationForest(n_estimators=2, max_samples=256).fit on the env's last
 * min(CYG_S_LOGS, CYG_DET_WINDOW) hop-log records, read from the internal ring.  The slot written is bit-identical to what
 * the host uploads after that seeded scikit-learn 1.9 fit (cygym_b200/csrc/cyg_iforest.cuh restates ensemble/_iforest.py,
 * ensemble/_bagging.py, utils/_random.pyx and tree/_splitter.pyx, _partitioner.pyx, _criterion.pyx, _tree.pyx).
 * An env without a slot (det_of_env[b] < 0) takes slot *next_slot, in env order, and *next_slot advances: next_slot is a
 * device int32 owned by the caller and shared with whatever assigns slots on the host.  A fitted env keeps
 * CYG_FL_DET_TRAINED and loses CYG_FL_DET_PENDING.  An env that cannot be fitted -- no slot left, or
 * min(CYG_S_LOGS, CYG_DET_WINDOW) > log_cap -- stays pending and gets CYG_FL_ERR_DETECTOR.  Three launches on `stream`
 * (slot assignment in two passes over the whole batch, then the fits), no host synchronisation.  CYG_E_INVAL when the
 * handle has no detector slots. */
int cyg_fit_detectors(cyg_handle h, const uint32_t* seeds, int32_t* next_slot, void* stream);

/* Replaces sample_action() (CyberDefenseEnv.py:555-578) for every env; writes hdr[B][4], mask[B][W]. */
int cyg_sample_actions(cyg_handle h, int32_t mode, uint32_t* hdr, uint32_t* mask, void* stream);
/* The same, also writing device_indices in the DRAW order of random.sample (CyberDefenseEnv.py:565) into
 * order[B][order_stride] (uint16, order_stride >= numOfDevice): pass it back as cyg_actions.order for a step that
 * visits the devices exactly in the reference's order. */
int cyg_sample_actions_ordered(cyg_handle h, int32_t mode, uint32_t* hdr, uint32_t* mask, uint16_t* order,
                               int32_t order_stride, void* stream);

/* Replaces _get_defender_state / _get_attacker_state / _get_state (CyberDefenseEnv.py:241/194/146). */
int cyg_observe(cyg_handle h, int32_t obs_mode, float* obs, void* stream);

/* IPPO / MAPPO glue (IPPO.py:559-570, MAPPO.py same lines): every device of every env drew an action type
 * (per_dev_types[B][M]); the devices the role sees (build_visibility_mask, IPPO.py:74-96: role 1 defender = not
 * Not_yet_added and attacker_owned, role 2 attacker = that and Known_to_attacker, role 0 = all; `visible`[B][M], when
 * given, is the caller's own 0 / 1 mask, ANDed with the role's) are grouped by type into
 * the n_types - 1 action groups of one cyg_step(CYG_STEP_GROUPED) call, ascending type order without `noop`; a type
 * with no device becomes a no-op group (the reference skips it).  Types 11 / 12 keep ONE device: single_choice[B][2]
 * (the reference's random.choice) or, when NULL, the lowest.  Writes hdr[n_types-1][B][4], mask[n_types-1][B][W]. */
int cyg_group_actions(cyg_handle h, int32_t mode, int32_t role, const int32_t* per_dev_types, const uint8_t* visible,
                      const int32_t* exp_idx, const int32_t* app_idx, const int32_t* single_choice, int32_t n_types, int32_t noop, uint32_t* hdr,
                      uint32_t* mask, void* stream);

/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t cyg_launch_count(cyg_handle h);

#ifdef __cplusplus
}
#endif
#endif /* CYGYM_B200_H */
