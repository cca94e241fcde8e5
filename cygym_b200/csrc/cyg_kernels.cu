/*
 * cyg_kernels.cu -- sm_100a kernels + the C-ABI of include/cygym_b200.h.
 *
 * cyg_step_kernel<W, PLAIN>: ONE launch per env step (volt_typhoon_env.py:818-1333 / :694-779).
 *   A CTA owns a block of NB consecutive envs.  Their internal records (cyg_core.cuh) are one
 *   contiguous span of HBM, so the CTA moves them with a single TMA bulk copy into shared
 *   memory (cp.async.bulk + mbarrier), steps them there, and writes them back with a single
 *   bulk store: HBM sees exactly one full-sector read and one write of the state per step.
 *   The hot network tables (adjacency bit rows, device masks, CSR) ride in on the same mbarrier.
 *   Work mapping is thread-per-env over bit-planes (32 devices per integer op), in three phases
 *   separated by __syncthreads():
 *     1. prologue  thread t -> env t      : epoch, executed action type, busy tick
 *     2. action    thread t -> env perm[t]: envs are counting-sorted by (mode, action type) inside
 *                                           the CTA so that a warp runs one action type and the 14
 *                                           defender / 3+X attacker branches do not serialise
 *     3. epilogue  thread t -> env t      : work, arrivals, reward, counters, evolve_network,
 *                                           coalesced outputs, optional fused observation rows
 * cyg_fit_assign_kernel + cyg_fit_kernel: the detector fit of defender action 10 (cyg_iforest.cuh), one warp per
 *   pending env.
 * No tensor cores: the path has no dense contraction.  No CPU fallback anywhere in this file.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <new>
#include <string>

#include "cyg_coop.cuh"
#include "cyg_core.cuh"
#include "cyg_iforest.cuh"
#include "cyg_tables.h"

using namespace cyg;

/* ---- small PTX wrappers (mbarrier + 1-D TMA bulk copies) ------------------- */
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_read() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

/* ---- kernel parameters ---------------------------------------------------- */
struct StepParams {
  Net net;              /* pointers into the device copy of the table blob */
  uint32_t* recs;       /* [B][S] internal records */
  uint32_t* ckpt;       /* [B][M] canonical checkpoint words */
  uint32_t* xtra;       /* [B][xcap] extra edges */
  const uint32_t* hdr;  /* [G][B][4] */
  const uint32_t* mask; /* [G][B][W] */
  const uint16_t* order;
  float* raw;
  float* shaped;
  int32_t* done;
  uint32_t* pre_masks;
  float* obs;
  unsigned long long* dbg_cycles; /* optional [B]: SM cycles each env's step took (diagnostics) */
  uint32_t* logs;                 /* [B][log_cap] hop-log rings (NULL when log_cap == 0) */
  const uint32_t* det_slots;      /* uploaded detectors (cyg_set_detectors) */
  const int32_t* det_of_env;      /* [B] slot of env, -1 none */
  const uint8_t* bl_env;          /* optional [B]: base_line per env (CYG_BL_*); NULL = cfg.base_line for all */
  int bl_stride;                  /* fused steps: bl_env row of step t starts at t * bl_stride (0: one row for all) */
  int B, env_id0, G, order_stride, obs_mode, block_envs;
  uint32_t flags;
  /* rollouts (cyg_rollout): action rows are shared by runs of envs -- env b reads row (row_base + b) / envs_per_row of
   * the n_rows rows of a step (envs_per_row == 0: one row per env, n_rows == B) -- and the raw rewards are summed per env */
  long long row_base;
  int envs_per_row, n_rows;
  int id_run, id_stride; /* cyg_set_env_id_stride (ROLL only): see strided_index() */
  const int32_t* block_order; /* optional (ROLL only): CTA b steps the envs [block_order[b] * block_envs, +block_envs) */
  double* ret_acc;      /* optional [2][B]: += raw reward, row 0 defender turns, row 1 attacker turns */
  int T;                /* plain steps fused into this launch (cyg_step_multi): hdr / mask hold T consecutive batches,
                           raw / shaped / done T consecutive [B] rows; the records stay in shared memory in between */
};

#define CYG_NKEYS 48 /* sort keys: (mode, executed action type) in 0..31; 32..47 = block / unblock envs of a plain step
                        bucketed by listed-device count, longest first (the warp-per-env tasks of phase B run in that order) */
#define CYG_KEY_FLIP0 32
#define CYG_TMA_STORE 1 /* records go back with one bulk store; plain coalesced stores measured the same (the
                          write-back is bound by the per-SM path to L2: ~16k cycles for 210 KB either way) */
#define CYG_MAX_BLOCK_ENVS 512   /* envs per CTA */
#ifndef CYG_MAX_BLOCK_THREADS
#define CYG_MAX_BLOCK_THREADS 640 /* threads per CTA at one CTA per SM: 20 warps with up to 93 registers each.  Phases A / C
                                    use one thread per env, the warp-per-env phase B every warp.  Measured with the final
                                    kernel (4 fused steps / one launch per step): 896 threads (72 registers, 88 B of spills)
                                    46.4 / 56.6 us, 768: 44.1 / 54.7, 640: 42.5 / 53.7, 576: 43.2 / 55.8, 512: 44.0 / 56.8 */
#endif

/* cyg_set_env_id_stride: env index (env id minus env_id0) of a slot -- runs of `run` consecutive ids, `stride` ids apart */
__host__ __device__ __forceinline__ uint32_t strided_index(uint32_t slot, uint32_t run, uint32_t stride) {
  const uint32_t c = slot / run;
  return c * stride + (slot - c * run);
}

/* one record from shared to global memory by one warp: 4 bytes per lane, 128 words per round, predicated tail */
__device__ __forceinline__ void copy_record(uint32_t* dst, const uint32_t* src, int S, int lane) {
  for (int base = 0; base < S; base += 128) {
    const int i0 = base + lane, i1 = i0 + 32, i2 = i0 + 64, i3 = i0 + 96;
    uint32_t v0 = 0, v1 = 0, v2 = 0, v3 = 0;
    if (i0 < S) v0 = src[i0];
    if (i1 < S) v1 = src[i1];
    if (i2 < S) v2 = src[i2];
    if (i3 < S) v3 = src[i3];
    if (i0 < S) dst[i0] = v0;
    if (i1 < S) dst[i1] = v1;
    if (i2 < S) dst[i2] = v2;
    if (i3 < S) dst[i3] = v3;
  }
}

/* Observation rows (CyberDefenseEnv.py:146-257; obs_mode as in cyg_step_out) of n_envs consecutive records: one warp per
 * (env, plane word) = 32 devices, the lanes on consecutive OUTPUT floats (coalesced stores): an element is a static
 * table value (OS id, version) or one bit of the four plane words the whole warp shares. */
template <int W, int F>
__device__ __forceinline__ void observe_rows_f(const Net& n, const uint32_t* recs, int S, int n_envs, int obs_mode, float* out, int warp,
                                               int nwarps, int lane) {
  const int M = n.M, Wm = n.Wm, dim = F == 4 ? 4 * M + n.cfg.X : 6 * M;
  const float* osv = (const float*)(n.blob + n.o_os);
  const float* verv = (const float*)(n.blob + n.o_ver);
  for (int chunk = warp; chunk < n_envs * Wm; chunk += nwarps) {
    const int el = chunk / Wm, w = chunk - el * Wm;
    const uint32_t* pl = recs + (size_t)el * S + CYG_REC_PLANES;
    const uint32_t c = pl[P_COMP * W + w], k = pl[P_KNOWN * W + w], y = pl[P_NYA * W + w], o = pl[P_OWNED * W + w];
    const uint32_t vis = F == 4 ? (k & ~y & o) : (obs_mode == 1 ? (~y & o) : 0xFFFFFFFFu); /* rows outside are -1 */
    const int nelem = min(32, M - 32 * w) * F;
    float* row = out + (size_t)el * dim + 32 * w * F;
    if ((((uintptr_t)row) & 7) == 0) { /* uniform */
      /* pairs of floats: F is even, a device's row is (OS, version) (compromised, 0 | 1) [(known, not-yet-added)], so a
       * lane produces the two fields of ONE pair of ONE device and stores 8 bytes -- half the rounds and a third of the
       * instructions per float of the element-wise form below (which cost more warp instructions than the step itself) */
      constexpr int P = F / 2; /* pairs per device */
      const int npair = nelem >> 1;
#pragma unroll
      for (int t = 0; t < P; t++) {
        const int pi = t * 32 + lane;
        if (pi >= npair) continue;
        const int sd = pi / P, fp = pi - sd * P, d = 32 * w + sd;
        float2 v;
        if (!((vis >> sd) & 1u)) { v.x = -1.f; v.y = -1.f; }
        else if (fp == 0) { v.x = osv[d]; v.y = verv[d]; }
        else if (fp == 1) {
          v.x = (F == 6 && obs_mode == 1) ? -1.f : (float)((c >> sd) & 1u);
          v.y = F == 4 ? 1.f : 0.f;
        } else { v.x = (float)((k >> sd) & 1u); v.y = (float)((y >> sd) & 1u); }
        reinterpret_cast<float2*>(row)[pi] = v;
      }
      if (F == 4 && w == 0 && lane < n.cfg.X) out[(size_t)el * dim + 4 * M + lane] = lane < n.cfg.n_exploits ? 1.f : 0.f;
      continue;
    }
#pragma unroll
    for (int t = 0; t < F; t++) {
      const int e = t * 32 + lane;
      if (e >= nelem) continue;
      const int sd = e / F, f = e - sd * F, d = 32 * w + sd;
      float v;
      if (!((vis >> sd) & 1u)) v = -1.f;
      else if (f == 0) v = osv[d];
      else if (f == 1) v = verv[d];
      else if (F == 4) v = f == 2 ? (float)((c >> sd) & 1u) : 1.f;
      else v = f == 2 ? (obs_mode == 1 ? -1.f : (float)((c >> sd) & 1u)) : f == 3 ? 0.f : f == 4 ? (float)((k >> sd) & 1u) : (float)((y >> sd) & 1u);
      row[e] = v;
    }
    if (F == 4 && w == 0 && lane < n.cfg.X) out[(size_t)el * dim + 4 * M + lane] = lane < n.cfg.n_exploits ? 1.f : 0.f;
  }
}
template <int W>
__device__ __forceinline__ void observe_rows(const Net& n, const uint32_t* recs, int S, int n_envs, int obs_mode, float* out, int warp,
                                             int nwarps, int lane) {
  if (obs_mode == 2) observe_rows_f<W, 4>(n, recs, S, n_envs, obs_mode, out, warp, nwarps, lane);
  else observe_rows_f<W, 6>(n, recs, S, n_envs, obs_mode, out, warp, nwarps, lane);
}

/* shared-memory carve-up for a CTA of NB envs (all offsets 16-byte aligned; tables first, at word 0) */
struct SmemPlan {
  size_t off_tables, off_recs, off_out, off_perm, off_cnt, off_def, off_bar, total;
};
__host__ __device__ inline size_t smem_take(size_t& o, size_t bytes) { size_t r = o; o += (bytes + 15) & ~(size_t)15; return r; }
__host__ __device__ inline SmemPlan smem_plan(uint32_t hot_words, int S, int NB) {
  SmemPlan p;
  size_t o = 0;
  p.off_tables = smem_take(o, (size_t)hot_words * 4);
  p.off_recs = smem_take(o, (size_t)NB * S * 4);
  p.off_out = smem_take(o, (size_t)NB * 2 * 4); /* phase B -> C carry: action cost, topology-dirty flag */
  p.off_perm = smem_take(o, (size_t)NB * 2);
  p.off_cnt = smem_take(o, (size_t)(CYG_NKEYS + 7) * 4); /* key histogram / run ends + four task counters + warps past phase A + warps past step_pre */
  p.off_def = smem_take(o, (size_t)(CYG_MAX_BLOCK_ENVS / 32) * 4); /* bit pos: perm[pos] is finished by phases B / C, not A */
  p.off_bar = smem_take(o, 8);
  p.total = o;
  return p;
}

/* CTA-level phase timestamps (profiling build -DCYG_CTA_TIMING: thread 0 writes clock64 at the phase boundaries) */
#ifdef CYG_CTA_TIMING
#define CYG_CTA_MARK(i) do { if (p.dbg_cycles && threadIdx.x == 0) p.dbg_cycles[(size_t)blockIdx.x * 8 + (i)] = (unsigned long long)clock64(); } while (0)
/* per-warp timestamps inside phase B (after the block/unblock, deposit and attack task loops): slots of 4 behind the CTA marks */
#define CYG_WARP_MARK(i) do { if (p.dbg_cycles && (threadIdx.x & 31) == 0) p.dbg_cycles[2048 + ((size_t)blockIdx.x * 32 + (threadIdx.x >> 5)) * 4 + (i)] = (unsigned long long)clock64(); } while (0)
#else
#define CYG_CTA_MARK(i) do { } while (0)
#define CYG_WARP_MARK(i) do { } while (0)
#endif

/* PLAIN: one ungrouped action per env, device lists as sets (no order array) -- the hot form: thread-per-env phases
 * A / C plus the warp-per-env phase B.  !PLAIN: grouped steps and explicit order lists, everything thread-per-env
 * (the sequential forms of every action live only in this instantiation). */
/* ROLL: the cyg_rollout form of the plain kernel -- action rows shared by runs of envs, raw rewards summed per env.  A
 * separate instantiation: compiled into the step kernel proper, the row indexing and the accumulation cost it 4.5 us per
 * step (registers) although no step ever takes those branches. */
/* LOG: the env keeps a hop-log ring and may hold a trained detector (cfg.log_cap > 0): the lateral-movement scan writes
 * its hops, scans consult the detector.  Also its own instantiation (the handles that keep only the log's length --
 * every throughput run -- take the kernel without that code: ~1 us per step). */
template <int W, bool PLAIN, bool ROLL = false, bool LOG = true>
__global__ void __launch_bounds__(CYG_MAX_BLOCK_THREADS, 1) cyg_step_kernel(const __grid_constant__ StepParams p) {
  unsigned char* smem = reinterpret_cast<unsigned char*>(cyg_smem);
  const int NB = p.block_envs, NT = blockDim.x, tid = threadIdx.x; /* NB envs, NT >= NB threads */
  CYG_CTA_MARK(0);
  const int S = p.net.S, M = p.net.M;
  int blk_i = (int)blockIdx.x;
  if constexpr (ROLL) { if (p.block_order) blk_i = p.block_order[blockIdx.x]; }
  const int env0 = blk_i * NB;
  const int nb = min(NB, p.B - env0);
  const SmemPlan sp = smem_plan(p.net.hot_words, S, NB);
  uint32_t* s_tab = (uint32_t*)(smem + sp.off_tables);
  uint32_t* s_rec = (uint32_t*)(smem + sp.off_recs);
  float* s_out = (float*)(smem + sp.off_out);
  uint16_t* s_perm = (uint16_t*)(smem + sp.off_perm);
  uint32_t* s_cnt = (uint32_t*)(smem + sp.off_cnt);
  uint32_t* s_def = (uint32_t*)(smem + sp.off_def);
  uint64_t* bar = (uint64_t*)(smem + sp.off_bar);
  const bool grouped = PLAIN ? false : (p.flags & CYG_STEP_GROUPED) != 0;

  uint32_t* g_rec = p.recs + (size_t)env0 * S;
  const uint32_t rec_bytes = (uint32_t)nb * S * 4u;
  const uint32_t tab_bytes = p.net.hot_words * 4u;
  const bool bulk_ok = (rec_bytes & 15u) == 0 && ((((size_t)g_rec) & 15) == 0);

  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_expect_tx(bar, tab_bytes + (bulk_ok ? rec_bytes : 0u));
    bulk_g2s(s_tab, p.net.blob, tab_bytes, bar);
    if (bulk_ok) bulk_g2s(s_rec, g_rec, rec_bytes, bar);
  }
  const int T = PLAIN ? (p.T < 1 ? 1 : p.T) : 1;
  const int lane = tid & 31;
  for (int t = 0; t < T; t++) { /* the steps fused into this launch; the records stay in shared memory */
  const bool last = t == T - 1;
  const uint32_t* hdr_t = p.hdr + (size_t)t * (ROLL ? p.n_rows : p.B) * 4 * (PLAIN ? 1 : 0);
  const uint32_t* mask_t = p.mask + (size_t)t * (ROLL ? p.n_rows : p.B) * W * (PLAIN ? 1 : 0);
  float* raw_t = p.raw + (size_t)t * p.B;
  float* shaped_t = p.shaped + (size_t)t * p.B;
  int32_t* done_t = p.done + (size_t)t * p.B;
  const uint8_t* bl_t = p.bl_env ? p.bl_env + (size_t)t * p.bl_stride : nullptr; /* base_line rows may change per step */
  /* the action row of env (index into this step's rows) */
  /* env id (draw streams, action row) of slot env_i minus env_id0: the slot itself unless the rollout handle strides */
  auto idx_of = [&](int env_i) -> uint32_t {
    if constexpr (ROLL) {
      if (p.id_run > 0) return strided_index((uint32_t)env_i, (uint32_t)p.id_run, (uint32_t)p.id_stride);
    }
    return (uint32_t)env_i;
  };
  auto arow = [&](int env_i) -> size_t {
    if constexpr (ROLL) return (size_t)(((uint32_t)p.row_base + idx_of(env_i)) / (uint32_t)p.envs_per_row);
    else return (size_t)env_i;
  };
  if (PLAIN && !ROLL && !last && tid < nb) { /* the next step's action rows of this block: into L2 while this step runs */
    asm volatile("prefetch.global.L2 [%0];" ::"l"(hdr_t + ((size_t)p.B + env0 + tid) * 4));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(mask_t + ((size_t)p.B + env0 + tid) * W));
  }
  for (int i = tid; i < CYG_NKEYS + 7; i += NT) s_cnt[i] = 0; /* ... + one "past pass 0" flag per owning warp */
  __syncthreads(); /* mbarrier initialised, counters zeroed (t > 0: the previous step is complete) */
  CYG_CTA_MARK(1);

  /* ---- sort the block's envs by the action type they will execute (needs only the action headers, so it
   *      overlaps the bulk copies): a warp then runs ONE branch of the 14 defender / 3+X attacker actions ---- */
  int key = 0;
  if (tid < nb) {
    if (!grouped) {
      const size_t r0 = arow(env0 + tid);
      const uint4 hv = *reinterpret_cast<const uint4*>(hdr_t + r0 * 4);
      const uint32_t h0 = hv.x;
      const int blk = bl_t ? (int)bl_t[r0] : p.net.cfg.base_line;
      const int xt = Env<W, 1>::exec_type(p.net.cfg, h0, blk) & 15;
      key = (int)(((h0 >> 8) & 1u) << 4) | xt;
      if (PLAIN && (key == 6 || key == 9)) { /* longest-processing-time first: 8 buckets of 16 listed devices */
        int nd = (int)(hv.z & 0xFFFFu);
        nd = nd < 0 ? 0 : (nd > 127 ? 127 : nd);
        key = CYG_KEY_FLIP0 + 2 * (7 - (nd >> 4)) + (key == 9 ? 1 : 0);
      }
    }
    atomicAdd(&s_cnt[key + 1], 1u);
  }
  __syncthreads();
  if (tid < 32) { /* exclusive prefix over the keys (count of key k sits in s_cnt[k + 1]): one warp, two keys per lane */
    static_assert(CYG_NKEYS > 32 && CYG_NKEYS <= 64, "two keys per lane");
    const uint32_t c0 = s_cnt[1 + tid];
    const uint32_t c1 = tid < CYG_NKEYS - 32 ? s_cnt[33 + tid] : 0u;
    uint32_t x0 = c0, x1 = c1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t y0 = __shfl_up_sync(0xFFFFFFFFu, x0, d), y1 = __shfl_up_sync(0xFFFFFFFFu, x1, d);
      if (tid >= d) { x0 += y0; x1 += y1; }
    }
    const uint32_t total0 = __shfl_sync(0xFFFFFFFFu, x0, 31);
    s_cnt[1 + tid] = x0 - c0;
    if (tid < CYG_NKEYS - 32) s_cnt[33 + tid] = total0 + x1 - c1;
  }
  __syncthreads();
  if (tid < nb) {
    uint32_t pos = atomicAdd(&s_cnt[key + 1], 1u);
    s_perm[pos] = (uint16_t)tid;
  }
  if (t == 0) {
    if (!bulk_ok) {
      for (int i = tid; i < nb * S; i += NT) s_rec[i] = g_rec[i];
    }
    mbar_wait(bar, 0);
  }
  __syncthreads();
  CYG_CTA_MARK(2);

  /* ---- the step in two passes over ONE copy of the thread-per-env code (the loop is not unrolled: step_post alone
   *      is ~10k SASS instructions, and the kernel's instruction footprint is what its warps miss on):
   *      pass 0  thread per env (env perm[tid]): epoch + busy tick, then either the whole rest of the step, or -- for
   *              the draw-heavy actions -- the env is handed to phase B;
   *      pass 1  phase B, warp per env, then the rest of the step (step_post) of those envs by their own threads.
   *      After either pass a warp sends the records its threads finished home (one warp-wide copy per record), so the
   *      write-back of the ~2/3 of the block that phase A completes drains under phase B. ---- */
  constexpr bool coop_ok = PLAIN;
  const bool lower = (tid & ~31) < nb; /* warps that own envs in the thread-per-env phases */
  bool deferred = false;
  const int el = tid < nb ? (int)s_perm[tid] : 0, env = env0 + el;
  Env<W, 1> e(&p.net, nullptr, p.ckpt + (size_t)env * M, p.xtra + (size_t)env * p.net.cfg.xcap,
                 (uint32_t)p.env_id0 + idx_of(env), (uint32_t)(sp.off_recs / 4) + (uint32_t)(el * S), (uint32_t)(sp.off_tables / 4));
  const size_t my_row = arow(env); /* this step's action row of the env this thread owns */
  /* the hop-log ring and the uploaded detector of an env (both optional, global memory) */
  auto bind_aux = [&](Env<W, 1>& ee, int env_i) {
    if constexpr (LOG) {
      ee.logs = p.logs ? p.logs + (size_t)env_i * p.net.cfg.log_cap : nullptr;
      ee.det = (p.det_slots && p.det_of_env[env_i] >= 0) ? p.det_slots + (size_t)p.det_of_env[env_i] * CYG_DET_WORDS : nullptr;
    }
  };
  if (tid < nb) bind_aux(e, env);
  long long t_begin = 0;
#ifdef CYG_PHASE_TIMING
  long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  e.phase_t = ph;
#endif
  int mode = 0;
  uint32_t home_mask = 0; /* lanes of this warp whose env's record is finished and not yet sent home (uniform) */
  auto send_some = [&](int k) {
    while (home_mask && k-- > 0) {
      const int src = __ffs((int)home_mask) - 1;
      home_mask &= home_mask - 1u;
      const int el_s = __shfl_sync(0xFFFFFFFFu, el, src);
      copy_record(g_rec + (size_t)el_s * S, s_rec + el_s * S, S, lane);
    }
  };
#pragma unroll /* two copies of the thread-per-env code: un-unrolled, ptxas spills inside the warp-per-env routines (measured slower) */
  for (int pass = 0; pass < (PLAIN ? 2 : 1); pass++) {
    double cost = 0.0;
    bool dirty = false, do_post = false;
    if (pass == 0) {
      uint32_t act[4 + W]; /* this env's action (group 0), in registers */
      const uint16_t* ord = (!PLAIN && p.order) ? p.order + (size_t)env * p.order_stride : nullptr;
      int atype = 0;
      if (tid < nb) {
        uint4 hv = *reinterpret_cast<const uint4*>(hdr_t + my_row * 4);
        act[0] = hv.x; act[1] = hv.y; act[2] = hv.z; act[3] = hv.w;
#pragma unroll
        for (int w = 0; w < W; w++) act[4 + w] = mask_t[my_row * W + w];
        t_begin = p.dbg_cycles ? clock64() : 0;
        mode = (int)((act[0] >> 8) & 1u);
        if (bl_t) e.bl = (int)bl_t[my_row];
        atype = e.step_pre(act, p.flags);
        deferred = coop_ok && Coop<W>::is_heavy(e, mode, atype) && !(mode == CYG_MODE_ATTACKER && e.bl == CYG_BL_NO_ATTACK);
      }
      if (coop_ok) {
        /* once every env has its epoch open and its busy tick done (s_cnt[CYG_NKEYS + 6] counts the owning warps that
         * got there) phase B may touch any deferred env: the warps that own no env start it right away, the owning
         * warps join after their thread-per-env work -- and check the same counter, a warp whose envs are all deferred
         * gets to phase B before the others are through step_pre */
        const uint32_t dmask = __ballot_sync(0xFFFFFFFFu, deferred);
        if (lower) {
          __syncwarp();
          if (lane == 0) { s_def[tid >> 5] = dmask; __threadfence_block(); atomicAdd(&s_cnt[CYG_NKEYS + 6], 1u); }
        }
      }
      if (tid < nb && !deferred) {
        if (PLAIN) e.template step_act<true>(act, act + 4, nullptr, 0, 0, 0, 1, p.flags, atype, cost, dirty);
        else if (!grouped) e.step_act(act, act + 4, ord, 0, 0, 0, 1, p.flags, atype, cost, dirty);
        else e.step_act(hdr_t + (size_t)env * 4, mask_t + (size_t)env * W, ord, (size_t)p.B * 4, (size_t)p.B * W,
                        (size_t)p.B * p.order_stride, p.G, p.flags, atype, cost, dirty);
        do_post = true;
      }
    } else {
      if constexpr (PLAIN) {
  CYG_CTA_MARK(3);
        if (lane == 0) while (atomicAdd(&s_cnt[CYG_NKEYS + 6], 0u) < (uint32_t)((nb + 31) >> 5)) __nanosleep(32);
        __syncwarp();
        auto load_action = [&](size_t row_b, uint32_t* act) {
          const uint4 hv = __ldg(reinterpret_cast<const uint4*>(hdr_t + row_b * 4)); /* phase A read these lines: L1 */
          act[0] = hv.x; act[1] = hv.y; act[2] = hv.z; act[3] = hv.w;
#pragma unroll
          for (int w = 0; w < W; w++) act[4 + w] = __ldg(mask_t + row_b * W + w);
        };
        /* B1: block / unblock (keys 6, 9; the longest lists first), B2: attacker exploit + lateral movement (key 16|1),
         * B3: clean / revert / upgrade (keys 1, 3, 4).  One env per warp; perm[] holds each kind as a contiguous run. */
#pragma unroll
        for (int kind = 0; kind < 3; kind++) {
          int lo0, n0, lo1 = 0, n1 = 0, lo2 = 0, n2 = 0;
          if (kind == 0) { lo0 = (int)s_cnt[CYG_KEY_FLIP0]; n0 = (int)s_cnt[CYG_NKEYS] - lo0; }
          else if (kind == 1) { lo0 = (int)s_cnt[17]; n0 = (int)s_cnt[18] - lo0; }
          else {
            lo0 = (int)s_cnt[1]; n0 = (int)s_cnt[2] - lo0; lo1 = (int)s_cnt[3]; n1 = (int)s_cnt[4] - lo1;
            lo2 = (int)s_cnt[4]; n2 = (int)s_cnt[5] - lo2;
          }
          const int ntasks = n0 + n1 + n2;
          for (;;) {
            int task = 0;
            if (lane == 0) task = (int)atomicAdd(&s_cnt[CYG_NKEYS + 1 + kind], 1u);
            task = __shfl_sync(0xFFFFFFFFu, task, 0);
            if (task >= ntasks) break;
            const int ppos = task < n0 ? lo0 + task : (task < n0 + n1 ? lo1 + task - n0 : lo2 + task - n0 - n1);
            if (!((s_def[ppos >> 5] >> (ppos & 31)) & 1u)) continue; /* its own thread did it in phase A */
            const int el_b = s_perm[ppos];
            const int env_b = env0 + el_b;
            Env<W, 1> eb(&p.net, nullptr, p.ckpt + (size_t)env_b * M, p.xtra + (size_t)env_b * p.net.cfg.xcap,
                            (uint32_t)p.env_id0 + idx_of(env_b), (uint32_t)(sp.off_recs / 4) + (uint32_t)(el_b * S), (uint32_t)(sp.off_tables / 4));
            const size_t row_b = arow(env_b);
            eb.resume_epoch();
            if (LOG && kind == 1) eb.logs = p.logs ? p.logs + (size_t)env_b * p.net.cfg.log_cap : nullptr; /* the attack logs its hops */
            uint32_t act[4 + W];
            load_action(row_b, act);
            typename Env<W, 1>::Act a;
            Env<W, 1>::decode(act, act + 4, nullptr, a);
            double tcost = 0.0;
            bool tdirty = false;
            long long tb0 = p.dbg_cycles ? clock64() : 0;
            if (lane == 0) eb.load_costs();
            if (kind == 0) {
              Coop<W>::template flip<32>(eb, a, (int)(act[0] & 0xFFu), tcost, tdirty); /* flip keys only hold executed types 6 / 9 == the header's */
            } else if (kind == 1) {
              Coop<W>::template attack<LOG>(eb, a);
            } else {
              const int atype_b = Env<W, 1>::exec_type(p.net.cfg, act[0], bl_t ? (int)bl_t[row_b] : p.net.cfg.base_line);
              Coop<W>::defender(eb, a, atype_b, tcost, tdirty);
            }
            if (lane == 0) {
#if !defined(CYG_PHASE_TIMING) && !defined(CYG_CTA_TIMING)
              if (p.dbg_cycles) p.dbg_cycles[env_b] = (unsigned long long)(clock64() - tb0); /* heavy envs: phase-B cycles */
#endif
#ifdef CYG_COUNT_ROUNDS
              if (p.dbg_cycles && kind == 0) p.dbg_cycles[env_b] = (unsigned long long)eb.dbg_rounds;
#endif
              eb.store_costs();
              s_out[el_b] = (float)tcost;
              s_out[NB + el_b] = __int_as_float(tdirty ? 1 : 0);
            }
            __syncwarp();
          }
          CYG_WARP_MARK(kind);
        }
        __syncthreads();
  CYG_CTA_MARK(4);
        /* ---- phase C, thread per env again: the rest of the step for the envs phase B handled ---- */
        if (deferred) {
          e = Env<W, 1>(&p.net, nullptr, p.ckpt + (size_t)env * M, p.xtra + (size_t)env * p.net.cfg.xcap, (uint32_t)p.env_id0 + idx_of(env),
                           (uint32_t)(sp.off_recs / 4) + (uint32_t)(el * S), (uint32_t)(sp.off_tables / 4)); /* nothing of it stays live across phase B */
          if (bl_t) e.bl = (int)bl_t[my_row];
          bind_aux(e, env);
          e.resume_epoch();
          cost = (double)s_out[el];
          dirty = __float_as_int(s_out[NB + el]) != 0;
          do_post = true;
        }
      }
    }
    if (do_post) {
      float raw, shaped;
      int32_t done;
      e.step_post(mode, cost, dirty, p.flags, &raw, &shaped, &done, p.pre_masks ? p.pre_masks + (size_t)env * 3 * W : nullptr);
      if constexpr (ROLL) p.ret_acc[(size_t)mode * p.B + env] += (double)raw;
      else { raw_t[env] = raw; shaped_t[env] = shaped; done_t[env] = done; }
    }
    if (pass == 0 && tid < nb) {
#ifdef CYG_PHASE_TIMING
      if (p.dbg_cycles) for (int i = 0; i < 8; i++) p.dbg_cycles[(size_t)env * 8 + i] = (unsigned long long)(ph[i] - t_begin);
#elif !defined(CYG_CTA_TIMING)
      if (p.dbg_cycles && !deferred) p.dbg_cycles[env] = (unsigned long long)(clock64() - t_begin);
#endif
    }
    if (PLAIN && last && lower) {
      /* The records this warp's threads just finished go home by warp-wide copies, right away.  Measured alternatives:
       * 4 records after each phase-B task of the warp (38.3 / 50.5 us fused / single against 37.8 / 48.1), a shared
       * claim counter with 4 records per claim (37.8 / 49.5), ONE warp copying for the whole block (45.1 / 67.5: a
       * single warp cannot keep enough stores in flight), per-warp step_post batches right after the warp's phase-B
       * tasks instead of the barrier + phase C (42.3 / 49.1: the ~10k-cycle chain runs with a handful of lanes). */
      home_mask = __ballot_sync(0xFFFFFFFFu, do_post);
      send_some(32);
    }
  }
  __syncthreads();
  CYG_CTA_MARK(5);
  } /* fused steps */

  /* ---- optional fused observation rows (post-evolve view, CyberDefenseEnv.py:146-257) ---- */
  if (p.obs && p.obs_mode) {
    const int dim = p.obs_mode == 2 ? 4 * M + p.net.cfg.X : 6 * M;
    observe_rows<W>(p.net, s_rec, S, nb, p.obs_mode, p.obs + (size_t)env0 * dim, tid >> 5, NT >> 5, lane);
  }

  /* ---- write the block's records back ---- */
  if constexpr (PLAIN) { /* every warp sent its records home already */
    CYG_CTA_MARK(6);
  } else
#ifdef CYG_TMA_STORE
  if (bulk_ok) { /* one bulk store; every writer fences generic -> async proxy first */
    fence_proxy_async();
    __syncthreads();
    CYG_CTA_MARK(6);
    if (tid == 0) {
      bulk_s2g(g_rec, s_rec, rec_bytes);
      bulk_commit_wait_read();
    }
  } else
#endif
  {
    /* coalesced 16-byte stores by all warps (tail blocks whose span is not 16-byte sized / aligned) */
    if (bulk_ok) {
      const uint4* s4 = reinterpret_cast<const uint4*>(s_rec);
      uint4* g4 = reinterpret_cast<uint4*>(g_rec);
      const int n4 = (int)(rec_bytes >> 4);
      for (int i = tid; i < n4; i += NT) g4[i] = s4[i];
    } else {
      for (int i = tid; i < nb * S; i += NT) g_rec[i] = s_rec[i];
    }
    CYG_CTA_MARK(6);
  }
}

/* ---- large networks (128 < M <= 2048, BASELINE.json config C4): the adjacency bit matrix (M x 64 words) exceeds
 *      shared memory, so this first correct path steps one env per thread straight on the records in global
 *      memory with the tables read through L2.  Same transition code (cyg_core.cuh), no staging, no sort. ---- */
template <int W>
__global__ void __launch_bounds__(256) cyg_step_generic_kernel(const __grid_constant__ StepParams p) {
  /* block_envs envs per CTA, spread over all SMs (B = 1024 -> 7 per CTA); their records (~6.4 KB each at M = 2000) are
   * staged in shared memory by coalesced copies.  Phase A, thread per env: epoch, busy tick and the actions whose cost
   * is a few passes over the 64-word planes.  Phase B, warp per env: block / unblock and the lateral-movement scan
   * (BigCoop, cyg_coop.cuh) -- one thread walking ~1000 listed devices or ~800 sources over 64-word rows took 6-9 ms
   * per launch.  Phase C, thread per env: the rest of the step. */
  const int NB = p.block_envs, S = p.net.S, M = p.net.M, tid = threadIdx.x, NT = blockDim.x, lane = tid & 31;
  const int env0 = blockIdx.x * NB, nb = min(NB, p.B - env0), Wm = p.net.Wm;
  uint32_t* g_rec = p.recs + (size_t)env0 * S;
  uint32_t* s_misc = cyg_smem + (size_t)NB * S + 4; /* per env: heavy kind, cost (float bits), dirty, atype */
  const uint32_t tab_off = (uint32_t)(NB * S + 4 + 4 * NB); /* the hot tables (masks, device ranges, unit table = CSR) behind them */
  for (int i = tid; i < nb * S; i += NT) cyg_smem[i] = g_rec[i];
  for (int i = tid; i < (int)p.net.hot_words; i += NT) cyg_smem[tab_off + i] = p.net.blob[i];
  __syncthreads();
  const bool plain = !(p.flags & CYG_STEP_GROUPED) && p.order == nullptr;
  const int env = env0 + tid;
  int mode = 0;
  if (tid < nb) {
    Env<W, 2> e(&p.net, nullptr, p.ckpt + (size_t)env * M, p.xtra + (size_t)env * p.net.cfg.xcap, (uint32_t)(p.env_id0 + env), (uint32_t)(tid * S), tab_off);
    if (p.bl_env) e.bl = (int)p.bl_env[env];
    e.logs = p.logs ? p.logs + (size_t)env * p.net.cfg.log_cap : nullptr;
    e.det = (p.det_slots && p.det_of_env[env] >= 0) ? p.det_slots + (size_t)p.det_of_env[env] * CYG_DET_WORDS : nullptr;
    const uint32_t* hdr = p.hdr + (size_t)env * 4;
    const uint16_t* ord = p.order ? p.order + (size_t)env * p.order_stride : nullptr;
    mode = (int)((hdr[0] >> 8) & 1u);
    int atype = e.step_pre(hdr, p.flags);
    int heavy = 0;
    if (plain) {
      if (mode == CYG_MODE_DEFENDER && (atype == 6 || atype == 9)) heavy = 1;
      if (mode == CYG_MODE_ATTACKER && atype == 1 && e.bl != CYG_BL_NO_ATTACK) heavy = 2;
    }
    double cost = 0.0;
    bool dirty = false;
    if (!heavy) atype = e.step_act(hdr, p.mask + (size_t)env * Wm, ord, (size_t)p.B * 4, (size_t)p.B * Wm, (size_t)p.B * p.order_stride, p.G, p.flags, atype, cost, dirty);
    s_misc[4 * tid] = (uint32_t)heavy; s_misc[4 * tid + 1] = __float_as_uint((float)cost); s_misc[4 * tid + 2] = dirty ? 1u : 0u; s_misc[4 * tid + 3] = (uint32_t)atype;
  }
  __syncthreads();
  for (int el = tid >> 5; el < nb; el += NT >> 5) { /* phase B: one warp per heavy env */
    const int heavy = (int)s_misc[4 * el];
    if (!heavy) continue;
    const int env_b = env0 + el;
    Env<W, 2> e(&p.net, nullptr, p.ckpt + (size_t)env_b * M, p.xtra + (size_t)env_b * p.net.cfg.xcap, (uint32_t)(p.env_id0 + env_b), (uint32_t)(el * S), tab_off);
    if (p.bl_env) e.bl = (int)p.bl_env[env_b];
    e.logs = p.logs ? p.logs + (size_t)env_b * p.net.cfg.log_cap : nullptr;
    e.resume_epoch();
    typename Env<W, 2>::Act a;
    Env<W, 2>::decode(p.hdr + (size_t)env_b * 4, p.mask + (size_t)env_b * Wm, nullptr, a);
    double cost = 0.0;
    bool dirty = false;
    if (lane == 0) e.load_costs();
    const bool done = heavy == 1 ? BigCoop<W>::flip(e, a, (int)s_misc[4 * el + 3], cost, dirty) : BigCoop<W>::attack(e, a);
    if (lane == 0) {
      if (!done) { /* extra edges / inconsistent header: the one-lane form */
        int at = (int)s_misc[4 * el + 3];
        e.step_act(p.hdr + (size_t)env_b * 4, p.mask + (size_t)env_b * Wm, nullptr, 0, 0, 0, 1, p.flags, at, cost, dirty);
      } else {
        e.store_costs();
      }
      s_misc[4 * el + 1] = __float_as_uint((float)cost); s_misc[4 * el + 2] = dirty ? 1u : 0u;
    }
    __syncwarp();
  }
  __syncthreads();
  if (tid < nb) {
    Env<W, 2> e(&p.net, nullptr, p.ckpt + (size_t)env * M, p.xtra + (size_t)env * p.net.cfg.xcap, (uint32_t)(p.env_id0 + env), (uint32_t)(tid * S), tab_off);
    if (p.bl_env) e.bl = (int)p.bl_env[env];
    e.resume_epoch();
    float raw, shaped;
    int32_t done;
    e.step_post(mode, (double)__uint_as_float(s_misc[4 * tid + 1]), s_misc[4 * tid + 2] != 0, p.flags, &raw, &shaped, &done,
                p.pre_masks ? p.pre_masks + (size_t)env * 3 * Wm : nullptr);
    p.raw[env] = raw; p.shaped[env] = shaped; p.done[env] = done;
  }
  __syncthreads();
  for (int i = tid; i < nb * S; i += NT) g_rec[i] = cyg_smem[i];
}

/* ---- randomize_compromise_and_ownership: thread per env on the global record ---- */
struct SimpleParams {
  Net net;
  uint32_t* recs;
  uint32_t* xtra;
  const uint8_t* env_mask;
  uint32_t* hdr;
  uint32_t* mask;
  int B, env_id0, mode;
  uint16_t* order;  /* optional [B][order_stride]: device_indices in draw order (cyg_sample_actions_ordered) */
  int order_stride;
  int id_run, id_stride; /* cyg_set_env_id_stride */
  __device__ __forceinline__ uint32_t env_id(int slot) const {
    return (uint32_t)env_id0 + (id_run > 0 ? strided_index((uint32_t)slot, (uint32_t)id_run, (uint32_t)id_stride) : (uint32_t)slot);
  }
};

template <int W>
__global__ void cyg_randomize_kernel(const __grid_constant__ SimpleParams p) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= p.B) return;
  if (p.env_mask && !p.env_mask[env]) return;
  Env<W> e(&p.net, p.recs + (size_t)env * p.net.S, nullptr, p.xtra + (size_t)env * p.net.cfg.xcap, p.env_id(env));
  e.randomize();
}

/* _rebuild_graph_cache() called from outside a step (DoubleOracle.restore, do_agent.py:891-895; reset(from_init),
 * volt:1933-1936): the rebuilt cache forgets every block (volt:476).  New edges are visible to the kernels at once. */
template <int W>
__global__ void cyg_rebuild_kernel(const __grid_constant__ SimpleParams p) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= p.B) return;
  if (p.env_mask && !p.env_mask[env]) return;
  Env<W> e(&p.net, p.recs + (size_t)env * p.net.S, nullptr, p.xtra + (size_t)env * p.net.cfg.xcap, p.env_id(env));
  e.rebuild_cache();
}

template <int W>
__global__ void cyg_sample_kernel(const __grid_constant__ SimpleParams p) {
  int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= p.B) return;
  uint32_t rec[CYG_NSCAL];
  uint32_t* g = p.recs + (size_t)env * p.net.S;
  for (int i = 0; i < CYG_NSCAL; i++) rec[i] = g[i];
  Env<W> e(&p.net, rec, nullptr, nullptr, p.env_id(env));
  uint32_t h[4], m[W];
  e.sample_action(p.mode, h, m, p.order ? p.order + (size_t)env * p.order_stride : nullptr);
  g[CYG_S_EPOCH] = rec[CYG_S_EPOCH];
  for (int i = 0; i < 4; i++) p.hdr[(size_t)env * 4 + i] = h[i];
  for (int w = 0; w < W; w++) if (w < p.net.Wm) p.mask[(size_t)env * p.net.Wm + w] = m[w];
}

/* ---- canonical <-> internal conversion: one warp per env, ballots build the planes ---- */
struct ConvParams {
  Net net;
  uint32_t* recs;
  uint32_t* ckpt_int;
  uint32_t* xtra_int;
  uint32_t *dev, *ckpt, *blocked, *extra, *scal;
  int B;
  uint32_t* logs_int; /* [B][log_cap] internal ring */
  uint32_t* logs;     /* optional canonical [B][log_cap] */
};

template <int W>
__global__ void cyg_import_kernel(const __grid_constant__ ConvParams p) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= p.B) return;
  const Net& n = p.net;
  uint32_t* rec = p.recs + (size_t)warp * n.S;
  const int M = n.M;
  uint32_t err = 0;
  for (int w = 0; w < W; w++) {
    int d = w * 32 + lane;
    uint32_t x = d < M ? p.dev[(size_t)warp * M + d] : 0u;
    uint32_t b = (x >> CYG_DEV_BUSY_SHIFT) & CYG_DEV_BUSY_MASK;
    if (b > CYG_BUSY_MAX) { b = CYG_BUSY_MAX; err = CYG_FL_ERR_BUSY; }
    const uint32_t cbits[7] = {CYG_DEV_COMP, CYG_DEV_KNOWN, CYG_DEV_NYA, CYG_DEV_OWNED, CYG_DEV_HASWL, CYG_DEV_BUSYSET, CYG_DEV_ACTSET};
    for (int pnum = 0; pnum < 7; pnum++) { /* planes P_COMP .. P_ACTSET */
      uint32_t m = __ballot_sync(0xFFFFFFFFu, (x & cbits[pnum]) != 0);
      if (lane == 0) rec[CYG_REC_PLANES + pnum * W + w] = m;
    }
    uint32_t pt = (x >> CYG_DEV_PT_SHIFT) & CYG_DEV_PT_MASK;
    for (int k = 0; k < 3; k++) {
      uint32_t m = __ballot_sync(0xFFFFFFFFu, (pt >> k) & 1u);
      if (lane == 0) rec[CYG_REC_PLANES + (P_PT0 + k) * W + w] = m;
    }
    for (int k = 0; k < 4; k++) {
      uint32_t m = __ballot_sync(0xFFFFFFFFu, (b >> k) & 1u);
      if (lane == 0) rec[CYG_REC_PLANES + (P_BUSY0 + k) * W + w] = m;
    }
    uint32_t cb = (x >> CYG_DEV_CBY_SHIFT) & CYG_DEV_CBY_MASK;
    for (int k = 0; k < n.ncby; k++) {
      uint32_t m = __ballot_sync(0xFFFFFFFFu, (cb >> k) & 1u);
      if (lane == 0) rec[CYG_REC_PLANES + (P_CBY0 + k) * W + w] = m;
    }
    if (d < M) p.ckpt_int[(size_t)warp * M + d] = ((p.ckpt ? p.ckpt[(size_t)warp * M + d] : 0u) & ~CYG_CKI_REMOVED) | ((x & CYG_DEV_REMOVED) ? CYG_CKI_REMOVED : 0u);
  }
  err = __reduce_or_sync(0xFFFFFFFFu, err);
  if (lane < CYG_NSCAL) {
    uint32_t v = p.scal[(size_t)warp * CYG_NSCAL + lane];
    if (lane == CYG_S_FLAGS) v |= err;
    rec[lane] = v;
  }
  /* canonical blocked[] (bit e = base pair e) -> the unit bitset: zero it, then every blocked pair sets its 2 m units */
  for (int i = n.off_inc + lane; i < n.S; i += 32) rec[i] = 0u;
  __syncwarp();
  uint32_t nblk = 0;
  const uint32_t* bo = p.blocked + (size_t)warp * n.EW;
  for (int i = lane; i < n.EW; i += 32) {
    uint32_t x = bo[i];
    if (i == n.EW - 1 && (n.E & 31)) x &= (1u << (n.E & 31)) - 1u;
    if (n.E == 0) x = 0;
    nblk += (uint32_t)__popc(x);
    while (x) {
      const int e = i * 32 + __ffs((int)x) - 1;
      x &= x - 1;
      pair_units(&n, e, [&](int wi, uint32_t m) { atomicOr(&rec[n.off_inc + wi], m); });
    }
  }
  nblk = __reduce_add_sync(0xFFFFFFFFu, nblk);
  for (int i = lane; i < n.cfg.xcap; i += 32) p.xtra_int[(size_t)warp * n.cfg.xcap + i] = p.extra[(size_t)warp * n.cfg.xcap + i];
  __syncwarp();
  if (lane == 0) rec[n.off_aux] = nblk;
  if (p.logs_int) /* the hop-log ring (zeroed when the caller has none to import) */
    for (int i = lane; i < n.cfg.log_cap; i += 32) p.logs_int[(size_t)warp * n.cfg.log_cap + i] = p.logs ? p.logs[(size_t)warp * n.cfg.log_cap + i] : 0u;
}

template <int W>
__global__ void cyg_export_kernel(const __grid_constant__ ConvParams p) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= p.B) return;
  const Net& n = p.net;
  const uint32_t* rec = p.recs + (size_t)warp * n.S;
  const int M = n.M;
  for (int w = 0; w < W; w++) {
    int d = w * 32 + lane;
    if (d >= M) continue;
    uint32_t ck = p.ckpt_int[(size_t)warp * M + d];
    p.dev[(size_t)warp * M + d] = export_device<W>(&n, rec, d, ck);
    if (p.ckpt) p.ckpt[(size_t)warp * M + d] = ck & ~CYG_CKI_REMOVED;
  }
  if (lane < CYG_NSCAL) p.scal[(size_t)warp * CYG_NSCAL + lane] = rec[lane];
  for (int i = lane; i < n.EW; i += 32) {
    uint32_t x = 0;
    for (int j = 0; j < 32 && i * 32 + j < n.E; j++) x |= (pair_blocked(&n, rec, i * 32 + j) ? 1u : 0u) << j;
    p.blocked[(size_t)warp * n.EW + i] = x;
  }
  for (int i = lane; i < n.cfg.xcap; i += 32) p.extra[(size_t)warp * n.cfg.xcap + i] = p.xtra_int[(size_t)warp * n.cfg.xcap + i];
  if (p.logs && p.logs_int)
    for (int i = lane; i < n.cfg.log_cap; i += 32) p.logs[(size_t)warp * n.cfg.log_cap + i] = p.logs_int[(size_t)warp * n.cfg.log_cap + i];
}

/* ---- IPPO / MAPPO glue: per-device action types -> the per-type action groups of one grouped step (IPPO.py:559-570),
 *      with the role's visibility mask (build_visibility_mask, IPPO.py:74-96) read straight from the bit-planes.
 *      One warp per env, lanes on 32 devices; group g = the g-th action type other than the no-op. ---- */
struct GroupParams {
  Net net;
  const uint32_t* recs;
  const int32_t* types;   /* [B][M] action type each device drew */
  const int32_t* exp_idx; /* [B] */
  const int32_t* app_idx; /* [B] */
  const uint8_t* visible; /* optional [B][M]: the policy's own mask (> 0 = the device counts), ANDed with the role's */
  const int32_t* single;  /* optional [B][2]: device kept for the single-device types 11 / 12 (random.choice, IPPO.py:567) */
  uint32_t* hdr;          /* [n_types - 1][B][4] */
  uint32_t* mask;         /* [n_types - 1][B][Wm] */
  int B, mode, role, n_types, noop;
};
#if defined(CYG_TU_W) && CYG_TU_W == 4 /* one copy: the kernel is not templated on the plane width */
/* the groups of ONE env by one warp: lane g < G ends up with group g's device words (handed to `put` word by word) and its
 * header (returned through h4) */
template <typename Put>
__device__ __forceinline__ void group_one_env(const GroupParams& p, int b, int lane, uint32_t* slot, uint32_t h4[4], Put put) {
  const Net& n = p.net;
  const int M = n.M, Wm = n.Wm, Wp = n.W;
  const uint32_t* pl = p.recs + (size_t)b * n.S + CYG_REC_PLANES;
  const int G = p.n_types - 1;
  int ndev = 0;            /* lane g: devices of group g */
  int first = -1;          /* lane g: lowest device of group g */
  const int t_mine = lane < G ? (lane < p.noop ? lane : lane + 1) : -1; /* the type of group `lane` */
  for (int w = 0; w < Wm; w++) {
    const int d = 32 * w + lane;
    uint32_t vis = 0xFFFFFFFFu;
    if (p.role == 1) vis = ~pl[P_NYA * Wp + w] & pl[P_OWNED * Wp + w];
    else if (p.role == 2) vis = ~pl[P_NYA * Wp + w] & pl[P_OWNED * Wp + w] & pl[P_KNOWN * Wp + w];
    const int ty = d < M ? p.types[(size_t)b * M + d] : -1;
    const bool on = d < M && ((vis >> lane) & 1u) && (!p.visible || p.visible[(size_t)b * M + d] != 0);
    /* lanes with the same type find each other with ONE match (13 ballots + selects before: the kernel was bound by its
     * instruction count, 60 us for 65 536 envs); the lowest lane of every type posts the set, lane g picks up its type's */
    slot[lane] = 0u;
    slot[lane + 32] = 0u;
    __syncwarp();
    const uint32_t same = __match_any_sync(0xFFFFFFFFu, on ? ty : -1);
    if (on && ty >= 0 && ty < 64 && (same & ((1u << lane) - 1u)) == 0u) slot[ty] = same;
    __syncwarp();
    uint32_t mine = lane < G ? slot[t_mine] : 0u;
    __syncwarp();
    if (lane < G) {
      if (t_mine == 11 || t_mine == 12) { /* single-device types: the chosen device if it is in the set, else (no choice given) the lowest */
        if (p.single) {
          const int c = p.single[(size_t)b * 2 + (t_mine - 11)];
          mine &= (c >= 32 * w && c < 32 * w + 32) ? (1u << (c & 31)) : 0u;
        } else {
          mine = first < 0 ? (mine & (0u - mine)) : 0u;
        }
      }
      if (mine && first < 0) first = 32 * w + __ffs((int)mine) - 1;
      ndev += __popc(mine);
      put(w, mine);
    }
  }
  const int at = ndev > 0 ? t_mine : p.noop;
  h4[0] = (uint32_t)(at & 0xFF) | ((uint32_t)p.mode << 8) | (1u << 16);
  h4[1] = (uint32_t)(p.exp_idx ? p.exp_idx[b] : 0) & 0xFFu;
  h4[2] = (uint32_t)ndev;
  h4[3] = (uint32_t)(p.app_idx ? p.app_idx[b] : 0);
}

/* any plane width: one warp per env, every lane < G writes its group's words straight to [g][b] (4-byte pieces, one per
 * group and word: fine for the few envs of a large network) */
__global__ void cyg_group_kernel(const __grid_constant__ GroupParams p) {
  const int b = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = (int)(threadIdx.x & 31);
  if (b >= p.B) return;
  const int G = p.n_types - 1, Wm = p.net.Wm;
  __shared__ uint32_t s_slot[4][64]; /* per warp: the device set of every type, one plane word at a time */
  uint32_t h4[4];
  uint32_t* const mrow = p.mask + ((size_t)lane * p.B + b) * Wm;
  if (Wm == 4 && (((uintptr_t)p.mask) & 15) == 0) { /* the outputs are [g][b][..]: ONE 16-byte store per group instead of four 4-byte pieces */
    uint32_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
    group_one_env(p, b, lane, s_slot[(threadIdx.x >> 5) & 3], h4, [&](int w, uint32_t m) { m0 = w == 0 ? m : m0; m1 = w == 1 ? m : m1; m2 = w == 2 ? m : m2; m3 = w == 3 ? m : m3; });
    if (lane < G) *reinterpret_cast<uint4*>(mrow) = make_uint4(m0, m1, m2, m3);
  } else {
    group_one_env(p, b, lane, s_slot[(threadIdx.x >> 5) & 3], h4, [&](int w, uint32_t m) { mrow[w] = m; });
  }
  if (lane < G) *reinterpret_cast<uint4*>(p.hdr + ((size_t)lane * p.B + b) * 4) = make_uint4(h4[0], h4[1], h4[2], h4[3]);
}

#endif

/* cyg_unpack_actions: compact action rows [B][2 + Wm] (include/cygym_b200.h) -> hdr [B][4] + mask [B][Wm].  One thread
 * per env; the rows are what a host-buffer step moves over PCIe (24 bytes per env at M <= 128 instead of 32). */
struct UnpackParams {
  const uint32_t* rows;
  uint32_t* hdr;
  uint32_t* mask;
  int B, Wm;
};
#if defined(CYG_TU_W) && CYG_TU_W == 4
__global__ void cyg_unpack_kernel(const __grid_constant__ UnpackParams p) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= p.B) return;
  const uint32_t* r = p.rows + (size_t)env * (2 + p.Wm);
  const uint32_t w0 = r[0], w1 = r[1];
  uint32_t exw = 0;
#pragma unroll
  for (int i = 0; i < 4; i++) { /* four signed 4-bit exploit indices -> four signed bytes */
    const int x = (int)((w1 >> (4 * i)) & 15u);
    exw |= (uint32_t)((x >= 8 ? x - 16 : x) & 0xFF) << (8 * i);
  }
  const int app = (int)(int16_t)(w1 >> 16);
  uint4 h;
  h.x = (w0 & 0x1FFu) | (((w0 >> 9) & 7u) << 16);       /* type | mode << 8 | n_ex << 16 */
  h.y = exw;
  h.z = ((w0 >> 12) & 0xFFFu) | ((w0 >> 24) << 16);     /* n_dev | (first + 1) << 16 */
  h.w = (uint32_t)app;
  *reinterpret_cast<uint4*>(p.hdr + (size_t)env * 4) = h;
  for (int w = 0; w < p.Wm; w++) p.mask[(size_t)env * p.Wm + w] = r[2 + w];
}
extern "C" void cyg_unpack_launch(int blocks, int threads, cudaStream_t st, const UnpackParams& p) { cyg_unpack_kernel<<<blocks, threads, 0, st>>>(p); }
/* cyg_pack_done: done flags [B] (int32) -> one bit per env (bit b % 32 of word b / 32) */
__global__ void cyg_pack_done_kernel(const int32_t* done, uint32_t* bits, int B) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t m = __ballot_sync(0xFFFFFFFFu, env < B && done[env] != 0);
  if ((threadIdx.x & 31) == 0 && env < B) bits[env >> 5] = m;
}
extern "C" void cyg_pack_done_launch(int blocks, int threads, cudaStream_t st, const int32_t* done, uint32_t* bits, int B) {
  cyg_pack_done_kernel<<<blocks, threads, 0, st>>>(done, bits, B);
}
#endif

/* ---- detector fits (cyg_fit_detectors; cyg_iforest.cuh) ---- */
struct FitParams {
  uint32_t* recs;          /* internal records [B][S] (the scalars lead each) */
  const uint32_t* logs;    /* internal hop-log rings [B][log_cap], NULL when log_cap == 0 */
  uint32_t* slots;         /* detector slots [n_slots][CYG_DET_WORDS] */
  int32_t* det_of_env;     /* [B] */
  const uint32_t* seeds;   /* [B] */
  int32_t* next_slot;      /* first free slot */
  int32_t* work;           /* [2 + B]: envs to fit, the fit kernel's cursor, their list */
  int S, B, log_cap, n_slots;
};
#define CYG_FIT_WARPS 4 /* fitting warps per CTA (cyg_iforest::Scratch each, in shared memory) */
#if defined(CYG_TU_W) && CYG_TU_W == 4
/* Block-wide exclusive count of `v` over the threads below this one; *total = count over the block. */
__device__ __forceinline__ int block_rank(bool v, int* warp_tot, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
  const uint32_t m = __ballot_sync(0xFFFFFFFFu, v);
  if (lane == 0) warp_tot[warp] = __popc(m);
  __syncthreads();
  int before = 0, all = 0;
  for (int w = 0; w < nwarps; w++) {
    before += w < warp ? warp_tot[w] : 0;
    all += warp_tot[w];
  }
  __syncthreads();
  *total = all;
  return before + __popc(m & ((1u << lane) - 1u));
}
/* One CTA walks the envs in order: slots go to pending envs without one in env order (deterministic, and the same
 * order service_detectors() uses); the envs that can be fitted are listed for cyg_fit_kernel. */
__global__ void __launch_bounds__(1024) cyg_fit_assign_kernel(const __grid_constant__ FitParams p) {
  __shared__ int warp_tot[32];
  const int first = *p.next_slot;
  int taken = 0, listed = 0;
  for (int c = 0; c < p.B; c += blockDim.x) {
    const int b = c + (int)threadIdx.x;
    bool pend = false, fits_ring = false;
    int cur = -1;
    uint32_t flags = 0;
    if (b < p.B) {
      const uint32_t* sc = p.recs + (size_t)b * p.S;
      flags = sc[CYG_S_FLAGS];
      pend = (flags & CYG_FL_DET_PENDING) != 0;
      if (pend) {
        const uint32_t nl = sc[CYG_S_LOGS];
        const uint32_t win = nl < (uint32_t)CYG_DET_WINDOW ? nl : (uint32_t)CYG_DET_WINDOW;
        fits_ring = p.logs != nullptr && win >= 1u && win <= (uint32_t)p.log_cap;
        cur = p.det_of_env[b];
      }
    }
    const bool need = pend && fits_ring && cur < 0;
    int n_need, n_ok;
    const int slot = first + taken + block_rank(need, warp_tot, &n_need);
    const bool ok = pend && fits_ring && (cur >= 0 || slot < p.n_slots);
    const int at = listed + block_rank(ok, warp_tot, &n_ok);
    if (need && slot < p.n_slots) p.det_of_env[b] = slot;
    if (pend && !ok) p.recs[(size_t)b * p.S + CYG_S_FLAGS] = flags | CYG_FL_ERR_DETECTOR;
    if (ok) p.work[2 + at] = b;
    taken += n_need;
    listed += n_ok;
  }
  if (threadIdx.x == 0) {
    const int next = first + taken;
    *p.next_slot = next <= p.n_slots ? next : (first > p.n_slots ? first : p.n_slots);
    p.work[0] = listed;
    p.work[1] = 0;
  }
}
/* Persistent warps take the listed envs one by one: lane 0 runs the serial fit (streams, row sampling, tree builds)
 * in shared memory, all lanes zero the slot and fill the verdict table. */
__global__ void __launch_bounds__(32 * CYG_FIT_WARPS) cyg_fit_kernel(const __grid_constant__ FitParams p) {
  extern __shared__ __align__(16) unsigned char fit_smem[];
  iforest::Scratch& s = reinterpret_cast<iforest::Scratch*>(fit_smem)[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int n = p.work[0];
  for (;;) {
    int i = 0;
    if (lane == 0) i = atomicAdd(&p.work[1], 1);
    i = __shfl_sync(0xFFFFFFFFu, i, 0);
    if (i >= n) break;
    const int b = p.work[2 + i];
    uint32_t* slot = p.slots + (size_t)p.det_of_env[b] * CYG_DET_WORDS;
    uint32_t* sc = p.recs + (size_t)b * p.S;
    for (int w = lane; w < CYG_DET_WORDS; w += 32) slot[w] = 0u;
    __syncwarp();
    if (lane == 0) iforest::fit_serial(s, p.logs + (size_t)b * p.log_cap, (uint32_t)p.log_cap, sc[CYG_S_LOGS], p.seeds[b], slot);
    __syncwarp();
    iforest::verdict_words(s, slot, lane, 32);
    if (lane == 0) sc[CYG_S_FLAGS] &= ~CYG_FL_DET_PENDING;
    __syncwarp();
  }
}
extern "C" int cyg_fit_launch(int n_sms, cudaStream_t st, const FitParams& p) {
  const size_t smem = sizeof(iforest::Scratch) * CYG_FIT_WARPS;
  cudaError_t e = cudaFuncSetAttribute(cyg_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  cyg_fit_assign_kernel<<<1, 1024, 0, st>>>(p);
  cyg_fit_kernel<<<3 * n_sms, 32 * CYG_FIT_WARPS, smem, st>>>(p); /* 3 CTAs of 4 Scratch each fit one SM's shared memory */
  return (int)cudaGetLastError();
}
#endif

struct ObsParams {
  Net net;
  const uint32_t* recs;
  float* obs;
  int B, obs_mode;
};
template <int W>
__global__ void cyg_observe_kernel(const __grid_constant__ ObsParams p) {
  const int nwarps = (int)((gridDim.x * blockDim.x) >> 5), warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  observe_rows<W>(p.net, p.recs, p.net.S, p.B, p.obs_mode, p.obs, warp, nwarps, (int)(threadIdx.x & 31));
}

/* ===========================================================================
 * Per-W launch table.  The library is built from several translation units of THIS file: one per plane width W
 * (-DCYG_TU_W=1|2|3|4|64: the kernels of that width and their launchers, compiled without --split-compile so that the
 * register allocation of the hot kernels does not depend on what else is in the module) and one with the C-ABI
 * (no CYG_TU_W: no kernel is instantiated there).
 * ======================================================================== */
struct WOps {
  cudaError_t (*set_smem_optin)(int max_optin);
  void (*step)(bool plain, int blocks, int threads, size_t smem, cudaStream_t st, const StepParams& p);
  void (*rollout)(int blocks, int threads, size_t smem, cudaStream_t st, const StepParams& p);
  void (*import_state)(int blocks, int threads, cudaStream_t st, const ConvParams& p);
  void (*export_state)(int blocks, int threads, cudaStream_t st, const ConvParams& p);
  void (*randomize)(int blocks, int threads, cudaStream_t st, const SimpleParams& p);
  void (*rebuild)(int blocks, int threads, cudaStream_t st, const SimpleParams& p);
  void (*sample)(int blocks, int threads, cudaStream_t st, const SimpleParams& p);
  void (*observe)(int blocks, int threads, cudaStream_t st, const ObsParams& p);
};
#define CYG_WOPS_NAME2(w) cyg_wops_##w
#define CYG_WOPS_NAME(w) CYG_WOPS_NAME2(w)

#ifdef CYG_TU_W
#if CYG_TU_W == 4
extern "C" void cyg_group_launch(int blocks, int threads, cudaStream_t st, const GroupParams& p) { cyg_group_kernel<<<blocks, threads, 0, st>>>(p); }
#endif
template <int KW>
struct WImpl {
  static cudaError_t set_smem_optin(int max_optin) {
    if constexpr (KW <= CYG_MAX_W) {
      cudaError_t e = cudaFuncSetAttribute(cyg_step_kernel<KW, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin);
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute(cyg_step_kernel<KW, true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin);
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute(cyg_step_kernel<KW, true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin);
      if (e != cudaSuccess) return e;
      return cudaFuncSetAttribute(cyg_step_kernel<KW, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin);
    } else {
      return cudaFuncSetAttribute(cyg_step_generic_kernel<KW>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin);
    }
  }
  static void step(bool plain, int blocks, int threads, size_t smem, cudaStream_t st, const StepParams& p) {
    if constexpr (KW <= CYG_MAX_W) {
      if (plain && !p.logs) cyg_step_kernel<KW, true, false, false><<<blocks, threads, smem, st>>>(p);
      else if (plain) cyg_step_kernel<KW, true><<<blocks, threads, smem, st>>>(p);
      else cyg_step_kernel<KW, false><<<blocks, threads, smem, st>>>(p);
    } else {
      cyg_step_generic_kernel<KW><<<blocks, threads, smem, st>>>(p);
    }
  }
  static void rollout(int blocks, int threads, size_t smem, cudaStream_t st, const StepParams& p) {
    if constexpr (KW <= CYG_MAX_W) cyg_step_kernel<KW, true, true, false><<<blocks, threads, smem, st>>>(p);
  }
  static void import_state(int blocks, int threads, cudaStream_t st, const ConvParams& p) { cyg_import_kernel<KW><<<blocks, threads, 0, st>>>(p); }
  static void export_state(int blocks, int threads, cudaStream_t st, const ConvParams& p) { cyg_export_kernel<KW><<<blocks, threads, 0, st>>>(p); }
  static void randomize(int blocks, int threads, cudaStream_t st, const SimpleParams& p) { cyg_randomize_kernel<KW><<<blocks, threads, 0, st>>>(p); }
  static void rebuild(int blocks, int threads, cudaStream_t st, const SimpleParams& p) { cyg_rebuild_kernel<KW><<<blocks, threads, 0, st>>>(p); }
  static void sample(int blocks, int threads, cudaStream_t st, const SimpleParams& p) { cyg_sample_kernel<KW><<<blocks, threads, 0, st>>>(p); }
  static void observe(int blocks, int threads, cudaStream_t st, const ObsParams& p) { cyg_observe_kernel<KW><<<blocks, threads, 0, st>>>(p); }
};
extern "C" const WOps* CYG_WOPS_NAME(CYG_TU_W)(void) {
  typedef WImpl<CYG_TU_W> I;
  static const WOps ops = {I::set_smem_optin, I::step, I::rollout, I::import_state, I::export_state, I::randomize, I::rebuild, I::sample, I::observe};
  return &ops;
}
#else /* ---- the C-ABI translation unit ---- */
extern "C" {
void cyg_group_launch(int blocks, int threads, cudaStream_t st, const GroupParams& p);
void cyg_unpack_launch(int blocks, int threads, cudaStream_t st, const UnpackParams& p);
void cyg_pack_done_launch(int blocks, int threads, cudaStream_t st, const int32_t* done, uint32_t* bits, int B);
int cyg_fit_launch(int n_sms, cudaStream_t st, const FitParams& p);
const WOps* cyg_wops_4(void);
#ifndef CYG_FAST_BUILD /* profiling builds link the W = 4 unit only (config C3) */
const WOps* cyg_wops_1(void);
const WOps* cyg_wops_2(void);
const WOps* cyg_wops_3(void);
const WOps* cyg_wops_64(void);
#endif
}
static const WOps* wops(int W) {
  switch (W) {
    case 4: return cyg_wops_4();
#ifndef CYG_FAST_BUILD
    case 1: return cyg_wops_1();
    case 2: return cyg_wops_2();
    case 3: return cyg_wops_3();
    default: return cyg_wops_64();
#else
    default: return nullptr;
#endif
  }
}

/* ===========================================================================
 * C-ABI (include/cygym_b200.h)
 * ======================================================================== */
struct cyg_env_s {
  TableBlob blob;
  Net net;           /* device pointers */
  uint32_t* d_blob;
  uint32_t* state;   /* bound internal buffer: [B][S] records then [B][M] checkpoint words */
  int B, env_id0, device, W, NB, n_sms;
  unsigned long long* dbg_cycles;
  const uint32_t* det_slots; /* uploaded detectors (device memory of the caller) */
  const int32_t* det_of_env;
  int n_det_slots;
  int32_t* fit_work; /* [2 + B] device words of cyg_fit_detectors (allocated with the detector slots) */
  const uint8_t* bl_env;
  int bl_rows;       /* rows of [B] codes behind bl_env (cyg_set_base_line_per_env_steps; 1 otherwise) */
  int id_run, id_stride; /* cyg_set_env_id_stride (0: env id = env_id0 + slot) */
  size_t smem_bytes;
  int64_t launches;
};

static thread_local std::string g_last_error;
static int fail(int code, const std::string& msg) { g_last_error = msg; return code; }
static int cuda_fail(cudaError_t e, const char* what) {
  return fail(CYG_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                                         \
  do {                                                   \
    cudaError_t _e = (call);                             \
    if (_e != cudaSuccess) return cuda_fail(_e, #call);  \
  } while (0)

struct DeviceGuard {
  int prev;
  bool ok;
  explicit DeviceGuard(int dev) : prev(-1), ok(false) {
    if (cudaGetDevice(&prev) != cudaSuccess) return;
    ok = (prev == dev) || (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static int pick_block_envs(const cyg_env_s* h, int requested) {
  /* envs (= threads) per CTA.  One CTA per SM: the bigger the block, the purer the per-warp action types after
   * the in-CTA sort.  Spread B over the SMs in one wave, bounded by shared memory and 512 threads. */
  if (requested > 0) return requested;
  const size_t budget = 226 * 1024;
  int per_sm = (h->B + h->n_sms - 1) / h->n_sms;
  int nb = ((per_sm + 3) / 4) * 4; /* a multiple of 4 records keeps every CTA's span 16-byte sized (bulk copies) whatever S is;
                                      65 536 envs on 148 SMs: 444 per CTA = 148 CTAs (448 = 147 CTAs and an idle SM: 1 % slower) */
  if (nb > CYG_MAX_BLOCK_ENVS) nb = CYG_MAX_BLOCK_ENVS;
  if (nb < 32) nb = 32;
  while (nb > 32 && smem_plan(h->net.hot_words, h->net.S, nb).total > budget) nb -= 4;
  return nb;
}

static int configure_step(cyg_env_s* h) {
  if (!wops(h->W)) return fail(CYG_E_INVAL, "this build has no kernels for the network's plane width");
  if (h->W > CYG_MAX_W) { /* large networks: a few envs per CTA so that every SM gets some, records staged in shared memory */
    int per_sm = (h->B + h->n_sms - 1) / h->n_sms;
    const size_t rec_bytes = (size_t)h->net.S * 4;
    const size_t tab_bytes = (size_t)h->net.hot_words * 4;
    if (tab_bytes + rec_bytes + 64 > 220 * 1024) return fail(CYG_E_INVAL, "network tables do not fit in shared memory");
    int cap = (int)((220 * 1024 - tab_bytes - 64) / (rec_bytes + 16));
    if (cap < 1) return fail(CYG_E_INVAL, "a record does not fit in shared memory");
    h->NB = per_sm < 1 ? 1 : (per_sm > cap ? cap : per_sm);
    if (h->NB > 128) h->NB = 128;
    h->smem_bytes = (size_t)h->NB * rec_bytes + 16 + (size_t)h->NB * 16 + tab_bytes; /* records, pad, 4 words of phase hand-over per env, hot tables */
    int max_optin = 0;
    CU(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    CU(wops(h->W)->set_smem_optin(max_optin));
    return CYG_OK;
  }
  SmemPlan sp = smem_plan(h->net.hot_words, h->net.S, h->NB);
  h->smem_bytes = sp.total;
  /* opt in to the device maximum once (handles with different block sizes share the kernel) */
  int max_optin = 0;
  CU(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
  if ((int)sp.total > max_optin) return fail(CYG_E_INVAL, "record block does not fit in shared memory");
  CU(wops(h->W)->set_smem_optin(max_optin));
  return CYG_OK;
}

extern "C" {

int cyg_version(void) { return CYG_ABI_VERSION; }
const char* cyg_last_error(void) { return g_last_error.c_str(); }

int cyg_create(cyg_handle* out, const cyg_config* cfg, const cyg_network* host_net, int32_t B, int32_t env_id0, int32_t device) {
  if (!out || !cfg || !host_net || !host_net->row_ptr || !host_net->col || !host_net->dev_static)
    return fail(CYG_E_INVAL, "null argument");
  if (B < 1) return fail(CYG_E_INVAL, "B must be >= 1");
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(CYG_E_INVAL, "bad CUDA device ordinal");
  cyg_env_s* h = new (std::nothrow) cyg_env_s();
  if (!h) return fail(CYG_E_NOMEM, "out of host memory");
  std::string err = build_tables(*cfg, *host_net, h->blob);
  if (!err.empty()) { delete h; return fail(CYG_E_INVAL, err); }
  h->B = B; h->env_id0 = env_id0; h->device = device; h->state = nullptr; h->launches = 0; h->dbg_cycles = nullptr; h->bl_env = nullptr; h->bl_rows = 1; h->id_run = 0; h->id_stride = 0;
  h->det_slots = nullptr; h->det_of_env = nullptr; h->n_det_slots = 0; h->fit_work = nullptr;
  h->W = h->blob.net.W;
  DeviceGuard g(device);
  if (!g.ok) { delete h; return fail(CYG_E_CUDA, "cudaSetDevice failed"); }
  size_t bytes = h->blob.words.size() * 4;
  cudaError_t e = cudaMalloc((void**)&h->d_blob, bytes);
  if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaMalloc(tables)"); }
  e = cudaMemcpy(h->d_blob, h->blob.words.data(), bytes, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(h->d_blob); delete h; return cuda_fail(e, "cudaMemcpy(tables)"); }
  relocate(h->blob, h->d_blob, h->net);
  cudaDeviceGetAttribute(&h->n_sms, cudaDevAttrMultiProcessorCount, device);
  if (h->n_sms < 1) h->n_sms = 148;
  const char* nb_env = getenv("CYG_BLOCK_ENVS");
  h->NB = pick_block_envs(h, nb_env ? atoi(nb_env) : 0);
  if (h->NB < 1 || h->NB > CYG_MAX_BLOCK_ENVS) { cudaFree(h->d_blob); delete h; return fail(CYG_E_INVAL, "CYG_BLOCK_ENVS must be in 1..512"); }
  int rc = CYG_OK;
  rc = configure_step(h);
  if (rc != CYG_OK) { cudaFree(h->d_blob); delete h; return rc; }
  *out = h;
  return CYG_OK;
}

int cyg_destroy(cyg_handle h) {
  if (!h) return CYG_OK;
  DeviceGuard g(h->device);
  cudaFree(h->d_blob);
  if (h->fit_work) cudaFree(h->fit_work);
  delete h;
  return CYG_OK;
}

int cyg_set_base_line(cyg_handle h, int32_t base_line) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  h->net.cfg.base_line = base_line;
  return CYG_OK;
}

int cyg_block_envs(cyg_handle h, int32_t* block_envs) {
  if (!h || !block_envs) return fail(CYG_E_INVAL, "null argument");
  *block_envs = h->NB;
  return CYG_OK;
}

int cyg_set_env_id_stride(cyg_handle h, int32_t run, int32_t stride) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  if (run <= 0) { h->id_run = 0; h->id_stride = 0; return CYG_OK; }
  if (stride < run || h->B % run != 0) return fail(CYG_E_INVAL, "cyg_set_env_id_stride: run must divide B and stride >= run");
  if ((int64_t)(h->B / run - 1) * stride + run - 1 + h->env_id0 > 0x7FFFFFFFll) return fail(CYG_E_INVAL, "cyg_set_env_id_stride: env ids beyond 2^31");
  h->id_run = run; h->id_stride = stride;
  return CYG_OK;
}

int cyg_set_base_line_per_env(cyg_handle h, const uint8_t* base_line) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  h->bl_env = base_line;
  h->bl_rows = 1;
  return CYG_OK;
}

int cyg_set_base_line_per_env_steps(cyg_handle h, const uint8_t* base_line, int32_t n_rows) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  if (base_line && n_rows < 1) return fail(CYG_E_INVAL, "n_rows must be >= 1");
  h->bl_env = base_line;
  h->bl_rows = base_line ? n_rows : 1;
  return CYG_OK;
}

static uint32_t* logs_of(cyg_handle h);
int cyg_set_detectors(cyg_handle h, const uint32_t* slots, int32_t n_slots, const int32_t* det_of_env) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  if ((slots == nullptr) != (det_of_env == nullptr) || (slots && n_slots < 1)) return fail(CYG_E_INVAL, "slots and det_of_env go together");
  if (slots && !h->fit_work) {
    DeviceGuard g(h->device);
    CU(cudaMalloc((void**)&h->fit_work, sizeof(int32_t) * (2 + (size_t)h->B)));
  }
  h->det_slots = slots;
  h->det_of_env = det_of_env;
  h->n_det_slots = slots ? n_slots : 0;
  return CYG_OK;
}

/* Detector.train of every pending env on the device (CDSimulator.py:687-695; cyg_iforest.cuh restates scikit-learn's
 * ensemble/_iforest.py, ensemble/_bagging.py, utils/_random.pyx, tree/_splitter.pyx, _partitioner.pyx, _criterion.pyx,
 * _tree.pyx and numpy's legacy MT19937). */
int cyg_fit_detectors(cyg_handle h, const uint32_t* seeds, int32_t* next_slot, void* stream) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  if (!h->det_slots) return fail(CYG_E_INVAL, "cyg_fit_detectors: the handle has no detector slots (cyg_set_detectors)");
  if (!seeds || !next_slot) return fail(CYG_E_INVAL, "null argument");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  DeviceGuard g(h->device);
  FitParams p = {h->state, logs_of(h), const_cast<uint32_t*>(h->det_slots), const_cast<int32_t*>(h->det_of_env), seeds, next_slot,
                 h->fit_work, (int)h->net.S, h->B, h->net.cfg.log_cap, h->n_det_slots};
  const int e = cyg_fit_launch(h->n_sms, (cudaStream_t)stream, p);
  h->launches += 2;
  if (e != 0) return cuda_fail((cudaError_t)e, "cyg_fit_detectors");
  return CYG_OK;
}

int cyg_internal_words(cyg_handle h, int64_t* words_per_env) {
  if (!h || !words_per_env) return fail(CYG_E_INVAL, "null argument");
  *words_per_env = (int64_t)h->net.S + h->net.M + h->net.cfg.xcap + h->net.cfg.log_cap;
  return CYG_OK;
}

int cyg_bind(cyg_handle h, uint32_t* internal_state) {
  if (!h || !internal_state) return fail(CYG_E_INVAL, "null argument");
  if (((uintptr_t)internal_state) & 15) return fail(CYG_E_INVAL, "internal state must be 16-byte aligned");
  h->state = internal_state;
  return CYG_OK;
}

static uint32_t* ckpt_of(cyg_handle h) { return h->state + (size_t)h->B * h->net.S; }
static uint32_t* xtra_of(cyg_handle h) { return ckpt_of(h) + (size_t)h->B * h->net.M; }
static uint32_t* logs_of(cyg_handle h) { return h->net.cfg.log_cap > 0 ? xtra_of(h) + (size_t)h->B * h->net.cfg.xcap : nullptr; }

int cyg_import_state(cyg_handle h, const cyg_state* c, void* stream) {
  if (!h || !c || !c->dev || !c->blocked || !c->extra || !c->scal) return fail(CYG_E_INVAL, "null argument");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  DeviceGuard g(h->device);
  ConvParams p = {h->net, h->state, ckpt_of(h), xtra_of(h), c->dev, c->ckpt, c->blocked, c->extra, c->scal, h->B, logs_of(h), c->logs};
  int threads = 128, blocks = (int)(((size_t)h->B * 32 + threads - 1) / threads);
  wops(h->W)->import_state(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_export_state(cyg_handle h, const cyg_state* c, void* stream) {
  if (!h || !c || !c->dev || !c->blocked || !c->extra || !c->scal) return fail(CYG_E_INVAL, "null argument");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  DeviceGuard g(h->device);
  ConvParams p = {h->net, h->state, ckpt_of(h), xtra_of(h), c->dev, c->ckpt, c->blocked, c->extra, c->scal, h->B, logs_of(h), c->logs};
  int threads = 128, blocks = (int)(((size_t)h->B * 32 + threads - 1) / threads);
  wops(h->W)->export_state(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

static int step_impl(cyg_handle h, const cyg_actions* a, int n_steps, uint32_t step_flags, const cyg_step_out* out, void* stream);

int cyg_step(cyg_handle h, const cyg_actions* a, uint32_t step_flags, const cyg_step_out* out, void* stream) {
  return step_impl(h, a, 1, step_flags, out, stream);
}

int cyg_step_multi(cyg_handle h, const cyg_actions* a, int32_t n_steps, uint32_t step_flags, const cyg_step_out* out, void* stream) {
  if (n_steps < 1) return fail(CYG_E_INVAL, "n_steps must be >= 1");
  if (n_steps > 1) {
    if (!h || !a || !out) return fail(CYG_E_INVAL, "null argument");
    if (h->bl_env && h->bl_rows > 1 && h->bl_rows < n_steps) return fail(CYG_E_INVAL, "cyg_step_multi: fewer base_line rows than steps");
    if ((step_flags & CYG_STEP_GROUPED) || a->order || a->n_groups != 1) return fail(CYG_E_INVAL, "cyg_step_multi: plain steps only (no groups, no order array)");
    if (out->obs || out->pre_masks) return fail(CYG_E_INVAL, "cyg_step_multi: no obs / pre_masks outputs");
    if (h->W > CYG_MAX_W) return fail(CYG_E_INVAL, "cyg_step_multi: networks of at most 128 device slots");
  }
  return step_impl(h, a, n_steps, step_flags, out, stream);
}

static int step_impl(cyg_handle h, const cyg_actions* a, int n_steps, uint32_t step_flags, const cyg_step_out* out, void* stream) {
  if (!h || !a || !out || !a->hdr || !a->mask || !out->raw_reward || !out->shaped_reward || !out->done)
    return fail(CYG_E_INVAL, "null argument");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  if (h->id_run > 0) return fail(CYG_E_INVAL, "strided env ids (cyg_set_env_id_stride): cyg_rollout only");
  const bool grouped = (step_flags & CYG_STEP_GROUPED) != 0;
  if (a->n_groups < 1 || (!grouped && a->n_groups != 1)) return fail(CYG_E_INVAL, "n_groups must be 1 unless CYG_STEP_GROUPED");
  if (a->order && a->order_stride < 1) return fail(CYG_E_INVAL, "order_stride must be >= 1 with an order array");
  if (out->obs && (out->obs_mode < 1 || out->obs_mode > 3)) return fail(CYG_E_INVAL, "obs_mode must be 1..3 when obs is given");
  if (((uintptr_t)a->hdr) & 15) return fail(CYG_E_INVAL, "hdr must be 16-byte aligned");
  DeviceGuard g(h->device);
  StepParams p;
  p.net = h->net;
  p.recs = h->state; p.ckpt = ckpt_of(h); p.xtra = xtra_of(h);
  p.hdr = a->hdr; p.mask = a->mask; p.order = a->order;
  p.raw = out->raw_reward; p.shaped = out->shaped_reward; p.done = out->done;
  p.pre_masks = out->pre_masks; p.obs = out->obs; p.dbg_cycles = h->dbg_cycles; p.bl_env = h->bl_env; p.bl_stride = (h->bl_env && h->bl_rows > 1) ? h->B : 0;
  p.B = h->B; p.env_id0 = h->env_id0; p.G = a->n_groups; p.order_stride = a->order_stride;
  p.obs_mode = out->obs ? out->obs_mode : 0;
  p.flags = step_flags;
  p.T = n_steps;
  p.row_base = 0; p.envs_per_row = 0; p.n_rows = h->B; p.ret_acc = nullptr; p.id_run = 0; p.id_stride = 0; p.block_order = nullptr;
  p.logs = logs_of(h); p.det_slots = h->det_slots; p.det_of_env = h->det_of_env;
  p.block_envs = h->NB;
  const bool plain = !(step_flags & CYG_STEP_GROUPED) && a->order == nullptr; /* the hot form: see cyg_step_kernel */
  int blocks = (h->B + h->NB - 1) / h->NB;
  int threads = ((2 * h->NB + 31) / 32) * 32;
  if (threads > CYG_MAX_BLOCK_THREADS) threads = CYG_MAX_BLOCK_THREADS;
  if (threads < h->NB) threads = ((h->NB + 31) / 32) * 32;
  if (h->W > CYG_MAX_W) {
    wops(h->W)->step(false, (h->B + h->NB - 1) / h->NB, 256, h->smem_bytes, (cudaStream_t)stream, p);
    if (out->obs) { /* post-evolve observation rows: a second launch on the generic path */
      h->launches++;
      CU(cudaGetLastError());
      return cyg_observe(h, out->obs_mode, out->obs, stream);
    }
  } else {
    wops(h->W)->step(plain, blocks, threads, h->smem_bytes, (cudaStream_t)stream, p);
  }
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_rollout(cyg_handle h, const cyg_rollout_args* a, uint32_t step_flags, void* stream) {
  if (!h || !a || !a->hdr || !a->mask || !a->returns) return fail(CYG_E_INVAL, "null argument");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  if (h->W > CYG_MAX_W) return fail(CYG_E_INVAL, "cyg_rollout: networks of at most 128 device slots");
  if (h->net.cfg.log_cap > 0) return fail(CYG_E_INVAL, "cyg_rollout: handles with a hop-log ring (log_cap > 0) step through cyg_step");
  if (a->n_steps < 1 || a->n_rows < 1 || a->envs_per_row < 1 || a->row_base < 0 || a->row_base + h->B > 0x7FFFFFFFll) return fail(CYG_E_INVAL, "cyg_rollout: bad sizes");
  const int64_t last_idx = h->id_run > 0 ? (int64_t)strided_index((uint32_t)(h->B - 1), (uint32_t)h->id_run, (uint32_t)h->id_stride) : (int64_t)h->B - 1;
  if (a->row_base + last_idx > 0x7FFFFFFFll || (a->row_base + last_idx) / a->envs_per_row >= a->n_rows) return fail(CYG_E_INVAL, "cyg_rollout: an env's action row is beyond n_rows");
  if (step_flags & CYG_STEP_GROUPED) return fail(CYG_E_INVAL, "cyg_rollout: plain steps only");
  if (((uintptr_t)a->hdr) & 15) return fail(CYG_E_INVAL, "hdr must be 16-byte aligned");
  DeviceGuard g(h->device);
  StepParams p;
  p.net = h->net;
  p.recs = h->state; p.ckpt = ckpt_of(h); p.xtra = xtra_of(h);
  p.hdr = a->hdr; p.mask = a->mask; p.order = nullptr;
  p.raw = nullptr; p.shaped = nullptr; p.done = nullptr; p.pre_masks = nullptr; p.obs = nullptr; p.dbg_cycles = nullptr;
  p.bl_env = a->base_line; p.bl_stride = a->base_line ? a->n_rows : 0;
  p.B = h->B; p.env_id0 = h->env_id0; p.G = 1; p.order_stride = 0; p.obs_mode = 0; p.flags = step_flags; p.T = a->n_steps;
  p.row_base = a->row_base; p.envs_per_row = a->envs_per_row; p.n_rows = a->n_rows; p.ret_acc = a->returns;
  p.id_run = h->id_run; p.id_stride = h->id_stride; p.block_order = a->block_order;
  p.logs = logs_of(h); p.det_slots = h->det_slots; p.det_of_env = h->det_of_env;
  p.block_envs = h->NB;
  int blocks = (h->B + h->NB - 1) / h->NB;
  int threads = ((2 * h->NB + 31) / 32) * 32;
  if (threads > CYG_MAX_BLOCK_THREADS) threads = CYG_MAX_BLOCK_THREADS;
  if (threads < h->NB) threads = ((h->NB + 31) / 32) * 32;
  wops(h->W)->rollout(blocks, threads, h->smem_bytes, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_randomize(cyg_handle h, const uint8_t* env_mask, void* stream) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  DeviceGuard g(h->device);
  SimpleParams p = {h->net, h->state, xtra_of(h), env_mask, nullptr, nullptr, h->B, h->env_id0, 0, nullptr, 0, h->id_run, h->id_stride};
  int threads = 128, blocks = (h->B + threads - 1) / threads;
  wops(h->W)->randomize(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_rebuild_graph_cache(cyg_handle h, const uint8_t* env_mask, void* stream) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  DeviceGuard g(h->device);
  SimpleParams p = {h->net, h->state, xtra_of(h), env_mask, nullptr, nullptr, h->B, h->env_id0, 0, nullptr, 0, h->id_run, h->id_stride};
  int threads = 128, blocks = (h->B + threads - 1) / threads;
  wops(h->W)->rebuild(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_sample_actions(cyg_handle h, int32_t mode, uint32_t* hdr, uint32_t* mask, void* stream) {
  return cyg_sample_actions_ordered(h, mode, hdr, mask, nullptr, 0, stream);
}

int cyg_sample_actions_ordered(cyg_handle h, int32_t mode, uint32_t* hdr, uint32_t* mask, uint16_t* order, int32_t order_stride,
                               void* stream) {
  if (!h || !hdr || !mask) return fail(CYG_E_INVAL, "null argument");
  if (order && order_stride < h->net.cfg.num_of_device) return fail(CYG_E_INVAL, "order_stride must hold numOfDevice entries");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  if (mode != CYG_MODE_DEFENDER && mode != CYG_MODE_ATTACKER) return fail(CYG_E_INVAL, "mode must be 0 or 1");
  DeviceGuard g(h->device);
  SimpleParams p = {h->net, h->state, xtra_of(h), nullptr, hdr, mask, h->B, h->env_id0, mode, order, order_stride, h->id_run, h->id_stride};
  int threads = 128, blocks = (h->B + threads - 1) / threads;
  wops(h->W)->sample(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_observe(cyg_handle h, int32_t obs_mode, float* obs, void* stream) {
  if (!h || !obs) return fail(CYG_E_INVAL, "null argument");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  if (obs_mode < 1 || obs_mode > 3) return fail(CYG_E_INVAL, "obs_mode must be 1..3");
  DeviceGuard g(h->device);
  ObsParams p = {h->net, h->state, obs, h->B, obs_mode};
  int threads = 256;
  size_t total = (size_t)h->B * (obs_mode == 2 ? 4 * h->net.M + h->net.cfg.X : 6 * h->net.M);
  int blocks = (int)((total + threads - 1) / threads);
  if (blocks > 148 * 16) blocks = 148 * 16;
  wops(h->W)->observe(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_unpack_actions(cyg_handle h, const uint32_t* rows, uint32_t* hdr, uint32_t* mask, void* stream) {
  if (!h || !rows || !hdr || !mask) return fail(CYG_E_INVAL, "null argument");
  if (((uintptr_t)hdr) & 15) return fail(CYG_E_INVAL, "hdr must be 16-byte aligned");
  if (h->net.M > 254) return fail(CYG_E_INVAL, "compact action rows: networks of at most 254 device slots");
  DeviceGuard g(h->device);
  UnpackParams p = {rows, hdr, mask, h->B, h->net.Wm};
  const int threads = 256, blocks = (h->B + threads - 1) / threads;
  cyg_unpack_launch(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_pack_done(cyg_handle h, const int32_t* done, uint32_t* bits, void* stream) {
  if (!h || !done || !bits) return fail(CYG_E_INVAL, "null argument");
  DeviceGuard g(h->device);
  const int threads = 256, blocks = (h->B + threads - 1) / threads;
  cyg_pack_done_launch(blocks, threads, (cudaStream_t)stream, done, bits, h->B);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int cyg_group_actions(cyg_handle h, int32_t mode, int32_t role, const int32_t* per_dev_types, const uint8_t* visible, const int32_t* exp_idx,
                      const int32_t* app_idx, const int32_t* single_choice, int32_t n_types, int32_t noop, uint32_t* hdr, uint32_t* mask, void* stream) {
  if (!h || !per_dev_types || !hdr || !mask) return fail(CYG_E_INVAL, "null argument");
  if (!h->state) return fail(CYG_E_INVAL, "cyg_bind() first");
  if (n_types < 2 || n_types > 33 || noop < 0 || noop >= n_types) return fail(CYG_E_INVAL, "n_types must be 2..33 and noop one of them");
  if (role < 0 || role > 2 || (mode != CYG_MODE_DEFENDER && mode != CYG_MODE_ATTACKER)) return fail(CYG_E_INVAL, "bad role / mode");
  if (((uintptr_t)hdr) & 15) return fail(CYG_E_INVAL, "hdr must be 16-byte aligned");
  DeviceGuard g(h->device);
  GroupParams p = {h->net, h->state, per_dev_types, exp_idx, app_idx, visible, single_choice, hdr, mask, h->B, mode, role, n_types, noop};
  const int threads = 128, blocks = (int)(((size_t)h->B * 32 + threads - 1) / threads);
  cyg_group_launch(blocks, threads, (cudaStream_t)stream, p);
  h->launches++;
  CU(cudaGetLastError());
  return CYG_OK;
}

int64_t cyg_launch_count(cyg_handle h) { return h ? h->launches : 0; }

int cyg_set_debug_cycles(cyg_handle h, uint64_t* per_env_cycles) {
  if (!h) return fail(CYG_E_INVAL, "null handle");
  h->dbg_cycles = (unsigned long long*)per_env_cycles;
  return CYG_OK;
}

} /* extern "C" */
#endif /* CYG_TU_W */
