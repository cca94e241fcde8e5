/*
 * cyg_core.cuh -- per-env transition of the CyGym step path on the INTERNAL bit-plane record.
 *
 * One thread owns one env.  The env's whole dynamic state is a record of S uint32 words
 * that the step kernel stages in shared memory (TMA bulk copy in, bulk copy out):
 *
 *   [0, 16)                          the 16 scalars of include/cygym_b200.h (CYG_S_*)
 *   [16 + p*W, 16 + (p+1)*W)         bit-plane p, W = ceil(M/32) words, bit d = device d
 *   [off_inc, off_inc + UW)          blocked-edge bitset in INCIDENCE-UNIT order: device d owns the contiguous bit
 *                                    range [ip[d], ip[d+1]) -- one bit per out-edge (ascending neighbour id, a pair of
 *                                    multiplicity m as m adjacent bits: the order of _outnbrs, volt:456-473), then one
 *                                    per in-edge (ascending source id).  A blocked pair has all its 2m bits set, so the
 *                                    pool of block / unblock (volt:485-511) is ONE window, its weight a popcount and
 *                                    the hop count of the lateral-movement scan (volt:1148-1185) a popcount as well
 *   [off_aux]                        number of blocked base pairs (derived; spares the scans a walk over the bitset)
 * (the rarely used per-env extra attacker hub-star edges and the per-device checkpoint words
 * live in side arrays in global memory and are touched only by the actions that need them)
 *
 * Bit-planes turn every O(M) loop of the reference (busy tick volt_typhoon_env.py:904-908,
 * workload advance :1242-1261, _count_comp :563-572, candidate lists of
 * CDSimulator.py:244-348, evolve_network's active/inactive sets CyberDefenseEnv.py:654-659)
 * into W word-wide boolean operations, and the lateral-movement scan (:1148-1185) into
 * "first set bit of adj[src] & candidates".  Multi-bit fields (busy_time, processing_time,
 * compromised_by) are bit-sliced across planes.
 *
 * Every function is written once, as plain integer C++ with no warp intrinsics, so the very
 * same source also compiles for the host: tests/emu builds it with g++ and replays the golden
 * trajectories through it on the CPU-only build container (logic check of the device source;
 * it is not shipped and the product library has no CPU path).
 *
 * Statement order and quirks follow the reference; the line numbers cited are the reference's.
 */
#ifndef CYG_CORE_CUH
#define CYG_CORE_CUH

#include <math.h>
#include <stdint.h>

#include "../../include/cygym_b200.h"

#if defined(__CUDACC__)
#define CYG_HD __host__ __device__ __forceinline__
#define CYG_HDN __host__ __device__ __noinline__
#else
#define CYG_HD inline
#define CYG_HDN inline
#endif

namespace cyg {

/* draw sites: oracle/draws.py (each is one RNG call site of the reference) */
enum {
  SITE_STALL = 1, SITE_BLOCK = 2, SITE_UNBLOCK = 3, SITE_ZDAY = 4, SITE_PROBE = 5, SITE_WL_SAMPLE = 6,
  SITE_WL_TRI = 7, SITE_WL_LAZY = 8, SITE_EV_POISSON = 9, SITE_EV_ADD = 10, SITE_EV_PICK = 11,
  SITE_EV_ATT = 12, SITE_SHUFFLE = 13, SITE_DETECT = 14, SITE_SA_TYPE = 15, SITE_SA_NDEV = 16,
  SITE_SA_DEVS = 17, SITE_SA_EXP = 18, SITE_SA_APP = 19
};

/* bit-plane ids */
enum {
  P_COMP = 0, P_KNOWN = 1, P_NYA = 2, P_OWNED = 3, P_HASWL = 4, P_BUSYSET = 5, P_ACTSET = 6,
  P_PT0 = 7, P_BUSY0 = 10, P_CBY0 = 14
};
#define CYG_REC_PLANES 16 /* word offset of plane 0 inside a record */
#define CYG_CKI_REMOVED 0x40000000u /* internal checkpoint word, spare bit: Device.removed_before (never read by step) */
#define CYG_MAX_W 4       /* M <= 128: the shared-memory bit-matrix step kernel (W = ceil(M/32) words per plane) */
#define CYG_BIG_W 64      /* 128 < M <= 2048: planes padded to 64 words, stepped by the generic global-memory kernel */

/* ---- shared network tables + derived sizes -------------------------------------------------
 * All tables live in ONE blob of uint32 words (cyg_tables.h); the Net holds word OFFSETS into it.  The step
 * kernel receives the Net by value as a __grid_constant__ parameter, so every size and offset below is a
 * constant-bank operand, and reads the hot prefix of the blob [0, hot_words) from its shared-memory copy. */
struct Net {
  cyg_config cfg;
  int M, W, E, EW, NP, S, ncby, off_inc, off_aux;
  int U2, UW;                 /* incidence units (2 x sum of multiplicities) and the words of their bitset */
  int Wm;                     /* ceil(M/32): words per device mask in the C-ABI arrays (== W unless the planes are padded) */
  double inv_M;               /* 1.0 / M */
  uint32_t hot_words;         /* prefix of the blob that a CTA stages in shared memory */
  /* hot tables */
  uint32_t o_adj;             /* [M][W] out-neighbour bit rows (unique pairs; _outnbrs, volt:456-473) */
  uint32_t o_dc, o_server, o_reach, o_valid; /* [W] masks over devices */
  uint32_t o_napps;           /* [8][W] bit-planes of len(device.apps) */
  uint32_t o_vuln;            /* [X][W] device has an app vulnerability in exploits[e].target */
  uint32_t o_dinfo;           /* [M+1] ip[d] | out-units(d) << 16: device d owns units [ip[d], ip[d+1]) */
  uint32_t o_unit;            /* [U2] twin run start | far endpoint << 16 | (m - 1) << 28 | offset in own run << 30 */
  uint32_t o_omulti;          /* [M] multi-edge runs of the out list: pair rank | (m-1) << 8, two 10-bit entries (0xFF = none);
                                 bit 31 = more than two (walk the units) */
  uint32_t o_static;          /* [M] CYG_ST_* */
  /* cold tables (global memory only) */
  uint32_t o_pair2unit;       /* [E] first out-unit of base pair e (canonical blocked[] <-> units) */
  uint32_t o_os, o_ver;       /* [M] float: os_to_float(d.OS), float(d.version) */
  const uint32_t* blob;       /* the blob in global (device) / host memory */
};

/* fields of a unit entry (Net::o_unit) */
CYG_HD int unit_twin(uint32_t u) { return (int)(u & 0xFFFFu); }
CYG_HD int unit_other(uint32_t u) { return (int)((u >> 16) & 0xFFFu); }
CYG_HD int unit_m(uint32_t u) { return (int)((u >> 28) & 3u) + 1; }
CYG_HD int unit_off(uint32_t u) { return (int)(u >> 30); }

CYG_HD int popc(uint32_t x) {
#ifdef __CUDA_ARCH__
  return __popc(x);
#else
  return __builtin_popcount(x);
#endif
}
CYG_HD int ctz(uint32_t x) { /* x != 0 */
#ifdef __CUDA_ARCH__
  return __ffs((int)x) - 1;
#else
  return __builtin_ctz(x);
#endif
}
CYG_HD uint32_t below(uint32_t x, uint32_t n) { /* floor(x*n/2^32): oracle/draws.py:below */
#ifdef __CUDA_ARCH__
  return __umulhi(x, n);
#else
  return (uint32_t)(((uint64_t)x * n) >> 32);
#endif
}
CYG_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, int sh) { /* bits [sh, sh+32) of hi:lo, 0 <= sh < 32 */
#ifdef __CUDA_ARCH__
  return __funnelshift_r(lo, hi, (uint32_t)sh);
#else
  return (uint32_t)((((uint64_t)hi << 32) | lo) >> sh);
#endif
}
/* all-ones when a == b.  Per-word updates are written branch-free (x |= bit & eqmask(w, idx)) on purpose: a
 * conditional store inside an unrolled loop is merged by the compiler into ONE dynamically indexed access, which
 * forces the whole array out of registers into local memory. */
CYG_HD uint32_t eqmask(int a, int b) { return a == b ? 0xFFFFFFFFu : 0u; }
CYG_HD uint32_t lowmask(int nbits) { /* the low nbits bits, 0 <= nbits; all ones from 32 up */
#ifdef __CUDA_ARCH__
  uint32_t m;
  asm("bmsk.clamp.b32 %0, %1, %2;" : "=r"(m) : "r"(0), "r"(nbits)); /* one BMSK */
  return m;
#else
  return nbits >= 32 ? 0xFFFFFFFFu : ((1u << nbits) - 1u);
#endif
}
CYG_HD uint32_t lowmask0(int nbits) { return lowmask(nbits < 0 ? 0 : nbits); } /* ... and none below 0 */
CYG_HD float u2f(uint32_t u) {
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f; __builtin_memcpy(&f, &u, 4); return f;
#endif
}
CYG_HD uint32_t f2u(float f) {
#ifdef __CUDA_ARCH__
  return __float_as_uint(f);
#else
  uint32_t u; __builtin_memcpy(&u, &f, 4); return u;
#endif
}

/* position of the r-th (0-based) set bit of x; r < popc(x) */
CYG_HD int select_in_word(uint32_t x, int r) {
  int pos = 0;
#pragma unroll
  for (int sh = 16; sh >= 1; sh >>= 1) {
    int c = popc((x >> pos) & ((1u << sh) - 1u));
    if (r >= c) { r -= c; pos += sh; }
  }
  return pos;
}

/* ---- Philox4x32-10 and the addressable draw contract (oracle/draws.py) ---- */
CYG_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t o[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
#ifdef __CUDA_ARCH__
    uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
#else
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t h0 = (uint32_t)(p0 >> 32), l0 = (uint32_t)p0, h1 = (uint32_t)(p1 >> 32), l1 = (uint32_t)p1;
#endif
    uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}

struct Rng { uint32_t k0, k1, env, epoch; };

/* sequential reader of one site's draws k = 0, 1, 2, ... inside the current epoch.  `blk` = index of the Philox block
 * held in b0..b3 (0xFFFFFFFF: none yet): next() computes a block only when the draw index leaves the held one, and
 * load() fetches block 0 ahead of time so that several streams' Philox rounds overlap instead of chaining. */
struct Stream {
  uint32_t k, blk, b0, b1, b2, b3;
  int site;
  CYG_HD explicit Stream(int s) : k(0), blk(0xFFFFFFFFu), b0(0), b1(0), b2(0), b3(0), site(s) {}
  CYG_HD void fetch(const Rng& r, uint32_t block) {
    uint32_t o[4];
    philox4x32_10(r.env, r.epoch, (uint32_t)site, block, r.k0, r.k1, o);
    b0 = o[0]; b1 = o[1]; b2 = o[2]; b3 = o[3];
    blk = block;
  }
  CYG_HD void load(const Rng& r) { fetch(r, k >> 2); }
  CYG_HD uint32_t next(const Rng& r) {
    if ((k >> 2) != blk) fetch(r, k >> 2);
    uint32_t j = k & 3u;
    k++;
    return j == 0 ? b0 : j == 1 ? b1 : j == 2 ? b2 : b3;
  }
  /* continue at draw index k + n (n draws are skipped unread) */
  CYG_HD void skip(const Rng& r, uint32_t nskip) { (void)r; k += nskip; }
};

/* ---- per-env view over an internal record ---------------------------------
 * SM = 1    : the record and the hot tables are addressed as offsets into the kernel's dynamic shared memory
 * SM = 2    : the record and the hot PREFIX of the tables in shared memory, the rest of the tables (large networks: the
 *             adjacency bit rows) through pointers
 *             (every access is an LDS with a constant-bank offset);
 * SM = 0    : plain pointers (host build, and the small kernels that work on records in global memory). */
#ifdef __CUDACC__
extern __shared__ __align__(128) uint32_t cyg_smem[];
#endif
/* defender action 5 with a TRAINED detector, as a stand-alone call that builds its own Env: the ~2 KB of local arrays
 * (30 scored records, the CPython set emulation) and the tree walks stay out of the register allocation of the step
 * kernels, and no Env of a hot path has its address taken.  Returns the _stall stream's draw index afterwards. */
template <int W, int SM>
CYG_HDN uint32_t scan_trained_call(const Net* n, uint32_t* rec, uint32_t ro, uint32_t to, uint32_t* logs, const uint32_t* det, uint32_t env_id,
                                   uint32_t stall_k, int reps);

template <int W, int SM = 0>
struct Env {
  const Net* n;
  uint32_t* rec;   /* the record (SM: unused) */
  const uint32_t* th; /* hot tables (SM: unused) */
  const uint32_t* tc; /* cold tables: the blob in global / host memory */
  uint32_t ro, to; /* SM: word offsets of the record / the hot tables inside cyg_smem */
  uint32_t* ckpt;  /* canonical per-device checkpoint words of this env [M] (global memory) */
  uint32_t* xtra;  /* extra (attacker hub-star) edges of this env [xcap] (global memory) */
  uint32_t* logs = nullptr;      /* hop-log ring of this env [cfg.log_cap] (global memory); nullptr: only the length is kept */
  const uint32_t* det = nullptr; /* detector slot of this env (CYG_DET_WORDS, global memory); nullptr: none uploaded */
  Rng rng;
  Stream stall;    /* SITE_STALL is shared by every group of a grouped step */
  int bl;          /* base_line in effect for this env (CYG_BL_*): cfg.base_line unless the caller set one per env */
  double defcost, cleancost;

  CYG_HD Env(const Net* net, uint32_t* record, uint32_t* ck, uint32_t* xt, uint32_t env_id, uint32_t rec_off = 0,
             uint32_t tab_off = 0)
      : n(net), rec(record), th(net->blob), tc(net->blob), ro(rec_off), to(tab_off), ckpt(ck), xtra(xt), stall(SITE_STALL),
        bl(net->cfg.base_line), defcost(0.0), cleancost(0.0) {
    rng.k0 = (uint32_t)net->cfg.seed;
    rng.k1 = (uint32_t)(net->cfg.seed >> 32);
    rng.env = env_id;
    rng.epoch = 0;
  }
  /* record word i / hot-table word i */
  CYG_HD uint32_t& R(int i) {
#ifdef __CUDA_ARCH__
    if (SM) return cyg_smem[ro + i];
#endif
    return rec[i];
  }
  CYG_HD uint32_t T(uint32_t i) const {
#ifdef __CUDA_ARCH__
    if (SM == 1) return cyg_smem[to + i];
    if (SM == 2 && i < n->hot_words) return cyg_smem[to + i];
#endif
    return th[i];
  }
  CYG_HD const uint32_t* Tp(uint32_t i) const {
#ifdef __CUDA_ARCH__
    if (SM == 1) return cyg_smem + to + i;
#endif
    return th + i;
  }
  CYG_HD uint32_t dinfo(int d) const { return T(n->o_dinfo + d); }
  CYG_HD int ip(int d) const { return (int)(dinfo(d) & 0xFFFFu); }      /* first unit of device d */
  CYG_HD int nout(int d) const { return (int)(dinfo(d) >> 16); }        /* its out-units; the in-units follow */
  CYG_HD uint32_t unit(int q) const { return T(n->o_unit + q); }
  CYG_HD uint32_t adj(int u, int w) const { return T(n->o_adj + u * W + w); }
  CYG_HD uint32_t m_dc(int w) const { return T(n->o_dc + w); }
  CYG_HD uint32_t m_server(int w) const { return T(n->o_server + w); }
  CYG_HD uint32_t m_reach(int w) const { return T(n->o_reach + w); }
  CYG_HD uint32_t m_valid(int w) const { return T(n->o_valid + w); }
  CYG_HD uint32_t m_vuln(int e, int w) const { return T(n->o_vuln + e * W + w); }
  CYG_HD bool devbit(uint32_t off, int d) const { return (T(off + (d >> 5)) >> (d & 31)) & 1u; }
  CYG_HD uint32_t dev_static(int d) const { return T(n->o_static + d); }
  CYG_HD uint32_t& scal(int i) { return R(i); }
  CYG_HD uint32_t& pl(int p, int w) { return R(CYG_REC_PLANES + p * W + w); }
  CYG_HD uint32_t* inc() { return &R(n->off_inc); } /* blocked bits in incidence-unit order */
  CYG_HD bool ubit(int q) { return (inc()[q >> 5] >> (q & 31)) & 1u; }
  CYG_HD uint32_t& nblk() { return R(n->off_aux); } /* number of blocked base pairs */
  CYG_HD uint32_t* extra() { return xtra; }
  CYG_HD int n_extra() { return (int)(R(CYG_S_PREV_X) >> 16); }

  /* open a draw epoch (one per step / randomize / sample_action call) */
  CYG_HD void begin_epoch() {
    rng.epoch = scal(CYG_S_EPOCH);
    scal(CYG_S_EPOCH) = rng.epoch + 1u;
    stall = Stream(SITE_STALL);
  }

  /* ---- single-device accessors ---- */
  CYG_HD bool bit(int p, int d) { return (pl(p, d >> 5) >> (d & 31)) & 1u; }
  CYG_HD void setb(int p, int d) { pl(p, d >> 5) |= 1u << (d & 31); }
  CYG_HD void clrb(int p, int d) { pl(p, d >> 5) &= ~(1u << (d & 31)); }
  CYG_HD uint32_t field(int p0, int nb, int d) {
    uint32_t v = 0;
    for (int k = 0; k < nb; k++) v |= ((pl(p0 + k, d >> 5) >> (d & 31)) & 1u) << k;
    return v;
  }
  CYG_HD void set_field(int p0, int nb, int d, uint32_t v) {
    uint32_t m = 1u << (d & 31);
    int w = d >> 5;
    for (int k = 0; k < nb; k++) {
      uint32_t x = pl(p0 + k, w) & ~m;
      if ((v >> k) & 1u) x |= m;
      pl(p0 + k, w) = x;
    }
  }
  CYG_HD uint32_t busy(int d) { return field(P_BUSY0, 4, d); }
  CYG_HD void set_busy(int d, uint32_t b) {
    if (b > CYG_BUSY_MAX) { b = CYG_BUSY_MAX; scal(CYG_S_FLAGS) |= CYG_FL_ERR_BUSY; }
    set_field(P_BUSY0, 4, d, b);
  }
  CYG_HD void drop_wl(int d) { clrb(P_HASWL, d); set_field(P_PT0, 3, d, 0); }
  CYG_HD uint32_t cby(int d) { return field(P_CBY0, n->ncby, d); }
  CYG_HD void clr_cby(int d) { set_field(P_CBY0, n->ncby, d, 0); }
  CYG_HD uint32_t stall_draw(int low, int high) { /* _stall: random.randint(low, high) (volt:135-138) */
    return (uint32_t)low + below(stall.next(rng), (uint32_t)(high - low + 1));
  }

  /* ---- word-wide helpers ---- */
  CYG_HD uint32_t busy_nz(int w) { return pl(P_BUSY0, w) | pl(P_BUSY0 + 1, w) | pl(P_BUSY0 + 2, w) | pl(P_BUSY0 + 3, w); }
  CYG_HD int count(int p) {
    int c = 0;
    for (int w = 0; w < W; w++) c += popc(pl(p, w));
    return c;
  }
  /* busy_time += 1 for every device in mask m[] (saturating at CYG_BUSY_MAX, flagged) */
  CYG_HD void busy_inc(const uint32_t* m) {
    for (int w = 0; w < W; w++) {
      uint32_t c = m[w];
      for (int k = 0; k < 4; k++) {
        uint32_t b = pl(P_BUSY0 + k, w);
        pl(P_BUSY0 + k, w) = b ^ c;
        c &= b;
      }
      if (c) { /* 15 + 1: saturate */
        for (int k = 0; k < 4; k++) pl(P_BUSY0 + k, w) |= c;
        scal(CYG_S_FLAGS) |= CYG_FL_ERR_BUSY;
      }
    }
  }
  /* busy_time -= 1 for every device in mask m[] that has busy_time > 0 */
  CYG_HD void busy_dec(const uint32_t* m) {
    for (int w = 0; w < W; w++) {
      uint32_t c = m[w] & busy_nz(w);
      for (int k = 0; k < 4; k++) {
        uint32_t b = pl(P_BUSY0 + k, w);
        pl(P_BUSY0 + k, w) = b ^ c;
        c &= ~b;
      }
    }
  }
  /* pop the lowest member of mask m[] (-1 when empty).  ONE loop over all W words keeps the lanes of a warp on the
   * same loop body (a loop per word would be unrolled into W copies that the lanes enter at different times). */
  CYG_HD int pop_lowest(uint32_t* m) {
    int w0 = -1;
    uint32_t x = 0;
    for (int w = W - 1; w >= 0; w--) { bool nz = m[w] != 0; w0 = nz ? w : w0; x = nz ? m[w] : x; }
    if (w0 < 0) return -1;
    uint32_t lb = x & (0u - x);
    for (int w = 0; w < W; w++) m[w] ^= lb & eqmask(w, w0);
    return w0 * 32 + ctz(lb);
  }
  /* r-th (0-based, ascending id) member of mask m[]; r < total popcount */
  CYG_HD int select_nth(const uint32_t* m, int r) { /* branch-free over the words: ONE select_in_word */
    int cum = 0, wsel = -1, base = 0;
    uint32_t xw = 0;
    for (int w = 0; w < W; w++) {
      int c = popc(m[w]);
      bool take = r >= cum && r < cum + c;
      xw = take ? m[w] : xw;
      wsel = take ? w : wsel;
      base = take ? cum : base;
      cum += c;
    }
    if (wsel < 0) return -1;
    return wsel * 32 + select_in_word(xw, r - base);
  }

  /* ---- topology: base bit rows + blocked unit bitset + extra edges ---------------- */
  CYG_HD bool any_blocked() {
    if (nblk() != 0) return true;
    uint32_t o = 0;
    int nx = n_extra();
    const uint32_t* x = extra();
    for (int j = 0; j < nx; j++) o |= x[j] & CYG_X_BLOCKED;
    return o != 0;
  }
  /* units of [a, a + len) whose blocked bit XOR flip is set (flipw = 0: blocked ones, ~0: unblocked ones) */
  CYG_HD int range_count(int a, int len, uint32_t flipw) {
    if (len <= 0) return 0;
    const uint32_t* b = inc();
    const int z = a + len, wa = a >> 5, wz = (z - 1) >> 5;
    int c = 0;
    for (int wi = wa; wi <= wz; wi++) {
      uint32_t x = b[wi] ^ flipw;
      if (wi == wa) x &= ~lowmask(a & 31);
      if (wi == wz) x &= lowmask(((z - 1) & 31) + 1);
      c += popc(x);
    }
    return c;
  }
  /* the r-th (0-based) such unit, as an absolute unit index; r < range_count */
  CYG_HD int range_select(int a, int len, uint32_t flipw, int r) {
    const uint32_t* b = inc();
    const int z = a + len, wa = a >> 5, wz = (z - 1) >> 5;
    for (int wi = wa; wi <= wz; wi++) {
      uint32_t x = b[wi] ^ flipw;
      if (wi == wa) x &= ~lowmask(a & 31);
      if (wi == wz) x &= lowmask(((z - 1) & 31) + 1);
      const int c = popc(x);
      if (r < c) return wi * 32 + select_in_word(x, r);
      r -= c;
    }
    return -1;
  }
  /* extra units the multi-edge runs add before pair rank rk of u's out list */
  CYG_HD int multi_before(int u, int rk) {
    const uint32_t dm = T(n->o_omulti + u);
    int c = 0;
    if (!(dm >> 31)) {
      for (int k = 0; k < 2; k++) {
        const int off = (int)((dm >> (10 * k)) & 0xFFu);
        c += (off != 0xFF && off < rk) ? (int)((dm >> (8 + 10 * k)) & 3u) : 0;
      }
      return c;
    }
    int q = ip(u);
    const int a = q;
    for (int pairs = 0; pairs < rk; pairs++) q += unit_m(unit(q)); /* more than two runs: walk the list, one run per pair */
    return (q - a) - rk;
  }
  CYG_HD int rank_in_row(int u, int v) { /* out-pairs of u with a neighbour id below v */
    int rk = 0;
    for (int w = 0; w < W; w++) {
      const uint32_t r = adj(u, w);
      rk += popc(r & (w < (v >> 5) ? 0xFFFFFFFFu : (lowmask(v & 31) & eqmask(w, v >> 5))));
    }
    return rk;
  }
  /* out-units of u that precede neighbour id v (v itself need not be a neighbour) */
  CYG_HD int units_before_out(int u, int v) {
    const int rk = rank_in_row(u, v);
    return rk + multi_before(u, rk);
  }
  /* in-units of v whose source id is below u: a walk over the in list (only the extra-edge paths need it) */
  CYG_HD int units_before_in(int v, int u) {
    const int a = ip(v) + nout(v), z = ip(v + 1);
    int c = 0;
    for (int q = a; q < z; q++) c += unit_other(unit(q)) < u ? 1 : 0;
    return c;
  }
  CYG_HD int unit_of(int u, int v) { return ip(u) + units_before_out(u, v); } /* first out-unit of base pair (u, v) */
  CYG_HD bool has_edge(int u, int v) { /* g.get_eid(u, v) != -1 (CyberDefenseEnv.py:752-770) */
    if ((adj(u, (v >> 5)) >> (v & 31)) & 1u) return true;
    int nx = n_extra();
    const uint32_t* x = extra();
    uint32_t key = (uint32_t)u | ((uint32_t)v << CYG_X_V_SHIFT);
    for (int j = 0; j < nx; j++) if ((x[j] & 0xFFFFFFu) == key) return true;
    return false;
  }
  /* block / unblock the base pair that unit q belongs to: all its units on both sides */
  CYG_HD void set_pair_blocked(int q, bool b) {
    const uint32_t ui = unit(q);
    const int s = q - unit_off(ui), t = unit_twin(ui), m = unit_m(ui);
    uint32_t* bits = inc();
    const uint32_t was = (bits[s >> 5] >> (s & 31)) & 1u;
    for (int k = 0; k < m; k++) {
      const int q0 = s + k, q1 = t + k;
      if (b) { bits[q0 >> 5] |= 1u << (q0 & 31); bits[q1 >> 5] |= 1u << (q1 & 31); }
      else { bits[q0 >> 5] &= ~(1u << (q0 & 31)); bits[q1 >> 5] &= ~(1u << (q1 & 31)); }
    }
    if (b) nblk() += 1u - was; else nblk() -= was;
  }
  /* _rebuild_graph_cache (volt:456-483) forgets every block (:476) */
  CYG_HD void rebuild_cache() {
    uint32_t* b = inc();
    for (int i = 0; i < n->UW; i++) b[i] = 0;
    nblk() = 0;
    int nx = n_extra();
    uint32_t* x = extra();
    for (int j = 0; j < nx; j++) x[j] &= ~CYG_X_BLOCKED;
  }
  /* id-space rows of the extra edges of device u: xo[] = targets of its extra out-edges whose blocked flag == want_blocked */
  CYG_HD void extra_out_row(int u, bool want_blocked, uint32_t* xo) {
    for (int w = 0; w < W; w++) xo[w] = 0;
    int nx = n_extra();
    const uint32_t* x = extra();
    for (int j = 0; j < nx; j++) {
      const uint32_t xe = x[j];
      if ((int)(xe & CYG_X_IDMASK) != u) continue;
      if (((xe & CYG_X_BLOCKED) != 0) != want_blocked) continue;
      const int v = (int)((xe >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
      for (int w = 0; w < W; w++) xo[w] |= (1u << (v & 31)) & eqmask(w, v >> 5);
    }
  }
  /* ids of the base out-neighbours of u whose pair is blocked */
  CYG_HD void blocked_out_ids(int u, uint32_t* bl) {
    for (int w = 0; w < W; w++) bl[w] = 0;
    const int a = ip(u), no = nout(u);
    if (no <= 0) return;
    const uint32_t* b = inc();
    const int z = a + no, wa = a >> 5, wz = (z - 1) >> 5;
    for (int wi = wa; wi <= wz; wi++) {
      uint32_t x = b[wi];
      if (wi == wa) x &= ~lowmask(a & 31);
      if (wi == wz) x &= lowmask(((z - 1) & 31) + 1);
      while (x) {
        const int q = wi * 32 + ctz(x);
        x &= x - 1;
        const int v = unit_other(unit(q));
        for (int w = 0; w < W; w++) bl[w] |= (1u << (v & 31)) & eqmask(w, v >> 5);
      }
    }
  }

  /* ---- busy tick over _busy_devices (volt:904-908) ---- */
  CYG_HD void tick_busyset() {
    uint32_t m[W];
    for (int w = 0; w < W; w++) m[w] = pl(P_BUSYSET, w);
    busy_dec(m);
  }
  CYG_HD void tick_all() { /* _tick_busy_time_once (volt:607-610) */
    uint32_t m[W];
    for (int w = 0; w < W; w++) m[w] = 0xFFFFFFFFu;
    busy_dec(m);
  }

  /* ---- action decoding (include/cygym_b200.h "actions") ---- */
  struct Act {
    int mode, atype, n_ex, n_dev, app_index;
    int first; /* device_indices[0] carried by a set-form header (hdr[2] >> 16, minus 1); -1: the lowest listed id */
    uint32_t exw;
    const uint32_t* mask;
    const uint16_t* order;
    CYG_HD int ex(int i) const { return (int)(int8_t)((exw >> (8 * i)) & 0xFFu); }
  };
  CYG_HD static void decode(const uint32_t* hdr, const uint32_t* mask, const uint16_t* order, Act& a) {
    uint32_t h0 = hdr[0];
    int at = (int)(h0 & 0xFFu);
    a.atype = at == (int)CYG_ATYPE_NONE ? -1000 : (int)(int8_t)at;
    a.mode = (int)((h0 >> 8) & 1u);
    a.n_ex = (int)((h0 >> 16) & 0xFFu);
    if (a.n_ex > 4) a.n_ex = 4;
    a.exw = hdr[1];
    a.n_dev = (int)(hdr[2] & 0xFFFFu);
    a.first = (int)(hdr[2] >> 16) - 1;
    a.app_index = (int)hdr[3];
    a.mask = mask;
    a.order = order;
  }
  /* iterator over device_indices: explicit order array, or ascending bits of the mask */
  struct DevIter {
    int i, cur;
    CYG_HD DevIter() : i(0), cur(0) {}
  };
  CYG_HD int next_dev(const Act& a, DevIter& it) {
    if (a.order) return (int)a.order[it.i++];
    it.i++;
    int d = it.cur, M = n->M;
    while (d < M) {
      uint32_t x = a.mask[d >> 5] >> (d & 31);
      if (x) { d += ctz(x); break; }
      d = (d | 31) + 1;
    }
    it.cur = d + 1;
    return d < M ? d : -1;
  }
  CYG_HD int first_dev(const Act& a) { /* device_indices[0] */
    DevIter it;
    if (!a.order && a.first >= 0 && a.first < n->M) return a.first; /* sample_action's first draw (CyberDefenseEnv.py:565) */
    return a.n_dev > 0 ? next_dev(a, it) : -1;
  }

  /* ---- defender actions ---- */
  /* busy_time = randint(0, high) for every device of mask a[] in ascending id order (one _stall draw each) */
  CYG_HD void stall_deposit(const uint32_t* a, int low, int high) {
    uint32_t range = (uint32_t)(high - low + 1);
    for (int w = 0; w < W; w++) { /* word by word: the word index stays a compile-time constant */
      uint32_t bits = a[w];
      if (!bits) continue;
      uint32_t r0 = 0, r1 = 0, r2 = 0, r3 = 0;
      while (bits) {
        uint32_t lb = bits & (0u - bits);
        bits ^= lb;
        uint32_t v = (uint32_t)low + below(stall.next(rng), range);
        if (v > CYG_BUSY_MAX) { v = CYG_BUSY_MAX; scal(CYG_S_FLAGS) |= CYG_FL_ERR_BUSY; }
        r0 |= lb & (0u - (v & 1u));
        r1 |= lb & (0u - ((v >> 1) & 1u));
        r2 |= lb & (0u - ((v >> 2) & 1u));
        r3 |= lb & (0u - ((v >> 3) & 1u));
      }
      uint32_t keep = ~a[w];
      pl(P_BUSY0, w) = (pl(P_BUSY0, w) & keep) | r0;
      pl(P_BUSY0 + 1, w) = (pl(P_BUSY0 + 1, w) & keep) | r1;
      pl(P_BUSY0 + 2, w) = (pl(P_BUSY0 + 2, w) & keep) | r2;
      pl(P_BUSY0 + 3, w) = (pl(P_BUSY0 + 3, w) & keep) | r3;
    }
  }
  /* clear isCompromised, compromised_by and the workload of every device in a[] */
  CYG_HD void wipe(const uint32_t* a, bool comp_too) {
    for (int w = 0; w < W; w++) {
      uint32_t keep = ~a[w];
      if (comp_too) {
        pl(P_COMP, w) &= keep;
        for (int k = 0; k < n->ncby; k++) pl(P_CBY0 + k, w) &= keep;
      }
      pl(P_HASWL, w) &= keep;
      pl(P_PT0, w) &= keep; pl(P_PT0 + 1, w) &= keep; pl(P_PT0 + 2, w) &= keep;
    }
  }
  /* device_indices as a set: the first n_dev bits of the mask (what the reference loop visits) */
  CYG_HD void listed(const Act& a, uint32_t* l) {
    int nl = 0;
    for (int w = 0; w < W; w++) { l[w] = (w < n->Wm ? a.mask[w] : 0u) & m_valid(w); nl += popc(l[w]); }
    if (a.n_dev >= nl) return;
    int keep = a.n_dev < 0 ? 0 : a.n_dev, seen = 0; /* inconsistent header: fewer entries than mask bits */
    for (int w = 0; w < W; w++) {
      uint32_t lm = l[w], out = 0;
      while (lm) { uint32_t lb = lm & (0u - lm); lm ^= lb; if (seen++ < keep) out |= lb; }
      l[w] = out;
    }
  }

  /* clean every listed device: volt_typhoon_env.py:996-1011 (and :676-690 in the grouped path), set form.
   * Three pieces so that the kernel can run the draw-bearing part with a whole warp: */
  CYG_HD void clean_mask(const Act& act, uint32_t* a) { /* the devices that get cleaned */
    listed(act, a);
    for (int w = 0; w < W; w++) a[w] &= ~pl(P_NYA, w) & ~pl(P_OWNED, w);
  }
  CYG_HD void clean_scalar(const uint32_t* a, double ds, double& cost) { /* rewards, discovery flags, state wipe */
    int nc = 0, nu = 0;
    uint32_t disc = 0;
    for (int w = 0; w < W; w++) {
      nc += popc(a[w] & pl(P_COMP, w));
      nu += popc(a[w] & ~pl(P_COMP, w));
      for (int k = 0; k < n->ncby; k++) if (pl(P_CBY0 + k, w) & a[w]) disc |= 1u << k;
    }
    cost += (nc * 0.3 - nu * 0.01) * ds;
    cleancost += (nc * 0.3 + nu * 0.01) * ds;
    defcost += (nc * 0.3 + nu * 0.01) * ds;
    scal(CYG_S_FLAGS) |= disc << CYG_FL_DISC_SHIFT; /* exp.discovered = True */
    wipe(a, true);
  }
  CYG_HD void clean_set(const Act& act, double ds, double& cost) {
    uint32_t a[W];
    clean_mask(act, a);
    clean_scalar(a, ds, cost);
    stall_deposit(a, 0, n->cfg.default_high); /* busy_time = randint(0, high) each */
  }
  CYG_HD void clean_device(int d, double ds, double& cost) { /* same, one device (explicit order form) */
    if (bit(P_OWNED, d)) return;
    bool comp = bit(P_COMP, d);
    cost += (comp ? 0.3 : -0.01) * ds;
    cleancost += (comp ? 0.3 : 0.01) * ds;
    defcost += (comp ? 0.3 : 0.01) * ds;
    scal(CYG_S_FLAGS) |= cby(d) << CYG_FL_DISC_SHIFT;
    clr_cby(d);
    clrb(P_COMP, d);
    set_busy(d, stall_draw(0, n->cfg.default_high));
    drop_wl(d);
  }

  /* meta actions shared by step (volt:918-976) and _step_apply_only (volt:627-668) */
  CYG_HD void defender_meta(const Act& a, int atype, bool grouped, double& cost, bool& dirty) {
    const cyg_config& c = n->cfg;
    double ds = (double)c.def_scale;
    if (atype == 2) {
      scal(CYG_S_CKPT)++;
      scal(CYG_S_FLAGS) |= CYG_FL_HAS_CKPT; /* checkpoint_variables stores an alias, not a copy */
      cost += -0.5 * a.n_dev * ds;
      defcost += 0.5 * a.n_dev * ds;
      uint32_t m[W];
      for (int w = 0; w < W; w++) m[w] = busy_nz(w);
      busy_inc(m);
    } else if (atype == 3) {
      scal(CYG_S_REVERT)++;
      if (scal(CYG_S_FLAGS) & CYG_FL_HAS_CKPT) { /* every device: busy = randint(0, high), workload dropped */
        uint32_t all[W];
        for (int w = 0; w < W; w++) all[w] = m_valid(w);
        stall_deposit(all, 0, c.default_high);
        for (int w = 0; w < W; w++) { pl(P_HASWL, w) = 0; pl(P_PT0, w) = 0; pl(P_PT0 + 1, w) = 0; pl(P_PT0 + 2, w) = 0; }
        cost += -1.0 * a.n_dev * ds;
        dirty = true;
      }
    } else if (atype == 10) {
      if (!grouped) { /* volt:946-953; the grouped variant has no busy bump (volt:650-659) */
        if (a.n_dev > 0) {
          int d = first_dev(a);
          if (d >= 0 && d < n->M) set_busy(d, busy(d) + 1);
        } else {
          uint32_t m[W];
          for (int w = 0; w < W; w++) m[w] = busy_nz(w);
          busy_inc(m);
        }
      }
      cost += -1.0 * ds;
      if (scal(CYG_S_LOGS) > 0) /* detector.train(last <= 2000 logs): pending until a fit between launches (cyg_fit_detectors, or detector.py on the host) */
        scal(CYG_S_FLAGS) |= CYG_FL_DET_TRAINED | (n->cfg.turbo ? 0u : CYG_FL_DET_PENDING);
    } else if (atype == 11) {
      int d = first_dev(a); /* the host raises ValueError when n_dev == 0 (volt:965-966) */
      if (d >= 0 && d < n->M) {
        uint32_t k = CYG_CK_VALID;
        if (bit(P_COMP, d)) k |= CYG_CK_COMP;
        if (bit(P_KNOWN, d)) k |= CYG_CK_KNOWN;
        if (bit(P_NYA, d)) k |= CYG_CK_NYA;
        if (dev_static(d) & CYG_ST_REACH) k |= CYG_CK_REACH;
        if (bit(P_HASWL, d)) k |= CYG_CK_HASWL | (field(P_PT0, 3, d) << CYG_DEV_PT_SHIFT);
        k |= busy(d) << CYG_DEV_BUSY_SHIFT;
        k |= cby(d) << CYG_DEV_CBY_SHIFT;
        ckpt[d] = k | (ckpt[d] & CYG_CKI_REMOVED);
        scal(CYG_S_CKPT)++;
        cost += -0.1 * ds;
        defcost += 0.1 * ds;
      }
    }
  }

  CYG_HD void restore_device(int d) { /* _apply_device_state (volt:430-437) */
    uint32_t k = ckpt[d];
    if (k & CYG_CK_COMP) setb(P_COMP, d); else clrb(P_COMP, d);
    if (k & CYG_CK_KNOWN) setb(P_KNOWN, d); else clrb(P_KNOWN, d);
    if (k & CYG_CK_NYA) setb(P_NYA, d); else clrb(P_NYA, d);
    drop_wl(d);
    if (k & CYG_CK_HASWL) { setb(P_HASWL, d); set_field(P_PT0, 3, d, (k >> CYG_DEV_PT_SHIFT) & CYG_DEV_PT_MASK); }
    set_busy(d, (k >> CYG_DEV_BUSY_SHIFT) & CYG_DEV_BUSY_MASK);
    set_field(P_CBY0, n->ncby, d, (k >> CYG_DEV_CBY_SHIFT) & CYG_DEV_CBY_MASK);
  }

  /* block / unblock one incident edge of d (volt:1071-1080, :1091-1100, :485-511):
   * pool = out-edges then in-edges whose blocked flag == want, each repeated `multiplicity` times == the units of
   * [ip[d], ip[d+1]) with that flag: its size is a popcount and the pick a select. */
  CYG_HD bool flip_incident(int d, bool want, Stream& st) {
    if (n_extra() > 0) return flip_incident_general(d, want, st);
    const uint32_t flipw = want ? 0u : 0xFFFFFFFFu;
    const int a = ip(d), len = ip(d + 1) - a;
    const int total = range_count(a, len, flipw);
    if (total == 0) return false;
    const int q = range_select(a, len, flipw, (int)below(st.next(rng), (uint32_t)total));
    set_pair_blocked(q, !want);
    return true;
  }
  /* The same for an env with extra (hub-star) edges: those sit in the per-env list, not in the unit bitset, and enter
   * the out list / in list at their place in ascending neighbour order.  A merged walk: per list, the extras of d in
   * ascending far-endpoint id, each preceded by the base units in front of it. */
  CYG_HD bool flip_incident_general(int d, bool want, Stream& st) {
    const uint32_t flipw = want ? 0u : 0xFFFFFFFFu;
    const int a = ip(d), no = nout(d), z = ip(d + 1);
    const int nx = n_extra();
    uint32_t* x = extra();
    int nxe = 0;
    for (int j = 0; j < nx; j++) {
      const uint32_t xe = x[j];
      const int u = (int)(xe & CYG_X_IDMASK), v = (int)((xe >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
      if ((u == d || v == d) && (((xe & CYG_X_BLOCKED) != 0) == want)) nxe++;
    }
    const int total = range_count(a, z - a, flipw) + nxe;
    if (total == 0) return false;
    int r = (int)below(st.next(rng), (uint32_t)total);
    for (int side = 0; side < 2; side++) { /* out list, then in list */
      int cursor = side ? a + no : a;
      const int end = side ? z : a + no;
      int last = -1;
      for (;;) { /* next extra of this side in ascending far-endpoint id */
        int best = -1, bid = 0x7FFFFFFF;
        for (int j = 0; j < nx; j++) {
          const uint32_t xe = x[j];
          const int u = (int)(xe & CYG_X_IDMASK), v = (int)((xe >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
          if ((side ? v : u) != d || (((xe & CYG_X_BLOCKED) != 0) != want)) continue;
          const int far_id = side ? u : v;
          if (far_id > last && far_id < bid) { bid = far_id; best = j; }
        }
        if (best < 0) break;
        last = bid;
        const int p = side ? a + no + units_before_in(d, bid) : a + units_before_out(d, bid);
        const int cb = range_count(cursor, p - cursor, flipw);
        if (r < cb) { set_pair_blocked(range_select(cursor, p - cursor, flipw, r), !want); return true; }
        r -= cb;
        cursor = p;
        if (r == 0) { if (want) x[best] &= ~CYG_X_BLOCKED; else x[best] |= CYG_X_BLOCKED; return true; }
        r--;
      }
      const int cb = range_count(cursor, end - cursor, flipw);
      if (r < cb) { set_pair_blocked(range_select(cursor, end - cursor, flipw, r), !want); return true; }
      r -= cb;
    }
    return false; /* not reached: r < total */
  }

  /* set / clear the units [s, s + m) of the bitset (m <= 4: at most one word boundary) */
  CYG_HD void set_run(uint32_t* bits, int s, int m, bool b) {
    const int sh = s & 31;
    const uint32_t lo = lowmask(m) << sh;
    uint32_t& w0 = bits[s >> 5];
    w0 = b ? (w0 | lo) : (w0 & ~lo);
    if (sh + m > 32) {
      const uint32_t hi = lowmask(m) >> (32 - sh);
      uint32_t& w1 = bits[(s >> 5) + 1];
      w1 = b ? (w1 | hi) : (w1 & ~hi);
    }
  }
  /* block / unblock for every device of act[] in ascending id order (the set form of volt:1071-1100), one thread per
   * env.  The pool of a device with at most 128 units is a 4-word window of the unit bitset, read, weighed and
   * selected from with no data-dependent branch, so that the 32 envs of a warp walk their lists in lock step (one
   * iteration per listed device, whatever its degree).  Returns the number of flips. */
  CYG_HD uint32_t flip_walk(uint32_t* act, bool want, int site) {
    const uint32_t flipw = want ? 0u : 0xFFFFFFFFu;
    Stream st(site);
    uint32_t cnt = 0;
    uint32_t* b = inc();
    const bool has_x = n_extra() > 0;
    for (;;) {
      const int d = pop_lowest(act);
      if (d < 0) break;
      if (has_x) { cnt += flip_incident_general(d, want, st) ? 1u : 0u; continue; }
      const uint32_t di = dinfo(d), di1 = dinfo(d + 1);
      const int a = (int)(di & 0xFFFFu), nt = (int)(di1 & 0xFFFFu) - a;
      int q;
      if (nt <= 128) {
        const int wa = a >> 5, sh = a & 31;
        uint32_t x[4];
        uint32_t lo = b[wa];
        for (int i = 0; i < 4; i++) {
#ifdef __CUDA_ARCH__
          const uint32_t hi = SM ? b[wa + i + 1] : (wa + i + 1 <= n->UW ? b[wa + i + 1] : 0u); /* shared memory: whatever follows is readable and masked off */
#else
          const uint32_t hi = wa + i + 1 <= n->UW ? b[wa + i + 1] : 0u;
#endif
          x[i] = (funnel_r(lo, hi, sh) ^ flipw) & lowmask0(nt - 32 * i);
          lo = hi;
        }
        const int c0 = popc(x[0]), c1 = popc(x[1]), c2 = popc(x[2]), c3 = popc(x[3]);
        const int total = c0 + c1 + c2 + c3;
        if (total == 0) continue;
        const int r = (int)below(st.next(rng), (uint32_t)total);
        /* word holding unit r, branch-free */
        const bool g1 = r >= c0, g2 = r >= c0 + c1, g3 = r >= c0 + c1 + c2;
        const uint32_t xw = g3 ? x[3] : g2 ? x[2] : g1 ? x[1] : x[0];
        const int base = g3 ? c0 + c1 + c2 : g2 ? c0 + c1 : g1 ? c0 : 0;
        const int wsel = (g1 ? 1 : 0) + (g2 ? 1 : 0) + (g3 ? 1 : 0);
        q = a + 32 * wsel + select_in_word(xw, r - base);
      } else {
        const int total = range_count(a, nt, flipw);
        if (total == 0) continue;
        q = range_select(a, nt, flipw, (int)below(st.next(rng), (uint32_t)total));
      }
      const uint32_t ui = unit(q);
      const int m = unit_m(ui);
      set_run(b, q - unit_off(ui), m, !want);
      set_run(b, unit_twin(ui), m, !want);
      cnt++;
    }
    if (!has_x) { if (want) nblk() -= cnt; else nblk() += cnt; }
    return cnt;
  }

  /* devices of act[] with app_index < len(device.apps) (volt:1014-1016): bit-sliced compare over the napps planes */
  CYG_HD void upgrade_mask(const uint32_t* act, int app_index, uint32_t* up) {
    for (int w = 0; w < W; w++) {
      uint32_t gt = 0, eq = 0xFFFFFFFFu;
      for (int bb = 7; bb >= 0; bb--) {
        uint32_t nb = T(n->o_napps + bb * W + w), ab = ((app_index >> bb) & 1) ? 0xFFFFFFFFu : 0u;
        gt |= eq & nb & ~ab;
        eq &= ~(nb ^ ab);
      }
      up[w] = (app_index >= 0 && app_index < 256) ? (act[w] & gt) : 0u;
    }
  }
  /* listed (first n_dev mask bits) & active */
  CYG_HD int listed_active(const Act& a, uint32_t* act) {
    int na = 0;
    listed(a, act);
    for (int w = 0; w < W; w++) { act[w] &= ~pl(P_NYA, w); na += popc(act[w]); }
    return na;
  }

  /* per-device defender actions when device_indices is a SET (ascending, duplicate-free): the loop of
   * volt:989-1123 collapses to word-wide operations for every type but block / unblock */
  CYG_HD void defender_per_device_set(const Act& a, int atype, double& cost, bool& dirty) {
    const cyg_config& c = n->cfg;
    double ds = (double)c.def_scale;
    if (atype == 1) { clean_set(a, ds, cost); return; }
    uint32_t act[W];
    int na = listed_active(a, act);
    if (na == 0) return;
    switch (atype) {
      case 4: { /* volt:1013-1018 */
        cost += -1.0 * ds * na;
        uint32_t up[W];
        upgrade_mask(act, a.app_index, up);
        stall_deposit(up, 0, c.default_high);
      } break;
      case 5: /* volt:1020-1069: an untrained detector predicts "D" for everything; a trained one is consulted */
        scal(CYG_S_SCAN) += (uint32_t)na;
        if (scal(CYG_S_LOGS) > 0) {
          if ((scal(CYG_S_FLAGS) & CYG_FL_DET_TRAINED) && !n->cfg.turbo) /* turbo: predictions = [] (volt:1055) */
            stall.k = scan_trained_call<W, SM>(n, rec, ro, to, logs, det, rng.env, stall.k, na);
          cost += -0.5 * ds * na;
          defcost += 0.5 * ds * na;
        }
        break;
      case 6: case 9: {
        cost += -0.5 * ds * na;
        defcost += 0.5 * ds * na;
        const uint32_t cnt = flip_walk(act, atype == 9, atype == 6 ? SITE_BLOCK : SITE_UNBLOCK);
        if (cnt) { scal(atype == 6 ? CYG_S_EBLK : CYG_S_EADD) += cnt; dirty = true; }
      } break;
      case 7: /* volt:1082-1089 */
        cost += -0.5 * ds * na;
        for (int w = 0; w < W; w++) pl(P_NYA, w) |= act[w];
        wipe(act, true);
        dirty = true;
        break;
      case 12: { /* acts on device_indices[0] once per listed active device (volt:1102-1109) */
        int dev0 = first_dev(a);
        if (ckpt[dev0] & CYG_CK_VALID) {
          /* the first restore rewrites Not_yet_added of dev0 itself: when dev0 is not the first active listed device
           * (sample_action's draw order), its own iteration is skipped / taken by the CHECKPOINTED flag */
          uint32_t l[W];
          listed(a, l);
          int before = 0;
          bool l0 = false, a0 = false;
          for (int w = 0; w < W; w++) {
            const uint32_t b0 = (1u << (dev0 & 31)) & eqmask(w, dev0 >> 5);
            before += popc(act[w] & (w < (dev0 >> 5) ? 0xFFFFFFFFu : ((b0 - 1u) & eqmask(w, dev0 >> 5))));
            l0 = l0 || (l[w] & b0) != 0;
            a0 = a0 || (act[w] & b0) != 0;
          }
          const int others = na - (a0 ? 1 : 0);
          const bool cnt0 = before > 0 ? (l0 && !(ckpt[dev0] & CYG_CK_NYA)) : a0;
          const int total = others + (cnt0 ? 1 : 0);
          if (total > 0) {
            restore_device(dev0);
            cost += -1.0 * ds * total;
            defcost += 1.0 * ds * total;
          }
        }
      } break;
      case 13: { /* volt:1111-1123: only the last of the `na` _stall draws survives */
        int dev0 = first_dev(a);
        clrb(P_COMP, dev0);
        clr_cby(dev0);
        drop_wl(dev0);
        stall.skip(rng, (uint32_t)(na - 1));
        set_busy(dev0, stall_draw(3, c.default_high + 3));
        cost += -3.0 * ds * na;
        cleancost += 3.0 * ds * na;
        defcost += 3.0 * ds * na;
      } break;
      default: break;
    }
  }

  /* per-device defender actions in listed order (volt:989-1123): explicit order form (may repeat devices) */
  CYG_HD void defender_per_device_seq(const Act& a, int atype, double& cost, bool& dirty) {
    const cyg_config& c = n->cfg;
    double ds = (double)c.def_scale;
    int dev0 = first_dev(a);
    DevIter it;
    Stream sblk(SITE_BLOCK), sunb(SITE_UNBLOCK);
    for (int i = 0; i < a.n_dev; i++) {
      int d = next_dev(a, it);
      if (d < 0 || d >= n->M) break;
      if (bit(P_NYA, d)) continue;
      switch (atype) {
        case 1: clean_device(d, ds, cost); break;
        case 4:
          cost += -1.0 * ds;
          if (a.app_index >= 0 && a.app_index < (int)((dev_static(d) >> CYG_ST_NAPPS_SHIFT) & 0xFFu))
            set_busy(d, stall_draw(0, c.default_high));
          break;
        case 5:
          scal(CYG_S_SCAN)++;
          if (scal(CYG_S_LOGS) > 0) {
            if ((scal(CYG_S_FLAGS) & CYG_FL_DET_TRAINED) && !n->cfg.turbo) /* turbo: predictions = [] (volt:1055) */
              stall.k = scan_trained_call<W, SM>(n, rec, ro, to, logs, det, rng.env, stall.k, 1);
            cost += -0.5 * ds;
            defcost += 0.5 * ds;
          }
          break;
        case 6:
          cost += -0.5 * ds;
          defcost += 0.5 * ds;
          if (flip_incident(d, false, sblk)) { scal(CYG_S_EBLK)++; dirty = true; }
          break;
        case 7:
          cost += -0.5 * ds;
          setb(P_NYA, d);
          clrb(P_COMP, d);
          clr_cby(d);
          drop_wl(d);
          dirty = true;
          break;
        case 9:
          cost += -0.5 * ds;
          defcost += 0.5 * ds;
          if (flip_incident(d, true, sunb)) { scal(CYG_S_EADD)++; dirty = true; }
          break;
        case 12:
          if (ckpt[dev0] & CYG_CK_VALID) {
            restore_device(dev0);
            cost += -1.0 * ds;
            defcost += 1.0 * ds;
          }
          break;
        case 13:
          clrb(P_COMP, dev0);
          clr_cby(dev0);
          drop_wl(dev0);
          set_busy(dev0, stall_draw(3, c.default_high + 3));
          cost += -3.0 * ds;
          cleancost += 3.0 * ds;
          defcost += 3.0 * ds;
          break;
        default: break;
      }
    }
  }
  CYG_HD void defender_per_device(const Act& a, int atype, double& cost, bool& dirty) {
    if (a.order) defender_per_device_seq(a, atype, cost, dirty);
    else defender_per_device_set(a, atype, cost, dirty);
  }

  /* ---- attacker actions (volt:1126-1202) ---- */
  /* unblocked out-neighbours of s (base row minus blocked pairs, plus unblocked extra edges) */
  CYG_HD void live_row(int s, bool has_blk, int nx, uint32_t* row) {
    uint32_t bl[W], xo[W];
    for (int w = 0; w < W; w++) { bl[w] = 0; xo[w] = 0; }
    if (has_blk) blocked_out_ids(s, bl);
    if (nx > 0) extra_out_row(s, false, xo);
    for (int w = 0; w < W; w++) row[w] = (adj(s, w) & ~bl[w]) | xo[w];
  }
  /* One source of the lateral-movement loop (volt:1148-1185): scan the unblocked out-neighbours of s in ascending
   * order; a DomainController source hits the first one, otherwise the first that is reachable_by_attacker or
   * (not compromised, known, vulnerable to the exploit).  comp[] = current isCompromised words, kv[] = known &
   * vulnerable, xrow = unblocked extra out-neighbours of s (nullptr: none).  Returns the hit device (-1: none); cnt =
   * hops logged before the hit (log_communication, volt:1161: every repeat of a multi-edge counts) = unblocked units in
   * front of the hit's first unit; rule3 = the hit relied on "not yet compromised". */
  CYG_HD int attack_source(int s, const uint32_t* comp, const uint32_t* kv, bool has_blk, const uint32_t* xrow, int& cnt, bool& rule3) {
    const bool is_dc = devbit(n->o_dc, s);
    const int a = ip(s), no = nout(s);
    uint32_t row[W], cand[W], xc[W];
    for (int w = 0; w < W; w++) {
      const uint32_t ok = is_dc ? 0xFFFFFFFFu : (m_reach(w) | (~comp[w] & kv[w]));
      row[w] = adj(s, w);
      xc[w] = xrow ? (xrow[w] & ok) : 0u;
      cand[w] = (row[w] & ok) | xc[w];
    }
    int vw = -1, upos = no; /* units walked in front of the hit (all of them when nothing is hit) */
    uint32_t hitbit = 0;
    for (;;) { /* first candidate whose edge is not blocked (volt:1157-1159) */
      int w0 = -1;
      uint32_t cw = 0, xw = 0;
      for (int w = W - 1; w >= 0; w--) { bool nz = cand[w] != 0; w0 = nz ? w : w0; cw = nz ? cand[w] : cw; xw = nz ? xc[w] : xw; }
      if (w0 < 0) break;
      const uint32_t lb = cw & (0u - cw);
      int rk = 0;
      for (int w = 0; w < W; w++) rk += popc(row[w] & ((w < w0 ? 0xFFFFFFFFu : 0u) | ((lb - 1u) & eqmask(w, w0))));
      const int up = rk + multi_before(s, rk);
      if (!(xw & lb) && has_blk && ubit(a + up)) { /* a blocked base pair: not walked, not logged */
        for (int w = 0; w < W; w++) cand[w] ^= lb & eqmask(w, w0);
        continue;
      }
      vw = w0; hitbit = lb; upos = up;
      break;
    }
    cnt = upos;
    if (has_blk) { /* minus the blocked units in front of the hit */
#ifdef __CUDA_ARCH__
      if (SM && W <= CYG_MAX_W) { /* shared memory, out lists of at most 128 units: a 4-word window, no data-dependent loop */
        const uint32_t* b = inc();
        const int wa = a >> 5, sh = a & 31;
        uint32_t lo = b[wa];
        int blk_n = 0;
        bool fits = upos <= 128;
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const uint32_t hi = b[wa + i + 1];
          blk_n += popc(funnel_r(lo, hi, sh) & lowmask0(upos - 32 * i));
          lo = hi;
        }
        cnt -= fits ? blk_n : range_count(a, upos, 0u);
      } else
#endif
      cnt -= range_count(a, upos, 0u);
    }
    if (xrow) { /* unblocked extra edges in front of the hit (all of them when nothing is hit) */
      for (int w = 0; w < W; w++) {
        const uint32_t bm = vw < 0 ? 0xFFFFFFFFu : ((w < vw ? 0xFFFFFFFFu : 0u) | ((hitbit - 1u) & eqmask(w, vw)));
        cnt += popc(xrow[w] & bm);
      }
    }
    if (vw < 0) { rule3 = false; return -1; }
    const int v = vw * 32 + ctz(hitbit);
    rule3 = !is_dc && !devbit(n->o_reach, v);
    return v;
  }
  /* The hop-log records of one source of the lateral-movement loop (log_communication, volt:1161 ->
   * CDSimulator.py:667-673): every unblocked out-edge walked in front of the hit, then the hit -- base units in unit
   * order, the unblocked extra edges (xrow, id space) at their place in ascending neighbour order.  Record k of the
   * source gets log index idx0 + k and is written to the ring when that index is >= lo_keep (a warp that logs several
   * sources at once only writes what a ring of log_cap records will still hold). */
  CYG_HD void log_source(int s, int hit, bool has_blk, const uint32_t* xrow, uint32_t idx0, uint32_t lo_keep) {
    const uint32_t cap = (uint32_t)n->cfg.log_cap;
    uint32_t* ring = logs;
    uint32_t xr[W];
    for (int w = 0; w < W; w++) xr[w] = xrow ? xrow[w] : 0u;
    uint32_t idx = idx0;
    /* the extra edges with a neighbour id below v, ascending */
    auto extras_below = [&](int v) {
      for (int w = 0; w < W; w++) {
        while (xr[w]) {
          const int d = w * 32 + ctz(xr[w]);
          if (d >= v) return;
          xr[w] &= xr[w] - 1u;
          if (idx >= lo_keep) ring[idx % cap] = (uint32_t)s | ((uint32_t)d << 16);
          idx++;
        }
      }
    };
    const int a = ip(s), z = a + nout(s);
    for (int q = a; q < z; q++) {
      const int v = unit_other(unit(q));
      if (hit >= 0 && v > hit) break;
      if (hit >= 0 && v == hit) { /* the hit is this base pair: its first unit, nothing behind it */
        extras_below(v);
        if (idx >= lo_keep) ring[idx % cap] = (uint32_t)s | ((uint32_t)v << 16);
        return;
      }
      if (has_blk && ubit(q)) continue;
      extras_below(v);
      if (idx >= lo_keep) ring[idx % cap] = (uint32_t)s | ((uint32_t)v << 16);
      idx++;
    }
    if (hit >= 0) { /* the hit is an extra edge */
      extras_below(hit);
      if (idx >= lo_keep) ring[idx % cap] = (uint32_t)s | ((uint32_t)hit << 16);
    } else {
      extras_below(0x7FFFFFFF);
    }
  }

  /* ---- trained detector: predict == two tree walks + the verdict bit of the leaf pair (include/cygym_b200.h CYG_DET_*;
   *      CDSimulator.py:714-723).  sklearn: a float32 sample goes left when X[feature] <= threshold (float64). ---- */
  CYG_HD int det_leaf(const uint32_t* tree, double from, double to) const {
    int node = 0;
    for (;;) {
      const uint32_t* nd = tree + 4 * node;
      const int feat = (int)(nd[3] & 0xFFFFu);
      if (feat >= 2) return (int)(nd[3] >> 16);
      const uint64_t bits = (uint64_t)nd[0] | ((uint64_t)nd[1] << 32);
      double thr;
#ifdef __CUDA_ARCH__
      thr = __longlong_as_double((long long)bits);
#else
      __builtin_memcpy(&thr, &bits, 8);
#endif
      node = ((feat == 0 ? from : to) <= thr) ? (int)(nd[2] & 0xFFFFu) : (int)(nd[2] >> 16);
    }
  }
  CYG_HD bool det_anomaly(int from, int to) const {
    const int l0 = det_leaf(det + CYG_DET_TREE0, (double)from, (double)to);
    const int l1 = det_leaf(det + CYG_DET_TREE0 + CYG_DET_TREE_STRIDE, (double)from, (double)to);
    const uint32_t idx = (uint32_t)l0 * det[0] + (uint32_t)l1;
    return (det[CYG_DET_TABLE + (idx >> 5)] >> (idx & 31)) & 1u;
  }
  /* Iteration order of the CPython set built by inserting the small non-negative ints vals[0..n) in that order: the
   * reference walks `flagged_senders`, a set, handing out one _stall draw per member (volt:1062-1069).  Objects/
   * setobject.c (3.12): hash(v) == v, open addressing with 9 linear probes, then i = i*5 + 1 + (perturb >>= 5);
   * the table grows to the first power of two > 4 * used once fill * 5 >= mask * 3.  n <= 30 here. */
  CYG_HD static int pyset_order(const int* vals, int cnt_in, int* out) {
    int table[128], tmp[128];
    int mask = 7, fill = 0;
    for (int i = 0; i <= mask; i++) table[i] = -1;
    for (int k = 0; k < cnt_in; k++) {
      const int key = vals[k];
      uint64_t perturb = (uint64_t)key;
      uint32_t i = (uint32_t)key & (uint32_t)mask;
      int placed = 0;
      while (!placed) {
        int probes = (i + 9u <= (uint32_t)mask) ? 9 : 0;
        uint32_t j = i;
        do {
          if (table[j] < 0) { table[j] = key; fill++; placed = 1; break; }
          if (table[j] == key) { placed = 2; break; }
          j++;
        } while (probes--);
        if (placed) break;
        perturb >>= 5;
        i = (uint32_t)((i * 5ull + 1ull + perturb) & (uint64_t)mask);
      }
      if (placed == 1 && !((uint64_t)fill * 5ull < (uint64_t)mask * 3ull)) {
        int newsize = 8;
        while (newsize <= fill * 4) newsize <<= 1;
        const int newmask = newsize - 1;
        for (int q = 0; q <= newmask; q++) tmp[q] = -1;
        for (int q = 0; q <= mask; q++) {
          if (table[q] < 0) continue;
          const int kk = table[q];
          uint64_t pb = (uint64_t)kk;
          uint32_t ii = (uint32_t)kk & (uint32_t)newmask;
          for (;;) {
            int probes = (ii + 9u <= (uint32_t)newmask) ? 9 : 0;
            uint32_t jj = ii;
            bool ok = false;
            do { if (tmp[jj] < 0) { tmp[jj] = kk; ok = true; break; } jj++; } while (probes--);
            if (ok) break;
            pb >>= 5;
            ii = (uint32_t)((ii * 5ull + 1ull + pb) & (uint64_t)newmask);
          }
        }
        mask = newmask;
        for (int q = 0; q <= mask; q++) table[q] = tmp[q];
      }
    }
    int c = 0;
    for (int q = 0; q <= mask; q++) if (table[q] >= 0) out[c++] = table[q];
    return c;
  }
  /* `reps` iterations of the scan body volt:1052-1069 (one per listed active device; the log does not change in
   * between, so the predictions are the same in each): the last 30 records are scored; with a majority of anomalies
   * every flagged sender is un-compromised and stalled -- one _stall draw each per iteration, in set order, of which
   * the last iteration's survive. */
  CYG_HD void scan_trained_body(int reps) {
    const cyg_config& c = n->cfg;
    const uint32_t nlogs = scal(CYG_S_LOGS);
    if (!det || !logs || (scal(CYG_S_FLAGS) & CYG_FL_DET_PENDING) || (c.log_cap < 30 && (uint32_t)c.log_cap < nlogs)) {
      scal(CYG_S_FLAGS) |= CYG_FL_ERR_DETECTOR;
      return;
    }
    const int nw = nlogs < 30u ? (int)nlogs : 30;
    int senders[30], order[30], ns = 0, n_anom = 0;
    for (int k = 0; k < nw; k++) {
      const uint32_t r = logs[(nlogs - (uint32_t)nw + (uint32_t)k) % (uint32_t)c.log_cap];
      const int from = (int)(r & 0xFFFFu), to = (int)(r >> 16);
      if (det_anomaly(from, to)) { n_anom++; senders[ns++] = from; }
    }
    if (n_anom < nw / 2 + 1) return;
    const int cnt = pyset_order(senders, ns, order);
    stall.skip(rng, (uint32_t)(reps - 1) * (uint32_t)cnt);
    for (int k = 0; k < cnt; k++) {
      const int d = order[k];
      clrb(P_COMP, d);
      set_busy(d, stall_draw(0, c.default_high));
    }
  }

  /* the exploit slot an attack uses: zero-day remap (volt:1131-1146); -1 = no such exploit */
  CYG_HD int resolve_exploit(int raw, uint32_t zday_draw) {
    const cyg_config& c = n->cfg;
    if (c.zero_day && !(raw >= 0 && raw < 32 && ((c.zero_day_mask >> raw) & 1u))) /* volt:1135-1136 */
      raw = select_in_word(c.zero_day_mask, (int)below(zday_draw, (uint32_t)popc(c.zero_day_mask)));
    return (raw >= 0 && raw < c.n_exploits) ? raw : -1; /* ids are strings: an int never matches (volt:1141) */
  }
  CYG_HD bool needs_zday_draw(int raw) {
    const cyg_config& c = n->cfg;
    return c.zero_day && !(raw >= 0 && raw < 32 && ((c.zero_day_mask >> raw) & 1u));
  }

  CYG_HD void attacker_act(const Act& a, int atype, double& cost) {
    if (bl == CYG_BL_NO_ATTACK) return;
    if (atype != 1 && atype != 2) return;
    uint32_t src[W]; /* snapshot of compromised-or-owned devices, taken before the loop (volt:1127-1128) */
    int ns = 0;
    for (int w = 0; w < W; w++) { src[w] = pl(P_COMP, w) | pl(P_OWNED, w); ns += popc(src[w]); }
    const bool has_blk = any_blocked();
    const int nx = n_extra();
    if (atype == 1) {
      Stream zday(SITE_ZDAY);
      uint32_t logs = scal(CYG_S_LOGS);
      uint32_t comp[W], known[W];
      for (int w = 0; w < W; w++) { comp[w] = pl(P_COMP, w); known[w] = pl(P_KNOWN, w); }
      for (int xi = 0; xi < a.n_ex; xi++) {
        int raw = a.ex(xi);
        raw = resolve_exploit(raw, needs_zday_draw(raw) ? zday.next(rng) : 0u);
        if (raw < 0) continue;
        uint32_t kv[W], dcby[W]; /* known & vulnerable to this exploit; compromised_by additions */
        for (int w = 0; w < W; w++) { kv[w] = known[w] & m_vuln(raw, w); dcby[w] = 0; }
        uint32_t todo[W];
        for (int w = 0; w < W; w++) todo[w] = src[w];
        for (;;) {
          const int s = pop_lowest(todo);
          if (s < 0) break;
          int cnt;
          bool rule3;
          uint32_t xrow[W];
          if (nx > 0) extra_out_row(s, false, xrow);
          const int v = attack_source(s, comp, kv, has_blk, nx > 0 ? xrow : (const uint32_t*)0, cnt, rule3);
          if (this->logs) log_source(s, v, has_blk, nx > 0 ? xrow : (const uint32_t*)0, logs, 0u);
          logs += (uint32_t)cnt + (v >= 0 ? 1u : 0u);
          if (v >= 0) {
            const bool is_dc = devbit(n->o_dc, s);
            for (int w = 0; w < W; w++) {
              uint32_t hb = (1u << (v & 31)) & eqmask(w, v >> 5);
              comp[w] |= hb;
              dcby[w] |= is_dc ? hb : 0u;
            }
          }
        }
        for (int w = 0; w < W; w++) if (dcby[w]) pl(P_CBY0 + raw, w) |= dcby[w];
      }
      for (int w = 0; w < W; w++) pl(P_COMP, w) = comp[w];
      scal(CYG_S_LOGS) = logs;
    } else { /* probe (volt:1187-1202) */
      if (ns > 0) {
        Stream sp(SITE_PROBE);
        int s = select_nth(src, (int)below(sp.next(rng), (uint32_t)ns));
        uint32_t row[W];
        live_row(s, has_blk, nx, row);
        for (int w = 0; w < W; w++) {
          uint32_t cand = row[w] & ~pl(P_KNOWN, w);
          if (cand) { pl(P_KNOWN, w) |= cand & (0u - cand); cost += 0.1; break; }
        }
      }
    }
  }

  /* ---- workload advance (volt:1242-1261); returns current_work ---- */
  CYG_HD int workload_advance() {
    int cur = 0;
    for (int w = 0; w < W; w++) {
      uint32_t p0 = pl(P_PT0, w), p1 = pl(P_PT0 + 1, w), p2 = pl(P_PT0 + 2, w);
      uint32_t m = ~busy_nz(w) & ~pl(P_NYA, w) & pl(P_HASWL, w) & (p0 | p1 | p2);
      uint32_t b = m; /* processing_time -= 1 on m */
      uint32_t q0 = p0 ^ b; b &= ~p0;
      uint32_t q1 = p1 ^ b; b &= ~p1;
      uint32_t q2 = p2 ^ b;
      uint32_t fin = m & ~(q0 | q1 | q2);
      pl(P_PT0, w) = q0; pl(P_PT0 + 1, w) = q1; pl(P_PT0 + 2, w) = q2;
      pl(P_HASWL, w) &= ~fin;
      cur += popc(fin);
    }
    scal(CYG_S_WORK) += (uint32_t)cur;
    return cur;
  }

  /* ---- arrivals (volt:575-596, :141-145, :184-191, :266-293; CDSimulator.py:244-348) ---- */
  CYG_HD void generate_workloads(int num_loads, bool server, int n_active, Stream& ssamp, Stream& stri) {
    const cyg_config& c = n->cfg;
    if (n_active <= 0) return;                                  /* volt:205-207 */
    if (c.wl_cap >= 0 && num_loads > c.wl_cap) num_loads = c.wl_cap; /* volt:210-211 */
    if (c.turbo) { /* cap + ramp (volt:219-231) */
      int frac_cap = (int)((server ? c.turbo_frac_servers : c.turbo_frac_clients) * (double)n_active);
      if (frac_cap < 1) frac_cap = 1;
      int hard_cap = server ? c.turbo_max_servers : c.turbo_max_clients;
      double ramp = (double)scal(CYG_S_STEP) / (double)(c.turbo_ramp_steps > 1 ? c.turbo_ramp_steps : 1);
      if (ramp > 1.0) ramp = 1.0;
      int base = frac_cap < hard_cap ? frac_cap : hard_cap;
      int turbo_cap = (int)rint((double)base * ramp); /* Python round(): half to even */
      if (turbo_cap < 1) turbo_cap = 1;
      if (num_loads > turbo_cap) num_loads = turbo_cap;
    }
    if (num_loads > n_active) num_loads = n_active;             /* volt:234 */
    if (num_loads <= 0) return;
    uint32_t cand[W];
    int nc = 0;
    for (int w = 0; w < W; w++) {
      uint32_t t = m_valid(w) & ~pl(P_NYA, w) & ~pl(P_HASWL, w) & ~busy_nz(w);
      t &= server ? m_server(w) : ~m_server(w);
      cand[w] = t;
      nc += popc(t);
    }
    int k = num_loads < nc ? num_loads : nc;
    for (int j = 0; j < k; j++) { /* random.sample: pop the r-th remaining candidate (CDSimulator.py:298) */
      int r = (int)below(ssamp.next(rng), (uint32_t)(nc - j));
      int did = select_nth(cand, r);
      for (int w = 0; w < W; w++) cand[w] &= ~((1u << (did & 31)) & eqmask(w, did >> 5));
      uint32_t xt = stri.next(rng); /* CDSimulator.py:308 */
      int pt = 1;
      for (int v = 0; v < 8; v++) pt += xt >= c.tri_tab[v];
      if (pt > c.tri_high) pt = c.tri_high;
      setb(P_HASWL, did);
      set_field(P_PT0, 3, did, (uint32_t)pt);
    }
  }
  CYG_HD void arrivals_if_due() {
    const cyg_config& c = n->cfg;
    int n_active = 0, idle = 0, free_s = 0;
    for (int w = 0; w < W; w++) {
      uint32_t act = m_valid(w) & ~pl(P_NYA, w);
      uint32_t idl = act & ~busy_nz(w) & ~pl(P_HASWL, w);
      n_active += popc(act);
      idle += popc(idl);
      free_s += popc(idl & m_server(w));
    }
    int free_c = idle - free_s;
    /* _arrival_period (volt:141-145) */
    int period; /* int(base + 0.5 * sqrt(max(1, n_active))) == base + max{k : 4k^2 <= n} for base >= 0 */
    {
      int na1 = n_active > 1 ? n_active : 1;
      if (c.wl_period_base >= 0) {
        int k = 0;
        while (4 * (k + 1) * (k + 1) <= na1) k++;
        period = c.wl_period_base + k;
      } else {
        period = (int)(c.wl_period_base + 0.5 * sqrt((double)na1));
      }
    }
    if (period < 10) period = 10;
    if (period > c.wl_period_max) period = c.wl_period_max;
    if (scal(CYG_S_STEP) % (uint32_t)period != 0) return;
    if (n_active == 0 || 10 * idle < n_active) return; /* _idle_fraction() < 0.10 (volt:580) */
    int nC = 100, nS = 10;
    if (c.scaling_vulnerability) { /* _scaled_numloads (volt:266-293) */
      int req_c = 2 * n_active;
      int req_s = (2 * n_active + 5) / 10;
      if (req_c < 1) req_c = 1;
      if (req_s < 1) req_s = 1;
      int cap_c = free_c > 1 ? free_c : 1, cap_s = free_s > 1 ? free_s : 1;
      nC = req_c < cap_c ? req_c : cap_c;
      nS = req_s < cap_s ? req_s : cap_s;
    }
    if (c.wl_cap > 0) { /* volt:588-593 */
      int total = nC + nS;
      if (total > c.wl_cap) {
        double ratio = (double)c.wl_cap / (double)total;
        nC = (int)(nC * ratio); if (nC < 0) nC = 0;
        nS = (int)(nS * ratio); if (nS < 0) nS = 0;
      }
    }
    Stream ssamp(SITE_WL_SAMPLE), stri(SITE_WL_TRI);
    generate_workloads(nC, false, n_active, ssamp, stri);
    generate_workloads(nS, true, n_active, ssamp, stri);
  }

  /* ---- evolve_network (CyberDefenseEnv.py:583-875) ----
   * Written for a warp of 32 envs in lock step: the Poisson count comes first (half of the envs draw 0 events), the
   * Philox blocks of the three per-event sites are fetched together before the loop, and an event is ONE code path
   * for both kinds (activate / deactivate differ only in the masks they apply), entered only by the lanes whose event
   * acts -- a removal is a no-op while the network sits at its floor size, which is most of them. */
  CYG_HD void evolve_network() {
    const cyg_config& c = n->cfg;
    if (!(scal(CYG_S_FLAGS) & CYG_FL_SETS_INIT)) { /* :654-659 */
      for (int w = 0; w < W; w++) pl(P_ACTSET, w) = m_valid(w) & ~pl(P_NYA, w);
      scal(CYG_S_FLAGS) |= CYG_FL_SETS_INIT;
    }
    Stream sp(SITE_EV_POISSON);
    const uint32_t xp = sp.next(rng); /* :668 */
    int num_events = 0; /* #{j : xp >= tab[j]}; the table is ascending: count over all 16 entries with fixed indices
                           (a walk with a per-thread index serialises the constant-bank loads of a warp) */
    for (int j = 0; j < 16; j++) num_events += (xp >= c.poisson_tab[j]) ? 1 : 0;
    if (num_events > 0) {
      int n_act = count(P_ACTSET);
      const int floor_n = c.num_of_device > c.min_network_size ? c.num_of_device : c.min_network_size;
      Stream sadd(SITE_EV_ADD), spick(SITE_EV_PICK), satt(SITE_EV_ATT);
      sadd.load(rng); spick.load(rng); satt.load(rng);
      for (int ev = 0; ev < num_events; ev++) {
        const bool add = (uint64_t)sadd.next(rng) < c.thr_p_add; /* :679 */
        const int pool_n = add ? n->M - n_act : n_act;
        if (add ? (pool_n > 0) : (n_act > floor_n)) { /* :680-712 */
          uint32_t m[W];
          const uint32_t inv = add ? 0xFFFFFFFFu : 0u; /* the inactive set, or the active one */
          for (int w = 0; w < W; w++) m[w] = m_valid(w) & (pl(P_ACTSET, w) ^ inv);
          const int node = select_nth(m, (int)below(spick.next(rng), (uint32_t)pool_n)); /* :675 */
          const int nw = node >> 5;
          const uint32_t bit = 1u << (node & 31);
          const uint32_t on = add ? bit : 0u, off = add ? 0u : bit;
          pl(P_NYA, nw) = (pl(P_NYA, nw) & ~bit) | off;
          pl(P_ACTSET, nw) = (pl(P_ACTSET, nw) & ~bit) | on;
          n_act += add ? 1 : -1;
          if (add) {
            const uint32_t xt = satt.next(rng); /* :690: the draw is consumed even when p_attacker == 0 */
            if ((uint64_t)xt < c.thr_p_attacker) { pl(P_COMP, nw) |= bit; pl(P_OWNED, nw) |= bit; pl(P_KNOWN, nw) |= bit; }
          } else { /* :701-712: workload dropped, busy_time 0, removed_before */
            pl(P_HASWL, nw) &= ~bit;
            pl(P_PT0, nw) &= ~bit; pl(P_PT0 + 1, nw) &= ~bit; pl(P_PT0 + 2, nw) &= ~bit;
            pl(P_BUSY0, nw) &= ~bit; pl(P_BUSY0 + 1, nw) &= ~bit; pl(P_BUSY0 + 2, nw) &= ~bit; pl(P_BUSY0 + 3, nw) &= ~bit;
#ifdef __CUDA_ARCH__
            atomicOr(&ckpt[node], CYG_CKI_REMOVED); /* removed_before: a RED, nobody waits for the global-memory round trip */
#else
            ckpt[node] |= CYG_CKI_REMOVED;
#endif
          }
        }
      }
    }
    /* bidirectional hub-star among active attacker-owned devices, hub = lowest id (:738-774) */
    int hub = -1;
    uint32_t oa[W];
    for (int w = W - 1; w >= 0; w--) {
      oa[w] = pl(P_OWNED, w) & pl(P_ACTSET, w);
      if (oa[w]) hub = w * 32 + ctz(oa[w]);
    }
    if (hub < 0) return;
    /* the hub's out- and in-neighbours: base rows plus ONE pass over the extra list (global memory: the loads are
     * independent and pipeline) instead of one has_edge() scan per direction and device */
    uint32_t need_out[W], need_in[W];
    uint32_t any = 0;
    {
      uint32_t xo[W], xi[W];
      for (int w = 0; w < W; w++) { xo[w] = 0; xi[w] = 0; }
      const int nx0 = n_extra();
      const uint32_t* x = extra();
      for (int j = 0; j < nx0; j++) {
        const uint32_t xe = x[j];
        const int u = (int)(xe & CYG_X_IDMASK), v = (int)((xe >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
        for (int w = 0; w < W; w++) {
          xo[w] |= (u == hub) ? ((1u << (v & 31)) & eqmask(w, v >> 5)) : 0u;
          xi[w] |= (v == hub) ? ((1u << (u & 31)) & eqmask(w, u >> 5)) : 0u;
        }
      }
      for (int w = 0; w < W; w++) {
        const uint32_t rest = oa[w] & ~((1u << (hub & 31)) & eqmask(w, hub >> 5));
        need_out[w] = rest & ~(adj(hub, w) | xo[w]); /* i lacks hub -> i */
        uint32_t ni = rest & ~xi[w], r = ni;          /* i lacks i -> hub: not an extra edge and not in i's base row */
        while (r) {
          const int b = ctz(r);
          r &= r - 1;
          if ((adj(w * 32 + b, hub >> 5) >> (hub & 31)) & 1u) ni &= ~(1u << b);
        }
        need_in[w] = ni;
        any |= need_out[w] | ni;
      }
    }
    if (any == 0) return; /* the star is complete: the usual case */
    bool changed = false;
    for (int w = 0; w < W; w++) {
      uint32_t rest = need_out[w] | need_in[w];
      while (rest) { /* ascending i; per device hub -> i first, then i -> hub (:752-770) */
        const int b = ctz(rest);
        rest &= rest - 1;
        const int i = w * 32 + b;
        for (int dir = 0; dir < 2; dir++) {
          if (!(((dir ? need_in[w] : need_out[w]) >> b) & 1u)) continue;
          const int u = dir ? i : hub, v = dir ? hub : i;
          int nx = n_extra();
          if (nx >= c.xcap) { scal(CYG_S_FLAGS) |= CYG_FL_ERR_XCAP; continue; }
          extra()[nx] = (uint32_t)u | ((uint32_t)v << CYG_X_V_SHIFT);
          scal(CYG_S_PREV_X) = (scal(CYG_S_PREV_X) & 0xFFFFu) | ((uint32_t)(nx + 1) << 16);
          changed = true;
        }
      }
    }
    /* the preferential-attachment repair (:776-843) needs a degree-0 vertex: build_tables refuses such networks */
    if (changed) rebuild_cache();
  }

  CYG_HD void count_comp(int& n_comp, int& n_comp_dc) { /* _count_comp (volt:563-572) */
    int a = 0, b = 0;
    for (int w = 0; w < W; w++) {
      uint32_t m = pl(P_COMP, w) & ~pl(P_NYA, w) & ~pl(P_OWNED, w);
      a += popc(m);
      b += popc(m & m_dc(w));
    }
    n_comp = a; n_comp_dc = b;
  }

  /* ---- the step (volt_typhoon_env.py:818-1333; grouped: :694-779) ---- */
  /* the action type step() ends up executing: None fill (volt:847-874), clamp into the action space
   * (:879-884), defender forced to the no-op unless base_line == "Nash" (:913-914).  Needs no env state,
   * so the kernel can sort a block's envs by it before their records arrive. */
  CYG_HD static int exec_type(const cyg_config& c, uint32_t h0, int base_line) {
    int at = (int)(h0 & 0xFFu);
    int mode = (int)((h0 >> 8) & 1u);
    int atype = at == (int)CYG_ATYPE_NONE ? -1000 : (int)(int8_t)at;
    if (atype == -1000) {
      if (mode == CYG_MODE_DEFENDER) atype = (base_line == CYG_BL_NO_DEFENSE) ? 8 : 7;
      else atype = (base_line == CYG_BL_NO_ATTACK) ? 3 : 2;
    }
    if (mode == CYG_MODE_DEFENDER) { if (!(atype >= 0 && atype < c.def_space_n)) atype = 8; }
    else { if (!(atype >= 0 && atype < c.att_space_n)) atype = 3; }
    if (mode == CYG_MODE_DEFENDER && base_line != CYG_BL_NASH) atype = 8;
    return atype;
  }

  /* The step in three pieces (the kernel may run the middle one with a whole warp per env):
   * step_pre : open the epoch, resolve the executed action type, busy tick (volt:847-908)
   * step_act : the action(s) (volt:913-1202; grouped: :612-692, :607-610)
   * step_post: work, arrivals, reward, counters, evolve_network (volt:1207-1333) */
  CYG_HD int step_pre(const uint32_t* hdr, uint32_t flags) {
    begin_epoch();
    if (flags & CYG_STEP_GROUPED) return 0;
    int atype = exec_type(n->cfg, hdr[0], bl);
    tick_busyset(); /* volt:904-908 */
    return atype;
  }
  CYG_HD void load_costs() {
    defcost = (double)u2f(scal(CYG_S_DEFCOST));
    cleancost = (double)u2f(scal(CYG_S_CLEANCOST));
  }
  CYG_HD void store_costs() {
    scal(CYG_S_DEFCOST) = f2u((float)defcost);
    scal(CYG_S_CLEANCOST) = f2u((float)cleancost);
  }
  /* the action types the plain-step kernel hands to a whole warp (cyg_coop.cuh) */
  CYG_HD static bool coop_type(int mode, int atype) {
    if (mode == CYG_MODE_ATTACKER) return atype == 1;
    return atype == 1 || atype == 3 || atype == 4;
  }
  /* ... plus block / unblock.  (Measured: the owning thread walking the list itself -- flip_walk, ~135 instructions per
   * listed device, branch-free -- is a ~90k-cycle dependent chain for a 46-device list; the warp-per-env windows of
   * cyg_coop.cuh take ~11k.  profiles/NOTES_r02.md.) */
  CYG_HD bool deferred_type(int mode, int atype) {
    if (mode == CYG_MODE_DEFENDER && (atype == 6 || atype == 9)) return true;
    return coop_type(mode, atype);
  }
  /* LIGHT: a plain (ungrouped, set-form) step whose cooperative types are handled elsewhere -- they return at once
   * here (the only one that can arrive is the attacker's type 1 under base_line "No Attack", a no-op), which lets the
   * compiler drop their thread-per-env code from the kernel that never runs it */
  template <bool LIGHT = false>
  CYG_HD int step_act(const uint32_t* hdr, const uint32_t* mask, const uint16_t* order, size_t hdr_gs, size_t mask_gs,
                      size_t order_gs, int G, uint32_t flags, int atype, double& cost, bool& dirty) {
    const cyg_config& c = n->cfg;
    const bool grouped = LIGHT ? false : (flags & CYG_STEP_GROUPED) != 0;
    if (LIGHT) order = nullptr;
    load_costs();
    Act a;
    decode(hdr, mask, order, a);
    const int mode = a.mode;
    if (LIGHT && deferred_type(mode, atype)) { store_costs(); return atype; }
    if (!grouped) {
      if (a.atype == -1000) { a.n_dev = 0; a.first = -1; a.n_ex = 1; a.exw = 0; a.app_index = 0; }
      if (mode == CYG_MODE_DEFENDER) {
        defender_meta(a, atype, false, cost, dirty);
        if (atype == 1 || atype == 4 || atype == 5 || atype == 6 || atype == 7 || atype == 9 || atype == 12 || atype == 13)
          defender_per_device(a, atype, cost, dirty);
      } else {
        attacker_act(a, atype, cost);
      }
    } else {
      atype = 0;
      for (int g = 0; g < G; g++) { /* _step_apply_only (volt:612-692) */
        Act ga;
        decode(hdr + g * hdr_gs, mask + g * mask_gs, order ? order + g * order_gs : (const uint16_t*)0, ga);
        int gt = ga.atype == -1000 ? 0 : ga.atype;
        if (gt == 0) gt = (mode == CYG_MODE_DEFENDER) ? 8 : 3;
        if (mode == CYG_MODE_DEFENDER) {
          if (bl != CYG_BL_NASH) gt = 8;
          defender_meta(ga, gt, true, cost, dirty);
          if (gt == 1) {
            double ds = (double)c.def_scale;
            if (!ga.order) {
              clean_set(ga, ds, cost);
            } else {
              DevIter it;
              for (int i = 0; i < ga.n_dev; i++) {
                int d = next_dev(ga, it);
                if (d < 0 || d >= n->M) break;
                if (bit(P_NYA, d)) continue;
                clean_device(d, ds, cost);
              }
            }
          }
        }
        atype = gt;
      }
      tick_all(); /* _tick_busy_time_once (volt:607-610) */
    }
    store_costs();
    return atype;
  }
  CYG_HD void step_post(int mode, double cost, bool dirty, uint32_t flags, float* raw_out, float* shaped_out,
                        int32_t* done_out, uint32_t* pre_masks) {
    const cyg_config& c = n->cfg;
    const bool grouped = (flags & CYG_STEP_GROUPED) != 0;
    const bool skip_work = (flags & CYG_STEP_SKIP_WORK) != 0;
    /* work, arrivals, reward, counters, evolve (volt:1207-1333) */
    int cur_work = 0;
    if (!skip_work || grouped) {
      cur_work = workload_advance();
      arrivals_if_due();
    }
    double def_work = (double)c.work_scale * cur_work;
    int n_comp, n_comp_dc;
    count_comp(n_comp, n_comp_dc);
    if (!grouped) scal(CYG_S_COMPCNT) += (uint32_t)n_comp; /* volt:1267-1270; absent from step_grouped */
    double raw, shaped;
    if (mode == CYG_MODE_DEFENDER) {
      raw = cost + def_work - n_comp * (double)c.comp_scale;
      shaped = raw;
    } else {
      raw = cost + (double)c.comp_scale * (n_comp + 10 * n_comp_dc);
      double phi = (double)n_comp * n->inv_M; /* n_comp / len(net): within 1 ulp of the division */
      double gam = (double)c.gamma;
      uint32_t pn = scal(CYG_S_PREV_X) & 0xFFFFu;
      double prev = (pn == 0xFFFFu) ? phi : gam * ((double)pn * n->inv_M);
      double bonus = 0.1 * (gam * phi - prev);
      scal(CYG_S_PREV_X) = (scal(CYG_S_PREV_X) & 0xFFFF0000u) | (uint32_t)n_comp;
      shaped = raw + bonus;
    }
    if (pre_masks) { /* the `state` step() returns is the pre-evolve view (volt:1306) */
      const int Wm = n->Wm;
      for (int w = 0; w < W; w++) {
        if (w >= Wm) break;
        pre_masks[0 * Wm + w] = pl(P_COMP, w);
        pre_masks[1 * Wm + w] = pl(P_KNOWN, w);
        pre_masks[2 * Wm + w] = pl(P_NYA, w);
      }
    }
    if (!skip_work || grouped) {
      scal(CYG_S_STEP)++;
      if (mode == CYG_MODE_ATTACKER) scal(CYG_S_ATT_STEP)++; else scal(CYG_S_DEF_STEP)++;
    }
    int done = scal(CYG_S_STEP) > 1000u; /* _check_done (CyberDefenseEnv.py:547-552) */
    bool periodic = (scal(CYG_S_STEP) % (uint32_t)c.evolve_period) == 0;
    if (dirty || periodic) evolve_network();
    if (!grouped) { /* volt:1330 */
      for (int w = 0; w < W; w++) pl(P_BUSYSET, w) = busy_nz(w);
    }
    *raw_out = (float)raw; *shaped_out = (float)shaped; *done_out = done;
  }

  CYG_HD int step(const uint32_t* hdr, const uint32_t* mask, const uint16_t* order, size_t hdr_gs, size_t mask_gs,
                  size_t order_gs, int G, uint32_t flags, float* raw_out, float* shaped_out, int32_t* done_out,
                  uint32_t* pre_masks) {
    int atype = step_pre(hdr, flags);
    double cost = 0.0;
    bool dirty = false;
    atype = step_act(hdr, mask, order, hdr_gs, mask_gs, order_gs, G, flags, atype, cost, dirty);
    step_post((int)((hdr[0] >> 8) & 1u), cost, dirty, flags, raw_out, shaped_out, done_out, pre_masks);
    return atype;
  }
  CYG_HD void resume_epoch() { /* re-attach to the epoch step_pre opened (the kernel changes threads between pieces) */
    rng.epoch = scal(CYG_S_EPOCH) - 1u;
    stall = Stream(SITE_STALL);
  }

  /* ---- randomize_compromise_and_ownership (volt:330-383) ---- */
  CYG_HD void randomize() {
    begin_epoch();
    uint32_t pool[W];
    int np = 0, k_owned = 0, k_comp = 0;
    for (int w = 0; w < W; w++) {
      uint32_t p = m_valid(w) & ~pl(P_NYA, w) & ~m_dc(w);
      pool[w] = p;
      np += popc(p);
      k_owned += popc(p & pl(P_OWNED, w));
      k_comp += popc(p & pl(P_COMP, w));
    }
    if (np == 0 || (k_owned == 0 && k_comp == 0)) return;
    int extra_c = k_comp - k_owned;
    if (extra_c < 0) extra_c = 0;
    for (int w = 0; w < W; w++) { pl(P_OWNED, w) &= ~pool[w]; pl(P_COMP, w) &= ~pool[w]; pl(P_KNOWN, w) &= ~pool[w]; }
    Stream ss(SITE_SHUFFLE);
    int rem = np;
    for (int j = 0; j < k_owned + extra_c && j < np; j++) { /* shuffle == successive uniform picks */
      int r = rem > 1 ? (int)below(ss.next(rng), (uint32_t)rem) : 0;
      int d = select_nth(pool, r);
      for (int w = 0; w < W; w++) pool[w] &= ~((1u << (d & 31)) & eqmask(w, d >> 5));
      rem--;
      if (j < k_owned) setb(P_OWNED, d);
      setb(P_COMP, d);
      setb(P_KNOWN, d);
    }
  }

  /* ---- sample_action (CyberDefenseEnv.py:555-578): device_indices as a set; the draw order of random.sample is kept
   *      for device_indices[0] (header field) and, when `order` is given, for the whole list ---- */
  CYG_HD void sample_action(int mode, uint32_t* hdr, uint32_t* mask, uint16_t* order = nullptr) {
    const cyg_config& c = n->cfg;
    begin_epoch();
    Stream st(SITE_SA_TYPE), sn(SITE_SA_NDEV), sd(SITE_SA_DEVS), sx(SITE_SA_EXP), sa(SITE_SA_APP);
    int space = mode == CYG_MODE_DEFENDER ? c.def_space_n : c.att_space_n;
    int atype = (int)below(st.next(rng), (uint32_t)space);
    int ndev = 1 + (int)below(sn.next(rng), (uint32_t)c.num_of_device);
    uint32_t pool[W], pick[W];
    for (int w = 0; w < W; w++) { pool[w] = m_valid(w); pick[w] = 0; }
    int rem = n->M, first = 0;
    for (int j = 0; j < ndev; j++) {
      int d = select_nth(pool, (int)below(sd.next(rng), (uint32_t)rem));
      for (int w = 0; w < W; w++) { uint32_t bw = (1u << (d & 31)) & eqmask(w, d >> 5); pool[w] &= ~bw; pick[w] |= bw; }
      rem--;
      if (order) order[j] = (uint16_t)d;
      first = j == 0 ? d : first;
    }
    int ex = (int)below(sx.next(rng), (uint32_t)c.X);
    int app = c.n_app_ids > 0 ? (int)below(sa.next(rng), (uint32_t)c.n_app_ids) : 0;
    hdr[0] = (uint32_t)(atype & 0xFF) | ((uint32_t)mode << 8) | (1u << 16);
    hdr[1] = (uint32_t)(ex & 0xFF);
    hdr[2] = (uint32_t)ndev | ((uint32_t)(first + 1) << 16); /* device_indices[0] = the first device drawn */
    hdr[3] = (uint32_t)app;
    for (int w = 0; w < W; w++) if (w < n->Wm) mask[w] = pick[w];
  }
};

template <int W, int SM>
CYG_HDN uint32_t scan_trained_call(const Net* n, uint32_t* rec, uint32_t ro, uint32_t to, uint32_t* logs, const uint32_t* det, uint32_t env_id,
                                   uint32_t stall_k, int reps) {
  Env<W, SM> e(n, rec, nullptr, nullptr, env_id, ro, to);
  e.logs = logs;
  e.det = det;
  e.resume_epoch();
  e.stall.k = stall_k;
  e.scan_trained_body(reps);
  return e.stall.k;
}

/* ---- canonical device word <-> bit-planes (include/cygym_b200.h) ------------ */
template <int W>
CYG_HD void import_device(const Net* n, uint32_t* rec, int d, uint32_t w) {
  uint32_t m = 1u << (d & 31);
  int wi = d >> 5;
  uint32_t* pl = rec + CYG_REC_PLANES;
  auto put = [&](int p, bool v) { if (v) pl[p * W + wi] |= m; else pl[p * W + wi] &= ~m; };
  put(P_COMP, w & CYG_DEV_COMP); put(P_KNOWN, w & CYG_DEV_KNOWN); put(P_NYA, w & CYG_DEV_NYA);
  put(P_OWNED, w & CYG_DEV_OWNED); put(P_HASWL, w & CYG_DEV_HASWL);
  put(P_BUSYSET, w & CYG_DEV_BUSYSET); put(P_ACTSET, w & CYG_DEV_ACTSET);
  uint32_t pt = (w >> CYG_DEV_PT_SHIFT) & CYG_DEV_PT_MASK;
  for (int k = 0; k < 3; k++) put(P_PT0 + k, (pt >> k) & 1u);
  uint32_t b = (w >> CYG_DEV_BUSY_SHIFT) & CYG_DEV_BUSY_MASK;
  if (b > CYG_BUSY_MAX) { b = CYG_BUSY_MAX; rec[CYG_S_FLAGS] |= CYG_FL_ERR_BUSY; }
  for (int k = 0; k < 4; k++) put(P_BUSY0 + k, (b >> k) & 1u);
  uint32_t cb = (w >> CYG_DEV_CBY_SHIFT) & CYG_DEV_CBY_MASK;
  for (int k = 0; k < n->ncby; k++) put(P_CBY0 + k, (cb >> k) & 1u);
}
template <int W>
CYG_HD uint32_t export_device(const Net* n, const uint32_t* rec, int d, uint32_t ckpt_internal) {
  int wi = d >> 5, s = d & 31;
  const uint32_t* pl = rec + CYG_REC_PLANES;
  auto get = [&](int p) -> uint32_t { return (pl[p * W + wi] >> s) & 1u; };
  uint32_t w = 0;
  if (get(P_COMP)) w |= CYG_DEV_COMP;
  if (get(P_KNOWN)) w |= CYG_DEV_KNOWN;
  if (get(P_NYA)) w |= CYG_DEV_NYA;
  if (get(P_OWNED)) w |= CYG_DEV_OWNED;
  if (ckpt_internal & CYG_CKI_REMOVED) w |= CYG_DEV_REMOVED;
  if (get(P_HASWL)) w |= CYG_DEV_HASWL;
  if (get(P_BUSYSET)) w |= CYG_DEV_BUSYSET;
  if (get(P_ACTSET)) w |= CYG_DEV_ACTSET;
  for (int k = 0; k < 3; k++) w |= get(P_PT0 + k) << (CYG_DEV_PT_SHIFT + k);
  for (int k = 0; k < 4; k++) w |= get(P_BUSY0 + k) << (CYG_DEV_BUSY_SHIFT + k);
  for (int k = 0; k < n->ncby; k++) w |= get(P_CBY0 + k) << (CYG_DEV_CBY_SHIFT + k);
  return w;
}

/* canonical blocked[] (bit e = base pair e, out-list pair order; include/cygym_b200.h) <-> the unit bitset of a record.
 * set_units: the word / mask pairs a blocked pair e sets (2 m bits: its run in the source's out list and the twin run in
 * the target's in list); `put(word_index, mask)` is the caller's store (plain on the host, atomicOr in the import kernel) */
template <class Put>
CYG_HD void pair_units(const Net* n, int e, Put put) {
  const int q = (int)n->blob[n->o_pair2unit + e];
  const uint32_t ui = n->blob[n->o_unit + q];
  const int t = unit_twin(ui), m = unit_m(ui);
  for (int k = 0; k < m; k++) { put((q + k) >> 5, 1u << ((q + k) & 31)); put((t + k) >> 5, 1u << ((t + k) & 31)); }
}
CYG_HD bool pair_blocked(const Net* n, const uint32_t* rec, int e) {
  const int q = (int)n->blob[n->o_pair2unit + e];
  return (rec[n->off_inc + (q >> 5)] >> (q & 31)) & 1u;
}

/* one element of an observation row (CyberDefenseEnv.py:146-257); obs_mode as in cyg_step_out */
template <int W>
CYG_HD float observe_elem(const Net* n, const uint32_t* rec, int obs_mode, int j) {
  int M = n->M;
  const uint32_t* pl = rec + CYG_REC_PLANES;
  if (obs_mode == 2) {
    if (j >= 4 * M) return (j - 4 * M) < n->cfg.n_exploits ? 1.f : 0.f;
    int d = j >> 2, k = j & 3, wi = d >> 5, s = d & 31;
    bool known = (pl[P_KNOWN * W + wi] >> s) & 1u, nya = (pl[P_NYA * W + wi] >> s) & 1u, owned = (pl[P_OWNED * W + wi] >> s) & 1u;
    if (!known || nya || !owned) return -1.f;
    if (k == 0) return ((const float*)(n->blob + n->o_os))[d];
    if (k == 1) return ((const float*)(n->blob + n->o_ver))[d];
    if (k == 2) return ((pl[P_COMP * W + wi] >> s) & 1u) ? 1.f : 0.f;
    return 1.f; /* known */
  }
  int d = j / 6, k = j - 6 * d, wi = d >> 5, s = d & 31;
  bool known = (pl[P_KNOWN * W + wi] >> s) & 1u, nya = (pl[P_NYA * W + wi] >> s) & 1u, owned = (pl[P_OWNED * W + wi] >> s) & 1u;
  bool comp = (pl[P_COMP * W + wi] >> s) & 1u;
  if (obs_mode == 1 && (nya || !owned)) return -1.f;
  switch (k) {
    case 0: return ((const float*)(n->blob + n->o_os))[d];
    case 1: return ((const float*)(n->blob + n->o_ver))[d];
    case 2: return obs_mode == 1 ? -1.f : (comp ? 1.f : 0.f);
    case 3: return 0.f; /* anomaly_score stays 0 under fast_scan (volt:46) */
    case 4: return known ? 1.f : 0.f;
    default: return nya ? 1.f : 0.f;
  }
}

}  // namespace cyg
#endif /* CYG_CORE_CUH */
