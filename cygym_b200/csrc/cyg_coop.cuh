/*
 * cyg_coop.cuh -- warp-per-env forms of the draw-heavy defender actions (device only).
 *
 * Thread-per-env is the right mapping for the word-wide parts of a step, but four defender actions walk the
 * listed devices one by one, each with its own random draw: clean (volt_typhoon_env.py:996-1011), revert
 * (:928-943), upgrade (:1013-1018) and block / unblock (:1071-1100 -> :485-511).  One thread doing that for ~90
 * devices is a ~10^5-cycle dependent chain that the rest of the CTA waits for.  Here a whole warp takes ONE env
 * and its 32 lanes take 32 consecutive listed devices.
 *
 * Draws are addressable (oracle/draws.py: x = Philox(seed; env, epoch, site, k)), so lane i simply computes the
 * draw of ITS device, k = (draws consumed so far) + (rank of the device among those that draw).
 *
 *  - clean / revert / upgrade: every listed device draws, nothing a device does depends on another device, so
 *    the result is one ballot per busy_time bit-plane.
 *  - block / unblock is sequential in the reference: the pool of device i (its incident edges with the wanted
 *    blocked flag) shrinks when an EARLIER device flips an edge that also touches i.  The lanes pick
 *    speculatively against the state at the start of the round; a pick is invalid only if a lower lane picked an
 *    edge whose far endpoint is that lane's device.  The round commits the lanes below the first such lane and
 *    restarts from it, so the outcome is bit-identical to the sequential walk.
 *
 * All lanes call these functions with identical arguments; only lane 0 touches per-env scalars and cost sums.
 */
#ifndef CYG_COOP_CUH
#define CYG_COOP_CUH

#include "cyg_core.cuh"

namespace cyg {

#define CYG_FULL 0xFFFFFFFFu

__device__ __forceinline__ int lane_id() { return (int)(threadIdx.x & 31u); }
__device__ __forceinline__ uint32_t lanes_below(int lane) { return (1u << lane) - 1u; }

/* k-th draw of `site` in the current epoch */
__device__ __forceinline__ uint32_t draw_at(const Rng& r, int site, uint32_t k) {
  uint32_t o[4];
  philox4x32_10(r.env, r.epoch, (uint32_t)site, k >> 2, r.k0, r.k1, o);
  uint32_t j = k & 3u;
  return j == 0 ? o[0] : j == 1 ? o[1] : j == 2 ? o[2] : o[3];
}

template <bool V> struct HasX { static constexpr bool value = V; };

template <int W>
struct Coop {
  typedef Env<W, 1> E;

  /* busy_time = low + below(draw, range) for the devices of A[] (lane-uniform), draws k_base, k_base+1, ... in
   * ascending device order (the set form of _stall, volt:135-138) */
  static __device__ __forceinline__ void deposit(E& e, const uint32_t* A, int low, int high, uint32_t k_base) {
    const int lane = lane_id();
    const uint32_t range = (uint32_t)(high - low + 1);
    uint32_t kw = k_base;
    bool over = false;
    /* one Philox block per lane = draws [4 (k_base/4 + lane), +4): 128 draws cover every device of a W <= 4 env, so a
     * device fetches its draw from lane (k - k_base_aligned) / 4 by shuffle instead of running its own Philox */
    uint32_t blk[4];
    philox4x32_10(e.rng.env, e.rng.epoch, (uint32_t)SITE_STALL, (k_base >> 2) + (uint32_t)lane, e.rng.k0, e.rng.k1, blk);
    const uint32_t k_al = k_base & ~3u;
#pragma unroll
    for (int w = 0; w < W; w++) {
      const uint32_t aw = A[w];
      if (aw == 0) continue; /* uniform */
      const bool on = ((aw >> lane) & 1u) != 0;
      const uint32_t k = kw + (uint32_t)popc(aw & lanes_below(lane));
      const uint32_t rel = k - k_al; /* < 128 + 3 */
      const int from = (int)(rel >> 2) & 31;
      const uint32_t x0 = __shfl_sync(CYG_FULL, blk[0], from), x1 = __shfl_sync(CYG_FULL, blk[1], from);
      const uint32_t x2 = __shfl_sync(CYG_FULL, blk[2], from), x3 = __shfl_sync(CYG_FULL, blk[3], from);
      const uint32_t j = rel & 3u;
      uint32_t x = j == 0 ? x0 : j == 1 ? x1 : j == 2 ? x2 : x3;
      uint32_t v = 0;
      if (on) {
        if (rel >= 128u) x = draw_at(e.rng, SITE_STALL, k); /* only when k_base is not a multiple of 4 */
        v = (uint32_t)low + below(x, range);
        if (v > CYG_BUSY_MAX) { v = CYG_BUSY_MAX; over = true; }
      }
      const uint32_t r0 = __ballot_sync(CYG_FULL, v & 1u), r1 = __ballot_sync(CYG_FULL, v & 2u);
      const uint32_t r2 = __ballot_sync(CYG_FULL, v & 4u), r3 = __ballot_sync(CYG_FULL, v & 8u);
      if (lane == 0) {
        const uint32_t keep = ~aw;
        e.pl(P_BUSY0, w) = (e.pl(P_BUSY0, w) & keep) | r0;
        e.pl(P_BUSY0 + 1, w) = (e.pl(P_BUSY0 + 1, w) & keep) | r1;
        e.pl(P_BUSY0 + 2, w) = (e.pl(P_BUSY0 + 2, w) & keep) | r2;
        e.pl(P_BUSY0 + 3, w) = (e.pl(P_BUSY0 + 3, w) & keep) | r3;
      }
      kw += (uint32_t)popc(aw);
    }
    if (__any_sync(CYG_FULL, over) && lane == 0) e.scal(CYG_S_FLAGS) |= CYG_FL_ERR_BUSY;
    __syncwarp();
  }

  /* block (6) / unblock (9) one incident edge per listed active device, in listed order (volt:1071-1100 -> :485-511).
   *
   * The pool of a device is the window [ip[d], ip[d+1]) of the unit bitset (cyg_core.cuh): weight = popcount, pick =
   * select.  Devices with at most 32 incident units -- all but the few star centres -- hold their window in ONE
   * register, and a run of up to 32 consecutive listed devices of that kind is a WINDOW of lanes: lane i speculates the
   * pick of its device on the state at the start of the window; a pick is wrong only if a LOWER lane flips an edge
   * that ends at this lane's device (that edge leaves the pool).  Each pass tells every lane which lower lanes
   * currently do that ("attackers"), the lane drops those edges from its start-of-window pool and picks again; the
   * picks are a function of the lower lanes' picks only, so the pass where nothing changes is the sequential walk's
   * outcome and all flips commit at once.  A device with more than 32 units ends the window and is done alone, exactly,
   * by the whole warp (lane l holds word l of its window).  The draw index of a device = draws consumed + non-empty
   * pools in front of it; lane l computed Philox block l of the site once per task, draws are fetched by shuffle.
   *
   * Envs with extra (hub-star) edges keep those in the per-env list (lane j holds extra j): an extra edge sits in its
   * endpoint's out / in list at its place in ascending neighbour order, so its index in the pool = pool units in front
   * of that place + pool extras with a smaller far endpoint; a pick that lands on such an index takes the extra edge,
   * the picks behind it shift by one. */
  template <int G>
  static __device__ __forceinline__ void flip(E& e, const typename E::Act& a, int atype, double& cost, bool& dirty) {
    const int lane = lane_id();
    const bool want = atype == 9;
    const int site = want ? SITE_UNBLOCK : SITE_BLOCK;
    const uint32_t flipw = want ? 0u : 0xFFFFFFFFu; /* pool bits = blocked bits XOR flipw */
    const double ds = (double)e.n->cfg.def_scale;
    uint32_t act[W];
    const int na = e.listed_active(a, act);
    if (na == 0) return;
    if (lane == 0) { cost += -0.5 * ds * na; e.defcost += 0.5 * ds * na; }
    const int nx = e.n_extra();
    uint32_t cnt = 0;
    if (nx > 32) { /* more extra edges than lanes: the sequential form, one lane (rare: many attacker arrivals) */
      if (lane == 0) {
        Stream st(site);
        for (;;) {
          const int d = e.pop_lowest(act);
          if (d < 0) break;
          if (e.flip_incident(d, want, st)) cnt++;
        }
      }
      cnt = __shfl_sync(CYG_FULL, cnt, 0);
    } else {
      uint32_t* const bits = e.inc();
      /* the env's extra edges: lane j holds extra j */
      uint32_t xe = 0;
      if (lane < nx) xe = e.extra()[lane];
      const int xu = (int)(xe & CYG_X_IDMASK), xv = (int)((xe >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
      uint32_t xflags = __ballot_sync(CYG_FULL, (xe & CYG_X_BLOCKED) != 0); /* bit j: extra j is blocked */
      uint32_t lto = 0, lti = 0; /* bit k: extra k has my source and a smaller target / my target and a smaller source */
      int xpo = 0, xpi = 0;      /* units of xu's out list in front of xv / of xv's in list in front of xu */
      for (int k = 0; k < nx; k++) { /* uniform */
        const int ku = __shfl_sync(CYG_FULL, xu, k), kv = __shfl_sync(CYG_FULL, xv, k);
        lto |= (ku == xu && kv < xv) ? (1u << k) : 0u;
        lti |= (kv == xv && ku < xu) ? (1u << k) : 0u;
      }
      if (lane < nx) { xpo = e.units_before_out(xu, xv); xpi = e.units_before_in(xv, xu); }
      /* draws of the site: lane l holds Philox block l = draws 4 l .. 4 l + 3 (a W <= 4 env lists at most 128 devices) */
      uint32_t blk[4];
      philox4x32_10(e.rng.env, e.rng.epoch, (uint32_t)site, (uint32_t)lane, e.rng.k0, e.rng.k1, blk);
      auto draw = [&](uint32_t k) -> uint32_t {
        const int from = (int)(k >> 2) & 31;
        const uint32_t x0 = __shfl_sync(CYG_FULL, blk[0], from), x1 = __shfl_sync(CYG_FULL, blk[1], from);
        const uint32_t x2 = __shfl_sync(CYG_FULL, blk[2], from), x3 = __shfl_sync(CYG_FULL, blk[3], from);
        const uint32_t j = k & 3u;
        return j == 0 ? x0 : j == 1 ? x1 : j == 2 ? x2 : x3;
      };
      int pos = 0;
      uint32_t kbase = 0;
      while (pos < na) { /* uniform */
        const int idx = pos + lane;
        const bool valid0 = idx < na;
        const int d = valid0 ? e.select_nth(act, idx) : 0;
        const uint32_t di = e.dinfo(d), di1 = e.dinfo(d + 1);
        const int a0 = (int)(di & 0xFFFFu), no = (int)(di >> 16), nt = (int)(di1 & 0xFFFFu) - a0;
        const uint32_t bigm = __ballot_sync(CYG_FULL, valid0 && nt > 128);
        if (bigm & 1u) {
          /* ---- the device at `pos` has more than 128 units: alone, exactly, lane l on word l of its window ---- */
          const int d0 = __shfl_sync(CYG_FULL, d, 0), ab = __shfl_sync(CYG_FULL, a0, 0);
          const int nob = __shfl_sync(CYG_FULL, no, 0), ntb = __shfl_sync(CYG_FULL, nt, 0);
          uint32_t hx = 0;
          if (32 * lane < ntb) {
            const int q0 = ab + 32 * lane;
            hx = (funnel_r(bits[q0 >> 5], bits[(q0 >> 5) + 1], q0 & 31) ^ flipw) & lowmask0(ntb - 32 * lane);
          }
          uint32_t imo = 0, imi = 0;
          for (int j = 0; j < nx; j++) {
            const int ju = __shfl_sync(CYG_FULL, xu, j), jv = __shfl_sync(CYG_FULL, xv, j);
            const bool memb = (((xflags >> j) & 1u) != 0) == want;
            imo |= (memb && ju == d0) ? (1u << j) : 0u;
            imi |= (memb && jv == d0) ? (1u << j) : 0u;
          }
          const int pc = popc(hx);
          const int tot = (int)__reduce_add_sync(CYG_FULL, (uint32_t)pc) + popc(imo) + popc(imi);
          if (tot > 0) { /* uniform */
            const int r = (int)below(draw(kbase), (uint32_t)tot);
            int sel = -1, passed = 0;
            for (int j = 0; j < nx; j++) { /* uniform: imo / imi are */
              const bool bo = (imo >> j) & 1u, bi = (imi >> j) & 1u;
              if (!(bo | bi)) continue;
              const int P = bo ? __shfl_sync(CYG_FULL, xpo, j) : nob + __shfl_sync(CYG_FULL, xpi, j);
              const int cb = (int)__reduce_add_sync(CYG_FULL, (uint32_t)popc(hx & lowmask0(P - 32 * lane)));
              const uint32_t lo_j = __shfl_sync(CYG_FULL, lto, j), li_j = __shfl_sync(CYG_FULL, lti, j);
              const int mi = cb + (bo ? popc(imo & lo_j) : popc(imo) + popc(imi & li_j));
              if (mi == r) sel = j;
              passed += mi < r ? 1 : 0;
            }
            if (sel >= 0) {
              if (lane == 0) { if (want) e.extra()[sel] &= ~CYG_X_BLOCKED; else e.extra()[sel] |= CYG_X_BLOCKED; }
              xflags = want ? (xflags & ~(1u << sel)) : (xflags | (1u << sel));
            } else {
              const int rr = r - passed;
              int incl = pc;
#pragma unroll
              for (int dd = 1; dd < 32; dd <<= 1) {
                const int y = __shfl_up_sync(CYG_FULL, incl, dd);
                if (lane >= dd) incl += y;
              }
              const int excl = incl - pc;
              const bool mine = rr >= excl && rr < incl;
              int q = mine ? ab + 32 * lane + select_in_word(hx, rr - excl) : 0;
              const uint32_t mm = __ballot_sync(CYG_FULL, mine);
              q = __shfl_sync(CYG_FULL, q, __ffs((int)mm) - 1);
              if (lane == 0) e.set_pair_blocked(q, !want);
            }
            cnt++; kbase++;
          }
          pos += 1;
          __threadfence_block();
          __syncwarp();
          continue;
        }
        /* ---- a window of lanes: the listed devices up to the next big one ---- */
        const int c = bigm ? (__ffs((int)bigm) - 1) : 32;
        const bool valid = valid0 && lane < c;
        const int nwin = min(c, na - pos);
        uint32_t x0[4] = {0u, 0u, 0u, 0u}; /* the pool window of my device at the start of the window of lanes (up to 128 units) */
        if (valid) {
          const int wa = a0 >> 5, sh = a0 & 31;
          uint32_t lo = bits[wa];
#pragma unroll
          for (int i = 0; i < 4; i++) { /* whatever follows the bitset in shared memory is readable and masked off */
            const uint32_t hi = bits[wa + i + 1];
            x0[i] = (funnel_r(lo, hi, sh) ^ flipw) & lowmask0(nt - 32 * i);
            lo = hi;
          }
        }
        uint32_t imo0 = 0, imi0 = 0; /* bit j: extra j is in the pool of my out list / in list at the start of the window */
        for (int j = 0; j < nx; j++) {
          const int ju = __shfl_sync(CYG_FULL, xu, j), jv = __shfl_sync(CYG_FULL, xv, j);
          const bool memb = valid && ((((xflags >> j) & 1u) != 0) == want);
          imo0 |= (memb && ju == d) ? (1u << j) : 0u;
          imi0 |= (memb && jv == d) ? (1u << j) : 0u;
        }
        const uint32_t xd = draw(kbase + (uint32_t)lane);
        uint32_t x[4] = {x0[0], x0[1], x0[2], x0[3]}, imo = imo0, imi = imi0;
        int key = -2;  /* the pick: run start unit of a base pair, 0x10000 | j for extra edge j, -1 none */
        int tw = 0, mrun = 1;
        uint32_t nem = 0;
        bool had_att = false; /* some lane's pool of the current pass had edges removed (uniform) */
        /* the fixed-point passes, compiled twice: for envs without extra edges (every env of a fresh network) nothing of the
         * extra-edge bookkeeping is in the loop, for envs with extras all of it is */
        auto passes = [&](auto has_x) {
        constexpr bool HX = decltype(has_x)::value;
        for (;;) {
          const int c0 = popc(x[0]), c1 = popc(x[1]), c2 = popc(x[2]), c3 = popc(x[3]);
          const int tot = c0 + c1 + c2 + c3 + (HX ? popc(imo) + popc(imi) : 0);
          nem = __ballot_sync(CYG_FULL, tot > 0);
          const uint32_t xr = __shfl_sync(CYG_FULL, xd, popc(nem & lanes_below(lane)));
          int nkey = -1, other = -1, ntw = 0, nm = 1;
          const int r = tot > 0 ? (int)below(xr, (uint32_t)tot) : 0;
          int sel = -1, passed = 0;
          /* only the extras that sit in SOME lane's pool matter (with the hub outside the window that is a third of them) */
          uint32_t rel = HX ? __reduce_or_sync(CYG_FULL, imo | imi) : 0u;
          while (rel) { /* uniform: does r land on an extra edge, how many extras sit in front of it */
            const int j = __ffs((int)rel) - 1;
            rel &= rel - 1u;
            const int po_j = __shfl_sync(CYG_FULL, xpo, j), pi_j = __shfl_sync(CYG_FULL, xpi, j);
            const uint32_t lo_j = __shfl_sync(CYG_FULL, lto, j), li_j = __shfl_sync(CYG_FULL, lti, j);
            const int ju = __shfl_sync(CYG_FULL, xu, j), jv = __shfl_sync(CYG_FULL, xv, j);
            const bool bo = (imo >> j) & 1u, bi = (imi >> j) & 1u;
            if (bo | bi) {
              const int P = bo ? po_j : no + pi_j;
              const int mi = popc(x[0] & lowmask0(P)) + popc(x[1] & lowmask0(P - 32)) + popc(x[2] & lowmask0(P - 64)) + popc(x[3] & lowmask0(P - 96)) +
                             (bo ? popc(imo & lo_j) : popc(imo) + popc(imi & li_j));
              if (mi == r) { sel = j; other = bo ? jv : ju; }
              passed += mi < r ? 1 : 0;
            }
          }
          if (tot > 0) {
            if (HX && sel >= 0) {
              nkey = 0x10000 | sel;
            } else {
              const int rr = r - passed; /* word holding unit rr of the window, branch-free */
              const bool g1 = rr >= c0, g2 = rr >= c0 + c1, g3 = rr >= c0 + c1 + c2;
              const uint32_t xw = g3 ? x[3] : g2 ? x[2] : g1 ? x[1] : x[0];
              const int base = g3 ? c0 + c1 + c2 : g2 ? c0 + c1 : g1 ? c0 : 0;
              const int q = a0 + 32 * ((g1 ? 1 : 0) + (g2 ? 1 : 0) + (g3 ? 1 : 0)) + select_in_word(xw, rr - base);
              const uint32_t ui = e.unit(q);
              nkey = q - unit_off(ui);
              ntw = unit_twin(ui); nm = unit_m(ui); other = unit_other(ui);
            }
          }
          const bool changed = __any_sync(CYG_FULL, nkey != key);
          key = nkey; tw = ntw; mrun = nm;
          if (!changed) break;
          /* victim of this lane's pick: the lane (above this one) whose device is the far endpoint */
          int vl = -1;
          if (nkey >= 0) {
            const int ow = other >> 5;
            const uint32_t ob = 1u << (other & 31);
            uint32_t in = 0;
            int rank = 0;
#pragma unroll
            for (int w = 0; w < W; w++) {
              in |= act[w] & ob & eqmask(w, ow);
              rank += popc(act[w] & (w < ow ? 0xFFFFFFFFu : (ob - 1u) & eqmask(w, ow)));
            }
            const int l = rank - pos;
            if (in != 0 && l > lane && l < nwin) vl = l;
          }
          const uint32_t bv = __ballot_sync(CYG_FULL, vl >= 0);
          if (bv == 0 && !had_att) break; /* nobody is touched and the picks came from untouched pools: final */
          uint32_t att = bv;
#pragma unroll
          for (int k = 0; k < 5; k++) {
            const uint32_t bk = __ballot_sync(CYG_FULL, vl >= 0 && ((vl >> k) & 1));
            att &= ((lane >> k) & 1) ? bk : ~bk;
          }
          had_att = bv != 0;
          x[0] = x0[0]; x[1] = x0[1]; x[2] = x0[2]; x[3] = x0[3];
          if (HX) { imo = imo0; imi = imi0; }
          while (__any_sync(CYG_FULL, att != 0)) {
            const int from = att ? (__ffs((int)att) - 1) : lane;
            const int kj = __shfl_sync(CYG_FULL, key, from);
            const int tj = __shfl_sync(CYG_FULL, tw, from), mj = __shfl_sync(CYG_FULL, mrun, from);
            if (att) {
              if (HX && (kj & 0x10000)) { imo &= ~(1u << (kj & 31)); imi &= ~(1u << (kj & 31)); }
              else { /* the run [tj, tj + mj) of my window: at most one word boundary */
                const int pp = tj - a0, sh = pp & 31;
                const uint32_t m0 = lowmask(mj) << sh, m1 = sh + mj > 32 ? lowmask(mj) >> (32 - sh) : 0u;
#pragma unroll
                for (int i = 0; i < 4; i++) x[i] &= ~((m0 & eqmask(i, pp >> 5)) | (m1 & eqmask(i, (pp >> 5) + 1)));
              }
              att &= att - 1u;
            }
          }
        }
        };
        if (nx) passes(HasX<true>{}); else passes(HasX<false>{}); /* uniform */
        /* commit: every lane's pick is final */
        const bool pick_x = key >= 0 && (key & 0x10000) != 0, pick_b = key >= 0 && !pick_x;
        if (pick_b) {
          for (int k = 0; k < mrun; k++) {
            const int q0 = key + k, q1 = tw + k;
            if (!want) { atomicOr(&bits[q0 >> 5], 1u << (q0 & 31)); atomicOr(&bits[q1 >> 5], 1u << (q1 & 31)); }
            else { atomicAnd(&bits[q0 >> 5], ~(1u << (q0 & 31))); atomicAnd(&bits[q1 >> 5], ~(1u << (q1 & 31))); }
          }
        }
        if (pick_x) {
          uint32_t* xp = e.extra() + (key & 0xFFFF);
          if (!want) atomicOr(xp, CYG_X_BLOCKED); else atomicAnd(xp, ~CYG_X_BLOCKED);
        }
        const uint32_t xpicked = __reduce_or_sync(CYG_FULL, pick_x ? (1u << (key & 31)) : 0u);
        xflags = want ? (xflags & ~xpicked) : (xflags | xpicked);
        const uint32_t nbase = (uint32_t)popc(__ballot_sync(CYG_FULL, pick_b));
        if (lane == 0) { if (want) e.nblk() -= nbase; else e.nblk() += nbase; }
        const uint32_t done = (uint32_t)popc(nem);
        cnt += done; kbase += done; pos += nwin;
        __threadfence_block();
        __syncwarp();
      }
    }
    if (lane == 0 && cnt) {
      e.scal(want ? CYG_S_EADD : CYG_S_EBLK) += cnt;
      dirty = true;
    }
    __syncwarp();
  }

  /* attacker action 1, exploit + lateral movement (volt:1126-1185), one warp per env: the 32 lanes take 32
   * consecutive sources of the snapshot.  A source's scan depends on earlier sources only through isCompromised
   * of its own hit (a "not yet compromised" hit is invalid if a lower lane hit the same device), so a round
   * commits the lanes below the first such lane and restarts from it: bit-identical to the sequential loop. */
  template <bool LOG = true>
  static __device__ __forceinline__ void attack(E& e, const typename E::Act& a) {
    const int lane = lane_id();
    uint32_t src[W];
    int ns = 0;
#pragma unroll
    for (int w = 0; w < W; w++) { src[w] = e.pl(P_COMP, w) | e.pl(P_OWNED, w); ns += popc(src[w]); }
    const bool has_blk = e.any_blocked();
    const int nx = e.n_extra();
    /* the env's extra (hub-star) edges (every env after randomize_compromise_and_ownership moved the owned set): lane j
     * holds extra j; a source's unblocked extra out-neighbours join its candidates as an id-space bit row */
    uint32_t xe = 0;
    if (nx <= 32 && lane < nx) xe = e.extra()[lane];
    __syncwarp();
    uint32_t logs_add = 0, zk = 0;
    uint32_t log_base = e.scal(CYG_S_LOGS); /* hop-log index of the next record (uniform; only used with a log ring) */
    const bool logging = LOG && e.logs != nullptr;
    for (int xi = 0; xi < a.n_ex; xi++) { /* uniform */
      int raw = a.ex(xi);
      uint32_t zx = 0;
      if (e.needs_zday_draw(raw)) zx = draw_at(e.rng, SITE_ZDAY, zk++);
      raw = e.resolve_exploit(raw, zx);
      if (raw < 0) continue;
      uint32_t kv[W];
#pragma unroll
      for (int w = 0; w < W; w++) kv[w] = e.pl(P_KNOWN, w) & e.m_vuln(raw, w);
      /* the rounds, compiled twice: without extra edges (every env of a fresh network) no candidate row of extras exists */
      auto rounds = [&](auto has_x) {
      constexpr bool HX = decltype(has_x)::value;
      int pos = 0;
      while (pos < ns) { /* uniform */
        const int idx = pos + lane;
        const bool valid = idx < ns;
        const int s = valid ? e.select_nth(src, idx) : 0;
        uint32_t comp[W], xrow[W];
#pragma unroll
        for (int w = 0; w < W; w++) { comp[w] = e.pl(P_COMP, w); xrow[w] = 0; }
        if (!HX) {
        } else if (nx > 32) {
          if (valid) e.extra_out_row(s, false, xrow);
        } else {
          for (int j = 0; j < nx; j++) { /* uniform */
            const uint32_t jw = __shfl_sync(CYG_FULL, xe, j);
            const int jv = (int)((jw >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
            const bool mine = valid && (int)(jw & CYG_X_IDMASK) == s && !(jw & CYG_X_BLOCKED);
#pragma unroll
            for (int w = 0; w < W; w++) xrow[w] |= mine ? ((1u << (jv & 31)) & eqmask(w, jv >> 5)) : 0u;
          }
        }
        int cnt = 0, v = -1;
        bool rule3 = false;
        if (valid) v = e.attack_source(s, comp, kv, has_blk, HX ? xrow : (const uint32_t*)nullptr, cnt, rule3);
        const uint32_t same = __match_any_sync(CYG_FULL, v >= 0 ? v : (0x1000 + lane));
        const bool conflict = valid && rule3 && (same & lanes_below(lane)) != 0;
        const uint32_t conf = __ballot_sync(CYG_FULL, conflict);
        int c = conf ? (__ffs((int)conf) - 1) : 32;
        if (c > ns - pos) c = ns - pos;
        if (logging) { /* uniform: the committed lanes write their hops, in source order, into the ring */
          const uint32_t nrec = (valid && lane < c) ? (uint32_t)cnt + (v >= 0 ? 1u : 0u) : 0u;
          uint32_t incl = nrec;
#pragma unroll
          for (int dd = 1; dd < 32; dd <<= 1) {
            const uint32_t y = __shfl_up_sync(CYG_FULL, incl, dd);
            if (lane >= dd) incl += y;
          }
          const uint32_t tot = __shfl_sync(CYG_FULL, incl, 31), cap = (uint32_t)e.n->cfg.log_cap;
          const uint32_t end = log_base + tot;
          if (nrec) e.log_source(s, v, has_blk, HX ? xrow : (const uint32_t*)nullptr, log_base + incl - nrec, end > cap ? end - cap : 0u);
          log_base = end;
        }
        if (valid && lane < c) {
          logs_add += (uint32_t)cnt + (v >= 0 ? 1u : 0u);
          if (v >= 0) {
            atomicOr(&e.pl(P_COMP, v >> 5), 1u << (v & 31));
            if (e.devbit(e.n->o_dc, s)) atomicOr(&e.pl(P_CBY0 + raw, v >> 5), 1u << (v & 31));
          }
        }
        pos += c;
        __syncwarp();
      }
      };
      if (nx) rounds(HasX<true>{}); else rounds(HasX<false>{}); /* uniform */
    }
    logs_add = __reduce_add_sync(CYG_FULL, logs_add);
    if (lane == 0) e.scal(CYG_S_LOGS) += logs_add;
    __syncwarp();
  }

  static __device__ __forceinline__ bool is_heavy(E& e, int mode, int atype) { return e.deferred_type(mode, atype); }

  /* the deposit-type heavy defender actions (clean / revert / upgrade) of a plain set-form step, one warp per env;
   * lane 0 owns cost / dirty / scalars */
  static __device__ __forceinline__ void defender(E& e, const typename E::Act& a, int atype, double& cost, bool& dirty) {
    const int lane = lane_id();
    const cyg_config& c = e.n->cfg;
    const double ds = (double)c.def_scale;
    if (atype == 1) {
      uint32_t A[W];
      e.clean_mask(a, A);
      __syncwarp();
      /* clean_scalar (rewards, discovery flags, state wipe; volt:996-1011) with one lane per (plane, word) */
      const int ncby = e.n->ncby, items = (5 + ncby) * W;
      int nc = 0, nu = 0;
      uint32_t disc = 0;
      for (int t = lane; t < items; t += 32) {
        const int pi = t / W, w = t - pi * W;
        uint32_t aw = 0;
#pragma unroll
        for (int q = 0; q < W; q++) aw |= A[q] & eqmask(q, w);
        const int p = pi == 0 ? P_COMP : pi == 1 ? P_HASWL : pi < 5 ? P_PT0 + (pi - 2) : P_CBY0 + (pi - 5);
        const uint32_t old = e.pl(p, w);
        e.pl(p, w) = old & ~aw;
        if (pi == 0) { nc += popc(aw & old); nu += popc(aw & ~old); }
        if (pi >= 5 && (old & aw) != 0) disc |= 1u << (pi - 5);
      }
      nc = __reduce_add_sync(CYG_FULL, nc);
      nu = __reduce_add_sync(CYG_FULL, nu);
      disc = __reduce_or_sync(CYG_FULL, disc);
      if (lane == 0) {
        cost += (nc * 0.3 - nu * 0.01) * ds;
        e.cleancost += (nc * 0.3 + nu * 0.01) * ds;
        e.defcost += (nc * 0.3 + nu * 0.01) * ds;
        e.scal(CYG_S_FLAGS) |= disc << CYG_FL_DISC_SHIFT; /* exp.discovered = True */
      }
      __syncwarp();
      deposit(e, A, 0, c.default_high, 0);
    } else if (atype == 3) {
      const bool has = (e.scal(CYG_S_FLAGS) & CYG_FL_HAS_CKPT) != 0;
      __syncwarp();
      if (lane == 0) e.scal(CYG_S_REVERT)++;
      if (has) {
        uint32_t A[W];
#pragma unroll
        for (int w = 0; w < W; w++) A[w] = e.m_valid(w);
        deposit(e, A, 0, c.default_high, 0);
        if (lane == 0) {
#pragma unroll
          for (int w = 0; w < W; w++) { e.pl(P_HASWL, w) = 0; e.pl(P_PT0, w) = 0; e.pl(P_PT0 + 1, w) = 0; e.pl(P_PT0 + 2, w) = 0; }
          cost += -1.0 * a.n_dev * ds;
          dirty = true;
        }
      }
    } else if (atype == 4) {
      uint32_t act[W], up[W];
      const int na = e.listed_active(a, act);
      if (na > 0) {
        e.upgrade_mask(act, a.app_index, up);
        if (lane == 0) cost += -1.0 * ds * na;
        deposit(e, up, 0, c.default_high, 0);
      }
    }
    __syncwarp();
  }
};

/* ---- large networks (128 < M <= 2048, planes of CYG_BIG_W = 64 words; BASELINE.json config C4): warp-per-env forms
 *      of the two actions whose thread-per-env cost grows with devices x words -- block / unblock (one pick per listed
 *      device) and the lateral-movement scan (one scan per source).  The record sits in shared memory (Env<W, 2>), a
 *      64-word device mask is two words per lane, and the adjacency is walked as CSR rows: a device's out-units
 *      [ip[d], ip[d] + nout[d]) of the unit table (L2-resident), 32 units per warp step.  Both walks are sequential over
 *      devices, as in the reference; the lanes share the work inside one device.  Envs with extra (hub-star) edges take
 *      the one-lane forms of cyg_core.cuh. ---- */
template <int W>
struct BigCoop {
  typedef Env<W, 2> E;
  static_assert(W == 64, "two plane words per lane");

  /* lowest set bit over a lane-distributed 64-word mask (lane l holds words l and l + 32); clears it; -1 when empty */
  static __device__ __forceinline__ int pop_lowest(uint32_t& m0, uint32_t& m1, int lane) {
    const int c0 = m0 ? 32 * lane + __ffs((int)m0) - 1 : 0x7FFFFFFF;
    const int c1 = m1 ? 32 * (lane + 32) + __ffs((int)m1) - 1 : 0x7FFFFFFF;
    const int d = (int)__reduce_min_sync(CYG_FULL, (unsigned)min(c0, c1));
    if (d == 0x7FFFFFFF) return -1;
    if ((d >> 5) == lane) m0 &= m0 - 1u;
    if ((d >> 5) == lane + 32) m1 &= m1 - 1u;
    return d;
  }

  /* block (6) / unblock (9): volt:1071-1100 -> :485-511, set form.  Returns false when the env must take the one-lane
   * path instead (extra edges, inconsistent header). */
  /* lane-distributed mask of the devices that are an endpoint of an extra (hub-star) edge: src = sources only */
  static __device__ __forceinline__ void extra_endpoints(E& e, bool src_only, uint32_t& x0, uint32_t& x1, int lane) {
    x0 = 0; x1 = 0;
    const int nx = e.n_extra();
    const uint32_t* x = e.extra();
    for (int base = 0; base < nx; base += 32) { /* uniform */
      const uint32_t xe = base + lane < nx ? x[base + lane] : 0xFFFFFFFFu;
      const int cnt = min(32, nx - base);
      for (int t = 0; t < cnt; t++) {
        const uint32_t w = __shfl_sync(CYG_FULL, xe, t);
        const int u = (int)(w & CYG_X_IDMASK), v = (int)((w >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
        if ((u >> 5) == lane) x0 |= 1u << (u & 31);
        if ((u >> 5) == lane + 32) x1 |= 1u << (u & 31);
        if (!src_only) {
          if ((v >> 5) == lane) x0 |= 1u << (v & 31);
          if ((v >> 5) == lane + 32) x1 |= 1u << (v & 31);
        }
      }
    }
  }
  static __device__ __forceinline__ bool test_bit(uint32_t x0, uint32_t x1, int d) {
    const uint32_t w = __shfl_sync(CYG_FULL, (d >> 5) < 32 ? x0 : x1, (d >> 5) & 31);
    return (w >> (d & 31)) & 1u;
  }

  static __device__ __forceinline__ bool flip(E& e, const typename E::Act& a, int atype, double& cost, bool& dirty) {
    const int lane = lane_id();
    const bool has_x = e.n_extra() > 0;
    uint32_t xi0 = 0, xi1 = 0; /* devices with an incident extra edge: their pool is a merged list, walked by lane 0 alone */
    if (has_x) extra_endpoints(e, false, xi0, xi1, lane);
    const bool want = atype == 9;
    const int site = want ? SITE_UNBLOCK : SITE_BLOCK;
    const uint32_t flipw = want ? 0u : 0xFFFFFFFFu;
    const int Wm = e.n->Wm;
    uint32_t m0 = (lane < Wm ? a.mask[lane] : 0u) & e.m_valid(lane);
    uint32_t m1 = (lane + 32 < Wm ? a.mask[lane + 32] : 0u) & e.m_valid(lane + 32);
    const int nl = (int)__reduce_add_sync(CYG_FULL, (unsigned)(popc(m0) + popc(m1)));
    if (a.n_dev < nl) return false;
    m0 &= ~e.pl(P_NYA, lane); m1 &= ~e.pl(P_NYA, lane + 32);
    const int na = (int)__reduce_add_sync(CYG_FULL, (unsigned)(popc(m0) + popc(m1)));
    if (na == 0) return true;
    const double ds = (double)e.n->cfg.def_scale;
    if (lane == 0) { cost += -0.5 * ds * na; e.defcost += 0.5 * ds * na; }
    uint32_t* const bits = e.inc();
    uint32_t blk[4]; /* lane l: Philox block (kblk + l) of the site = draws 4 (kblk + l) .. + 3 */
    uint32_t kdraw = 0, kblk = 0xFFFFFFFFu, cnt = 0;
    for (;;) { /* uniform */
      const int d = pop_lowest(m0, m1, lane);
      if (d < 0) break;
      if (has_x && test_bit(xi0, xi1, d)) { /* uniform */
        uint32_t kn = kdraw, ok = 0;
        if (lane == 0) {
          Stream st(site);
          st.k = kdraw;
          ok = e.flip_incident_general(d, want, st) ? 1u : 0u;
          kn = st.k;
        }
        kdraw = __shfl_sync(CYG_FULL, kn, 0);
        cnt += __shfl_sync(CYG_FULL, ok, 0);
        __syncwarp();
        continue;
      }
      const uint32_t di = e.dinfo(d), di1 = e.dinfo(d + 1);
      const int a0 = (int)(di & 0xFFFFu), nt = (int)(di1 & 0xFFFFu) - a0;
      /* the pool: units [a0, a0 + nt) with the wanted flag.  At most 32 units (all but the hubs): one window word, every
       * lane computes the same weight and pick, no reduction; else 32 words (1024 units) per round across the lanes */
      const bool small = nt <= 32;
      uint32_t xs = 0;
      int total = 0;
      if (small) {
        xs = (funnel_r(bits[a0 >> 5], bits[(a0 >> 5) + 1], a0 & 31) ^ flipw) & lowmask(nt);
        total = popc(xs);
      } else {
        for (int base = 0; base < nt; base += 1024) {
          const int q0 = a0 + base + 32 * lane;
          uint32_t x = 0;
          if (base + 32 * lane < nt) x = (funnel_r(bits[q0 >> 5], bits[(q0 >> 5) + 1], q0 & 31) ^ flipw) & lowmask0(nt - base - 32 * lane);
          total += (int)__reduce_add_sync(CYG_FULL, (unsigned)popc(x));
        }
      }
      if (total == 0) continue;
      if ((kdraw >> 7) != kblk) { /* refill: 128 draws */
        kblk = kdraw >> 7;
        philox4x32_10(e.rng.env, e.rng.epoch, (uint32_t)site, (kblk << 5) + (uint32_t)lane, e.rng.k0, e.rng.k1, blk);
      }
      const int from = (int)((kdraw >> 2) & 31u);
      const uint32_t x0 = __shfl_sync(CYG_FULL, blk[0], from), x1 = __shfl_sync(CYG_FULL, blk[1], from);
      const uint32_t x2 = __shfl_sync(CYG_FULL, blk[2], from), x3 = __shfl_sync(CYG_FULL, blk[3], from);
      const uint32_t j = kdraw & 3u;
      kdraw++;
      int r = (int)below(j == 0 ? x0 : j == 1 ? x1 : j == 2 ? x2 : x3, (uint32_t)total);
      int q = -1;
      if (small) {
        q = a0 + select_in_word(xs, r);
      } else {
        for (int base = 0; base < nt && q < 0; base += 1024) { /* uniform: q is */
          const int q0 = a0 + base + 32 * lane;
          uint32_t x = 0;
          if (base + 32 * lane < nt) x = (funnel_r(bits[q0 >> 5], bits[(q0 >> 5) + 1], q0 & 31) ^ flipw) & lowmask0(nt - base - 32 * lane);
          const int pc = popc(x);
          int incl = pc;
#pragma unroll
          for (int dd = 1; dd < 32; dd <<= 1) {
            const int y = __shfl_up_sync(CYG_FULL, incl, dd);
            if (lane >= dd) incl += y;
          }
          const int tot_r = __shfl_sync(CYG_FULL, incl, 31), excl = incl - pc;
          const bool mine = r >= excl && r < incl;
          const uint32_t mm = __ballot_sync(CYG_FULL, mine);
          if (mm) {
            const int qq = mine ? q0 + select_in_word(x, r - excl) : 0;
            q = __shfl_sync(CYG_FULL, qq, __ffs((int)mm) - 1);
          } else {
            r -= tot_r;
          }
        }
      }
      if (lane == 0) e.set_pair_blocked(q, !want);
      cnt++;
      __syncwarp();
    }
    if (lane == 0 && cnt) { e.scal(want ? CYG_S_EADD : CYG_S_EBLK) += cnt; dirty = true; }
    __syncwarp();
    return true;
  }

  /* attacker action 1, exploit + lateral movement (volt:1126-1185): sources in ascending id order, each source's
   * out-units scanned 32 at a time (lane = unit): blocked units are skipped unlogged, the first unit whose far endpoint
   * qualifies is the hit, the unblocked units in front of it are the hops logged.  Returns false when the env must take
   * the one-lane path (extra edges). */
  static __device__ __forceinline__ bool attack(E& e, const typename E::Act& a) {
    const int lane = lane_id();
    const int nx = e.n_extra();
    uint32_t xs0 = 0, xs1 = 0; /* sources with extra out-edges */
    if (nx > 0) extra_endpoints(e, true, xs0, xs1, lane);
    const uint32_t* const xl = e.extra();
    uint32_t s0 = e.pl(P_COMP, lane) | e.pl(P_OWNED, lane), s1 = e.pl(P_COMP, lane + 32) | e.pl(P_OWNED, lane + 32);
    const bool has_blk = e.any_blocked();
    __syncwarp();
    const uint32_t* const bits = e.inc();
    uint32_t logs_add = 0, zk = 0;
    for (int xi = 0; xi < a.n_ex; xi++) { /* uniform */
      int raw = a.ex(xi);
      uint32_t zx = 0;
      if (e.needs_zday_draw(raw)) zx = draw_at(e.rng, SITE_ZDAY, zk++);
      raw = e.resolve_exploit(raw, zx);
      if (raw < 0) continue;
      uint32_t t0 = s0, t1 = s1;
      for (;;) {
        const int s = pop_lowest(t0, t1, lane);
        if (s < 0) break;
        const bool is_dc = e.devbit(e.n->o_dc, s);
        const uint32_t di = e.dinfo(s);
        const int a0 = (int)(di & 0xFFFFu), no = (int)(di >> 16);
        int hit = -1, walked = 0;
        /* extra out-edges of s (unblocked ones): the lowest qualifying target competes with the base scan, the unblocked
         * ones in front of the hit are logged like base hops */
        int ve = 0x7FFFFFFF;
        const bool sx = nx > 0 && test_bit(xs0, xs1, s);
        if (sx) {
          for (int base = 0; base < nx; base += 32) {
            const uint32_t xe = base + lane < nx ? xl[base + lane] : 0xFFFFFFFFu;
            int cand = 0x7FFFFFFF;
            if ((int)(xe & CYG_X_IDMASK) == s && !(xe & CYG_X_BLOCKED) && xe != 0xFFFFFFFFu) {
              const int v = (int)((xe >> CYG_X_V_SHIFT) & CYG_X_IDMASK);
              const uint32_t vb = 1u << (v & 31);
              const int vw = v >> 5;
              if (is_dc || (e.m_reach(vw) & vb) || (!(e.pl(P_COMP, vw) & vb) && (e.pl(P_KNOWN, vw) & vb) && (e.m_vuln(raw, vw) & vb))) cand = v;
            }
            ve = min(ve, (int)__reduce_min_sync(CYG_FULL, (unsigned)cand));
          }
        }
        bool stopped = false;
        for (int base = 0; base < no && !stopped; base += 32) { /* uniform */
          const int q = a0 + base + lane;
          const bool in = base + lane < no;
          int v = 0;
          bool open = false, ok = false;
          if (in) {
            v = unit_other(e.unit(q));
            open = !(has_blk && ((bits[q >> 5] >> (q & 31)) & 1u));
            const uint32_t vb = 1u << (v & 31);
            const int vw = v >> 5;
            ok = open && (is_dc || (e.m_reach(vw) & vb) || (!(e.pl(P_COMP, vw) & vb) && (e.pl(P_KNOWN, vw) & vb) && (e.m_vuln(raw, vw) & vb)));
          }
          const uint32_t openm = __ballot_sync(CYG_FULL, open), okm = __ballot_sync(CYG_FULL, ok);
          const uint32_t stopm = okm | __ballot_sync(CYG_FULL, in && v > ve); /* ascending ids: past ve the extra edge comes first */
          if (stopm) {
            const int hl = __ffs((int)stopm) - 1;
            const int vh = __shfl_sync(CYG_FULL, v, hl);
            if (((okm >> hl) & 1u) && vh < ve) hit = vh;
            walked += popc(openm & lanes_below(hl));
            stopped = true;
          } else {
            walked += popc(openm);
          }
        }
        if (hit < 0 && ve != 0x7FFFFFFF) hit = ve;
        if (e.logs != nullptr && lane == 0) { /* one lane writes this source's hops (the ring is a diagnostic at this size) */
          uint32_t xrow_l[W];
          if (sx) e.extra_out_row(s, false, xrow_l);
          e.log_source(s, hit, has_blk, sx ? xrow_l : (const uint32_t*)nullptr, e.scal(CYG_S_LOGS) + logs_add, 0u);
        }
        if (sx) { /* unblocked extra edges of s in front of the hit (all of them when nothing is hit) */
          for (int base = 0; base < nx; base += 32) {
            const uint32_t xe = base + lane < nx ? xl[base + lane] : 0xFFFFFFFFu;
            const bool mine = xe != 0xFFFFFFFFu && (int)(xe & CYG_X_IDMASK) == s && !(xe & CYG_X_BLOCKED) &&
                              (hit < 0 || (int)((xe >> CYG_X_V_SHIFT) & CYG_X_IDMASK) < hit);
            walked += popc(__ballot_sync(CYG_FULL, mine));
          }
        }
        logs_add += (uint32_t)walked + (hit >= 0 ? 1u : 0u);
        if (hit >= 0 && lane == 0) {
          e.pl(P_COMP, hit >> 5) |= 1u << (hit & 31);
          if (is_dc) e.pl(P_CBY0 + raw, hit >> 5) |= 1u << (hit & 31);
        }
        __syncwarp();
      }
    }
    if (lane == 0) e.scal(CYG_S_LOGS) += logs_add;
    __syncwarp();
    return true;
  }
};

}  // namespace cyg
#endif
