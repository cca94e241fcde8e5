/*
 * cyg_iforest.cuh -- the detector FIT of defender action 10 (CDSimulator.py:687-695) on the device.
 *
 * Detector.train fits scikit-learn's IsolationForest(n_estimators=2, max_samples=256) with random_state=None, i.e. from
 * numpy's global stream, on the last <= 2000 hop-log records.  Once that stream is seeded, the fit is a function of the
 * records and the seed only; this file restates it step by step so that the slot it writes is word for word
 * cygym_b200/detector.py: pack_detector(fit_detector(records, seed)) (scikit-learn 1.9, numpy 2.x):
 *
 *   IsolationForest.fit (ensemble/_iforest.py)   y = uniform(size=n); max_depth = ceil(log2(max(max_samples, 2)))
 *   BaseBagging._fit (ensemble/_bagging.py)      seeds = randint(2**31 - 1, size=2) from the same stream; tree i gets
 *                                                random_state = RandomState(seeds[i]).randint(2**31 - 1) and the rows
 *                                                sample_without_replacement(n, max_samples, RandomState(seeds[i])) as
 *                                                sample_weight = bincount(rows): the tree sees them in ascending order
 *   utils/_random.pyx                            ratio >= 0.99: reservoir sampling; else permutation(n)[:max_samples]
 *   tree/_splitter.pyx, _partitioner.pyx         RandomSplitter.node_split (max_features = 1), swap partition
 *   tree/_criterion.pyx                          MSE sums in the partitioner's sample order
 *   tree/_tree.pyx                               DepthFirstTreeBuilder: stack order (node ids), the EPSILON leaf tests
 *   tree/_utils.pyx, utils/_random.pxd           our_rand_r, rand_int, rand_uniform
 *   numpy legacy RandomState                     mt19937_seed (integer seed), the twist, the 53-bit double, masked
 *                                                rejection (randint, 32-bit path), random_interval (shuffle)
 *
 * Double arithmetic goes through dadd / dmul / ddiv: never contracted into FMAs, as on the host that fitted the
 * reference.  Feature values are float32 (scikit-learn's DTYPE).  The serial part (the streams, the sampling, the tree
 * builds) is one thread's work; zeroing the slot and the verdict table split over `nlanes` lanes.
 */
#ifndef CYG_IFOREST_CUH
#define CYG_IFOREST_CUH

#include <stdint.h>
#include <string.h>

#include "cyg_core.cuh"

namespace cyg {
namespace iforest {

enum { MAX_SAMPLES = 256, N_TREES = 2, MAX_NODES = 512, STACK = 16 };

CYG_HD double dadd(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}
CYG_HD double dsub(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dsub_rn(a, b);
#else
  return a - b;
#endif
}
CYG_HD double dmul(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
CYG_HD double ddiv(double a, double b) {
#ifdef __CUDA_ARCH__
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}
CYG_HD uint64_t dbits(double d) {
#ifdef __CUDA_ARCH__
  return (uint64_t)__double_as_longlong(d);
#else
  uint64_t u;
  memcpy(&u, &d, 8);
  return u;
#endif
}
CYG_HD double bitsd(uint64_t u) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)u);
#else
  double d;
  memcpy(&d, &u, 8);
  return d;
#endif
}

/* c(k) of sklearn.ensemble._iforest._average_path_length for k = 0 .. 256, float64 bits (it evaluates np.log; the
 * device reads the table instead).  tests/test_detector_fit.py regenerates it from scikit-learn and compares. */
#define CYG_APL_TABLE {                                                                                   \
  0x0000000000000000ull, 0x0000000000000000ull, 0x3ff0000000000000ull, 0x3ff3517aa6149ab3ull, \
  0x3ffda061f1c9bc30ull, 0x40029dbcb065482full, 0x4005a73320d012eaull, 0x400830770aab1fa0ull, \
  0x400a5eb92c6a3564ull, 0x400c48c76e764e64ull, 0x400dfdb50d2b7abcull, 0x400f88070ce856acull, \
  0x401077b1a145cf7dull, 0x40111cc3d48d15dcull, 0x4011b5708edfc2fcull, 0x40124375de7c31b6ull, \
  0x4012c839786935a5ull, 0x401344deb68e9feeull, 0x4013ba561d88341cull, 0x40142968947a05c9ull, \
  0x401492bfab870718ull, 0x4014f6ebd2f15730ull, 0x40155669195d1094ull, 0x4015b1a2d7bddfd4ull, \
  0x401608f69242f6cbull, 0x40165cb640ccd2d1ull, 0x4016ad2a23583fa5ull, 0x4016fa923d028d11ull, \
  0x40174527896896a8ull, 0x40178d1cfb36a197ull, 0x4017d2a04f2e2fe9ull, 0x401815dabc48cc63ull, \
  0x401856f187ad18e0ull, 0x4018960681b5ae30ull, 0x4018d338702de294ull, 0x40190ea3690f7f24ull, \
  0x401948612064c4daull, 0x401980892b6f90feull, 0x4019b7313acff8a2ull, 0x4019ec6d4d13b276ull, \
  0x401a204fdad72e8full, 0x401a52e9fd6d97c6ull, 0x401a844b90db5ce0ull, 0x401ab48351cd24c0ull, \
  0x401ae39ef81993c6ull, 0x401b11ab4e45c4a2ull, 0x401b3eb44671cd6dull, 0x401b6ac50d035613ull, \
  0x401b95e8195788e7ull, 0x401bc0273cbb0706ull, 0x401be98bafdda407ull, 0x401c121e1ef0315eull, \
  0x401c39e6b49450fcull, 0x401c60ed23c0edc2ull, 0x401c8738b0b96c91ull, 0x401cacd03931c8b7ull, \
  0x401cd1ba3bb67db5ull, 0x401cf5fcde6c4865ull, 0x401d199df539572full, 0x401d3ca30767646eull, \
  0x401d5f1154cc629aull, 0x401d80edda85cc50ull, 0x401da23d575149c1ull, 0x401dc3044f8c2964ull, \
  0x401de34710e21dbcull, 0x401e0309b5b2c664ull, 0x401e22502834bc8full, 0x401e411e255c258aull, \
  0x401e5f773f8a2dfeull, 0x401e7d5ee10a437aull, 0x401e9ad84e6164d0ull, 0x401eb7e6a8737363ull, \
  0x401ed48cee820cdfull, 0x401ef0ce00081dc5ull, 0x401f0cac9e750f0dull, 0x401f282b6eca2bdbull, \
  0x401f434cfb1c9dedull, 0x401f5e13b3fe280eull, 0x401f7881f1ce93a2ull, 0x401f9299f5f79a0cull, \
  0x401fac5dec14ea06ull, 0x401fc5cfeb09c4f8ull, 0x401fdef1f6058fb5ull, 0x401ff7c5fd789444ull, \
  0x40200826effd0c08ull, 0x40201445b59068a3ull, 0x402020402e275850ull, 0x40202c1730b8705bull, \
  0x402037cb8cda6521ull, 0x4020435e0b196de4ull, 0x40204ecf6d47e26full, 0x40205a206eca6387ull, \
  0x40206551c4dfd912ull, 0x402070641ee58b42ull, 0x40207b58269796bbull, 0x4020862e804df708ull, \
  0x402090e7cb365e51ull, 0x40209b84a18b0d37ull, 0x4020a60598c6da3eull, 0x4020b06b41d6948dull, \
  0x4020bab62947eaf8ull, 0x4020c4e6d775fd46ull, 0x4020cefdd0b3bafeull, 0x4020d8fb957430d4ull, \
  0x4020e2e0a270e34cull, 0x4020ecad70ce5341ull, 0x4020f662763ec724ull, 0x40210000252371deull, \
  0x40210986ecac0eb6ull, 0x402112f738f5081dull, 0x40211c5173243dd2ull, 0x4021259601847d88ull, \
  0x40212ec5479fbff6ull, 0x402137dfa6583b4eull, 0x402140e57c005aafull, 0x402149d72471a99aull, \
  0x402152b4f922c146ull, 0x40215b7f513c44daull, 0x4021643681acf904ull, 0x40216cdadd3d025eull, \
  0x4021756cb4a0559eull, 0x40217dec568863daull, 0x4021865a0fb50c7cull, 0x40218eb62b04de16ull, \
  0x40219700f184aeb4ull, 0x40219f3aaa7e93c1ull, 0x4021a7639b88412cull, 0x4021af7c0890d71eull, \
  0x4021b78433ee2505ull, 0x4021bf7c5e696876ull, 0x4021c764c74b8e0cull, 0x4021cf3dac68fa07ull, \
  0x4021d7074a2cde2dull, 0x4021dec1dba42222ull, 0x4021e66d9a87e31dull, 0x4021ee0abf478fa7ull, \
  0x4021f5998112a3e0ull, 0x4021fd1a15e20a5cull, 0x4022048cb28125c0ull, 0x40220bf18a9686c7ull, \
  0x40221348d0ac524aull, 0x40221a92b6385ad1ull, 0x402221cf6ba3f0c8ull, 0x402228ff20536c82ull, \
  0x4022302202ad7503ull, 0x402237384022063eull, 0x40223e420531398full, 0x4022453f7d71d2e9ull, \
  0x40224c30d3979520ull, 0x4022531631795faaull, 0x402259efc01717f7ull, 0x402260bda79f607dull, \
  0x402267800f751f82ull, 0x40226e371e34d76full, 0x402274e2f9b9d29eull, 0x40227b83c7232444ull, \
  0x40228219aad88026ull, 0x402288a4c88eeabdull, 0x40228f25434d432cull, 0x4022959b3d70a89cull, \
  0x40229c06d8b0bc41ull, 0x4022a2683623c173ull, 0x4022a8bf76429d0cull, 0x4022af0cb8ecb544ull, \
  0x4022b5501d6bb344ull, 0x4022bb89c277276cull, 0x4022c1b9c6381175ull, 0x4022c7e0464c4d6full, \
  0x4022cdfd5fc9e684ull, 0x4022d4112f425085ull, 0x4022da1bd0c5891aull, 0x4022e01d5fe5216bull, \
  0x4022e615f7b73120ull, 0x4022ec05b2d93382ull, 0x4022f1ecab72cf73ull, 0x4022f7cafb388afdull, \
  0x4022fda0bb6e6b39ull, 0x4023036e04ea8118ull, 0x40230932f01763deull, 0x40230eef94f699c5ull, \
  0x402314a40b22ef76ull, 0x40231a5069d2beeeull, 0x40231ff4c7da2648ull, 0x402325913bad2f08ull, \
  0x40232b25db61e65bull, 0x402330b2bcb266ceull, 0x40233637f4fed3f4ull, 0x40233bb5994f4876ull, \
  0x4023412bbe55b6eaull, 0x4023469a786fbdf1ull, 0x40234c01dba86ff7ull, 0x40235161fbba0effull, \
  0x402356baec0fbcd2ull, 0x40235c0cbfc71ffdull, 0x4023615789b1fde3ull, 0x4023669b5c57ca4dull, \
  0x40236bd849f72cbcull, 0x4023710e64877bd6ull, 0x4023763dbdba2f34ull, 0x40237b6666fc47e0ull, \
  0x402380887177afceull, 0x402385a3ee14908aull, 0x40238ab8ed7aa16aull, 0x40238fc780126d7aull, \
  0x402394cfb606916dull, 0x402399d19f44f1c3ull, 0x40239ecd4b7fe961ull, 0x4023a3c2ca2f70d8ull, \
  0x4023a8b22a923e8full, 0x4023ad9b7baee003ull, 0x4023b27ecc54cc4dull, 0x4023b75c2b1d7028ull, \
  0x4023bc33a66d339cull, 0x4023c1054c747983ull, 0x4023c5d12b309913ull, 0x4023ca97506cd190ull, \
  0x4023cf57c9c33864ull, 0x4023d412a49da1a5ull, 0x4023d8c7ee368351ull, 0x4023dd77b399d352ull, \
  0x4023e22201a5e071ull, 0x4023e6c6e50c265eull, 0x4023eb666a521cf2ull, 0x4023f0009dd202c7ull, \
  0x4023f4958bbba342ull, 0x4023f9254015183dull, 0x4023fdafc6bb8761ull, 0x402402352b63db4dull, \
  0x402406b5799b78b6ull, 0x40240b30bcc8ef86ull, 0x40240fa7002ca826ull, 0x402414184ee18d01ull, \
  0x40241884b3ddb060ull, 0x40241cec39f2eeb5ull, 0x4024214eebcf8d68ull, 0x402425acd3fed64cull, \
  0x40242a05fce9afb5ull, 0x40242e5a70d7316bull, 0x402432aa39ed366bull, 0x402436f56230eba0ull, \
  0x40243b3bf3875ba1ull, 0x40243f7df7b5f786ull, 0x402443bb78631ce8ull, 0x402447f47f16991full, \
  0x40244c29153a29c6ull, 0x402450594419fab4ull, 0x4024548514e52140ull, 0x402458ac90ae152cull, \
  0x40245ccfc06b2706ull, 0x402460eeacf6f428ull, 0x402465095f10d872ull, 0x4024691fdf5d5db4ull, \
  0x40246d323666a8e6ull, 0x402471406c9ce532ull, 0x4024754a8a56ace2ull, 0x4024795097d17047ull, \
  0x40247d529d31da8full, \
}
#ifdef __CUDACC__
static __constant__ uint64_t kAplDev[257] = CYG_APL_TABLE;
#endif
static const uint64_t kAplHost[257] = CYG_APL_TABLE;
#undef CYG_APL_TABLE
CYG_HD double avg_path_length(int k) {
#ifdef __CUDA_ARCH__
  return bitsd(kAplDev[k]);
#else
  return bitsd(kAplHost[k]);
#endif
}

/* ---- numpy's legacy RandomState (MT19937) ---- */
struct MT {
  uint32_t key[624];
  int pos;
};
CYG_HD void mt_seed(MT& s, uint32_t seed) { /* mt19937_seed: what RandomState(int) / np.random.seed(int) run */
  for (int i = 0; i < 624; i++) {
    s.key[i] = seed;
    seed = 1812433253u * (seed ^ (seed >> 30)) + (uint32_t)i + 1u;
  }
  s.pos = 624;
}
CYG_HD void mt_twist(MT& s) { /* mt19937_gen */
  int i = 0;
  for (; i < 624 - 397; i++) {
    const uint32_t y = (s.key[i] & 0x80000000u) | (s.key[i + 1] & 0x7FFFFFFFu);
    s.key[i] = s.key[i + 397] ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908B0DFu);
  }
  for (; i < 623; i++) {
    const uint32_t y = (s.key[i] & 0x80000000u) | (s.key[i + 1] & 0x7FFFFFFFu);
    s.key[i] = s.key[i + 397 - 624] ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908B0DFu);
  }
  const uint32_t y = (s.key[623] & 0x80000000u) | (s.key[0] & 0x7FFFFFFFu);
  s.key[623] = s.key[396] ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908B0DFu);
  s.pos = 0;
}
CYG_HD uint32_t mt_next(MT& s) {
  if (s.pos == 624) mt_twist(s);
  uint32_t y = s.key[s.pos++];
  y ^= y >> 11;
  y ^= (y << 7) & 0x9D2C5680u;
  y ^= (y << 15) & 0xEFC60000u;
  return y ^ (y >> 18);
}
CYG_HD double mt_double(MT& s) { /* random_sample / uniform(0, 1): 0.0 + 1.0 * d == d */
  const uint32_t a = mt_next(s) >> 5, b = mt_next(s) >> 6;
  return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
}
/* An integer in [0, rng] by masked rejection: randint(low, high) = low + mt_bounded(high - 1 - low) on the 32-bit path
 * (buffered_bounded_masked_uint32; rng == 0 draws nothing), and random_interval(rng), shuffle's draw. */
CYG_HD uint32_t mt_bounded(MT& s, uint32_t rng) {
  if (rng == 0) return 0;
  uint32_t mask = rng;
  mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
  uint32_t v;
  while ((v = mt_next(s) & mask) > rng) {
  }
  return v;
}

/* ---- scikit-learn's rand_r (tree/_utils.pyx, utils/_random.pxd) ---- */
#define CYG_RAND_R_MAX 2147483647u
CYG_HD uint32_t our_rand_r(uint32_t& seed) {
  if (seed == 0) seed = 1u; /* DEFAULT_SEED */
  seed ^= seed << 13;
  seed ^= seed >> 17;
  seed ^= seed << 5;
  return seed % (CYG_RAND_R_MAX + 1u);
}
CYG_HD int rand_int(int low, int high, uint32_t& seed) { return low + (int)(our_rand_r(seed) % (uint32_t)(high - low)); }
CYG_HD double rand_uniform(double low, double high, uint32_t& seed) {
  return dadd(ddiv(dmul(dsub(high, low), (double)our_rand_r(seed)), (double)CYG_RAND_R_MAX), low);
}

/* Per-fit working memory (one per fitting warp; shared memory on the device). */
struct Scratch {
  MT mt;
  union {
    uint16_t perm[CYG_DET_WINDOW];     /* permutation(n) while the rows are drawn */
    struct {
      double y[N_TREES][MAX_SAMPLES];  /* the target uniforms of each tree's rows */
      double lv[N_TREES][MAX_SAMPLES]; /* per leaf: depth + c(n_leaf) - 1.0 */
    } t;
  } u;
  uint32_t sel[(CYG_DET_WINDOW + 31) / 32];
  uint16_t rows[N_TREES][MAX_SAMPLES]; /* each tree's rows (ascending log positions) */
  uint32_t rec[MAX_SAMPLES];           /* the record of row k of the tree being built */
  uint16_t samples[MAX_SAMPLES];       /* the splitter's sample order (indices k) */
  float fv[MAX_SAMPLES];               /* the partitioner's feature_values */
  int n_leaves[N_TREES];
  int ms;                              /* max_samples = min(256, n) */
};

CYG_HD float feature_of(uint32_t rec, int f) { return (float)(f == 0 ? (rec & 0xFFFFu) : (rec >> 16)); }

struct Split {
  int feature, pos;
  double threshold, improvement, imp_left, imp_right;
};
struct Crit { /* MSE over samples[start, end) with unit weights (RegressionCriterion / MSE of _criterion.pyx) */
  int start, end, pos;
  double sum_total, sq_sum_total, wn_node, sum_left, sum_right, wn_left, wn_right;
};

CYG_HD void crit_init(Crit& c, const Scratch& s, const double* y, int start, int end) {
  c.start = start; c.end = end;
  c.sum_total = 0.0; c.sq_sum_total = 0.0; c.wn_node = 0.0;
  for (int p = start; p < end; p++) {
    const double yi = y[s.samples[p]];
    const double wy = dmul(1.0, yi);
    c.sum_total = dadd(c.sum_total, wy);
    c.sq_sum_total = dadd(c.sq_sum_total, dmul(wy, yi));
    c.wn_node = dadd(c.wn_node, 1.0);
  }
  c.pos = start; c.sum_left = 0.0; c.sum_right = c.sum_total; c.wn_left = 0.0; c.wn_right = c.wn_node; /* reset() */
}
CYG_HD void crit_reset(Crit& c) { c.pos = c.start; c.sum_left = 0.0; c.sum_right = c.sum_total; c.wn_left = 0.0; c.wn_right = c.wn_node; }
CYG_HD void crit_update(Crit& c, const Scratch& s, const double* y, int new_pos) {
  if (new_pos - c.pos <= c.end - new_pos) {
    for (int p = c.pos; p < new_pos; p++) {
      c.sum_left = dadd(c.sum_left, dmul(1.0, y[s.samples[p]]));
      c.wn_left = dadd(c.wn_left, 1.0);
    }
  } else {
    c.pos = c.end; c.sum_right = 0.0; c.sum_left = c.sum_total; c.wn_right = 0.0; c.wn_left = c.wn_node; /* reverse_reset() */
    for (int p = c.end - 1; p >= new_pos; p--) {
      c.sum_left = dsub(c.sum_left, dmul(1.0, y[s.samples[p]]));
      c.wn_left = dsub(c.wn_left, 1.0);
    }
  }
  c.wn_right = dsub(c.wn_node, c.wn_left);
  c.sum_right = dsub(c.sum_total, c.sum_left);
  c.pos = new_pos;
}
CYG_HD double crit_node_impurity(const Crit& c) {
  const double m = ddiv(c.sum_total, c.wn_node);
  return dsub(ddiv(c.sq_sum_total, c.wn_node), dmul(m, m));
}
CYG_HD double crit_proxy(const Crit& c) {
  return dadd(ddiv(dmul(c.sum_left, c.sum_left), c.wn_left), ddiv(dmul(c.sum_right, c.sum_right), c.wn_right));
}
CYG_HD void crit_children(const Crit& c, const Scratch& s, const double* y, double& il, double& ir) {
  double sq_left = 0.0;
  for (int p = c.start; p < c.pos; p++) {
    const double yi = y[s.samples[p]];
    sq_left = dadd(sq_left, dmul(dmul(1.0, yi), yi));
  }
  const double sq_right = dsub(c.sq_sum_total, sq_left);
  const double ml = ddiv(c.sum_left, c.wn_left), mr = ddiv(c.sum_right, c.wn_right);
  il = dsub(ddiv(sq_left, c.wn_left), dmul(ml, ml));
  ir = dsub(ddiv(sq_right, c.wn_right), dmul(mr, mr));
}
CYG_HD double crit_improvement(const Crit& c, double wn_samples, double imp, double il, double ir) {
  return dmul(ddiv(c.wn_node, wn_samples),
              dsub(dsub(imp, dmul(ddiv(c.wn_right, c.wn_node), ir)), dmul(ddiv(c.wn_left, c.wn_node), il)));
}

/* RandomSplitter.node_split with max_features = 1 (tree/_splitter.pyx); features / constant_features persist across
 * the nodes of a tree, n_const is the parent record's n_constant_features (updated for the children). */
CYG_HD void node_split(Scratch& s, const double* y, int start, int end, double impurity, int& n_const, int* features,
                       int* constant_features, uint32_t& rstate, double wn_samples, Crit& c, Split& best) {
  best.pos = end; best.feature = 0; best.threshold = 0.0; best.improvement = -INFINITY;
  best.imp_left = INFINITY; best.imp_right = INFINITY;
  Split cur = best;
  double best_proxy = -INFINITY;
  int f_i = 2, n_found = 0, n_drawn = 0;
  const int n_known = n_const;
  int n_total = n_known, n_visited = 0;
  while (f_i > n_total && (n_visited < 1 || n_visited <= n_found + n_drawn)) {
    n_visited++;
    int f_j = rand_int(n_drawn, f_i - n_found, rstate);
    if (f_j < n_known) {
      const int t = features[n_drawn]; features[n_drawn] = features[f_j]; features[f_j] = t;
      n_drawn++;
      continue;
    }
    f_j += n_found;
    cur.feature = features[f_j];
    /* find_min_max */
    float mn = feature_of(s.rec[s.samples[start]], cur.feature), mx = mn;
    s.fv[start] = mn;
    for (int p = start + 1; p < end; p++) {
      const float v = feature_of(s.rec[s.samples[p]], cur.feature);
      s.fv[p] = v;
      if (v < mn) mn = v;
      else if (v > mx) mx = v;
    }
    if (mx <= mn + 1e-7f) { /* FEATURE_THRESHOLD: a constant feature */
      features[f_j] = features[n_total]; features[n_total] = cur.feature;
      n_found++; n_total++;
      continue;
    }
    f_i--;
    { const int t = features[f_i]; features[f_i] = features[f_j]; features[f_j] = t; }
    cur.threshold = rand_uniform((double)mn, (double)mx, rstate);
    if (cur.threshold == (double)mx) cur.threshold = (double)mn;
    /* partition_samples */
    int ps = start, pe = end;
    while (ps < pe) {
      if ((double)s.fv[ps] <= cur.threshold) {
        ps++;
      } else {
        pe--;
        const float tv = s.fv[ps]; s.fv[ps] = s.fv[pe]; s.fv[pe] = tv;
        const uint16_t ts = s.samples[ps]; s.samples[ps] = s.samples[pe]; s.samples[pe] = ts;
      }
    }
    cur.pos = pe;
    if (cur.pos - start < 1 || end - cur.pos < 1) continue; /* min_samples_leaf */
    crit_reset(c);
    crit_update(c, s, y, cur.pos);
    const double proxy = crit_proxy(c);
    if (proxy > best_proxy) { best_proxy = proxy; best = cur; }
  }
  if (best.pos < end) { /* with max_features = 1 the best split is the last one partitioned */
    crit_reset(c);
    crit_update(c, s, y, best.pos);
    crit_children(c, s, y, best.imp_left, best.imp_right);
    best.improvement = crit_improvement(c, wn_samples, impurity, best.imp_left, best.imp_right);
  }
  for (int i = 0; i < n_known; i++) features[i] = constant_features[i];
  for (int i = 0; i < n_found; i++) constant_features[n_known + i] = features[n_known + i];
  n_const = n_total;
}

/* DepthFirstTreeBuilder.build on the rows s.rows[t] (targets s.u.t.y[t]): node words into `tree` (the slot's tree t,
 * zeroed by the caller), the leaves' depth + c(n_leaf) - 1.0 into s.u.t.lv[t].  Returns the node count. */
CYG_HD int build_tree(Scratch& s, int t, uint32_t rstate, uint32_t* tree) {
  const double EPS = 2.220446049250313e-16; /* np.finfo('double').eps */
  const double* y = s.u.t.y[t];
  const int ms = s.ms;
  int max_depth = 0;
  while ((1 << max_depth) < (ms < 2 ? 2 : ms)) max_depth++;
  for (int k = 0; k < ms; k++) s.samples[k] = (uint16_t)k;
  int features[2] = {0, 1}, constant_features[2] = {0, 0};
  struct Rec { int start, end, depth, parent, is_left, n_const; double impurity; } stack[STACK];
  int sp = 0;
  stack[sp++] = {0, ms, 0, -1, 0, 0, INFINITY};
  Split split;
  split.pos = 0; split.feature = 0; split.threshold = 0.0; split.improvement = 0.0; split.imp_left = 0.0; split.imp_right = 0.0;
  Crit c;
  bool first = true;
  int n_nodes = 0, n_leaves = 0;
  const double wn_samples = (double)ms;
  while (sp > 0) {
    Rec r = stack[--sp];
    const int n_node = r.end - r.start;
    crit_init(c, s, y, r.start, r.end); /* splitter.node_reset */
    bool is_leaf = r.depth >= max_depth || n_node < 2;
    double impurity = r.impurity;
    if (first) { impurity = crit_node_impurity(c); first = false; }
    is_leaf = is_leaf || impurity <= EPS;
    int n_const = r.n_const;
    if (!is_leaf) {
      node_split(s, y, r.start, r.end, impurity, n_const, features, constant_features, rstate, wn_samples, c, split);
      is_leaf = split.pos >= r.end || dadd(split.improvement, EPS) < 0.0;
    }
    const int id = n_nodes++;
    if (r.parent >= 0) tree[4 * r.parent + 2] |= r.is_left ? (uint32_t)id : ((uint32_t)id << 16);
    uint32_t* w = tree + 4 * id;
    if (is_leaf) {
      const uint64_t tb = dbits(-2.0); /* _TREE_UNDEFINED */
      w[0] = (uint32_t)tb; w[1] = (uint32_t)(tb >> 32);
      w[3] = 2u | ((uint32_t)n_leaves << 16);
      /* compute_node_depths (root = 1) + _average_path_length(n_node_samples) - 1.0 */
      s.u.t.lv[t][n_leaves++] = dsub(dadd((double)(r.depth + 1), avg_path_length(n_node)), 1.0);
    } else {
      const uint64_t tb = dbits(split.threshold);
      w[0] = (uint32_t)tb; w[1] = (uint32_t)(tb >> 32);
      w[3] = (uint32_t)split.feature;
      stack[sp++] = {split.pos, r.end, r.depth + 1, id, 0, n_const, split.imp_right};
      stack[sp++] = {r.start, split.pos, r.depth + 1, id, 1, n_const, split.imp_left};
    }
  }
  s.n_leaves[t] = n_leaves;
  return n_nodes;
}

/* Row selection of one tree: sample_without_replacement(n, ms, RandomState(seed)) as an ascending list. */
CYG_HD void draw_rows(Scratch& s, int t, int n, uint32_t seed) {
  const int ms = s.ms;
  const int nw = (n + 31) >> 5;
  for (int i = 0; i < nw; i++) s.sel[i] = 0;
  if (n <= ms) {
    for (int i = 0; i < n; i++) s.sel[i >> 5] |= 1u << (i & 31);
  } else {
    mt_seed(s.mt, seed);
    if (ddiv((double)ms, (double)n) < 0.99) { /* permutation(n)[:ms]: legacy shuffle, i = n-1 .. 1 */
      for (int i = 0; i < n; i++) s.u.perm[i] = (uint16_t)i;
      for (int i = n - 1; i >= 1; i--) {
        const uint32_t j = mt_bounded(s.mt, (uint32_t)i);
        const uint16_t v = s.u.perm[i]; s.u.perm[i] = s.u.perm[j]; s.u.perm[j] = v;
      }
    } else { /* reservoir sampling */
      for (int i = 0; i < ms; i++) s.u.perm[i] = (uint16_t)i;
      for (int i = ms; i < n; i++) {
        const uint32_t j = mt_bounded(s.mt, (uint32_t)i); /* randint(0, i + 1) */
        if ((int)j < ms) s.u.perm[j] = (uint16_t)i;
      }
    }
    for (int k = 0; k < ms; k++) s.sel[s.u.perm[k] >> 5] |= 1u << (s.u.perm[k] & 31);
  }
  int k = 0;
  for (int i = 0; i < nw; i++)
    for (uint32_t m = s.sel[i]; m; m &= m - 1) s.rows[t][k++] = (uint16_t)(32 * i + ctz(m));
}

/* The serial part of one fit: `ring` holds the env's hop log (record i at i % log_cap), n_logs records in all; the last
 * n = min(n_logs, CYG_DET_WINDOW) <= log_cap are fitted.  `slot` (CYG_DET_WORDS) must be zero; the tree words and slot[0]
 * are written, the leaf values stay in `s` for verdict_words. */
CYG_HD void fit_serial(Scratch& s, const uint32_t* ring, uint32_t log_cap, uint32_t n_logs, uint32_t seed, uint32_t* slot) {
  const int n = (int)(n_logs < (uint32_t)CYG_DET_WINDOW ? n_logs : (uint32_t)CYG_DET_WINDOW);
  s.ms = n < MAX_SAMPLES ? n : MAX_SAMPLES;
  /* the global stream: y = uniform(size=n) (stepped over here, drawn again below), then the two estimator seeds */
  mt_seed(s.mt, seed);
  for (int i = 0; i < 2 * n; i++) mt_next(s.mt);
  uint32_t est_seed[N_TREES], rstate[N_TREES];
  for (int t = 0; t < N_TREES; t++) est_seed[t] = mt_bounded(s.mt, 0x7FFFFFFEu);
  for (int t = 0; t < N_TREES; t++) {
    mt_seed(s.mt, est_seed[t]);
    const uint32_t tree_seed = mt_bounded(s.mt, 0x7FFFFFFEu); /* _set_random_states */
    mt_seed(s.mt, tree_seed);
    rstate[t] = mt_bounded(s.mt, CYG_RAND_R_MAX - 1u); /* Splitter.init: randint(0, RAND_R_MAX) */
    draw_rows(s, t, n, est_seed[t]);
  }
  /* y again, kept for the selected rows only */
  mt_seed(s.mt, seed);
  int at[N_TREES] = {0, 0};
  for (int i = 0; i < n; i++) {
    const double d = mt_double(s.mt);
    for (int t = 0; t < N_TREES; t++)
      if (at[t] < s.ms && s.rows[t][at[t]] == i) s.u.t.y[t][at[t]++] = d;
  }
  for (int t = 0; t < N_TREES; t++) {
    for (int k = 0; k < s.ms; k++) s.rec[k] = ring[((n_logs - (uint32_t)n) + s.rows[t][k]) % log_cap];
    build_tree(s, t, rstate[t], slot + CYG_DET_TREE0 + t * CYG_DET_TREE_STRIDE);
  }
  slot[0] = (uint32_t)s.n_leaves[1];
}

/* Verdict words [w0, w0 + nlanes, ...) of the table: bit l0 * L1 + l1 is set when 2 ** -q > 0.5 (predict == -1, "A"),
 * q = (lv0 + lv1) / (2 c(max_samples)).  numpy's power gives 2 ** -q > 0.5 exactly when q <= 1 - 2**-52, so no exp2 is
 * evaluated; a zero denominator (max_samples = 1) makes q = 1 (np.divide's `where`). */
CYG_HD void verdict_words(const Scratch& s, uint32_t* slot, int lane, int nlanes) {
  const int L0 = s.n_leaves[0], L1 = s.n_leaves[1];
  const double den = dmul(2.0, avg_path_length(s.ms));
  const double qmax = bitsd(0x3FEFFFFFFFFFFFFEull); /* 1 - 2**-52 */
  const int nbits = L0 * L1, nwords = (nbits + 31) >> 5;
  for (int w = lane; w < nwords; w += nlanes) {
    uint32_t bits = 0;
    if (den != 0.0) {
      int l0 = (32 * w) / L1, l1 = (32 * w) % L1;
      for (int b = 0; b < 32 && 32 * w + b < nbits; b++) {
        const double q = ddiv(dadd(s.u.t.lv[0][l0], s.u.t.lv[1][l1]), den);
        if (q <= qmax) bits |= 1u << b;
        if (++l1 == L1) { l1 = 0; l0++; }
      }
    }
    slot[CYG_DET_TABLE + w] = bits;
  }
}

/* One whole fit on one thread (the host build; the kernel splits the same calls over a warp). */
CYG_HD void fit_slot(Scratch& s, const uint32_t* ring, uint32_t log_cap, uint32_t n_logs, uint32_t seed, uint32_t* slot) {
  for (int i = 0; i < CYG_DET_WORDS; i++) slot[i] = 0;
  fit_serial(s, ring, log_cap, n_logs, seed, slot);
  verdict_words(s, slot, 0, 1);
}

}  // namespace iforest
}  // namespace cyg
#endif /* CYG_IFOREST_CUH */
