/*
 * cyg_emu_iforest.cpp -- host build of the DEVICE detector fit cygym_b200/csrc/cyg_iforest.cuh (TEST INFRASTRUCTURE).
 *
 * Compiles the fit the CUDA kernel runs with g++ and exposes one fit and numpy's stream primitives as restated there,
 * so that the CPU-only build container can compare them with scikit-learn and numpy (tests/test_detector_fit.py).
 * It is never loaded by the product package.
 */
#include <stdint.h>

#include "../../cygym_b200/csrc/cyg_iforest.cuh"

using namespace cyg;

extern "C" {
/* One detector fit (cyg_fit_detectors for one env): the ring holds n_logs records at i % log_cap -> slot [CYG_DET_WORDS]. */
int emu_fit_detector(const uint32_t* ring, uint32_t log_cap, uint32_t n_logs, uint32_t seed, uint32_t* slot) {
  const uint32_t n = n_logs < (uint32_t)CYG_DET_WINDOW ? n_logs : (uint32_t)CYG_DET_WINDOW;
  if (n == 0 || n > log_cap) return CYG_E_INVAL;
  static iforest::Scratch s;
  iforest::fit_slot(s, ring, log_cap, n_logs, seed, slot);
  return 0;
}
/* numpy's legacy stream after seed(seed): ops[i] = (kind, arg) -- kind 0: one uniform(); 1: randint(0, arg + 1) on the
 * 32-bit path (mt_bounded(arg)); 2: permutation(arg) (arg outputs).  Outputs go to out[], their count is returned. */
int emu_np_stream(uint32_t seed, const int64_t* ops, int n_ops, double* out) {
  static iforest::MT mt;
  static uint16_t perm[65536];
  iforest::mt_seed(mt, seed);
  int k = 0;
  for (int i = 0; i < n_ops; i++) {
    const int64_t kind = ops[2 * i], arg = ops[2 * i + 1];
    if (kind == 0) out[k++] = iforest::mt_double(mt);
    else if (kind == 1) out[k++] = (double)iforest::mt_bounded(mt, (uint32_t)arg);
    else {
      for (int j = 0; j < arg; j++) perm[j] = (uint16_t)j;
      for (int j = (int)arg - 1; j >= 1; j--) {
        const uint32_t r = iforest::mt_bounded(mt, (uint32_t)j);
        const uint16_t v = perm[j]; perm[j] = perm[r]; perm[r] = v;
      }
      for (int j = 0; j < arg; j++) out[k++] = perm[j];
    }
  }
  return k;
}
}
