/* stub, see Rinternals.h in this directory: R's RNG entry points (R_ext/Random.h).  The stand-in RNG lives here, in the
 * translation unit that includes it: a 64-bit LCG started at a fixed state replaces R's Mersenne twister, so a sequence
 * of draws is reproducible from the state below (tests/test_gpu_dosage.py restates it). */
#ifndef STUB_R_EXT_RANDOM_H
#define STUB_R_EXT_RANDOM_H
static unsigned long long minir_rng_state = 20251017ull;
static inline void GetRNGstate(void) {}
static inline void PutRNGstate(void) {}
static inline double unif_rand(void) {
  minir_rng_state = minir_rng_state * 6364136223846793005ull + 1442695040888963407ull;
  return (double)(minir_rng_state >> 11) * (1.0 / 9007199254740992.0);
}
#endif
