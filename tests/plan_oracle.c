/*
 * plan_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Exports the oracle's counter-based N(0, 1) pair (noise2 of oracle/sg_oracle.c, included unchanged), the noise
 * sg_plan_sample draws (include/sg_b200.h), for a batch of counters.  Built by tests/plan_oracle.py into a
 * temporary directory with the oracle's flags: no FMA contraction.
 */
#include "sg_oracle.c"

/* z[2*j], z[2*j + 1] = noise2(seed, i[j], k) for j < n */
void sgp_noise2(uint64_t seed, const int64_t* i, int64_t n, int k, double* z) {
  for (int64_t j = 0; j < n; ++j) noise2(seed, i[j], k, z + 2 * j);
}
