/* sweep_run.c — a plain C caller of lbft_create_sweep: 96 four-author instances over three parameter sets (the reference's
 * defaults, uniform delays, a silent node with another pacemaker), interleaved.  Prints one line per instance
 * ("inst <i> <set> <commit counts> <state keys>") for the test to check against the oracle, then "sweep ok". */
#include <stdio.h>
#include <string.h>

#include "lbft.h"

#define I 96
#define N 4

static int fail(const char* what, int rc) {
  printf("%s failed (%d): %s\n", what, rc, lbft_last_error());
  return 1;
}

int main(void) {
  uint64_t seeds[I];
  uint32_t set_of[I];
  for (uint32_t i = 0; i < I; i++) {
    seeds[i] = 500 + i;
    set_of[i] = (i * 7 + i / 5) % 3;
  }
  lbft_param_set sets[3];
  memset(sets, 0, sizeof sets);
  for (int k = 0; k < 3; k++) {
    sets[k].struct_size = sizeof(lbft_param_set);
    sets[k].delay_kind = LBFT_DELAY_LOGNORMAL;
    sets[k].delay_mean = 10.0;
    sets[k].delay_variance = 4.0;
    sets[k].target_commit_interval = 100000;
    sets[k].delta = 20;
    sets[k].gamma = 2.0;
    sets[k].lambda = 0.5;
  }
  sets[1].delay_kind = LBFT_DELAY_UNIFORM;
  sets[1].delay_lo = 2;
  sets[1].delay_hi = 12;
  sets[2].silent_mask = 1u << 3;
  sets[2].delta = 30;
  lbft_config c;
  memset(&c, 0, sizeof c);
  c.struct_size = sizeof(lbft_config);
  c.num_instances = I;
  c.num_nodes = N;
  c.seeds = seeds;
  c.max_clock = 1000;
  c.commands_per_epoch = 30000;
  lbft_sim* sim = NULL;
  int rc = lbft_create_sweep(&c, sets, 3, set_of, &sim);
  if (rc) return fail("lbft_create_sweep", rc);
  if ((rc = lbft_run(sim))) return fail("lbft_run", rc);
  uint32_t counts[I * N];
  uint64_t states[I * N];
  if ((rc = lbft_commit_counts(sim, counts))) return fail("lbft_commit_counts", rc);
  if ((rc = lbft_last_states(sim, states))) return fail("lbft_last_states", rc);
  for (uint32_t i = 0; i < I; i++) {
    printf("inst %u %u", i, set_of[i]);
    for (int n = 0; n < N; n++) printf(" %u", counts[i * N + n]);
    for (int n = 0; n < N; n++) printf(" %llu", (unsigned long long)states[i * N + n]);
    printf("\n");
  }
  char name[128];
  if ((rc = lbft_kernel_info(sim, name, sizeof name))) return fail("lbft_kernel_info", rc);
  printf("kernel %s\n", name);
  size_t bytes = 0;
  if (lbft_snapshot_size(sim, &bytes) != LBFT_ERR_STATE) return fail("lbft_snapshot_size on a sweep handle", -1);
  lbft_destroy(sim);
  printf("sweep ok\n");
  return 0;
}
