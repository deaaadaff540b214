/* ser_internal.h -- shared between the host C side (ser_host.c) and the CUDA side (ser_kernels.cu) */
#ifndef SER_INTERNAL_H
#define SER_INTERNAL_H

#include "../../include/seriation_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

struct ser_dataset {
  int32_t N, M, nh;
  uint8_t *X;    /* N*M row-major 0/1 */
  uint8_t *hard; /* N */
  char **taxon_names; /* M or NULL */
  char **site_names;  /* N or NULL */
  int32_t *site_mn;   /* MN unit per site */
  double *site_age;   /* age in Ma per site */
  uint8_t *site_star; /* '*' flag seen in the .sites file */
};

void ser_set_error(const char *fmt, ...);

/* raw exp_data sums of one local chain: sum(-loglik), sum(exp c), sum(exp d), #samples */
int ser_run_chain_sums(ser_run *run, int32_t chain, double sums[3], int32_t *n_samples);
int ser_run_dims(const ser_run *run, int32_t *N, int32_t *M, int32_t *nh, int32_t *n_chains);
const uint8_t *ser_run_hard_flags(const ser_run *run);
int ser_run_is_manycd(const ser_run *run);
/* local index of GLOBAL chain id g on this run, -1 when the run does not hold it */
int ser_run_local_chain(const ser_run *run, int32_t g);

#ifdef __cplusplus
}
#endif
#endif
