/* r3d_snapshot_oracle.h -- TEST INFRASTRUCTURE ONLY: the CPU restatement of the energy snapshots (include/r3d_gpu.h,
 * r3d_set_snapshots).  Same layouts as r3d_fetch_snapshots and r3d_test_advance_time. */
#ifndef R3D_SNAPSHOT_ORACLE_H_
#define R3D_SNAPSHOT_ORACLE_H_
#include "r3d_gpu.h"
#include "r3d_oracle.h"
#ifdef __cplusplus
extern "C" {
#endif

/* R3D_EINVAL for what r3d_set_snapshots rejects (here also s == NULL and n_times == 0: nothing to compute); 0 otherwise,
 * with the voxel count in *n_vox (may be NULL) */
int r3d_oracle_check_snapshots(const r3d_model_desc *d, const r3d_snapshot_desc *s, uint64_t *n_vox);

/* Trace phonons [first, first+n) as r3d_oracle_run does and ACCUMULATE their snapshot records into energy / count
 * [n_times][dims[2]][dims[1]][dims[0]][2] and outside_energy / outside_count [n_times][2] (any may be NULL); finals (may
 * be NULL) receives the n end states.  Returns 0, R3D_EINVAL (see r3d_oracle_check_snapshots) or R3D_ENOMEM. */
int r3d_oracle_run_snapshots(const r3d_model_desc *d, uint64_t first, uint64_t n, uint64_t seed, const r3d_snapshot_desc *s,
                             double *energy, uint64_t *count, double *outside_energy, uint64_t *outside_count,
                             r3d_phonon_final *finals);

/* r3d_test_advance_time's rows: in[i] = {cell, type, x,y,z, theta, phi, dt}; out[i] as r3d_test_advance */
void r3d_oracle_advance_time(const r3d_model_desc *d, const double *in, uint32_t n, double *out);

#ifdef __cplusplus
}
#endif
#endif
