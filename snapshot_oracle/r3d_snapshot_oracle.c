/* r3d_snapshot_oracle.c -- TEST INFRASTRUCTURE ONLY (never part of the product path).
 *
 * Plain-C restatement of the energy snapshots of include/r3d_gpu.h (r3d_set_snapshots): the deposit rule and the partial
 * advance to a travel time, on top of the CPU oracle.  The oracle (oracle/r3d_oracle.c) is pinned to the reference's own
 * compiled code and is included here unchanged, so that its cell geometry, draws and events are used as they are;
 * propagate_snap() below is its propagate() with the deposit before each Phonon::Move.  The reference has no snapshots, so
 * nothing pins this part to it: the exact count invariant and the ballistic case of tests/test_oracle_snapshots.py do.
 */
#include "../oracle/r3d_oracle.c"
#include "r3d_snapshot_oracle.h"

#define SNAP_NEWTON 5     /* R3D_SNAP_NEWTON of radiative3d_b200/csrc/r3d_device.cuh */

/* advance_time (r3d_device.cuh): the point at travel time dt along the move of length len_seg, time time_seg from
 * (loc, th, ph) in `cell`.  Straight rays at constant speed: len = dt v.  Curved rays: SNAP_NEWTON Newton steps on the
 * length from the proportional guess, d(time)/d(len) = 1 / v at the current end point, each kept inside [0, len_seg]. */
static travel_t advance_time(const r3d_model_desc *d, uint32_t cell, int rt, double dt, v3 loc, double th, double ph,
                             double len_seg, double time_seg) {
  const double *c = cellp(d, cell);
  double v = 0.0;
  if (d->cell_kind == R3D_CELL_CYLINDER) v = c[rt];
  else if (d->cell_kind == R3D_CELL_SHELL && c[rt] == 0) v = c[2 + rt];
  if (v > 0.0) return advance_length(d, cell, rt, dt * v, loc, th, ph);
  double len = len_seg * (dt / time_seg);
  travel_t t = advance_length(d, cell, rt, len, loc, th, ph);
  for (int i = 0; i < SNAP_NEWTON; i++) {
    len -= (t.time - dt) * veloc_at(d, cell, rt, t.loc);
    len = fmin(fmax(len, 0.0), len_seg);
    t = advance_length(d, cell, rt, len, loc, th, ph);
  }
  return t;
}

typedef struct {
  const r3d_snapshot_desc *s;
  uint64_t n_vox;
  double *energy; uint64_t *count;          /* [K][n_vox + 1][2], outside = voxel n_vox */
} snap_acc_t;

/* the records of one move of p (state before Phonon::Move) along tr: every t_k in [t_a, t_b) */
static void deposit(const r3d_model_desc *d, const snap_acc_t *S, const phonon_t *p, const travel_t *tr) {
  const double t_a = p->time, t_b = p->time + tr->time;       /* t_b: the value Phonon::Move gives p->time */
  for (uint32_t k = 0; k < S->s->n_times; k++) {
    const double tk = S->s->times[k];
    if (!(t_a <= tk && tk < t_b)) continue;
    travel_t t = advance_time(d, p->cell, p->type, tk - t_a, p->loc, p->th, p->ph, tr->len, tr->time);
    const double amp = p->amp * t.atten;
    const double x[3] = {t.loc.x, t.loc.y, t.loc.z};
    uint64_t v = 0, stride = 1;
    int inside = 1;
    for (int a = 0; a < 3; a++) {
      const double f = floor((x[a] - S->s->origin[a]) / S->s->voxel[a]);
      inside = inside && f >= 0.0 && f < (double)S->s->dims[a];
      if (inside) v += (uint64_t)f * stride;
      stride *= S->s->dims[a];
    }
    const size_t at = ((size_t)k * (S->n_vox + 1) + (inside ? v : S->n_vox)) * 2 + (size_t)p->type;
    S->energy[at] += amp * amp;
    S->count[at] += 1;
  }
}

/* propagate() of oracle/r3d_oracle.c, with deposit() before each ph_move() */
static uint32_t propagate_snap(const r3d_model_desc *d, phonon_t *p, rng_t *g, accum_t *A, const snap_acc_t *S) {
  for (;;) {
    p->iters++;
    if (p->time > d->ttl) return R3D_FATE_TIMEOUT;
    if ((p->moves % 128) == 127) {
      int why = -1;
      if (isnan(p->pathlen)) why = R3D_INV_PATH_NAN;
      else if (isnan(p->time)) why = R3D_INV_TIME_NAN;
      else if (p->pathlen < 0) why = R3D_INV_PATH_NEGATIVE;
      else if ((p->time < 0) || (p->recent < 0)) why = R3D_INV_TIME_NEGATIVE;
      else if (p->recent == 0) why = R3D_INV_STUCK;
      else if (p->recent < d->slow_concern) why = R3D_INV_SLOW;
      else if (p->moves > d->loop_concern) why = R3D_INV_LOOP_EXCEED;
      if (why >= 0) return R3D_FATE_INVALID | ((1u << why) << 8);
      p->recent = 0;
    }
    travel_t tr = path_to_boundary(d, p->cell, p->type, p->loc, p->th, p->ph);
    if (tr.len == PINF) return R3D_FATE_TIMEOUT;
    uint32_t scat = d->cell_scat[p->cell];
    double r = ((double)rng_next(g)) / (R3D_RAND_MAX + 1);
    r = 1.0 - r;
    double scatlen = -log(r) * d->scat_mfp[scat * 2 + p->type];
    if (scatlen < tr.len) {
      tr = advance_length(d, p->cell, p->type, scatlen, p->loc, p->th, p->ph);
      deposit(d, S, p, &tr);
      ph_move(p, &tr);
      double rth, rph, rpol = 0; int otype;
      if (d->no_deflect) { rth = nudge(d, 0); rph = 0; otype = p->type; }
      else {
        uint32_t conv = cdf_search(d->scat_whole_cdf + (scat * 2 + p->type) * 4, 4, rng_next(g));
        otype = conv & 1;
        uint32_t ti = cdf_search(d->scat_cdf + ((size_t)scat * 4 + conv) * d->n_toa, d->n_toa, rng_next(g));
        if (conv == 3) rpol = d->scat_spol[(size_t)scat * d->n_toa + ti];
        rth = nudge(d, d->toa_theta[ti]); rph = d->toa_phi[ti];
      }
      transform(&p->th, &p->ph, &p->pol, rth, rph, rpol);
      p->type = otype;
      p->scatters++;
      continue;
    }
    deposit(d, S, p, &tr);
    ph_move(p, &tr);
    uint8_t fl = d->face_flags[p->cell * d->faces_per_cell + tr.face];
    if (fl & R3D_FACE_COLLECT) report_collected(d, p, A);
    if (fl & R3D_FACE_REFLECT) { refraction_fullrt(d, p, tr.face, g); continue; }
    if (fl & R3D_FACE_ADJOIN) {
      uint32_t other = d->face_other_cell[p->cell * d->faces_per_cell + tr.face];
      if (fl & R3D_FACE_DISCON) refraction_fullrt(d, p, tr.face, g);
      else if (velocity_jump(d, p->cell, other, p->loc) > 0.00001) refraction_bend(d, p, tr.face);
      else p->cell = other;
      continue;
    }
    return R3D_FATE_LOST;
  }
}

/* the rejections of r3d_set_snapshots; *n_vox receives the voxel count */
int r3d_oracle_check_snapshots(const r3d_model_desc *d, const r3d_snapshot_desc *s, uint64_t *n_vox) {
  if (!d || !s || !s->n_times || s->n_times > R3D_SNAP_MAX_TIMES || !s->times) return R3D_EINVAL;
  for (uint32_t k = 0; k < s->n_times; k++) {
    const double t = s->times[k];
    if (!isfinite(t) || t < 0 || t > d->ttl) return R3D_EINVAL;
    if (k && !(t > s->times[k - 1])) return R3D_EINVAL;
  }
  uint64_t nv = 1;
  for (int a = 0; a < 3; a++) {
    if (!isfinite(s->origin[a]) || !isfinite(s->voxel[a]) || !(s->voxel[a] > 0) || !s->dims[a]) return R3D_EINVAL;
    nv *= s->dims[a];
    if (nv > R3D_SNAP_MAX_CELLS) return R3D_EINVAL;
  }
  if ((uint64_t)s->n_times * (nv + 1) * 2 > R3D_SNAP_MAX_CELLS) return R3D_EINVAL;
  if (n_vox) *n_vox = nv;
  return 0;
}

int r3d_oracle_run_snapshots(const r3d_model_desc *d, uint64_t first, uint64_t n, uint64_t seed, const r3d_snapshot_desc *s,
                             double *energy, uint64_t *count, double *outside_energy, uint64_t *outside_count,
                             r3d_phonon_final *finals) {
  uint64_t nv = 0;
  if (r3d_oracle_check_snapshots(d, s, &nv)) return R3D_EINVAL;
  const size_t cells = (size_t)s->n_times * (nv + 1) * 2;
  snap_acc_t S = {s, nv, (double *)calloc(cells, sizeof(double)), (uint64_t *)calloc(cells, sizeof(uint64_t))};
  if (!S.energy || !S.count) { free(S.energy); free(S.count); return R3D_ENOMEM; }
  accum_t A = {NULL, NULL, NULL};
  for (uint64_t i = 0; i < n; i++) {
    rng_t g = {seed, first + i, 0};
    phonon_t p;
    generate(d, &p, &g);
    uint32_t fate = propagate_snap(d, &p, &g, &A, &S);
    if (finals) {
      r3d_phonon_final *f = finals + i;
      f->time = p.time; f->pathlen = p.pathlen; f->amp = p.amp;
      f->loc[0] = p.loc.x; f->loc[1] = p.loc.y; f->loc[2] = p.loc.z;
      f->theta = p.th; f->phi = p.ph; f->pol = p.pol;
      f->moves = p.moves; f->cell = p.cell; f->type = p.type; f->fate = fate;
      f->draws = g.ordinal; f->catches = p.catches; f->scatters = p.scatters; f->iters = p.iters;
    }
  }
  /* accumulate into the caller's arrays, in the layout of r3d_fetch_snapshots */
  for (size_t k = 0; k < s->n_times; k++) {
    const size_t at = k * (nv + 1) * 2;
    for (size_t i = 0; i < nv * 2; i++) {
      if (energy) energy[k * nv * 2 + i] += S.energy[at + i];
      if (count) count[k * nv * 2 + i] += S.count[at + i];
    }
    for (int t = 0; t < 2; t++) {
      if (outside_energy) outside_energy[2 * k + t] += S.energy[at + nv * 2 + t];
      if (outside_count) outside_count[2 * k + t] += S.count[at + nv * 2 + t];
    }
  }
  free(S.energy); free(S.count);
  return 0;
}

void r3d_oracle_advance_time(const r3d_model_desc *d, const double *in, uint32_t n, double *out) {
  for (uint32_t i = 0; i < n; i++) {
    const double *x = in + 8 * i;
    const uint32_t cell = (uint32_t)x[0];
    const int rt = (int)x[1];
    const v3 loc = V(x[2], x[3], x[4]);
    const travel_t seg = path_to_boundary(d, cell, rt, loc, x[5], x[6]);
    travel_t t = advance_time(d, cell, rt, x[7], loc, x[5], x[6], seg.len, seg.time);
    t.face = -1;
    put_travel(&t, out + 9 * i);
  }
}
