// Host-side sequencing of one frame of the atmosphere (OOPAO/Atmosphere.py:350-428, `update`): which layers take an add_row
// this frame and in which direction, window origins and canvas re-centring, generator counters, the sub-pixel tap
// weights — then the launches themselves, through the same entry points the Python layer uses.  The arithmetic is that of
// rlao_b200/Atmosphere.py (_plan_layer, _update_layers, _extrude_group, _publish), which stays the path for injected /
// host-generated innovations; both work on the SAME state block (aoenv_atm_state_t is shared with Python through ctypes),
// so the two can be mixed freely.  What this buys is host time: ~10 launches per frame cost ~70-100 us of interpreter
// work, a few us here — the difference is the whole step when the batch is small.
#include <math.h>
#include <string.h>

#include "common.cuh"

using namespace aoenv;

namespace {

struct Step { int sx, sy; };

inline double sign_of(double v) { return v > 0 ? 1.0 : (v < 0 ? -1.0 : 0.0); }

// Atmosphere.py:350-404 (integer part of updateLayer): the add_row steps of one layer for this frame, in order
int plan_layer(const aoenv_atm_state_t& st, aoenv_layer_state_t& ly, Step* steps, int max_steps) {
  int count = 0;
  if (ly.vX == 0.0 && ly.vY == 0.0) return 0;
  if (ly.not_done_once) {
    ly.not_done_once = 0;
    ly.ratio[0] = ly.vX * st.sampling_time / st.ps_loop;
    ly.ratio[1] = ly.vY * st.sampling_time / st.ps_loop;
    ly.buff[0] = ly.buff[1] = 0.0;
  }
  double a[2] = {fabs(ly.ratio[0]), fabs(ly.ratio[1])};
  long n[2];
  for (int k = 0; k < 2; ++k) n[k] = isinf(a[k]) ? 0 : (long)a[k];
  const double sg[2] = {sign_of(ly.ratio[0]), sign_of(ly.ratio[1])};
  const long nmin = n[0] < n[1] ? n[0] : n[1], nmax = n[0] < n[1] ? n[1] : n[0];
  for (long r = 0; r < nmin && count < max_steps; ++r) steps[count++] = {(int)sg[0], (int)sg[1]};
  for (long r = 0; r < nmax - nmin && count < max_steps; ++r)
    steps[count++] = {n[0] == nmin ? 0 : (int)sg[0], n[1] == nmin ? 0 : (int)sg[1]};
  if (nmax > max_steps) return -1;
  for (int k = 0; k < 2; ++k) ly.buff[k] += fmod(fabs(ly.ratio[k]), 1.0) * sg[k];
  if (fabs(ly.buff[0]) >= 1.0 || fabs(ly.buff[1]) >= 1.0) {
    if (count >= max_steps) return -1;
    steps[count++] = {fabs(ly.buff[0]) < 1.0 ? 0 : (int)sign_of(ly.buff[0]), fabs(ly.buff[1]) < 1.0 ? 0 : (int)sign_of(ly.buff[1])};
  }
  for (int k = 0; k < 2; ++k) ly.buff[k] = fmod(fabs(ly.buff[k]), 1.0) * sign_of(ly.buff[k]);
  return count;
}

inline int pick_origin(double v, int S, int align) {
  const int o = v > 0 ? S : (v < 0 ? 0 : S / 2);
  return o / align * align;
}

inline float* window(const aoenv_atm_state_t& st, int i, int buf, int oy, int ox) {
  return (float*)st.maps[i][buf] + ((size_t)oy * st.pitch + ox);
}

// tools/vonkarman.py cubic_tap_weights: first tap offset and the four weights of the shift by `buff` pixels
void tap_weights(double buff, int kernel, int* off, float* w) {
  const double f = floor(-buff), frac = -buff - f;
  *off = (int)f - 1;
  double x, v[4];
  if (kernel == 0) {          // scikit-image 0.18.3: cubic through four equispaced nodes, argument (r - first tap) / 3
    x = (frac + 1.0) / 3.0;
    v[0] = 1.0 + x * (-5.5 + x * (9.0 + x * -4.5));
    v[1] = x * (9.0 + x * (-22.5 + x * 13.5));
    v[2] = x * (-4.5 + x * (18.0 + x * -13.5));
    v[3] = x * (1.0 + x * (-4.5 + x * 4.5));
  } else {                    // Catmull-Rom (scikit-image >= 0.19)
    x = frac;
    v[0] = 0.5 * x * (-1.0 + x * (2.0 - x));
    v[1] = 1.0 + 0.5 * x * x * (-5.0 + 3.0 * x);
    v[2] = 0.5 * x * (1.0 + x * (4.0 - 3.0 * x));
    v[3] = 0.5 * x * x * (x - 1.0);
  }
  for (int k = 0; k < 4; ++k) w[k] = (float)v[k];
}

int extrude_group(aoenv_atm_state_t& st, const int* layers, const Step* steps, int G, const void* w_planes, void* stream) {
  const void* wins[AOENV_MAX_LAYERS];
  int32_t sxs[AOENV_MAX_LAYERS], sys_[AOENV_MAX_LAYERS];
  uint64_t seeds[AOENV_MAX_LAYERS], ids[AOENV_MAX_LAYERS];
  const int S = st.S;
  for (int g = 0; g < G; ++g) {
    const int i = layers[g];
    aoenv_layer_state_t& ly = st.layer[i];
    const int sx = steps[g].sx, sy = steps[g].sy;
    if (!(0 <= ly.org[0] - sy && ly.org[0] - sy <= S && 0 <= ly.org[1] - sx && ly.org[1] - sx <= S)) {
      const int foy = pick_origin(ly.vY, S, 1), fox = pick_origin(ly.vX, S, 4);
      int rc = aoenv_atm_compact(window(st, i, ly.cur, ly.org[0], ly.org[1]), window(st, i, 1 - ly.cur, foy, fox), st.B, st.M,
                                 st.pitch, st.env_stride, (uint64_t*)st.ext[i],
                                 (int64_t)(foy - ly.org[0]) * st.pitch + (fox - ly.org[1]), stream);
      if (rc) return rc;
      ly.cur = 1 - ly.cur;
      ly.org[0] = foy;
      ly.org[1] = fox;
      if (!(0 <= foy - sy && foy - sy <= S && 0 <= fox - sx && fox - sx <= S))
        return fail(-2, "atm_update: canvas slack too small for this wind direction change");
    }
    wins[g] = window(st, i, ly.cur, ly.org[0], ly.org[1]);
    sxs[g] = sx;
    sys_[g] = sy;
    seeds[g] = ly.philox_seed;
    ids[g] = ((ly.events << 8) | (uint64_t)i) + (st.env_offset << 40);
    ly.events += 1;
  }
  const bool tc = st.use_tc && G * st.B > AOENV_SKINNY_MAX_ROWS;       // a few rows: exact FP32, one warp per ring pixel
  int rc = aoenv_atm_gather_multi(wins, sxs, sys_, seeds, ids, G, st.B, st.M, st.pitch, st.env_stride, (const int32_t*)st.inner_rc,
                                  st.nI, st.nO, nullptr, tc ? nullptr : (float*)st.zx, st.ldz, tc ? st.zx_planes : nullptr,
                                  st.parts, stream);
  if (rc) return rc;
  if (tc)
    rc = aoenv_gemm_tn_tc(st.zx_planes, w_planes, st.ldz, st.parts, (float*)st.X, st.ldx, G * st.B, st.nO, st.ldz, 1.0f, stream);
  else
    rc = aoenv_gemm_tn((const float*)st.zx, st.ldz, (const float*)st.w_f32, st.ldz, (float*)st.X, st.ldx, G * st.B, st.nO, st.ldz,
                       1.0f, stream);
  if (rc) return rc;
  void* wins2[AOENV_MAX_LAYERS];
  int64_t offs[AOENV_MAX_LAYERS];
  void* exts[AOENV_MAX_LAYERS];
  for (int g = 0; g < G; ++g) {
    aoenv_layer_state_t& ly = st.layer[layers[g]];
    ly.org[0] -= steps[g].sy;
    ly.org[1] -= steps[g].sx;
    wins2[g] = window(st, layers[g], ly.cur, ly.org[0], ly.org[1]);
    offs[g] = (int64_t)ly.org[0] * st.pitch + ly.org[1];
    exts[g] = st.ext[layers[g]];
  }
  return aoenv_atm_ring_multi(wins2, offs, exts, G, st.B, st.M, st.pitch, st.env_stride, st.nO, (const float*)st.X, st.ldx,
                              (int32_t*)st.flag, 0, stream);
}

}  // namespace

extern "C" {

int aoenv_atm_update(aoenv_atm_state_t* state, const void* w_planes, float* opd_out, void* stream) {
  AOENV_CHECK_ARG(state != nullptr && opd_out != nullptr, "atm_update: null state / output");
  aoenv_atm_state_t& st = *state;
  const int L = st.nLayer;
  AOENV_CHECK_ARG(L >= 1 && L <= AOENV_MAX_LAYERS && st.group_max >= 1, "atm_update: %d layers", L);
  AOENV_CHECK_ARG(!st.use_tc || w_planes != nullptr, "atm_update: the operator planes are missing");
  constexpr int kMaxSteps = 64;
  static thread_local Step plans[AOENV_MAX_LAYERS][kMaxSteps];
  int count[AOENV_MAX_LAYERS], rounds = 0;
  for (int i = 0; i < L; ++i) {
    count[i] = plan_layer(st, st.layer[i], plans[i], kMaxSteps);
    if (count[i] < 0) return fail(-2, "atm_update: more than %d add_row steps in one frame (layer %d)", kMaxSteps, i);
    if (count[i] > rounds) rounds = count[i];
  }
  // the r-th add_row of every layer that has one this frame goes through one gather / GEMM / ring sequence
  for (int r = 0; r < rounds; ++r) {
    int layers[AOENV_MAX_LAYERS], G = 0;
    Step steps[AOENV_MAX_LAYERS];
    for (int i = 0; i < L; ++i)
      if (count[i] > r) {
        layers[G] = i;
        steps[G++] = plans[i][r];
      }
    for (int k = 0; k < G; k += st.group_max) {
      const int g = G - k < st.group_max ? G - k : st.group_max;
      const int rc = extrude_group(st, layers + k, steps + k, g, w_planes, stream);
      if (rc) return rc;
    }
  }
  // sub-pixel shift of every layer + weighted sum (Atmosphere.py:406-407,439-478)
  const float* canv[AOENV_MAX_LAYERS];
  const uint64_t* exts[AOENV_MAX_LAYERS];
  int32_t org[2 * AOENV_MAX_LAYERS], roff[AOENV_MAX_LAYERS], coff[AOENV_MAX_LAYERS];
  float wr[4 * AOENV_MAX_LAYERS], wc[4 * AOENV_MAX_LAYERS];
  for (int i = 0; i < L; ++i) {
    const aoenv_layer_state_t& ly = st.layer[i];
    canv[i] = (const float*)st.maps[i][ly.cur];
    exts[i] = (const uint64_t*)st.ext[i];
    org[2 * i] = ly.org[0];
    org[2 * i + 1] = ly.org[1];
    tap_weights(ly.buff[0], st.warp_kernel, &coff[i], &wc[4 * i]);      // x -> columns
    tap_weights(ly.buff[1], st.warp_kernel, &roff[i], &wr[4 * i]);      // y -> rows
  }
  return aoenv_atm_phase(canv, exts, org, L, st.B, st.R, st.M, st.Mc, st.pitch, st.fp_off, roff, coff, wr, wc, st.weight,
                         st.opd_scale, opd_out, stream);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// The rest of env.step for the Shack-Hartmann / integrator configuration, as one call: spots (with the DM surface
// evaluated in place) -> slopes -> reconstruction -> observation, reward, Strehl -> command update -> T = C gx of the new
// command.  Exactly the entry points rlao_b200/OOPAOEnv/OOPAOEnvRazor.py calls one by one (OOPAOEnvRazor.py:474-514 of
// the reference), in the same order on the same stream.
// ---------------------------------------------------------------------------------------------------------
extern "C" int aoenv_sh_step(const aoenv_sh_step_t* c, int parts, const float* opd_a, const float* dm_rows_cur,
                             const aoenv_detector_t* det, const float* action, float* coefs_next, float* dm_rows_next,
                             float* obs, float* reward, float* strehl, float* total, float* residual, void* stream) {
  AOENV_CHECK_ARG(c != nullptr && parts >= 1 && parts <= 7, "sh_step: bad arguments");
  AOENV_CHECK_ARG(!(parts & 1) || (opd_a != nullptr && dm_rows_cur != nullptr), "sh_step: null wavefront argument");
  AOENV_CHECK_ARG(!(parts & 2) || (obs != nullptr && reward != nullptr && strehl != nullptr), "sh_step: null output argument");
  AOENV_CHECK_ARG(!(parts & 4) || (action != nullptr && coefs_next != nullptr && dm_rows_next != nullptr), "sh_step: null command argument");
  const bool tc = c->use_tc && c->B > AOENV_SKINNY_MAX_ROWS;
  int rc = 0;
  if ((parts & 1) && c->geometric) {  // geometric slopes (DM surface in place)
    aoenv_dm_sep_t dm = c->dm;
    dm.rows = dm_rows_cur;
    rc = aoenv_shwfs_geometric(opd_a, nullptr, &dm, (const float*)c->pupil, (const float*)c->amp, (const int32_t*)c->valid_idx,
                               c->nV, c->B, c->nS, c->n, c->phase_scale, c->inv_units, (float*)c->slopes, c->lds,
                               tc ? c->slope_planes : nullptr, 2, (double*)c->stats, stream);
    if (rc) return rc;
  } else if (parts & 1) {           // spots (DM surface in place) + slopes
    aoenv_dm_sep_t dm = c->dm;
    dm.rows = dm_rows_cur;
    rc = aoenv_shwfs_frame_dm(opd_a, nullptr, &dm, (const int32_t*)c->order, (const float*)c->pupil, (const float*)c->amp,
                              (const uint8_t*)c->valid, c->B, c->nS, c->n, c->phase_scale, det, 0, (float*)c->frame,
                              (int32_t*)c->envmax, (double*)c->stats, stream);
    if (rc) return rc;
    rc = aoenv_shwfs_slopes((const float*)c->frame, (const int32_t*)c->envmax, 0, (const int32_t*)c->valid_idx, c->nV,
                            (const float*)c->ref_xy, c->inv_units, c->threshold_cog, c->B, c->nS, c->n, (float*)c->slopes, c->lds,
                            tc ? c->slope_planes : nullptr, 2, stream);
    if (rc) return rc;
  }
  if (parts & 2) {                  // reconstruction + observation / reward / Strehl
    if (tc)
      rc = aoenv_gemm_tn_tc(c->slope_planes, c->rec_planes, c->lds, c->rec_parts, (float*)c->rec, c->ldr, c->B, c->nA, c->lds,
                            1.0f, stream);
    else
      rc = aoenv_gemm_tn((const float*)c->slopes, c->lds, (const float*)c->rec_f32, c->lds, (float*)c->rec, c->ldr, c->B, c->nA,
                         c->lds, 1.0f, stream);
    if (rc) return rc;
    rc = aoenv_observe((const float*)c->rec, c->ldr, (const int32_t*)c->act_idx, c->B, c->nA, c->nAct2, (const double*)c->stats,
                       c->n_pupil, c->phase_scale, obs, reward, strehl, total, residual, stream);
    if (rc) return rc;
  }
  if (parts & 4) {                  // command update + T = C gx of the new command
    rc = aoenv_command_update(action, (const int32_t*)c->act_idx, c->B, c->nA, c->nAct2, c->leak, coefs_next, (float*)c->dm_prev,
                              c->ldc, stream);
    if (rc) return rc;
    rc = aoenv_dm_rows(coefs_next, c->ldc, (const int32_t*)c->act_pos, c->nA, c->nAct, c->dm.nActP, (const float*)c->wx,
                       (const int32_t*)c->j0x, c->W, c->B, c->nS * c->n, dm_rows_next, stream);
  }
  return rc;
}
