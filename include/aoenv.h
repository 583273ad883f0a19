/*
 * aoenv.h — C ABI of libaoenv_b200.so: the closed-loop adaptive-optics environment step on B200 (sm_100a).
 *
 * The reference (artiom-matvei/RLAO, drl4ao + OOPAO) has no FFI: its boundary is the Python object protocol
 * (Telescope / Atmosphere / DeformableMirror / ShackHartmann / Detector objects and the gym-style
 * OOPAO.step).  rlao_b200 keeps that protocol in Python and calls the entry points below through ctypes.
 * Each entry point names the reference code it replaces (paths under /root/reference/drl4ao/:
 * OOPAO/ = AO_OOPAO/OOPAO/, MAIN/ = MAIN_CODE/).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name starts with h_ (host);
 *   - all arrays are dense row-major float32 unless stated otherwise; "B" is the number of environments
 *     stepped in lock-step on this GPU, and is always the slowest-varying (leading) dimension;
 *   - `stream` is a cudaStream_t passed as void*; no entry point synchronises the device or the stream;
 *   - the caller owns every buffer; return value 0 = success, otherwise a negative error code whose text
 *     is available (per calling thread) from aoenv_last_error().
 */
#ifndef AOENV_H_
#define AOENV_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AOENV_MAX_LAYERS 8
#define AOENV_ABI_VERSION 1

int aoenv_abi_version(void);
const char* aoenv_last_error(void);
/* Number of kernels launched by this library in the calling process since load (bench.py's gpu_launches). */
uint64_t aoenv_launch_count(void);
/* Programmatic dependent launch between the kernels of the step (default on; AOENV_PDL=0 in the environment turns it off
 * at load).  With it the next kernel of the chain is scheduled while the last wave of the current one drains.  Results are
 * bit-identical either way (the toggle exists for A/B timing and tests).  Returns the previous setting. */
int aoenv_set_pdl(int enabled);

/* ---------------------------------------------------------------------------------------------------------
 * Atmosphere — OOPAO/Atmosphere.py
 *
 * State per layer: a canvas [B][Mc][pitch] holding the reference's layer.mapShift (side M = R + 6) as a WINDOW at a
 * movable origin.  The reference shifts the whole map by one pixel at every add_row (Atmosphere.py:301-311); here the
 * window origin moves by -step instead and only the 4M-4 ring pixels are written.  A window is passed as a pointer
 * to its origin pixel plus `pitch` (floats per canvas row) and `env_stride` (floats per environment canvas).
 * `ext` [3][B][2] (uint64) tracks minimum / maximum WITH position — (monotone key of the float) << 32 | element
 * index in the canvas.  Block 0 [B][2]: the whole window, which is the clip range of skimage.warp
 * (tools/tools.py:215-217) and all that aoenv_atm_phase reads; block 1 [B][2]: the window interior (the window without
 * its outer ring), which is what survives an add_row — the ring is redrawn every time; block 2 [B][2]: entry 0 =
 * (1 << 32) | window origin at the previous add_row (0: none), from which the ring kernel knows which lines became
 * interior.
 * ------------------------------------------------------------------------------------------------------- */

/* add_row, step 1 (Atmosphere.py:303-307): gathers, for every environment, the two inner rings Z of the map
 * shifted by (sx, sy) in {-1,0,1}^2 pixels (tx = sx along columns, ty = sy along rows) into zx[b][0..nI), and
 * the innovation xi ~ N(0,1) into zx[b][nI..nI+nO): injected from `xi` [B][nO] when non-null, else Philox
 * (seed, stream_id, b).  zx rows have `ldz` floats (ldz >= nI+nO; the tail is zero-filled).  `win` is the window
 * BEFORE the shift.  inner_rc [nI][2] holds (row, col) of the inner-ring pixels in window coordinates, in the
 * reference's boolean-mask (row-major) order.  zx_planes (nullable): [parts][B][ldz] bf16, the same vector in the
 * split-bf16 operand format of aoenv_gemm_tn_tc, written in the same pass; zx may then be NULL (no float32 copy). */
int aoenv_atm_gather(const float* win, int B, int M, int pitch, int64_t env_stride, int sx, int sy,
                     const int32_t* inner_rc, int nI, int nO, const float* xi,
                     uint64_t seed, uint64_t stream_id, float* zx, int ldz, void* zx_planes, int parts, void* stream);

/* add_row, step 3 (Atmosphere.py:309-310): writes the freshly extruded outer ring X [B][ldx] (X = A Z + B xi, from
 * the GEMM on zx and the stacked operator [A | B]) on the border of `win`, the window AFTER the shift, ring pixels in
 * the order of numpy's boolean mask `outerMask` (row 0, then the (r,0),(r,M-1) pairs, then row M-1; nO = 4M-4).
 * win_offset = element index of the window origin inside the canvas.  Updates ext [3][B][2]: interior extrema whose
 * pixel is still in the interior of the new window are kept and merged with the pixels that just became interior;
 * otherwise (or when force_rescan) the environment is flagged in flag [B] and its interior is rescanned exactly; the
 * window extrema are the better of the interior's and the new ring's. */
int aoenv_atm_ring(float* win, int B, int M, int pitch, int64_t env_stride, int64_t win_offset, int nO, const float* X,
                   int ldx, uint64_t* ext, int32_t* flag, int force_rescan, void* stream);

/* The same two steps for G <= AOENV_MAX_LAYERS layers at once (the layers of one atmosphere whose add_row falls in the
 * same round of a step share the operator [A | B], so their Z / X rows stack into ONE GEMM of G*B rows):
 * wins, sx, sy, seeds, stream_ids, win_offsets, exts are HOST arrays of G per-layer values with the meaning of the
 * single-layer arguments; zx / zx_planes / X / flag / xi hold G*B rows, layer-major ((g*B + b)). */
int aoenv_atm_gather_multi(const void* const* wins, const int32_t* sx, const int32_t* sy, const uint64_t* seeds,
                           const uint64_t* stream_ids, int G, int B, int M, int pitch, int64_t env_stride,
                           const int32_t* inner_rc, int nI, int nO, const float* xi, float* zx, int ldz,
                           void* zx_planes, int parts, void* stream);
int aoenv_atm_ring_multi(void* const* wins, const int64_t* win_offsets, void* const* exts, int G, int B, int M,
                         int pitch, int64_t env_stride, int nO, const float* X, int ldx, int32_t* flag,
                         int force_rescan, void* stream);

/* Episode reset of a subset of the environments (zero-shift add_row, as after a new screen): the same two steps for the k
 * environments env_idx [k] (device, int32, distinct, each in [0, B)) of G layers at their windows' CURRENT origin.
 * Workspace row g*k + j belongs to environment env_idx[j].  The gather reads Z from that environment's window (no shift)
 * and draws xi from Philox (seeds[g]; counter = ring index, env_idx[j], stream_ids[g]): the caller keys these draws in a
 * domain of its own, so that they are none of the per-frame add_row draws.  The ring kernel writes row g*k + j of X on
 * environment env_idx[j]'s window and always rescans its extrema: all three blocks of ext [3][B][2] are exact for the
 * listed environments afterwards and untouched for the others.  flag: G*k entries. */
int aoenv_atm_gather_envs(const void* const* wins, const uint64_t* seeds, const uint64_t* stream_ids, int G,
                          const int32_t* env_idx, int k, int M, int pitch, int64_t env_stride, const int32_t* inner_rc,
                          int nI, int nO, float* zx, int ldz, void* zx_planes, int parts, void* stream);
int aoenv_atm_ring_envs(void* const* wins, const int64_t* win_offsets, void* const* exts, int G, const int32_t* env_idx,
                        int k, int B, int M, int pitch, int64_t env_stride, int nO, const float* X, int ldx, int32_t* flag,
                        void* stream);

/* Canvas re-centring: copies the window from src_win to dst_win (another canvas buffer, origin 16-byte aligned) and
 * adds pos_delta to the positions stored in ext [3][B][2]. */
int aoenv_atm_compact(const float* src_win, float* dst_win, int B, int M, int pitch, int64_t env_stride, uint64_t* ext,
                      int64_t pos_delta, void* stream);

/* Episode reset (Atmosphere.py:560-592 -> OOPAO/phaseStats.py:190-318, ft_phase_screen + ft_sh_phase_screen): S von
 * Karman screens of N x N points, written into the interior of S layer windows (dst = window row 1, column 1 of
 * environment 0; pitch floats per row, env_stride floats per environment).  N = R + 4 is not a power of two, so the
 * transform fftshift(fft2(fftshift(cn))) runs as two dense products with the DFT matrix on the tensor cores (the
 * fftshifts folded into signs), with a transposition in between; the three 3 x 3 sub-harmonic grids and the removal of
 * their mean are applied by the last kernel.  Five launches.
 *   cn = (n_re + i n_im) sqrt(PSD) del_f with n ~ N(0, 1) from Philox4x32-10 (seed; counter = stream position, screen0 + s),
 *   or from `inject` [S][2][N][N] (real-part draws then imaginary-part draws, in the reference's order) when non-null.
 *   As in the reference, the sub-harmonic coefficients reuse the first 54 positions of the real-part stream
 *   (phaseStats.py:268,272 seed both generators alike).
 *   amp [N][N] = sqrt(PSD) del_f (-1)^(a+b);  wa_planes: split-bf16 planes [parts][2N][Kp] of
 *   [[Wr, -Wi], [Wi, Wr]], W[y][a] = (-1)^y exp(-2 pi i y a / N);  wb_planes: [parts][N][Kp] of [Wr | -Wi];  Kp >= 2N, % 16.
 *   sh_ex / sh_ey: float2 [3][2][N] = exp(2 pi i g x), g in {-1/(3^p D), 0}; h_amp [3][2][2], h_mx / h_my [3][2][2] (HOST):
 *   sub-harmonic amplitudes sqrt(PSD) df and the grid means of sh_ex / sh_ey.
 *   Workspaces (caller-owned): work_planes bf16 [parts][S*N][Kp], work_a [S*N][lda >= 2N], work_b [S*N][ldb >= N]. */
int aoenv_vk_screens(uint64_t seed, uint32_t screen0, int S, int N, const float* amp, const float* inject, const void* wa_planes,
                     const void* wb_planes, int Kp, int parts, const float* sh_ex, const float* sh_ey, const float* h_amp,
                     const float* h_mx, const float* h_my, void* work_planes, float* work_a, int lda, float* work_b, int ldb,
                     float* dst, int pitch, int64_t env_stride, void* stream);

/* aoenv_vk_screens for a list of environments: screen s is drawn from Philox stream screen0 + env_idx[s] (the stream
 * aoenv_vk_screens gives environment env_idx[s] when it draws the whole batch from screen0) and written into the window
 * interior of environment env_idx[s] (dst = row 1, column 1 of environment 0's window).  env_idx [S]: device int32,
 * distinct.  No injected draws; workspaces as above, sized for S screens. */
int aoenv_vk_screens_envs(uint64_t seed, uint32_t screen0, const int32_t* env_idx, int S, int N, const float* amp,
                          const void* wa_planes, const void* wb_planes, int Kp, int parts, const float* sh_ex,
                          const float* sh_ey, const float* h_amp, const float* h_mx, const float* h_my, void* work_planes,
                          float* work_a, int lda, float* work_b, int ldb, float* dst, int pitch, int64_t env_stride,
                          void* stream);

/* updateLayer tail + fill_phase_support + set_OPD (Atmosphere.py:406-407,439-450,474-478): for each layer the
 * bicubic (4x4 tap) sub-pixel shift of the map, clipped to the map's [min,max], cropped to the R x R pupil
 * footprint, weighted by sqrt(fractionalR0) and summed; opd_out [B][R][R] = sum * opd_scale (lambda/2pi).
 * h_canvas / h_ext: host arrays of nLayer device pointers (canvas base [B][Mc][pitch], extrema); h_org [nLayer][2] =
 * window origin (row, col) in each canvas.  h_row_off / h_col_off: first tap offset relative to the output pixel's own
 * window row / column (tap k reads window row i + fp_off + h_row_off[l] + k).  h_wrow / h_wcol [nLayer][4]: tap
 * weights (computed by the host in float64 from layer.buff).  h_weight [nLayer] = sqrt(fractionalR0).
 * fp_off = window index of footprint pixel 0 (3 for fov = 0).  The input windows are staged with TMA box loads. */
int aoenv_atm_phase(const float* const* h_canvas, const uint64_t* const* h_ext, const int32_t* h_org, int nLayer, int B,
                    int R, int M, int Mc, int pitch, int fp_off, const int32_t* h_row_off, const int32_t* h_col_off,
                    const float* h_wrow, const float* h_wcol, const float* h_weight, float opd_scale, float* opd_out,
                    void* stream);
/* aoenv_atm_phase for the k environments env_idx [k] (device int32, each in [0, B)) of the batch of B: writes their rows of
 * opd_out [B][R][R] only, with the same per-environment arithmetic (bit for bit what aoenv_atm_phase writes there). */
int aoenv_atm_phase_envs(const float* const* h_canvas, const uint64_t* const* h_ext, const int32_t* h_org, int nLayer,
                         int B, int R, int M, int Mc, int pitch, int fp_off, const int32_t* h_row_off,
                         const int32_t* h_col_off, const float* h_wrow, const float* h_wcol, const float* h_weight,
                         float opd_scale, const int32_t* env_idx, int k, float* opd_out, void* stream);

/* One frame of Atmosphere.update() (OOPAO/Atmosphere.py:350-428) sequenced on the host side of the library instead of by
 * the Python layer: per layer the add_row steps of this frame (integer part of updateLayer), canvas re-centring, the
 * grouped gather / GEMM / ring launches above, then aoenv_atm_phase with the tap weights of the sub-pixel remainders.
 * `state` is shared with the caller (rlao_b200/Atmosphere.py maps it with ctypes and keeps using it for the paths that
 * inject innovations); it is read AND updated: ratio / buff / not_done_once / events / cur / org.
 *   ratio, buff: pixels per frame and accumulated sub-pixel shift along (x = columns, y = rows); vX, vY wind (m/s);
 *   events: add_row count so far (Philox stream id); cur: canvas buffer in use; org: window origin (row, col).
 *   maps[l][2]: the two canvas buffers [B][Mc][pitch] of layer l; ext[l]: extrema [3][B][2]; S: canvas slack (Mc = M + S);
 *   zx / zx_planes / X / flag: the add_row workspaces for group_max * B rows; w_f32 [nO][ldz]: [A | B] (SIMT back end,
 *   use_tc = 0); w_planes (argument: it is rebuilt when r0 changes): its split-bf16 planes [parts][nO][ldz];
 *   weight[l] = sqrt(fractionalR0); warp_kernel: 0 = scikit-image 0.18.3 cubic, 1 = Catmull-Rom. */
typedef struct {
  double ratio[2];
  double buff[2];
  double vX, vY;
  uint64_t events;
  uint64_t philox_seed;
  int32_t not_done_once;
  int32_t cur;
  int32_t org[2];
} aoenv_layer_state_t;

typedef struct {
  int32_t nLayer, B, R, M, Mc, pitch, S, nI, nO, ldz, ldx, group_max, parts, fp_off, warp_kernel, use_tc;
  int64_t env_stride;
  uint64_t env_offset;
  double sampling_time, ps_loop;
  float opd_scale, reserved;
  float weight[AOENV_MAX_LAYERS];
  void* maps[AOENV_MAX_LAYERS][2];
  void* ext[AOENV_MAX_LAYERS];
  const void* inner_rc;
  void* zx;
  void* zx_planes;
  void* X;
  void* flag;
  const void* w_f32;
  aoenv_layer_state_t layer[AOENV_MAX_LAYERS];
} aoenv_atm_state_t;

int aoenv_atm_update(aoenv_atm_state_t* state, const void* w_planes, float* opd_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Dense contractions — DeformableMirror.coefs setter (OOPAO/DeformableMirror.py:534-570: OPD = modes @ coefs),
 * add_row's X = A Z + B xi (OOPAO/Atmosphere.py:308), reconstruction (MAIN/OOPAOEnv/OOPAOEnvRazor.py:496-499).
 * D[m][n] = alpha * sum_k X[m][k] * W[n][k]     (both operands K-contiguous; D row-major, ldd floats/row)
 * ------------------------------------------------------------------------------------------------------- */
/* Up to AOENV_SKINNY_MAX_ROWS rows of X (a single or a few environments) take a warp-per-column kernel in exact FP32; the
 * host layers route such products here instead of to the tensor-core kernel, whose set-up dominates at that size. */
#define AOENV_SKINNY_MAX_ROWS 8
int aoenv_gemm_tn(const float* X, int ldx, const float* W, int ldw, float* D, int ldd,
                  int M, int N, int K, float alpha, void* stream);

/* Tensor-core variant (tcgen05.mma with TMEM accumulators, TMA-fed, sm_100a) of the same contraction with FP32-grade
 * accuracy: both operands are given as `parts` (2 or 3) stacked bf16 planes x = x_0 + x_1 (+ x_2) produced by
 * aoenv_split_bf16 — Xs [parts][MX][ldk], Ws [parts][NW][ldk], ldk % 8 == 0, zero padded beyond K.  parts = 2 keeps the
 * three leading cross products (relative error ~2^-17), parts = 3 the six leading ones (~2^-24).
 * D[x][w] = alpha * sum_k X[x][k] W[w][k], D row-major with ldd floats per row. */
int aoenv_split_bf16(const float* src, int lds, int rows, int K, int parts, void* dst, int ldk, void* stream);
int aoenv_gemm_tn_tc(const void* Xs, const void* Ws, int ldk, int parts, float* D, int ldd, int MX, int NW, int K,
                     float alpha, void* stream);

/* DM surface for the reference's default geometry (DeformableMirror.py:286-305,494-514: Cartesian actuator grid,
 * axis-aligned Gaussian influence functions): modes @ coefs factorises as OPD = gy^T (C gx) with C the nAct x nAct
 * command image.  coefs [B][ldc] (valid actuators only), act_pos [nA] = row*nAct + col of each valid actuator,
 * gx / gy [nAct][R] = exp(-a (g - u0)^2) per actuator column / row, band_x / band_y [R][2] = first and last actuator
 * index kept for each pixel column / row (the rest is below float32 resolution).  opd [B][R][R] metres. */
int aoenv_dm_surface_separable(const float* coefs, int ldc, const int32_t* act_pos, int nA, int nAct, const float* gx,
                               const float* gy, const int32_t* band_x, const int32_t* band_y, const float* wx,
                               const int32_t* j0x, const float* wyp, const int32_t* i0y, int W, int B, int R, float* opd,
                               void* stream);
/* Optional banded tables (W = 12 or 16, else pass W = 0 and NULLs): wx [R][W] / j0x [R] = weights and first actuator
 * column of pixel column x; wyp [R/2][2][W] / i0y [R/2] = weights and first actuator row of the pixel-row pair
 * (2k, 2k+1).  With them the kernel runs fully unrolled on fixed-width bands. */

/* ---------------------------------------------------------------------------------------------------------
 * Shack-Hartmann WFS + detector — OOPAO/ShackHartmann.py:511-601 (and :605-674), OOPAO/Detector.py:190-301
 * ------------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t photon_noise;    /* Detector.photonNoise: Poisson(frame)                       (Detector.py:204) */
  int32_t sensor_emccd;    /* 1: gain applied before the read noise (EMCCD), else after  (:249-266)        */
  int32_t has_fwc;         /* FWC is not None: clip to [0, FWC]                           (:177-181)        */
  int32_t bits;            /* 0 = no ADC; else quantise frame/FWC*(2^bits-1), truncate    (:190-201)        */
  float qe;                /* quantum efficiency                                          (:172-174)        */
  float dark_electrons;    /* darkCurrent * integrationTime, Poisson mean per pixel       (:224-229)        */
  float fwc;
  float gain;
  float readout_noise;     /* e- rms; round(N(0,1) * RON)                                 (:218-221)        */
  uint32_t reserved;       /* stages to run, 0 = all: 1 integrate (photon noise, QE), 2 dark + full well + EM gain,
                              4 read noise + gain + ADC (long exposures: :279-301 per sub-frame, :232-276 once) */
  uint64_t seed;           /* Philox key                                                                    */
  uint64_t frame_counter;  /* advances once per call: independent draws per step                            */
} aoenv_detector_t;

/* OOPAO/Detector.py:279-301 + 232-276 (integrate + readout) applied in place to B frames of rows x cols photons
 * (the camera pass of aoenv_shwfs_frame as a stand-alone call: Poisson photon noise, QE, dark current, full well,
 * read-out noise, gain, ADC).  One Philox stream per (pixel, frame index, det->seed, det->frame_counter). */
int aoenv_detector_integrate(float* frame, int B, int rows, int cols, const aoenv_detector_t* det, void* stream);

/* The camera of the WFS as its own step: the same chain applied in place to B noise-free frames of nS x nS lenslets of
 * n x n pixels, and envmax [B] (or [1] when shared_max) = maximum over the pixels of the valid lenslets AFTER the
 * camera (the centroiding threshold of ShackHartmann.py:314-316 is taken on the detector output).  This is the second
 * half of aoenv_shwfs_frame with a detector; aoenv_shwfs_fused + this + aoenv_shwfs_slopes is the noisy step.  Any n > 0
 * (the camera works per pixel and looks up the lenslet of a pixel only for the maximum). */
int aoenv_shwfs_camera(float* frame, const uint8_t* valid, int B, int nS, int n, const aoenv_detector_t* det, int shared_max,
                       int32_t* envmax, void* stream);

/* Selects the implementation of the n = 6 frame kernel: 2 = factorised transform (radix 2 x Good-Thomas 2 x 3) on three
 * lanes per lenslet (default), 1 = the same transform on one thread per lenslet, 0 = term-by-term pruned DFT.  Same frame
 * to float32 rounding; returns the previous setting. */
int aoenv_set_wfs6_variant(int variant);

/* wfs_measure, diffractive branch up to the detector: per lenslet, the transposed n x n tile of
 * phase = (opd_a + opd_b) * pupil * phase_scale is zero-padded to 2n x 2n, multiplied by sqrt(flux) and the
 * half-pixel phasor, Fourier transformed, |.|^2 / (2n)^2, binned 2x2 -> n x n spot, written at tile (i, j) of
 * frame [B][R][R] after the detector chain `det` (det == NULL: ideal detector).  Lenslets with valid[k] == 0
 * contribute zero light (their pixels still see dark/read noise).  opd_b may be NULL.
 * amp [R][R] = sqrt(fluxMap).  envmax [B] receives max over the environment's valid-lenslet pixels (float bits
 * in a monotone int32 encoding, initialised by this call); shared_max != 0 -> one max for the whole batch in
 * envmax[0] (the interaction-matrix branch, ShackHartmann.py:659).
 * stats [B][4] (float64): sums over pupil pixels of {a, a^2, t, t^2}, a = opd_a - opd_a[centre], t = opd - opd[centre]
 * in metres (centred on the pupil-centre pixel: only variances are derived from them), for env.total /
 * env.residual / get_strehl (MAIN/OOPAOEnv/OOPAOEnvRazor.py:484,502,604-605). May be NULL.
 * n (pixels per lenslet) must be one of the compiled sizes (4, 6, 8, 10, 12).  n = 10, 12 run on n / 2 lanes per lenslet
 * and only with the default frame variant (aoenv_set_wfs6_variant(0)); another variant is rejected for them. */
int aoenv_shwfs_frame(const float* opd_a, const float* opd_b, const float* pupil, const float* amp,
                      const uint8_t* valid, int B, int nS, int n, float phase_scale,
                      const aoenv_detector_t* det, int shared_max,
                      float* frame, int32_t* envmax, double* stats, void* stream);

/* centroid + slopes (ShackHartmann.py:314-324,580-601): threshold at thr * max, first moments along the
 * lenslet map's axis 1 -> X and axis 2 -> Y, NaN/Inf -> 0, minus reference, divided by slopes_units.
 * valid_idx [nV]: lenslet numbers k = i*nS + j of the valid lenslets (row-major); ref_xy [2][nV].
 * slopes [B][lds]: first nV entries X, next nV entries Y (= wfs.signal).  slope_planes (nullable): [parts][B][lds]
 * bf16, the same vector as operand planes of aoenv_gemm_tn_tc (the reconstruction), written in the same pass.
 * n: 4, 6, 8, 10 or 12. */
int aoenv_shwfs_slopes(const float* frame, const int32_t* envmax, int shared_max, const int32_t* valid_idx,
                       int nV, const float* ref_xy, float inv_units, float threshold_cog, int B, int nS, int n,
                       float* slopes, int lds, void* slope_planes, int parts, void* stream);

/* The three steps DM surface -> lenslet spots -> slopes of one frame as ONE kernel (thread-block cluster per
 * environment; the production path of env.step): DeformableMirror.py:534-570 (separable default geometry, see
 * aoenv_dm_surface_separable), ShackHartmann.py:340-353,529-577 (ideal detector), :314-324,580-601, and the pupil
 * statistics of MAIN/OOPAOEnv/OOPAOEnvRazor.py:484,502,604-605.  Neither the DM surface nor atmosphere + DM are
 * written to memory; the camera frame only when `frame` is non-null.
 *   opd_a [B][R][R]: first OPD term (atmosphere, metres, no pupil).  Second term: either `dm` (the column half
 *   T = C gx of the separable surface from aoenv_dm_rows + the row weights) or `opd_b` [B][R][R] (any surface), or neither.
 *   pupil8 [R][R]: 1 inside the pupil (the flux must be uniform over the pupil: amp0 = sqrt(fluxMap) there).  R % 4 == 0.
 *   cluster: CTAs per environment (<= 16; > 8 needs the non-portable cluster size); CTA r owns the lenslet rows
 *   [h_row_start[r], h_row_start[r+1]) (HOST array of cluster + 1 entries, 0 ... nS).  order [cluster][rows_max * nS]
 *   (rows_max = tallest strip): lenslet ids inside each strip (row_in_strip * nS + column), the lit ones first;
 *   nlit [cluster]: how many are lit.  slot_of [nS*nS]: position of a lenslet in the valid list (= its slope index), -1
 *   if invalid.  groups: warp groups per CTA.
 *   slopes (nullable; then only the frame is produced, envmax is reset for the camera pass) / slope_planes / ref_xy /
 *   inv_units / threshold_cog / envmax / stats: as in aoenv_shwfs_slopes and aoenv_shwfs_frame, except that stats
 *   holds the plain sums {sum a, sum a^2, sum t, sum t^2} over the pupil (a = opd_a, t = opd_a + DM).
 *   n: 4, 6, 8 only (other sizes are rejected). */
typedef struct {
  const float* rows;             /* [B][nActP][R] T = C gx from aoenv_dm_rows (rows >= nAct are zero); NULL = no separable DM */
  const float* wlr;              /* [R][2 * pad4((WL+1)/2)] weights of pixel row y on the actuator rows ilr[y / n] + t, t < WL,  */
                                 /* stored as two halves of (WL+1)/2 entries, each padded to a multiple of 4 floats               */
  const int32_t* ilr;            /* [nS] first actuator row of the window of every lenslet row, non-decreasing                   */
  int32_t nActP;                 /* rows per environment in `rows` (>= nAct + WL)                                                */
  int32_t WL;                    /* window height: 14 or 18                                                                      */
  int32_t t_rows;                /* max over strips of ilr[last row] + WL - ilr[first row]                                       */
  int32_t reserved;
} aoenv_dm_sep_t;

int aoenv_shwfs_fused(const float* opd_a, const float* opd_b, const aoenv_dm_sep_t* dm, const uint8_t* pupil8, float amp0,
                      const int32_t* h_row_start, const int32_t* order, const int32_t* nlit, const int32_t* slot_of, int B,
                      int nS, int n, int cluster, int groups, float phase_scale, const float* ref_xy, int nV, float inv_units,
                      float threshold_cog, float* frame, float* slopes, int lds, void* slope_planes, int parts,
                      int32_t* envmax, double* stats, void* stream);
/* aoenv_shwfs_frame as env.step calls it.  Second OPD term: `opd_b` (a surface in memory), or `dm` (the separable DM surface
 * in factored form: T = C gx from aoenv_dm_rows + the row-weight windows; t_rows is not used), or neither.  With `dm` every
 * lenslet evaluates the surface of its own n x n pixels in registers, so DeformableMirror.py:534-570 costs one small kernel
 * per command (aoenv_dm_rows) and the [B][R][R] surface is neither written nor read (stats: the total is then centred on the
 * atmosphere's centre value — the variance is shift invariant).
 * order (nullable) [nS*nS]: a permutation of the lenslet numbers, the valid (lit) ones first: thread k works on lenslet
 * order[k], so whole warps are lit or dark and the dark ones skip the transform (21 % of the lenslets of a circular pupil).
 * The variants selected by aoenv_set_wfs6_variant ignore `dm` = NULL-only and `order`.  n: as aoenv_shwfs_frame (4, 6, 8, 10,
 * 12); WL 14 or 18 for every n (the window is counted in actuator rows, and a lenslet spans about one actuator pitch). */
int aoenv_shwfs_frame_dm(const float* opd_a, const float* opd_b, const aoenv_dm_sep_t* dm, const int32_t* order,
                         const float* pupil, const float* amp, const uint8_t* valid, int B, int nS, int n, float phase_scale,
                         const aoenv_detector_t* det, int shared_max, float* frame, int32_t* envmax, double* stats,
                         void* stream);
/* Shared memory per CTA (bytes) the kernel above needs when its tallest strip has rows_max lenslet rows, or -1 for an
 * invalid configuration (t_rows = 0: no separable DM).  The limit is 227 KB. */
int aoenv_shwfs_fused_smem(int nS, int n, int rows_max, int groups, int t_rows, int WL);
/* Column half of the separable DM surface, once per command: rows [B][nActP][R], rows[b][i][x] = sum_q C_b[i][j0x[x] + q]
 * wx[x][q] for i < nAct (C_b = command image of environment b, see aoenv_dm_surface_separable for the tables; W = 12 or
 * 16); rows i >= nAct are not written (the caller keeps them zero). */
int aoenv_dm_rows(const float* coefs, int ldc, const int32_t* act_pos, int nA, int nAct, int nActP, const float* wx,
                  const int32_t* j0x, int W, int B, int R, float* rows, void* stream);

/* env.step after the atmosphere, as one call (MAIN/OOPAOEnv/OOPAOEnvRazor.py:488-514 with a Shack-Hartmann, the separable
 * mirror evaluated in place, the integrator's command update): aoenv_shwfs_frame_dm -> aoenv_shwfs_slopes ->
 * aoenv_gemm_tn(_tc) (reconstructor) -> aoenv_observe -> aoenv_command_update -> aoenv_dm_rows, on `stream`, with the
 * arguments those entry points document.  `c` holds what does not change between steps; per call: the atmosphere OPD, the
 * T rows of the surface commanded at the previous step (dm_rows_cur), the camera description of this frame (NULL = ideal),
 * the action [B][nAct2], where the new commands and their T rows go, and the output tensors.  Host time is what this
 * saves: six interpreter-driven calls become one (the step of a single small environment is launch-bound). */
/* geometric != 0: part 1 runs aoenv_shwfs_geometric instead of aoenv_shwfs_frame_dm + aoenv_shwfs_slopes; `amp` then holds the
 * flux weights [R][R] (fluxMap, not its square root), and frame / envmax / order / ref_xy / threshold_cog / det are not used. */
typedef struct {
  int32_t B, nS, n, nV, lds, nA, nAct, nAct2, ldc, ldr, W, rec_parts, use_tc, geometric;
  float phase_scale, inv_units, threshold_cog, leak;
  double n_pupil;
  const void *pupil, *amp, *valid, *order, *valid_idx, *ref_xy;        /* aoenv_shwfs_frame_dm / aoenv_shwfs_slopes */
  void *frame, *envmax, *stats, *slopes, *slope_planes;
  aoenv_dm_sep_t dm;                                                  /* wlr, ilr, nActP, WL; rows is taken per call */
  const void *rec_planes, *rec_f32;                                   /* reconstructor [nA][lds]: bf16 planes / float32 */
  void* rec;                                                          /* [B][ldr] */
  const void* act_idx;
  void* dm_prev;
  const void *act_pos, *wx, *j0x;                                     /* aoenv_dm_rows */
} aoenv_sh_step_t;

/* parts: bit 0 = spots + slopes, bit 1 = reconstruction + observation / reward / Strehl, bit 2 = command update + T rows
 * (7 = the whole chain).  A caller that runs the next frame's atmosphere on a side stream issues it after part 1, so that
 * it fills the SMs the small kernels of the rest leave idle; a host-facing caller starts the download of the observation
 * after part 2 and waits for the uploaded action before part 4. */
int aoenv_sh_step(const aoenv_sh_step_t* c, int parts, const float* opd_a, const float* dm_rows_cur, const aoenv_detector_t* det,
                  const float* action, float* coefs_next, float* dm_rows_next, float* obs, float* reward, float* strehl,
                  float* total, float* residual, void* stream);

/* Calibration-grade measurement (init only): the two steps above in float64 with the ideal detector, for the
 * reference slopes / slope units (ShackHartmann.py:254-312) and the interaction matrix pushes
 * (calibration/InteractionMatrix.py:79-84), whose 1 nm pokes move the spots by ~1e-3 pixel.  opd [F][R][R]
 * float32 (OPD_no_pupil, metres); frame [F][R][R], slopes [F][lds], ref_xy [2][nV] float64; envmax [F] (or [1]
 * when shared_max) scratch.  n: 4, 6, 8, 10 or 12. */
int aoenv_shwfs_measure_f64(const float* opd, const float* pupil, const float* amp, const uint8_t* valid,
                            const int32_t* valid_idx, int nV, const double* ref_xy, double inv_units, double threshold_cog,
                            int F, int nS, int n, double phase_scale, int shared_max, double* frame, uint64_t* envmax,
                            double* slopes, int lds, void* stream);

/* Geometric Shack-Hartmann sensor (ShackHartmann(is_geometric=True); defined in DESIGN.md §2 as the geometric-optics limit of
 * the diffractive sensor above): per valid lenslet (i, j), the flux-weighted mean over its n x n pixels
 * [i*n, (i+1)*n) x [j*n, (j+1)*n) of the gradient of the phase (opd_a + second term) * phase_scale, taken as np.gradient
 * with unit spacing (central differences inside the R x R array, one-sided first differences on its outer rows and columns;
 * axis 1 -> X, axis 0 -> Y), times inv_units.  No reference is subtracted (a flat wavefront has zero gradient), no detector
 * runs and no threshold applies.  The OPD terms are the pupil-less ones (OPD_no_pupil): pixels just outside the pupil take
 * part in the central differences.
 *   opd_a [B][R][R]; second term: `opd_b` [B][R][R], or `dm` (the separable DM in factored form, as aoenv_shwfs_frame_dm takes
 *   it; t_rows is not used), or neither.  flux [R][R] = fluxMap (weights); pupil [R][R] (> 0 inside) for the statistics.
 *   valid_idx [nV]: ascending lenslet numbers i*nS + j of the valid lenslets.  slopes [B][lds]: X block, then Y block
 *   (= wfs.signal); slope_planes (nullable) [parts][B][lds] bf16, as aoenv_shwfs_slopes writes them; stats (nullable) [B][4]
 *   float64 with the definition of aoenv_shwfs_frame_dm (with `dm`, the total is centred on the atmosphere's centre value).
 * One CTA per (environment, strip of lenslet rows): the strip's pixel rows and a one-row halo are staged in shared memory with
 * 128-bit loads (64-bit when R % 4 != 0), the DM surface is evaluated in registers and never written; slopes are reduced
 * without atomics (deterministic).  Two launches when stats is given (its reset, then the kernel), else one.
 * n: 4, 6, 8, 10 or 12; with `dm`, WL 14 or 18. */
int aoenv_shwfs_geometric(const float* opd_a, const float* opd_b, const aoenv_dm_sep_t* dm, const float* pupil,
                          const float* flux, const int32_t* valid_idx, int nV, int B, int nS, int n, float phase_scale,
                          float inv_units, float* slopes, int lds, void* slope_planes, int parts, double* stats, void* stream);

/* Calibration-grade twin (init only: slope units, interaction-matrix pushes): the same measurement in float64 arithmetic on
 * F wavefronts opd [F][R][R] (float32, OPD_no_pupil, metres); slopes [F][lds] float64 = gradient means * phase_scale *
 * inv_units.  n: 4, 6, 8, 10 or 12. */
int aoenv_shwfs_geometric_f64(const float* opd, const float* flux, const int32_t* valid_idx, int nV, int F, int nS, int n,
                              double phase_scale, double inv_units, double* slopes, int lds, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Pyramid WFS — OOPAO/Pyramid.py:469-504 (pyramid_transform), :581-603 (modulation), :987-1002 (detector binning)
 *
 * frame [B][N/bin][N/bin] = bin x bin sums of  sum_theta | ifft2( fft2( support_theta * phasor ) * mask ) |^2, where
 * support_theta is the pupil field amp * exp(i (phase + px_theta Tip + py_theta Tilt)) zero padded to N x N (centred),
 * phase = (opd_a + opd_b) * pupil * phase_scale, Tip / Tilt = lin[x] / lin[y] * pupil (lin = linspace(-pi, pi, R)),
 * mod [nTheta][2] = (px, py), phasor = exp(-i pi (N+1)/N (x + y)).  amp [R][R] = sqrt(flux / nTheta) * reflectivity.
 * mask_s: complex64 [N][N], the pyramid mask exp(i m) with BOTH axes in the transform's digit-scrambled order: position
 * p = j1 * N2 + j2 holds frequency j1 + N1 * j2 (N = N1 * N2 = 16 * 18 or 16 * 8).  Hand-written FFT kernels (no
 * library); aoenv_pyramid_supported(N) tells whether N is a compiled size.
 * Workspaces (caller-owned): work_x1 complex64 [B][nTheta][N][R], work_yt complex64 [B][nTheta][N][N],
 * intensity float32 [B][N][N] (the un-binned sum, also an output).
 * ------------------------------------------------------------------------------------------------------- */
int aoenv_pyramid_supported(int N);
int aoenv_pyramid_frames(const float* opd_a, const float* opd_b, const float* pupil, const float* amp, const float* lin,
                         const float* mod, const float* mask_s, int B, int R, int N, int nTheta, int bin, float phase_scale,
                         float* work_x1, float* work_yt, float* intensity, float* frame, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Command update and observation — MAIN/OOPAOEnv/OOPAOEnvRazor.py:479,492-500,514,621-641
 * ------------------------------------------------------------------------------------------------------- */

/* coefs = dm_prev * leak + img_to_vec(action) * 1e-6 ; dm_prev = coefs.   action [B][nAct][nAct] (micrometres),
 * act_idx [nA]: flat index xvalid*nAct + yvalid of each valid actuator. coefs/dm_prev [B][ldc]. */
int aoenv_command_update(const float* action, const int32_t* act_idx, int B, int nA, int nAct2, float leak,
                         float* coefs, float* dm_prev, int ldc, void* stream);

/* obs = vec_to_img(-rec) * 1e6 with rec [B][ldr] = reconstructor @ signal (from aoenv_gemm_tn);
 * reward = -||obs||_2; strehl = exp(-var(phase[pupil])) ; total / residual = std(OPD[pupil]) * 1e9, from `stats`
 * (see aoenv_shwfs_frame) and n_pupil = number of pupil pixels.  obs [B][nAct2] is fully overwritten. */
int aoenv_observe(const float* rec, int ldr, const int32_t* act_idx, int B, int nA, int nAct2,
                  const double* stats, double n_pupil, float phase_scale,
                  float* obs, float* reward, float* strehl, float* total, float* residual, void* stream);

/* Exploration noise (MAIN/OOPAOEnv/OOPAOEnvRazor.py:616-619: F @ np.random.normal(0, sigma, nValidAct), as an actuator
 * image): aoenv_normal_fill draws z [rows][ld] = sigma * N(0, 1) (columns >= cols are zero) from Philox4x32-10 keyed by
 * `seed` with `counter` = the call number, as float32 and (planes non-null) as the split-bf16 operand of
 * aoenv_gemm_tn_tc; the product with F is that GEMM; aoenv_vec_to_img scatters vec [B][ldv] * scale into
 * img [B][nAct2] (zero at invalid actuators; vec_to_img of OOPAOEnvRazor.py:621-630). */
int aoenv_normal_fill(uint64_t seed, uint64_t counter, int rows, int cols, int ld, float sigma, float* out, void* planes,
                      int parts, void* stream);
int aoenv_vec_to_img(const float* vec, int ldv, const int32_t* act_idx, int B, int nA, int nAct2, float scale, float* img,
                     void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Science-path PSF Strehl — OOPAO/Telescope.py:260-360 (computePSF(zp) -> PropagateField), PSF.max()
 * The reference pads the pupil field to N = os*zp*R (os = 2 for even image sizes), takes |FFT/N|^2 and bins
 * os x os.  This entry point evaluates that PSF on the central `win` x `win` binned pixels only (pruned DFT)
 * and returns their maximum in psf_max [B]; psf_win [B][win][win] may be NULL.  Three launches: the pupil field
 * written transposed in split-bf16 form, the row transform as one tcgen05 GEMM (M = B*R, N = 2*Wu, K = 2*R,
 * Wu = os*win), the column transform + |.|^2 + binning + maximum.
 * w1_planes: bf16 [2][2*Wu][ldk], the two split-bf16 parts (aoenv_split_bf16) of the real operator
 *   [[Wr, -Wi], [Wi, Wr]], (Wr + i Wi)[u][y] = exp(-i pi (pad + y)(2 d_u + 1) / N), pad = (N-R)/2,
 *   d_u = os*((N/os)/2 - win/2) + u - N/2, columns [0,R) multiply Re(field), [R,2R) Im(field), zero padded to ldk;
 * g2: float2 [R][Wu], g2[x][v] = exp(-i pi (pad + x)(2 d_v + 1) / N);  both host-computed in float64;
 * field_planes: bf16 workspace [2][B*R][ldk] whose columns [2R, ldk) are zero; ldk % 8 == 0;
 * scratch: B*R * 2*Wu floats.
 * ------------------------------------------------------------------------------------------------------- */
int aoenv_psf_peak(const float* opd_a, const float* opd_b, const float* pupil, const float* amp,
                   const void* w1_planes, const float* g2, int B, int R, int N, int os, int win, float phase_scale,
                   void* field_planes, int ldk, float* scratch, float* psf_win, float* psf_max, void* stream);

/* The whole PSF image (tel.computePSF(zp) / computePSF(detector=cam): Telescope.py:260-360 with img_resolution = win):
 * the central win x win binned pixels, any win up to N / os.  Both transforms are tensor-core GEMMs with the operator of
 * aoenv_psf_peak (w_planes [2][2*Wu][ldk], Wu = os * win; the DFT kernel is the same along both axes), with a
 * transposition in between; five launches.  Workspaces (caller-owned): field_planes bf16 [2][B*R][ldk] (columns
 * [2R, ldk) zero), work_t [B*R][2*Wu], planes_u bf16 [2][B*Wu][ldk] (columns [2R, ldk) zero), work_f [B*Wu][2*Wu].
 * psf [B][win][win]; psf_max [B]. */
int aoenv_psf_image(const float* opd_a, const float* opd_b, const float* pupil, const float* amp, const void* w_planes, int B,
                    int R, int N, int os, int win, float phase_scale, void* field_planes, int ldk, float* work_t, void* planes_u,
                    float* work_f, float* psf, float* psf_max, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AOENV_H_ */
