// Shack-Hartmann wavefront sensor + detector (OOPAO/ShackHartmann.py:511-601, OOPAO/Detector.py:190-301),
// batched over environments.  One thread owns one lenslet: its n x n field lives in registers, the zero-padded
// 2n-point DFTs are done as two passes of constant-twiddle complex FMAs (only the n non-zero inputs are
// visited), intensities are binned 2x2 on the fly and pushed through the detector chain before the single
// store of the camera frame.
#include <stdlib.h>
#include <mutex>

#include "common.cuh"
#include "wfs_twiddles.inc"

namespace aoenv {

constexpr int kMaxN = 8;                 // pixels per lenslet side
// c_tw[u * n + a] = exp(-i pi (a + n/2) (2u + N + 1) / N),  N = 2n: the N-point DFT kernel restricted to the n
// non-zero inputs (which sit at padded positions n/2 .. n/2+n-1, ShackHartmann.py:344), times the half-pixel
// phasor exp(-i pi (N+1)/N x) of ShackHartmann.py:208-209.
__constant__ float2 c_tw[2 * kMaxN * kMaxN];
__constant__ double2 c_twd[2 * kMaxN * kMaxN];   // float64 copy for the calibration-grade kernels

// ---- per-pixel random stream: Philox counter = (pixel, env, frame_lo, frame_hi16 << 16 | block) -------------------
// Block 0 of a pixel's stream feeds the photon draw (words x, y) and the read-out normal (z, w); block 1 the dark
// current; blocks 16.. / 32.. the (rare) further attempts of the rejection sampler.  Every lane of a warp therefore
// calls the generator at the same program points — a lazily refilled buffer would refill at different call sites in
// different lanes and serialise the ten Philox rounds once per site.
struct PixelRng {
  Philox ph;
  uint32_t c0, c1, c2, c3hi;
  __device__ __forceinline__ PixelRng(uint64_t seed, uint32_t pixel, uint32_t env, uint64_t frame)
      : ph(seed), c0(pixel), c1(env), c2((uint32_t)frame), c3hi(((uint32_t)(frame >> 32)) << 16) {}
  __device__ __forceinline__ uint4 block(uint32_t i) const { return ph(c0, c1, c2, c3hi | (i & 0xffffu)); }
};

// log(k!) for the PTRS acceptance test: table below 10, Stirling's series above (error < 1e-7 relative there)
__constant__ float c_logfact[10] = {0.f, 0.f, 0.6931471806f, 1.7917594692f, 3.1780538303f, 4.7874917428f,
                                    6.5792512120f, 8.5251613611f, 10.6046029027f, 12.8018274801f};
__device__ __forceinline__ float log_factorial(float k) {
  if (k < 10.f) return c_logfact[(int)k];
  const float r = __frcp_rn(k);
  return (k + 0.5f) * __logf(k) - k + 0.9189385332f + r * (0.0833333333f - 0.00277777778f * r * r);
}

struct RcpTable { float v[64]; };
constexpr RcpTable make_rcp() {
  RcpTable t{};
  t.v[0] = 0.f;
  for (int k = 1; k < 64; ++k) t.v[k] = 1.0f / (float)k;
  return t;
}
__constant__ RcpTable c_rcp_table = make_rcp();

// n = 10, 12: only the float64 calibration kernel reads a table (their spots kernel uses literal twiddles), so they get a
// float64 table of their own, declared after the tables the n <= 8 kernels read so that those kernels' constant-bank
// offsets do not move
constexpr int kMaxWideN = 12;
__constant__ double2 c_twd_wide[2 * kMaxWideN * kMaxWideN];
template <int n>
__device__ __forceinline__ double2 twd(int i) {
  if constexpr (n <= kMaxN) return c_twd[i];
  else return c_twd_wide[i];
}
static int g_tw_n[64] = {0};             // per device: n for which c_tw / c_twd (c_twd_wide) are currently valid
static std::mutex g_tw_mutex;

static int ensure_twiddles(int n, cudaStream_t stream) {
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(g_tw_mutex);
  if (dev < 64 && g_tw_n[dev] == n) return 0;
  const int N = 2 * n;
  float2 h[2 * kMaxWideN * kMaxWideN];
  double2 hd[2 * kMaxWideN * kMaxWideN];
  for (int u = 0; u < N; ++u)
    for (int a = 0; a < n; ++a) {
      const long m = ((long)(a + n / 2) * (2 * u + N + 1)) % (2L * N);
      const double ang = -M_PI * (double)m / (double)N;
      hd[u * n + a] = make_double2(cos(ang), sin(ang));
      h[u * n + a] = make_float2((float)cos(ang), (float)sin(ang));
    }
  // synchronous on purpose: `h` is a stack buffer; happens once per (device, n)
  cudaError_t e = cudaSuccess;
  if (n <= kMaxN) {
    e = cudaMemcpyToSymbol(c_tw, h, sizeof(float2) * N * n);
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_twd, hd, sizeof(double2) * N * n);
  } else {
    e = cudaMemcpyToSymbol(c_twd_wide, hd, sizeof(double2) * N * n);
  }
  if (e != cudaSuccess) return fail(-3, "twiddle upload: %s", cudaGetErrorString(e));
  if (dev < 64) g_tw_n[dev] = n;
  (void)stream;
  return 0;
}

// Poisson(lambda), lambda < 12, by inversion of the uniform u in (0, 1): sequential search from k = 0.  The first
// sixteen terms are unrolled with literal reciprocals (four FP32 instructions and a branch per term, no table load); the
// table loop takes over beyond (P(k > 16 | lambda < 12) < 8 %).
__device__ __forceinline__ float poisson_small(float lam, float u) {
  if (!(lam > 0.f)) return 0.f;
  float p = __expf(-lam), F = p;
#pragma unroll
  for (int j = 1; j <= 16; ++j) {
    if (!(u > F)) return (float)(j - 1);
    p *= lam * (1.0f / (float)j);
    F += p;
  }
  int k = 16;
  while (u > F && k < 63) {              // P(k >= 63 | lambda < 12) < 1e-24
    ++k;
    p *= lam * c_rcp_table.v[k];
    F += p;
  }
  return (float)k;
}
// the same search as a loop (rare call sites: the dark-current draw)
__device__ __noinline__ float poisson_small_loop(float lam, float u) {
  float p = __expf(-lam), F = p;
  int k = 0;
  while (u > F && k < 63) {
    ++k;
    p *= lam * c_rcp_table.v[k];
    F += p;
  }
  return (float)k;
}

// Hormann's PTRS transformed rejection for lambda >= 12 (the algorithm numpy's legacy generator also uses for
// lambda >= 10), one attempt at a time: two uniform words per attempt.
struct Ptrs {
  float lam, loglam, bb, a, invalpha, vr;
  __device__ __forceinline__ explicit Ptrs(float l) : lam(l) {
    const float slam = sqrtf(l);
    loglam = __logf(l);
    bb = 0.931f + 2.53f * slam;
    a = -0.059f + 0.02483f * bb;
    invalpha = 1.1239f + __fdividef(1.1328f, bb - 3.4f);
    vr = 0.9277f - __fdividef(3.6224f, bb - 2.f);
  }
  // true: accepted, k holds the draw
  __device__ __forceinline__ bool attempt(uint32_t w0, uint32_t w1, float& k) const {
    const float U = u32_to_unit(w0) - 0.5f;
    const float V = u32_to_unit(w1);
    const float us = 0.5f - fabsf(U);
    k = floorf((__fdividef(2.f * a, us) + bb) * U + lam + 0.43f);
    if (us >= 0.07f && V <= vr) return true;
    if (k < 0.f || (us < 0.013f && V > us)) return false;
    return __logf(V * invalpha * __frcp_rn(__fdividef(a, us * us) + bb)) <= -lam + k * loglam - log_factorial(k);
  }
};
constexpr int kPtrsMaxAttempts = 15;

// Poisson(lambda) from the uniform words (w0, w1), any lambda, attempts after the first from block `retry_block + attempt`
// of the pixel's stream (the in-lane form: used where the draws are too rare to be worth queueing)
__device__ __forceinline__ float poisson_draw(float lam, uint32_t w0, uint32_t w1, const PixelRng& rng, uint32_t retry_block) {
  if (!(lam > 0.f)) return 0.f;
  if (lam < 12.f) return poisson_small_loop(lam, u32_to_unit(w0) * 0.99999994f);
  const Ptrs pt(lam);
  for (int it = 0; it < kPtrsMaxAttempts; ++it) {
    if (it > 0) {
      const uint4 r = rng.block(retry_block + (uint32_t)it);
      w0 = r.x;
      w1 = r.y;
    }
    float k;
    if (pt.attempt(w0, w1, k)) return k;
  }
  return rintf(lam);
}

// OOPAO/Detector.py:279-301 (integrate) then :232-276 (readout), one pixel, split around the photon draw:
//   electrons = Poisson(flux) * QE + Poisson(dark); clip to the full well; (+ EM gain); + round(N(0,1) RON); gain; ADC.
// `stages` (aoenv_detector_t.reserved; 0 = all): bit 0 = integrate (photon noise, QE: Detector.py:279-301), bit 1 = first
// half of readout (dark current, full well, EM gain: :232-251), bit 2 = second half (read noise, gain, ADC: :256-268).
// Long exposures integrate sub-frames into a buffer (bit 0 each), then read the sum out once (bits 1 | 2); detector
// binning (:252-254) sits between the two halves.
__device__ __forceinline__ float detector_finish(float photons, float dark, float ron, const aoenv_detector_t& d, uint32_t stages) {
  float x = photons;
  if (stages & 1u) x *= d.qe;
  if (stages & 2u) {
    x += dark;
    if (d.has_fwc) x = fminf(fmaxf(x, 0.f), d.fwc);
    if (d.sensor_emccd) x *= d.gain;
  }
  if (stages & 4u) {
    x += ron;
    if (!d.sensor_emccd) x *= d.gain;
    if (d.bits > 0) {
      const float full = (float)((1u << d.bits) - 1u);
      x = truncf(x / d.fwc * full);
      x = fminf(x, full);
    }
  }
  return x;
}

// The camera as its own pass over the noise-free frame.  A warp walks kDetPerLane * 32 consecutive pixels (coalesced
// loads and stores, no block barrier).  Every lane does the cheap, uniform part of a pixel — one Philox block, the
// read-out normal, the dark-current draw, and the photon draw when the flux is below 12 (sequential inversion).  Pixels
// in the transformed-rejection regime (the bright cores, about a third of the lit pixels) are queued in the warp's
// shared-memory list and drawn afterwards by consecutive lanes, so the PTRS path runs on full warps.  Rejected attempts
// are not retried in the lane (one rejecting lane in 32 would make the whole warp pay for another Philox block and
// another attempt — ncu: 550 instructions per queued pixel, 40 % of the kernel): they are compacted into the front of the
// same list and the next round works on the rejected ones only, again on full warps.
// The random stream of a pixel depends only on (pixel, env, frame counter): block 0 -> photon words x, y / normal z, w;
// the four low bytes that u32_to_unit drops make a fifth independent word for the dark current; attempt i > 0 of the
// rejection sampler uses block 16 + i; dark currents >= 12 e- take block 1 (retries: blocks 32..).
constexpr int kDetPerLane = 8;
// w0 / w1: the photon words; their low bytes (which u32_to_unit drops) carry the pixel's dark-current draw, a whole number
// of electrons, as a 16-bit count — the entry stays at 20 bytes (40 KB of queues per CTA)
struct DetQueued { float lam, ron; uint32_t w0, w1; int pix; };

__device__ __forceinline__ uint32_t spare_word(const uint4& r) {
  return (r.x & 0xffu) | ((r.y & 0xffu) << 8) | ((r.z & 0xffu) << 16) | (r.w << 24);
}

__global__ void __launch_bounds__(256)
shwfs_detector_kernel(float* __restrict__ frame, const uint8_t* __restrict__ valid, int nS, int n, float inv_R, float inv_n,
                      const __grid_constant__ aoenv_detector_t det, int shared_max, int32_t* __restrict__ envmax,
                      int n_pixels) {
  pdl_enter();
  __shared__ DetQueued queue[8][kDetPerLane * 32];
  const int R = nS * n, P = n_pixels > 0 ? n_pixels : R * R;
  const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int first = (blockIdx.x * 8 + warp) * (kDetPerLane * 32);
  float* __restrict__ img = frame + (size_t)b * P;
  DetQueued* __restrict__ q = queue[warp];
  int queued = 0;                                   // warp-uniform
  float vmax = -INFINITY;
  const uint32_t stages = det.reserved ? det.reserved : 7u;
  const bool photon_noise = det.photon_noise && (stages & 1u);
  const bool has_dark = det.dark_electrons > 0.f && (stages & 2u);
  const bool has_ron = det.readout_noise != 0.f && (stages & 4u);
  const float dark_p0 = has_dark ? __expf(-det.dark_electrons) : 1.f;

  auto is_lit = [&](int pix) {
    if (valid == nullptr) return envmax != nullptr;            // stand-alone camera: every pixel counts
    const int y = (int)(((float)pix + 0.5f) * inv_R);          // exact: P < 2^24, fraction >= 1/(2R) from an integer
    const int x = pix - y * R;
    const int li = (int)(((float)y + 0.5f) * inv_n), lj = (int)(((float)x + 0.5f) * inv_n);
    return valid[li * nS + lj] != 0;
  };
  // the maximum runs over the lit lenslets only; the lookup is needed for the few values that would raise it
  auto track = [&](int pix, float val) {
    if (val > vmax && is_lit(pix)) vmax = val;
  };
  // dark current of one pixel (Detector.py:232-238): almost always zero — one comparison against exp(-dark)
  auto dark_draw = [&](const uint4& r0, const PixelRng& rng) {
    if (!has_dark) return 0.f;
    const uint32_t w = spare_word(r0);
    const float u = u32_to_unit(w) * 0.99999994f;
    if (!(u > dark_p0)) return 0.f;
    if (det.dark_electrons < 12.f) return poisson_small_loop(det.dark_electrons, u);
    const uint4 r1 = rng.block(1);
    return poisson_draw(det.dark_electrons, r1.x, r1.y, rng, 32);
  };

#pragma unroll 2
  for (int j = 0; j < kDetPerLane; ++j) {
    const int pix = first + j * 32 + lane;
    const bool in = pix < P;
    const float lam = in ? img[pix] : 0.f;
    const PixelRng rng(det.seed, (uint32_t)pix, (uint32_t)b, det.frame_counter);
    const uint4 r0 = rng.block(0);
    float ron = 0.f;
    if (has_ron)                        // Box-Muller with the SFU logarithm / cosine: the draw is rounded to whole electrons
      ron = rintf(sqrtf(-2.0f * __logf(u32_to_unit(r0.z))) * __cosf(6.283185307179586f * u32_to_unit(r0.w)) * det.readout_noise);
    const float dark = dark_draw(r0, rng);
    const bool ptrs = in && photon_noise && lam >= 12.f;
    if (!ptrs && in) {
      const float photons = photon_noise ? poisson_small(lam, u32_to_unit(r0.x) * 0.99999994f) : lam;
      const float val = detector_finish(photons, dark, ron, det, stages);
      img[pix] = val;
      track(pix, val);
    }
    const unsigned m = __ballot_sync(0xffffffffu, ptrs);
    if (ptrs) {
      const uint32_t dk = (uint32_t)fminf(dark, 65535.f);
      q[queued + __popc(m & ((1u << lane) - 1u))] = {lam, ron, (r0.x & ~0xffu) | (dk & 0xffu), (r0.y & ~0xffu) | (dk >> 8), pix};
    }
    queued += __popc(m);
  }
  __syncwarp();
  // rounds of one attempt per queued pixel; the rejected ones move to the front of the list for the next round
  for (int round = 0; queued > 0; ++round) {
    int kept = 0;                                   // warp-uniform
    for (int e0 = 0; e0 < queued; e0 += 32) {
      const int e = e0 + lane;
      const bool have = e < queued;
      DetQueued it = q[have ? e : 0];
      bool rejected = false;
      if (have) {
        const float dark = (float)((it.w0 & 0xffu) | ((it.w1 & 0xffu) << 8));
        if (round > 0) {
          const PixelRng rng(det.seed, (uint32_t)it.pix, (uint32_t)b, det.frame_counter);
          const uint4 r = rng.block(16u + (uint32_t)round);
          it.w0 = (r.x & ~0xffu) | (it.w0 & 0xffu);
          it.w1 = (r.y & ~0xffu) | (it.w1 & 0xffu);
        }
        const Ptrs pt(it.lam);
        float photons;
        bool ok = pt.attempt(it.w0, it.w1, photons);
        if (!ok && round == kPtrsMaxAttempts - 1) { photons = rintf(it.lam); ok = true; }
        if (ok) {
          const float val = detector_finish(photons, dark, it.ron, det, stages);
          img[it.pix] = val;
          track(it.pix, val);
        }
        rejected = !ok;
      }
      __syncwarp();                                 // every lane has read its entry before the front of the list is rewritten
      const unsigned m = __ballot_sync(0xffffffffu, rejected);
      if (rejected) q[kept + __popc(m & ((1u << lane) - 1u))] = it;      // kept + rank <= e: never ahead of the reads
      kept += __popc(m);
    }
    __syncwarp();
    queued = kept;
  }
  if (envmax != nullptr) {
    vmax = warp_max(vmax);
    if (lane == 0 && vmax > -INFINITY) atomicMax(&envmax[shared_max ? 0 : b], float_to_ordered(vmax));
  }
}

// WL > 0: the second OPD term is the separable DM surface, evaluated in place from the column half T = C gx
// (aoenv_dm_rows) and the row weights of `dm` (see aoenv_dm_sep_t) instead of being read from opd_b: each lenslet sums
// its n x n pixels over the WL actuator rows of its lenslet row's window.  The surface is then never written to memory.
template <int n, int WL = 0>
__global__ void __launch_bounds__(128)
shwfs_frame_kernel(const float* __restrict__ opd_a, const float* __restrict__ opd_b, const float* __restrict__ pupil,
                   const float* __restrict__ amp, const uint8_t* __restrict__ valid, int nS, float phase_scale,
                   int track_max, int shared_max, float* __restrict__ frame,
                   int32_t* __restrict__ envmax, double* __restrict__ stats, const __grid_constant__ aoenv_dm_sep_t dm,
                   const int32_t* __restrict__ order) {
  constexpr int N = 2 * n;
  pdl_enter();
  const int R = nS * n;
  const int b = blockIdx.y;
  // `order` (nullable): a permutation of the lenslet numbers with the lit ones first — warps are then all lit or all
  // dark, and the dark ones skip the transform as a whole instead of idling in the lanes of a mixed warp
  const int k0 = blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = k0 < nS * nS;
  const int k = (active && order != nullptr) ? __ldg(&order[k0]) : k0;
  const int li = active ? k / nS : 0, lj = active ? k % nS : 0;
  const bool lit = active && valid[k] != 0;
  const float phase_turns = phase_scale * 0.15915494309189535f;      // radians -> turns

  // field E[a][b] = tile^T (ShackHartmann.py:341-345 tiles phase.T), kept as pairs along b:
  // er2[a][k] = (Re E[a][2k], Re E[a][2k+1]) so that the first DFT pass runs on packed FP32 (FFMA2)
  float2 er2[n][n / 2], ei2[n][n / 2];
  // Pupil statistics for std(OPD) / var(phase): variance is shift invariant, so each thread accumulates its n*n
  // pixels in float32 relative to the value at the pupil centre (removes the piston that would otherwise dominate
  // sum x^2), and only the per-thread partial sums are promoted to float64 for the reduction.
  float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f;
  if (active) {
    const size_t tile = (size_t)(li * n) * R + lj * n;
    const float* __restrict__ pa = opd_a + (size_t)b * R * R + tile;
    const float* __restrict__ pb = (WL == 0 && opd_b) ? opd_b + (size_t)b * R * R + tile : nullptr;
    const size_t centre = (size_t)b * R * R + (size_t)(R / 2) * R + R / 2;
    const float ka = stats ? __ldg(opd_a + centre) : 0.f;
    // (variance is shift invariant: with the in-place DM the total is centred on the atmosphere's centre value)
    const float kt = stats ? (pb ? ka + __ldg(opd_b + centre) : ka) : 0.f;
    // DM surface of this lenslet's tile: dmv[bb][a2] = pixels (row bb, columns 2 a2, 2 a2 + 1)
    float2 dmv[WL > 0 ? n : 1][n / 2];
    if (WL > 0) {
      constexpr int half = (WL + 1) / 2, hp = (half + 3) / 4 * 4;
#pragma unroll
      for (int bb = 0; bb < n; ++bb)
#pragma unroll
        for (int a2 = 0; a2 < n / 2; ++a2) dmv[WL > 0 ? bb : 0][a2] = make_float2(0.f, 0.f);
      const float* __restrict__ trow = dm.rows + ((size_t)b * dm.nActP + __ldg(&dm.ilr[li])) * R + lj * n;
      const float* __restrict__ wrow = dm.wlr + (size_t)(li * n) * (2 * hp);
#pragma unroll
      for (int g = 0; g < 2 * hp / 4; ++g) {
        float4 w4[n];
#pragma unroll
        for (int bb = 0; bb < n; ++bb) w4[bb] = __ldg(reinterpret_cast<const float4*>(wrow + (size_t)bb * (2 * hp)) + g);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int j = 4 * g + e, hh = j / hp, kk = j % hp;
          if (kk >= half) continue;                      // padding entries of the weight rows
          const int t = hh * half + kk;
          if (t >= WL) continue;
          float2 tv[n / 2];
#pragma unroll
          for (int a2 = 0; a2 < n / 2; ++a2) tv[a2] = __ldg(reinterpret_cast<const float2*>(trow + (size_t)t * R) + a2);
#pragma unroll
          for (int bb = 0; bb < n; ++bb) {
            const float w = e == 0 ? w4[bb].x : (e == 1 ? w4[bb].y : (e == 2 ? w4[bb].z : w4[bb].w));
#pragma unroll
            for (int a2 = 0; a2 < n / 2; ++a2) dmv[WL > 0 ? bb : 0][a2] = fma2(dup2(w), tv[a2], dmv[WL > 0 ? bb : 0][a2]);
          }
        }
      }
    }
#pragma unroll
    for (int bb = 0; bb < n; ++bb) {
#pragma unroll
      for (int a2 = 0; a2 < n / 2; ++a2) {
        // two neighbouring pixels per 64-bit load (tile rows start on even columns: lj * n with n even, R even)
        const int o2 = bb * R + 2 * a2;
        const float2 av = __ldg(reinterpret_cast<const float2*>(pa + o2));
        const float2 bv = WL > 0 ? dmv[WL > 0 ? bb : 0][a2]
                                 : (pb ? __ldg(reinterpret_cast<const float2*>(pb + o2)) : make_float2(0.f, 0.f));
        const float2 pv = __ldg(reinterpret_cast<const float2*>(pupil + tile + o2));
        const float2 mv = lit ? __ldg(reinterpret_cast<const float2*>(amp + tile + o2)) : make_float2(0.f, 0.f);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int aa = 2 * a2 + e;
          const float a = e ? av.y : av.x;
          const float t = a + (e ? bv.y : bv.x);
          const float pu = e ? pv.y : pv.x;
          const float in_pupil = pu > 0.f ? 1.f : 0.f;
          const float da = (a - ka) * in_pupil, dt = (t - kt) * in_pupil;
          f0 += da; f1 = fmaf(da, da, f1); f2 += dt; f3 = fmaf(dt, dt, f3);
          // phase / 2pi reduced to [-1/2, 1/2] exactly, then the SFU sine/cosine (abs. error ~4e-7 on [-pi, pi])
          const float turns = t * pu * phase_turns;
          // nearest integer by the 1.5 * 2^23 trick (two FADDs; rintf would go through the transcendental pipe, which
          // the sine and cosine already load): exact for |turns| < 2^22
          const float ang = (turns - ((turns + 12582912.0f) - 12582912.0f)) * 6.283185307179586f;
          const float sn = __sinf(ang), cs = __cosf(ang);
          const float am = e ? mv.y : mv.x;
          if ((bb & 1) == 0) { er2[aa][bb >> 1].x = am * cs; ei2[aa][bb >> 1].x = am * sn; }
          else { er2[aa][bb >> 1].y = am * cs; ei2[aa][bb >> 1].y = am * sn; }
        }
      }
    }
  }
  double s0 = (double)f0, s1 = (double)f1, s2 = (double)f2, s3 = (double)f3;

  if (stats != nullptr) {       // one atomic per warp and statistic: no block barrier, warps drift freely between phases
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2); s3 = warp_sum(s3);
    if ((threadIdx.x & 31) == 0) {
      double* __restrict__ st = stats + (size_t)b * 4;
      atomicAdd(st, s0); atomicAdd(st + 1, s1); atomicAdd(st + 2, s2); atomicAdd(st + 3, s3);
    }
  }

  float vmax = -INFINITY;
  if (active) {
    float* __restrict__ fout = frame + (size_t)b * R * R + (size_t)(li * n) * R + lj * n;
    const float norm = 1.0f / (float)(N * N);
    // Radix-2 split of both DFT passes: G[u + n][a] = (-1)^(a + n/2) G[u][a] (the half-pixel phasor keeps the
    // symmetry), so output rows u and u + n share their even-/odd-class partial sums P, Q:  Y_u = P + Q,
    // Y_{u+n} = P - Q, and likewise for the columns.  Binned row pp collects u = 2pp, 2pp+1; row pp + n/2 collects
    // u + n.
    // Both passes run on packed pairs: pass 1 on pairs of columns b (twiddle = broadcast scalar from the constant
    // bank), pass 2 on the pair (row u, row u + n), which share their twiddles (broadcast immediates).  Each
    // FFMA2 / FADD2 / FMUL2 is two IEEE FP32 operations in one issue slot, in the same order as the scalar formulation.
    constexpr int h = n / 2;
#pragma unroll 1
    for (int pp = 0; pp < h; ++pp) {
      float2 acc[n];                         // acc[q] = (binned row pp, binned row pp + n/2) at binned column q
#pragma unroll
      for (int q = 0; q < n; ++q) acc[q] = make_float2(0.f, 0.f);
      if (lit) {
#pragma unroll
        for (int du = 0; du < 2; ++du) {
          const int u = 2 * pp + du;
          float2 pr[h], pi[h], qr[h], qi[h];
#pragma unroll
          for (int k = 0; k < h; ++k) { pr[k] = pi[k] = qr[k] = qi[k] = make_float2(0.f, 0.f); }
#pragma unroll
          for (int aa = 0; aa < n; ++aa) {
            const float2 g = c_tw[u * n + aa];
            const float2 gx = dup2(g.x), gy = dup2(g.y), ngy = dup2(-g.y);
            if (((aa + h) & 1) == 0) {
#pragma unroll
              for (int k = 0; k < h; ++k) {
                pr[k] = fma2(gx, er2[aa][k], fma2(ngy, ei2[aa][k], pr[k]));
                pi[k] = fma2(gx, ei2[aa][k], fma2(gy, er2[aa][k], pi[k]));
              }
            } else {
#pragma unroll
              for (int k = 0; k < h; ++k) {
                qr[k] = fma2(gx, er2[aa][k], fma2(ngy, ei2[aa][k], qr[k]));
                qi[k] = fma2(gx, ei2[aa][k], fma2(gy, er2[aa][k], qi[k]));
              }
            }
          }
          // Y[b] = (row u: P + Q, row u + n: P - Q)
          float2 yr[n], yi[n];
#pragma unroll
          for (int bb = 0; bb < n; ++bb) {
            const float p_r = (bb & 1) ? pr[bb >> 1].y : pr[bb >> 1].x, q_r = (bb & 1) ? qr[bb >> 1].y : qr[bb >> 1].x;
            const float p_i = (bb & 1) ? pi[bb >> 1].y : pi[bb >> 1].x, q_i = (bb & 1) ? qi[bb >> 1].y : qi[bb >> 1].x;
            yr[bb] = make_float2(p_r + q_r, p_r - q_r);
            yi[bb] = make_float2(p_i + q_i, p_i - q_i);
          }
#pragma unroll
          for (int v = 0; v < n; ++v) {
            float2 er_ = make_float2(0.f, 0.f), ei_ = er_, or_ = er_, oi_ = er_;
#pragma unroll
            for (int bb = 0; bb < n; ++bb) {
              // v, bb are compile-time after unrolling: literal twiddles -> broadcast-immediate FFMA2s
              const float gx = WfsTw<n>::re(v * n + bb), gy = WfsTw<n>::im(v * n + bb);
              if (((bb + h) & 1) == 0) {
                er_ = fma2(yr[bb], dup2(gx), fma2(yi[bb], dup2(-gy), er_));
                ei_ = fma2(yr[bb], dup2(gy), fma2(yi[bb], dup2(gx), ei_));
              } else {
                or_ = fma2(yr[bb], dup2(gx), fma2(yi[bb], dup2(-gy), or_));
                oi_ = fma2(yr[bb], dup2(gy), fma2(yi[bb], dup2(gx), oi_));
              }
            }
            const float2 f0r = add2(er_, or_), f0i = add2(ei_, oi_);     // F[row][v]
            const float2 f1r = sub2(er_, or_), f1i = sub2(ei_, oi_);     // F[row][v + n]
            acc[v >> 1] = add2(acc[v >> 1], fma2(f0r, f0r, mul2(f0i, f0i)));
            acc[(v >> 1) + h] = add2(acc[(v >> 1) + h], fma2(f1r, f1r, mul2(f1i, f1i)));
          }
        }
      }
#pragma unroll
      for (int r2 = 0; r2 < 2; ++r2) {
        const int p = pp + r2 * h;
#pragma unroll
        for (int q = 0; q < n; ++q) {
          const float val = (r2 == 0 ? acc[q].x : acc[q].y) * norm;
          fout[(size_t)p * R + q] = val;
          if (lit) vmax = fmaxf(vmax, val);
        }
      }
    }
  }
  if (track_max) {            // with a camera model the maximum is taken after the detector pass
    vmax = warp_max(vmax);
    if ((threadIdx.x & 31) == 0 && vmax > -INFINITY) atomicMax(&envmax[shared_max ? 0 : b], float_to_ordered(vmax));
  }
}

// ---------------------------------------------------------------------------------------------------------
// n = 6 (the reference's 6 pixels per subaperture, N = 12): the same frame as shwfs_frame_kernel<6>, with the pruned
// DFTs factorised instead of summed term by term.
//   * the half-pixel phasor exp(-i pi 13 (a+3)/12) exp(-i pi 13 (b+3)/12) is folded into the angle of the field;
//     the remaining kernel is W^{(a+3)u} = W^{3u} W^{au}, W = exp(-2 pi i / 12), and the unit factor W^{3u} (W^{3v}) does
//     not change |F|^2, so each pass is a plain 12-point DFT of 6 inputs at indices 0..5;
//   * u = 2k + r:  H[2k + r] = DFT6( x[a] W^{r a} )[k]  — two 6-point DFTs, the second on the twiddled sequence;
//   * DFT6 = Good-Thomas 2 x 3 (no inner twiddles): s[a2] = z[2 a2] +- z[2 a2 + 3], then a 3-point DFT;
//     output k = (3 k1 + 4 k2) mod 6.
// Packed FP32 throughout: pass 1 carries (r = 0, r = 1) in the two lanes, pass 2 the row pair (2p, 2p + 1) — exactly
// the four samples a binned pixel sums.  Rows are produced in two phases (k1 = 0: binned rows 0, 4, 2; k1 = 1: rows
// 3, 1, 5) so that only half of the intermediate lives in registers; the field waits in shared memory, one column of
// 72 floats per thread.  2.1 k FP32 pipe slots per lenslet for transform + intensities instead of 3.5 k.
// ---------------------------------------------------------------------------------------------------------
struct C2 { float2 r, i; };          // two complex numbers, lane-wise
__device__ __forceinline__ C2 cadd(const C2& a, const C2& b) { return {add2(a.r, b.r), add2(a.i, b.i)}; }
__device__ __forceinline__ C2 csub(const C2& a, const C2& b) { return {sub2(a.r, b.r), sub2(a.i, b.i)}; }
// a * (wr + i wi), constants
__device__ __forceinline__ C2 cmulc(const C2& a, float wr, float wi) {
  return {fma2(a.r, dup2(wr), mul2(a.i, dup2(-wi))), fma2(a.r, dup2(wi), mul2(a.i, dup2(wr)))};
}
__device__ __forceinline__ void dft3(const C2& z0, const C2& z1, const C2& z2, C2& y0, C2& y1, C2& y2) {
  constexpr float c = 0.8660254037844386f;
  const C2 t = cadd(z1, z2), d = csub(z1, z2);
  y0 = cadd(z0, t);
  const C2 m = {fma2(dup2(-0.5f), t.r, z0.r), fma2(dup2(-0.5f), t.i, z0.i)};
  y1 = {fma2(dup2(c), d.i, m.r), fma2(dup2(-c), d.r, m.i)};      // m - i c d
  y2 = {fma2(dup2(-c), d.i, m.r), fma2(dup2(c), d.r, m.i)};      // m + i c d
}
// one half of DFT6 (k1 = 0: outputs k = 0, 4, 2; k1 = 1: outputs k = 3, 1, 5), inputs z[0..5]
template <int K1>
__device__ __forceinline__ void dft6_half(const C2 (&z)[6], C2& y0, C2& y1, C2& y2) {
  const C2 s0 = K1 == 0 ? cadd(z[0], z[3]) : csub(z[0], z[3]);
  const C2 s1 = K1 == 0 ? cadd(z[2], z[5]) : csub(z[2], z[5]);
  const C2 s2 = K1 == 0 ? cadd(z[4], z[1]) : csub(z[4], z[1]);
  dft3(s0, s1, s2, y0, y1, y2);
}
// z[a] * W^a, W = exp(-2 pi i / 12)
__device__ __forceinline__ void twiddle6(const C2 (&z)[6], C2 (&w)[6]) {
  constexpr float c = 0.8660254037844386f;
  w[0] = z[0];
  w[1] = cmulc(z[1], c, -0.5f);
  w[2] = cmulc(z[2], 0.5f, -c);
  w[3] = {z[3].i, mul2(z[3].r, dup2(-1.0f))};                    // * (-i)
  w[4] = cmulc(z[4], -0.5f, -c);
  w[5] = cmulc(z[5], -c, -0.5f);
}
__host__ __device__ constexpr int dft6_row(int k1, int k2) { return (3 * k1 + 4 * k2) % 6; }

// pass 1 of one phase: Hp[k2][b] = (DFT6(x)[k], DFT6(x W^a)[k]) for k = dft6_row(K1, k2)
template <int K1>
__device__ __forceinline__ void wfs6_pass1(const float* __restrict__ sF, C2 (&Hp)[3][6]) {
  constexpr float c = 0.8660254037844386f;
#pragma unroll
  for (int b = 0; b < 6; ++b) {
    C2 z[6];
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      const float xr = sF[(2 * (a * 6 + b)) * 128], xi = sF[(2 * (a * 6 + b) + 1) * 128];
      float wr, wi;                                              // x * W^a
      if (a == 0) { wr = xr; wi = xi; }
      else if (a == 1) { wr = fmaf(xr, c, xi * 0.5f); wi = fmaf(xi, c, xr * -0.5f); }
      else if (a == 2) { wr = fmaf(xr, 0.5f, xi * c); wi = fmaf(xi, 0.5f, xr * -c); }
      else if (a == 3) { wr = xi; wi = -xr; }
      else if (a == 4) { wr = fmaf(xr, -0.5f, xi * c); wi = fmaf(xi, -0.5f, xr * -c); }
      else { wr = fmaf(xr, -c, xi * 0.5f); wi = fmaf(xi, -c, xr * -0.5f); }
      z[a] = {make_float2(xr, wr), make_float2(xi, wi)};
    }
    dft6_half<K1>(z, Hp[0][b], Hp[1][b], Hp[2][b]);
  }
}

// pass 2 of one phase + intensities + binning + store of three binned rows
template <int K1>
__device__ __forceinline__ void wfs6_pass2(const C2 (&Hp)[3][6], float norm, float* __restrict__ fout, int R, float& vmax) {
#pragma unroll
  for (int k2 = 0; k2 < 3; ++k2) {
    const int p = dft6_row(K1, k2);                              // lanes = frame rows (2p, 2p + 1) before binning
    C2 yw[6];
    twiddle6(Hp[k2], yw);
    float row[6];
#pragma unroll
    for (int q1 = 0; q1 < 2; ++q1) {
      C2 e[3], o[3];
      if (q1 == 0) { dft6_half<0>(Hp[k2], e[0], e[1], e[2]); dft6_half<0>(yw, o[0], o[1], o[2]); }
      else { dft6_half<1>(Hp[k2], e[0], e[1], e[2]); dft6_half<1>(yw, o[0], o[1], o[2]); }
#pragma unroll
      for (int q2 = 0; q2 < 3; ++q2) {
        const float2 i0 = fma2(e[q2].r, e[q2].r, mul2(e[q2].i, e[q2].i));       // v = 2q
        const float2 i1 = fma2(o[q2].r, o[q2].r, mul2(o[q2].i, o[q2].i));       // v = 2q + 1
        const float2 t = add2(i0, i1);
        row[dft6_row(q1, q2)] = (t.x + t.y) * norm;
      }
    }
#pragma unroll
    for (int q = 0; q < 6; ++q) {
      fout[(size_t)p * R + q] = row[q];
      vmax = fmaxf(vmax, row[q]);
    }
  }
}

__global__ void __launch_bounds__(128, 3)
shwfs_frame6_kernel(const float* __restrict__ opd_a, const float* __restrict__ opd_b, const float* __restrict__ pupil,
                    const float* __restrict__ amp, const uint8_t* __restrict__ valid, int nS, float phase_scale,
                    int track_max, int shared_max, float* __restrict__ frame, int32_t* __restrict__ envmax,
                    double* __restrict__ stats) {
  constexpr int n = 6, N = 12;
  __shared__ float sF_all[2 * n * n * 128];      // field, element-major: thread t owns sF_all[e * 128 + t]
  float* __restrict__ sF = sF_all + threadIdx.x;
  const int R = nS * n;
  const int b = blockIdx.y;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = k < nS * nS;
  const int li = active ? k / nS : 0, lj = active ? k % nS : 0;
  const bool lit = active && valid[k] != 0;
  const float phase_turns = phase_scale * 0.15915494309189535f;      // radians -> turns
  float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f;                      // pupil statistics, see shwfs_frame_kernel
  if (active) {
    const size_t tile = (size_t)(li * n) * R + lj * n;
    const float* __restrict__ pa = opd_a + (size_t)b * R * R + tile;
    const float* __restrict__ pb = opd_b ? opd_b + (size_t)b * R * R + tile : nullptr;
    const size_t centre = (size_t)b * R * R + (size_t)(R / 2) * R + R / 2;
    const float ka = stats ? __ldg(opd_a + centre) : 0.f;
    const float kt = stats ? (opd_b ? ka + __ldg(opd_b + centre) : ka) : 0.f;
#pragma unroll
    for (int bb = 0; bb < n; ++bb) {
#pragma unroll
      for (int aa = 0; aa < n; ++aa) {
        const int o = bb * R + aa;
        const float a = __ldg(pa + o);
        const float t = pb ? a + __ldg(pb + o) : a;
        const float pu = __ldg(pupil + tile + o);
        const float in_pupil = pu > 0.f ? 1.f : 0.f;
        const float da = (a - ka) * in_pupil, dt = (t - kt) * in_pupil;
        f0 += da; f1 = fmaf(da, da, f1); f2 += dt; f3 = fmaf(dt, dt, f3);
        if (lit) {
          // phase / 2pi plus the half-pixel phasor of both axes, -13 (a + b + 6) / 24 turns (compile-time constant)
          constexpr double kTurn = -13.0 / 24.0;
          const double cst = kTurn * (double)(aa + bb + n);
          const float cfrac = (float)(cst - (double)(long long)(cst - 0.5));      // reduced to [-0.5, 0.5]
          const float turns = fmaf(t * pu, phase_turns, cfrac);
          const float ang = (turns - ((turns + 12582912.0f) - 12582912.0f)) * 6.283185307179586f;
          const float am = __ldg(amp + tile + o);
          sF[(2 * (aa * n + bb)) * 128] = am * __cosf(ang);
          sF[(2 * (aa * n + bb) + 1) * 128] = am * __sinf(ang);
        }
      }
    }
  }
  if (stats != nullptr) {
    double s0 = warp_sum((double)f0), s1 = warp_sum((double)f1), s2 = warp_sum((double)f2), s3 = warp_sum((double)f3);
    if ((threadIdx.x & 31) == 0) {
      double* __restrict__ st = stats + (size_t)b * 4;
      atomicAdd(st, s0); atomicAdd(st + 1, s1); atomicAdd(st + 2, s2); atomicAdd(st + 3, s3);
    }
  }
  float vmax = -INFINITY;
  if (active) {
    float* __restrict__ fout = frame + (size_t)b * R * R + (size_t)(li * n) * R + lj * n;
    if (lit) {
      const float norm = 1.0f / (float)(N * N);
      C2 Hp[3][6];
      wfs6_pass1<0>(sF, Hp);
      wfs6_pass2<0>(Hp, norm, fout, R, vmax);
      wfs6_pass1<1>(sF, Hp);
      wfs6_pass2<1>(Hp, norm, fout, R, vmax);
    } else {
#pragma unroll
      for (int p = 0; p < n; ++p)
#pragma unroll
        for (int q = 0; q < n; ++q) fout[(size_t)p * R + q] = 0.f;
    }
  }
  if (track_max) {
    vmax = warp_max(vmax);
    if ((threadIdx.x & 31) == 0 && vmax > -INFINITY) atomicMax(&envmax[shared_max ? 0 : b], float_to_ordered(vmax));
  }
}

// ---------------------------------------------------------------------------------------------------------
// n = 6, THREE LANES PER LENSLET (the production frame kernel): the factorised transform above, split so that no thread
// ever holds more than a third of a lenslet.  Lane t of a lenslet owns tile rows 2t, 2t+1 = columns b = 2t, 2t+1 of the
// transposed field: it loads those 12 pixels, forms the field (half-pixel phasor folded into the angle) and runs pass 1
// — the 12-point DFT over a of its two columns, as two 6-point Good-Thomas DFTs packed in the FP32x2 lanes (r = 0, 1) —
// which yields H[k][b] for all six row pairs k.  The three lanes then swap thirds through a warp-private patch of shared
// memory (no block barrier anywhere: a __syncwarp orders the exchange): lane t keeps the row pairs k = (4t) mod 6 and
// (3 + 4t) mod 6, for which it runs pass 2 over all six columns, the intensities and the 2x2 binning, and stores binned
// rows k with 64-bit stores.  Every lane of a warp executes the same instruction stream (the passes do not depend on which
// column / row pair they work on), 10 lenslets per warp, ~80 registers instead of 165, 2.1 k instead of 3.5 k FP32 pipe
// slots per lenslet.
// ---------------------------------------------------------------------------------------------------------
constexpr int kS6Lenslets = 10;                     // lenslets per warp (lanes 30, 31 idle)
constexpr int kS6Warps = 4;

// dft6_half for both K1 at once on one column; outputs indexed [K1][k2]
__device__ __forceinline__ void dft6_both(const C2 (&z)[6], C2 (&y)[2][3]) {
  dft6_half<0>(z, y[0][0], y[0][1], y[0][2]);
  dft6_half<1>(z, y[1][0], y[1][1], y[1][2]);
}

__global__ void __launch_bounds__(kS6Warps * 32, 4)
shwfs_frame6s_kernel(const float* __restrict__ opd_a, const float* __restrict__ opd_b, const float* __restrict__ pupil,
                     const float* __restrict__ amp, const uint8_t* __restrict__ valid, int nS, float phase_scale,
                     int track_max, int shared_max, float* __restrict__ frame, int32_t* __restrict__ envmax,
                     double* __restrict__ stats) {
  constexpr int n = 6, N = 12;
  constexpr float c = 0.8660254037844386f;
  // exchange buffer: [warp][value 0..47][lane]; value = ((K1 * 3 + k2) * 2 + col) * 4 + component
  __shared__ float xch[kS6Warps][48][33];        // row stride 33: the three lanes of a lenslet hit different banks
  const int R = nS * n;
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = lane / 3, t = lane - slot * 3;                        // lenslet of the warp, third of the lenslet
  const int k = (blockIdx.x * kS6Warps + warp) * kS6Lenslets + slot;
  const bool active = slot < kS6Lenslets && k < nS * nS;
  const int li = active ? k / nS : 0, lj = active ? k - li * nS : 0;
  const bool lit = active && valid[k] != 0;
  const float phase_turns = phase_scale * 0.15915494309189535f;
  const size_t tile = (size_t)(li * n) * R + lj * n;
  float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f;                         // pupil statistics, see shwfs_frame_kernel
  // ---- field of tile rows 2t, 2t+1 + pass 1 ------------------------------------------------------------------------
  C2 y[2][2][3];                                                          // [column][K1][k2]
  if (active) {
    const float* __restrict__ pa = opd_a + (size_t)b * R * R + tile;
    const float* __restrict__ pb = opd_b ? opd_b + (size_t)b * R * R + tile : nullptr;
    const size_t centre = (size_t)b * R * R + (size_t)(R / 2) * R + R / 2;
    const float ka = stats ? __ldg(opd_a + centre) : 0.f;
    const float kt = stats ? (opd_b ? ka + __ldg(opd_b + centre) : ka) : 0.f;
    // reduced phasor angle of row bb = 2t + e, in turns: -13 (bb + 3) / 24 mod 1 (literal constants, exact to 6e-8)
    constexpr float kCf[6] = {0.375f, -0.16666667f, 0.29166667f, -0.25f, 0.20833333f, -0.33333333f};
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int bb = 2 * t + e;
      const float cfb = e == 0 ? (t == 0 ? kCf[0] : t == 1 ? kCf[2] : kCf[4]) : (t == 0 ? kCf[1] : t == 1 ? kCf[3] : kCf[5]);
      C2 z[6];
#pragma unroll
      for (int a2 = 0; a2 < 3; ++a2) {
        const int o2 = bb * R + 2 * a2;
        const float2 av = __ldg(reinterpret_cast<const float2*>(pa + o2));
        const float2 bv = pb ? __ldg(reinterpret_cast<const float2*>(pb + o2)) : make_float2(0.f, 0.f);
        const float2 pv = __ldg(reinterpret_cast<const float2*>(pupil + tile + o2));
        const float2 mv = lit ? __ldg(reinterpret_cast<const float2*>(amp + tile + o2)) : make_float2(0.f, 0.f);
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
          const int aa = 2 * a2 + h2;
          const float a = h2 ? av.y : av.x;
          const float tt = a + (h2 ? bv.y : bv.x);
          const float pu = h2 ? pv.y : pv.x;
          const float in_pupil = pu > 0.f ? 1.f : 0.f;
          const float da = (a - ka) * in_pupil, dt = (tt - kt) * in_pupil;
          f0 += da; f1 = fmaf(da, da, f1); f2 += dt; f3 = fmaf(dt, dt, f3);
          const float turns = fmaf(tt * pu, phase_turns, kCf[aa] + cfb);
          const float ang = (turns - ((turns + 12582912.0f) - 12582912.0f)) * 6.283185307179586f;
          const float am = h2 ? mv.y : mv.x;
          const float xr = am * __cosf(ang), xi = am * __sinf(ang);
          float wr, wi;                                                   // x * W^a, W = exp(-2 pi i / 12): the r = 1 lane
          if (aa == 0) { wr = xr; wi = xi; }
          else if (aa == 1) { wr = fmaf(xr, c, xi * 0.5f); wi = fmaf(xi, c, xr * -0.5f); }
          else if (aa == 2) { wr = fmaf(xr, 0.5f, xi * c); wi = fmaf(xi, 0.5f, xr * -c); }
          else if (aa == 3) { wr = xi; wi = -xr; }
          else if (aa == 4) { wr = fmaf(xr, -0.5f, xi * c); wi = fmaf(xi, -0.5f, xr * -c); }
          else { wr = fmaf(xr, -c, xi * 0.5f); wi = fmaf(xi, -c, xr * -0.5f); }
          z[aa] = {make_float2(xr, wr), make_float2(xi, wi)};
        }
      }
      dft6_both(z, y[e]);
    }
  }
  if (stats != nullptr) {
    double s0 = warp_sum((double)f0), s1 = warp_sum((double)f1), s2 = warp_sum((double)f2), s3 = warp_sum((double)f3);
    if (lane == 0) {
      double* __restrict__ st = stats + (size_t)b * 4;
      atomicAdd(st, s0); atomicAdd(st + 1, s1); atomicAdd(st + 2, s2); atomicAdd(st + 3, s3);
    }
  }
  // ---- the three lanes of a lenslet swap thirds: lane t2 receives H[K1][k2 = t2][all six columns] ----------------------
  float (*x)[33] = xch[warp];
  const bool any_lit = __any_sync(0xffffffffu, lit);
  float vmax = -INFINITY;
  if (any_lit) {
    if (lit) {
#pragma unroll
      for (int e = 0; e < 2; ++e)
#pragma unroll
        for (int K1 = 0; K1 < 2; ++K1)
#pragma unroll
          for (int k2 = 0; k2 < 3; ++k2) {
            // destination lane = slot * 3 + k2; written at its address, indexed by (K1, source column 2t + e)
            const int dst = slot * 3 + k2;
            const C2 v = y[e][K1][k2];
            // value index: (K1 * 6 + column) * 4 + component -> 48 values per destination lane
            // (column = 2t + e is lane-dependent: the index is computed, the stores stay conflict-free per component)
            const int base = (K1 * 6 + 2 * t + e) * 4;
            x[base + 0][dst] = v.r.x; x[base + 1][dst] = v.r.y; x[base + 2][dst] = v.i.x; x[base + 3][dst] = v.i.y;
          }
    }
    __syncwarp();
    if (lit) {
      float* __restrict__ fout = frame + (size_t)b * R * R + tile;
      const float norm = 1.0f / (float)(N * N);
#pragma unroll
      for (int K1 = 0; K1 < 2; ++K1) {
        const int p = (3 * K1 + 4 * t) % 6;                              // binned row = row pair (2p, 2p + 1)
        C2 Hr[6];
#pragma unroll
        for (int bcol = 0; bcol < 6; ++bcol) {
          const int base = (K1 * 6 + bcol) * 4;
          Hr[bcol] = {make_float2(x[base + 0][lane], x[base + 1][lane]), make_float2(x[base + 2][lane], x[base + 3][lane])};
        }
        C2 yw[6];
        twiddle6(Hr, yw);
        float row[6];
#pragma unroll
        for (int q1 = 0; q1 < 2; ++q1) {
          C2 e[3], o[3];
          if (q1 == 0) { dft6_half<0>(Hr, e[0], e[1], e[2]); dft6_half<0>(yw, o[0], o[1], o[2]); }
          else { dft6_half<1>(Hr, e[0], e[1], e[2]); dft6_half<1>(yw, o[0], o[1], o[2]); }
#pragma unroll
          for (int q2 = 0; q2 < 3; ++q2) {
            const float2 i0 = fma2(e[q2].r, e[q2].r, mul2(e[q2].i, e[q2].i));       // v = 2q
            const float2 i1 = fma2(o[q2].r, o[q2].r, mul2(o[q2].i, o[q2].i));       // v = 2q + 1
            const float2 tt = add2(i0, i1);
            row[dft6_row(q1, q2)] = (tt.x + tt.y) * norm;
          }
        }
#pragma unroll
        for (int q2 = 0; q2 < 3; ++q2) {
          *reinterpret_cast<float2*>(fout + (size_t)p * R + 2 * q2) = make_float2(row[2 * q2], row[2 * q2 + 1]);
          vmax = fmaxf(vmax, fmaxf(row[2 * q2], row[2 * q2 + 1]));
        }
      }
    }
  }
  if (active && !lit) {                                                   // dark lenslet: rows 2t, 2t+1 of its tile
    float* __restrict__ fout = frame + (size_t)b * R * R + tile;
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
      for (int q2 = 0; q2 < 3; ++q2) *reinterpret_cast<float2*>(fout + (size_t)(2 * t + e) * R + 2 * q2) = make_float2(0.f, 0.f);
  }
  if (track_max) {
    vmax = warp_max(vmax);
    if (lane == 0 && vmax > -INFINITY) atomicMax(&envmax[shared_max ? 0 : b], float_to_ordered(vmax));
  }
}

// ---------------------------------------------------------------------------------------------------------
// n / 2 LANES PER LENSLET, term-by-term transform (all compiled n): the arithmetic of shwfs_frame_kernel — radix-2 split
// of both pruned DFT passes, packed FP32, literal twiddles — with the lenslet spread over T = n / 2 lanes of one warp.
// Lane t owns tile rows 2t, 2t+1 = the column pair (2t, 2t+1) of the transposed field: it forms those fields and runs
// pass 1 for them (all n output rows u: the twiddles depend on (u, a) only, so every lane executes the same code).  The
// lanes of a lenslet swap through a warp-private patch of shared memory (__syncwarp, no block barrier); lane p then runs
// pass 2 for the output rows 2p, 2p+1 (and n + those), |.|^2 and the binning, and stores binned rows p and p + n/2.
// A third of the registers of the one-thread-per-lenslet kernel -> twice the resident warps.
// ---------------------------------------------------------------------------------------------------------
template <int n>
__global__ void __launch_bounds__(128, 4)
shwfs_frame_split_kernel(const float* __restrict__ opd_a, const float* __restrict__ opd_b, const float* __restrict__ pupil,
                         const float* __restrict__ amp, const uint8_t* __restrict__ valid, int nS, float phase_scale,
                         int track_max, int shared_max, float* __restrict__ frame, int32_t* __restrict__ envmax,
                         double* __restrict__ stats) {
  constexpr int N = 2 * n, T = n / 2, h = n / 2, LPW = 32 / T, S = LPW + 1;
  // exchange: [warp][((kind * T + k) * n + u)][slot] float2, kind = Pr, Pi, Qr, Qi of output row u, column pair k
  __shared__ float2 xch[4][4 * T * n][S];
  const int R = nS * n;
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = lane / T, t = lane - slot * T;
  const int k = (blockIdx.x * 4 + warp) * LPW + slot;
  const bool active = slot < LPW && k < nS * nS;
  const int li = active ? k / nS : 0, lj = active ? k - li * nS : 0;
  const bool lit = active && valid[k] != 0;
  const float phase_turns = phase_scale * 0.15915494309189535f;
  const size_t tile = (size_t)(li * n) * R + lj * n;
  float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f;                         // pupil statistics, see shwfs_frame_kernel
  float2 er2[n], ei2[n];                                                  // (E[a][2t], E[a][2t+1])
  if (active) {
    const float* __restrict__ pa = opd_a + (size_t)b * R * R + tile;
    const float* __restrict__ pb = opd_b ? opd_b + (size_t)b * R * R + tile : nullptr;
    const size_t centre = (size_t)b * R * R + (size_t)(R / 2) * R + R / 2;
    const float ka = stats ? __ldg(opd_a + centre) : 0.f;
    const float kt = stats ? (opd_b ? ka + __ldg(opd_b + centre) : ka) : 0.f;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int bb = 2 * t + e;
#pragma unroll
      for (int a2 = 0; a2 < h; ++a2) {
        const int o2 = bb * R + 2 * a2;
        const float2 av = __ldg(reinterpret_cast<const float2*>(pa + o2));
        const float2 bv = pb ? __ldg(reinterpret_cast<const float2*>(pb + o2)) : make_float2(0.f, 0.f);
        const float2 pv = __ldg(reinterpret_cast<const float2*>(pupil + tile + o2));
        const float2 mv = lit ? __ldg(reinterpret_cast<const float2*>(amp + tile + o2)) : make_float2(0.f, 0.f);
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
          const int aa = 2 * a2 + h2;
          const float a = h2 ? av.y : av.x;
          const float tt = a + (h2 ? bv.y : bv.x);
          const float pu = h2 ? pv.y : pv.x;
          const float in_pupil = pu > 0.f ? 1.f : 0.f;
          const float da = (a - ka) * in_pupil, dt = (tt - kt) * in_pupil;
          f0 += da; f1 = fmaf(da, da, f1); f2 += dt; f3 = fmaf(dt, dt, f3);
          const float turns = tt * pu * phase_turns;
          const float ang = (turns - ((turns + 12582912.0f) - 12582912.0f)) * 6.283185307179586f;
          const float am = h2 ? mv.y : mv.x;
          const float cs = am * __cosf(ang), sn = am * __sinf(ang);
          if (e == 0) { er2[aa].x = cs; ei2[aa].x = sn; } else { er2[aa].y = cs; ei2[aa].y = sn; }
        }
      }
    }
  }
  if (stats != nullptr) {
    double s0 = warp_sum((double)f0), s1 = warp_sum((double)f1), s2 = warp_sum((double)f2), s3 = warp_sum((double)f3);
    if (lane == 0) {
      double* __restrict__ st = stats + (size_t)b * 4;
      atomicAdd(st, s0); atomicAdd(st + 1, s1); atomicAdd(st + 2, s2); atomicAdd(st + 3, s3);
    }
  }
  float2 (*x)[S] = xch[warp];
  const bool any_lit = __any_sync(0xffffffffu, lit);
  float vmax = -INFINITY;
  if (any_lit) {
    if (lit) {
      // pass 1 for this lane's column pair, every output row u < n (rows u + n follow by the radix-2 symmetry)
#pragma unroll
      for (int u = 0; u < n; ++u) {
        float2 pr = make_float2(0.f, 0.f), pi = pr, qr = pr, qi = pr;
#pragma unroll
        for (int aa = 0; aa < n; ++aa) {
          const float gx = WfsTw<n>::re(u * n + aa), gy = WfsTw<n>::im(u * n + aa);
          if (((aa + h) & 1) == 0) {
            pr = fma2(dup2(gx), er2[aa], fma2(dup2(-gy), ei2[aa], pr));
            pi = fma2(dup2(gx), ei2[aa], fma2(dup2(gy), er2[aa], pi));
          } else {
            qr = fma2(dup2(gx), er2[aa], fma2(dup2(-gy), ei2[aa], qr));
            qi = fma2(dup2(gx), ei2[aa], fma2(dup2(gy), er2[aa], qi));
          }
        }
        x[(0 * T + t) * n + u][slot] = pr;
        x[(1 * T + t) * n + u][slot] = pi;
        x[(2 * T + t) * n + u][slot] = qr;
        x[(3 * T + t) * n + u][slot] = qi;
      }
    }
    __syncwarp();
    if (lit) {
      float* __restrict__ fout = frame + (size_t)b * R * R + tile;
      const float norm = 1.0f / (float)(N * N);
      float2 acc[n];                         // acc[q] = (binned row t, binned row t + n/2) at binned column q
#pragma unroll
      for (int q = 0; q < n; ++q) acc[q] = make_float2(0.f, 0.f);
#pragma unroll
      for (int du = 0; du < 2; ++du) {
        const int u = 2 * t + du;
        float2 yr[n], yi[n];                 // (row u: P + Q, row u + n: P - Q)
#pragma unroll
        for (int kk = 0; kk < T; ++kk) {
          const float2 pr = x[(0 * T + kk) * n + u][slot], pi = x[(1 * T + kk) * n + u][slot];
          const float2 qr = x[(2 * T + kk) * n + u][slot], qi = x[(3 * T + kk) * n + u][slot];
          yr[2 * kk] = make_float2(pr.x + qr.x, pr.x - qr.x);
          yr[2 * kk + 1] = make_float2(pr.y + qr.y, pr.y - qr.y);
          yi[2 * kk] = make_float2(pi.x + qi.x, pi.x - qi.x);
          yi[2 * kk + 1] = make_float2(pi.y + qi.y, pi.y - qi.y);
        }
#pragma unroll
        for (int v = 0; v < n; ++v) {
          float2 er_ = make_float2(0.f, 0.f), ei_ = er_, or_ = er_, oi_ = er_;
#pragma unroll
          for (int bb = 0; bb < n; ++bb) {
            const float gx = WfsTw<n>::re(v * n + bb), gy = WfsTw<n>::im(v * n + bb);
            if (((bb + h) & 1) == 0) {
              er_ = fma2(yr[bb], dup2(gx), fma2(yi[bb], dup2(-gy), er_));
              ei_ = fma2(yr[bb], dup2(gy), fma2(yi[bb], dup2(gx), ei_));
            } else {
              or_ = fma2(yr[bb], dup2(gx), fma2(yi[bb], dup2(-gy), or_));
              oi_ = fma2(yr[bb], dup2(gy), fma2(yi[bb], dup2(gx), oi_));
            }
          }
          const float2 f0r = add2(er_, or_), f0i = add2(ei_, oi_);     // F[row][v]
          const float2 f1r = sub2(er_, or_), f1i = sub2(ei_, oi_);     // F[row][v + n]
          acc[v >> 1] = add2(acc[v >> 1], fma2(f0r, f0r, mul2(f0i, f0i)));
          acc[(v >> 1) + h] = add2(acc[(v >> 1) + h], fma2(f1r, f1r, mul2(f1i, f1i)));
        }
      }
#pragma unroll
      for (int q2 = 0; q2 < h; ++q2) {
        const float2 lo = make_float2(acc[2 * q2].x * norm, acc[2 * q2 + 1].x * norm);
        const float2 hi = make_float2(acc[2 * q2].y * norm, acc[2 * q2 + 1].y * norm);
        *reinterpret_cast<float2*>(fout + (size_t)t * R + 2 * q2) = lo;
        *reinterpret_cast<float2*>(fout + (size_t)(t + h) * R + 2 * q2) = hi;
        vmax = fmaxf(vmax, fmaxf(fmaxf(lo.x, lo.y), fmaxf(hi.x, hi.y)));
      }
    }
  }
  if (active && !lit) {                                                   // dark lenslet: rows 2t, 2t+1 of its tile
    float* __restrict__ fout = frame + (size_t)b * R * R + tile;
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
      for (int q2 = 0; q2 < h; ++q2) *reinterpret_cast<float2*>(fout + (size_t)(2 * t + e) * R + 2 * q2) = make_float2(0.f, 0.f);
  }
  if (track_max) {
    vmax = warp_max(vmax);
    if (lane == 0 && vmax > -INFINITY) atomicMax(&envmax[shared_max ? 0 : b], float_to_ordered(vmax));
  }
}

// ---------------------------------------------------------------------------------------------------------
// n = 10, 12 (the spots kernel of the wide lenslets, both in aoenv_shwfs_frame and in aoenv_shwfs_frame_dm): the arithmetic
// of shwfs_frame_kernel — radix-2 split of both pruned DFT passes, packed FP32, literal twiddles — on T = n / 2 lanes per
// lenslet.  One thread per lenslet would hold the 2 n^2 floats of the field next to the pass-2 rows and accumulators
// (~360 live floats at n = 12).  Lane t owns tile rows 2t, 2t+1 (= the column pair (2t, 2t+1) of the
// transposed field): it loads those 2n pixels, evaluates their DM surface in place (WL > 0, the same operations in the
// same order as shwfs_frame_kernel<n, WL>), accumulates the pupil statistics and forms the field.  Then two rounds, one per
// parity du of the output row: every lane runs pass 1 of its column pair for the rows u = 2p + du (p < T), the lanes of
// a lenslet swap those rows through a warp-private patch of shared memory (__syncwarp, no block barrier), and lane p runs
// pass 2 of row u = 2p + du (and u + n), |.|^2 and the binning into binned rows p and p + n/2.  Splitting by du halves the
// patch (27 KB per 128-thread CTA at n = 12 instead of 55 KB) at no cost in arithmetic.  `order` (nullable) visits the
// lenslets lit-first, as in shwfs_frame_kernel.
// ---------------------------------------------------------------------------------------------------------
template <int n, int WL>
__global__ void __launch_bounds__(128, n == 12 ? 3 : 4)      // n = 12: 168 registers, no spills (at 128 it spills)
shwfs_frame_wide_kernel(const float* __restrict__ opd_a, const float* __restrict__ opd_b, const float* __restrict__ pupil,
                        const float* __restrict__ amp, const uint8_t* __restrict__ valid, int nS, float phase_scale,
                        int track_max, int shared_max, float* __restrict__ frame, int32_t* __restrict__ envmax,
                        double* __restrict__ stats, const __grid_constant__ aoenv_dm_sep_t dm, const int32_t* __restrict__ order) {
  constexpr int N = 2 * n, T = n / 2, h = n / 2, LPW = 32 / T, S = LPW + 1;
  // exchange of one round: [warp][(kind * T + source lane) * T + destination lane][slot] float2, kind = Pr, Pi, Qr, Qi
  __shared__ float2 xch[4][4 * T * T][S];
  pdl_enter();
  const int R = nS * n;
  const int b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = lane / T, t = lane - slot * T;
  const int k0 = (blockIdx.x * 4 + warp) * LPW + slot;
  const bool active = slot < LPW && k0 < nS * nS;
  const int k = (active && order != nullptr) ? __ldg(&order[k0]) : k0;
  const int li = active ? k / nS : 0, lj = active ? k - li * nS : 0;
  const bool lit = active && valid[k] != 0;
  const float phase_turns = phase_scale * 0.15915494309189535f;
  const size_t tile = (size_t)(li * n) * R + lj * n;
  float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f;                         // pupil statistics, see shwfs_frame_kernel
  float2 er2[n], ei2[n];                                                  // (E[a][2t], E[a][2t+1])
  if (active) {
    const float* __restrict__ pa = opd_a + (size_t)b * R * R + tile;
    const float* __restrict__ pb = (WL == 0 && opd_b) ? opd_b + (size_t)b * R * R + tile : nullptr;
    const size_t centre = (size_t)b * R * R + (size_t)(R / 2) * R + R / 2;
    const float ka = stats ? __ldg(opd_a + centre) : 0.f;
    // (with the in-place DM the total is centred on the atmosphere's centre value, as in shwfs_frame_kernel)
    const float kt = stats ? (pb ? ka + __ldg(opd_b + centre) : ka) : 0.f;
    // DM surface of tile rows 2t + e: dmv[e][a2] = pixels (columns 2 a2, 2 a2 + 1)
    float2 dmv[2][WL > 0 ? h : 1];
    if constexpr (WL > 0) {
      constexpr int half = (WL + 1) / 2, hp = (half + 3) / 4 * 4;
#pragma unroll
      for (int e = 0; e < 2; ++e)
#pragma unroll
        for (int a2 = 0; a2 < h; ++a2) dmv[e][a2] = make_float2(0.f, 0.f);
      const float* __restrict__ trow = dm.rows + ((size_t)b * dm.nActP + __ldg(&dm.ilr[li])) * R + lj * n;
      const float* __restrict__ wrow = dm.wlr + (size_t)(li * n + 2 * t) * (2 * hp);
#pragma unroll
      for (int g = 0; g < 2 * hp / 4; ++g) {
        float4 w4[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) w4[e] = __ldg(reinterpret_cast<const float4*>(wrow + (size_t)e * (2 * hp)) + g);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int j = 4 * g + c, hh = j / hp, kk = j % hp;
          if (kk >= half) continue;                      // padding entries of the weight rows
          const int tr = hh * half + kk;
          if (tr >= WL) continue;
          float2 tv[h];
#pragma unroll
          for (int a2 = 0; a2 < h; ++a2) tv[a2] = __ldg(reinterpret_cast<const float2*>(trow + (size_t)tr * R) + a2);
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const float w = c == 0 ? w4[e].x : (c == 1 ? w4[e].y : (c == 2 ? w4[e].z : w4[e].w));
#pragma unroll
            for (int a2 = 0; a2 < h; ++a2) dmv[e][a2] = fma2(dup2(w), tv[a2], dmv[e][a2]);
          }
        }
      }
    }
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int bb = 2 * t + e;
#pragma unroll
      for (int a2 = 0; a2 < h; ++a2) {
        const int o2 = bb * R + 2 * a2;
        const float2 av = __ldg(reinterpret_cast<const float2*>(pa + o2));
        float2 bv;
        if constexpr (WL > 0) bv = dmv[e][a2];
        else bv = pb ? __ldg(reinterpret_cast<const float2*>(pb + o2)) : make_float2(0.f, 0.f);
        const float2 pv = __ldg(reinterpret_cast<const float2*>(pupil + tile + o2));
        const float2 mv = lit ? __ldg(reinterpret_cast<const float2*>(amp + tile + o2)) : make_float2(0.f, 0.f);
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
          const int aa = 2 * a2 + h2;
          const float a = h2 ? av.y : av.x;
          const float tt = a + (h2 ? bv.y : bv.x);
          const float pu = h2 ? pv.y : pv.x;
          const float in_pupil = pu > 0.f ? 1.f : 0.f;
          const float da = (a - ka) * in_pupil, dt = (tt - kt) * in_pupil;
          f0 += da; f1 = fmaf(da, da, f1); f2 += dt; f3 = fmaf(dt, dt, f3);
          const float turns = tt * pu * phase_turns;
          const float ang = (turns - ((turns + 12582912.0f) - 12582912.0f)) * 6.283185307179586f;
          const float am = h2 ? mv.y : mv.x;
          const float cs = am * __cosf(ang), sn = am * __sinf(ang);
          if (e == 0) { er2[aa].x = cs; ei2[aa].x = sn; } else { er2[aa].y = cs; ei2[aa].y = sn; }
        }
      }
    }
  }
  if (stats != nullptr) {       // one atomic per warp and statistic
    double s0 = warp_sum((double)f0), s1 = warp_sum((double)f1), s2 = warp_sum((double)f2), s3 = warp_sum((double)f3);
    if (lane == 0) {
      double* __restrict__ st = stats + (size_t)b * 4;
      atomicAdd(st, s0); atomicAdd(st + 1, s1); atomicAdd(st + 2, s2); atomicAdd(st + 3, s3);
    }
  }
  float2 (*x)[S] = xch[warp];
  const bool any_lit = __any_sync(0xffffffffu, lit);
  float vmax = -INFINITY;
  if (any_lit) {                                                          // warp-uniform: every lane meets the __syncwarps
    float2 acc[n];                         // acc[q] = (binned row t, binned row t + n/2) at binned column q
#pragma unroll
    for (int q = 0; q < n; ++q) acc[q] = make_float2(0.f, 0.f);
#pragma unroll
    for (int du = 0; du < 2; ++du) {
      if (lit) {
        // pass 1 for this lane's column pair, output rows u = 2p + du (rows u + n follow by the radix-2 symmetry)
#pragma unroll
        for (int p = 0; p < T; ++p) {
          const int u = 2 * p + du;
          float2 pr = make_float2(0.f, 0.f), pi = pr, qr = pr, qi = pr;
#pragma unroll
          for (int aa = 0; aa < n; ++aa) {
            const float gx = WfsTw<n>::re(u * n + aa), gy = WfsTw<n>::im(u * n + aa);
            if (((aa + h) & 1) == 0) {
              pr = fma2(dup2(gx), er2[aa], fma2(dup2(-gy), ei2[aa], pr));
              pi = fma2(dup2(gx), ei2[aa], fma2(dup2(gy), er2[aa], pi));
            } else {
              qr = fma2(dup2(gx), er2[aa], fma2(dup2(-gy), ei2[aa], qr));
              qi = fma2(dup2(gx), ei2[aa], fma2(dup2(gy), er2[aa], qi));
            }
          }
          x[(0 * T + t) * T + p][slot] = pr;
          x[(1 * T + t) * T + p][slot] = pi;
          x[(2 * T + t) * T + p][slot] = qr;
          x[(3 * T + t) * T + p][slot] = qi;
        }
      }
      __syncwarp();
      if (lit) {
        float2 yr[n], yi[n];                 // (row u: P + Q, row u + n: P - Q), u = 2t + du
#pragma unroll
        for (int kk = 0; kk < T; ++kk) {
          const float2 pr = x[(0 * T + kk) * T + t][slot], pi = x[(1 * T + kk) * T + t][slot];
          const float2 qr = x[(2 * T + kk) * T + t][slot], qi = x[(3 * T + kk) * T + t][slot];
          yr[2 * kk] = make_float2(pr.x + qr.x, pr.x - qr.x);
          yr[2 * kk + 1] = make_float2(pr.y + qr.y, pr.y - qr.y);
          yi[2 * kk] = make_float2(pi.x + qi.x, pi.x - qi.x);
          yi[2 * kk + 1] = make_float2(pi.y + qi.y, pi.y - qi.y);
        }
#pragma unroll
        for (int v = 0; v < n; ++v) {
          float2 er_ = make_float2(0.f, 0.f), ei_ = er_, or_ = er_, oi_ = er_;
#pragma unroll
          for (int bb = 0; bb < n; ++bb) {
            const float gx = WfsTw<n>::re(v * n + bb), gy = WfsTw<n>::im(v * n + bb);
            if (((bb + h) & 1) == 0) {
              er_ = fma2(yr[bb], dup2(gx), fma2(yi[bb], dup2(-gy), er_));
              ei_ = fma2(yr[bb], dup2(gy), fma2(yi[bb], dup2(gx), ei_));
            } else {
              or_ = fma2(yr[bb], dup2(gx), fma2(yi[bb], dup2(-gy), or_));
              oi_ = fma2(yr[bb], dup2(gy), fma2(yi[bb], dup2(gx), oi_));
            }
          }
          const float2 f0r = add2(er_, or_), f0i = add2(ei_, oi_);     // F[row][v]
          const float2 f1r = sub2(er_, or_), f1i = sub2(ei_, oi_);     // F[row][v + n]
          acc[v >> 1] = add2(acc[v >> 1], fma2(f0r, f0r, mul2(f0i, f0i)));
          acc[(v >> 1) + h] = add2(acc[(v >> 1) + h], fma2(f1r, f1r, mul2(f1i, f1i)));
        }
      }
      __syncwarp();                                                       // the patch is rewritten by the next round
    }
    if (lit) {
      float* __restrict__ fout = frame + (size_t)b * R * R + tile;
      const float norm = 1.0f / (float)(N * N);
#pragma unroll
      for (int q2 = 0; q2 < h; ++q2) {
        const float2 lo = make_float2(acc[2 * q2].x * norm, acc[2 * q2 + 1].x * norm);
        const float2 hi = make_float2(acc[2 * q2].y * norm, acc[2 * q2 + 1].y * norm);
        *reinterpret_cast<float2*>(fout + (size_t)t * R + 2 * q2) = lo;
        *reinterpret_cast<float2*>(fout + (size_t)(t + h) * R + 2 * q2) = hi;
        vmax = fmaxf(vmax, fmaxf(fmaxf(lo.x, lo.y), fmaxf(hi.x, hi.y)));
      }
    }
  }
  if (active && !lit) {                                                   // dark lenslet: rows 2t, 2t+1 of its tile
    float* __restrict__ fout = frame + (size_t)b * R * R + tile;
#pragma unroll
    for (int e = 0; e < 2; ++e)
#pragma unroll
      for (int q2 = 0; q2 < h; ++q2) *reinterpret_cast<float2*>(fout + (size_t)(2 * t + e) * R + 2 * q2) = make_float2(0.f, 0.f);
  }
  if (track_max) {            // with a camera model the maximum is taken after the detector pass
    vmax = warp_max(vmax);
    if (lane == 0 && vmax > -INFINITY) atomicMax(&envmax[shared_max ? 0 : b], float_to_ordered(vmax));
  }
}

// centroid + slopes: one thread per (valid lenslet, environment).  n is a template parameter so that the 6 x 6 (4 x 4,
// 8 x 8, 10 x 10, 12 x 12) spot is read with fully unrolled 64-bit loads (tile rows start on even columns: lj * n with n
// even).
template <int n>
__global__ void __launch_bounds__(128)
shwfs_slopes_kernel(const float* __restrict__ frame, const int32_t* __restrict__ envmax, int shared_max,
                    const int32_t* __restrict__ valid_idx, int nV, const float* __restrict__ ref_xy, float inv_units,
                    float threshold_cog, int nS, float* __restrict__ slopes, int lds,
                    __nv_bfloat16* __restrict__ planes, int parts) {
  const int b = blockIdx.y;
  pdl_enter();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nV) return;
  const int R = nS * n;
  const int k = __ldg(&valid_idx[t]);
  const int li = k / nS, lj = k - li * nS;
  const float thr = threshold_cog * ordered_to_float(__ldg(&envmax[shared_max ? 0 : b]));
  const float* __restrict__ f = frame + (size_t)b * R * R + (size_t)(li * n) * R + lj * n;
  float2 v[n][n / 2];
#pragma unroll
  for (int p = 0; p < n; ++p)
#pragma unroll
    for (int h = 0; h < n / 2; ++h) v[p][h] = __ldg(reinterpret_cast<const float2*>(f + (size_t)p * R) + h);
  float s = 0.f, sx = 0.f, sy = 0.f;
#pragma unroll
  for (int p = 0; p < n; ++p)
#pragma unroll
    for (int q = 0; q < n; ++q) {
      float x = (q & 1) ? v[p][q >> 1].y : v[p][q >> 1].x;
      x = x < thr ? 0.f : x;
      s += x;
      sx = fmaf(x, (float)p, sx);   // axis 1 of maps_intensity -> centroid[:,0] -> SX (ShackHartmann.py:321,596)
      sy = fmaf(x, (float)q, sy);   // axis 2 -> centroid[:,1] -> SY
    }
  float cx = sx / s, cy = sy / s;
  if (!isfinite(cx)) cx = 0.f;      // ShackHartmann.py:583-593
  if (!isfinite(cy)) cy = 0.f;
  const float sx_ = (cx - __ldg(&ref_xy[t])) * inv_units, sy_ = (cy - __ldg(&ref_xy[nV + t])) * inv_units;
  slopes[(size_t)b * lds + t] = sx_;
  slopes[(size_t)b * lds + nV + t] = sy_;
  if (planes != nullptr) {      // operand planes of the reconstruction GEMM (padding columns stay zero from allocation)
    store_bf16_planes(planes, (size_t)gridDim.y * lds, (size_t)b * lds + t, parts, sx_);
    store_bf16_planes(planes, (size_t)gridDim.y * lds, (size_t)b * lds + nV + t, parts, sy_);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Calibration-grade (float64) variant: ideal detector, used at init for the reference slopes, the slope units
// (ShackHartmann.py:254-312) and the interaction matrix (calibration/InteractionMatrix.py), whose 1 nm pokes move
// the spots by ~1e-3 pixel — below what float32 centroids resolve to 1e-4.  Intensities are >= 0, so the bit
// pattern of a double orders like the value and atomicMax on unsigned long long gives the frame maximum.
// ---------------------------------------------------------------------------------------------------------
template <int n>
__global__ void __launch_bounds__(64)
shwfs_frame_f64_kernel(const float* __restrict__ opd, const float* __restrict__ pupil, const float* __restrict__ amp,
                       const uint8_t* __restrict__ valid, int nS, double phase_scale, int shared_max,
                       double* __restrict__ frame, unsigned long long* __restrict__ envmax) {
  constexpr int N = 2 * n;
  const int R = nS * n;
  const int b = blockIdx.y;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nS * nS) return;
  const int li = k / nS, lj = k % nS;
  const bool lit = valid[k] != 0;
  const size_t tile = (size_t)(li * n) * R + lj * n;
  double* __restrict__ fout = frame + (size_t)b * R * R + tile;
  if (!lit) {
    for (int p = 0; p < n; ++p)
      for (int q = 0; q < n; ++q) fout[(size_t)p * R + q] = 0.0;
    return;
  }
  double er[n][n], ei[n][n];
  const float* __restrict__ pa = opd + (size_t)b * R * R + tile;
#pragma unroll
  for (int bb = 0; bb < n; ++bb)
#pragma unroll
    for (int aa = 0; aa < n; ++aa) {
      const int o = bb * R + aa;
      double sn, cs;
      sincos((double)__ldg(pa + o) * (double)__ldg(pupil + tile + o) * phase_scale, &sn, &cs);
      const double am = (double)__ldg(amp + tile + o);
      er[aa][bb] = am * cs;
      ei[aa][bb] = am * sn;
    }
  double vmax = 0.0;
  const double norm = 1.0 / (double)(N * N);
  for (int p = 0; p < n; ++p) {
    double acc[n];
#pragma unroll
    for (int q = 0; q < n; ++q) acc[q] = 0.0;
    for (int du = 0; du < 2; ++du) {
      const int u = 2 * p + du;
      double yr[n], yi[n];
#pragma unroll
      for (int bb = 0; bb < n; ++bb) { yr[bb] = 0.0; yi[bb] = 0.0; }
#pragma unroll
      for (int aa = 0; aa < n; ++aa) {
        const double2 g = twd<n>(u * n + aa);
#pragma unroll
        for (int bb = 0; bb < n; ++bb) {
          yr[bb] += g.x * er[aa][bb] - g.y * ei[aa][bb];
          yi[bb] += g.x * ei[aa][bb] + g.y * er[aa][bb];
        }
      }
#pragma unroll
      for (int v = 0; v < N; ++v) {
        double fr = 0.0, fi = 0.0;
#pragma unroll
        for (int bb = 0; bb < n; ++bb) {
          const double2 g = twd<n>(v * n + bb);
          fr += yr[bb] * g.x - yi[bb] * g.y;
          fi += yr[bb] * g.y + yi[bb] * g.x;
        }
        acc[v >> 1] += fr * fr + fi * fi;
      }
    }
#pragma unroll
    for (int q = 0; q < n; ++q) {
      const double val = acc[q] * norm;
      fout[(size_t)p * R + q] = val;
      vmax = fmax(vmax, val);
    }
  }
  atomicMax(&envmax[shared_max ? 0 : b], (unsigned long long)__double_as_longlong(vmax));
}

__global__ void __launch_bounds__(128)
shwfs_slopes_f64_kernel(const double* __restrict__ frame, const unsigned long long* __restrict__ envmax, int shared_max,
                        const int32_t* __restrict__ valid_idx, int nV, const double* __restrict__ ref_xy,
                        double inv_units, double threshold_cog, int nS, int n, double* __restrict__ slopes, int lds) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nV) return;
  const int R = nS * n;
  const int k = __ldg(&valid_idx[t]);
  const int li = k / nS, lj = k % nS;
  const double thr = threshold_cog * __longlong_as_double((long long)envmax[shared_max ? 0 : b]);
  const double* __restrict__ f = frame + (size_t)b * R * R + (size_t)(li * n) * R + lj * n;
  double s = 0.0, sx = 0.0, sy = 0.0;
  for (int p = 0; p < n; ++p)
    for (int q = 0; q < n; ++q) {
      double v = f[(size_t)p * R + q];
      v = v < thr ? 0.0 : v;
      s += v;
      sx += v * (double)p;
      sy += v * (double)q;
    }
  double cx = sx / s, cy = sy / s;
  if (!isfinite(cx)) cx = 0.0;
  if (!isfinite(cy)) cy = 0.0;
  slopes[(size_t)b * lds + t] = (cx - ref_xy[t]) * inv_units;
  slopes[(size_t)b * lds + nV + t] = (cy - ref_xy[nV + t]) * inv_units;
}

// Resets the per-environment maxima and (optionally) the pupil statistics in one launch: a memset node between two kernels
// would cut the programmatic-dependent-launch chain of the step.
__global__ void envmax_init_kernel(int32_t* __restrict__ envmax, int count, double* __restrict__ stats, int n_stats) {
  pdl_enter();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) envmax[i] = float_to_ordered(-INFINITY);
  if (stats != nullptr && i < n_stats) stats[i] = 0.0;
}

}  // namespace aoenv

using namespace aoenv;

// Implementations of the same frame (aoenv_set_wfs6_variant / AOENV_WFS_FRAME=termwise|factorised|split6|split):
//   0 term-by-term transform, one thread per lenslet (shwfs_frame_kernel<n>)
//   1 factorised transform (radix 2 x Good-Thomas 2 x 3), one thread per lenslet, n = 6 (shwfs_frame6_kernel)
//   2 factorised transform on three lanes per lenslet, n = 6 (shwfs_frame6s_kernel)
//   3 term-by-term transform on n / 2 lanes per lenslet (shwfs_frame_split_kernel<n>)
// The tests run all of them against the oracle; the default is the one measured fastest on B200 (profiles/).
constexpr int kDefaultFrameVariant = 0;
static std::atomic<int> g_wfs6_factorised{[] {
  const char* e = getenv("AOENV_WFS_FRAME");      // termwise | factorised | split6 | split
  if (e && e[0] == 'f') return 1;
  if (e && e[0] == 's') return (e[5] == '6') ? 2 : 3;
  if (e && e[0] == 't') return 0;
  return kDefaultFrameVariant;
}()};

extern "C" {

int aoenv_set_wfs6_variant(int variant) {
  return g_wfs6_factorised.exchange(variant < 0 || variant > 3 ? kDefaultFrameVariant : variant);
}

static int shwfs_frame_impl(const float* opd_a, const float* opd_b, const aoenv_dm_sep_t* dm_in, const int32_t* order, const float* pupil,
                            const float* amp, const uint8_t* valid, int B, int nS, int n, float phase_scale,
                            const aoenv_detector_t* det, int shared_max, float* frame, int32_t* envmax, double* stats,
                            void* stream) {
  AOENV_CHECK_ARG(B > 0 && B <= 65535 && nS > 0, "shwfs_frame: bad shape B=%d nS=%d", B, nS);
  aoenv_dm_sep_t dm{};
  if (dm_in != nullptr) {
    dm = *dm_in;
    AOENV_CHECK_ARG(opd_b == nullptr, "shwfs_frame_dm: give either the separable DM or an explicit second OPD term");
    AOENV_CHECK_ARG(dm.rows != nullptr && dm.wlr != nullptr && dm.ilr != nullptr && dm.nActP > 0, "shwfs_frame_dm: bad DM tables");
    AOENV_CHECK_ARG(dm.WL == 14 || dm.WL == 18, "shwfs_frame_dm: DM window of %d actuator rows (14 or 18)", dm.WL);
    AOENV_CHECK_ARG((reinterpret_cast<uintptr_t>(dm.rows) & 7) == 0 && (reinterpret_cast<uintptr_t>(dm.wlr) & 15) == 0,
                    "shwfs_frame_dm: DM tables must be 16-byte aligned");
  }
  AOENV_CHECK_ARG(n == 4 || n == 6 || n == 8 || n == 10 || n == 12,
                  "shwfs_frame: %d pixels per lenslet is not a compiled size (4, 6, 8, 10, 12)", n);
  const int variant = g_wfs6_factorised.load(std::memory_order_relaxed);
  AOENV_CHECK_ARG(n <= 8 || variant == 0,
                  "shwfs_frame: the alternative frame variant %d (aoenv_set_wfs6_variant / AOENV_WFS_FRAME) is compiled for "
                  "4, 6, 8 pixels per lenslet, not %d", variant, n);
  cudaStream_t s = (cudaStream_t)stream;
  if (det) {
    AOENV_CHECK_ARG(!(det->bits > 0 && !det->has_fwc), "shwfs_frame: ADC without a full-well capacity is not supported");
    AOENV_CHECK_ARG(det->bits >= 0 && det->bits < 31, "shwfs_frame: bits=%d", det->bits);
  }
  int rc = ensure_twiddles(n, s);
  if (rc) return rc;
  AOENV_LAUNCH(envmax_init_kernel, dim3((4 * B + 255) / 256), 256, 0, s, envmax, shared_max ? 1 : B, stats, stats ? 4 * B : 0);
  AOENV_LAUNCH_CHECK("envmax_init");
  dim3 grid((nS * nS + 127) / 128, B);
  if (n > 8) {                                 // n / 2 lanes per lenslet, 4 warps per CTA
    const int per_block = 4 * (32 / (n / 2));
    dim3 gw((nS * nS + per_block - 1) / per_block, B);
#define AOENV_WFS_WIDE(NN, WW)                                                                                            \
  AOENV_LAUNCH((shwfs_frame_wide_kernel<NN, WW>), gw, 128, 0, s, opd_a, opd_b, pupil, amp, valid, nS, phase_scale,        \
               (int)(det == nullptr), shared_max, frame, envmax, stats, dm, order)
    if (n == 10) {
      if (dm.WL == 14) AOENV_WFS_WIDE(10, 14);
      else if (dm.WL == 18) AOENV_WFS_WIDE(10, 18);
      else AOENV_WFS_WIDE(10, 0);
    } else {
      if (dm.WL == 14) AOENV_WFS_WIDE(12, 14);
      else if (dm.WL == 18) AOENV_WFS_WIDE(12, 18);
      else AOENV_WFS_WIDE(12, 0);
    }
#undef AOENV_WFS_WIDE
  } else if (variant == 3 && dm.WL == 0) {     // n / 2 lanes per lenslet, any compiled n
    const int per_block = 4 * (32 / (n / 2));
    dim3 g3((nS * nS + per_block - 1) / per_block, B);
    if (n == 4) shwfs_frame_split_kernel<4><<<g3, 128, 0, s>>>(opd_a, opd_b, pupil, amp, valid, nS, phase_scale, det == nullptr, shared_max, frame, envmax, stats);
    else if (n == 6) shwfs_frame_split_kernel<6><<<g3, 128, 0, s>>>(opd_a, opd_b, pupil, amp, valid, nS, phase_scale, det == nullptr, shared_max, frame, envmax, stats);
    else shwfs_frame_split_kernel<8><<<g3, 128, 0, s>>>(opd_a, opd_b, pupil, amp, valid, nS, phase_scale, det == nullptr, shared_max, frame, envmax, stats);
  } else
#define AOENV_WFS_CASE(NN)                                                                                   \
  case NN:                                                                                                   \
    if (dm.WL == 14)                                                                                         \
      AOENV_LAUNCH((shwfs_frame_kernel<NN, 14>), grid, 128, 0, s, opd_a, opd_b, pupil, amp, valid, nS, phase_scale, \
                   (int)(det == nullptr), shared_max, frame, envmax, stats, dm, order);                             \
    else if (dm.WL == 18)                                                                                    \
      AOENV_LAUNCH((shwfs_frame_kernel<NN, 18>), grid, 128, 0, s, opd_a, opd_b, pupil, amp, valid, nS, phase_scale, \
                   (int)(det == nullptr), shared_max, frame, envmax, stats, dm, order);                             \
    else                                                                                                     \
      AOENV_LAUNCH((shwfs_frame_kernel<NN, 0>), grid, 128, 0, s, opd_a, opd_b, pupil, amp, valid, nS, phase_scale,  \
                   (int)(det == nullptr), shared_max, frame, envmax, stats, dm, order);                             \
    break;
  switch (n) {
    AOENV_WFS_CASE(4)
    AOENV_WFS_CASE(8)
    case 6:
      if (dm.WL != 0) {
        if (dm.WL == 14) {
          AOENV_LAUNCH((shwfs_frame_kernel<6, 14>), grid, 128, 0, s, opd_a, opd_b, pupil, amp, valid, nS, phase_scale,
                       (int)(det == nullptr), shared_max, frame, envmax, stats, dm, order);
        } else
          AOENV_LAUNCH((shwfs_frame_kernel<6, 18>), grid, 128, 0, s, opd_a, opd_b, pupil, amp, valid, nS, phase_scale,
                       (int)(det == nullptr), shared_max, frame, envmax, stats, dm, order);
      } else if (variant == 2) {
        dim3 g3((nS * nS + kS6Warps * kS6Lenslets - 1) / (kS6Warps * kS6Lenslets), B);
        shwfs_frame6s_kernel<<<g3, kS6Warps * 32, 0, s>>>(opd_a, opd_b, pupil, amp, valid, nS, phase_scale, det == nullptr,
                                                          shared_max, frame, envmax, stats);
      } else if (variant == 1)
        shwfs_frame6_kernel<<<grid, 128, 0, s>>>(opd_a, opd_b, pupil, amp, valid, nS, phase_scale, det == nullptr, shared_max,
                                                 frame, envmax, stats);
      else
        AOENV_LAUNCH((shwfs_frame_kernel<6, 0>), grid, 128, 0, s, opd_a, opd_b, pupil, amp, valid, nS, phase_scale,
                     (int)(det == nullptr), shared_max, frame, envmax, stats, dm, order);
      break;
  }
#undef AOENV_WFS_CASE
  AOENV_LAUNCH_CHECK("shwfs_frame");
  if (det) {
    const int R = nS * n;
    AOENV_CHECK_ARG(R * R < (1 << 24), "shwfs_frame: frame of %d x %d pixels is too large for the camera pass", R, R);
    dim3 gd((R * R + 8 * kDetPerLane * 32 - 1) / (8 * kDetPerLane * 32), B);
    AOENV_LAUNCH(shwfs_detector_kernel, gd, 256, 0, s, frame, valid, nS, n, 1.0f / (float)R, 1.0f / (float)n, *det, shared_max, envmax, 0);
    AOENV_LAUNCH_CHECK("shwfs_detector");
  }
  return 0;
}

int aoenv_shwfs_frame(const float* opd_a, const float* opd_b, const float* pupil, const float* amp,
                      const uint8_t* valid, int B, int nS, int n, float phase_scale, const aoenv_detector_t* det,
                      int shared_max, float* frame, int32_t* envmax, double* stats, void* stream) {
  return shwfs_frame_impl(opd_a, opd_b, nullptr, nullptr, pupil, amp, valid, B, nS, n, phase_scale, det, shared_max, frame, envmax, stats, stream);
}

int aoenv_shwfs_frame_dm(const float* opd_a, const float* opd_b, const aoenv_dm_sep_t* dm, const int32_t* order,
                         const float* pupil, const float* amp, const uint8_t* valid, int B, int nS, int n, float phase_scale,
                         const aoenv_detector_t* det, int shared_max, float* frame, int32_t* envmax, double* stats,
                         void* stream) {
  return shwfs_frame_impl(opd_a, opd_b, dm, order, pupil, amp, valid, B, nS, n, phase_scale, det, shared_max, frame, envmax, stats, stream);
}

int aoenv_shwfs_camera(float* frame, const uint8_t* valid, int B, int nS, int n, const aoenv_detector_t* det, int shared_max,
                       int32_t* envmax, void* stream) {
  AOENV_CHECK_ARG(B > 0 && B <= 65535 && nS > 0 && n > 0, "shwfs_camera: bad shape B=%d nS=%d", B, nS);
  AOENV_CHECK_ARG(det != nullptr && valid != nullptr && envmax != nullptr, "shwfs_camera: detector, lenslet mask and envmax are required");
  AOENV_CHECK_ARG(!(det->bits > 0 && !det->has_fwc), "shwfs_camera: ADC without a full-well capacity is not supported");
  AOENV_CHECK_ARG(det->bits >= 0 && det->bits < 31, "shwfs_camera: bits=%d", det->bits);
  const int R = nS * n;
  AOENV_CHECK_ARG(R * R < (1 << 24), "shwfs_camera: frame of %d x %d pixels is too large for the camera pass", R, R);
  cudaStream_t s = (cudaStream_t)stream;
  AOENV_LAUNCH(envmax_init_kernel, dim3((B + 255) / 256), 256, 0, s, envmax, shared_max ? 1 : B, (double*)nullptr, 0);
  AOENV_LAUNCH_CHECK("envmax_init");
  dim3 gd((R * R + 8 * kDetPerLane * 32 - 1) / (8 * kDetPerLane * 32), B);
  shwfs_detector_kernel<<<gd, 256, 0, s>>>(frame, valid, nS, n, 1.0f / (float)R, 1.0f / (float)n, *det, shared_max, envmax, 0);
  AOENV_LAUNCH_CHECK("shwfs_detector");
  return 0;
}

int aoenv_detector_integrate(float* frame, int B, int rows, int cols, const aoenv_detector_t* det, void* stream) {
  AOENV_CHECK_ARG(B > 0 && B <= 65535 && rows > 0 && cols > 0 && (long long)rows * cols < (1 << 24), "detector_integrate: bad shape");
  AOENV_CHECK_ARG(det != nullptr, "detector_integrate: no detector given");
  AOENV_CHECK_ARG(!(det->bits > 0 && !det->has_fwc), "detector_integrate: ADC without a full-well capacity is not supported");
  AOENV_CHECK_ARG(det->bits >= 0 && det->bits < 31, "detector_integrate: bits=%d", det->bits);
  const int P = rows * cols;
  dim3 gd((P + 8 * kDetPerLane * 32 - 1) / (8 * kDetPerLane * 32), B);
  // the kernel only needs P = R * R pixels per frame when no lenslet mask is given: pass nS * n = 1 * P via (nS, n) = (P, 1)
  shwfs_detector_kernel<<<gd, 256, 0, (cudaStream_t)stream>>>(frame, nullptr, 1, 1, 1.0f, 1.0f, *det, 0, nullptr, P);
  AOENV_LAUNCH_CHECK("detector_integrate");
  return 0;
}

int aoenv_shwfs_slopes(const float* frame, const int32_t* envmax, int shared_max, const int32_t* valid_idx, int nV,
                       const float* ref_xy, float inv_units, float threshold_cog, int B, int nS, int n, float* slopes,
                       int lds, void* slope_planes, int parts, void* stream) {
  AOENV_CHECK_ARG(B > 0 && B <= 65535 && nV > 0 && lds >= 2 * nV, "shwfs_slopes: bad shape B=%d nV=%d lds=%d", B, nV, lds);
  AOENV_CHECK_ARG(n == 4 || n == 6 || n == 8 || n == 10 || n == 12,
                  "shwfs_slopes: %d pixels per lenslet is not a compiled size (4, 6, 8, 10, 12)", n);
  AOENV_CHECK_ARG((reinterpret_cast<uintptr_t>(frame) & 7) == 0, "shwfs_slopes: frame must be 8-byte aligned");
  dim3 grid((nV + 127) / 128, B);
#define AOENV_SLOPES_CASE(NN)                                                                                          \
  case NN:                                                                                                             \
    AOENV_LAUNCH(shwfs_slopes_kernel<NN>, grid, 128, 0, (cudaStream_t)stream, frame, envmax, shared_max, valid_idx, nV, \
                 ref_xy, inv_units, threshold_cog, nS, slopes, lds, (__nv_bfloat16*)slope_planes, parts);              \
    break;
  switch (n) {
    AOENV_SLOPES_CASE(4)
    AOENV_SLOPES_CASE(6)
    AOENV_SLOPES_CASE(8)
    AOENV_SLOPES_CASE(10)
    AOENV_SLOPES_CASE(12)
  }
#undef AOENV_SLOPES_CASE
  AOENV_LAUNCH_CHECK("shwfs_slopes");
  return 0;
}

int aoenv_shwfs_measure_f64(const float* opd, const float* pupil, const float* amp, const uint8_t* valid,
                            const int32_t* valid_idx, int nV, const double* ref_xy, double inv_units, double threshold_cog,
                            int F, int nS, int n, double phase_scale, int shared_max, double* frame, uint64_t* envmax,
                            double* slopes, int lds, void* stream) {
  AOENV_CHECK_ARG(F > 0 && F <= 65535 && nS > 0 && nV > 0 && lds >= 2 * nV, "shwfs_measure_f64: bad shape");
  AOENV_CHECK_ARG(n == 4 || n == 6 || n == 8 || n == 10 || n == 12,
                  "shwfs_measure_f64: %d pixels per lenslet is not a compiled size (4, 6, 8, 10, 12)", n);
  cudaStream_t s = (cudaStream_t)stream;
  int rc = ensure_twiddles(n, s);
  if (rc) return rc;
  cudaError_t e = cudaMemsetAsync(envmax, 0, sizeof(uint64_t) * (shared_max ? 1 : (size_t)F), s);
  if (e != cudaSuccess) return fail(-3, "shwfs_measure_f64 memset: %s", cudaGetErrorString(e));
  dim3 grid((nS * nS + 63) / 64, F);
  unsigned long long* em = reinterpret_cast<unsigned long long*>(envmax);
  switch (n) {
    case 4: shwfs_frame_f64_kernel<4><<<grid, 64, 0, s>>>(opd, pupil, amp, valid, nS, phase_scale, shared_max, frame, em); break;
    case 6: shwfs_frame_f64_kernel<6><<<grid, 64, 0, s>>>(opd, pupil, amp, valid, nS, phase_scale, shared_max, frame, em); break;
    case 8: shwfs_frame_f64_kernel<8><<<grid, 64, 0, s>>>(opd, pupil, amp, valid, nS, phase_scale, shared_max, frame, em); break;
    case 10: shwfs_frame_f64_kernel<10><<<grid, 64, 0, s>>>(opd, pupil, amp, valid, nS, phase_scale, shared_max, frame, em); break;
    case 12: shwfs_frame_f64_kernel<12><<<grid, 64, 0, s>>>(opd, pupil, amp, valid, nS, phase_scale, shared_max, frame, em); break;
  }
  AOENV_LAUNCH_CHECK("shwfs_frame_f64");
  dim3 g2((nV + 127) / 128, F);
  shwfs_slopes_f64_kernel<<<g2, 128, 0, s>>>(frame, em, shared_max, valid_idx, nV, ref_xy, inv_units, threshold_cog, nS, n,
                                             slopes, lds);
  AOENV_LAUNCH_CHECK("shwfs_slopes_f64");
  return 0;
}

}  // extern "C"
