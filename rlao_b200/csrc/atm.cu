// Atmosphere kernels: von Karman infinite phase screens (Assemat et al. 2006) as OOPAO/Atmosphere.py runs them,
// batched over environments.  All are HBM-bound streaming kernels; the dense part of add_row (X = A Z + B xi)
// is a GEMM (gemm_tc.cu / gemm.cu).
//
// Sliding window: the reference shifts the whole (R+6)^2 map by one pixel at every add_row.  Here each layer map
// lives in a larger canvas and only the WINDOW ORIGIN moves (by -step); add_row then writes just the 4M-4 ring
// pixels of the new window border.  The canvas is re-centred ("compacted") once every S events.  A "window" is
// addressed as (pointer to its origin, pitch = canvas pitch, env_stride = canvas size).
#include "common.cuh"
#include "tma.cuh"

namespace aoenv {

// ---------------------------------------------------------------------------------------------------------
// add_row step 1: gather the two inner rings of the one-pixel-shifted map + the innovation vector
// (OOPAO/Atmosphere.py:303-308).  One thread per entry of zx[b][:].
// ---------------------------------------------------------------------------------------------------------
// Several layers whose add_row falls in the same round of a step are processed by one launch: gridDim.z = layers in
// the group, per-layer arguments in a __grid_constant__ block (indexed loads from the constant bank).
struct AtmGroup {
  float* win[AOENV_MAX_LAYERS];                  // window origin (gather: the NEW origin; ring: canvas base)
  unsigned long long* ext[AOENV_MAX_LAYERS];
  unsigned long long seed[AOENV_MAX_LAYERS], stream_id[AOENV_MAX_LAYERS];
  uint32_t win_offset[AOENV_MAX_LAYERS];
  int sx[AOENV_MAX_LAYERS], sy[AOENV_MAX_LAYERS];
};

// kEnvs: workspace row b belongs to environment env_idx[b] (the episode reset of a subset, aoenv_atm_gather_envs); the
// environment index is also the Philox counter word, so a row's innovation does not depend on which others are listed.
template <bool kEnvs>
__global__ void __launch_bounds__(256)
atm_gather_kernel(const __grid_constant__ AtmGroup grp, int M, int pitch, size_t env_stride,
                  const int2* __restrict__ inner_rc, int nI, int nO, const float* __restrict__ xi,
                  float* __restrict__ zx, int ldz, __nv_bfloat16* __restrict__ planes, int parts,
                  const int32_t* __restrict__ env_idx) {
  pdl_enter();
  const int b = blockIdx.y, g = blockIdx.z;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= ldz) return;
  const int e = kEnvs ? __ldg(&env_idx[b]) : b;
  const size_t row = (size_t)g * gridDim.y + b;
  float v = 0.f;
  if (k < nI) {
    const int2 rc = __ldg(&inner_rc[k]);
    const float* __restrict__ map = grp.win[g];
    v = __ldg(&map[(size_t)e * env_stride + (size_t)(rc.x - grp.sy[g]) * pitch + (rc.y - grp.sx[g])]);
  } else if (k < nI + nO) {
    const int j = k - nI;
    if (xi != nullptr) {
      v = __ldg(&xi[row * nO + j]);
    } else {
      const unsigned long long stream_id = grp.stream_id[g];
      Philox rng(grp.seed[g]);
      const uint4 r = rng((uint32_t)j, (uint32_t)e, (uint32_t)stream_id, (uint32_t)(stream_id >> 32));
      v = box_muller(r.x, r.y).x;
    }
  }
  if (zx != nullptr) zx[row * ldz + k] = v;        // float32 copy only for the SIMT GEMM back end / inspection
  if (planes != nullptr) store_bf16_planes(planes, (size_t)gridDim.z * gridDim.y * ldz, row * ldz + k, parts, v);
}

// ---------------------------------------------------------------------------------------------------------
// Map extrema (the clip range of skimage.warp, tools/tools.py:215-217) are tracked WITH their position:
// ext[b][0] = packed minimum, ext[b][1] = packed maximum, packed = (monotone 32-bit key of the value) << 32 | pos,
// pos = element index inside the environment's canvas.  The array holds three blocks per layer, [3][B][2]:
// block 0 = extrema of the whole window (what atm_phase clips with), block 1 = extrema of the window INTERIOR (the
// window without its outer ring), block 2 = [b][0]: (1 << 32) | window origin at the previous add_row (0 = none yet).  The ring is redrawn at every add_row, so an extremum sitting on it (where a
// von Karman screen likes to put them) says nothing about the next window; the interior pixels keep their values, and
// an interior extremum survives an add_row unless its pixel leaves the interior on the trailing side.  Per add_row:
// new interior extrema = best(old ones if they survive, the one or two edge lines of the new interior that were ring
// pixels before the step); window extrema = best(interior, new ring).  Only when an interior
// extremum is lost is the environment flagged and atm_rescan_kernel recomputes the interior exactly.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t key_of(float f) { return (uint32_t)float_to_ordered(f) ^ 0x80000000u; }
__device__ __forceinline__ float value_of(unsigned long long packed) {
  return ordered_to_float((int32_t)((uint32_t)(packed >> 32) ^ 0x80000000u));
}
__device__ __forceinline__ unsigned long long pack(float f, uint32_t pos) { return ((unsigned long long)key_of(f) << 32) | pos; }

__device__ __forceinline__ void block_reduce_ext(unsigned long long& lo, unsigned long long& hi) {
  __shared__ unsigned long long s_lo[32], s_hi[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
    lo = l2 < lo ? l2 : lo;
    hi = h2 > hi ? h2 : hi;
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s_lo[w] = lo; s_hi[w] = hi; }
  __syncthreads();
  if (w == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    lo = l < nw ? s_lo[l] : ~0ull;
    hi = l < nw ? s_hi[l] : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
      lo = l2 < lo ? l2 : lo;
      hi = h2 > hi ? h2 : hi;
    }
  }
}

// add_row step 3 (OOPAO/Atmosphere.py:309): one CTA per environment writes the ring of the NEW window (ring index in
// numpy boolean-mask order of `outerMask`, :263-264: row 0, then the (r,0),(r,M-1) pairs, then row M-1), reduces the
// ring extrema and decides whether the tracked extrema survive.
// kEnvs: CTA b writes environment env_idx[b] of nB (the extrema blocks hold nB environments); workspace rows stay b.
template <bool kEnvs>
__global__ void __launch_bounds__(256)
atm_ring_kernel(const __grid_constant__ AtmGroup grp, int M, int pitch, size_t env_stride,
                const float* __restrict__ X, int ldx, int32_t* __restrict__ flag, int force_rescan,
                const int32_t* __restrict__ env_idx, int nB) {
  pdl_enter();
  const int b = blockIdx.x, g = blockIdx.y;
  const int e = kEnvs ? __ldg(&env_idx[b]) : b;
  const size_t nEnv = kEnvs ? (size_t)nB : (size_t)gridDim.x;
  const size_t row = (size_t)g * gridDim.x + b;
  const uint32_t win_offset = grp.win_offset[g];
  unsigned long long* __restrict__ ext = grp.ext[g];
  float* __restrict__ w = grp.win[g] + (size_t)e * env_stride;
  const float* __restrict__ xb = X + row * ldx;
  const int nO = 4 * M - 4;
  // Which lines became interior with this step: the window moved by (dy, dx) = new origin - previous origin (block 2 of
  // the extrema array remembers the previous one); origin - 1 along an axis exposes line 1 of that axis, + 1 line M - 2.
  // Unknown history (first call, forced rescan) -> all four edge lines of the interior.
  unsigned long long* __restrict__ ext_prev = ext + 4 * nEnv + 2 * e;
  const unsigned long long prev = *ext_prev;
  const int oy = win_offset / pitch, ox = win_offset % pitch;
  int line_r[2], line_c[2], nr = 0, nc = 0;                     // rows / columns of the window to merge
  {
    const int py = (int)((uint32_t)prev / (uint32_t)pitch), px = (int)((uint32_t)prev % (uint32_t)pitch);
    const int dy = oy - py, dx = ox - px;
    if ((prev >> 32) != 1ull || force_rescan || dy < -1 || dy > 1 || dx < -1 || dx > 1) {
      line_r[0] = 1; line_r[1] = M - 2; nr = 2;
      line_c[0] = 1; line_c[1] = M - 2; nc = 2;
    } else {
      if (dy != 0) line_r[nr++] = dy < 0 ? 1 : M - 2;
      if (dx != 0) line_c[nc++] = dx < 0 ? 1 : M - 2;
    }
  }
  const int nE = (nr + nc) * (M - 2);
  // their loads go first (the column ones are one 32-byte sector each), the ring is written while they are in flight
  constexpr int kEdge = 8;
  float ev[kEdge];
  uint32_t erel[kEdge];
#pragma unroll
  for (int i = 0; i < kEdge; ++i) {
    const int k = threadIdx.x + i * 256;
    erel[i] = 0;
    ev[i] = 0.f;
    if (k < nE) {
      const int side = k / (M - 2), t = 1 + k % (M - 2);
      const int r = side < nr ? line_r[side] : t, c = side < nr ? t : line_c[side - nr];
      erel[i] = (uint32_t)(r * pitch + c);
      ev[i] = w[erel[i]];
    }
  }
  unsigned long long lo = ~0ull, hi = 0ull;
  for (int k = threadIdx.x; k < nO; k += blockDim.x) {
    int r, c;
    if (k < M) { r = 0; c = k; }
    else if (k >= M + 2 * (M - 2)) { r = M - 1; c = k - (M + 2 * (M - 2)); }
    else { const int t = k - M; r = 1 + (t >> 1); c = (t & 1) ? M - 1 : 0; }
    const float v = __ldg(&xb[k]);
    const uint32_t rel = (uint32_t)(r * pitch + c);
    w[rel] = v;
    const unsigned long long pk = pack(v, win_offset + rel);
    lo = pk < lo ? pk : lo;
    hi = pk > hi ? pk : hi;
  }
  unsigned long long ilo = ~0ull, ihi = 0ull;
#pragma unroll
  for (int i = 0; i < kEdge; ++i) {
    if (threadIdx.x + i * 256 < nE) {
      const unsigned long long pk = pack(ev[i], win_offset + erel[i]);
      ilo = pk < ilo ? pk : ilo;
      ihi = pk > ihi ? pk : ihi;
    }
  }
  for (int k = threadIdx.x + kEdge * 256; k < nE; k += 256) {   // windows wider than 514 pixels with all four lines
    const int side = k / (M - 2), t = 1 + k % (M - 2);
    const int r = side < nr ? line_r[side] : t, c = side < nr ? t : line_c[side - nr];
    const uint32_t rel = (uint32_t)(r * pitch + c);
    const unsigned long long pk = pack(w[rel], win_offset + rel);
    ilo = pk < ilo ? pk : ilo;
    ihi = pk > ihi ? pk : ihi;
  }
  block_reduce_ext(lo, hi);
  __syncthreads();                       // the reduction scratch is reused
  block_reduce_ext(ilo, ihi);
  if (threadIdx.x == 0) {
    unsigned long long* __restrict__ ext_in = ext + 2 * nEnv;                   // block 1: interior extrema
    const unsigned long long old_lo = ext_in[2 * e], old_hi = ext_in[2 * e + 1];
    *ext_prev = (1ull << 32) | win_offset;
    auto retained = [&](unsigned long long pk) {
      const uint32_t pos = (uint32_t)pk;
      const int r = (int)(pos / pitch) - oy, c = (int)(pos % pitch) - ox;
      return r >= 1 && r <= M - 2 && c >= 1 && c <= M - 2;
    };
    const bool ok = !force_rescan && retained(old_lo) && retained(old_hi);
    if (ok) {
      ilo = old_lo < ilo ? old_lo : ilo;
      ihi = old_hi > ihi ? old_hi : ihi;
    }
    ext_in[2 * e] = ilo;                  // not ok: the edge lines only, the rescan merges the rest
    ext_in[2 * e + 1] = ihi;
    ext[2 * e] = ilo < lo ? ilo : lo;
    ext[2 * e + 1] = ihi > hi ? ihi : hi;
    flag[row] = ok ? 0 : 1;
  }
}

// Exact extrema of the window interior for the flagged environments, merged into ext (which already holds the ring's).
// A CTA scans `rows_per_block` interior rows with aligned 128-bit loads, four rows (64 bytes) per thread in flight; the
// running extrema are kept as (value, position) pairs under plain float comparisons and packed once at the end.  Rows
// start on arbitrary columns (the window origin moves pixel by pixel), so the first / last vector of a row is masked.
// Needs pitch and env_stride to be multiples of 4 floats (then every row has the same misalignment).
template <bool kEnvs>
__global__ void __launch_bounds__(256)
atm_rescan_kernel(const __grid_constant__ AtmGroup grp, int M, int pitch, size_t env_stride,
                  const int32_t* __restrict__ flag, int rows_per_block, const int32_t* __restrict__ env_idx, int nB) {
  pdl_enter();
  const int b = blockIdx.y, g = blockIdx.z;
  if (__ldg(&flag[(size_t)g * gridDim.y + b]) == 0) return;
  const int e = kEnvs ? __ldg(&env_idx[b]) : b;
  const size_t nEnv = kEnvs ? (size_t)nB : (size_t)gridDim.y;
  const uint32_t win_offset = grp.win_offset[g];
  unsigned long long* __restrict__ ext = grp.ext[g];
  const float* __restrict__ w = grp.win[g] + (size_t)e * env_stride;
  const int r_begin = 1 + blockIdx.x * rows_per_block;
  const int r_end = min(M - 1, r_begin + rows_per_block);
  const int mis = (int)((reinterpret_cast<uintptr_t>(w) >> 2) & 3);      // window column 0 sits `mis` floats into a 16-byte line
  const int nvec = (M - 1 + mis + 3) >> 2;                                // vectors covering columns -mis .. M-2
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  float vlo = INFINITY, vhi = -INFINITY;
  uint32_t plo = 0, phi = 0;
  constexpr int kRows = 4;
  for (int r0 = r_begin + ty * kRows; r0 < r_end; r0 += 4 * kRows) {
    for (int v4 = tx; v4 < nvec; v4 += 64) {
      const int c0 = 4 * v4 - mis;
      float4 q[kRows];
#pragma unroll
      for (int i = 0; i < kRows; ++i)
        q[i] = (r0 + i < r_end) ? __ldg(reinterpret_cast<const float4*>(w + (size_t)(r0 + i) * pitch + c0)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < kRows; ++i) {
        if (r0 + i >= r_end) break;
        const uint32_t base = (uint32_t)((r0 + i) * pitch + c0);
        const float e[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int c = c0 + k;
          if (c >= 1 && c < M - 1) {
            if (e[k] < vlo) { vlo = e[k]; plo = base + k; }
            if (e[k] > vhi) { vhi = e[k]; phi = base + k; }
          }
        }
      }
    }
  }
  unsigned long long lo = vlo < INFINITY ? pack(vlo, win_offset + plo) : ~0ull;
  unsigned long long hi = vhi > -INFINITY ? pack(vhi, win_offset + phi) : 0ull;
  block_reduce_ext(lo, hi);
  if (threadIdx.x == 0 && r_begin < r_end) {
    unsigned long long* __restrict__ ext_in = ext + 2 * nEnv;                    // block 1: interior extrema
    atomicMin(&ext_in[2 * e], lo);
    atomicMax(&ext_in[2 * e + 1], hi);
    atomicMin(&ext[2 * e], lo);
    atomicMax(&ext[2 * e + 1], hi);
  }
}

// Canvas compaction: copies the window to its new origin in the other canvas buffer (dst origin column is a multiple
// of 4, so the stores are aligned 128-bit) and moves the tracked extremum positions along.
__global__ void __launch_bounds__(256)
atm_compact_kernel(const float* __restrict__ src, float* __restrict__ dst, int M, int pitch, size_t env_stride,
                   unsigned long long* __restrict__ ext, int pos_delta, int rows_per_block) {
  pdl_enter();
  const int b = blockIdx.y;
  const float* __restrict__ s = src + (size_t)b * env_stride;
  float* __restrict__ d = dst + (size_t)b * env_stride;
  const int r_begin = blockIdx.x * rows_per_block;
  const int r_end = min(M, r_begin + rows_per_block);
  const int nvec = (M + 3) >> 2;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  for (int r = r_begin + ty; r < r_end; r += 4) {
    const float* __restrict__ sr = s + (size_t)r * pitch;
    float* __restrict__ dr = d + (size_t)r * pitch;
    for (int v4 = tx; v4 < nvec; v4 += 64) {
      const int c = v4 << 2;
      if (c + 3 < M) {
        *reinterpret_cast<float4*>(dr + c) = make_float4(__ldg(sr + c), __ldg(sr + c + 1), __ldg(sr + c + 2), __ldg(sr + c + 3));
      } else {
        for (int k = 0; c + k < M; ++k) dr[c + k] = __ldg(sr + c + k);
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < 5) {     // the three blocks of the extrema array: window, interior, previous origin
    const size_t i = (size_t)(threadIdx.x >> 1) * 2 * gridDim.y + 2 * b + (threadIdx.x & 1);
    const unsigned long long e = ext[i];
    ext[i] = (e & 0xffffffff00000000ull) | (uint32_t)((int)(uint32_t)e + pos_delta);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Sub-pixel shift + clip + footprint crop + Cn2-weighted layer sum (OOPAO/Atmosphere.py:406-407,439-450,474-478;
// interpolation: scikit-image 0.18.3 bicubic, see oracle/warp018.py).  Each thread produces a 1 x ROWS column
// strip: the horizontal 4-tap pass is done once per input row and reused by the vertical 4-tap pass.
// ---------------------------------------------------------------------------------------------------------
struct AtmPhaseParams {
  CUtensorMap map[AOENV_MAX_LAYERS];                 // canvas [B][Mc][pitch] of each layer (3-D tensor map)
  const unsigned long long* ext[AOENV_MAX_LAYERS];
  int row0[AOENV_MAX_LAYERS];                        // canvas row / column of the first tap of footprint pixel (0, 0)
  int col0[AOENV_MAX_LAYERS];
  float wrow[AOENV_MAX_LAYERS][4];
  float wcol[AOENV_MAX_LAYERS][4];
  float weight[AOENV_MAX_LAYERS];
  int nLayer;
};

// Tile = 128 x 32 output pixels per CTA of 128 threads; each thread owns a 4 (columns) x 8 (rows) register block.
// Per layer one TMA box load (cp.async.bulk.tensor.3d) brings the (32+3) x (128+8) input window to shared memory with
// zero fill outside the canvas; two buffers let the load of layer l+1 overlap the interpolation of layer l.  TMA needs
// the innermost start coordinate 16-byte aligned, so the box starts at the window column rounded down to a multiple
// of 4 and the remainder `mis` (uniform per CTA and layer) is resolved in registers: three 128-bit shared loads per
// input row cover the 7 taps of a thread's 4 outputs for any mis in 0..3.
constexpr int kPhTileW = 128, kPhTileH = 32, kPhThreadsX = 32, kPhThreadsY = 4, kPhRows = 8;
constexpr int kPhBoxW = kPhTileW + 8, kPhBoxH = kPhTileH + 3;
constexpr uint32_t kPhBoxBytes = kPhBoxW * kPhBoxH * sizeof(float);
constexpr int kPhBufFloats = (kPhBoxW * kPhBoxH + 31) / 32 * 32;      // each TMA destination 128-byte aligned

// Tensor maps must be addressed in parameter space: a dynamically indexed `&p.map[l]` would make the compiler copy the
// parameter block to local memory, which TMA cannot read.  Constant indices keep the generic address in param space.
__device__ __forceinline__ const CUtensorMap* layer_map(const AtmPhaseParams& p, int l) {
  switch (l) {
    case 0: return &p.map[0];
    case 1: return &p.map[1];
    case 2: return &p.map[2];
    case 3: return &p.map[3];
    case 4: return &p.map[4];
    case 5: return &p.map[5];
    case 6: return &p.map[6];
    default: return &p.map[7];
  }
}

template <int MIS>
__device__ __forceinline__ void phase_rows(const float* __restrict__ tbase, float wc0, float wc1, float wc2, float wc3,
                                           float (&h)[kPhRows + 3][4]) {
#pragma unroll
  for (int t = 0; t < kPhRows + 3; ++t) {
    const float* __restrict__ trow = tbase + t * kPhBoxW;
    const float4 a = *reinterpret_cast<const float4*>(trow);
    const float4 b = *reinterpret_cast<const float4*>(trow + 4);
    const float4 c = *reinterpret_cast<const float4*>(trow + 8);
    const float v[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      h[t][k] = wc0 * v[MIS + k] + wc1 * v[MIS + k + 1] + wc2 * v[MIS + k + 2] + wc3 * v[MIS + k + 3];
  }
}

// kEnvs: grid layer z computes environment env_idx[z] (same arithmetic as the whole-batch launch, per environment)
template <bool kEnvs>
__global__ void __launch_bounds__(kPhThreadsX * kPhThreadsY)
atm_phase_kernel(const __grid_constant__ AtmPhaseParams p, int R, float opd_scale, float* __restrict__ opd_out,
                 const int32_t* __restrict__ env_idx) {
  pdl_enter();
  __shared__ __align__(128) float tile[2][kPhBufFloats];
  __shared__ __align__(8) uint64_t bar[2];
  const int b = kEnvs ? __ldg(&env_idx[blockIdx.z]) : (int)blockIdx.z;
  const int j0 = blockIdx.x * kPhTileW, i0 = blockIdx.y * kPhTileH;
  const int tx = threadIdx.x, ty = threadIdx.y;
  const bool leader = (tx == 0 && ty == 0);
  if (leader) {
    tma::mbar_init(&bar[0], 1);
    tma::mbar_init(&bar[1], 1);
    tma::mbar_fence_init();
  }
  __syncthreads();
  if (leader) {
    tma::mbar_expect_tx(&bar[0], kPhBoxBytes);
    tma::load_3d(layer_map(p, 0), &bar[0], &tile[0][0], (p.col0[0] + j0) & ~3, p.row0[0] + i0, b);
  }
  float acc[kPhRows][4];
#pragma unroll
  for (int r = 0; r < kPhRows; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;

  for (int l = 0; l < p.nLayer; ++l) {
    const int buf = l & 1;
    if (leader && l + 1 < p.nLayer) {     // buffer buf^1 was released by the __syncthreads that ended iteration l-1
      tma::mbar_expect_tx(&bar[buf ^ 1], kPhBoxBytes);
      tma::load_3d(layer_map(p, l + 1), &bar[buf ^ 1], &tile[buf ^ 1][0], (p.col0[l + 1] + j0) & ~3, p.row0[l + 1] + i0, b);
    }
    const float lo = value_of(__ldg(&p.ext[l][2 * b + 0]));
    const float hi = value_of(__ldg(&p.ext[l][2 * b + 1]));
    const float wc0 = p.wcol[l][0], wc1 = p.wcol[l][1], wc2 = p.wcol[l][2], wc3 = p.wcol[l][3];
    const float wr0 = p.wrow[l][0], wr1 = p.wrow[l][1], wr2 = p.wrow[l][2], wr3 = p.wrow[l][3];
    const float w = p.weight[l];
    tma::mbar_wait(&bar[buf], (l >> 1) & 1);
    float h[kPhRows + 3][4];
    const float* __restrict__ tbase = &tile[buf][(ty * kPhRows) * kPhBoxW + tx * 4];
    switch ((p.col0[l] + j0) & 3) {                                     // uniform across the CTA
      case 0: phase_rows<0>(tbase, wc0, wc1, wc2, wc3, h); break;
      case 1: phase_rows<1>(tbase, wc0, wc1, wc2, wc3, h); break;
      case 2: phase_rows<2>(tbase, wc0, wc1, wc2, wc3, h); break;
      default: phase_rows<3>(tbase, wc0, wc1, wc2, wc3, h); break;
    }
#pragma unroll
    for (int t = 0; t < kPhRows; ++t)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float v = wr0 * h[t][c] + wr1 * h[t + 1][c] + wr2 * h[t + 2][c] + wr3 * h[t + 3][c];
        v = fminf(fmaxf(v, lo), hi);
        acc[t][c] += w * v;
      }
    __syncthreads();                       // everyone is done with tile[buf] before it is refilled
  }
  float* __restrict__ out = opd_out + (size_t)b * R * R;
  const int jc = j0 + tx * 4;
#pragma unroll
  for (int t = 0; t < kPhRows; ++t) {
    const int i = i0 + ty * kPhRows + t;
    if (i >= R || jc >= R) continue;
    float* __restrict__ o = out + (size_t)i * R + jc;
    if (jc + 3 < R && ((R & 3) == 0)) {
      *reinterpret_cast<float4*>(o) = make_float4(acc[t][0] * opd_scale, acc[t][1] * opd_scale, acc[t][2] * opd_scale, acc[t][3] * opd_scale);
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (jc + c < R) o[c] = acc[t][c] * opd_scale;
    }
  }
}

}  // namespace aoenv

using namespace aoenv;

static int rows_per_block_for(int B, int M) {
  // enough blocks to fill 148 SMs a few times over even for a handful of environments
  int chunks = (4 * kNumSMs + B - 1) / B;
  if (chunks < 1) chunks = 1;
  if (chunks > M) chunks = M;
  return (M + chunks - 1) / chunks;
}

namespace {

int gather_launch(const void* const* wins, const int32_t* sx, const int32_t* sy, const uint64_t* seeds, const uint64_t* stream_ids,
                  int G, int B, int M, int pitch, int64_t env_stride, const int32_t* inner_rc, int nI, int nO, const float* xi,
                  float* zx, int ldz, void* zx_planes, int parts, const int32_t* env_idx, void* stream) {
  AOENV_CHECK_ARG(G > 0 && G <= AOENV_MAX_LAYERS, "atm_gather: %d layers in one group (max %d)", G, AOENV_MAX_LAYERS);
  AOENV_CHECK_ARG(B > 0 && B <= 65535 && M > 6 && pitch >= M && env_stride >= (int64_t)M * pitch, "atm_gather: bad shape B=%d M=%d pitch=%d", B, M, pitch);
  AOENV_CHECK_ARG(ldz >= nI + nO, "atm_gather: ldz=%d < nI+nO=%d", ldz, nI + nO);
  AOENV_CHECK_ARG(zx_planes == nullptr || parts == 2 || parts == 3, "atm_gather: parts must be 2 or 3");
  AOENV_CHECK_ARG(zx != nullptr || zx_planes != nullptr, "atm_gather: neither zx nor zx_planes given");
  AtmGroup grp{};
  for (int g = 0; g < G; ++g) {
    AOENV_CHECK_ARG(sx[g] >= -1 && sx[g] <= 1 && sy[g] >= -1 && sy[g] <= 1, "atm_gather: shift must be in {-1,0,1}");
    grp.win[g] = (float*)wins[g];
    grp.sx[g] = sx[g];
    grp.sy[g] = sy[g];
    grp.seed[g] = seeds ? seeds[g] : 0;
    grp.stream_id[g] = stream_ids ? stream_ids[g] : 0;
  }
  dim3 grid((ldz + 255) / 256, B, G);
  if (env_idx)
    AOENV_LAUNCH(atm_gather_kernel<true>, grid, 256, 0, (cudaStream_t)stream, grp, M, pitch, (size_t)env_stride,
                 (const int2*)inner_rc, nI, nO, xi, zx, ldz, (__nv_bfloat16*)zx_planes, parts, env_idx);
  else
    AOENV_LAUNCH(atm_gather_kernel<false>, grid, 256, 0, (cudaStream_t)stream, grp, M, pitch, (size_t)env_stride,
                 (const int2*)inner_rc, nI, nO, xi, zx, ldz, (__nv_bfloat16*)zx_planes, parts, env_idx);
  AOENV_LAUNCH_CHECK("atm_gather");
  return 0;
}

// rows = workspace rows per layer (B, or k listed environments); nB = environments in the extrema blocks
int ring_launch(void* const* wins, const int64_t* win_offsets, void* const* exts, int G, int rows, int nB, int M, int pitch,
                int64_t env_stride, int nO, const float* X, int ldx, int32_t* flag, int force_rescan, const int32_t* env_idx,
                void* stream) {
  AOENV_CHECK_ARG(G > 0 && G <= AOENV_MAX_LAYERS, "atm_ring: %d layers in one group (max %d)", G, AOENV_MAX_LAYERS);
  AOENV_CHECK_ARG(rows > 0 && rows <= 65535 && nB >= rows && M > 6 && pitch >= M && pitch % 4 == 0 && env_stride % 4 == 0,
                  "atm_ring: bad shape (pitch and env_stride must be multiples of 4 floats)");
  AOENV_CHECK_ARG(nO == 4 * M - 4 && ldx >= nO, "atm_ring: ring has %d pixels, got nO=%d ldx=%d", 4 * M - 4, nO, ldx);
  AtmGroup grp{};
  for (int g = 0; g < G; ++g) {
    AOENV_CHECK_ARG(win_offsets[g] >= 0 && win_offsets[g] + (int64_t)M * pitch <= env_stride + pitch && env_stride < (1ll << 32),
                    "atm_ring: window leaves the canvas");
    grp.win[g] = (float*)wins[g];
    grp.ext[g] = (unsigned long long*)exts[g];
    grp.win_offset[g] = (uint32_t)win_offsets[g];
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (env_idx)
    AOENV_LAUNCH(atm_ring_kernel<true>, dim3(rows, G), 256, 0, s, grp, M, pitch, (size_t)env_stride, X, ldx, flag, force_rescan,
                 env_idx, nB);
  else
    AOENV_LAUNCH(atm_ring_kernel<false>, dim3(rows, G), 256, 0, s, grp, M, pitch, (size_t)env_stride, X, ldx, flag, force_rescan,
                 env_idx, nB);
  AOENV_LAUNCH_CHECK("atm_ring");
  const int rpb = 32;                          // >= 8 CTAs per flagged environment; unflagged ones exit at once (8 rows per CTA measured slower: 169 vs 138 us)
  dim3 grid((M - 2 + rpb - 1) / rpb, rows, G);
  if (env_idx)
    AOENV_LAUNCH(atm_rescan_kernel<true>, grid, 256, 0, s, grp, M, pitch, (size_t)env_stride, flag, rpb, env_idx, nB);
  else
    AOENV_LAUNCH(atm_rescan_kernel<false>, grid, 256, 0, s, grp, M, pitch, (size_t)env_stride, flag, rpb, env_idx, nB);
  AOENV_LAUNCH_CHECK("atm_rescan");
  return 0;
}

}  // namespace

extern "C" {

int aoenv_atm_gather_multi(const void* const* wins, const int32_t* sx, const int32_t* sy, const uint64_t* seeds,
                           const uint64_t* stream_ids, int G, int B, int M, int pitch, int64_t env_stride,
                           const int32_t* inner_rc, int nI, int nO, const float* xi, float* zx, int ldz, void* zx_planes,
                           int parts, void* stream) {
  return gather_launch(wins, sx, sy, seeds, stream_ids, G, B, M, pitch, env_stride, inner_rc, nI, nO, xi, zx, ldz, zx_planes,
                       parts, nullptr, stream);
}

int aoenv_atm_gather_envs(const void* const* wins, const uint64_t* seeds, const uint64_t* stream_ids, int G,
                          const int32_t* env_idx, int k, int M, int pitch, int64_t env_stride, const int32_t* inner_rc, int nI,
                          int nO, float* zx, int ldz, void* zx_planes, int parts, void* stream) {
  AOENV_CHECK_ARG(env_idx != nullptr, "atm_gather_envs: no environment list");
  const int32_t zero[AOENV_MAX_LAYERS] = {};
  return gather_launch(wins, zero, zero, seeds, stream_ids, G, k, M, pitch, env_stride, inner_rc, nI, nO, nullptr, zx, ldz,
                       zx_planes, parts, env_idx, stream);
}

int aoenv_atm_gather(const float* win, int B, int M, int pitch, int64_t env_stride, int sx, int sy,
                     const int32_t* inner_rc, int nI, int nO, const float* xi, uint64_t seed, uint64_t stream_id,
                     float* zx, int ldz, void* zx_planes, int parts, void* stream) {
  const void* wins[1] = {win};
  const int32_t sxs[1] = {sx}, sys[1] = {sy};
  const uint64_t seeds[1] = {seed}, ids[1] = {stream_id};
  return aoenv_atm_gather_multi(wins, sxs, sys, seeds, ids, 1, B, M, pitch, env_stride, inner_rc, nI, nO, xi, zx, ldz,
                                zx_planes, parts, stream);
}

int aoenv_atm_ring_multi(void* const* wins, const int64_t* win_offsets, void* const* exts, int G, int B, int M, int pitch,
                         int64_t env_stride, int nO, const float* X, int ldx, int32_t* flag, int force_rescan, void* stream) {
  return ring_launch(wins, win_offsets, exts, G, B, B, M, pitch, env_stride, nO, X, ldx, flag, force_rescan, nullptr, stream);
}

int aoenv_atm_ring_envs(void* const* wins, const int64_t* win_offsets, void* const* exts, int G, const int32_t* env_idx, int k,
                        int B, int M, int pitch, int64_t env_stride, int nO, const float* X, int ldx, int32_t* flag,
                        void* stream) {
  AOENV_CHECK_ARG(env_idx != nullptr, "atm_ring_envs: no environment list");
  return ring_launch(wins, win_offsets, exts, G, k, B, M, pitch, env_stride, nO, X, ldx, flag, 1, env_idx, stream);
}

int aoenv_atm_ring(float* win, int B, int M, int pitch, int64_t env_stride, int64_t win_offset, int nO, const float* X,
                   int ldx, uint64_t* ext, int32_t* flag, int force_rescan, void* stream) {
  void* wins[1] = {win};
  void* exts[1] = {ext};
  const int64_t offs[1] = {win_offset};
  return aoenv_atm_ring_multi(wins, offs, exts, 1, B, M, pitch, env_stride, nO, X, ldx, flag, force_rescan, stream);
}

int aoenv_atm_compact(const float* src_win, float* dst_win, int B, int M, int pitch, int64_t env_stride, uint64_t* ext,
                      int64_t pos_delta, void* stream) {
  AOENV_CHECK_ARG(B > 0 && B <= 65535 && M > 6 && pitch >= M && pitch % 4 == 0, "atm_compact: bad shape");
  AOENV_CHECK_ARG((reinterpret_cast<uintptr_t>(dst_win) & 15) == 0, "atm_compact: destination window must be 16-byte aligned");
  const int rpb = rows_per_block_for(B, M);
  dim3 grid((M + rpb - 1) / rpb, B);
  AOENV_LAUNCH(atm_compact_kernel, grid, 256, 0, (cudaStream_t)stream, src_win, dst_win, M, pitch, (size_t)env_stride,
                                                             reinterpret_cast<unsigned long long*>(ext), (int)pos_delta, rpb);
  AOENV_LAUNCH_CHECK("atm_compact");
  return 0;
}

}  // extern "C"

namespace {

// grid layers: B environments, or the k of env_idx (the tensor maps always describe the whole batch of B canvases)
int phase_launch(const float* const* h_canvas, const uint64_t* const* h_ext, const int32_t* h_org, int nLayer, int B, int R,
                 int M, int Mc, int pitch, int fp_off, const int32_t* h_row_off, const int32_t* h_col_off, const float* h_wrow,
                 const float* h_wcol, const float* h_weight, float opd_scale, const int32_t* env_idx, int k, float* opd_out,
                 void* stream) {
  AOENV_CHECK_ARG(k > 0 && k <= B, "atm_phase: %d environments listed of %d", k, B);
  AOENV_CHECK_ARG(nLayer >= 1 && nLayer <= AOENV_MAX_LAYERS, "atm_phase: nLayer=%d out of range", nLayer);
  AOENV_CHECK_ARG(B > 0 && B <= 65535, "atm_phase: B=%d out of range (1..65535)", B);
  AOENV_CHECK_ARG(pitch % 4 == 0 && pitch >= Mc && Mc >= M, "atm_phase: bad canvas Mc=%d pitch=%d", Mc, pitch);
  tma::EncodeTiledFn enc = tma::get_encode();
  if (!enc) return fail(-4, "cuTensorMapEncodeTiled is not available from the CUDA driver");
  AtmPhaseParams p;
  p.nLayer = nLayer;
  for (int l = 0; l < nLayer; ++l) {
    const int oy = h_org[2 * l], ox = h_org[2 * l + 1];
    AOENV_CHECK_ARG(oy >= 0 && ox >= 0 && oy + M <= Mc && ox + M <= pitch, "atm_phase: window of layer %d leaves the canvas", l);
    // every tap of every footprint pixel must lie inside the window
    const int lo_r = fp_off + h_row_off[l], hi_r = fp_off + R - 1 + h_row_off[l] + 3;
    const int lo_c = fp_off + h_col_off[l], hi_c = fp_off + R - 1 + h_col_off[l] + 3;
    AOENV_CHECK_ARG(lo_r >= 0 && lo_c >= 0 && hi_r < M && hi_c < M, "atm_phase: taps of layer %d leave the map", l);
    AOENV_CHECK_ARG((reinterpret_cast<uintptr_t>(h_canvas[l]) & 15) == 0, "atm_phase: canvas must be 16-byte aligned");
    static thread_local tma::MapCache<2 * AOENV_MAX_LAYERS> cache;       // two canvas buffers per layer
    const tma::MapKey key{h_canvas[l], ((unsigned long long)(unsigned)pitch << 32) | (unsigned)Mc, (unsigned long long)(unsigned)B};
    const int mrc = cache.get(key, &p.map[l], [&](CUtensorMap* out) {
      cuuint64_t dims[3] = {(cuuint64_t)pitch, (cuuint64_t)Mc, (cuuint64_t)B};
      cuuint64_t strides[2] = {(cuuint64_t)pitch * 4, (cuuint64_t)Mc * pitch * 4};
      cuuint32_t box[3] = {(cuuint32_t)kPhBoxW, (cuuint32_t)kPhBoxH, 1};
      cuuint32_t estr[3] = {1, 1, 1};
      CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(h_canvas[l]), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(-4, "atm_phase: cuTensorMapEncodeTiled failed (%d)", (int)r);
      return 0;
    });
    if (mrc) return mrc;
    p.ext[l] = reinterpret_cast<const unsigned long long*>(h_ext[l]);
    p.row0[l] = oy + fp_off + h_row_off[l];
    p.col0[l] = ox + fp_off + h_col_off[l];
    for (int k = 0; k < 4; ++k) {
      p.wrow[l][k] = h_wrow[4 * l + k];
      p.wcol[l][k] = h_wcol[4 * l + k];
    }
    p.weight[l] = h_weight[l];
  }
  dim3 block(kPhThreadsX, kPhThreadsY);
  dim3 grid((R + kPhTileW - 1) / kPhTileW, (R + kPhTileH - 1) / kPhTileH, k);
  if (env_idx)
    AOENV_LAUNCH(atm_phase_kernel<true>, grid, block, 0, (cudaStream_t)stream, p, R, opd_scale, opd_out, env_idx);
  else
    AOENV_LAUNCH(atm_phase_kernel<false>, grid, block, 0, (cudaStream_t)stream, p, R, opd_scale, opd_out, env_idx);
  AOENV_LAUNCH_CHECK("atm_phase");
  return 0;
}

}  // namespace

extern "C" {

int aoenv_atm_phase(const float* const* h_canvas, const uint64_t* const* h_ext, const int32_t* h_org, int nLayer, int B,
                    int R, int M, int Mc, int pitch, int fp_off, const int32_t* h_row_off, const int32_t* h_col_off,
                    const float* h_wrow, const float* h_wcol, const float* h_weight, float opd_scale, float* opd_out,
                    void* stream) {
  return phase_launch(h_canvas, h_ext, h_org, nLayer, B, R, M, Mc, pitch, fp_off, h_row_off, h_col_off, h_wrow, h_wcol, h_weight,
                      opd_scale, nullptr, B, opd_out, stream);
}

int aoenv_atm_phase_envs(const float* const* h_canvas, const uint64_t* const* h_ext, const int32_t* h_org, int nLayer, int B,
                         int R, int M, int Mc, int pitch, int fp_off, const int32_t* h_row_off, const int32_t* h_col_off,
                         const float* h_wrow, const float* h_wcol, const float* h_weight, float opd_scale, const int32_t* env_idx,
                         int k, float* opd_out, void* stream) {
  AOENV_CHECK_ARG(env_idx != nullptr, "atm_phase_envs: no environment list");
  return phase_launch(h_canvas, h_ext, h_org, nLayer, B, R, M, Mc, pitch, fp_off, h_row_off, h_col_off, h_wrow, h_wcol, h_weight,
                      opd_scale, env_idx, k, opd_out, stream);
}

}  // extern "C"
