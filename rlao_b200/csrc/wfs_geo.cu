// Geometric Shack-Hartmann sensor: the geometric-optics limit of the diffractive sensor of wfs.cu (DESIGN.md §2).  Per
// lenslet, the flux-weighted mean of the phase gradient (np.gradient: central differences inside the array, one-sided
// first differences on its outer rows and columns) over its n x n pixels of the pupil-less OPD.  No spots, no camera,
// no threshold: one streaming pass over the OPD per environment.
#include "common.cuh"

namespace aoenv {
namespace {

constexpr int kGeoThreads = 256;                 // threads per CTA; a CTA owns a strip of lenslet rows of one environment
constexpr int kGeoSmemLimit = 227 * 1024;

template <int V>
__device__ __forceinline__ void load_vec(const float* __restrict__ p, float (&v)[V]) {
  if constexpr (V == 4) {
    const float4 q = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  } else {
    const float2 q = __ldg(reinterpret_cast<const float2*>(p));
    v[0] = q.x; v[1] = q.y;
  }
}

template <int V>
__device__ __forceinline__ void store_vec(float* p, const float (&v)[V]) {
  if constexpr (V == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  else *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
}

// Staged rows: the strip's n * rows pixel rows plus one halo row above and below (the central differences along y read
// them), as two planes: opd_a (for the pupil statistics) and the total OPD opd_a + second term (for the gradients).  With
// the separable DM (WL > 0) the second term is evaluated while staging, from T = C gx and the row weights, with the same
// operations in the same order as shwfs_frame_kernel: the surface is bit-identical to the one the frame kernel sees.
// Then one thread per lenslet sums its n x n pixels in row-major order — weighted gradients, weights, and the four pupil
// statistics in float32 exactly as the frame kernel does per lenslet — so slopes need no atomics and the statistics equal
// the frame kernel's up to the order of the float64 reduction (at 4 to 8 pixels; the wide frame kernel of 10 and 12 pixels
// splits a lenslet over n / 2 lanes and adds its float32 partial sums in another order: agreement to float32 rounding).
template <int n, int V, int WL>
__global__ void __launch_bounds__(kGeoThreads)
shwfs_geometric_kernel(const float* __restrict__ opd_a, const float* __restrict__ opd_b, const __grid_constant__ aoenv_dm_sep_t dm,
                       const float* __restrict__ pupil, const float* __restrict__ flux, const int32_t* __restrict__ valid_idx,
                       int nV, int nS, int SL, float scale, float* __restrict__ slopes, int lds,
                       __nv_bfloat16* __restrict__ planes, int parts, double* __restrict__ stats) {
  extern __shared__ float4 geo_smem[];
  pdl_enter();
  const int R = nS * n, b = blockIdx.y;
  const int l0 = blockIdx.x * SL, nl = min(SL, nS - l0);        // lenslet rows [l0, l0 + nl)
  const int y0 = l0 * n - 1;                                      // image row of staged row 0 (the upper halo)
  const int P = SL * n + 2;
  const bool second = WL > 0 || opd_b != nullptr;
  float* sA = reinterpret_cast<float*>(geo_smem);
  float* sT = second ? sA + (size_t)P * R : sA;
  const size_t env = (size_t)b * R * R;
  const int rlo = y0 < 0 ? 1 : 0, rhi = min(nl * n + 2, R - y0);
  const int vpr = R / V;

  if constexpr (WL == 0) {
#pragma unroll 4
    for (int idx = rlo * vpr + threadIdx.x; idx < rhi * vpr; idx += blockDim.x) {
      const int r = idx / vpr, c = (idx - r * vpr) * V, y = y0 + r;
      const size_t o = env + (size_t)y * R + c;
      float a[V];
      load_vec<V>(opd_a + o, a);
      store_vec<V>(sA + (size_t)r * R + c, a);
      if (second) {
        float d[V];
        load_vec<V>(opd_b + o, d);
#pragma unroll
        for (int e = 0; e < V; ++e) d[e] = a[e] + d[e];
        store_vec<V>(sT + (size_t)r * R + c, d);
      }
    }
  } else {
    // One item = V columns of the n pixel rows of one lenslet row (or of one halo row): the rows share their window of T
    // rows, so each T value is loaded once for all of them.
    constexpr int half = (WL + 1) / 2, hp = (half + 3) / 4 * 4;
    for (int it = threadIdx.x; it < (nl + 2) * vpr; it += blockDim.x) {
      const int g = it / vpr, c = (it - g * vpr) * V;
      const int r0 = g == 0 ? 0 : 1 + (g - 1) * n;
      const int nr = (g == 0 || g == nl + 1) ? 1 : n;
      if (r0 < rlo || r0 >= rhi) continue;                        // halo row outside the image
      const int yb = y0 + r0;
      const float* __restrict__ trow = dm.rows + ((size_t)b * dm.nActP + __ldg(&dm.ilr[yb / n])) * R + c;
      const float* __restrict__ wrow = dm.wlr + (size_t)yb * (2 * hp);
      float2 acc[n][V / 2];
#pragma unroll
      for (int bb = 0; bb < n; ++bb)
#pragma unroll
        for (int h = 0; h < V / 2; ++h) acc[bb][h] = make_float2(0.f, 0.f);
#pragma unroll
      for (int t = 0; t < WL; ++t) {
        float tv[V];
        load_vec<V>(trow + (size_t)t * R, tv);
#pragma unroll
        for (int bb = 0; bb < n; ++bb) {
          if (bb < nr) {
            const float w = __ldg(wrow + (size_t)bb * (2 * hp) + (t / half) * hp + t % half);
#pragma unroll
            for (int h = 0; h < V / 2; ++h) acc[bb][h] = fma2(dup2(w), make_float2(tv[2 * h], tv[2 * h + 1]), acc[bb][h]);
          }
        }
      }
#pragma unroll
      for (int bb = 0; bb < n; ++bb) {
        if (bb < nr) {
          const int r = r0 + bb;
          float a[V], d[V];
          load_vec<V>(opd_a + env + (size_t)(yb + bb) * R + c, a);
          store_vec<V>(sA + (size_t)r * R + c, a);
#pragma unroll
          for (int h = 0; h < V / 2; ++h) { d[2 * h] = a[2 * h] + acc[bb][h].x; d[2 * h + 1] = a[2 * h + 1] + acc[bb][h].y; }
          store_vec<V>(sT + (size_t)r * R + c, d);
        }
      }
    }
  }
  __syncthreads();

  const size_t centre = env + (size_t)(R / 2) * R + R / 2;
  const float ka = stats ? __ldg(opd_a + centre) : 0.f;
  // (as in the frame kernel: with the in-place DM the total is centred on the atmosphere's centre value)
  const float kt = stats ? ((WL == 0 && opd_b != nullptr) ? ka + __ldg(opd_b + centre) : ka) : 0.f;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int base = 0; base < nl * nS; base += blockDim.x) {
    const int k = base + threadIdx.x;
    if (k >= nl * nS) break;
    const int lr = k / nS, lj = k - lr * nS;
    float f0 = 0.f, f1 = 0.f, f2 = 0.f, f3 = 0.f, sw = 0.f, swx = 0.f, swy = 0.f;
#pragma unroll
    for (int bb = 0; bb < n; ++bb) {
      const int r = 1 + lr * n + bb, y = y0 + r;
      const float* tr = sT + (size_t)r * R;
      const float* ar = sA + (size_t)r * R;
      const float* up = y == 0 ? tr : tr - R;
      const float* dn = y == R - 1 ? tr : tr + R;
      const float gys = (y == 0 || y == R - 1) ? 1.f : 0.5f;
#pragma unroll
      for (int aa = 0; aa < n; ++aa) {
        const int x = lj * n + aa;
        const int xl = x == 0 ? 0 : x - 1, xr = x == R - 1 ? x : x + 1;
        const float gxs = (x == 0 || x == R - 1) ? 1.f : 0.5f;
        const float t = tr[x], a = ar[x];
        const float gx = gxs * (tr[xr] - tr[xl]);
        const float gy = gys * (dn[x] - up[x]);
        const float pu = __ldg(pupil + (size_t)y * R + x), w = __ldg(flux + (size_t)y * R + x);
        const float in_pupil = pu > 0.f ? 1.f : 0.f;
        const float da = (a - ka) * in_pupil, dt = (t - kt) * in_pupil;
        f0 += da; f1 = fmaf(da, da, f1); f2 += dt; f3 = fmaf(dt, dt, f3);
        sw += w; swx = fmaf(w, gx, swx); swy = fmaf(w, gy, swy);
      }
    }
    s0 += (double)f0; s1 += (double)f1; s2 += (double)f2; s3 += (double)f3;
    // slope index = position of the lenslet in valid_idx (ascending lenslet numbers): lower bound
    const int kid = (l0 + lr) * nS + lj;
    int lo = 0, hi = nV;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(&valid_idx[mid]) < kid) lo = mid + 1;
      else hi = mid;
    }
    if (lo < nV && __ldg(&valid_idx[lo]) == kid) {
      const float sx = swx / sw * scale, sy = swy / sw * scale;
      slopes[(size_t)b * lds + lo] = sx;
      slopes[(size_t)b * lds + nV + lo] = sy;
      if (planes != nullptr) {      // operand planes of the reconstruction GEMM, as aoenv_shwfs_slopes writes them
        store_bf16_planes(planes, (size_t)gridDim.y * lds, (size_t)b * lds + lo, parts, sx);
        store_bf16_planes(planes, (size_t)gridDim.y * lds, (size_t)b * lds + nV + lo, parts, sy);
      }
    }
  }
  if (stats != nullptr) {           // one atomic per warp and statistic, as the frame kernel
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2); s3 = warp_sum(s3);
    if ((threadIdx.x & 31) == 0) {
      double* __restrict__ st = stats + (size_t)b * 4;
      atomicAdd(st, s0); atomicAdd(st + 1, s1); atomicAdd(st + 2, s2); atomicAdd(st + 3, s3);
    }
  }
}

__global__ void geo_stats_init_kernel(double* __restrict__ stats, int count) {
  pdl_enter();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) stats[i] = 0.0;
}

// Calibration-grade twin (init only: slope units, interaction-matrix pushes): float64 arithmetic on the float32 OPD, one
// thread per (valid lenslet, frame), no statistics.
template <int n>
__global__ void __launch_bounds__(128)
shwfs_geometric_f64_kernel(const float* __restrict__ opd, const float* __restrict__ flux, const int32_t* __restrict__ valid_idx,
                           int nV, int nS, double scale, double* __restrict__ slopes, int lds) {
  const int f = blockIdx.y, t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nV) return;
  const int R = nS * n;
  const int k = __ldg(&valid_idx[t]), li = k / nS, lj = k - li * nS;
  const float* __restrict__ o = opd + (size_t)f * R * R;
  double sw = 0.0, swx = 0.0, swy = 0.0;
  for (int bb = 0; bb < n; ++bb) {
    const int y = li * n + bb;
    const int yu = y == 0 ? 0 : y - 1, yd = y == R - 1 ? y : y + 1;
    const double gys = (y == 0 || y == R - 1) ? 1.0 : 0.5;
    for (int aa = 0; aa < n; ++aa) {
      const int x = lj * n + aa;
      const int xl = x == 0 ? 0 : x - 1, xr = x == R - 1 ? x : x + 1;
      const double gxs = (x == 0 || x == R - 1) ? 1.0 : 0.5;
      const double gx = gxs * ((double)__ldg(o + (size_t)y * R + xr) - (double)__ldg(o + (size_t)y * R + xl));
      const double gy = gys * ((double)__ldg(o + (size_t)yd * R + x) - (double)__ldg(o + (size_t)yu * R + x));
      const double w = (double)__ldg(flux + (size_t)y * R + x);
      sw += w;
      swx += w * gx;
      swy += w * gy;
    }
  }
  slopes[(size_t)f * lds + t] = swx / sw * scale;
  slopes[(size_t)f * lds + nV + t] = swy / sw * scale;
}

inline size_t geo_smem_bytes(int SL, int n, int R, bool second) {
  return (size_t)(second ? 2 : 1) * (size_t)(SL * n + 2) * R * sizeof(float);
}

template <int n, int V, int WL>
int launch_geometric(dim3 grid, size_t smem, cudaStream_t s, const float* opd_a, const float* opd_b, const aoenv_dm_sep_t& dm,
                     const float* pupil, const float* flux, const int32_t* valid_idx, int nV, int nS, int SL, float scale,
                     float* slopes, int lds, __nv_bfloat16* planes, int parts, double* stats) {
  // once per instantiation and device: allow the strips the host sizes up to 227 KB
  static std::atomic<uint64_t> attr_set{0};
  int dev = 0;
  cudaGetDevice(&dev);
  const uint64_t bit = 1ull << (dev & 63);
  if (!(attr_set.load(std::memory_order_relaxed) & bit)) {
    cudaError_t e = cudaFuncSetAttribute(shwfs_geometric_kernel<n, V, WL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         kGeoSmemLimit);
    if (e != cudaSuccess) return fail(-3, "shwfs_geometric: %s", cudaGetErrorString(e));
    attr_set.fetch_or(bit, std::memory_order_relaxed);
  }
  AOENV_LAUNCH((shwfs_geometric_kernel<n, V, WL>), grid, kGeoThreads, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS,
               SL, scale, slopes, lds, planes, parts, stats);
  return 0;
}

template <int n, int V>
int dispatch_wl(int WL, dim3 grid, size_t smem, cudaStream_t s, const float* opd_a, const float* opd_b, const aoenv_dm_sep_t& dm,
                const float* pupil, const float* flux, const int32_t* valid_idx, int nV, int nS, int SL, float scale,
                float* slopes, int lds, __nv_bfloat16* planes, int parts, double* stats) {
  if (WL == 14)
    return launch_geometric<n, V, 14>(grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds,
                                      planes, parts, stats);
  if (WL == 18)
    return launch_geometric<n, V, 18>(grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds,
                                      planes, parts, stats);
  return launch_geometric<n, V, 0>(grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes,
                                   parts, stats);
}

template <int n>
int dispatch_v(int V, int WL, dim3 grid, size_t smem, cudaStream_t s, const float* opd_a, const float* opd_b,
               const aoenv_dm_sep_t& dm, const float* pupil, const float* flux, const int32_t* valid_idx, int nV, int nS, int SL,
               float scale, float* slopes, int lds, __nv_bfloat16* planes, int parts, double* stats) {
  if (V == 4)
    return dispatch_wl<n, 4>(WL, grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes,
                             parts, stats);
  return dispatch_wl<n, 2>(WL, grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes,
                           parts, stats);
}

}  // namespace
}  // namespace aoenv

using namespace aoenv;

extern "C" {

int aoenv_shwfs_geometric(const float* opd_a, const float* opd_b, const aoenv_dm_sep_t* dm_in, const float* pupil,
                          const float* flux, const int32_t* valid_idx, int nV, int B, int nS, int n, float phase_scale,
                          float inv_units, float* slopes, int lds, void* slope_planes, int parts, double* stats, void* stream) {
  AOENV_CHECK_ARG(B > 0 && B <= 65535 && nS > 0 && nV > 0 && lds >= 2 * nV, "shwfs_geometric: bad shape B=%d nS=%d nV=%d lds=%d",
                  B, nS, nV, lds);
  AOENV_CHECK_ARG(n == 4 || n == 6 || n == 8 || n == 10 || n == 12,
                  "shwfs_geometric: %d pixels per lenslet is not a compiled size (4, 6, 8, 10, 12)", n);
  AOENV_CHECK_ARG(opd_a != nullptr && pupil != nullptr && flux != nullptr && valid_idx != nullptr && slopes != nullptr,
                  "shwfs_geometric: null argument");
  AOENV_CHECK_ARG(slope_planes == nullptr || parts == 2 || parts == 3, "shwfs_geometric: parts=%d", parts);
  const int R = nS * n;
  const int V = R % 4 == 0 ? 4 : 2;
  aoenv_dm_sep_t dm{};
  if (dm_in != nullptr) {
    dm = *dm_in;
    AOENV_CHECK_ARG(opd_b == nullptr, "shwfs_geometric: give either the separable DM or an explicit second OPD term");
    AOENV_CHECK_ARG(dm.rows != nullptr && dm.wlr != nullptr && dm.ilr != nullptr && dm.nActP > 0, "shwfs_geometric: bad DM tables");
    AOENV_CHECK_ARG(dm.WL == 14 || dm.WL == 18, "shwfs_geometric: DM window of %d actuator rows (14 or 18)", dm.WL);
    AOENV_CHECK_ARG((reinterpret_cast<uintptr_t>(dm.rows) & (4 * V - 1)) == 0 && (reinterpret_cast<uintptr_t>(dm.wlr) & 15) == 0,
                    "shwfs_geometric: DM tables must be %d-byte aligned", 4 * V);
  }
  AOENV_CHECK_ARG((reinterpret_cast<uintptr_t>(opd_a) & (4 * V - 1)) == 0 &&
                      (opd_b == nullptr || (reinterpret_cast<uintptr_t>(opd_b) & (4 * V - 1)) == 0),
                  "shwfs_geometric: OPD terms must be %d-byte aligned", 4 * V);
  const bool second = dm.WL != 0 || opd_b != nullptr;
  int SL = nS < kGeoThreads ? kGeoThreads / nS : 1;         // lenslet rows per CTA: about one lenslet per thread
  if (SL > nS) SL = nS;
  while (SL > 1 && geo_smem_bytes(SL, n, R, second) > (size_t)kGeoSmemLimit) --SL;
  const size_t smem = geo_smem_bytes(SL, n, R, second);
  AOENV_CHECK_ARG(smem <= (size_t)kGeoSmemLimit, "shwfs_geometric: %d pixel rows do not fit in shared memory", R);
  cudaStream_t s = (cudaStream_t)stream;
  if (stats != nullptr) {
    AOENV_LAUNCH(geo_stats_init_kernel, dim3((4 * B + 255) / 256), 256, 0, s, stats, 4 * B);
    AOENV_LAUNCH_CHECK("shwfs_geometric_stats_init");
  }
  dim3 grid((nS + SL - 1) / SL, B);
  const float scale = (float)((double)phase_scale * (double)inv_units);
  __nv_bfloat16* planes = (__nv_bfloat16*)slope_planes;
  int rc = 0;
  switch (n) {
    case 4: rc = dispatch_v<4>(V, dm.WL, grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes, parts, stats); break;
    case 6: rc = dispatch_v<6>(V, dm.WL, grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes, parts, stats); break;
    case 8: rc = dispatch_v<8>(V, dm.WL, grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes, parts, stats); break;
    case 10: rc = dispatch_v<10>(V, dm.WL, grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes, parts, stats); break;
    default: rc = dispatch_v<12>(V, dm.WL, grid, smem, s, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, nS, SL, scale, slopes, lds, planes, parts, stats); break;
  }
  if (rc) return rc;
  AOENV_LAUNCH_CHECK("shwfs_geometric");
  return 0;
}

int aoenv_shwfs_geometric_f64(const float* opd, const float* flux, const int32_t* valid_idx, int nV, int F, int nS, int n,
                              double phase_scale, double inv_units, double* slopes, int lds, void* stream) {
  AOENV_CHECK_ARG(F > 0 && F <= 65535 && nS > 0 && nV > 0 && lds >= 2 * nV, "shwfs_geometric_f64: bad shape");
  AOENV_CHECK_ARG(n == 4 || n == 6 || n == 8 || n == 10 || n == 12,
                  "shwfs_geometric_f64: %d pixels per lenslet is not a compiled size (4, 6, 8, 10, 12)", n);
  AOENV_CHECK_ARG(opd != nullptr && flux != nullptr && valid_idx != nullptr && slopes != nullptr, "shwfs_geometric_f64: null argument");
  cudaStream_t s = (cudaStream_t)stream;
  dim3 grid((nV + 127) / 128, F);
  const double scale = phase_scale * inv_units;
  switch (n) {
    case 4: shwfs_geometric_f64_kernel<4><<<grid, 128, 0, s>>>(opd, flux, valid_idx, nV, nS, scale, slopes, lds); break;
    case 6: shwfs_geometric_f64_kernel<6><<<grid, 128, 0, s>>>(opd, flux, valid_idx, nV, nS, scale, slopes, lds); break;
    case 8: shwfs_geometric_f64_kernel<8><<<grid, 128, 0, s>>>(opd, flux, valid_idx, nV, nS, scale, slopes, lds); break;
    case 10: shwfs_geometric_f64_kernel<10><<<grid, 128, 0, s>>>(opd, flux, valid_idx, nV, nS, scale, slopes, lds); break;
    default: shwfs_geometric_f64_kernel<12><<<grid, 128, 0, s>>>(opd, flux, valid_idx, nV, nS, scale, slopes, lds); break;
  }
  AOENV_LAUNCH_CHECK("shwfs_geometric_f64");
  return 0;
}

}  // extern "C"
