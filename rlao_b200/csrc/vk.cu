// Episode reset: von Karman phase screens by the FFT method with three sub-harmonic grids (OOPAO/phaseStats.py:190-318,
// ft_phase_screen + ft_sh_phase_screen; called by Atmosphere.generateNewPhaseScreen, OOPAO/Atmosphere.py:560-592), for a
// batch of screens at once.
//
// The layer grid has N = R + 4 points per side (244, 484, ...: not a power of two, prime factor 61), so the 2-D transform
//     hi[y][x] = Re( fftshift(fft2(fftshift(cn))) ),  cn = (n_re + i n_im) sqrt(PSD) del_f
// is evaluated as two DENSE products with the N x N DFT matrix on the tensor cores (aoenv_gemm_tn_tc, split-bf16 operands):
//     pass A   U[b][y] = sum_a cn'[a][b] W[y][a]          rows (screen, b), K = (a, re|im), columns (y, re|im)
//     pass B   hi[y][x] = Re sum_b U[b][y] W[x][b]        rows (screen, y), K = (b, re|im), columns x
// with the two fftshifts folded into signs: cn' = (-1)^(a+b) cn, W[y][a] = (-1)^y exp(-2 pi i y a / N).
// This file holds the kernels around the two GEMMs: the random spectrum in operand form, the transposition between the
// passes, and the finish (sub-harmonics, mean removal, store into the layer canvas).
#include "common.cuh"

namespace aoenv {

// standard normal of the reference's stream position `flat` (row-major index into the N x N draw) of screen `s`:
// component 0 = the real-part draw, 1 = the imaginary-part draw
__device__ __forceinline__ float2 vk_normals(const Philox& rng, const float* __restrict__ inject, int S, int N, uint32_t s,
                                             uint32_t flat) {
  if (inject != nullptr) {
    const size_t base = (size_t)s * 2 * N * N;
    return make_float2(__ldg(inject + base + flat), __ldg(inject + base + (size_t)N * N + flat));
  }
  const uint4 w = rng(flat, s, 0x564bu, 0u);
  return box_muller(w.x, w.y);
}

// Philox stream of screen s: screen0 + s, or screen0 + env_idx[s] when the screens go to a list of environments
__device__ __forceinline__ uint32_t vk_stream(uint32_t screen0, const int32_t* __restrict__ env_idx, int s) {
  return screen0 + (uint32_t)(env_idx ? __ldg(&env_idx[s]) : s);
}

// planes[(s, b)][k]: k < N -> Re cn'[a = k][b], N <= k < 2N -> Im cn'[a = k - N][b], zero beyond (operand of pass A)
__global__ void __launch_bounds__(256)
vk_spectrum_kernel(unsigned long long seed, uint32_t screen0, int S, int N, const float* __restrict__ amp,
                   const float* __restrict__ inject, __nv_bfloat16* __restrict__ planes, int Kp, int parts,
                   const int32_t* __restrict__ env_idx) {
  const int s = blockIdx.z, b = blockIdx.y;
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= Kp) return;
  const size_t row = (size_t)s * N + b;
  const size_t stride = (size_t)S * N * Kp;
  if (a < N) {
    Philox rng(seed);
    const uint32_t flat = (uint32_t)a * N + b;
    const float2 z = vk_normals(rng, inject, S, N, inject ? (uint32_t)s : vk_stream(screen0, env_idx, s), flat);
    const float w = __ldg(&amp[flat]);                       // sqrt(PSD) del_f (-1)^(a+b)
    store_bf16_planes(planes, stride, row * Kp + a, parts, z.x * w);
    store_bf16_planes(planes, stride, row * Kp + N + a, parts, z.y * w);
  } else if (a >= 2 * N) {
    for (int p = 0; p < parts; ++p) planes[(size_t)p * stride + row * Kp + a] = __float2bfloat16_rn(0.f);
  }
}

// out planes[(s, y)][k] = src[(s, b = k mod N)][(k / N) * N + y]: the [b][y] -> [y][b] transposition between the passes,
// through a 32 x 32 shared-memory tile, written directly in split-bf16 operand form
__global__ void __launch_bounds__(256)
vk_transpose_kernel(const float* __restrict__ src, int lds, int S, int N, __nv_bfloat16* __restrict__ planes, int Kp, int parts) {
  __shared__ float tile[32][33];
  const int s = blockIdx.z / 2, half = blockIdx.z & 1;      // half 0: real part, 1: imaginary part
  const int b0 = blockIdx.y * 32, y0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;    // 32 x 8
  for (int r = ty; r < 32; r += 8) {
    const int b = b0 + r, y = y0 + tx;
    tile[r][tx] = (b < N && y < N) ? __ldg(&src[((size_t)s * N + b) * lds + half * N + y]) : 0.f;
  }
  __syncthreads();
  const size_t stride = (size_t)S * N * Kp;
  for (int r = ty; r < 32; r += 8) {
    const int y = y0 + r, b = b0 + tx;
    if (y < N && b < N) store_bf16_planes(planes, stride, ((size_t)s * N + y) * Kp + half * N + b, parts, tile[tx][r]);
  }
  // zero padding of the K axis (columns 2N .. Kp), once per row
  if (blockIdx.y == 0 && half == 0) {
    for (int r = ty; r < 32; r += 8) {
      const int y = y0 + r;
      if (y < N)
        for (int k = 2 * N + tx; k < Kp; k += 32)
          for (int p = 0; p < parts; ++p) planes[(size_t)p * stride + ((size_t)s * N + y) * Kp + k] = __float2bfloat16_rn(0.f);
    }
  }
}

struct VkSubharmonics {
  const float2* ex;      // [3][2][N] exp(2 pi i gx x)   (gx = -df_p, 0)
  const float2* ey;      // [3][2][N] exp(2 pi i gy y)
  float amp[3][2][2];    // sqrt(PSD) df_p at (i, j)     (gy index i, gx index j)
  float2 mx[3][2], my[3][2];   // means of ex / ey over the grid (for the analytic mean of the low-frequency screen)
};

// screen = hi + lo - mean(lo), stored into the interior of the layer window (the reference's layer.phase) of environment
// s, or env_idx[s]
__global__ void __launch_bounds__(256)
vk_finish_kernel(const float* __restrict__ hi, int ldh, unsigned long long seed, uint32_t screen0, int S, int N,
                 const float* __restrict__ inject, const __grid_constant__ VkSubharmonics sh, float* __restrict__ dst, int pitch,
                 size_t env_stride, const int32_t* __restrict__ env_idx) {
  __shared__ float2 cs[3][2][2];
  __shared__ float mean;
  const int s = blockIdx.z, y = blockIdx.y;
  if (threadIdx.x < 12) {
    // The reference seeds the sub-harmonic draws like the FFT draws (phaseStats.py:268,272): grid p takes, for its real
    // parts, the stream positions 18 (p-1) + 3 i + j of the real-part draw, and 9 further on for its imaginary parts.
    const int p = threadIdx.x / 4, i = (threadIdx.x >> 1) & 1, j = threadIdx.x & 1;
    Philox rng(seed);
    const uint32_t sid = inject ? (uint32_t)s : vk_stream(screen0, env_idx, s);
    const float re = vk_normals(rng, inject, S, N, sid, 18u * p + 3u * i + j).x;
    const float im = vk_normals(rng, inject, S, N, sid, 18u * p + 9u + 3u * i + j).x;
    cs[p][i][j] = make_float2(re * sh.amp[p][i][j], im * sh.amp[p][i][j]);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int p = 0; p < 3; ++p)
      for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2; ++j) {
          const float2 e = make_float2(sh.my[p][i].x * sh.mx[p][j].x - sh.my[p][i].y * sh.mx[p][j].y,
                                       sh.my[p][i].x * sh.mx[p][j].y + sh.my[p][i].y * sh.mx[p][j].x);
          m += cs[p][i][j].x * e.x - cs[p][i][j].y * e.y;
        }
    mean = m;
  }
  __syncthreads();
  // per row: t[p][j] = sum_i cs[p][i][j] ey[p][i][y]
  float2 t[3][2];
#pragma unroll
  for (int p = 0; p < 3; ++p)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      float2 acc = make_float2(0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const float2 e = __ldg(&sh.ey[(p * 2 + i) * N + y]), c = cs[p][i][j];
        acc.x += c.x * e.x - c.y * e.y;
        acc.y += c.x * e.y + c.y * e.x;
      }
      t[p][j] = acc;
    }
  float* __restrict__ out = dst + (size_t)(env_idx ? __ldg(&env_idx[s]) : s) * env_stride + (size_t)y * pitch;
  const float* __restrict__ h = hi + ((size_t)s * N + y) * ldh;
  for (int x = threadIdx.x; x < N; x += blockDim.x) {
    float lo = 0.f;
#pragma unroll
    for (int p = 0; p < 3; ++p)
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const float2 e = __ldg(&sh.ex[(p * 2 + j) * N + x]);
        lo += t[p][j].x * e.x - t[p][j].y * e.y;
      }
    out[x] = __ldg(&h[x]) + lo - mean;
  }
}

}  // namespace aoenv

using namespace aoenv;

namespace {

int vk_screens(uint64_t seed, uint32_t screen0, const int32_t* env_idx, int S, int N, const float* amp, const float* inject,
               const void* wa_planes, const void* wb_planes, int Kp, int parts, const float* sh_ex, const float* sh_ey,
               const float* h_amp, const float* h_mx, const float* h_my, void* work_planes, float* work_a, int lda, float* work_b,
               int ldb, float* dst, int pitch, int64_t env_stride, void* stream) {
  AOENV_CHECK_ARG(S > 0 && 2 * S <= 65535 && N >= 8 && N <= 32768, "vk_screens: bad shape S=%d N=%d", S, N);
  AOENV_CHECK_ARG(Kp >= 2 * N && Kp % 16 == 0 && lda >= 2 * N && ldb >= N && pitch >= N, "vk_screens: bad leading dimensions");
  AOENV_CHECK_ARG(parts == 2 || parts == 3, "vk_screens: parts must be 2 or 3");
  cudaStream_t st = (cudaStream_t)stream;
  __nv_bfloat16* planes = (__nv_bfloat16*)work_planes;
  // random spectrum, operand form of pass A
  vk_spectrum_kernel<<<dim3((Kp + 255) / 256, N, S), 256, 0, st>>>(seed, screen0, S, N, amp, inject, planes, Kp, parts, env_idx);
  AOENV_LAUNCH_CHECK("vk_spectrum");
  // pass A: U[(s, b)][(y, re|im)] = sum_(a, re|im) cn'[(s, b)][(a, re|im)] WA[(y, re|im)][(a, re|im)]
  int rc = aoenv_gemm_tn_tc(planes, wa_planes, Kp, parts, work_a, lda, S * N, 2 * N, Kp, 1.0f, stream);
  if (rc) return rc;
  vk_transpose_kernel<<<dim3((N + 31) / 32, (N + 31) / 32, 2 * S), 256, 0, st>>>(work_a, lda, S, N, planes, Kp, parts);
  AOENV_LAUNCH_CHECK("vk_transpose");
  // pass B: hi[(s, y)][x] = sum_(b, re|im) U[(s, y)][(b, re|im)] WB[x][(b, re|im)]
  rc = aoenv_gemm_tn_tc(planes, wb_planes, Kp, parts, work_b, ldb, S * N, N, Kp, 1.0f, stream);
  if (rc) return rc;
  VkSubharmonics sh;
  sh.ex = reinterpret_cast<const float2*>(sh_ex);
  sh.ey = reinterpret_cast<const float2*>(sh_ey);
  for (int p = 0; p < 3; ++p)
    for (int i = 0; i < 2; ++i) {
      for (int j = 0; j < 2; ++j) sh.amp[p][i][j] = h_amp[(p * 2 + i) * 2 + j];
      sh.mx[p][i] = make_float2(h_mx[(p * 2 + i) * 2], h_mx[(p * 2 + i) * 2 + 1]);
      sh.my[p][i] = make_float2(h_my[(p * 2 + i) * 2], h_my[(p * 2 + i) * 2 + 1]);
    }
  vk_finish_kernel<<<dim3(1, N, S), 256, 0, st>>>(work_b, ldb, seed, screen0, S, N, inject, sh, dst, pitch, (size_t)env_stride,
                                              env_idx);
  AOENV_LAUNCH_CHECK("vk_finish");
  return 0;
}

}  // namespace

extern "C" {

int aoenv_vk_screens(uint64_t seed, uint32_t screen0, int S, int N, const float* amp, const float* inject, const void* wa_planes,
                     const void* wb_planes, int Kp, int parts, const float* sh_ex, const float* sh_ey, const float* h_amp,
                     const float* h_mx, const float* h_my, void* work_planes, float* work_a, int lda, float* work_b, int ldb,
                     float* dst, int pitch, int64_t env_stride, void* stream) {
  return vk_screens(seed, screen0, nullptr, S, N, amp, inject, wa_planes, wb_planes, Kp, parts, sh_ex, sh_ey, h_amp, h_mx, h_my,
                    work_planes, work_a, lda, work_b, ldb, dst, pitch, env_stride, stream);
}

int aoenv_vk_screens_envs(uint64_t seed, uint32_t screen0, const int32_t* env_idx, int S, int N, const float* amp,
                          const void* wa_planes, const void* wb_planes, int Kp, int parts, const float* sh_ex, const float* sh_ey,
                          const float* h_amp, const float* h_mx, const float* h_my, void* work_planes, float* work_a, int lda,
                          float* work_b, int ldb, float* dst, int pitch, int64_t env_stride, void* stream) {
  AOENV_CHECK_ARG(env_idx != nullptr, "vk_screens_envs: no environment list");
  return vk_screens(seed, screen0, env_idx, S, N, amp, nullptr, wa_planes, wb_planes, Kp, parts, sh_ex, sh_ey, h_amp, h_mx, h_my,
                    work_planes, work_a, lda, work_b, ldb, dst, pitch, env_stride, stream);
}

}  // extern "C"
