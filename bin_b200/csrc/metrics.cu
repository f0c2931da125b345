// Image-quality metrics of the evaluation loop on uint8 HWC images: MSE, MAE and SSIM per image pair.
//
//   BIN_SSIM_BOX7    skimage 0.14-0.16 compare_ssim(X, Y, multichannel=True) with its defaults (test.py:35):
//                    7x7 uniform window, sample covariance (x 49/48), K1 = 0.01, K2 = 0.03, L = 255, map cropped by
//                    3 px, mean over channels of the per-channel means.
//   BIN_SSIM_GAUSS11 utils/util.py:211-231 ssim(): outer product of cv2.getGaussianKernel(11, 1.5), population
//                    moments, same K1 / K2, [5:-5, 5:-5] crop, mean over every element (util.py:246-247 averages
//                    three identical values for 3-channel input).
//
// Both references crop exactly the outputs whose window reaches past the image, so both are valid-region filters:
// output (oy, ox) of the (h-K+1) x (w-K+1) map reads input rows [oy, oy+K) and columns [ox, ox+K), and no kernel here
// handles a border.
//
// One CTA per (tile of kTH x kTW outputs, channel, pair).  It stages the (kTH+K-1) x (kTW+K-1) halo of both images in
// shared memory, runs a row pass and then a column pass over the five moments x, y, x^2, y^2, xy, and reduces its SSIM
// values and the integer sums of (a-b)^2 and |a-b| over the input pixels it owns.  Partials go to a workspace slab and
// a second kernel sums each pair's partials in a fixed order: no atomics, so a pair's result is bit-identical across
// calls and does not depend on which other pairs share the launch.
//
// Exactness: BOX7 window sums are integers (49 * 255^2 < 2^24), and so are the covariance numerators 49*Sxx - Sx^2;
// only the final ratio is floating point.  GAUSS11 runs its moments in fp64 (an fp32 E[x^2] - mu^2 cancels to ~1e-3).
// MSE and MAE are exact integer sums divided once, as numpy's mean of exactly representable float64 integers is.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <type_traits>

#include "internal.h"

namespace binb {

namespace {

constexpr int kMTW = 64;       // outputs per tile row
constexpr int kMTH = 16;       // output rows per tile
constexpr int kMThreads = 256;
constexpr double kC1 = (0.01 * 255) * (0.01 * 255);   // (K1 L)^2, util.py:212, skimage compare_ssim
constexpr double kC2 = (0.03 * 255) * (0.03 * 255);   // (K2 L)^2

struct MetricArgs {
  const uint8_t* a[BIN_MAX_METRIC_PAIRS];
  const uint8_t* b[BIN_MAX_METRIC_PAIRS];
  int h, w, c;
  int Ho, Wo, tiles_x, ntiles;
  double g[11];                // GAUSS11 weights (host-computed as cv2.getGaussianKernel does)
};

struct TilePartial {           // one per (pair, channel, tile)
  double ssim;                 // sum of the tile's SSIM map values
  unsigned long long sse, sae; // sum of (a-b)^2 and |a-b| over the input pixels the tile owns
};

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int K>
constexpr size_t tile_smem_bytes(bool gauss) {
  return 5 * (size_t)(kMTH + K - 1) * kMTW * (gauss ? sizeof(double) : sizeof(int)) +
         2 * (size_t)(kMTH + K - 1) * (kMTW + K - 1) * sizeof(int);
}

template <int K, bool GAUSS>
__global__ void __launch_bounds__(kMThreads) ssim_tile_kernel(const __grid_constant__ MetricArgs P,
                                                              TilePartial* __restrict__ part) {
  using Acc = typename std::conditional<GAUSS, double, int>::type;
  constexpr int HW = kMTW + K - 1, HH = kMTH + K - 1;
  extern __shared__ __align__(16) unsigned char smem[];
  Acc* rs = reinterpret_cast<Acc*>(smem);                                   // [5][HH][kMTW] row-pass moments
  int* ta = reinterpret_cast<int*>(smem + 5 * (size_t)HH * kMTW * sizeof(Acc));   // [HH][HW] halo of a
  int* tb = ta + HH * HW;                                                   // [HH][HW] halo of b

  const int tile = blockIdx.x, ch = blockIdx.y, pair = blockIdx.z;
  const int x0 = (tile % P.tiles_x) * kMTW, y0 = (tile / P.tiles_x) * kMTH;
  const uint8_t* A = P.a[pair];
  const uint8_t* B = P.b[pair];
  // Input pixels this tile counts for MSE / MAE: its own kMTW x kMTH block, extended to the image edge on the last
  // tile column / row (whose halo reaches the edge), so that the tiles partition the image.
  const int ox1 = x0 + kMTW >= P.Wo ? P.w : x0 + kMTW;
  const int oy1 = y0 + kMTH >= P.Ho ? P.h : y0 + kMTH;
  unsigned long long sse = 0, sae = 0;
  for (int i = threadIdx.x; i < HH * HW; i += kMThreads) {
    const int y = y0 + i / HW, x = x0 + i % HW;
    int va = 0, vb = 0;
    if (y < P.h && x < P.w) {
      const size_t off = ((size_t)y * P.w + x) * P.c + ch;
      va = A[off];
      vb = B[off];
      if (y < oy1 && x < ox1) {
        const int d = va - vb;
        sse += (unsigned)(d * d);
        sae += (unsigned)abs(d);
      }
    }
    ta[i] = va;
    tb[i] = vb;
  }
  __syncthreads();

  // row pass: horizontal window sums of the five moments for every halo row and every output column
  for (int i = threadIdx.x; i < HH * kMTW; i += kMThreads) {
    const int r = i / kMTW, col = i % kMTW;
    const int* pa = ta + r * HW + col;
    const int* pb = tb + r * HW + col;
    Acc sx = 0, sy = 0, sxx = 0, syy = 0, sxy = 0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const int xa = pa[j], xb = pb[j];
      if constexpr (GAUSS) {
        const double g = P.g[j];
        sx += g * (double)xa;
        sy += g * (double)xb;
        sxx += g * (double)(xa * xa);
        syy += g * (double)(xb * xb);
        sxy += g * (double)(xa * xb);
      } else {
        sx += xa;
        sy += xb;
        sxx += xa * xa;
        syy += xb * xb;
        sxy += xa * xb;
      }
    }
    rs[0 * HH * kMTW + i] = sx;
    rs[1 * HH * kMTW + i] = sy;
    rs[2 * HH * kMTW + i] = sxx;
    rs[3 * HH * kMTW + i] = syy;
    rs[4 * HH * kMTW + i] = sxy;
  }
  __syncthreads();

  // column pass + SSIM of each valid output; each thread sums its outputs in a fixed order
  double acc = 0.0;
  for (int i = threadIdx.x; i < kMTH * kMTW; i += kMThreads) {
    const int r = i / kMTW, col = i % kMTW;
    if (y0 + r >= P.Ho || x0 + col >= P.Wo) continue;
    Acc m[5] = {0, 0, 0, 0, 0};
#pragma unroll
    for (int j = 0; j < K; ++j) {
#pragma unroll
      for (int q = 0; q < 5; ++q) {
        const Acc v = rs[q * HH * kMTW + (r + j) * kMTW + col];
        if constexpr (GAUSS) m[q] += P.g[j] * v;
        else m[q] += v;
      }
    }
    if constexpr (GAUSS) {
      // util.py:218-229, term for term, each product and sum rounded on its own as numpy does (no FMA contraction:
      // it keeps numerator and denominator rounding alike, so an identical pair gives exactly 1)
      const double mu1 = m[0], mu2 = m[1];
      const double mu1_sq = __dmul_rn(mu1, mu1), mu2_sq = __dmul_rn(mu2, mu2), mu1_mu2 = __dmul_rn(mu1, mu2);
      const double s1 = __dsub_rn(m[2], mu1_sq), s2 = __dsub_rn(m[3], mu2_sq), s12 = __dsub_rn(m[4], mu1_mu2);
      const double num = __dmul_rn(__dadd_rn(__dmul_rn(2.0, mu1_mu2), kC1), __dadd_rn(__dmul_rn(2.0, s12), kC2));
      const double den = __dmul_rn(__dadd_rn(__dadd_rn(mu1_sq, mu2_sq), kC1), __dadd_rn(__dadd_rn(s1, s2), kC2));
      acc += num / den;
    } else {
      // skimage's (A1 A2) / (B1 B2) with ux = Sx/N, vx = (N Sxx - Sx^2) / (N (N-1)), N = 49: the common factors
      // 1/N^2 and 1/(N(N-1)) cancel, leaving exact integer numerators
      constexpr int N = K * K;
      const long long sx = m[0], sy = m[1];
      const long long nx = N * (long long)m[2] - sx * sx;
      const long long ny = N * (long long)m[3] - sy * sy;
      const long long nxy = N * (long long)m[4] - sx * sy;
      const double a1 = (double)(2 * sx * sy) + (double)(N * N) * kC1;
      const double a2 = (double)(2 * nxy) + (double)(N * (N - 1)) * kC2;
      const double b1 = (double)(sx * sx + sy * sy) + (double)(N * N) * kC1;
      const double b2 = (double)(nx + ny) + (double)(N * (N - 1)) * kC2;
      acc += (a1 * a2) / (b1 * b2);
    }
  }

  __shared__ double wd[kMThreads / 32];
  __shared__ unsigned long long we[kMThreads / 32], wa[kMThreads / 32];
  acc = warp_sum(acc);
  sse = warp_sum(sse);
  sae = warp_sum(sae);
  const int wid = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    wd[wid] = acc;
    we[wid] = sse;
    wa[wid] = sae;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    TilePartial t{0.0, 0ull, 0ull};
    for (int k = 0; k < kMThreads / 32; ++k) {
      t.ssim += wd[k];
      t.sse += we[k];
      t.sae += wa[k];
    }
    part[((size_t)pair * P.c + ch) * P.ntiles + tile] = t;
  }
}

// One CTA per pair: sums the pair's partials in a fixed order and writes res[pair] = {mse, mae, ssim}.
__global__ void __launch_bounds__(kMThreads) metrics_finalize_kernel(const TilePartial* __restrict__ part, int c,
                                                                     int ntiles, int h, int w, int Ho, int Wo,
                                                                     int gauss, double* __restrict__ res) {
  const int pair = blockIdx.x;
  __shared__ double wd[kMThreads / 32];
  __shared__ unsigned long long we[kMThreads / 32], wa[kMThreads / 32];
  double ssim_total = 0.0;
  unsigned long long sse_total = 0, sae_total = 0;
  const double nmap = (double)Ho * (double)Wo;
  for (int ch = 0; ch < c; ++ch) {
    const TilePartial* p = part + ((size_t)pair * c + ch) * ntiles;
    double s = 0.0;
    unsigned long long e = 0, a = 0;
    for (int t = threadIdx.x; t < ntiles; t += kMThreads) {
      s += p[t].ssim;
      e += p[t].sse;
      a += p[t].sae;
    }
    s = warp_sum(s);
    e = warp_sum(e);
    a = warp_sum(a);
    if ((threadIdx.x & 31) == 0) {
      wd[threadIdx.x >> 5] = s;
      we[threadIdx.x >> 5] = e;
      wa[threadIdx.x >> 5] = a;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double sc = 0.0;
      for (int k = 0; k < kMThreads / 32; ++k) {
        sc += wd[k];
        sse_total += we[k];
        sae_total += wa[k];
      }
      // BOX7: mean of the per-channel means; GAUSS11: one mean over every element of the (Ho, Wo, c) map
      ssim_total += gauss ? sc : sc / nmap;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double n = (double)h * (double)w * (double)c;
    res[pair * 3 + 0] = (double)sse_total / n;
    res[pair * 3 + 1] = (double)sae_total / n;
    res[pair * 3 + 2] = gauss ? ssim_total / (nmap * c) : ssim_total / c;
  }
}

int window_of(int kind) { return kind == BIN_SSIM_BOX7 ? 7 : (kind == BIN_SSIM_GAUSS11 ? 11 : 0); }

}  // namespace

size_t image_metrics_workspace_bytes(int npairs, int h, int w, int c, int kind) {
  const int K = window_of(kind);
  if (K == 0 || npairs < 1 || npairs > BIN_MAX_METRIC_PAIRS || (c != 1 && c != 3) || h < K || w < K) return 0;
  const size_t tiles = (size_t)((w - K + 1 + kMTW - 1) / kMTW) * ((h - K + 1 + kMTH - 1) / kMTH);
  return tiles * c * npairs * sizeof(TilePartial);
}

int launch_image_metrics_u8(const uint8_t* const* a, const uint8_t* const* b, int npairs, int h, int w, int c, int kind,
                            double* res, void* ws, size_t ws_bytes, cudaStream_t s) {
  const int K = window_of(kind);
  if (K == 0) return fail(BIN_ERR_ARG, "image_metrics: unknown SSIM kind (BIN_SSIM_BOX7 or BIN_SSIM_GAUSS11)");
  if (npairs < 1 || npairs > BIN_MAX_METRIC_PAIRS)
    return fail(BIN_ERR_ARG, "image_metrics: npairs must be in 1..BIN_MAX_METRIC_PAIRS");
  if (c != 1 && c != 3) return fail(BIN_ERR_ARG, "image_metrics: channels must be 1 or 3");
  if (h < K || w < K)
    return fail(BIN_ERR_ARG, "image_metrics: image smaller than the " + std::to_string(K) + "x" + std::to_string(K) +
                                 " SSIM window");
  for (int k = 0; k < npairs; ++k)
    if (!a[k] || !b[k]) return fail(BIN_ERR_ARG, "image_metrics: null image pointer");
  if ((reinterpret_cast<uintptr_t>(ws) & 7) != 0) return fail(BIN_ERR_ARG, "image_metrics: workspace not 8-byte aligned");
  const size_t need = image_metrics_workspace_bytes(npairs, h, w, c, kind);
  if (ws_bytes < need)
    return fail(BIN_ERR_ARG, "image_metrics: workspace too small (" + std::to_string(ws_bytes) + " < " +
                                 std::to_string(need) + " bytes)");

  MetricArgs P;
  memset(&P, 0, sizeof(P));
  for (int k = 0; k < npairs; ++k) {
    P.a[k] = a[k];
    P.b[k] = b[k];
  }
  P.h = h;
  P.w = w;
  P.c = c;
  P.Ho = h - K + 1;
  P.Wo = w - K + 1;
  P.tiles_x = (P.Wo + kMTW - 1) / kMTW;
  P.ntiles = P.tiles_x * ((P.Ho + kMTH - 1) / kMTH);
  // cv2.getGaussianKernel(11, 1.5) in double: t_i = exp(-x_i^2 / (2 sigma^2)), then every t_i times 1 / sum(t)
  {
    const double sigma = 1.5, scale2 = -0.5 / (sigma * sigma);
    double sum = 0.0;
    for (int i = 0; i < 11; ++i) {
      const double x = i - (11 - 1) * 0.5;
      P.g[i] = exp(scale2 * x * x);
      sum += P.g[i];
    }
    sum = 1.0 / sum;
    for (int i = 0; i < 11; ++i) P.g[i] *= sum;
  }

  TilePartial* part = static_cast<TilePartial*>(ws);
  const dim3 grid((unsigned)P.ntiles, (unsigned)c, (unsigned)npairs);
  if (kind == BIN_SSIM_BOX7) {
    static std::atomic<unsigned long long> done{0};
    constexpr int smem = (int)tile_smem_bytes<7>(false);
    BIN_TRY(ensure_dynamic_smem(ssim_tile_kernel<7, false>, smem, done));
    ssim_tile_kernel<7, false><<<grid, kMThreads, smem, s>>>(P, part);
  } else {
    static std::atomic<unsigned long long> done{0};
    constexpr int smem = (int)tile_smem_bytes<11>(true);
    BIN_TRY(ensure_dynamic_smem(ssim_tile_kernel<11, true>, smem, done));
    ssim_tile_kernel<11, true><<<grid, kMThreads, smem, s>>>(P, part);
  }
  BIN_CUDA_OK(cudaGetLastError());
  metrics_finalize_kernel<<<npairs, kMThreads, 0, s>>>(part, c, P.ntiles, h, w, P.Ho, P.Wo, kind == BIN_SSIM_GAUSS11,
                                                       res);
  BIN_CUDA_OK(cudaGetLastError());
  return BIN_OK;
}

}  // namespace binb
