// bin_b200 -- training-batch assembly (DESIGN 5c rank 6): BINDataset.__getitem__ + DataLoader collation
// (data/BIN_dataset.py:30-54, Adobe_BIN_loader :63-183) on uint8 frames already in HBM.
//
// One launch builds a whole batch.  Sample b's 17 source frames arrive in the order the output slots want them
// (6 blurry, 6 sharp, 5 interpolation targets; the reference's random reversal is resolved by the caller through that
// order), with the crop offset (y0, x0) and the horizontal flip.  Every output value is float32(u8) / 255 correctly
// rounded, which is what read_img's `img.astype(np.float32) / 255.` computes (data/util.py:89), with BGR reordered to
// RGB (:42-44) and the layout made CHW (:47-49).  Outputs are slot-major ([slot][B][3][h][w]) so that every
// `LQs[:, i]` of feed_data (bin_model.py:147-202) is a contiguous (B, 3, h, w) tensor.
#include <string.h>

#include "common.cuh"
#include "internal.h"

namespace binb {

constexpr int kTdThreads = 256;
constexpr int kTdPix = 4;        // output pixels per thread (one float4 per plane)

struct TrainBatch {              // ~9.7 KB of kernel parameters at 64 samples (limit 32 KB)
  bin_train_sample_t smp[BIN_MAX_TRAIN_SAMPLES];
};

// grid = (pixel groups of one (h, w) crop, 17 slots, samples of this launch).  A thread reads the 4 * 3 source bytes of
// its 4 output pixels (contiguous in the frame, also when flipped) and writes 4 pixels of each of the 3 planes.
template <bool VEC>
__global__ void __launch_bounds__(kTdThreads) train_batch_u8_kernel(const __grid_constant__ TrainBatch P, int W, int h,
                                                                    int w, int b0, int Btot, float* __restrict__ lqs,
                                                                    float* __restrict__ gtenh, float* __restrict__ gtinp) {
  // the 256 possible values, one IEEE division per thread (the division's slow path is a call: keep it out of the
  // pixel loop, where it would cost spills)
  __shared__ float lut[256];
  static_assert(kTdThreads == 256, "one table entry per thread");
  lut[threadIdx.x] = __fdiv_rn((float)threadIdx.x, 255.f);
  __syncthreads();
  const int gw = (w + kTdPix - 1) / kTdPix;
  const int g = blockIdx.x * kTdThreads + threadIdx.x;
  if (g >= h * gw) return;
  const int slot = blockIdx.y, bl = blockIdx.z;
  const bin_train_sample_t& S = P.smp[bl];
  const int y = g / gw, x = (g - y * gw) * kTdPix;
  const int n = w - x < kTdPix ? w - x : kTdPix;                 // < 4 only in the last group of a row (w % 4 != 0)
  const uint8_t* row = S.src[slot] + ((size_t)(S.y0 + y) * W + S.x0) * 3;
  float* base;
  int k;
  if (slot < 6) { base = lqs; k = slot; }
  else if (slot < 12) { base = gtenh; k = slot - 6; }
  else { base = gtinp; k = slot - 12; }
  const size_t plane = (size_t)h * w;
  float* dst = base + ((size_t)k * Btot + b0 + bl) * 3 * plane + (size_t)y * w + x;
  float v[3][kTdPix];
#pragma unroll
  for (int i = 0; i < kTdPix; ++i) {
    if (i < n) {
      const int xs = S.flip ? w - 1 - (x + i) : x + i;          // np.fliplr of the crop (BIN_dataset.py:156-177)
      const uint8_t* px = row + (size_t)xs * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c][i] = lut[px[2 - c]];   // channel c = RGB <- BGR byte 2-c
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float* d = dst + (size_t)c * plane;
    if (VEC) {
      *reinterpret_cast<float4*>(d) = make_float4(v[c][0], v[c][1], v[c][2], v[c][3]);
    } else {
#pragma unroll
      for (int i = 0; i < kTdPix; ++i)
        if (i < n) d[i] = v[c][i];
    }
  }
}

int launch_train_batch_u8(const bin_train_sample_t* samples, int B, int H, int W, int h, int w, float* lqs, float* gtenh,
                          float* gtinp, cudaStream_t s) {
  if (B < 1) return fail(BIN_ERR_ARG, "train_batch: B must be at least 1");
  if (H < 1 || W < 1 || h < 1 || w < 1 || h > H || w > W)
    return fail(BIN_ERR_ARG, "train_batch: need 1 <= h <= H and 1 <= w <= W");
  if ((long long)H * W * 3 > (1ll << 40)) return fail(BIN_ERR_ARG, "train_batch: frame too large");
  for (int b = 0; b < B; ++b) {
    const bin_train_sample_t& S = samples[b];
    for (int f = 0; f < BIN_TRAIN_FRAMES; ++f)
      if (!S.src[f]) return fail(BIN_ERR_ARG, "train_batch: sample " + std::to_string(b) + " has a null frame pointer");
    if (S.y0 < 0 || S.x0 < 0 || S.y0 > H - h || S.x0 > W - w)
      return fail(BIN_ERR_ARG, "train_batch: crop of sample " + std::to_string(b) + " leaves the frame");
    if (S.flip != 0 && S.flip != 1) return fail(BIN_ERR_ARG, "train_batch: flip must be 0 or 1");
  }
  const bool vec = (w % kTdPix) == 0 &&
                   (((uintptr_t)lqs | (uintptr_t)gtenh | (uintptr_t)gtinp) & 15u) == 0;
  const int gw = (w + kTdPix - 1) / kTdPix;
  TrainBatch P;
  for (int b0 = 0; b0 < B; b0 += BIN_MAX_TRAIN_SAMPLES) {      // the sample table travels in the kernel parameters
    const int m = B - b0 < BIN_MAX_TRAIN_SAMPLES ? B - b0 : BIN_MAX_TRAIN_SAMPLES;
    memcpy(P.smp, samples + b0, (size_t)m * sizeof(bin_train_sample_t));
    const dim3 grid((unsigned)((h * gw + kTdThreads - 1) / kTdThreads), BIN_TRAIN_FRAMES, (unsigned)m);
    if (vec) train_batch_u8_kernel<true><<<grid, kTdThreads, 0, s>>>(P, W, h, w, b0, B, lqs, gtenh, gtinp);
    else train_batch_u8_kernel<false><<<grid, kTdThreads, 0, s>>>(P, W, h, w, b0, B, lqs, gtenh, gtinp);
    BIN_CUDA_OK(cudaGetLastError());
  }
  return BIN_OK;
}

}  // namespace binb
