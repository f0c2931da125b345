// bin_b200 -- extern "C" entry points (include/bin_b200.h) and the host-side orchestration of
// one backbone / one 6-frame window.  Host code only: every arithmetic step is a kernel in
// conv_igemm.cu / aux_kernels.cu.
#include <stdlib.h>
#include <string.h>

#include <initializer_list>
#include <string>
#include <vector>

#include "internal.h"

namespace binb {

static thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

static Options read_options() {
  Options o;
  auto env = [](const char* k) { const char* e = getenv(k); return (e && *e) ? e : nullptr; };
  const char* e;
  o.debug = (e = env("BIN_B200_DEBUG")) ? atoi(e) : 0;
  o.fuse_lff = !((e = env("BIN_B200_FUSE_LFF")) && *e == '0');
  o.tail_streams = !((e = env("BIN_B200_TAIL_STREAMS")) && *e == '0');
  o.pair = (e = env("BIN_B200_PAIR")) && *e == '1';     // CTA-pair kernels: opt-in until verified on hardware
  o.msplit = (e = env("BIN_B200_MSPLIT")) && *e == '1';
  o.quad = !((e = env("BIN_B200_QUAD")) && *e == '0');  // four MMA warps in the x-stacked conv: default (measured +8 %)
  o.tailq = (e = env("BIN_B200_TAILQ")) && *e == '1';
  o.spread = (e = env("BIN_B200_SPREAD")) && *e == '1';
  o.polite = (e = env("BIN_B200_POLITE")) && *e == '1';
  o.zigzag = (e = env("BIN_B200_ZIGZAG")) && *e == '1';
  o.stage_mmas = (e = env("BIN_B200_STAGE_MMAS")) ? atoi(e) : 12;
  if (o.stage_mmas < 1) o.stage_mmas = 12;
  o.band_budget = (e = env("BIN_B200_BAND_BUDGET_KB")) ? (size_t)atoll(e) << 10 : (~(size_t)0 >> 1);
  return o;
}
const Options& options() {
#ifdef BIN_B200_TOOLS
  static thread_local Options o;
  o = read_options();
  return o;
#else
  static const Options o = read_options();
  return o;
#endif
}

int num_sms() {
  static std::atomic<int> cache[64];
  int dev = 0;
  cudaGetDevice(&dev);
  int v = cache[dev & 63].load(std::memory_order_relaxed);
  if (v == 0) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    if (v <= 0) v = 148;
    cache[dev & 63].store(v, std::memory_order_relaxed);
  }
  return v;
}

int launch_nchw_to_p8(const float* x, int C, const bin_act_t& dst, int plane0, cudaStream_t s);
int launch_p8_to_nchw(const bin_act_t& src, int plane0, int C, float* y, cudaStream_t s);
int launch_pack_frames(const bin_frames_t& fr, int H, int W, const bin_act_t& dst, cudaStream_t s, int x3 = 0);
int launch_pack_weight(const float* w, int cout, int cin, int ks, int cout_pad, int cin_pad, int variant,
                       void* packed, cudaStream_t s, int x3 = 0);
int launch_pack_bias(const float* b, int cout, int cout_pad, float* dst, cudaStream_t s);
int launch_grad_scale(const float* const* gouts, int n, size_t numel, float target, float* scale_dev, unsigned* tmp_dev,
                      cudaStream_t s);
// batched packing: all tensors of one blob in one launch (aux_kernels.cu)
void* pack_batch_new();
int pack_batch_add_weight(void* hb, const float* w, int cout, int cin, int ks, int cout_pad, int cin_pad, int variant,
                          void* packed, int x3);
int pack_batch_add_weight_t(void* hb, const float* w, int cout, int cin, int ks, int row0, int nrows, int cout_pad_t,
                            int cin_pad_t, void* packed);
int pack_batch_add_bias(void* hb, const float* b, int cout, int cout_pad, float* dst);
int pack_batch_launch(void* hb, cudaStream_t s);   // launches and frees the batch
int launch_convlstm(const float* x, const float* c_prev, const float* h_prev, const float* w, const float* b,
                    float* h_out, float* c_out, int B, int H, int W, cudaStream_t s);
int launch_pixel_loss_fwd(const float* const* a, const float* const* b, int npairs, size_t n, int kind, float eps,
                          float* pair_loss, cudaStream_t s);
int launch_pixel_loss_bwd(const float* const* a, const float* const* b, float* const* da, float* const* db, int npairs,
                          size_t n, int kind, float eps, const float* upstream, cudaStream_t s);
int launch_adam_step(const bin_adam_tensor_t* table, const int* chunk_prefix, int ntensors, int nchunks, float lr,
                     float beta1, float beta2, float eps, float weight_decay, float bias_correction1,
                     float bias_correction2, float grad_scale, cudaStream_t s);
int launch_blur_average_u8(const uint8_t* frames, int T, size_t frame_bytes, int window_size, int first_mid, int stride,
                           int nwin, uint8_t* out, cudaStream_t s);
int launch_rdb_tail(const bin_act_t& x, int x_plane0, const bin_act_t& g, int g_plane0, const void* w_conv,
                    const float* b_conv, const void* w_lff, const float* b_lff, const bin_act_t& out, int out_plane0,
                    int b_begin, int b_count, int y_begin, int y_count, cudaStream_t s, bool reverse = false);
int launch_tensor2img_u8(const float* x, int Hs, int Ws, int top, int left, int h, int w, uint8_t* out, cudaStream_t s);
int launch_u8_to_frame(const uint8_t* img, int h, int w, int pl, int pr, int pt, int pb, float* out, cudaStream_t s);
int launch_convlstm_bwd(const float* x, const float* c_prev, const float* h_prev, const float* w, const float* b,
                        const float* dh, const float* dc, float* dgates_ws, float* dx, float* dc_prev, float* dh_prev,
                        float* dw, float* db, int B, int H, int W, cudaStream_t s);
size_t image_metrics_workspace_bytes(int npairs, int h, int w, int c, int kind);   // metrics.cu
int launch_image_metrics_u8(const uint8_t* const* a, const uint8_t* const* b, int npairs, int h, int w, int c, int kind,
                            double* res, void* ws, size_t ws_bytes, cudaStream_t s);
int launch_train_batch_u8(const bin_train_sample_t* samples, int B, int H, int W, int h, int w, float* lqs, float* gtenh,
                          float* gtinp, cudaStream_t s);   // train_data.cu

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------ backbone conv table
// Order = nn.Module registration order of the reference backbones (RDN.py:187-208): SFENet1,
// SFENet2, RDBs.{i}.convs.{0..3}, RDBs.{i}.LFF, GFF.0, GFF.1, UPNet.0, UPNet.2.
struct ConvSpec {
  int cin, cout, ks, cin_pad, cout_pad;
  size_t w_off, b_off;
};
constexpr int kG0 = 96, kD = 12, kCgrow = 4, kG = 32;

struct BackboneLayout {
  ConvSpec conv[BIN_BACKBONE_NCONV];
  size_t bytes;
};

static BackboneLayout backbone_layout(int nframes, int x3 = 0) {
  BackboneLayout L;
  int k = 0;
  auto add = [&](int cin, int cout, int ks, int cout_pad) {
    ConvSpec c;
    c.cin = cin; c.cout = cout; c.ks = ks;
    c.cin_pad = (int)align_up(cin, kKC);
    c.cout_pad = cout_pad;
    c.w_off = c.b_off = 0;
    L.conv[k++] = c;
  };
  add(12 * nframes, kG0, 5, 96);
  add(kG0, kG0, 3, 96);
  for (int i = 0; i < kD; ++i) {
    for (int c = 0; c < kCgrow; ++c) add(kG0 + c * kG, kG, 3, 32);
    add(kG0 + kCgrow * kG, kG0, 1, 96);
  }
  add(kD * kG0, kG0, 1, 96);
  add(kG0, kG0, 3, 96);
  add(kG0, 256, 3, 256);
  add(64, 3, 3, 16);
  size_t off = 0;
  for (int i = 0; i < BIN_BACKBONE_NCONV; ++i) {
    ConvSpec& c = L.conv[i];
    c.w_off = off;
    off = align_up(off + (size_t)c.cout_pad * c.cin_pad * c.ks * c.ks * sizeof(__half) * (x3 ? 3 : 1), 256);
    c.b_off = off;
    off = align_up(off + (size_t)c.cout_pad * sizeof(float), 256);
  }
  L.bytes = off;
  return L;
}

static bool valid_nframes(int n) { return n == 2 || n == 3 || n == 5; }

// ------------------------------------------------------------------ backbone workspace
struct BackboneWs {
  bin_act_t x0, f1, f2, cat, g, t1, t2, u;
  size_t bytes;
};
static BackboneWs backbone_ws(int nframes, int Btot, int H, int W, void* base, bool train = false, int x3 = 0) {
  BackboneWs w;
  const int h = H / 2, wd = W / 2;
  size_t off = 0;
  auto carve = [&](int planes, int hh, int ww) {
    bin_act_t t;
    t.ptr = base ? (void*)((uint8_t*)base + off) : nullptr;
    t.B = Btot; t.planes = planes * (x3 ? 2 : 1); t.H = hh; t.W = ww;      // x3: hi + lo plane groups
    off = align_up(off + (size_t)Btot * t.planes * hh * ww * 16, 256);
    return t;
  };
  w.x0 = carve((int)align_up(12 * nframes, kKC) / 8, h, wd);
  w.f1 = carve(12, h, wd);
  w.f2 = carve(12, h, wd);
  w.cat = carve(12 * kD, h, wd);
  w.g = carve(train ? 16 * kD : 16, h, wd);   // training keeps the growth maps of all 12 RDBs for the backward
  w.t1 = carve(12, h, wd);
  w.t2 = carve(12, h, wd);
  w.u = carve(8, H, W);
  w.bytes = off;
  return w;
}

static bin_conv_args_t conv_args(const void* blob, const ConvSpec& c, int x3 = 0) {
  bin_conv_args_t a;
  memset(&a, 0, sizeof(a));
  a.x3 = x3;
  a.w_packed = (const uint8_t*)blob + c.w_off;
  a.bias = (const float*)((const uint8_t*)blob + c.b_off);
  a.ksize = c.ks;
  a.cout_pad = c.cout_pad;
  return a;
}

// ------------------------------------------------------------------ L2 band plan for the RDB section
// An RDB run layer-by-layer over the whole (batched) image moves 2 240 B/position through HBM
// (each conv re-reads the growing concat); measured, that makes the RDB convs HBM-bound at ~50 % of
// the tensor peak.  Walking the RDB band by band -- all 5 layers for one band before the next --
// keeps x (192 B/px) + growth scratch (256 B/px) + x' (192 B/px) of the band inside the 126 MB L2,
// so only x in / x' out (384 B/position) touch HBM.  Bands overlap by the 3-row receptive field of
// the chained 3x3 convs (rows are recomputed, values identical).  Boundaries sit at rows 8k-3 so
// every layer of a band has the same number of 8-row tile rows, and k is chosen to minimise the
// number of 148-CTA waves.
struct Band { int b0, nb, y0, y1; };   // batch items [b0,b0+nb), LFF output rows [y0,y1)
constexpr size_t kBandBytesPerPx = 640;
static size_t band_budget() {            // BIN_B200_BAND_BUDGET_KB overrides (tests force many bands)
  // Measured on B200 (720p, 5 batched calls): with 10 bands the 10x launch count costs more
  // (prologue + drain per launch, ~4 us each) than the L2 residency saves: 41.5 ms vs 31.8 ms per
  // window.  Default = one band (off).
  return options().band_budget;
}

static std::vector<Band> plan_bands(int Btot, int h, int w) {
  std::vector<Band> out;
  const size_t px_max = band_budget() / kBandBytesPerPx;
  const size_t img = (size_t)h * w;
  if (img <= px_max) {                       // small images: several batch items per band, full rows
    const size_t per_sz = px_max / img;
    int per = per_sz >= (size_t)Btot ? Btot : (int)per_sz;
    if (per < 1) per = 1;
    for (int b = 0; b < Btot; b += per) out.push_back({b, (b + per <= Btot) ? per : Btot - b, 0, h});
    return out;
  }
  const int tx = (w + 29) / 30;
  const int T = (h + 7) / 8;                 // boundaries allowed at rows 8k-3, k = 1..T-1
  const int maxrows = (int)(px_max / w);
  const int sms = num_sms();
  auto waves = [&](int rows) { int t = ((rows + 7) / 8) * tx; return (t + sms - 1) / sms; };
  // dp[k] = min waves to cover rows [0, 8k-3) with bands ending at k; last band ends at h.
  const int INF = 1 << 30;
  std::vector<int> dp(T + 1, INF), prev(T + 1, -1);
  dp[0] = 0;
  int best = INF, best_k = -1;
  for (int k = 0; k < T; ++k) {
    if (dp[k] == INF) continue;
    const int start = k == 0 ? 0 : 8 * k - 3;
    for (int k2 = k + 1; k2 < T; ++k2) {     // middle band [start, 8*k2-3)
      const int end = 8 * k2 - 3;
      if (end <= start || end >= h) continue;
      if (end - start > maxrows) break;
      const int lo = start - 3 < 0 ? 0 : start - 3, hi = end + 3 > h ? h : end + 3;
      const int c = dp[k] + waves(hi - lo);
      if (c < dp[k2] || (c == dp[k2] && prev[k2] < k)) { dp[k2] = c; prev[k2] = k; }
    }
    if (h - start <= maxrows) {               // close with the last band [start, h)
      const int lo = start - 3 < 0 ? 0 : start - 3;
      const int c = dp[k] + waves(h - lo);
      if (c < best) { best = c; best_k = k; }
    }
  }
  std::vector<int> cuts;
  for (int k = best_k; k > 0; k = prev[k]) cuts.push_back(8 * k - 3);
  std::vector<int> edges = {0};
  for (auto it = cuts.rbegin(); it != cuts.rend(); ++it) edges.push_back(*it);
  edges.push_back(h);
  if (best_k < 0) edges = {0, h};
  for (int b = 0; b < Btot; ++b)
    for (size_t i = 0; i + 1 < edges.size(); ++i) out.push_back({b, 1, edges[i], edges[i + 1]});
  return out;
}

// One RDB: 4 x (conv3x3+ReLU -> growth planes) + LFF 1x1 + residual (RDN.py:149-165).
// The last conv and the LFF run as one kernel (rdb_tail.cu) in fp16 inference; training keeps them apart because the
// backward needs the fourth growth map, and the split-fp16 mode has no fused variant.  BIN_B200_FUSE_LFF=0 disables it.
static bool fuse_lff_enabled() { return options().fuse_lff; }
static int run_rdb(const void* blob, const BackboneLayout& L, int i, const bin_act_t& xin, int x_plane0,
                   const bin_act_t& g, const bin_act_t& out, int out_plane0, const std::vector<Band>& bands,
                   cudaStream_t s, int g_plane0 = 0, int x3 = 0, bool keep_growth = false) {
  const int base = 2 + i * (kCgrow + 1);
  const int h = xin.H;
  const bool fuse = !x3 && !keep_growth && fuse_lff_enabled();
  for (const Band& bd : bands) {
    for (int c = 0; c < (fuse ? kCgrow - 1 : kCgrow); ++c) {
      bin_conv_args_t a = conv_args(blob, L.conv[base + c], x3);
      a.in0 = xin; a.in0_plane0 = x_plane0; a.in0_planes = 12;
      a.in1 = g; a.in1_plane0 = g_plane0; a.in1_planes = 4 * c;
      a.relu = 1; a.epilogue = BIN_EPI_P8;
      a.out = g; a.out_plane0 = g_plane0 + 4 * c;
      const int ext = kCgrow - 1 - c;             // rows still needed by the convs downstream in this band
      const int lo = bd.y0 - ext < 0 ? 0 : bd.y0 - ext, hi = bd.y1 + ext > h ? h : bd.y1 + ext;
      a.b_begin = bd.b0; a.b_count = bd.nb; a.y_begin = lo; a.y_count = hi - lo;
      // zigzag: conv0 forward, conv1 backward, conv2 forward, tail backward -- every launch starts on the tiles its
      // predecessor touched last, which are the ones still in the 126 MB L2 (the tail ends at tile 0, where the next
      // RDB's conv0 starts)
      BIN_TRY(launch_conv(a, s, options().zigzag && (c & 1)));
    }
    if (fuse) {
      const ConvSpec& c3 = L.conv[base + kCgrow - 1];
      const ConvSpec& lf = L.conv[base + kCgrow];
      BIN_TRY(launch_rdb_tail(xin, x_plane0, g, g_plane0, (const uint8_t*)blob + c3.w_off,
                              (const float*)((const uint8_t*)blob + c3.b_off), (const uint8_t*)blob + lf.w_off,
                              (const float*)((const uint8_t*)blob + lf.b_off), out, out_plane0, bd.b0, bd.nb, bd.y0,
                              bd.y1 - bd.y0, s, options().zigzag));
      continue;
    }
    bin_conv_args_t a = conv_args(blob, L.conv[base + kCgrow], x3);
    a.in0 = xin; a.in0_plane0 = x_plane0; a.in0_planes = 12;
    a.in1 = g; a.in1_plane0 = g_plane0; a.in1_planes = 16;
    a.epilogue = BIN_EPI_P8;
    a.out = out; a.out_plane0 = out_plane0;
    a.res = xin; a.res_plane0 = x_plane0;
    a.b_begin = bd.b0; a.b_count = bd.nb; a.y_begin = bd.y0; a.y_count = bd.y1 - bd.y0;
    BIN_TRY(launch_conv(a, s));
  }
  return BIN_OK;
}

static int run_backbone(int nframes, const void* blob, const bin_frames_t& fr, int H, int W, void* workspace,
                        size_t workspace_bytes, cudaStream_t s, bool train = false, int x3 = 0) {
  if (!valid_nframes(nframes) || fr.nframes != nframes) return fail(BIN_ERR_ARG, "backbone: nframes must be 2, 3 or 5");
  if (fr.ncalls < 1 || fr.ncalls > BIN_MAX_CALLS || fr.Bc < 1) return fail(BIN_ERR_ARG, "backbone: bad call table");
  if ((H & 1) || (W & 1) || H < 2 || W < 2) return fail(BIN_ERR_ARG, "backbone: H and W must be even (RDN.py:123-128)");
  const int Btot = fr.ncalls * fr.Bc;
  if (train && x3) return fail(BIN_ERR_UNSUPPORTED, "backbone: training runs in the fp16 mode only");
  const BackboneLayout L = backbone_layout(nframes, x3);
  const BackboneWs ws = backbone_ws(nframes, Btot, H, W, workspace, train, x3);
  if (ws.bytes > workspace_bytes) return fail(BIN_ERR_WORKSPACE, "backbone: workspace too small");
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) != 0) return fail(BIN_ERR_ARG, "backbone: workspace must be 256-byte aligned");

  BIN_TRY(launch_pack_frames(fr, H, W, ws.x0, s, x3));                           // RDN.py:211
  {
    bin_conv_args_t a = conv_args(blob, L.conv[0], x3);                              // SFENet1 (RDN.py:212)
    a.in0 = ws.x0; a.in0_planes = ws.x0.planes / (x3 ? 2 : 1); a.epilogue = BIN_EPI_P8; a.out = ws.f1;
    BIN_TRY(launch_conv(a, s));
  }
  {
    bin_conv_args_t a = conv_args(blob, L.conv[1], x3);                              // SFENet2 (RDN.py:213)
    a.in0 = ws.f1; a.in0_planes = 12; a.epilogue = BIN_EPI_P8; a.out = ws.f2;
    BIN_TRY(launch_conv(a, s));
  }
  const std::vector<Band> bands = plan_bands(Btot, H / 2, W / 2);
  for (int i = 0; i < kD; ++i) {                                                 // RDN.py:215-217
    const int gp0 = train ? 16 * i : 0;
    if (i == 0) BIN_TRY(run_rdb(blob, L, i, ws.f2, 0, ws.g, ws.cat, 0, bands, s, gp0, x3, train));
    else BIN_TRY(run_rdb(blob, L, i, ws.cat, 12 * (i - 1), ws.g, ws.cat, 12 * i, bands, s, gp0, x3, train));
  }
  {
    bin_conv_args_t a = conv_args(blob, L.conv[62], x3);                             // GFF.0 on the 1152-ch concat (RDN.py:218)
    a.in0 = ws.cat; a.in0_planes = 12 * kD; a.epilogue = BIN_EPI_P8; a.out = ws.t1;
    BIN_TRY(launch_conv(a, s));
  }
  {
    bin_conv_args_t a = conv_args(blob, L.conv[63], x3);                             // GFF.1, x += f__1 (RDN.py:219)
    a.in0 = ws.t1; a.in0_planes = 12; a.epilogue = BIN_EPI_P8; a.out = ws.t2; a.res = ws.f1;
    BIN_TRY(launch_conv(a, s));
  }
  {
    bin_conv_args_t a = conv_args(blob, L.conv[64], x3);                             // UPNet.0 + PixelShuffle (RDN.py:205-206)
    a.in0 = ws.t2; a.in0_planes = 12; a.epilogue = BIN_EPI_PIXSHUF; a.out = ws.u;
    BIN_TRY(launch_conv(a, s));
  }
  {
    bin_conv_args_t a = conv_args(blob, L.conv[65], x3);                             // UPNet.2 + mean(frames) (RDN.py:207,221)
    a.in0 = ws.u; a.in0_planes = 8; a.epilogue = BIN_EPI_FINAL; a.fr = fr;
    BIN_TRY(launch_conv(a, s));
  }
  return BIN_OK;
}

// ------------------------------------------------------------------ backward of one backbone
// Data gradients reuse conv_igemm_kernel: for a stride-1 / pad k/2 conv, dX = conv(dY, V) with
// V[ci][co][ky][kx] = W[co][ci][k-1-ky][k-1-kx] (packed by launch_pack_weight_t, Cout' padded to a
// multiple of 96 and clipped by store_planes).  Gradients are fp16 P8 tensors scaled by *scale (loss
// scaling, a device scalar) and un-scaled when they leave the backbone (frame grads, dW, db).
int launch_pack_weight_t(const float* w, int cout, int cin, int ks, int row0, int nrows, int cout_pad_t, int cin_pad_t,
                         void* packed, cudaStream_t s);
int launch_p8_add(const bin_act_t& dst, int dplane0, const bin_act_t& src, int splane0, int nplanes, cudaStream_t s);
int launch_relu_mask(const bin_act_t& dg, int dplane0, const bin_act_t& g, int gplane0, int nplanes, cudaStream_t s);
int launch_pixel_unshuffle(const bin_act_t& du, const bin_act_t& dst, cudaStream_t s);
int launch_unpack_frames_grad(const bin_act_t& dx0, const bin_frames_t& dout, const bin_frames_t& dfr, int H, int W,
                              const float* scale, cudaStream_t s);
int launch_grad_out_to_p8(const bin_frames_t& dout, int H, int W, const bin_act_t& dst, const float* scale, cudaStream_t s);
int launch_bias_grad(const bin_act_t& dy, int plane0, int C, const float* scale, float* db, cudaStream_t s);
int launch_wgrad(const bin_act_t& x0, int x0_plane0, int x0_planes, const bin_act_t& x1, int x1_plane0, int x1_planes,
                 const bin_act_t& dy, int dy_plane0, int cout, int cin, int ks, const float* scale, float* dw,
                 float* partial_ws, cudaStream_t s);
static size_t wgrad_partial_bytes() { return (size_t)num_sms() * 128 * 512 * sizeof(float); }   // per-CTA accumulator slabs (grid = #SMs)

struct TSpec {          // one data-gradient conv: output rows [row0,row0+nrows) of the forward conv's Cin axis
  int conv, row0, nrows, cout_pad_t, cin_pad_t, ks;
  size_t off;
};
struct BackboneLayoutT {
  TSpec x[BIN_BACKBONE_NCONV];      // x part / whole input
  TSpec g[BIN_BACKBONE_NCONV];      // growth part (RDB convs c>=1 and LFF); nrows = 0 if absent
  size_t zero_bias_off, bytes;
};
static BackboneLayoutT backbone_layout_t(int nframes) {
  const BackboneLayout L = backbone_layout(nframes);
  BackboneLayoutT T;
  size_t off = 0;
  auto mk = [&](int conv, int row0, int nrows) {
    TSpec t;
    t.conv = conv; t.row0 = row0; t.nrows = nrows; t.ks = L.conv[conv].ks;
    t.cout_pad_t = nrows > 0 ? (int)align_up(nrows, 96) : 0;
    t.cin_pad_t = (int)align_up(L.conv[conv].cout, kKC);
    t.off = off;
    if (nrows > 0) off = align_up(off + (size_t)t.cout_pad_t * t.cin_pad_t * t.ks * t.ks * sizeof(__half), 256);
    return t;
  };
  for (int i = 0; i < BIN_BACKBONE_NCONV; ++i) {
    const ConvSpec& c = L.conv[i];
    const bool in_rdb = i >= 2 && i < 2 + kD * (kCgrow + 1);
    if (in_rdb) {
      T.x[i] = mk(i, 0, kG0);
      T.g[i] = mk(i, kG0, c.cin - kG0);          // 0 rows for conv 0 of each RDB
    } else {
      T.x[i] = mk(i, 0, c.cin);
      T.g[i] = mk(i, 0, 0);
    }
  }
  T.zero_bias_off = off;
  off = align_up(off + 1152 * sizeof(float), 256);
  T.bytes = off;
  return T;
}

struct GradWs {
  bin_act_t dout16, du, dup0, dt2, dt1, dcat, df2, dg, dx0;
  float* wg_partial;
  size_t bytes;
};
static GradWs grad_ws(int nframes, int Btot, int H, int W, void* base) {
  GradWs w;
  const int h = H / 2, wd = W / 2;
  size_t off = 0;
  auto carve = [&](int planes, int hh, int ww) {
    bin_act_t t;
    t.ptr = base ? (void*)((uint8_t*)base + off) : nullptr;
    t.B = Btot; t.planes = planes; t.H = hh; t.W = ww;
    off = align_up(off + (size_t)Btot * planes * hh * ww * 16, 256);
    return t;
  };
  w.dout16 = carve(4, H, W);
  w.du = carve(8, H, W);
  w.dup0 = carve(32, h, wd);
  w.dt2 = carve(12, h, wd);
  w.dt1 = carve(12, h, wd);
  w.dcat = carve(12 * kD, h, wd);
  w.df2 = carve(12, h, wd);
  w.dg = carve(16, h, wd);
  w.dx0 = carve((int)align_up(12 * nframes, kKC) / 8, h, wd);
  w.wg_partial = base ? (float*)((uint8_t*)base + off) : nullptr;
  off = align_up(off + wgrad_partial_bytes(), 256);
  w.bytes = off;
  return w;
}

struct GradParamLayout { size_t w[BIN_BACKBONE_NCONV], b[BIN_BACKBONE_NCONV], floats; };
static GradParamLayout grad_param_layout(int nframes) {
  const BackboneLayout L = backbone_layout(nframes);
  GradParamLayout g;
  size_t off = 0;
  for (int i = 0; i < BIN_BACKBONE_NCONV; ++i) {
    g.w[i] = off; off += (size_t)L.conv[i].cout * L.conv[i].cin * L.conv[i].ks * L.conv[i].ks;
    g.b[i] = off; off += (size_t)L.conv[i].cout;
  }
  g.floats = off;
  return g;
}

static int run_backbone_bwd(int nframes, const void* blob_t, const bin_frames_t& dout, const bin_frames_t& dfr, int H,
                            int W, const void* save_ws, void* gws_ptr, size_t gws_bytes, float* gparams,
                            const float* scale, cudaStream_t s) {
  if (!valid_nframes(nframes) || dfr.nframes != nframes) return fail(BIN_ERR_ARG, "backbone_bwd: nframes must be 2, 3 or 5");
  if (dout.ncalls != dfr.ncalls || dout.Bc != dfr.Bc || dout.ncalls < 1 || dout.ncalls > BIN_MAX_CALLS)
    return fail(BIN_ERR_ARG, "backbone_bwd: bad call tables");
  const int Btot = dout.ncalls * dout.Bc;
  const BackboneLayout L = backbone_layout(nframes);
  const BackboneLayoutT T = backbone_layout_t(nframes);
  const GradParamLayout GP = grad_param_layout(nframes);
  const BackboneWs ws = backbone_ws(nframes, Btot, H, W, const_cast<void*>(save_ws), true);
  const GradWs gw = grad_ws(nframes, Btot, H, W, gws_ptr);
  if (gw.bytes > gws_bytes) return fail(BIN_ERR_WORKSPACE, "backbone_bwd: gradient workspace too small");
  const float* zero_bias = (const float*)((const uint8_t*)blob_t + T.zero_bias_off);

  // dX (+)= conv(dY planes [dy_plane0, +dy_planes), V): writes `nstore` planes of `out` at out_plane0
  auto dgrad = [&](const TSpec& t, const bin_act_t& dy, int dy_plane0, int dy_planes, const bin_act_t& out, int out_plane0,
                   int nstore, bool accumulate) -> int {
    bin_conv_args_t a;
    memset(&a, 0, sizeof(a));
    a.in0 = dy; a.in0_plane0 = dy_plane0; a.in0_planes = dy_planes;
    a.w_packed = (const uint8_t*)blob_t + t.off; a.bias = zero_bias;
    a.ksize = t.ks; a.cout_pad = t.cout_pad_t; a.epilogue = BIN_EPI_P8;
    a.out = out; a.out_plane0 = out_plane0; a.store_planes = nstore;
    if (accumulate) { a.res = out; a.res_plane0 = out_plane0; }
    return launch_conv(a, s);
  };
  // dW += X^T dY, db += sum dY for forward conv `idx`
  auto wgrad = [&](int idx, const bin_act_t& x0, int x0p, int x0n, const bin_act_t& x1, int x1p, int x1n,
                   const bin_act_t& dy, int dyp) -> int {
    const ConvSpec& c = L.conv[idx];
    BIN_TRY(launch_bias_grad(dy, dyp, c.cout, scale, gparams + GP.b[idx], s));
    return launch_wgrad(x0, x0p, x0n, x1, x1p, x1n, dy, dyp, c.cout, c.cin, c.ks, scale, gparams + GP.w[idx], gw.wg_partial, s);
  };
  const bin_act_t none = {nullptr, 0, 0, 0, 0};

  BIN_TRY(launch_grad_out_to_p8(dout, H, W, gw.dout16, scale, s));
  BIN_TRY(wgrad(65, ws.u, 0, 8, none, 0, 0, gw.dout16, 0));                          // UPNet.2
  BIN_TRY(dgrad(T.x[65], gw.dout16, 0, 4, gw.du, 0, 8, false));
  BIN_TRY(launch_pixel_unshuffle(gw.du, gw.dup0, s));                               // nn.PixelShuffle backward
  BIN_TRY(wgrad(64, ws.t2, 0, 12, none, 0, 0, gw.dup0, 0));                          // UPNet.0
  BIN_TRY(dgrad(T.x[64], gw.dup0, 0, 32, gw.dt2, 0, 12, false));
  BIN_TRY(wgrad(63, ws.t1, 0, 12, none, 0, 0, gw.dt2, 0));                           // GFF.1
  BIN_TRY(dgrad(T.x[63], gw.dt2, 0, 12, gw.dt1, 0, 12, false));                      // dt2 doubles as d f__1 (RDN.py:219)
  BIN_TRY(wgrad(62, ws.cat, 0, 12 * kD, none, 0, 0, gw.dt1, 0));                     // GFF.0
  BIN_TRY(dgrad(T.x[62], gw.dt1, 0, 12, gw.dcat, 0, 12 * kD, false));
  BIN_CUDA_OK(cudaMemsetAsync(gw.df2.ptr, 0, (size_t)Btot * 12 * (H / 2) * (W / 2) * 16, s));
  for (int i = kD - 1; i >= 0; --i) {
    const int base = 2 + i * (kCgrow + 1);
    const bin_act_t& xin = i == 0 ? ws.f2 : ws.cat;           // forward input of RDB i
    const int xin_p = i == 0 ? 0 : 12 * (i - 1);
    const bin_act_t& dxin = i == 0 ? gw.df2 : gw.dcat;        // its gradient (accumulated)
    const int dxin_p = i == 0 ? 0 : 12 * (i - 1);
    const int dxo_p = 12 * i;                                 // d x_{i+1}, complete at this point
    BIN_TRY(wgrad(base + kCgrow, xin, xin_p, 12, ws.g, 16 * i, 16, gw.dcat, dxo_p));                 // LFF
    BIN_TRY(launch_p8_add(dxin, dxin_p, gw.dcat, dxo_p, 12, s));                                      // residual (RDN.py:165)
    BIN_TRY(dgrad(T.x[base + kCgrow], gw.dcat, dxo_p, 12, dxin, dxin_p, 12, true));
    BIN_TRY(dgrad(T.g[base + kCgrow], gw.dcat, dxo_p, 12, gw.dg, 0, 16, false));
    for (int c = kCgrow - 1; c >= 0; --c) {
      BIN_TRY(launch_relu_mask(gw.dg, 4 * c, ws.g, 16 * i + 4 * c, 4, s));                            // RDN.py:142
      BIN_TRY(wgrad(base + c, xin, xin_p, 12, ws.g, 16 * i, 4 * c, gw.dg, 4 * c));
      BIN_TRY(dgrad(T.x[base + c], gw.dg, 4 * c, 4, dxin, dxin_p, 12, true));
      if (c > 0) BIN_TRY(dgrad(T.g[base + c], gw.dg, 4 * c, 4, gw.dg, 0, 4 * c, true));
    }
  }
  BIN_TRY(wgrad(1, ws.f1, 0, 12, none, 0, 0, gw.df2, 0));                            // SFENet2
  BIN_TRY(dgrad(T.x[1], gw.df2, 0, 12, gw.dt2, 0, 12, true));                        // d f__1 complete
  BIN_TRY(wgrad(0, ws.x0, 0, ws.x0.planes, none, 0, 0, gw.dt2, 0));                  // SFENet1
  BIN_TRY(dgrad(T.x[0], gw.dt2, 0, 12, gw.dx0, 0, gw.dx0.planes, false));
  return launch_unpack_frames_grad(gw.dx0, dout, dfr, H, W, scale, s);
}

// ------------------------------------------------------------------ window orchestration
struct Call {
  const float* in[BIN_MAX_FRAMES];
  float* out;
};
static int run_stage(const bin_net_t* net, int which, int nframes, const std::vector<Call>& calls, int B, int H, int W,
                     void* ws, size_t ws_bytes, cudaStream_t s, int x3 = 0) {
  bin_frames_t fr;
  memset(&fr, 0, sizeof(fr));
  fr.ncalls = (int)calls.size(); fr.nframes = nframes; fr.Bc = B;
  for (int k = 0; k < fr.ncalls; ++k) {
    for (int f = 0; f < nframes; ++f) fr.frame[k][f] = calls[k].in[f];
    fr.out[k] = calls[k].out;
  }
  return run_backbone(nframes, net->blob[which], fr, H, W, ws, ws_bytes, s, false, x3);
}

static size_t window_ws_bytes(int B, int H, int W, int max_calls, int ntemp, int x3 = 0) {
  size_t bb = 0;
  const int nf[3] = {2, 3, 5};
  for (int i = 0; i < 3; ++i) {
    size_t v = backbone_ws(nf[i], max_calls * B, H, W, nullptr, false, x3).bytes;
    bb = v > bb ? v : bb;
  }
  return bb + (size_t)ntemp * align_up((size_t)B * 3 * H * W * sizeof(float), 256);
}

}  // namespace binb

using namespace binb;

extern "C" {

int bin_abi_version(void) { return BIN_ABI_VERSION; }
const char* bin_last_error(void) { return g_err.c_str(); }

int bin_check_device(void) {
  int dev = 0;
  BIN_CUDA_OK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  BIN_CUDA_OK(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(BIN_ERR_UNSUPPORTED, std::string("bin_b200 needs an sm_100 device, found sm_") +
                                                          std::to_string(prop.major) + std::to_string(prop.minor));
  return BIN_OK;
}

int bin_nchw_to_p8(const float* x, int C, bin_act_t dst, int plane0, bin_stream_t s) {
  return launch_nchw_to_p8(x, C, dst, plane0, (cudaStream_t)s);
}
int bin_p8_to_nchw(bin_act_t src, int plane0, int C, float* y, bin_stream_t s) {
  return launch_p8_to_nchw(src, plane0, C, y, (cudaStream_t)s);
}
int bin_pack_frames(const bin_frames_t* fr, int H, int W, bin_act_t dst, bin_stream_t s) {
  if (!fr) return fail(BIN_ERR_ARG, "pack_frames: null frame table");
  return launch_pack_frames(*fr, H, W, dst, (cudaStream_t)s);
}
size_t bin_packed_weight_bytes(int cout_pad, int cin_pad, int ksize) {
  return (size_t)cout_pad * cin_pad * ksize * ksize * sizeof(__half);
}
int bin_pack_conv_weight(const float* w_oihw, int cout, int cin, int ksize, int cout_pad, int cin_pad, int variant,
                         void* packed, bin_stream_t s) {
  return launch_pack_weight(w_oihw, cout, cin, ksize, cout_pad, cin_pad, variant, packed, (cudaStream_t)s);
}
int bin_pack_conv_weight_t(const float* w_oihw, int cout, int cin, int ksize, int row0, int nrows, int cout_pad_t,
                           int cin_pad_t, void* packed, bin_stream_t s) {
  return launch_pack_weight_t(w_oihw, cout, cin, ksize, row0, nrows, cout_pad_t, cin_pad_t, packed, (cudaStream_t)s);
}
size_t bin_conv_wgrad_workspace_bytes(void) { return wgrad_partial_bytes(); }
int bin_conv_wgrad(bin_act_t x0, int x0_plane0, int x0_planes, bin_act_t x1, int x1_plane0, int x1_planes, bin_act_t dy,
                   int dy_plane0, int cout, int cin, int ksize, const float* scale_dev, float* dw, void* workspace,
                   bin_stream_t s) {
  return launch_wgrad(x0, x0_plane0, x0_planes, x1, x1_plane0, x1_planes, dy, dy_plane0, cout, cin, ksize, scale_dev, dw,
                      (float*)workspace, (cudaStream_t)s);
}
int bin_conv_fwd(const bin_conv_args_t* a, bin_stream_t s) {
  if (!a) return fail(BIN_ERR_ARG, "conv: null args");
  return launch_conv(*a, (cudaStream_t)s);
}
int bin_convlstm_fwd(const float* x, const float* c_prev, const float* h_prev, const float* w, const float* b,
                     float* h_out, float* c_out, int B, int H, int W, bin_stream_t s) {
  return launch_convlstm(x, c_prev, h_prev, w, b, h_out, c_out, B, H, W, (cudaStream_t)s);
}

int bin_pixel_loss_fwd(const float* const* a_host, const float* const* b_host, int npairs, size_t n, int kind, float eps,
                       float* pair_loss, bin_stream_t s) {
  if (!a_host || !b_host || !pair_loss) return fail(BIN_ERR_ARG, "pixel_loss_fwd: null argument");
  return launch_pixel_loss_fwd(a_host, b_host, npairs, n, kind, eps, pair_loss, (cudaStream_t)s);
}
int bin_pixel_loss_bwd(const float* const* a_host, const float* const* b_host, float* const* da_host, float* const* db_host,
                       int npairs, size_t n, int kind, float eps, const float* upstream, bin_stream_t s) {
  if (!a_host || !b_host || !da_host || !upstream) return fail(BIN_ERR_ARG, "pixel_loss_bwd: null argument");
  return launch_pixel_loss_bwd(a_host, b_host, da_host, db_host, npairs, n, kind, eps, upstream, (cudaStream_t)s);
}
int bin_tensor2img_u8(const float* x, int Hs, int Ws, int top, int left, int h, int w, uint8_t* out, bin_stream_t s) {
  if (!x || !out) return fail(BIN_ERR_ARG, "tensor2img: null argument");
  return launch_tensor2img_u8(x, Hs, Ws, top, left, h, w, out, (cudaStream_t)s);
}
int bin_u8_to_frame(const uint8_t* img, int h, int w, int pad_l, int pad_r, int pad_t, int pad_b, float* out, bin_stream_t s) {
  if (!img || !out) return fail(BIN_ERR_ARG, "u8_to_frame: null argument");
  return launch_u8_to_frame(img, h, w, pad_l, pad_r, pad_t, pad_b, out, (cudaStream_t)s);
}
int bin_convlstm_bwd(const float* x, const float* c_prev, const float* h_prev, const float* w, const float* b,
                     const float* dh, const float* dc, float* dgates_ws, float* dx, float* dc_prev, float* dh_prev,
                     float* dw, float* db, int B, int H, int W, bin_stream_t s) {
  if (!x || !w || !b || !dgates_ws || !dx || !dw || !db) return fail(BIN_ERR_ARG, "convlstm_bwd: null argument");
  return launch_convlstm_bwd(x, c_prev, h_prev, w, b, dh, dc, dgates_ws, dx, dc_prev, dh_prev, dw, db, B, H, W, (cudaStream_t)s);
}

size_t bin_backbone_packed_bytes(int nframes) { return valid_nframes(nframes) ? backbone_layout(nframes).bytes : 0; }

// all 66 weights + 66 biases of a backbone in ONE launch
static int pack_backbone(int nframes, const float* const* w_host, const float* const* b_host, void* blob, int x3,
                         cudaStream_t s) {
  if (!w_host || !b_host || !blob) return fail(BIN_ERR_ARG, "backbone_pack: null argument");
  const BackboneLayout L = backbone_layout(nframes, x3);
  void* hb = pack_batch_new();
  int rc = BIN_OK;
  for (int i = 0; i < BIN_BACKBONE_NCONV && rc == BIN_OK; ++i) {
    const ConvSpec& c = L.conv[i];
    rc = pack_batch_add_weight(hb, w_host[i], c.cout, c.cin, c.ks, c.cout_pad, c.cin_pad, BIN_CONV_DEFAULT,
                               (uint8_t*)blob + c.w_off, x3);
    if (rc == BIN_OK) rc = pack_batch_add_bias(hb, b_host[i], c.cout, c.cout_pad, (float*)((uint8_t*)blob + c.b_off));
  }
  const int rl = pack_batch_launch(hb, s);      // always frees the batch
  return rc != BIN_OK ? rc : rl;
}

int bin_backbone_pack(int nframes, const float* const* w_host, const float* const* b_host, void* blob,
                      bin_stream_t s) {
  if (!valid_nframes(nframes)) return fail(BIN_ERR_ARG, "backbone_pack: nframes must be 2, 3 or 5");
  return pack_backbone(nframes, w_host, b_host, blob, 0, (cudaStream_t)s);
}

size_t bin_backbone_workspace_bytes(int nframes, int Btot, int H, int W) {
  return valid_nframes(nframes) ? backbone_ws(nframes, Btot, H, W, nullptr).bytes : 0;
}

int bin_backbone_fwd(int nframes, const void* blob, const bin_frames_t* fr, int H, int W, void* workspace,
                     size_t workspace_bytes, bin_stream_t s) {
  if (!fr || !blob) return fail(BIN_ERR_ARG, "backbone_fwd: null argument");
  return run_backbone(nframes, blob, *fr, H, W, workspace, workspace_bytes, (cudaStream_t)s);
}

size_t bin_backbone_packed_t_bytes(int nframes) { return valid_nframes(nframes) ? backbone_layout_t(nframes).bytes : 0; }

int bin_backbone_pack_t(int nframes, const float* const* w_host, void* blob_t, bin_stream_t s) {
  if (!valid_nframes(nframes)) return fail(BIN_ERR_ARG, "backbone_pack_t: nframes must be 2, 3 or 5");
  const BackboneLayout L = backbone_layout(nframes);
  const BackboneLayoutT T = backbone_layout_t(nframes);
  void* hb = pack_batch_new();
  int rc = BIN_OK;
  for (int i = 0; i < BIN_BACKBONE_NCONV && rc == BIN_OK; ++i) {
    const ConvSpec& c = L.conv[i];
    const TSpec* parts[2] = {&T.x[i], &T.g[i]};
    for (const TSpec* t : parts) {
      if (t->nrows <= 0 || rc != BIN_OK) continue;
      rc = pack_batch_add_weight_t(hb, w_host[i], c.cout, c.cin, c.ks, t->row0, t->nrows, t->cout_pad_t, t->cin_pad_t,
                                   (uint8_t*)blob_t + t->off);
    }
  }
  const int rl = pack_batch_launch(hb, (cudaStream_t)s);
  if (rc != BIN_OK) return rc;
  BIN_TRY(rl);
  BIN_CUDA_OK(cudaMemsetAsync((uint8_t*)blob_t + T.zero_bias_off, 0, 1152 * sizeof(float), (cudaStream_t)s));
  return BIN_OK;
}

size_t bin_backbone_train_workspace_bytes(int nframes, int Btot, int H, int W) {
  return valid_nframes(nframes) ? backbone_ws(nframes, Btot, H, W, nullptr, true).bytes : 0;
}
int bin_backbone_fwd_train(int nframes, const void* blob, const bin_frames_t* fr, int H, int W, void* save_ws,
                           size_t save_ws_bytes, bin_stream_t s) {
  if (!fr || !blob) return fail(BIN_ERR_ARG, "backbone_fwd_train: null argument");
  return run_backbone(nframes, blob, *fr, H, W, save_ws, save_ws_bytes, (cudaStream_t)s, true);
}
size_t bin_backbone_grad_workspace_bytes(int nframes, int Btot, int H, int W) {
  return valid_nframes(nframes) ? grad_ws(nframes, Btot, H, W, nullptr).bytes : 0;
}
size_t bin_backbone_grad_param_floats(int nframes) { return valid_nframes(nframes) ? grad_param_layout(nframes).floats : 0; }
int bin_backbone_bwd(int nframes, const void* blob_t, const bin_frames_t* dout, const bin_frames_t* dframes, int H, int W,
                     const void* save_ws, void* grad_ws_ptr, size_t grad_ws_bytes, float* grad_params,
                     const float* scale_dev, bin_stream_t s) {
  if (!blob_t || !dout || !dframes || !save_ws || !grad_params || !scale_dev)
    return fail(BIN_ERR_ARG, "backbone_bwd: null argument");
  return run_backbone_bwd(nframes, blob_t, *dout, *dframes, H, W, save_ws, grad_ws_ptr, grad_ws_bytes, grad_params,
                          scale_dev, (cudaStream_t)s);
}

int bin_grad_scale(const float* const* gouts_host, int n, size_t numel, float target, float* scale_dev, void* tmp4_dev,
                   bin_stream_t s) {
  if (!gouts_host || !scale_dev || !tmp4_dev) return fail(BIN_ERR_ARG, "grad_scale: null argument");
  return launch_grad_scale(gouts_host, n, numel, target, scale_dev, (unsigned*)tmp4_dev, (cudaStream_t)s);
}

int bin_rdb_fwd(const void* blob, int nframes, int index, const float* x, float* y, int B, int h, int w,
                void* workspace, size_t workspace_bytes, bin_stream_t s) {
  if (!valid_nframes(nframes) || index < 0 || index >= kD) return fail(BIN_ERR_ARG, "rdb_fwd: bad nframes/index");
  const BackboneLayout L = backbone_layout(nframes);
  size_t off = 0;
  auto carve = [&](int planes) {
    bin_act_t t;
    t.ptr = (uint8_t*)workspace + off; t.B = B; t.planes = planes; t.H = h; t.W = w;
    off = align_up(off + (size_t)B * planes * h * w * 16, 256);
    return t;
  };
  bin_act_t xin = carve(12), g = carve(16), out = carve(12);
  if (off > workspace_bytes) return fail(BIN_ERR_WORKSPACE, "rdb_fwd: workspace too small");
  BIN_TRY(launch_nchw_to_p8(x, kG0, xin, 0, (cudaStream_t)s));
  BIN_TRY(run_rdb(blob, L, index, xin, 0, g, out, 0, plan_bands(B, h, w), (cudaStream_t)s));
  return launch_p8_to_nchw(out, 0, kG0, y, (cudaStream_t)s);
}

static int window_fwd_impl(const bin_net_t* net, const float* const* F, float* const* o, int B, int H, int W, void* workspace,
                           size_t workspace_bytes, bin_stream_t s_, int x3) {
  if (!net || !F || !o) return fail(BIN_ERR_ARG, "window_fwd: null argument");
  cudaStream_t s = (cudaStream_t)s_;
  const size_t need = window_ws_bytes(B, H, W, BIN_MAX_CALLS, 9, x3);
  if (workspace_bytes < need) return fail(BIN_ERR_WORKSPACE, "window_fwd: workspace too small");
  const size_t fbytes = align_up((size_t)B * 3 * H * W * sizeof(float), 256);
  uint8_t* base = (uint8_t*)workspace;
  float* tmp[9];
  for (int i = 0; i < 9; ++i) tmp[i] = (float*)(base + i * fbytes);
  void* bws = base + 9 * fbytes;
  const size_t bws_bytes = workspace_bytes - 9 * fbytes;
  float *p4 = tmp[0], *p6 = tmp[1], *p8 = tmp[2], *p5 = tmp[3], *p7 = tmp[4], *p6b = tmp[5];
  float *t0 = tmp[6], *t1 = tmp[7], *t2 = tmp[8];
  // the cells of one recurrent hand-off are independent: one launch for all of them (grid.z = cell)
  auto lstm = [&](int k0, int n, std::initializer_list<const float*> xs, std::initializer_list<float*> hs) {
    LstmCells c;
    memset(&c, 0, sizeof(c));
    int i = 0;
    for (const float* x : xs) c.x[i++] = x;
    i = 0;
    for (float* h : hs) c.h_out[i++] = h;
    for (i = 0; i < n; ++i) { c.w[i] = net->lstm_w[k0 + i]; c.b[i] = net->lstm_b[k0 + i]; }
    return launch_convlstm_multi(c, n, B, H, W, s);
  };
  // Stage 1 (RDN.py:371-374): 4 calls of step 0 + the one stage-1 call of step 1 that is not a repeat.
  BIN_TRY(run_stage(net, 0, 2, {{{F[0], F[1]}, o[0]}, {{F[1], F[2]}, o[1]}, {{F[2], F[3]}, o[2]},
                               {{F[3], F[4]}, o[3]}, {{F[4], F[5]}, o[10]}}, B, H, W, bws, bws_bytes, s, x3));
  // recurrent hand-off for the stage-1 outputs (RDN.py:451-453)
  BIN_TRY(lstm(0, 3, {o[1], o[2], o[3]}, {p4, p6, p8}));
  // Stage 2: step 0 (RDN.py:384-386, "prev" slot duplicated) + step 1 (RDN.py:377-379) in ONE launch of 6 calls:
  // the step-1 calls only need stage-1 outputs and their ConvLSTM images, not step-0's stage 2.
  BIN_TRY(run_stage(net, 1, 3, {{{o[0], o[0], o[1]}, o[4]}, {{o[1], o[1], o[2]}, o[5]}, {{o[2], o[2], o[3]}, o[6]},
                               {{p4, o[1], o[2]}, t0}, {{p6, o[2], o[3]}, t1}, {{p8, o[3], o[10]}, o[11]}},
                    B, H, W, bws, bws_bytes, s, x3));
  BIN_TRY(lstm(3, 2, {o[5], o[6]}, {p5, p7}));                                    // RDN.py:454-455
  // Stage 3: step 0 (RDN.py:387-388) + step 1 (RDN.py:380-381)
  BIN_TRY(run_stage(net, 2, 5, {{{o[4], F[1], o[4], o[5], F[2]}, o[7]}, {{o[5], F[2], o[5], o[6], F[3]}, o[8]},
                               {{p5, F[2], t0, t1, F[3]}, t2}, {{p7, F[3], t1, o[11], F[4]}, o[12]}},
                    B, H, W, bws, bws_bytes, s, x3));
  BIN_TRY(lstm(5, 1, {o[8]}, {p6b}));                                             // RDN.py:456
  // Stage 4: step 0 (RDN.py:389) + step 1 (RDN.py:382)
  BIN_TRY(run_stage(net, 3, 5, {{{o[1], o[1], o[7], o[8], o[2]}, o[9]}, {{p6b, o[2], t2, o[12], o[3]}, o[13]}},
                    B, H, W, bws, bws_bytes, s, x3));
  return BIN_OK;
}

size_t bin_window_workspace_bytes(int B, int H, int W) { return window_ws_bytes(B, H, W, BIN_MAX_CALLS, 9); }
int bin_window_fwd(const bin_net_t* net, const float* const* F, float* const* o, int B, int H, int W, void* workspace,
                   size_t workspace_bytes, bin_stream_t s) {
  return window_fwd_impl(net, F, o, B, H, W, workspace, workspace_bytes, s, 0);
}
/* precision-parameterised twins (BIN_PREC_*) */
size_t bin_window_workspace_bytes_p(int B, int H, int W, int prec) { return window_ws_bytes(B, H, W, BIN_MAX_CALLS, 9, prec ? 1 : 0); }
int bin_window_fwd_p(const bin_net_t* net, const float* const* F, float* const* o, int B, int H, int W, void* workspace,
                     size_t workspace_bytes, int prec, bin_stream_t s) {
  return window_fwd_impl(net, F, o, B, H, W, workspace, workspace_bytes, s, prec ? 1 : 0);
}
size_t bin_backbone_packed_bytes_p(int nframes, int prec) { return valid_nframes(nframes) ? backbone_layout(nframes, prec ? 1 : 0).bytes : 0; }
int bin_backbone_pack_p(int nframes, const float* const* w_host, const float* const* b_host, void* blob, int prec,
                        bin_stream_t s) {
  if (!valid_nframes(nframes)) return fail(BIN_ERR_ARG, "backbone_pack: nframes must be 2, 3 or 5");
  return pack_backbone(nframes, w_host, b_host, blob, prec ? 1 : 0, (cudaStream_t)s);
}
size_t bin_backbone_workspace_bytes_p(int nframes, int Btot, int H, int W, int prec) {
  return valid_nframes(nframes) ? backbone_ws(nframes, Btot, H, W, nullptr, false, prec ? 1 : 0).bytes : 0;
}
int bin_backbone_fwd_p(int nframes, const void* blob, const bin_frames_t* fr, int H, int W, void* workspace,
                       size_t workspace_bytes, int prec, bin_stream_t s) {
  if (!fr || !blob) return fail(BIN_ERR_ARG, "backbone_fwd: null argument");
  return run_backbone(nframes, blob, *fr, H, W, workspace, workspace_bytes, (cudaStream_t)s, false, prec ? 1 : 0);
}

int bin_pyramid3_fwd(const bin_net_t* net, const float* const* F, float* const* o, int B, int H, int W,
                     void* workspace, size_t workspace_bytes, bin_stream_t s_) {
  if (!net || !F || !o) return fail(BIN_ERR_ARG, "pyramid3_fwd: null argument");
  cudaStream_t s = (cudaStream_t)s_;
  if (workspace_bytes < window_ws_bytes(B, H, W, BIN_MAX_CALLS, 9)) return fail(BIN_ERR_WORKSPACE, "pyramid3_fwd: workspace too small");
  BIN_TRY(run_stage(net, 0, 2, {{{F[0], F[1]}, o[0]}, {{F[1], F[2]}, o[1]}, {{F[2], F[3]}, o[2]}}, B, H, W, workspace,
                    workspace_bytes, s));
  BIN_TRY(run_stage(net, 1, 3, {{{o[0], o[0], o[1]}, o[3]}, {{o[1], o[1], o[2]}, o[4]}}, B, H, W, workspace,
                    workspace_bytes, s));
  return run_stage(net, 2, 5, {{{o[3], F[1], o[3], o[4], F[2]}, o[5]}}, B, H, W, workspace, workspace_bytes, s);
}

int bin_rdb_tail_fwd(const bin_act_t* x, int x_plane0, const bin_act_t* g, int g_plane0, const void* w_conv,
                     const float* b_conv, const void* w_lff, const float* b_lff, const bin_act_t* out, int out_plane0,
                     int b_begin, int b_count, int y_begin, int y_count, bin_stream_t s) {
  if (!x || !g || !out || !x->ptr || !g->ptr || !out->ptr || !w_conv || !b_conv || !w_lff || !b_lff)
    return fail(BIN_ERR_ARG, "rdb_tail_fwd: null argument");
  return launch_rdb_tail(*x, x_plane0, *g, g_plane0, w_conv, b_conv, w_lff, b_lff, *out, out_plane0, b_begin, b_count,
                         y_begin, y_count, (cudaStream_t)s);
}
int bin_adam_step(const bin_adam_tensor_t* table_dev, const int* chunk_prefix_dev, int ntensors, int nchunks, float lr,
                  float beta1, float beta2, float eps, float weight_decay, float bias_correction1,
                  float bias_correction2, float grad_scale, bin_stream_t s) {
  if (!table_dev || !chunk_prefix_dev) return fail(BIN_ERR_ARG, "adam_step: null argument");
  return launch_adam_step(table_dev, chunk_prefix_dev, ntensors, nchunks, lr, beta1, beta2, eps, weight_decay,
                          bias_correction1, bias_correction2, grad_scale, (cudaStream_t)s);
}
int bin_blur_average_u8(const uint8_t* frames, int T, size_t frame_bytes, int window_size, int first_mid, int stride,
                        int nwin, uint8_t* out, bin_stream_t s) {
  if (!frames || !out) return fail(BIN_ERR_ARG, "blur_average: null argument");
  return launch_blur_average_u8(frames, T, frame_bytes, window_size, first_mid, stride, nwin, out, (cudaStream_t)s);
}
size_t bin_image_metrics_workspace_bytes(int npairs, int h, int w, int c, int kind) {
  return image_metrics_workspace_bytes(npairs, h, w, c, kind);
}
int bin_image_metrics_u8(const uint8_t* const* a_host, const uint8_t* const* b_host, int npairs, int h, int w, int c,
                         int kind, double* res, void* ws, size_t ws_bytes, bin_stream_t s) {
  if (!a_host || !b_host || !res || !ws) return fail(BIN_ERR_ARG, "image_metrics: null argument");
  return launch_image_metrics_u8(a_host, b_host, npairs, h, w, c, kind, res, ws, ws_bytes, (cudaStream_t)s);
}
int bin_train_batch_u8(const bin_train_sample_t* samples, int B, int H, int W, int h, int w, float* lqs, float* gtenh,
                       float* gtinp, bin_stream_t s) {
  if (!samples || !lqs || !gtenh || !gtinp) return fail(BIN_ERR_ARG, "train_batch: null argument");
  return launch_train_batch_u8(samples, B, H, W, h, w, lqs, gtenh, gtinp, (cudaStream_t)s);
}

}  // extern "C"
