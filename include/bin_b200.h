/* bin_b200 -- C ABI of the B200-native BIN hot path (libbin_b200.so).
 *
 * The reference (laomao0/BIN) has no FFI layer: its boundary for this path is the Python
 * nn.Module contract reached through models/networks.py:9-10 -> models/archs/RDN.py:469-471
 * (SURVEY.md 8b).  This header is the "thin C-ABI extension" north_star asks for: every
 * entry point replaces one reference symbol (cited per function) and is called by the
 * Python mirror in bin_b200/rdn.py through ctypes.  Conventions:
 *   - all data pointers are DEVICE pointers unless the name ends in _host;
 *   - every call is asynchronous on the given CUDA stream (cudaStream_t passed as void*);
 *   - return 0 on success, non-zero error code otherwise; bin_last_error() gives the text
 *     (thread-local, valid until the next failing call on that thread);
 *   - no allocation inside: callers pass workspaces sized by the *_bytes() queries;
 *   - no global mutable state: re-entrant per (device, stream).
 *
 * Device layouts
 *   frames / outputs : fp32 NCHW, exactly what the reference module takes and returns.
 *   "planar-8" (P8)  : fp16 activations [B][C/8][H][W][8]  (8-channel planes; one pixel of one
 *                      plane = 16 B = one UMMA core-matrix row, so any pixel shift of a smem
 *                      tile is a 16-byte descriptor offset -> implicit GEMM without im2col).
 *   packed conv W    : fp16 [Cin_pad/32][kh][kw][4][Cout_pad][8]  (K-major B operand, one
 *                      contiguous slab per 32-channel K chunk), + fp32 bias[Cout_pad].
 *                      3x3 convs with Cout=32 (the RDB convs, 70 % of all FLOPs) use the
 *                      "x-stacked" layout [Cin_pad/32][kh][4][kw*32+cout][8]: the three horizontal
 *                      taps become GEMM columns (N=96) and are re-aligned in the epilogue.
 */
#ifndef BIN_B200_H_
#define BIN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BIN_ABI_VERSION 2
#define BIN_MAX_CALLS 6   /* same-weight backbone calls batched along N */
#define BIN_MAX_FRAMES 5  /* frames per backbone call (2, 3 or 5) */
#define BIN_MAX_LOSS_PAIRS 20 /* (prediction, target) pairs of one fused loss call */

enum { BIN_OK = 0, BIN_ERR_ARG = 1, BIN_ERR_CUDA = 2, BIN_ERR_UNSUPPORTED = 3, BIN_ERR_WORKSPACE = 4 };

typedef void* bin_stream_t; /* cudaStream_t */

int bin_abi_version(void);
const char* bin_last_error(void);
/* 0 if the current device is sm_100 (B200) and the driver exposes cuTensorMapEncodeTiled. */
int bin_check_device(void);

/* ---- P8 activation tensor view ------------------------------------------------------- */
typedef struct {
  void* ptr; /* fp16 [B][planes][H][W][8] */
  int B, planes, H, W;
} bin_act_t;

/* ---- frame pointer table (one row per batched backbone call) --------------------------- */
typedef struct {
  const float* frame[BIN_MAX_CALLS][BIN_MAX_FRAMES]; /* each (Bc,3,H,W) fp32 NCHW */
  float* out[BIN_MAX_CALLS];                          /* each (Bc,3,H,W) fp32 NCHW */
  int ncalls, nframes, Bc;
} bin_frames_t;

/* ---- layout helpers (tests, boundary) ----------------------------------------------- */
/* fp32 NCHW (B,C,H,W) -> P8 planes [plane0, plane0+ceil(C/8)); channels past C are zeroed. */
int bin_nchw_to_p8(const float* x, int C, bin_act_t dst, int plane0, bin_stream_t s);
/* P8 planes -> fp32 NCHW (B,C,H,W). */
int bin_p8_to_nchw(bin_act_t src, int plane0, int C, float* y, bin_stream_t s);

/* RDN.py:107-132 pixel_reshuffle(cat(frames),2) fused with the fp32->fp16 cast and channel
 * padding: dst is P8 (ncalls*Bc, cin_pad/8, H/2, W/2); channel (f*3+rgb)*4 + dy*2+dx. */
int bin_pack_frames(const bin_frames_t* fr, int H, int W, bin_act_t dst, bin_stream_t s);

/* ---- weights ------------------------------------------------------------------------- */
size_t bin_packed_weight_bytes(int cout_pad, int cin_pad, int ksize);
/* nn.Conv2d weight (cout,cin,k,k) fp32 OIHW -> packed fp16; rows/cols past cout/cin are zero. */
/* variant: BIN_CONV_DEFAULT, or BIN_CONV_PLAIN to force the un-stacked layout for 3x3/Cout=32. */
int bin_pack_conv_weight(const float* w_oihw, int cout, int cin, int ksize, int cout_pad, int cin_pad, int variant,
                         void* packed, bin_stream_t s);

/* ---- the implicit-GEMM convolution (tcgen05) ------------------------------------------ */
enum { BIN_EPI_P8 = 0, BIN_EPI_PIXSHUF = 1, BIN_EPI_FINAL = 2 };
enum { BIN_CONV_DEFAULT = 0, BIN_CONV_PLAIN = 1 };
/* Precision modes: fp16 storage / fp32 accumulate (<=1e-3 parity), or the split-fp16 "fp32-accurate" mode
 * (x = hi + lo, 3 MMAs per product, <=1e-5 parity; ~3x slower -- a correctness mode, not the benchmarked one). */
enum { BIN_PREC_F16 = 0, BIN_PREC_F32X3 = 1 };
typedef struct {
  /* input channels = planes [in0_plane0, +in0_planes) of in0 followed by planes of in1
   * (dense concat without a copy: RDN.py:147 torch.cat((x,out),1)); plane counts multiples of 4. */
  bin_act_t in0; int in0_plane0, in0_planes;
  bin_act_t in1; int in1_plane0, in1_planes; /* in1_planes = 0 -> unused */
  const void* w_packed; const float* bias;   /* bias: fp32[cout_pad] */
  int ksize;     /* 1, 3 or 5; stride 1, zero padding ksize/2 (all convs of RDN.py) */
  int cout_pad;  /* 16, 32, 256 or a multiple of 96 */
  int relu;      /* RDN.py:142 */
  int epilogue;  /* BIN_EPI_* */
  int variant;   /* BIN_CONV_*; must match the variant the weights were packed with */
  /* optional sub-range of the output: batch items [b_begin, b_begin+b_count) and rows
   * [y_begin, y_begin+y_count); counts of 0 mean "to the end".  Used to walk an RDB band by band
   * so that its intermediate tensors stay L2-resident. */
  int b_begin, b_count, y_begin, y_count;
  /* BIN_EPI_P8 only: number of output planes actually stored (0 = cout_pad/8); lets a conv whose Cout was
   * zero-padded up to a multiple of 96 (the data-gradient launches) write a narrower tensor. */
  int store_planes;
  /* 1 = fp32-accurate split mode: tensors carry (hi, lo) fp16 pairs -- per 32-channel chunk 4 planes of hi then
   * 4 planes of lo, so bin_act_t.planes is twice the logical plane count while every *_plane0 / *_planes field
   * stays LOGICAL (multiples of 4); weights must have been packed with BIN_PREC_F32X3. */
  int x3;
  /* BIN_EPI_P8: out planes [out_plane0, +cout_pad/8), optional residual (RDN.py:165, :219) */
  bin_act_t out; int out_plane0;
  bin_act_t res; int res_plane0; /* res.ptr = NULL -> none */
  /* BIN_EPI_PIXSHUF (RDN.py:206): cout_pad=256 -> out is P8 (B, 8 planes, 2H, 2W) */
  /* BIN_EPI_FINAL (RDN.py:207 + :221/:279/:333): cout_pad=16 (3 used); out = conv + bias +
   * mean(frames) written as fp32 NCHW to fr.out[call] */
  bin_frames_t fr;
} bin_conv_args_t;
int bin_conv_fwd(const bin_conv_args_t* a, bin_stream_t s);

/* Fused tail of one RDB (RDN.py:141-147 for the 4th RDB_Conv, :162-165): g3 = ReLU(conv3x3(cat(x, g0..g2))) and
 * out = LFF(cat(x, g0..g3)) + x in one kernel; g3 is never written.  x: 12 planes from x_plane0, g: the 12 planes of
 * g0..g2 from g_plane0, out: 12 planes from out_plane0 (may be other planes of x's tensor).  w_conv / w_lff are the
 * bin_pack_conv_weight outputs of the (32,192,3,3) conv (variant BIN_CONV_DEFAULT) and the (96,224,1,1) LFF; b_conv
 * has 32 floats, b_lff 96.  b/y sub-ranges as in the conv arguments: a count of 0 means "to the end".  fp16 mode only. */
int bin_rdb_tail_fwd(const bin_act_t* x, int x_plane0, const bin_act_t* g, int g_plane0, const void* w_conv,
                     const float* b_conv, const void* w_lff, const float* b_lff, const bin_act_t* out, int out_plane0,
                     int b_begin, int b_count, int y_begin, int y_count, bin_stream_t s);

/* Data-gradient weights of a conv (cout,cin,k): V[ci][co][ky][kx] = W[co][row0+ci][k-1-ky][k-1-kx] for ci < nrows,
 * packed like a forward conv with Cout' = cout_pad_t (multiple of 96), Cin' = cin_pad_t (multiple of 32):
 * bin_conv_fwd over dY with these weights gives dX[:, row0:row0+nrows]. */
int bin_pack_conv_weight_t(const float* w_oihw, int cout, int cin, int ksize, int row0, int nrows, int cout_pad_t,
                           int cin_pad_t, void* packed, bin_stream_t s);
/* Weight gradient of one conv: dw (cout,cin,k,k fp32 OIHW) += (1/ *scale_dev) * sum_px dY[px][co] X[px+tap][ci];
 * X = planes of x0 followed by planes of x1 (like bin_conv_args_t), dY = planes [dy_plane0, +ceil(cout/8)).
 * workspace: bin_conv_wgrad_workspace_bytes() bytes (per-CTA partial sums, reduced by a second kernel). */
size_t bin_conv_wgrad_workspace_bytes(void);
int bin_conv_wgrad(bin_act_t x0, int x0_plane0, int x0_planes, bin_act_t x1, int x1_plane0, int x1_planes, bin_act_t dy,
                   int dy_plane0, int cout, int cin, int ksize, const float* scale_dev, float* dw, void* workspace,
                   bin_stream_t s);

/* ---- ConvLSTMCell.forward, RDN.py:50-95 ------------------------------------------------ */
/* x,(c_prev,h_prev): (B,3,H,W) fp32; c_prev/h_prev NULL = zeros (RDN.py:57-68);
 * w: (12,6,3,3), b: (12); writes h_out and (optionally) c_out. */
int bin_convlstm_fwd(const float* x, const float* c_prev, const float* h_prev, const float* w, const float* b,
                     float* h_out, float* c_out, int B, int H, int W, bin_stream_t s);

/* Backward of the cell: dh/dc = gradients of the two outputs (either may be NULL = zero); dgates_ws = scratch
 * (B,12,H,W) fp32; writes dx (and dc_prev/dh_prev when a state was given), ACCUMULATES into dw (12,6,3,3) and db (12). */
int bin_convlstm_bwd(const float* x, const float* c_prev, const float* h_prev, const float* w, const float* b,
                     const float* dh, const float* dc, float* dgates_ws, float* dx, float* dc_prev, float* dh_prev,
                     float* dw, float* db, int B, int H, int W, bin_stream_t s);

/* ---- one backbone (RDN_residual_interp_{2,2_1,4_1}_input.forward, RDN.py:210-334) ---------- */
#define BIN_BACKBONE_NCONV 66 /* SFENet1, SFENet2, 12 x (4 conv + LFF), GFF.0, GFF.1, UPNet.0, UPNet.2 */
size_t bin_backbone_packed_bytes(int nframes);
/* w[i], b[i]: device fp32 parameters in nn.Module registration order (see bin_b200/rdn.py). */
int bin_backbone_pack(int nframes, const float* const* w_host, const float* const* b_host, void* blob,
                      bin_stream_t s);
size_t bin_backbone_workspace_bytes(int nframes, int Btot, int H, int W);
int bin_backbone_fwd(int nframes, const void* blob, const bin_frames_t* fr, int H, int W, void* workspace,
                     size_t workspace_bytes, bin_stream_t s);
/* ---- training: forward that keeps the activations + backward (bin_model.optimize_parameters,
 * bin_model.py:130-141 -> l_pix.backward()).  Gradients flow as loss-scaled fp16 P8 tensors:
 * *scale_dev (device float, a power of two chosen by the caller from max|dOut|) multiplies dOut on entry
 * and is divided out of every result (frame gradients, dW, db). */
size_t bin_backbone_packed_t_bytes(int nframes);             /* data-gradient (transposed, tap-flipped) weights */
int bin_backbone_pack_t(int nframes, const float* const* w_host, void* blob_t, bin_stream_t s);
size_t bin_backbone_train_workspace_bytes(int nframes, int Btot, int H, int W);   /* saved activations */
int bin_backbone_fwd_train(int nframes, const void* blob, const bin_frames_t* fr, int H, int W, void* save_ws,
                           size_t save_ws_bytes, bin_stream_t s);
size_t bin_backbone_grad_workspace_bytes(int nframes, int Btot, int H, int W);
size_t bin_backbone_grad_param_floats(int nframes);          /* fp32 [w0,b0,w1,b1,...] in nn.Module order */
/* dout->out[k]: dL/d(output of call k), (Bc,3,H,W) fp32.  dframes->frame[k][f]: receives dL/d(frame f of call k)
 * (written, not accumulated; the caller sums frames that feed several calls).  grad_params is ACCUMULATED into. */
int bin_backbone_bwd(int nframes, const void* blob_t, const bin_frames_t* dout, const bin_frames_t* dframes, int H, int W,
                     const void* save_ws, void* grad_ws, size_t grad_ws_bytes, float* grad_params,
                     const float* scale_dev, bin_stream_t s);
/* Loss scale for one backbone backward: *scale_dev = 2^floor(log2(target / max_k max|gouts[k]|)) (a power of two, so
 * scaling and un-scaling are exact), computed on the device -- no host synchronisation.  gouts_host: host array of n
 * (<= BIN_MAX_CALLS) device pointers to fp32 tensors of `numel` elements, 16-byte aligned; tmp4_dev: 4 bytes of scratch. */
int bin_grad_scale(const float* const* gouts_host, int n, size_t numel, float target, float* scale_dev, void* tmp4_dev,
                   bin_stream_t s);

/* Unit-test entry: one RDB (RDN.py:149-165) on fp32 NCHW (B,96,h,w), using RDB `index` of the blob. */
int bin_rdb_fwd(const void* blob, int nframes, int index, const float* x, float* y, int B, int h, int w,
                void* workspace, size_t workspace_bytes, bin_stream_t s);

/* ---- whole 6-frame window (RDN_residual_interp_5_input_ConvLSTM_L.forward, RDN.py:422-465) */
typedef struct {
  const void* blob[4];      /* packed model1_1, model2_1, model3_1, model4_1 */
  const float* lstm_w[6];   /* clstm_{4',6',8',5'',7'',6'''}.Gates.weight (12,6,3,3) */
  const float* lstm_b[6];
} bin_net_t;
size_t bin_window_workspace_bytes(int B, int H, int W);
/* frames[6], outs[14]: (B,3,H,W) fp32 NCHW device tensors.  Executes the 17 unique backbone
 * calls of the reference's 20 (the 3 repeated stage-1 calls are bit-identical) and the 6 live
 * ConvLSTM calls of its 12 (SURVEY.md Appendix A). */
int bin_window_fwd(const bin_net_t* net, const float* const* frames_host, float* const* outs_host, int B, int H,
                   int W, void* workspace, size_t workspace_bytes, bin_stream_t s);
/* Precision-parameterised twins of the calls above (prec = BIN_PREC_F16 | BIN_PREC_F32X3).  In BIN_PREC_F32X3 the
 * packed blob is 3x and the workspace 2x as large; results match the fp32 reference to <=1e-5. */
size_t bin_backbone_packed_bytes_p(int nframes, int prec);
int bin_backbone_pack_p(int nframes, const float* const* w_host, const float* const* b_host, void* blob, int prec,
                        bin_stream_t s);
size_t bin_backbone_workspace_bytes_p(int nframes, int Btot, int H, int W, int prec);
int bin_backbone_fwd_p(int nframes, const void* blob, const bin_frames_t* fr, int H, int W, void* workspace,
                       size_t workspace_bytes, int prec, bin_stream_t s);
size_t bin_window_workspace_bytes_p(int B, int H, int W, int prec);
int bin_window_fwd_p(const bin_net_t* net, const float* const* frames_host, float* const* outs_host, int B, int H,
                     int W, void* workspace, size_t workspace_bytes, int prec, bin_stream_t s);

/* BASELINE config 2a/3a: stages 1-3 on 4 frames -> 6 outputs [I2',I4',I6',I3',I5',I4'']. */
int bin_pyramid3_fwd(const bin_net_t* net, const float* const* frames_host, float* const* outs_host, int B, int H,
                     int W, void* workspace, size_t workspace_bytes, bin_stream_t s);

/* ---- fused pixel loss (SURVEY 8f rank 3): bin_model.get_loss, bin_model.py:395-425 ---------------------- */
/* kind: 0 = nn.L1Loss(reduction='sum') (bin_model.py:55), 1 = nn.MSELoss(reduction='sum') (:57),
 * 2 = CharbonnierLoss mean sqrt(d^2+eps) (loss.py:130-140).  pair_loss[k] (device fp32[npairs]) = cri_pix(a_k, b_k);
 * the caller's loss is their mean.  a_host/b_host: host arrays of npairs device pointers, n elements each. */
enum { BIN_LOSS_L1_SUM = 0, BIN_LOSS_L2_SUM = 1, BIN_LOSS_CHARBONNIER_MEAN = 2 };
int bin_pixel_loss_fwd(const float* const* a_host, const float* const* b_host, int npairs, size_t n, int kind, float eps,
                       float* pair_loss, bin_stream_t s);
/* da_k = (upstream/npairs) * d cri_pix / d a_k, db_k = -da_k (db_host or single entries may be NULL). */
int bin_pixel_loss_bwd(const float* const* a_host, const float* const* b_host, float* const* da_host, float* const* db_host,
                       int npairs, size_t n, int kind, float eps, const float* upstream, bin_stream_t s);

/* ---- image boundary of the caller loop (SURVEY 8f rank 2) ------------------------------------ */
/* utils/util.py:113-137 tensor2img + the crop of test.py:394-402 for ONE (3,Hs,Ws) fp32 RGB image:
 * clamp [0,1], *255, round-half-even, uint8 HWC BGR of the (top,left,h,w) window -> out (h*w*3 bytes, device). */
int bin_tensor2img_u8(const float* x, int Hs, int Ws, int top, int left, int h, int w, uint8_t* out, bin_stream_t s);
/* test.py:44-56 read_image + the ReplicationPad2d of test.py:366-371: uint8 HWC BGR (h,w,3) ->
 * fp32 CHW RGB /255 of size (3, h+pad_t+pad_b, w+pad_l+pad_r), edge-replicated. */
int bin_u8_to_frame(const uint8_t* img, int h, int w, int pad_l, int pad_r, int pad_t, int pad_b, float* out, bin_stream_t s);

/* ---- optimizer step (SURVEY 8f rank 3): torch.optim.Adam as bin_model.py:97-100 builds it and :141 steps it ----- */
/* One launch over every parameter tensor.  table (device): ntensors entries; chunk_prefix (device int[ntensors+1]):
 * chunk_prefix[t] = number of BIN_ADAM_CHUNK-element blocks before tensor t, chunk_prefix[ntensors] = nchunks.
 * Semantics of torch.optim.Adam(amsgrad=False, maximize=False): g' = grad_scale*g + weight_decay*p;
 * m += (g'-m)(1-beta1); v = beta2 v + (1-beta2) g'^2; p -= lr/bias_correction1 * m / (sqrt(v)/sqrt(bias_correction2) + eps)
 * with bias_correction_i = 1 - beta_i^step computed by the caller (as torch does, on the host). */
#define BIN_ADAM_CHUNK 4096
typedef struct {
  float* p;                 /* parameter (updated in place)        */
  const float* g;           /* gradient                            */
  float* m;                 /* exp_avg                             */
  float* v;                 /* exp_avg_sq                          */
  unsigned long long n;     /* elements                            */
} bin_adam_tensor_t;
int bin_adam_step(const bin_adam_tensor_t* table_dev, const int* chunk_prefix_dev, int ntensors, int nchunks, float lr,
                  float beta1, float beta2, float eps, float weight_decay, float bias_correction1,
                  float bias_correction2, float grad_scale, bin_stream_t s);

/* ---- training-data synthesis (SURVEY 8f rank 4): create_dataset_blur_N_frames_average.py:108-134 ------------------ */
/* frames: device uint8 [T][frame_bytes] (consecutive sharp frames, any pixel layout); out: [nwin][frame_bytes].
 * out[w] = uint8( sum_{j=-r..r} float32(frames[first_mid + w*stride + j]) / float32(2r+1) ), r = (window_size-1)/2
 * (script: window_size 11, first_mid 16, stride 8, nwin = floor(T/8) - 2). */
int bin_blur_average_u8(const uint8_t* frames, int T, size_t frame_bytes, int window_size, int first_mid, int stride,
                        int nwin, uint8_t* out, bin_stream_t s);

/* ---- evaluation metrics (DESIGN 5c rank 5): the PSNR / SSIM / interpolation error of test.py:404-458 and the
 * validation metrics of bin_model.compute_current_psnr_ssim (bin_model.py:564-589) ------------------------------ */
/* kind selects the SSIM definition; both are valid-region filters (no border handling):
 *   BIN_SSIM_BOX7    skimage 0.14-0.16 compare_ssim(X, Y, multichannel=True) with the defaults test.py:35 uses:
 *                    7x7 uniform window, sample covariance (x49/48), K1 = 0.01, K2 = 0.03, L = 255, map cropped by
 *                    3 px per side, mean over channels of the per-channel means;
 *   BIN_SSIM_GAUSS11 utils/util.py:211-231 ssim (and calculate_ssim, :234-252): 11x11 window = outer product of
 *                    cv2.getGaussianKernel(11, 1.5), population moments, same K1 / K2, [5:-5, 5:-5] crop, mean over
 *                    every element. */
enum { BIN_SSIM_BOX7 = 0, BIN_SSIM_GAUSS11 = 1 };
#define BIN_MAX_METRIC_PAIRS 64
/* Workspace of one call: per-CTA partial sums (0 for arguments the call would reject). */
size_t bin_image_metrics_workspace_bytes(int npairs, int h, int w, int c, int kind);
/* res (device double[npairs][3]) = {mse, mae, ssim} per pair; a_host/b_host: npairs device pointers to h*w*c uint8
 * (HWC, c = 1 or 3, h and w at least the window size).  mse = mean (a-b)^2 (util.py:203-205; PSNR =
 * 10 log10(255^2 / mse)), mae = mean |a-b| (test.py:431-435 interpolation error).  Sums are exact integers; the
 * reduction is deterministic (fixed order, no atomics) and a pair's result does not depend on the other pairs. */
int bin_image_metrics_u8(const uint8_t* const* a_host, const uint8_t* const* b_host, int npairs, int h, int w, int c,
                         int kind, double* res, void* ws, size_t ws_bytes, bin_stream_t s);

/* ---- training batches (DESIGN 5c rank 6): BINDataset.__getitem__ + DataLoader collation, data/BIN_dataset.py:30-183 -- */
/* One sample: its 17 source frames in output-slot order -- blurry B1..B11 (LQs), sharp I1..I11 (GTenh), sharp
 * I2..I10 (GTinp); the reference's random reversal (:68-109) is the caller's choice of this order -- and its crop
 * (rows y0.., columns x0..) and np.fliplr (:155-177).  Each src: device uint8 (H, W, 3) BGR, row-major HWC. */
#define BIN_TRAIN_FRAMES 17
#define BIN_MAX_TRAIN_SAMPLES 64 /* samples per kernel launch (the table travels in the kernel parameters) */
typedef struct {
  const uint8_t* src[BIN_TRAIN_FRAMES];
  int y0, x0, flip;
} bin_train_sample_t;
/* samples: host array of B >= 1 entries (one launch per BIN_MAX_TRAIN_SAMPLES of them; no copy, no synchronisation).
 * Writes fp32 float32(u8)/255 RGB crops of h x w (1 <= h <= H, 1 <= w <= W, crop inside the frame) slot-major:
 * lqs [6][B][3][h][w], gtenh [6][B][3][h][w], gtinp [5][B][3][h][w]. */
int bin_train_batch_u8(const bin_train_sample_t* samples, int B, int H, int W, int h, int w, float* lqs, float* gtenh,
                       float* gtinp, bin_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* BIN_B200_H_ */
