/* ievm.h -- C ABI of the B200 (sm_100a) engine for the hot path of
 * jaideepmurkute/Inference-Efficient-Vision-Models: the batched forward pass `outputs = model(images)`
 * of the pruned ResNet-18 student after static INT8 PTQ or FP16 casting, and of the ResNet-50 teacher.
 *
 * Reference interfaces replaced (the reference is pure Python; its "FFI" for this path is the
 * nn.Module call protocol plus the converted module's attribute / state-dict layout):
 *
 *   ievm_create        <- the converted module the caller holds: quantize_fx.convert_fx(...)
 *                         (quantization/engines.py:118, quantization/main.py:242) or
 *                         deepcopy(model).half() (quantization/engines.py:91-92, main.py:258/262)
 *   ievm_forward_i8    <- outputs = model(images), f32 NCHW in -> f32 logits out
 *                         (quantization/engines.py:27,31,60; quantization/main.py:287)
 *   ievm_forward_f16   <- outputs = model(images.half()) (quantization/engines.py:57-60; main.py:284-287)
 *                         and teacher_model(images) (knowledge_distillation/train.py:43-44)
 *   ievm_forward_*_host<- the same calls with `images` still on the host, as the reference's loops
 *                         hand them over (engines.py:52-60): H2D + forward + D2H in one call
 *   ievm_kd_loss       <- CE + T^2 * KLDiv(batchmean) soft-target loss
 *                         (knowledge_distillation/train.py:47-57; main.py:128-129)
 *   ievm_set_input_lut,
 *   ievm_forward_u8*   <- the dataset transform in front of the call, T.ToTensor() + T.Normalize(mean, std)
 *                         (quantization/dataset.py:14-19), fused with the graph's quantize_per_tensor node
 *   ievm_observe,
 *   ievm_observer_read <- the observer passes of PTQ calibration, `prepared_model(images)` over the calibration loader
 *                         (quantization/engines.py:123-133 `_calibrate`; quantization/main.py:236-239): float forward on
 *                         the FP16 engine, per-batch torch.aminmax of every observed tensor reduced on the device
 *   ievm_count_correct <- the accumulation of evaluate_accuracy (quantization/engines.py:59-63; main.py:288-290)
 *   ievm_debug_*       <- no reference counterpart: parity hooks (per-tensor activations and the
 *                         int32 accumulators torch never exposes)
 *
 * Conventions: every function returns 0 on success or a negative ievm_status; ievm_last_error()
 * describes the last failure on the calling thread.  Device pointers are plain CUDA device
 * pointers owned by the caller; `stream` is a cudaStream_t passed as void*.  Work is enqueued on the
 * caller's stream without synchronising or allocating (CUDA-graph capturable) unless stated.
 * A handle is bound to one device and is not re-entrant: calls on one handle come from one thread at a time.  All
 * forwards of a handle share one activation workspace; consecutive calls may use different streams (the engine orders
 * them with an event recorded at the end of every enqueue), but their work runs one after the other.  Every entry
 * point restores the calling thread's current CUDA device before it returns.  There is no CPU fallback: creation fails
 * with IEVM_ERR_CUDA when no sm_100 device is present.
 */
#ifndef IEVM_H_
#define IEVM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ievm_handle ievm_handle;

typedef enum ievm_status {
  IEVM_OK = 0,
  IEVM_ERR_BAD_ARG = -1,
  IEVM_ERR_UNSUPPORTED = -2,
  IEVM_ERR_CUDA = -3,
  IEVM_ERR_OOM = -4
} ievm_status;

typedef enum ievm_dtype { IEVM_DTYPE_I8 = 0, IEVM_DTYPE_F16 = 1 } ievm_dtype;

typedef enum ievm_op {
  IEVM_OP_CONV = 0,    /* conv (+folded BN) [+ReLU] [+residual add (+ReLU)] */
  IEVM_OP_MAXPOOL = 1, /* MaxPool2d(3, 2, 1) */
  IEVM_OP_HEAD = 2,    /* AdaptiveAvgPool2d(1) + flatten + Linear (+ dequantize) -> logits */
  IEVM_OP_ADD_RELU = 3 /* F16 only: out = relu(in_tensor + res_tensor), the BasicBlock's residual add left un-fused so
                          that calibration can observe the conv output in front of it (see ievm_observe) */
} ievm_op;

/* One node of the flattened graph.  Tensor id 0 is the network input (for INT8: the output of
 * quantize_per_tensor); every other id names the output of exactly one earlier layer. */
typedef struct ievm_layer_desc {
  int32_t op;          /* ievm_op */
  int32_t in_tensor;
  int32_t res_tensor;  /* residual operand of the fused add, or -1 */
  int32_t out_tensor;  /* ignored for IEVM_OP_HEAD */
  int32_t cin, cout;   /* real (un-padded) channel counts; HEAD: cin = features, cout = classes */
  int32_t ksize, stride, pad;
  int32_t relu;        /* I8: the module is ConvReLU2d (ReLU on the conv's own output; the fused
                          add_relu always clamps).  F16: ReLU is the layer's last operation
                          (after the residual add when res_tensor >= 0). */
  const void* weight;  /* host pointer. I8: int8 [cout][cin][k][k]; F16: IEEE half bits, BN folded */
  const float* bias;   /* host pointer, [cout] (BN folded) */
  const float* w_scale;/* host pointer, [cout], I8 only */
  float in_scale;  int32_t in_zp;    /* I8: qparams of in_tensor */
  float out_scale; int32_t out_zp;   /* I8: qparams of this layer's own output (module.scale/zero_point) */
  float res_scale; int32_t res_zp;   /* I8: qparams of res_tensor */
  float add_scale; int32_t add_zp;   /* I8: output qparams of quantized.add_relu (used iff res_tensor >= 0) */
} ievm_layer_desc;

typedef struct ievm_net_desc {
  int32_t dtype;       /* ievm_dtype */
  int32_t num_layers;
  int32_t in_c, in_h, in_w;
  int32_t num_classes;
  float in_scale;      /* I8: quantize_per_tensor scale / zero point of the network input */
  int32_t in_zp;
  const ievm_layer_desc* layers;
} ievm_net_desc;

/* Build an engine on `device`: pads/packs weights into the tensor-core layout, uploads them,
 * allocates the activation workspace for `max_batch` images and encodes the TMA descriptors.
 * Synchronous.  The descriptor and everything it points to may be freed after the call. */
int ievm_create(const ievm_net_desc* desc, int device, int max_batch, ievm_handle** out);
void ievm_destroy(ievm_handle* h);

/* x: device f32 [n][in_c][in_h][in_w]; logits: device f32 [n][num_classes]. n <= max_batch. */
int ievm_forward_i8(ievm_handle* h, const float* x_nchw, int n, float* logits, void* stream);
/* x: device f16 [n][in_c][in_h][in_w]; logits: device f16 [n][num_classes]. */
int ievm_forward_f16(ievm_handle* h, const void* x_nchw, int n, void* logits, void* stream);

/* Host-buffer variants (what a reference caller holds): copies x to the device, runs the forward
 * and copies the logits back; returns after the logits are in `logits_host`.  Pinned buffers make
 * the copies asynchronous on the handle's own stream. */
int ievm_forward_i8_host(ievm_handle* h, const float* x_nchw_host, int n, float* logits_host);
int ievm_forward_f16_host(ievm_handle* h, const void* x_nchw_host, int n, void* logits_host);

/* Pipelined host entry points for the reference's evaluation loops, which hand over one CPU batch per iteration
 * (quantization/engines.py:52-63, quantization/main.py:277-290).  ievm_submit_*_host ENQUEUES the H2D copy, the forward
 * and the D2H copy of the logits and returns a ticket without synchronising: the copy of call i+1 (copy stream)
 * overlaps the forward of call i (compute stream) through two device staging slots, so at most two tickets are in
 * flight -- a third submit first waits for the first.  x_host and logits_host must stay valid and untouched until
 * ievm_wait(ticket) returns (pinned memory makes the copies asynchronous; pageable memory works but serialises).
 * ievm_wait blocks the calling thread until that ticket's logits are in logits_host. */
int ievm_submit_i8_host(ievm_handle* h, const float* x_nchw_host, int n, float* logits_host, int64_t* ticket);
int ievm_submit_f16_host(ievm_handle* h, const void* x_nchw_host, int n, void* logits_host, int64_t* ticket);
int ievm_submit_u8_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host, int64_t* ticket);
int ievm_submit_u8_resize_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host, int64_t* ticket);
int ievm_wait(ievm_handle* h, int64_t ticket);

/* SURVEY 8(f)-1, the input pipeline in front of the hot path.  INT8 engines accept decoded 8-bit images,
 * x_nhwc = [n][224][224][3] u8 (RGB interleaved, what PIL / T.Resize hand to T.ToTensor in the reference's
 * quantization/dataset.py:14-19), and fuse ToTensor + Normalize + quantize_per_tensor into the front-end kernel
 * through a lookup table lut768 = [3][256] u8: lut[c][v] = quantised value of level v in channel c, which the host
 * computes once with the reference's own float ops (ievm_b200.input_lut), so logits are bit-identical to feeding
 * the f32 tensor.  Four times fewer input bytes over PCIe and HBM. */
int ievm_set_input_lut(ievm_handle* h, const uint8_t* lut768);
int ievm_forward_u8(ievm_handle* h, const uint8_t* x_nhwc, int n, float* logits, void* stream);
int ievm_forward_u8_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host);

/* The remaining step of that transform, T.Resize((H, W)) on the decoded image (quantization/dataset.py:15), is
 * Pillow's 8-bit bilinear ImagingResample; ievm_set_resize installs its per-output-pixel tables for source images of
 * src_h x src_w -- bounds_*[o] = {first source index, taps}, kk_*[o][ksize_*] = 22-bit fixed-point coefficients,
 * computed on the host exactly as Resample.c:precompute_coeffs does (ievm_b200.pipeline.pil_bilinear_coeffs) -- and
 * ievm_forward_u8_resize runs resize (horizontal, then vertical, 8-bit intermediate: bit-identical to PIL) +
 * ToTensor + Normalize + the quantized network on x_nhwc = [n][src_h][src_w][3] u8. */
int ievm_set_resize(ievm_handle* h, int src_h, int src_w, const int32_t* bounds_w, const int32_t* kk_w, int ksize_w,
                    const int32_t* bounds_h, const int32_t* kk_h, int ksize_h);
int ievm_forward_u8_resize(ievm_handle* h, const uint8_t* x_nhwc, int n, float* logits, void* stream);
int ievm_forward_u8_resize_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host);
/* Parity hook: only the resize, result [n][H][W][3] u8 copied to the host. */
int ievm_debug_resize(ievm_handle* h, const uint8_t* x_dev, int n, uint8_t* out_host, uint64_t out_bytes);

/* SURVEY 8(f)-4: calibration statistics on the device.  An FP16 engine built from the observer-instrumented float
 * model (ievm_b200.netdesc.from_prepared: residual adds as IEVM_OP_ADD_RELU layers) with options keep_tensors = 1 and
 * observe = 1 | 2 records, per ievm_observe call, what the reference's observers keep of a batch, for every observation
 * point of the LAST forward, on the caller's stream, without synchronising (two or three launches in all):
 *   point 0              the network input; x_f32 (device f32 [n][c][h][w], the un-rounded batch) when given, else the
 *                        f16 buffer the forward read
 *   point id, 1 <= id < T  tensor `id` over its real channels (T = ievm_num_tensors)
 *   point T              the AdaptiveAvgPool2d output (rounded to f16)
 *   point T + 1          the logits
 * observe = 1: the pair torch.aminmax(x) (MinMaxObserver, MovingAverageMinMaxObserver: quantization/main.py:196-207).
 * observe = 2: additionally torch.histc(x, 2048, min = lo, max = hi) over the running range [lo, hi] of the point's
 *   observer after this batch (HistogramObserver.forward; default fbgemm qconfig, quantization/engines.py:103), as exact
 *   integer counts.  prepare_fx lets several graph nodes share one observer instance; ievm_observer_set_groups maps
 *   every point to its observer (default: one observer per point) so that the running range is the observer's.
 * ievm_observer_read synchronises and copies the (min, max) log as f32 [records][points][2] (NaN = nothing observed),
 * ievm_observer_read_hist the histogram log as u32 [records][points][2048] plus, when range_host is not NULL, the
 * running (min, max) of all 64 observer groups as f32 [64][2]; both return the number of records.
 * ievm_observer_capacity is the number of records the log holds (4096, or 64 with histograms); ievm_observer_clear
 * empties the log but keeps the running ranges (a caller drains a full log and goes on); ievm_set_option(h, "observe",
 * mode) restarts everything.  The host replays the records into the prepared module's own observers
 * (ievm_b200.calibration.calibrate), after which convert_fx runs unchanged. */
int ievm_observer_points(const ievm_handle* h);
int ievm_observer_capacity(const ievm_handle* h);
int ievm_observer_set_groups(ievm_handle* h, const int32_t* group_of_point, int points);
int ievm_observe(ievm_handle* h, const float* x_f32, void* stream);
int ievm_observer_read(ievm_handle* h, float* minmax_host, int max_records);
int ievm_observer_read_hist(ievm_handle* h, uint32_t* hist_host, float* range_host, int max_records);
int ievm_observer_clear(ievm_handle* h);

/* Engine options: "conv_impl" 0 = tcgen05 tensor-core kernels (default), 1 = direct CUDA-core
 * cross-check kernels (tests only); "use_graph" 1 = replay forward() from a CUDA graph cached per
 * (n, x, logits) triple; "keep_tensors" 1 = one buffer per tensor (parity hooks); "profile" 1 =
 * per-launch event timing (see ievm_profile_read); "observe" 1 | 2 = (re)start the calibration observer log (F16 engines; 2 = with histograms), 0 = off. */
int ievm_set_option(ievm_handle* h, const char* name, int value);

/* Introspection used by the benchmark and tests. */
int ievm_num_tensors(const ievm_handle* h);
/* Shape of tensor `id` for the last forward: writes {n, h, w, c_real, c_pitch, elem_bytes}. */
int ievm_tensor_shape(const ievm_handle* h, int id, int32_t out6[6]);
/* Number of kernel launches one forward() enqueues. */
int ievm_launches_per_forward(const ievm_handle* h);
/* Index of the layer whose kernel launch computes `layer`: the layer itself, except that a residual block's 1x1
 * downsample conv runs as a second tile class of the block's first 3x3 conv (option "dual", default on) and the
 * max-pool runs inside the fused front end (layer 0).  -1 for a bad index. */
int ievm_layer_launch(const ievm_handle* h, int layer);

/* Per-launch device timing.  With ievm_set_option(h, "profile", 1) every forward brackets each of its
 * launches with CUDA events on the caller's stream and synchronises at the end (not for timed
 * throughput runs).  ievm_profile_read copies the accumulated milliseconds and call counts: slot 0 is
 * the input-quantize launch (INT8), slot 1 + i is layer i.  Returns the number of slots. */
int ievm_profile_read(const ievm_handle* h, int max_slots, float* ms_sum, int32_t* calls);

/* Parity hooks.  ievm_debug_read_tensor copies tensor `id` as left by the last forward into a host
 * buffer in the engine's layout [n][h][w][c_pitch] (synchronises the device).  Tensors share
 * workspace, so call ievm_set_option(h, "keep_tensors", 1) before the forward to give every tensor
 * its own buffer. */
int ievm_debug_read_tensor(ievm_handle* h, int id, void* host_out, uint64_t host_bytes);
/* Re-runs conv layer `layer` on its current input with accumulator dumping enabled and copies the
 * raw accumulators (int32 for I8, fp32 bits for F16) as [n*ho*wo][c_pitch] to the host. */
int ievm_debug_conv_acc(ievm_handle* h, int layer, int n, int32_t* host_out, uint64_t host_bytes);

/* Runs ONLY the fused front end (quantize + stem + ReLU + max-pool, frontend_v2.cuh) on the device batch
 * x_dev and copies the pooled tensor [n][ph][pw][c_pitch] (u8 / f16) to pooled_host; when acc_host is not
 * NULL also the stem's zero-point-corrected accumulators [n][ho][wo][c_pitch] (int32; fp32 bits for F16).
 * in_mode 0: x_dev is the engine's native input (f32 / f16 NCHW); 1: decoded 8-bit images, u8 [n][in_h][in_w][3]
 * through the lookup table of ievm_set_input_lut (INT8 engines).  Without acc_host the kernel the forward would
 * launch for that input runs. */
int ievm_debug_frontend(ievm_handle* h, const void* x_dev, int in_mode, int n, void* pooled_host, uint64_t pooled_bytes,
                        int32_t* acc_host, uint64_t acc_bytes);

/* Diagnostic: issue ONE im2col-mode TMA load (128 pixels x kc_bytes channels of a u8 NHWC tensor
 * with channel pitch c_pitch) for the tile that starts at output pixel m0, filter tap
 * (tap_x, tap_y), channel offset c0, and copy the raw (swizzled) shared-memory image, 128*kc_bytes
 * bytes, to out_dev.  Synchronous.  Lets the tests pin the TMA unit's im2col semantics
 * (bounding box, traversal stride, zero fill, swizzle) independently of the MMA path. */
int ievm_probe_im2col(const void* in_dev, int n, int h, int w, int c_pitch, int ksize, int stride, int pad,
                      int kc_bytes, int m0, int tap_x, int tap_y, int c0, void* out_dev);

/* Diagnostic: ONE tiled 4-D TMA box {rb bytes of C, box_w pixels, box_h rows, 1 image} of a u8 NHWC
 * tensor starting at pixel (w0, h0) of image `img` (negative / past-the-end coordinates are zero
 * filled), dumped raw (swizzled) from shared memory: box_w*box_h*rb bytes.  Pins the layout the
 * halo-patch convolution mode relies on. */
int ievm_probe_patch(const void* in_dev, int n, int h, int w, int c_pitch, int rb, int img, int w0, int h0, int box_w,
                     int box_h, void* out_dev);

/* SURVEY 8(f)-3: the accumulation step of evaluate_accuracy (quantization/engines.py:59-63) on the device.
 * logits: [n][classes] f32 (dtype IEVM_DTYPE_I8 engines) or f16 (IEVM_DTYPE_F16); labels int64 [n];
 * counters2 (device, u64[2]) += {number of rows whose arg-max (lowest index on ties) equals the label, n}. */
int ievm_count_correct(const void* logits, int dtype, const int64_t* labels, int n, int classes, uint64_t* counters2,
                       void* stream);

/* Soft-target KD evaluation loss over device logits (f32 [n][classes]) and labels (int64 [n]).
 * out3 (device, f32[3]) receives {mean CE, mean T^2*KL (batchmean), number correct};
 * total loss = (1 - alpha) * CE + alpha * KL. */
int ievm_kd_loss(const float* student_logits, const float* teacher_logits, const int64_t* labels, int n,
                 int classes, float temperature, float* out3, void* stream);

/* Measurement support (bench.py's roofline denominator): the rate at which THIS device's tensor cores retire a stream of
 * tcgen05.mma M128 x N256 x K32-byte instructions (kind::i8 for IEVM_DTYPE_I8, kind::f16 for IEVM_DTYPE_F16) issued
 * from one CTA per SM, timed with CUDA events: `iters` x 16 instructions per SM; *tera_ops = 2 * MACs / s / 1e12.
 * MEASURED_PEAKS.json holds a cuBLAS bf16 figure only; there is no library INT8 GEMM to measure against. */
int ievm_probe_mma_peak(int device, int dtype, int iters, double* tera_ops);

/* Every mbarrier wait inside the kernels is bounded: after `ms` milliseconds (default 2000) it records which pipeline
 * role was stuck and traps, so that a protocol bug fails a test instead of hanging a GPU box.  0 = wait forever: for
 * runs under ncu replay, compute-sanitizer or GPU time-slicing, where the limit can fire spuriously (also
 * IEVM_WAIT_LIMIT_MS in the environment at ievm_create). */
int ievm_set_wait_limit_ms(int device, int64_t ms);

const char* ievm_last_error(void);
/* "sm_100a" build tag and ABI version, for the loader to check. */
const char* ievm_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* IEVM_H_ */
