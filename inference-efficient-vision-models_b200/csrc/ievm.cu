// C-ABI implementation (include/ievm.h): graph planning, weight packing, TMA descriptor encoding and
// kernel sequencing for the INT8 / FP16 ResNet forward on sm_100a.
#include "../../include/ievm.h"

#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "conv_tc.cuh"
#include "conv_dual.cuh"
#include "conv_s2.cuh"
#include "simt_kernels.cuh"
#include "stem_tc.cuh"
#include "frontend_v2.cuh"
#include "observe.cuh"
#include "probe_mma.cuh"

namespace {

using namespace ievm;

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t e__ = (expr);                                                                       \
    if (e__ != cudaSuccess)                                                                         \
      return fail(e__ == cudaErrorMemoryAllocation ? IEVM_ERR_OOM : IEVM_ERR_CUDA, "%s failed: %s", \
                  #expr, cudaGetErrorString(e__));                                                  \
  } while (0)

// Every entry point runs on the handle's device and leaves the calling thread's current device as it found it.
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// ---- driver entry points for tensor-map encoding (resolved at run time: the library must load on a
// machine without libcuda so that the CPU-only test tier can check its exports) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode_tiled = nullptr;
EncodeIm2colFn g_encode_im2col = nullptr;

int load_driver_entry_points() {
  if (g_encode_tiled && g_encode_im2col) return IEVM_OK;
  cudaDriverEntryPointQueryResult q;
  void* fn = nullptr;
  CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  if (q != cudaDriverEntryPointSuccess || !fn) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled not available");
  g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
  fn = nullptr;
  CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q));
  if (q != cudaDriverEntryPointSuccess || !fn) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeIm2col not available");
  g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
  return IEVM_OK;
}

int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Launch with (optionally) the programmatic-stream-serialization attribute: the kernel may begin while its
// predecessor in the stream drains; it calls griddepcontrol.wait before touching the predecessor's output.
template <typename... KArgs, typename... Args>
cudaError_t launch_kernel_cluster(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s,
                                  bool pdl, unsigned cluster, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  unsigned na = 0;
  if (pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
template <typename... KArgs, typename... Args>
cudaError_t launch_kernel(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, bool pdl,
                          Args&&... args) {
  return launch_kernel_cluster(kernel, grid, block, smem, s, pdl, 1u, std::forward<Args>(args)...);
}

struct TensorInfo {
  int h = 0, w = 0, c = 0, pitch = 0;   // pitch in elements
  int elem = 1;
  int producer = -1;                    // layer index, -1 for the network input
  int last_use = -1;
  int buffer = -1;
  int hp = 0, wp = 0, pad_t = 0, pad_l = 0;   // stored with a constant border when hp > 0 (INT8 network input)
  size_t bytes_per_image() const {
    return hp > 0 ? static_cast<size_t>(hp) * wp * pitch * elem : static_cast<size_t>(h) * w * pitch * elem;
  }
};

struct LayerPlan {
  ievm_layer_desc d;
  bool is_stem = false;
  // conv geometry
  int h = 0, w = 0, ho = 0, wo = 0;
  int cin_pitch = 0, cout_pad = 0;
  int bn = 0, n_tiles = 0;
  int kc_bytes = 0, kc_elems = 0, kchunks = 0, cin_w = 0;
  int stages = 0, tmem_cols = 0, resident_b = 0;
  int mode = 0;                 // kModeIm2col | kModeHalo
  int fast_round = 0;           // see ConvTcParams::fast_round
  int cluster = 1;              // CTAs per cluster sharing the weight tile by TMA multicast
  int max_clusters = 0;         // co-resident clusters the device can hold (cluster > 1)
  int wp = 0, patch_rows = 0, a_stage_bytes = 0, a_tx_bytes = 0;
  int sub_rows = 0, subs_per_img = 0, band_subs = 0;   // halo (band) mode, conv_tc.cuh
  int kb_group = 1;             // im2col mode: k-blocks per barrier pair
  int two_cta = 0;              // halo mode, narrow INT8 layers: two 320-thread CTAs per SM (conv_tc.cuh, kEpiW = 8)
  size_t smem_bytes = 0;
  // device operands
  void* w_packed = nullptr;     // tensor-core layout [cout_pad][taps][cin_w]
  void* w_stem = nullptr;       // stem layout (CUDA-core kernels)
  void* w_stem_tc = nullptr;    // stem layout for the tensor-core kernel: [cout_pad][8 segments x 32 B]
  void* w_front2 = nullptr;     // frontend_v2.cuh weight operand image (two stem rows stacked in M)
  int* wsum = nullptr;
  int* zwsum = nullptr;         // in_zp * wsum
  int32_t* zcorr = nullptr;     // tensor-core convs with a non-zero input zero point: ConvTcParams::zcorr
  size_t stem_smem = 0;
  float* ep0 = nullptr;
  float* ep1 = nullptr;
  std::vector<float> ep0_host, ep1_host;   // copies for the kernel-parameter block (ConvTcParams::epc0 / epc1)
  CUtensorMap tmap_a, tmap_b;
  // conv_dual.cuh: a block's first 3x3 conv runs the block's 1x1 downsample (the next layer) as a second tile class
  int dual_partner = -1;        // on the 3x3: index of the downsample layer
  int dual_of = -1;             // on the downsample: index of the 3x3 whose launch computes it
  int dual_stages = 0, dual_kb_group = 1, dual_max_clusters = 0;
  size_t dual_smem_bytes = 0;
  CUtensorMap tmap_b2;          // the downsample's weights with the 3x3's N-tile box
  // pixel-pair form of the dual launch (conv_dual.cuh): INT8 3x3 stride-2 convs over 64-byte pixels
  int dual_wide = 0;
  // phase-patch form (conv_s2.cuh): the same layers as four stride-1 phase patches; preferred over the pixel-pair form
  int dual_s2 = 0, s2_stages = 0, s2_rows = 0, s2_phase_bytes = 0;
  size_t s2_smem_bytes = 0;
  CUtensorMap tmap_a_s2, tmap_b2_s2;
  void* w_wide = nullptr;       // on the 3x3: [cout_pad][3 x 2 wide taps][128]; on the downsample: [cout_pad][1][128]
  CUtensorMap tmap_a_wide, tmap_b_wide;
};

}  // namespace

struct ievm_handle {
  int device = 0;
  int dtype = 0;
  int elem = 1;
  int max_batch = 0;
  int num_sms = 0;
  int smem_optin = 0;
  int opt_halo = 1;        // IEVM_HALO=0 disables the halo-patch mode (all convs use per-tap im2col TMA)
  int opt_two_cta = 1;     // IEVM_TWO_CTA=0: one CTA per SM for every layer
  int opt_halo_static = 1; // IEVM_HALO_STATIC=0: run-time-shaped halo kernel (class 0) even for the specialised shapes
  int opt_fused_front = 1; // IEVM_FUSED_FRONT=0: separate quantize / stem / maxpool kernels
  int front2_ok = 0;       // the network's front end fits frontend_v2.cuh (224-wide input, <= 64 stem channels)
  int front_tpu = 0;       // IEVM_FRONT_TPU: pooled rows per work unit (0 = heuristic)
  uint8_t* lut_dev = nullptr;   // u8 input mode: [3][256] level -> quantised value (ievm_set_input_lut)
  // resize front stage (ievm_set_resize): Pillow bilinear tables and the two intermediate images
  int rs_in_h = 0, rs_in_w = 0, rs_ksize_w = 0, rs_ksize_h = 0;
  int2* rs_bounds_w = nullptr;
  int2* rs_bounds_h = nullptr;
  int* rs_kk_w = nullptr;
  int* rs_kk_h = nullptr;
  uint8_t* rs_tmp = nullptr;    // [max_batch][rs_in_h][in_w][3]
  uint8_t* rs_out = nullptr;    // [max_batch][in_h][in_w][3]
  size_t stage_in_bytes = 0;
  int opt_cluster = 1;     // IEVM_CLUSTER=0: no 2-CTA clusters / weight multicast
  int opt_pdl = 1;         // IEVM_PDL=0: no programmatic dependent launch
  int opt_fixed_bn = 0;    // IEVM_FIXED_BN=1: one N tile per <=256 channels (disables the tile-width heuristic)
  int opt_dual = 1;        // IEVM_DUAL=0 / option "dual": the 1x1 downsample convs run as launches of their own
  int opt_wide = 1;        // IEVM_WIDE=0: no pixel-pair form in dual launches (conv_dual.cuh)
  int opt_s2 = 1;          // IEVM_S2=0: no phase-patch form of the stride-2 dual launch (conv_s2.cuh)
  int opt_tiny = 1;        // IEVM_TINY=0: no single-accumulator form of the halo layers at small batches (launch_conv)
  int front_chunk = 0;     // IEVM_FRONT_CHUNK: images per front-end chunk (0 = whole batch at once, default)
  // IEVM_HALO_RB128=1: 64-byte pixels use 128-byte shared-memory rows in halo mode
  int in_c = 0, in_h = 0, in_w = 0, classes = 0;
  float in_scale = 1.f;
  int in_zp = 0;
  std::vector<LayerPlan> layers;
  std::vector<TensorInfo> tensors;
  std::vector<void*> buffers;
  std::vector<size_t> buffer_bytes;
  std::vector<void*> owned;            // device allocations freed at destroy
  // calibration observers (observe.cuh): per ievm_observe call one record of (min, max) pairs, order-encoded u32
  uint32_t* obs_log = nullptr;         // [kObsMaxRecords][points][2]
  uint32_t* obs_run = nullptr;         // [kObsMaxPoints][2] running (min, max) per observer group
  uint32_t* obs_hist = nullptr;        // [kObsHistRecords][points][kObsBins] (observe = 2)
  int obs_group[kObsMaxPoints] = {};   // point -> observer group (ievm_observer_set_groups; default: its own)
  int obs_mode = 0;                    // 0 off, 1 min/max, 2 min/max + histograms
  int obs_records = 0;
  __half* obs_pooled = nullptr;        // avgpool output of the last forward, [max_batch][head cin]; null = not calibrating
  __half* obs_pooled_alloc = nullptr;
  const void* last_x = nullptr;        // caller's buffers of the last forward (network input / logits)
  const void* last_logits = nullptr;
  int conv_impl = 0;
  int keep_tensors = 0;
  int use_graph = 0;
  int last_n = 0;
  unsigned int* stuck_host = nullptr;  // mapped pinned word
  unsigned int* stuck_dev = nullptr;
  cudaStream_t own_stream = nullptr;
  cudaStream_t copy_stream = nullptr;   // H2D copies of the *_host entry points
  std::vector<cudaEvent_t> copy_events;
  int host_chunk = 64;                  // IEVM_HOST_CHUNK: images per H2D/compute pipeline chunk (0 = no chunking)
  void* stage_in = nullptr;            // device staging for the *_host entry points
  void* stage_out = nullptr;
  void* pin_in = nullptr;              // pinned host staging
  void* pin_out = nullptr;
  size_t pin_in_bytes = 0;
  // CUDA graphs cached per (n, input mode, x, logits); bounded (kMaxGraphs, least recently used goes first)
  std::map<std::tuple<int, const void*, void*>, std::pair<cudaGraphExec_t, unsigned long long>> graphs;
  unsigned long long graph_clock = 0;
  // All forwards of a handle share one activation workspace: work enqueued on a different stream than the previous
  // forward's first waits for `order_event`, recorded at the end of every enqueue (ADVICE r1: y1 = model(x_cuda);
  // y2 = model(x_cpu) raced on the workspace).
  cudaEvent_t order_event = nullptr;
  cudaStream_t last_stream = nullptr;
  bool order_valid = false;
  // pipelined host entry points (ievm_submit_*_host / ievm_wait): two staging slots, no per-call stream synchronisation
  struct HostSlot {
    void* dev_in = nullptr;
    void* dev_out = nullptr;
    size_t in_bytes = 0;
    cudaEvent_t copied = nullptr, done = nullptr;
    long long ticket = -1;          // ticket in flight in this slot, -1 = free
  } slots[2];
  long long next_ticket = 0;
  // per-launch device timing (option "profile"): slot 0 = input quantize, slot 1 + i = layer i
  int profile = 0;
  std::vector<cudaEvent_t> prof_events;
  std::vector<double> prof_ms;
  std::vector<int> prof_calls;
};

namespace {

template <typename T>
int dev_upload(ievm_handle* h, const std::vector<T>& host, T** out) {
  void* p = nullptr;
  CUDA_TRY(cudaMalloc(&p, std::max<size_t>(host.size() * sizeof(T), 16)));
  h->owned.push_back(p);
  CUDA_TRY(cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = static_cast<T*>(p);
  return IEVM_OK;
}

// ----------------------------------------------------------------------------------------------
// Planning: shapes, channel pitches, tile configuration
// ----------------------------------------------------------------------------------------------
int plan_shapes(ievm_handle* h, const ievm_net_desc* nd) {
  int max_id = 0;
  for (int i = 0; i < nd->num_layers; ++i) {
    const ievm_layer_desc& d = nd->layers[i];
    max_id = std::max(max_id, std::max(d.in_tensor, std::max(d.res_tensor, d.out_tensor)));
  }
  h->tensors.assign(max_id + 1, TensorInfo());
  TensorInfo& t0 = h->tensors[0];
  t0.h = nd->in_h;
  t0.w = nd->in_w;
  t0.c = nd->in_c;
  if (h->dtype == IEVM_DTYPE_I8) {
    t0.pitch = 4;      // quantized NHWC4 inside a zero-point border (simt_kernels.cuh)
    t0.elem = 1;
    t0.hp = nd->in_h + kInPadH;
    t0.wp = nd->in_w + kInPadW;
    t0.pad_t = kInPadTop;
    t0.pad_l = kInPadLeft;
  } else {
    t0.pitch = nd->in_c;   // caller's f16 NCHW buffer is read in place by the stem
    t0.elem = 2;
  }
  h->layers.resize(nd->num_layers);
  for (int i = 0; i < nd->num_layers; ++i) {
    LayerPlan& L = h->layers[i];
    L.d = nd->layers[i];
    const ievm_layer_desc& d = L.d;
    if (d.in_tensor < 0 || d.in_tensor > max_id) return fail(IEVM_ERR_BAD_ARG, "layer %d: bad in_tensor", i);
    TensorInfo& tin = h->tensors[d.in_tensor];
    if (tin.h == 0) return fail(IEVM_ERR_BAD_ARG, "layer %d reads tensor %d before it is produced", i, d.in_tensor);
    tin.last_use = i;
    if (d.res_tensor >= 0) h->tensors[d.res_tensor].last_use = i;
    L.h = tin.h;
    L.w = tin.w;
    L.cin_pitch = tin.pitch;
    if (d.op == IEVM_OP_HEAD) {
      if (d.cin != tin.c) return fail(IEVM_ERR_BAD_ARG, "head: cin %d != producer channels %d", d.cin, tin.c);
      if (d.cout > kMaxClasses) return fail(IEVM_ERR_UNSUPPORTED, "head: more than %d classes", kMaxClasses);
      if (tin.pitch > kHeadSumWords) return fail(IEVM_ERR_UNSUPPORTED, "head: more than %d input channels", kHeadSumWords);
      continue;
    }
    if (d.out_tensor <= 0 || d.out_tensor > max_id || h->tensors[d.out_tensor].h != 0)
      return fail(IEVM_ERR_BAD_ARG, "layer %d: bad out_tensor", i);
    TensorInfo& tout = h->tensors[d.out_tensor];
    tout.producer = i;
    tout.elem = h->elem;
    if (d.op == IEVM_OP_MAXPOOL) {
      L.ho = (tin.h + 2 - 3) / 2 + 1;
      L.wo = (tin.w + 2 - 3) / 2 + 1;
      tout.h = L.ho;
      tout.w = L.wo;
      tout.c = tin.c;
      tout.pitch = tin.pitch;
      continue;
    }
    if (d.op == IEVM_OP_ADD_RELU) {
      if (h->dtype != IEVM_DTYPE_F16) return fail(IEVM_ERR_UNSUPPORTED, "layer %d: a stand-alone add_relu exists for F16 only "
                                                                       "(INT8: fused into the conv, res_tensor)", i);
      if (d.res_tensor < 0 || d.res_tensor > max_id) return fail(IEVM_ERR_BAD_ARG, "layer %d: add_relu needs res_tensor", i);
      const TensorInfo& tr = h->tensors[d.res_tensor];
      if (d.in_tensor == 0 || d.res_tensor == 0 || tr.h != tin.h || tr.w != tin.w || tr.c != tin.c || tr.pitch != tin.pitch ||
          tin.pitch % 8 != 0)
        return fail(IEVM_ERR_BAD_ARG, "layer %d: add_relu operands differ in shape", i);
      L.ho = tin.h;
      L.wo = tin.w;
      tout.h = tin.h;
      tout.w = tin.w;
      tout.c = tin.c;
      tout.pitch = tin.pitch;
      continue;
    }
    if (d.op != IEVM_OP_CONV) return fail(IEVM_ERR_BAD_ARG, "layer %d: unknown op %d", i, d.op);
    if (d.cin != tin.c) return fail(IEVM_ERR_BAD_ARG, "layer %d: cin %d != producer channels %d", i, d.cin, tin.c);
    L.ho = (tin.h + 2 * d.pad - d.ksize) / d.stride + 1;
    L.wo = (tin.w + 2 * d.pad - d.ksize) / d.stride + 1;
    L.n_tiles = (d.cout + 255) / 256;
    L.bn = round_up((d.cout + L.n_tiles - 1) / L.n_tiles, 16);
    L.cout_pad = L.n_tiles * L.bn;
    tout.h = L.ho;
    tout.w = L.wo;
    tout.c = d.cout;
    tout.pitch = L.cout_pad;
    L.is_stem = d.in_tensor == 0;
    if (L.is_stem) {
      if (d.cin != 3 || d.ksize != 7 || d.stride != 2 || d.pad != 3 || d.res_tensor >= 0 || L.n_tiles != 1)
        return fail(IEVM_ERR_UNSUPPORTED, "stem must be a 3-channel 7x7/2 pad-3 conv with <= 256 outputs");
      if (nd->in_w % 4 != 0 || nd->in_h % 2 != 0) return fail(IEVM_ERR_UNSUPPORTED, "input width must be a multiple of 4 and height even");
      continue;
    }
    if (!((d.ksize == 3 && d.pad == 1) || (d.ksize == 1 && d.pad == 0)) || d.stride < 1 || d.stride > 2)
      return fail(IEVM_ERR_UNSUPPORTED, "layer %d: only 3x3/pad1 and 1x1/pad0 convs with stride 1|2", i);
    if (d.res_tensor >= 0) {
      const TensorInfo& tr = h->tensors[d.res_tensor];
      if (tr.h != L.ho || tr.w != L.wo || tr.c != d.cout || tr.pitch != L.cout_pad)
        return fail(IEVM_ERR_BAD_ARG, "layer %d: residual shape mismatch", i);
    }
    const int row_bytes = L.cin_pitch * h->elem;
    constexpr int kMaxStages = 16;
    const int fixed = 1024 /*alignment slack*/ + 2 * L.cout_pad * 4 + (2 * kMaxStages + 2 * kMaxAcc + 1) * 8 + 16;
    const int avail = h->smem_optin - fixed;
    L.tmem_cols = 32;
    while (L.tmem_cols < 2 * L.bn) L.tmem_cols *= 2;
    // ---- halo (band) mode: 3x3 stride-1 convs whose pixel fits one shared-memory row, weights resident ----
    if (h->opt_halo && d.ksize == 3 && d.stride == 1 && d.pad == 1 && L.n_tiles == 1 && row_bytes <= 128 && L.w + 2 <= kTileM) {
      const int rb = row_bytes <= 64 ? 64 : 128;
      const int wp = L.w + 2;
      const int R = kTileM / wp;                        // whole output rows per sub-tile (row aligned)
      const int T = (L.h + R - 1) / R;
      int acc_stride = 32;
      while (acc_stride < L.bn) acc_stride *= 2;
      const int nacc = std::max(2, std::min(kMaxAcc, 512 / acc_stride));
      const int b_all = 9 * L.bn * rb;
      // Two CTAs per SM (two independent pipelines that fill each other's stalls) when weights + >= 2 patch stages fit in
      // half of the shared memory and the accumulators in half of TMEM: the 64-channel INT8 layers.
      if (h->opt_two_cta && h->dtype == IEVM_DTYPE_I8 && halo_shape_class(wp, rb, L.bn) == 1 && h->opt_halo_static) {
        const int half_smem = (h->smem_optin + 1024 /* per-CTA reservation */) / 2 - 1024 - 1024;
        const int nacc2 = std::max(2, std::min(kMaxAcc, 256 / acc_stride));
        const int S2 = std::max(1, std::min({kMaxBandSubs, nacc2 / 2, T}));
        const int a_stage2 = round_up((S2 * R + 2) * wp * rb, 1024);
        const int stages2 = std::min(8, (half_smem - fixed - b_all - 2048) / a_stage2);
        if (stages2 >= 2) {
          L.mode = kModeHalo;
          L.two_cta = 1;
          L.kc_bytes = rb;
          L.kc_elems = rb / h->elem;
          L.kchunks = 1;
          L.cin_w = L.kc_elems;
          L.wp = wp;
          L.sub_rows = R;
          L.subs_per_img = T;
          L.band_subs = S2;
          L.patch_rows = S2 * R + 2;
          L.a_tx_bytes = L.patch_rows * wp * rb;
          L.a_stage_bytes = a_stage2;
          L.resident_b = 1;
          L.stages = stages2;
          L.kb_group = 1;
          L.smem_bytes = static_cast<size_t>(L.stages) * a_stage2 + b_all + 2048 + fixed;
          continue;
        }
      }
      // largest band (sub-tiles per patch) that leaves the epilogue half of the accumulator ring and >= 2 patch stages
      int best_s = 0, best_stages = 0, best_stage_bytes = 0;
      for (int S = std::min({kMaxBandSubs, nacc / 2 > 0 ? nacc / 2 : 1, T}); S >= 1; --S) {
        const int a_tx = (S * R + 2) * wp * rb;
        const int a_stage = round_up(a_tx, 1024);
        // the last sub-tile's tap views run up to (130 - R * wp) rows past the patch: keep that much behind the last stage
        const int slack = round_up((130 - R * wp > 0 ? 130 - R * wp : 0) * rb, 1024);
        const int stages = std::min(8, (avail - b_all - slack) / a_stage);
        if (stages >= 2) {
          best_s = S;
          best_stages = stages;
          best_stage_bytes = a_stage;
          break;
        }
      }
      if (const char* e = getenv("IEVM_BAND_SUBS")) {     // diagnostics: force the band size
        const int S = std::max(1, std::min({atoi(e), kMaxBandSubs, nacc, T}));
        const int a_stage = round_up((S * R + 2) * wp * rb, 1024);
        const int stages = std::min(8, (avail - b_all - 2048) / a_stage);
        if (stages >= 2) {
          best_s = S;
          best_stages = stages;
          best_stage_bytes = a_stage;
        }
      }
      if (best_s > 0) {
        L.mode = kModeHalo;
        L.kc_bytes = rb;
        L.kc_elems = rb / h->elem;
        L.kchunks = 1;
        L.cin_w = L.kc_elems;
        L.wp = wp;
        L.sub_rows = R;
        L.subs_per_img = T;
        L.band_subs = best_s;
        L.patch_rows = best_s * R + 2;
        L.a_tx_bytes = L.patch_rows * wp * rb;
        L.a_stage_bytes = best_stage_bytes;
        L.resident_b = 1;
        L.stages = best_stages;
        L.kb_group = 1;
        L.smem_bytes = static_cast<size_t>(L.stages) * best_stage_bytes + b_all + 2048 + fixed;
        continue;
      }
    }
    // ---- im2col mode ----
    L.mode = kModeIm2col;
    L.kc_bytes = row_bytes <= 64 ? 64 : 128;
    L.kc_elems = L.kc_bytes / h->elem;
    L.kchunks = (d.cin * h->elem + L.kc_bytes - 1) / L.kc_bytes;
    L.cin_w = L.kchunks * L.kc_elems;
    {
      // N-tile width: the persistent grid runs ceil(tiles / #SMs) rounds of tiles, each costing about
      // (#k-blocks x k-steps) MMAs of max(bn/2, issue floor) cycles.  Narrower tiles waste less of the
      // last round (e.g. 7x7 layers: 98 M-tiles x 2 N-tiles on 148 SMs is 1.3 rounds, x 3 N-tiles is 2.0).
      const int num_kb_ = d.ksize * d.ksize * L.kchunks;
      const int ksteps = L.kc_bytes / 32;
      const long long m_tiles = (static_cast<long long>(h->max_batch) * L.ho * L.wo + kTileM - 1) / kTileM;
      long long best_cost = -1;
      int best_bn = L.bn, best_cluster = 1;
      for (int bn = 16; bn <= 256; bn += 16) {
        if (L.cout_pad % bn != 0) continue;
        const int ntl = L.cout_pad / bn;
        const bool resident = ntl == 1 && num_kb_ * bn * L.kc_bytes + 4 * kTileM * L.kc_bytes <= avail;
        for (int cl = 1; cl <= (h->opt_cluster && !resident ? 2 : 1); ++cl) {
          if (cl > 1 && ((bn / cl) % 8 != 0 || m_tiles < 2 * cl)) continue;
          const long long tiles = ((m_tiles + cl - 1) / cl) * ntl;              // cluster tiles
          const long long rounds = (tiles + h->num_sms / cl - 1) / (h->num_sms / cl);
          // a tile costs the slower of its MMAs (128 x bn x 32 B per instruction = bn/2 cycles) and the delivery of
          // its operands from L2 (measured ~40 B/clk/SM when every SM streams: layers 3-4 sit on this bound);
          // resident weights are loaded once, multicast splits the weight tile over the cluster
          const long long mma_cycles = static_cast<long long>(num_kb_) * ksteps * std::max(bn / 2, 24);
          const long long b_rows = resident ? 0 : bn / cl;
          const long long load_cycles = static_cast<long long>(num_kb_) * (kTileM + b_rows) * L.kc_bytes / 40;
          const long long tile_cycles = std::max(mma_cycles, load_cycles) + 600 + 6LL * bn;
          const long long cost = rounds * tile_cycles;
          if (best_cost < 0 || cost < best_cost || (cost == best_cost && bn > best_bn)) {
            best_cost = cost;
            best_bn = bn;
            best_cluster = cl;
          }
        }
      }
      if (!h->opt_fixed_bn) {
        L.bn = best_bn;
        L.cluster = best_cluster;
        L.n_tiles = L.cout_pad / L.bn;
        L.tmem_cols = 32;
        while (L.tmem_cols < 2 * L.bn) L.tmem_cols *= 2;
      }
    }
    // shared-memory plan: [A stages][B stages | all B k-blocks][epilogue tables][barriers]
    const int a_bytes = kTileM * L.kc_bytes;
    const int num_kb = d.ksize * d.ksize * L.kchunks;
    L.a_stage_bytes = L.a_tx_bytes = a_bytes;
    L.resident_b = (L.n_tiles == 1 && num_kb * L.bn * L.kc_bytes + 4 * a_bytes <= avail) ? 1 : 0;
    if (L.resident_b) L.cluster = 1;
    const int b_bytes = (L.bn / L.cluster) * L.kc_bytes;      // a pair CTA holds half of each weight k-block
    if (L.resident_b) L.stages = std::min(kMaxStages, (avail - num_kb * b_bytes) / a_bytes);
    else L.stages = std::min(kMaxStages, avail / (a_bytes + b_bytes));
    if (L.stages < 2) return fail(IEVM_ERR_UNSUPPORTED, "layer %d: tile does not fit in shared memory", i);
    // k-blocks per barrier pair: every mbarrier test by the MMA-issuing thread idles the tensor pipe for ~150 cycles
    // (conv_tc.cuh), so a stage is a GROUP of k-blocks -- the largest divisor of the k-block count (<= 4) that still
    // leaves three groups in flight
    {
      const int slots = L.stages;
      int G = 1;
      for (int g = 4; g >= 2; --g)
        if (num_kb % g == 0 && slots / g >= 3) {
          G = g;
          break;
        }
      if (const char* e = getenv("IEVM_KB_GROUP")) {
        const int g = atoi(e);
        if (g >= 1 && num_kb % g == 0 && slots / g >= 2) G = g;
      }
      L.kb_group = G;
      L.stages = slots / G;
    }
    L.smem_bytes = static_cast<size_t>(L.stages) * L.kb_group * a_bytes +
                   static_cast<size_t>(L.resident_b ? num_kb : L.stages * L.kb_group) * b_bytes + fixed;
  }
  // ---- dual launches (conv_dual.cuh): a 3x3 conv next to a 1x1 conv of the same stride on the same tensor (either order:
  // the FX graph of the INT8 module lists conv1 first, the FP16 flattening the downsample) ----
  for (size_t j = 0; j + 1 < 2 * h->layers.size(); ++j) {
    const size_t i = j / 2;
    if (i + 1 >= h->layers.size()) break;
    LayerPlan& P = h->layers[(j & 1) ? i + 1 : i];
    LayerPlan& D = h->layers[(j & 1) ? i : i + 1];
    const ievm_layer_desc& a = P.d;
    const ievm_layer_desc& b = D.d;
    if (P.dual_partner >= 0 || P.dual_of >= 0 || D.dual_partner >= 0 || D.dual_of >= 0) continue;
    if (a.op != IEVM_OP_CONV || b.op != IEVM_OP_CONV || P.is_stem || D.is_stem) continue;
    if (P.mode != kModeIm2col || D.mode != kModeIm2col || a.ksize != 3 || a.pad != 1 || b.ksize != 1 || b.pad != 0) continue;
    if (a.stride != b.stride || a.in_tensor != b.in_tensor || a.cout != b.cout || a.res_tensor >= 0 || b.res_tensor >= 0) continue;
    if (P.cout_pad != D.cout_pad || P.kc_bytes != D.kc_bytes || P.kchunks != D.kchunks) continue;
    if (h->dtype == IEVM_DTYPE_I8 && (a.in_zp != 0 || b.in_zp != 0)) continue;      // zero-point correction: separate launches
    constexpr int kMaxStages = 16;
    const int fixed2 = 1024 + 4 * P.cout_pad * 4 + (2 * kMaxStages + 2 * kMaxAcc + 1) * 8 + 16;
    const int avail2 = h->smem_optin - fixed2;
    // pixel-pair form: 64-byte pixels, stride 2, even width, weights resident
    const bool wide = h->dtype == IEVM_DTYPE_I8 && a.stride == 2 && P.kc_bytes == 64 && P.kchunks == 1 && P.cin_pitch == 64 &&
                      P.w % 2 == 0 && P.resident_b && P.cluster == 1 && h->opt_wide &&
                      (6 + 1) * P.bn * 128 + 4 * kTileM * 128 <= avail2;
    const int kcb = wide ? 128 : P.kc_bytes;
    const int a_bytes = kTileM * kcb;
    const int b_bytes = (P.bn / P.cluster) * kcb;
    const int num_kb = (wide ? 6 : 9) * P.kchunks;
    const int slots = P.resident_b ? std::min(kMaxStages, (avail2 - (num_kb + P.kchunks) * b_bytes) / a_bytes)
                                   : std::min(kMaxStages, avail2 / (a_bytes + b_bytes));
    if (slots < 2) continue;
    P.dual_wide = wide ? 1 : 0;
    // phase-patch form (conv_s2.cuh): 64-byte pixels, stride 2, one N tile of <= 128 channels, even input size
    if (h->opt_s2 && h->dtype == IEVM_DTYPE_I8 && a.stride == 2 && P.kc_bytes == 64 && P.kchunks == 1 && P.cin_pitch == 64 &&
        P.w % 2 == 0 && P.h % 2 == 0 && P.n_tiles == 1 && P.bn <= 128 && P.cluster == 1 && P.wo + 1 <= kTileM) {
      const int wp = P.wo + 1;
      const int R = kTileM / wp;
      const int pbytes = round_up((R + 1) * wp * 64, 1024);
      const int fixed_s2 = 1024 + 4 * P.cout_pad * 4 + (2 * kMaxStages + 2 * kMaxAcc + 1) * 8 + 16;
      const int stages = std::min(4, (h->smem_optin - fixed_s2 - 10 * P.bn * 64 - 1024) / (4 * pbytes));
      if (stages >= 2) {
        P.dual_s2 = 1;
        P.s2_rows = R;
        P.s2_phase_bytes = pbytes;
        P.s2_stages = stages;
        P.s2_smem_bytes = static_cast<size_t>(stages) * 4 * pbytes + 1024 + 10 * P.bn * 64 + fixed_s2;
      }
    }
    int G = 1;
    for (int g = 4; g >= 2; --g)
      if (num_kb % g == 0 && slots / g >= 3) {
        G = g;
        break;
      }
    P.dual_partner = static_cast<int>(&D - h->layers.data());
    D.dual_of = static_cast<int>(&P - h->layers.data());
    P.dual_kb_group = G;
    P.dual_stages = slots / G;
    P.dual_smem_bytes = static_cast<size_t>(P.dual_stages) * G * a_bytes +
                        static_cast<size_t>(P.resident_b ? num_kb + P.kchunks : P.dual_stages * G) * b_bytes + fixed2;
  }
  return IEVM_OK;
}

// ----------------------------------------------------------------------------------------------
// Weights and epilogue tables
// ----------------------------------------------------------------------------------------------
int upload_front2_weights(ievm_handle* h, LayerPlan& L);

int upload_conv_operands(ievm_handle* h, LayerPlan& L) {
  const ievm_layer_desc& d = L.d;
  const int taps = d.ksize * d.ksize;
  std::vector<float> ep0(L.cout_pad, 0.f), ep1(L.cout_pad, 0.f);
  if (h->dtype == IEVM_DTYPE_I8) {
    for (int c = 0; c < d.cout; ++c) {
      const float atw = d.in_scale * d.w_scale[c];
      ep0[c] = d.bias[c] / atw;
      ep1[c] = atw / d.out_scale;
    }
    // Magic-number rounding is exact while the value being rounded stays below 2^22 in magnitude.  Bound it over
    // every possible input: |acc| <= 255 * sum|w| (activations are u8, zero point 0 or a border of zero points).
    double vmax = 0.0;
    const int8_t* w = static_cast<const int8_t*>(d.weight);
    const size_t per_out = static_cast<size_t>(d.cin) * taps;
    for (int c = 0; c < d.cout; ++c) {
      double sw = 0.0;
      for (size_t i = 0; i < per_out; ++i) sw += std::abs(static_cast<int>(w[c * per_out + i]));
      vmax = std::max(vmax, (255.0 * sw + std::fabs(static_cast<double>(ep0[c]))) * std::fabs(static_cast<double>(ep1[c])));
    }
    if (d.res_tensor >= 0) vmax = std::max(vmax, 256.0 * (static_cast<double>(d.out_scale) + d.res_scale) / d.add_scale);
    L.fast_round = vmax < 2097152.0 ? 1 : 0;       // 2^21: a factor two of margin
    if (d.res_tensor >= 0 && d.relu) L.fast_round = 0;   // the fast fused add_relu assumes the conv's own lower clamp is 0
    if (const char* e = getenv("IEVM_FAST_ROUND")) L.fast_round = L.fast_round && atoi(e);
  } else {
    for (int c = 0; c < d.cout; ++c) ep0[c] = d.bias[c];
  }
  if (int rc = dev_upload(h, ep0, &L.ep0)) return rc;
  if (int rc = dev_upload(h, ep1, &L.ep1)) return rc;
  L.ep0_host = ep0;
  L.ep1_host = ep1;

  if (L.is_stem) {
    if (L.cout_pad == 64 && h->in_w == kF2W && h->in_h % 4 == 0 && h->in_h >= 8) {
      if (int rc = upload_front2_weights(h, L)) return rc;
      h->front2_ok = 1;
    }
    if (h->dtype == IEVM_DTYPE_I8) {
      const int8_t* w = static_cast<const int8_t*>(d.weight);     // [cout][3][7][7]
      std::vector<uint32_t> w4(static_cast<size_t>(49) * L.cout_pad, 0u);
      std::vector<int> wsum(L.cout_pad, 0);
      for (int co = 0; co < d.cout; ++co)
        for (int t = 0; t < 49; ++t) {
          uint32_t word = 0;
          for (int c = 0; c < 3; ++c) {
            const int8_t v = w[(static_cast<size_t>(co) * 3 + c) * 49 + t];
            word |= static_cast<uint32_t>(static_cast<uint8_t>(v)) << (8 * c);
            wsum[co] += v;
          }
          w4[static_cast<size_t>(t) * L.cout_pad + co] = word;
        }
      uint32_t* dw = nullptr;
      if (int rc = dev_upload(h, w4, &dw)) return rc;
      L.w_stem = dw;
      if (int rc = dev_upload(h, wsum, &L.wsum)) return rc;
      // tensor-core layout: K index = ky*32 + j*4 + c, window pixel j <-> kx = j - 1 (j = 0 is padding)
      std::vector<int8_t> wt(static_cast<size_t>(L.cout_pad) * kStemKBytes, 0);
      std::vector<int> zw(L.cout_pad, 0);
      for (int co = 0; co < d.cout; ++co) {
        for (int c = 0; c < 3; ++c)
          for (int ky = 0; ky < 7; ++ky)
            for (int kx = 0; kx < 7; ++kx)
              wt[static_cast<size_t>(co) * kStemKBytes + ky * 32 + (kx + 1) * 4 + c] =
                  w[(static_cast<size_t>(co) * 3 + c) * 49 + ky * 7 + kx];
        zw[co] = h->in_zp * wsum[co];
      }
      int8_t* dwt = nullptr;
      if (int rc = dev_upload(h, wt, &dwt)) return rc;
      L.w_stem_tc = dwt;
      if (int rc = dev_upload(h, zw, &L.zwsum)) return rc;
      L.tmem_cols = 32;
      while (L.tmem_cols < 2 * L.cout_pad) L.tmem_cols *= 2;
      L.stem_smem = 1024 + static_cast<size_t>(kStemStages) * 2 * kTileM * 128 + 2 * static_cast<size_t>(L.cout_pad) * 128 +
                    3 * static_cast<size_t>(L.cout_pad) * 4 + (2 * kStemStages + 5) * 8 + 16;
    } else {
      const uint16_t* w = static_cast<const uint16_t*>(d.weight);
      std::vector<uint16_t> ws(static_cast<size_t>(147) * L.cout_pad, 0);
      for (int co = 0; co < d.cout; ++co)
        for (int c = 0; c < 3; ++c)
          for (int t = 0; t < 49; ++t)
            ws[(static_cast<size_t>(t) * 3 + c) * L.cout_pad + co] = w[(static_cast<size_t>(co) * 3 + c) * 49 + t];
      uint16_t* dw = nullptr;
      if (int rc = dev_upload(h, ws, &dw)) return rc;
      L.w_stem = dw;
    }
    return IEVM_OK;
  }

  const size_t k_total = static_cast<size_t>(taps) * L.cin_w;
  if (h->dtype == IEVM_DTYPE_I8) {
    const int8_t* w = static_cast<const int8_t*>(d.weight);
    std::vector<int8_t> wp(static_cast<size_t>(L.cout_pad) * k_total, 0);
    for (int co = 0; co < d.cout; ++co)
      for (int ci = 0; ci < d.cin; ++ci)
        for (int t = 0; t < taps; ++t)
          wp[static_cast<size_t>(co) * k_total + static_cast<size_t>(t) * L.cin_w + ci] =
              w[(static_cast<size_t>(co) * d.cin + ci) * taps + t];
    int8_t* dw = nullptr;
    if (int rc = dev_upload(h, wp, &dw)) return rc;
    L.w_packed = dw;
    // pixel-pair form of the dual launch (conv_dual.cuh): a wide tap is 128 bytes = pixels (2j, 2j+1) x 64 channels
    if (L.dual_partner >= 0 && L.dual_wide) {
      // the 3x3: wide tap (ty, 0) = [unused pixel 2ox-2 | kx = 0], wide tap (ty, 1) = [kx = 1 | kx = 2]
      std::vector<int8_t> ww(static_cast<size_t>(L.cout_pad) * 6 * 128, 0);
      for (int co = 0; co < d.cout; ++co)
        for (int ci = 0; ci < d.cin; ++ci)
          for (int ky = 0; ky < 3; ++ky)
            for (int kx = 0; kx < 3; ++kx) {
              const int tx = kx == 0 ? 0 : 1, half = kx == 1 ? 0 : 1;
              ww[(static_cast<size_t>(co) * 6 + ky * 2 + tx) * 128 + half * 64 + ci] =
                  w[(static_cast<size_t>(co) * d.cin + ci) * 9 + ky * 3 + kx];
            }
      int8_t* dww = nullptr;
      if (int rc = dev_upload(h, ww, &dww)) return rc;
      L.w_wide = dww;
    }
    if (L.dual_of >= 0 && h->layers[L.dual_of].dual_wide) {
      // the 1x1 downsample: pixel (2oy, 2ox) = first half of wide tap (1, 1)
      std::vector<int8_t> ww(static_cast<size_t>(L.cout_pad) * 128, 0);
      for (int co = 0; co < d.cout; ++co)
        for (int ci = 0; ci < d.cin; ++ci) ww[static_cast<size_t>(co) * 128 + ci] = w[static_cast<size_t>(co) * d.cin + ci];
      int8_t* dww = nullptr;
      if (int rc = dev_upload(h, ww, &dww)) return rc;
      L.w_wide = dww;
    }
    if (d.in_zp != 0) {
      // border-aware zero-point correction (ConvTcParams::zcorr): class = (row-tap mask << k) | column-tap mask
      const int k = d.ksize, ncls = 1 << (2 * k);
      std::vector<int32_t> w2(static_cast<size_t>(d.cout) * taps, 0);           // sum over input channels per tap
      for (int co = 0; co < d.cout; ++co)
        for (int ci = 0; ci < d.cin; ++ci)
          for (int t = 0; t < taps; ++t) w2[static_cast<size_t>(co) * taps + t] += w[(static_cast<size_t>(co) * d.cin + ci) * taps + t];
      std::vector<int32_t> tab(static_cast<size_t>(ncls) * L.cout_pad, 0);
      for (int cls = 0; cls < ncls; ++cls) {
        const int my = cls >> k, mx = cls & ((1 << k) - 1);
        for (int co = 0; co < d.cout; ++co) {
          int32_t sum = 0;
          for (int ty = 0; ty < k; ++ty)
            for (int tx = 0; tx < k; ++tx)
              if (((my >> ty) & 1) && ((mx >> tx) & 1)) sum += w2[static_cast<size_t>(co) * taps + ty * k + tx];
          tab[static_cast<size_t>(cls) * L.cout_pad + co] = d.in_zp * sum;
        }
      }
      if (int rc = dev_upload(h, tab, &L.zcorr)) return rc;
    }
  } else {
    const uint16_t* w = static_cast<const uint16_t*>(d.weight);
    std::vector<uint16_t> wp(static_cast<size_t>(L.cout_pad) * k_total, 0);
    for (int co = 0; co < d.cout; ++co)
      for (int ci = 0; ci < d.cin; ++ci)
        for (int t = 0; t < taps; ++t)
          wp[static_cast<size_t>(co) * k_total + static_cast<size_t>(t) * L.cin_w + ci] =
              w[(static_cast<size_t>(co) * d.cin + ci) * taps + t];
    uint16_t* dw = nullptr;
    if (int rc = dev_upload(h, wp, &dw)) return rc;
    L.w_packed = dw;
  }
  return IEVM_OK;
}

// Weight operand of frontend_v2.cuh: A[m][k], m = 64 * r + cout (r = which of the tile's two stem rows),
// K bytes = line s (0 .. kSegs-1) x 64: record j (0..3) x 16 bytes; stored row-major [128][kSegs * 64] (the kernel
// copies it into tensor memory, one row per lane).
//   INT8: record byte = rp * 6 + cp * 3 + c, line s = input row pair: ky = 2 * (s - r) + rp - 1, kx = 2 * j + cp - 1
//   FP16: record half = cp * 3 + c,          line s = input row:      ky = s - 2 * r,             kx = 2 * j + cp - 1
int upload_front2_weights(ievm_handle* h, LayerPlan& L) {
  const ievm_layer_desc& d = L.d;
  const bool i8 = h->dtype == IEVM_DTYPE_I8;
  const int segs = i8 ? F2Cfg<kDtypeI8>::kSegs : F2Cfg<kDtypeF16>::kSegs;
  const int abytes = i8 ? F2Cfg<kDtypeI8>::kABytes : F2Cfg<kDtypeF16>::kABytes;
  std::vector<uint8_t> img(abytes, 0);
  const int row_bytes = abytes / 128;
  auto at = [&](int m, int kb) -> uint8_t* { return &img[static_cast<size_t>(m) * row_bytes + kb]; };
  for (int r = 0; r < 2; ++r)
    for (int co = 0; co < d.cout; ++co)
      for (int s = 0; s < segs; ++s)
        for (int j = 0; j < 4; ++j)
          for (int cp = 0; cp < 2; ++cp)
            for (int c = 0; c < 3; ++c) {
              const int kx = 2 * j + cp - 1;
              if (kx < 0 || kx > 6) continue;
              if (i8) {
                for (int rp = 0; rp < 2; ++rp) {
                  const int ky = 2 * (s - r) + rp - 1;
                  if (ky < 0 || ky > 6) continue;
                  const int8_t v = static_cast<const int8_t*>(d.weight)[(static_cast<size_t>(co) * 3 + c) * 49 + ky * 7 + kx];
                  *at(64 * r + co, s * 64 + j * 16 + rp * 6 + cp * 3 + c) = static_cast<uint8_t>(v);
                }
              } else {
                const int ky = s - 2 * r;
                if (ky < 0 || ky > 6) continue;
                const uint16_t v = static_cast<const uint16_t*>(d.weight)[(static_cast<size_t>(co) * 3 + c) * 49 + ky * 7 + kx];
                uint8_t* dst = at(64 * r + co, s * 64 + j * 16 + (cp * 3 + c) * 2);
                dst[0] = static_cast<uint8_t>(v & 0xff);
                dst[1] = static_cast<uint8_t>(v >> 8);
              }
            }
  uint8_t* dw = nullptr;
  if (int rc = dev_upload(h, img, &dw)) return rc;
  L.w_front2 = dw;
  return IEVM_OK;
}

int upload_head_operands(ievm_handle* h, LayerPlan& L) {
  const ievm_layer_desc& d = L.d;
  std::vector<float> ep0(kMaxClasses, 0.f), ep1(kMaxClasses, 0.f);
  if (h->dtype == IEVM_DTYPE_I8) {
    for (int c = 0; c < d.cout; ++c) {
      const float atw = d.in_scale * d.w_scale[c];
      ep0[c] = d.bias[c] / atw;
      ep1[c] = atw / d.out_scale;
    }
    const int8_t* w = static_cast<const int8_t*>(d.weight);   // [classes][cin]
    std::vector<int8_t> wp(static_cast<size_t>(d.cout) * L.cin_pitch, 0);
    for (int o = 0; o < d.cout; ++o)
      for (int c = 0; c < d.cin; ++c) wp[static_cast<size_t>(o) * L.cin_pitch + c] = w[static_cast<size_t>(o) * d.cin + c];
    int8_t* dw = nullptr;
    if (int rc = dev_upload(h, wp, &dw)) return rc;
    L.w_packed = dw;
  } else {
    for (int c = 0; c < d.cout; ++c) ep0[c] = d.bias[c];
    const uint16_t* w = static_cast<const uint16_t*>(d.weight);
    std::vector<uint16_t> wp(static_cast<size_t>(d.cout) * L.cin_pitch, 0);
    for (int o = 0; o < d.cout; ++o)
      for (int c = 0; c < d.cin; ++c) wp[static_cast<size_t>(o) * L.cin_pitch + c] = w[static_cast<size_t>(o) * d.cin + c];
    uint16_t* dw = nullptr;
    if (int rc = dev_upload(h, wp, &dw)) return rc;
    L.w_packed = dw;
  }
  if (int rc = dev_upload(h, ep0, &L.ep0)) return rc;
  if (int rc = dev_upload(h, ep1, &L.ep1)) return rc;
  return IEVM_OK;
}

// ----------------------------------------------------------------------------------------------
// Workspace: greedy buffer reuse by liveness (or one buffer per tensor with keep_tensors)
// ----------------------------------------------------------------------------------------------
bool front_end_is_chunked(const ievm_handle* h);
bool front_end_is_v2(const ievm_handle* h);

int assign_buffers(ievm_handle* h) {
  for (void* b : h->buffers) cudaFree(b);
  h->buffers.clear();
  h->buffer_bytes.clear();
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
  h->graphs.clear();
  std::vector<size_t> need;          // planned size per buffer
  std::vector<int> free_list;
  const bool f16 = h->dtype == IEVM_DTYPE_F16;
  // best fit: the smallest free buffer that is already big enough, else grow the largest free one
  auto take = [&](size_t bytes) {
    int best = -1;
    if (!h->keep_tensors) {
      for (size_t i = 0; i < free_list.size(); ++i) {
        if (best < 0) { best = static_cast<int>(i); continue; }
        const size_t cur = need[free_list[best]], cand = need[free_list[i]];
        const bool cur_fits = cur >= bytes, cand_fits = cand >= bytes;
        if ((cand_fits && (!cur_fits || cand < cur)) || (!cand_fits && !cur_fits && cand > cur)) best = static_cast<int>(i);
      }
    }
    if (best >= 0) {
      const int b = free_list[best];
      free_list.erase(free_list.begin() + best);
      need[b] = std::max(need[b], bytes);
      return b;
    }
    need.push_back(bytes);
    return static_cast<int>(need.size()) - 1;
  };
  for (auto& t : h->tensors) t.buffer = -1;
  const bool chunked = front_end_is_chunked(h);
  const size_t front_imgs = chunked ? static_cast<size_t>(std::min(h->max_batch, h->front_chunk)) : h->max_batch;
  if (!f16) h->tensors[0].buffer = take(h->tensors[0].bytes_per_image() * front_imgs);
  for (size_t i = 0; i < h->layers.size(); ++i) {
    const LayerPlan& L = h->layers[i];
    if (L.d.op != IEVM_OP_HEAD) {
      TensorInfo& t = h->tensors[L.d.out_tensor];
      if (t.buffer < 0)
        t.buffer = take(t.bytes_per_image() * ((chunked && i == 0) ? front_imgs : static_cast<size_t>(h->max_batch)));
      // a dual launch (conv_dual.cuh) writes both convs' outputs at the position of the first of the two
      const int mate = L.dual_partner >= 0 ? L.dual_partner : L.dual_of;
      if (mate > static_cast<int>(i)) {
        TensorInfo& tm = h->tensors[h->layers[mate].d.out_tensor];
        tm.buffer = take(tm.bytes_per_image() * static_cast<size_t>(h->max_batch));
      }
    }
    if (!h->keep_tensors)
      for (size_t ti = (f16 ? 0 : 1); ti < h->tensors.size(); ++ti) {   // the INT8 input keeps its bordered buffer
        const TensorInfo& t = h->tensors[ti];
        if (t.buffer >= 0 && t.last_use == static_cast<int>(i)) free_list.push_back(t.buffer);
      }
  }
  for (size_t b = 0; b < need.size(); ++b) {
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, need[b] + 256));
    const int fill = (!f16 && static_cast<int>(b) == h->tensors[0].buffer) ? h->in_zp : 0;   // zero-point border
    CUDA_TRY(cudaMemset(p, fill, need[b] + 256));
    h->buffers.push_back(p);
    h->buffer_bytes.push_back(need[b]);
  }
  return IEVM_OK;
}

void* tensor_ptr(const ievm_handle* h, int id) {
  const int b = h->tensors[id].buffer;
  return b < 0 ? nullptr : h->buffers[b];
}

int encode_maps(ievm_handle* h) {
  const CUtensorMapDataType dt = h->dtype == IEVM_DTYPE_I8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  for (size_t i = 0; i < h->layers.size(); ++i) {
    LayerPlan& L = h->layers[i];
    if (L.d.op == IEVM_OP_CONV && L.is_stem && h->dtype == IEVM_DTYPE_I8) {
      cuuint64_t dims[2] = {static_cast<cuuint64_t>(kStemKBytes), static_cast<cuuint64_t>(L.cout_pad)};
      cuuint64_t strides[1] = {static_cast<cuuint64_t>(kStemKBytes)};
      cuuint32_t box[2] = {128, static_cast<cuuint32_t>(L.cout_pad)};
      cuuint32_t estr[2] = {1, 1};
      const CUresult r = g_encode_tiled(&L.tmap_b, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, L.w_stem_tc, dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled failed for the stem: CUresult %d", (int)r);
      continue;
    }
    if (L.d.op != IEVM_OP_CONV || L.is_stem) continue;
    const CUtensorMapSwizzle sw = L.kc_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const size_t e = h->elem;
    if (L.mode == kModeHalo) {
      cuuint64_t dims[4] = {static_cast<cuuint64_t>(L.cin_pitch), static_cast<cuuint64_t>(L.w),
                            static_cast<cuuint64_t>(L.h), static_cast<cuuint64_t>(h->max_batch)};
      cuuint64_t strides[3] = {L.cin_pitch * e, static_cast<cuuint64_t>(L.w) * L.cin_pitch * e,
                               static_cast<cuuint64_t>(L.h) * L.w * L.cin_pitch * e};
      cuuint32_t box[4] = {static_cast<cuuint32_t>(L.kc_elems), static_cast<cuuint32_t>(L.wp),
                           static_cast<cuuint32_t>(L.patch_rows), 1};
      cuuint32_t estr[4] = {1, 1, 1, 1};
      const CUresult r = g_encode_tiled(&L.tmap_a, dt, 4, tensor_ptr(h, L.d.in_tensor), dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled (halo patch) failed for layer %zu: CUresult %d", i, (int)r);
    } else
    // activations as (C, W, H, N), im2col mode
    {
      cuuint64_t dims[4] = {static_cast<cuuint64_t>(L.cin_pitch), static_cast<cuuint64_t>(L.w),
                            static_cast<cuuint64_t>(L.h), static_cast<cuuint64_t>(h->max_batch)};
      cuuint64_t strides[3] = {L.cin_pitch * e, static_cast<cuuint64_t>(L.w) * L.cin_pitch * e,
                               static_cast<cuuint64_t>(L.h) * L.w * L.cin_pitch * e};
      int lower[2] = {-L.d.pad, -L.d.pad};
      int upper[2] = {L.d.pad - (L.d.ksize - 1), L.d.pad - (L.d.ksize - 1)};
      cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(L.d.stride), static_cast<cuuint32_t>(L.d.stride), 1};
      const CUresult r = g_encode_im2col(&L.tmap_a, dt, 4, tensor_ptr(h, L.d.in_tensor), dims, strides, lower, upper,
                                         static_cast<cuuint32_t>(L.kc_elems), kTileM, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeIm2col failed for layer %zu: CUresult %d", i, (int)r);
    }
    // packed weights as (K_total, cout_pad), tiled mode
    {
      const size_t k_total = static_cast<size_t>(L.d.ksize) * L.d.ksize * L.cin_w;
      cuuint64_t dims[2] = {k_total, static_cast<cuuint64_t>(L.cout_pad)};
      cuuint64_t strides[1] = {k_total * e};
      cuuint32_t box[2] = {static_cast<cuuint32_t>(L.kc_elems), static_cast<cuuint32_t>(L.bn / L.cluster)};
      cuuint32_t estr[2] = {1, 1};
      const CUresult r = g_encode_tiled(&L.tmap_b, dt, 2, L.w_packed, dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled failed for layer %zu: CUresult %d", i, (int)r);
    }
    if (L.dual_partner >= 0 && L.dual_s2) {
      // phase patches (conv_s2.cuh): a tiled box that walks W and H with traversal stride 2 -- (R + 1) x (W_out + 1) pixels of
      // one phase of the input, landing densely in shared memory
      cuuint64_t dims[4] = {static_cast<cuuint64_t>(L.cin_pitch), static_cast<cuuint64_t>(L.w), static_cast<cuuint64_t>(L.h),
                            static_cast<cuuint64_t>(h->max_batch)};
      cuuint64_t strides[3] = {L.cin_pitch * e, static_cast<cuuint64_t>(L.w) * L.cin_pitch * e,
                               static_cast<cuuint64_t>(L.h) * L.w * L.cin_pitch * e};
      cuuint32_t box[4] = {64, static_cast<cuuint32_t>(2 * (L.wo + 1)), static_cast<cuuint32_t>(2 * (L.s2_rows + 1)), 1};
      cuuint32_t estr[4] = {1, 2, 2, 1};
      const CUresult r = g_encode_tiled(&L.tmap_a_s2, dt, 4, tensor_ptr(h, L.d.in_tensor), dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled (phase patches) failed for layer %zu: CUresult %d", i, (int)r);
      const LayerPlan& D = h->layers[L.dual_partner];       // the downsample's weights, 64-byte rows, this layer's N tile
      cuuint64_t ddims[2] = {static_cast<cuuint64_t>(D.cin_w), static_cast<cuuint64_t>(D.cout_pad)};
      cuuint64_t dstr[1] = {D.cin_w * e};
      cuuint32_t dbox[2] = {64, static_cast<cuuint32_t>(L.bn)};
      cuuint32_t destr[2] = {1, 1};
      const CUresult r2 = g_encode_tiled(&L.tmap_b2_s2, dt, 2, D.w_packed, ddims, dstr, dbox, destr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                         CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r2 != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled (phase-patch downsample weights) failed for layer %zu: CUresult %d", i, (int)r2);
    }
    if (L.dual_partner >= 0 && L.dual_wide) {
      // pixel-pair form: the input as (128 B wide pixels, W / 2, H, N); 3 x 2 taps, stride (1, 2), padding left / top 1
      const LayerPlan& D = h->layers[L.dual_partner];
      cuuint64_t dims[4] = {128, static_cast<cuuint64_t>(L.w / 2), static_cast<cuuint64_t>(L.h), static_cast<cuuint64_t>(h->max_batch)};
      cuuint64_t strides[3] = {128, static_cast<cuuint64_t>(L.w) * L.cin_pitch, static_cast<cuuint64_t>(L.h) * L.w * L.cin_pitch};
      int lower[2] = {-1, -1};
      int upper[2] = {-1, -1};              // W: no right padding, 2 taps; H: padding 1, 3 taps
      cuuint32_t estr[4] = {1, 1, 2, 1};
      CUresult r = g_encode_im2col(&L.tmap_a_wide, dt, 4, tensor_ptr(h, L.d.in_tensor), dims, strides, lower, upper, 128, kTileM,
                                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeIm2col (pixel pairs) failed for layer %zu: CUresult %d", i, (int)r);
      cuuint32_t westr[2] = {1, 1};
      cuuint32_t wbox[2] = {128, static_cast<cuuint32_t>(L.bn)};
      cuuint64_t wdims[2] = {6 * 128, static_cast<cuuint64_t>(L.cout_pad)};
      cuuint64_t wstr[1] = {6 * 128};
      r = g_encode_tiled(&L.tmap_b_wide, dt, 2, L.w_wide, wdims, wstr, wbox, westr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r == CUDA_SUCCESS) {
        cuuint64_t ddims[2] = {128, static_cast<cuuint64_t>(D.cout_pad)};
        cuuint64_t dstr[1] = {128};
        r = g_encode_tiled(&L.tmap_b2, dt, 2, D.w_wide, ddims, dstr, wbox, westr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      }
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled (pixel-pair weights) failed for layer %zu: CUresult %d", i, (int)r);
    } else if (L.dual_partner >= 0) {
      // the downsample's packed weights (one tap) read with THIS layer's N-tile box
      const LayerPlan& D = h->layers[L.dual_partner];
      const size_t k_total = D.cin_w;
      cuuint64_t dims[2] = {k_total, static_cast<cuuint64_t>(D.cout_pad)};
      cuuint64_t strides[1] = {k_total * e};
      cuuint32_t box[2] = {static_cast<cuuint32_t>(L.kc_elems), static_cast<cuuint32_t>(L.bn / L.cluster)};
      cuuint32_t estr[2] = {1, 1};
      const CUresult r = g_encode_tiled(&L.tmap_b2, dt, 2, D.w_packed, dims, strides, box, estr,
                                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled (dual weights) failed for layer %zu: CUresult %d", i, (int)r);
    }
  }
  return IEVM_OK;
}

// ----------------------------------------------------------------------------------------------
// Launch helpers
// ----------------------------------------------------------------------------------------------
ConvTcParams make_conv_params(const ievm_handle* h, const LayerPlan& L, int n, int32_t* dump_acc) {
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  const ievm_layer_desc& d = L.d;
  p.m_total = n * L.ho * L.wo;
  p.ho = L.ho;
  p.wo = L.wo;
  p.stride = d.stride;
  p.pad = d.pad;
  p.ksize = d.ksize;
  p.kchunks = L.kchunks;
  p.kc_bytes = L.kc_bytes;
  p.kc_elems = L.kc_elems;
  p.bn = L.bn;
  p.n_tiles = L.n_tiles;
  p.m_tiles = L.mode == kModeHalo ? n * L.subs_per_img : (p.m_total + kTileM - 1) / kTileM;
  p.stages = L.stages;
  p.resident_b = L.resident_b;
  p.a_stage_bytes = L.a_stage_bytes;
  p.a_tx_bytes = L.a_tx_bytes;
  p.kb_group = L.kb_group;
  p.h_in = L.h;
  p.w_in = L.w;
  p.wp = L.wp;
  p.sub_rows = L.sub_rows;
  p.sub_pos = L.sub_rows * L.wp;
  p.subs_per_img = L.subs_per_img;
  p.band_subs = L.band_subs;
  p.total_subs = n * L.subs_per_img;
  // magic(d, n_max): ceil(2^32 / d) when every dividend n <= n_max satisfies n * d < 2^32, else 0 (plain division)
  auto magic = [](long long d, long long n_max) {
    return (d > 1 && n_max * d < 0x100000000ll) ? static_cast<uint32_t>((0x100000000ull + d - 1) / d) : 0u;
  };
  p.spi_magic = magic(L.subs_per_img, static_cast<long long>(n) * L.subs_per_img);
  p.wp_magic = magic(L.wp, kTileM);
  p.hw_magic = magic(static_cast<long long>(L.ho) * L.wo, static_cast<long long>(p.m_total) + 4 * kTileM);
  p.wo_magic = magic(L.wo, static_cast<long long>(L.ho) * L.wo);
  p.cout_pad = L.cout_pad;
  // accumulator ring: buffers a power-of-two number of columns apart, as many as TMEM's 512 columns hold (<= 8)
  p.acc_stride = 32;
  while (p.acc_stride < L.bn) p.acc_stride *= 2;
  p.nacc = std::max(2, std::min(kMaxAcc, (L.two_cta ? 256 : 512) / p.acc_stride));
  p.tmem_cols = p.nacc * p.acc_stride;
  p.fast_round = L.fast_round;
  const int mma_m = L.cluster > 1 ? 256 : 128;             // a CTA pair issues M = 256 instructions
  p.idesc = h->dtype == IEVM_DTYPE_I8 ? make_idesc_i8_u8s8(L.bn, mma_m) : make_idesc_f16(L.bn, mma_m);
  p.out = tensor_ptr(h, d.out_tensor);
  p.out_pitch = L.cout_pad;
  p.res = d.res_tensor >= 0 ? tensor_ptr(h, d.res_tensor) : nullptr;
  p.res_pitch = L.cout_pad;
  p.ep0 = L.ep0;
  p.ep1 = L.ep1;
  p.out_zp = d.out_zp;
  p.out_lo = d.relu ? d.out_zp : 0;
  p.a_scale = d.out_scale;
  p.res_scale = d.res_scale;
  p.res_zp = d.res_zp;
  p.inv_add_scale = d.res_tensor >= 0 ? 1.0f / d.add_scale : 0.f;
  p.add_zp = d.add_zp;
  p.relu = d.relu;
  p.zcorr = L.zcorr;
  p.dump_acc = dump_acc;
  p.dump_pitch = L.cout_pad;
  p.stuck_flag = h->stuck_dev;
  if (L.cout_pad <= kEpConst && !L.ep0_host.empty()) {
    memcpy(p.epc0, L.ep0_host.data(), L.cout_pad * sizeof(float));
    memcpy(p.epc1, L.ep1_host.data(), L.cout_pad * sizeof(float));
  }
#ifdef IEVM_EXP_TIMING
  p.timing_slot = static_cast<int>(&L - h->layers.data()) % kExpSlots;
#endif
  return p;
}

int launch_conv(ievm_handle* h, const LayerPlan& L, int n, cudaStream_t s, int32_t* dump_acc) {
  ConvTcParams p = make_conv_params(h, L, n, dump_acc);
  // Small batches: when no CTA of a halo layer gets more than one sub-tile, the accumulator ring is pointless and three
  // of the four epilogue groups would idle.  One accumulator instead: all sixteen epilogue warps drain the one tile
  // together (four per TMEM lane quadrant, interleaving 16-column chunks; the run-time-shaped kernel does that).
  const bool tiny = h->opt_tiny && L.mode == kModeHalo && h->conv_impl == 0 && p.total_subs <= h->num_sms;
  if (tiny) {
    p.nacc = 1;
    p.band_subs = 1;
    p.tmem_cols = std::max(32, p.acc_stride);
  }
  if (h->conv_impl == 1) {
    ConvDirectParams g;
    g.n = n; g.h = L.h; g.w = L.w; g.ho = L.ho; g.wo = L.wo;
    g.cin_pitch = L.cin_pitch; g.cin_w = L.cin_w; g.cin_real = L.d.cin; g.cout_pad = L.cout_pad;
    g.ksize = L.d.ksize; g.stride = L.d.stride; g.pad = L.d.pad;
    g.in_zp = h->dtype == IEVM_DTYPE_I8 ? L.d.in_zp : 0;
    const long long total = static_cast<long long>(p.m_total) * L.cout_pad;
    const unsigned blocks = static_cast<unsigned>((total + 127) / 128);
    if (h->dtype == IEVM_DTYPE_I8)
      conv_direct_i8_kernel<<<blocks, 128, 0, s>>>(static_cast<const uint8_t*>(tensor_ptr(h, L.d.in_tensor)),
                                                   static_cast<const int8_t*>(L.w_packed),
                                                   static_cast<uint8_t*>(p.out), g, p);
    else
      conv_direct_f16_kernel<<<blocks, 128, 0, s>>>(static_cast<const __half*>(tensor_ptr(h, L.d.in_tensor)),
                                                    static_cast<const __half*>(L.w_packed), g, p);
    CUDA_TRY(cudaGetLastError());
    return IEVM_OK;
  }
  const bool has_res = p.res != nullptr;
  const unsigned cl = static_cast<unsigned>(L.cluster);
  int grid = std::min(p.m_tiles * p.n_tiles, h->num_sms);
  if (cl > 1) {
    const int cluster_tiles = ((p.m_tiles + L.cluster - 1) / L.cluster) * p.n_tiles;
    grid = std::min(cluster_tiles, L.max_clusters > 0 ? L.max_clusters : h->num_sms / L.cluster) * L.cluster;
  }
#define IEVM_LAUNCH(DT, RES, MODE, CL, SH) \
  CUDA_TRY(launch_kernel_cluster(conv_tc_kernel<DT, RES, MODE, CL, SH>, grid, kConvThreads, L.smem_bytes, s, h->opt_pdl != 0, \
                                 static_cast<unsigned>(CL), L.tmap_a, L.tmap_b, p))
#define IEVM_LAUNCH_MODE(DT, RES, SH_A, SH_B)                              \
  do {                                                                     \
    if (L.mode == kModeHalo) {                                             \
      if (shape == SH_A) IEVM_LAUNCH(DT, RES, kModeHalo, 1, SH_A);         \
      else if (shape == SH_B) IEVM_LAUNCH(DT, RES, kModeHalo, 1, SH_B);    \
      else IEVM_LAUNCH(DT, RES, kModeHalo, 1, 0);                          \
    } else if (cl == 2) IEVM_LAUNCH(DT, RES, kModeIm2col, 2, 0);           \
    else IEVM_LAUNCH(DT, RES, kModeIm2col, 1, 0);                          \
  } while (0)
  // the shape-specialised kernels assume a zero input zero point (true for every post-ReLU tensor); others take class 0
  const int shape = (L.mode == kModeHalo && h->opt_halo_static && L.zcorr == nullptr && !tiny) ? halo_shape_class(L.wp, L.kc_bytes, L.bn) : 0;
  if (L.zcorr != nullptr && h->dtype == IEVM_DTYPE_I8) {
    // non-zero input zero point: the run-time-shaped kernels with the border-aware correction compiled in
#define IEVM_LAUNCH_ZC(RES, MODE, CL)                                                                                        \
  CUDA_TRY(launch_kernel_cluster(conv_tc_kernel<kDtypeI8, RES, MODE, CL, 0, kEpiWarps, true>, grid, kConvThreads, L.smem_bytes, s, \
                                 h->opt_pdl != 0, static_cast<unsigned>(CL), L.tmap_a, L.tmap_b, p))
    if (L.mode == kModeHalo) {
      if (has_res) IEVM_LAUNCH_ZC(true, kModeHalo, 1); else IEVM_LAUNCH_ZC(false, kModeHalo, 1);
    } else if (cl == 2) {
      if (has_res) IEVM_LAUNCH_ZC(true, kModeIm2col, 2); else IEVM_LAUNCH_ZC(false, kModeIm2col, 2);
    } else {
      if (has_res) IEVM_LAUNCH_ZC(true, kModeIm2col, 1); else IEVM_LAUNCH_ZC(false, kModeIm2col, 1);
    }
#undef IEVM_LAUNCH_ZC
    CUDA_TRY(cudaGetLastError());
    return IEVM_OK;
  }
  if (L.two_cta && shape == 1 && h->dtype == IEVM_DTYPE_I8) {
    const int grid2 = std::min(p.m_tiles, 2 * h->num_sms);
    if (has_res)
      CUDA_TRY(launch_kernel_cluster(conv_tc_kernel<kDtypeI8, true, kModeHalo, 1, 1, 8>, grid2, 64 + 32 * 8, L.smem_bytes, s,
                                     h->opt_pdl != 0, 1u, L.tmap_a, L.tmap_b, p));
    else
      CUDA_TRY(launch_kernel_cluster(conv_tc_kernel<kDtypeI8, false, kModeHalo, 1, 1, 8>, grid2, 64 + 32 * 8, L.smem_bytes, s,
                                     h->opt_pdl != 0, 1u, L.tmap_a, L.tmap_b, p));
    CUDA_TRY(cudaGetLastError());
    return IEVM_OK;
  }
  if (h->dtype == IEVM_DTYPE_I8) {
    if (has_res) IEVM_LAUNCH_MODE(kDtypeI8, true, 1, 2); else IEVM_LAUNCH_MODE(kDtypeI8, false, 1, 2);
  } else {
    if (has_res) IEVM_LAUNCH_MODE(kDtypeF16, true, 3, 3); else IEVM_LAUNCH_MODE(kDtypeF16, false, 3, 3);
  }
#undef IEVM_LAUNCH_MODE
#undef IEVM_LAUNCH
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

// Are the 1x1 downsample convs computed inside their block's first 3x3 launch (conv_dual.cuh)?
bool dual_active(const ievm_handle* h) { return h->opt_dual && h->conv_impl == 0; }

// Layer P (3x3) and its partner (the block's 1x1 downsample) in one launch; dump0 / dump1: debug accumulators per class.
int launch_conv_dual(ievm_handle* h, const LayerPlan& P, int n, cudaStream_t s, int32_t* dump0, int32_t* dump1) {
  const LayerPlan& D = h->layers[P.dual_partner];
  ConvTcParams p = make_conv_params(h, P, n, dump0);
  p.stages = P.dual_stages;
  p.kb_group = P.dual_kb_group;
  if (P.dual_wide && !P.dual_s2) {          // pixel-pair form: 128-byte wide pixels, 3 x 2 taps, stride (2, 1), left padding 1
    p.kc_bytes = 128;
    p.kc_elems = 128;
    p.kchunks = 1;
    p.a_stage_bytes = p.a_tx_bytes = kTileM * 128;
    p.kw = 2;
    p.stride_w = 1;
    p.pad_w = 1;
  }
  ConvDualParams x;
  memset(&x, 0, sizeof(x));
  x.out = tensor_ptr(h, D.d.out_tensor);
  x.ep0 = D.ep0;
  x.ep1 = D.ep1;
  x.out_zp = D.d.out_zp;
  x.out_lo = D.d.relu ? D.d.out_zp : 0;
  x.fast_round = D.fast_round;
  x.relu = D.d.relu;
  x.dump_acc = dump1;
  if (D.cout_pad <= kEpConst && !D.ep0_host.empty()) {
    memcpy(x.epc0, D.ep0_host.data(), D.cout_pad * sizeof(float));
    memcpy(x.epc1, D.ep1_host.data(), D.cout_pad * sizeof(float));
  }
  if (P.dual_s2) {
    // phase-patch form (conv_s2.cuh): sub-tiles of R output rows, four stride-1 phase patches per sub-tile
    const int wp = P.wo + 1, R = P.s2_rows, T = (P.ho + R - 1) / R;
    p.stages = P.s2_stages;
    p.kb_group = 1;
    p.wp = wp;
    p.sub_rows = R;
    p.sub_pos = R * wp;
    p.subs_per_img = T;
    p.total_subs = n * T;
    p.spi_magic = (T > 1 && static_cast<long long>(n) * T * T < 0x100000000ll) ? static_cast<uint32_t>((0x100000000ull + T - 1) / T) : 0u;
    p.wp_magic = static_cast<uint32_t>((0x100000000ull + wp - 1) / wp);
    p.phase_bytes = P.s2_phase_bytes;
    p.a_stage_bytes = 4 * P.s2_phase_bytes;
    p.a_tx_bytes = 4 * (R + 1) * wp * 64;
    p.acc_stride = 128;
    p.nacc = 4;
    p.tmem_cols = 512;
    const int grid = std::min(p.total_subs, h->num_sms);
    CUDA_TRY(launch_kernel_cluster(conv_s2_kernel, grid, kConvThreads, P.s2_smem_bytes, s, h->opt_pdl != 0, 1u, P.tmap_a_s2,
                                   P.tmap_b, P.tmap_b2_s2, p, x));
    CUDA_TRY(cudaGetLastError());
    return IEVM_OK;
  }
  const int cl = P.cluster;
  const int class_tiles = ((p.m_tiles + cl - 1) / cl) * p.n_tiles;
  const int max_cl = cl > 1 ? (P.dual_max_clusters > 0 ? P.dual_max_clusters : h->num_sms / cl) : h->num_sms;
  const int grid = std::min(2 * class_tiles, max_cl) * cl;
#define IEVM_LAUNCH_DUAL(DT, CL)                                                                                        \
  CUDA_TRY(launch_kernel_cluster(conv_dual_kernel<DT, CL>, grid, kConvThreads, P.dual_smem_bytes, s, h->opt_pdl != 0, \
                                 static_cast<unsigned>(CL), P.dual_wide ? P.tmap_a_wide : P.tmap_a,                  \
                                 P.dual_wide ? P.tmap_b_wide : P.tmap_b, P.tmap_b2, p, x))
  if (h->dtype == IEVM_DTYPE_I8) {
    if (cl == 2) IEVM_LAUNCH_DUAL(kDtypeI8, 2); else IEVM_LAUNCH_DUAL(kDtypeI8, 1);
  } else {
    if (cl == 2) IEVM_LAUNCH_DUAL(kDtypeF16, 2); else IEVM_LAUNCH_DUAL(kDtypeF16, 1);
  }
#undef IEVM_LAUNCH_DUAL
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

int launch_stem_tc(ievm_handle* h, const LayerPlan& L, const uint8_t* xq, uint8_t* out, int n, cudaStream_t s,
                   int32_t* dump_acc) {
  StemTcParams sp;
  memset(&sp, 0, sizeof(sp));
  sp.n = n; sp.h = L.h; sp.w = L.w; sp.ho = L.ho; sp.wo = L.wo;
  sp.m_total = n * L.ho * L.wo;
  sp.m_tiles = (sp.m_total + kTileM - 1) / kTileM;
  sp.cpad = L.cout_pad;
  sp.in_zp = h->in_zp;
  sp.tmem_cols = L.tmem_cols;
  sp.acc_stride = L.tmem_cols / 2;
  sp.idesc = make_idesc_i8_u8s8(L.cout_pad);
  sp.xq = xq;
  sp.out = out;
  sp.bdiv = L.ep0; sp.mult = L.ep1; sp.zwsum = L.zwsum;
  sp.out_zp = L.d.out_zp; sp.out_lo = L.d.relu ? L.d.out_zp : 0;
  sp.dump_acc = dump_acc;
  sp.stuck_flag = h->stuck_dev;
  const int grid = std::min(sp.m_tiles, h->num_sms);
  stem_tc_kernel<<<grid, kStemThreads, L.stem_smem, s>>>(L.tmap_b, sp);
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

int launch_quantize(ievm_handle* h, const float* x, int n, uint8_t* xq, cudaStream_t s) {
  const long long quads = static_cast<long long>(n) * h->in_h * h->in_w / 4;
  quantize_nchw3_to_nhwc4_kernel<<<static_cast<unsigned>((quads + 255) / 256), 256, 0, s>>>(
      x, xq, quads, h->in_h, h->in_w, 1.0f / h->in_scale, h->in_zp);
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

// Stem conv: `in` is the quantised NHWC4 tensor (INT8) or the caller's f16 NCHW batch (FP16).
int launch_stem(ievm_handle* h, const LayerPlan& L, const void* in, void* out, int n, cudaStream_t s) {
  const ievm_layer_desc& d = L.d;
  const long long m_total = static_cast<long long>(n) * L.ho * L.wo;
  if (h->dtype == IEVM_DTYPE_I8 && h->conv_impl == 0)
    return launch_stem_tc(h, L, static_cast<const uint8_t*>(in), static_cast<uint8_t*>(out), n, s, nullptr);
  if (h->dtype == IEVM_DTYPE_I8) {
    StemParams sp;
    sp.n = n; sp.h = L.h; sp.w = L.w; sp.ho = L.ho; sp.wo = L.wo; sp.cpad = L.cout_pad; sp.in_zp = h->in_zp;
    sp.w4 = static_cast<const uint32_t*>(L.w_stem); sp.wsum = L.wsum; sp.bdiv = L.ep0; sp.mult = L.ep1;
    sp.out_zp = d.out_zp; sp.out_lo = d.relu ? d.out_zp : 0;
    stem_conv7x7_simt_kernel<<<static_cast<unsigned>((m_total + 127) / 128), 128, 49 * L.cout_pad * 4, s>>>(
        static_cast<const uint8_t*>(in), static_cast<uint8_t*>(out), sp);
  } else {
    StemF16Params sp;
    sp.n = n; sp.h = L.h; sp.w = L.w; sp.ho = L.ho; sp.wo = L.wo; sp.cpad = L.cout_pad;
    sp.wt = static_cast<const __half*>(L.w_stem); sp.bias = L.ep0;
    const long long total = m_total * (L.cout_pad / 8);
    stem_conv7x7_f16_kernel<<<static_cast<unsigned>((total + 127) / 128), 128, 147 * L.cout_pad * 2, s>>>(
        static_cast<const __half*>(in), static_cast<__half*>(out), sp);
  }
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

int launch_maxpool(ievm_handle* h, const LayerPlan& L, const void* in, void* out, int n, cudaStream_t s) {
  const int pitch = L.cin_pitch;
  if (h->dtype == IEVM_DTYPE_I8) {
    const long long total = static_cast<long long>(n) * L.ho * L.wo * (pitch / 16);
    maxpool3x3s2_u8_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, s>>>(
        static_cast<const uint8_t*>(in), static_cast<uint8_t*>(out), n, L.h, L.w, L.ho, L.wo, pitch);
  } else {
    const long long total = static_cast<long long>(n) * L.ho * L.wo * (pitch / 8);
    maxpool3x3s2_f16_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, s>>>(
        static_cast<const __half*>(in), static_cast<__half*>(out), n, L.h, L.w, L.ho, L.wo, pitch);
  }
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

// The front end (quantize -> stem -> maxpool) is run in chunks of `front_chunk` images through two
// small reused buffers: the stem's 112x112xC output (the largest tensor of the net, 0.8 MB/image)
// is produced and consumed inside L2 and, because every chunk overwrites the same lines, never has
// to be written back to HBM.
// Second-generation fused front end (frontend_v2.cuh): INT8 and FP16, 224-wide inputs, <= 64 stem channels.
bool front_end_is_v2(const ievm_handle* h) {
  return h->front2_ok && h->opt_fused_front && h->conv_impl == 0 && !h->keep_tensors &&
         h->layers.size() >= 2 && h->layers[0].is_stem && h->layers[0].w_front2 != nullptr &&
         h->layers[1].d.op == IEVM_OP_MAXPOOL && h->layers[1].d.in_tensor == h->layers[0].d.out_tensor &&
         h->tensors[h->layers[0].d.out_tensor].last_use == 1;
}

int launch_frontend2(ievm_handle* h, const void* x, int n, cudaStream_t s, int32_t* dump_acc, bool u8_input = false) {
  const LayerPlan& Ls = h->layers[0];
  const LayerPlan& Lp = h->layers[1];
  const bool i8 = h->dtype == IEVM_DTYPE_I8;
  CUtensorMap tmap;
  if (u8_input) {
    // decoded images [n][H][W][3] u8 as (32-bit words of a row, H, n); a box = 4 rows x 176 words starting 16 bytes
    // before the row (TMA wants the box start on a 16-byte boundary)
    cuuint64_t dims[3] = {static_cast<cuuint64_t>(h->in_w) * 3 / 4, static_cast<cuuint64_t>(h->in_h), static_cast<cuuint64_t>(n)};
    cuuint64_t strides[2] = {static_cast<cuuint64_t>(h->in_w) * 3, static_cast<cuuint64_t>(h->in_w) * 3 * h->in_h};
    cuuint32_t box[3] = {F2Cfg<kDtypeI8, 1>::kU8RowBytes / 4, 4, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = g_encode_tiled(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<void*>(x), dims, strides, box, estr,
                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled (u8 input) failed: CUresult %d", (int)r);
  } else {
    // the input batch as (W, H, 3 * n) planes; boxes start 4 columns left of the image and are zero-filled outside
    const size_t es = i8 ? 4 : 2;
    cuuint64_t dims[3] = {static_cast<cuuint64_t>(h->in_w), static_cast<cuuint64_t>(h->in_h), static_cast<cuuint64_t>(3) * n};
    cuuint64_t strides[2] = {h->in_w * es, static_cast<cuuint64_t>(h->in_w) * h->in_h * es};
    cuuint32_t box[3] = {static_cast<cuuint32_t>(i8 ? F2Cfg<kDtypeI8>::kBoxW : F2Cfg<kDtypeF16>::kBoxW), 4, 3};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = g_encode_tiled(&tmap, i8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                                      const_cast<void*>(x), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                      CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "cuTensorMapEncodeTiled (front end input) failed: CUresult %d", (int)r);
  }
  Frontend2Params fp;
  memset(&fp, 0, sizeof(fp));
  fp.n = n;
  fp.h = h->in_h;
  fp.ho = Ls.ho;
  fp.ph = Lp.ho;
  fp.tpu = h->front_tpu > 0 ? std::min(h->front_tpu, fp.ph) : 0;
  fp.in_zp = h->in_zp;
  fp.inv_scale = i8 ? 1.0f / h->in_scale : 1.0f;
  fp.idesc = i8 ? make_idesc_i8_s8u8(kF2Wo) : make_idesc_f16(kF2Wo);
  fp.wpack = static_cast<const uint8_t*>(Ls.w_front2);
  fp.out = tensor_ptr(h, Lp.d.out_tensor);
  fp.bdiv = Ls.ep0;
  fp.mult = Ls.ep1;
  fp.zwsum = Ls.zwsum;
  fp.lut = h->lut_dev;
  fp.out_zp = Ls.d.out_zp;
  fp.out_lo = Ls.d.relu ? Ls.d.out_zp : 0;
  fp.fast_round = Ls.fast_round && fp.out_lo == 0;    // the fast instantiation folds both clamps into one instruction (lower = 0)
  fp.dump_acc = dump_acc;
  fp.stuck_flag = h->stuck_dev;
  const int grid = std::min(n * fp.ph, h->num_sms);       // contiguous ranges of pooled rows (frontend_v2.cuh: F2Walk)
  if (dump_acc != nullptr) {
    // debug instantiations (ievm_debug_frontend): the general rounding form, accumulators written out
    if (i8) frontend2_kernel<kDtypeI8, 0, false, true><<<grid, kF2Threads, F2Cfg<kDtypeI8>::kSmemBytes, s>>>(tmap, fp);
    else frontend2_kernel<kDtypeF16, 0, false, true><<<grid, kF2Threads, F2Cfg<kDtypeF16>::kSmemBytes, s>>>(tmap, fp);
  } else if (u8_input && fp.fast_round) frontend2_kernel<kDtypeI8, 1, true><<<grid, kF2Threads, F2Cfg<kDtypeI8, 1>::kSmemBytes, s>>>(tmap, fp);
  else if (u8_input) frontend2_kernel<kDtypeI8, 1><<<grid, kF2Threads, F2Cfg<kDtypeI8, 1>::kSmemBytes, s>>>(tmap, fp);
  else if (i8 && fp.fast_round) frontend2_kernel<kDtypeI8, 0, true><<<grid, kF2Threads, F2Cfg<kDtypeI8>::kSmemBytes, s>>>(tmap, fp);
  else if (i8) frontend2_kernel<kDtypeI8, 0><<<grid, kF2Threads, F2Cfg<kDtypeI8>::kSmemBytes, s>>>(tmap, fp);
  else frontend2_kernel<kDtypeF16, 0><<<grid, kF2Threads, F2Cfg<kDtypeF16>::kSmemBytes, s>>>(tmap, fp);
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

bool front_end_is_chunked(const ievm_handle* h) {
  return h->dtype == IEVM_DTYPE_I8 && h->front_chunk > 0 && !h->keep_tensors && h->layers.size() >= 2 &&
         h->layers[0].is_stem && h->layers[1].d.op == IEVM_OP_MAXPOOL &&
         h->layers[1].d.in_tensor == h->layers[0].d.out_tensor && h->tensors[h->layers[0].d.out_tensor].last_use == 1;
}

// Input modes of the forward entry points.
enum : int { kInNative = 0, kInU8 = 1, kInU8Resize = 2 };

int launch_resize(ievm_handle* h, const uint8_t* x, int n, cudaStream_t s) {
  if (!h->rs_out) return fail(IEVM_ERR_BAD_ARG, "call ievm_set_resize before ievm_forward_u8_resize");
  const uint8_t* src = x;
  if (h->rs_in_w != h->in_w) {      // horizontal pass: [n * rs_in_h rows][rs_in_w] -> [..][in_w]
    const long long rows = static_cast<long long>(n) * h->rs_in_h;
    uint8_t* dst = h->rs_in_h != h->in_h ? h->rs_tmp : h->rs_out;
    resize_rows_u8_kernel<<<static_cast<unsigned>((rows * h->in_w + 255) / 256), 256, 0, s>>>(
        src, dst, rows, h->rs_in_w, h->in_w, h->rs_bounds_w, h->rs_kk_w, h->rs_ksize_w);
    src = dst;
  }
  if (h->rs_in_h != h->in_h) {      // vertical pass
    const long long total = static_cast<long long>(n) * h->in_h * h->in_w;
    resize_cols_u8_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, s>>>(
        src, h->rs_out, n, h->rs_in_h, h->in_h, h->in_w, h->rs_bounds_h, h->rs_kk_h, h->rs_ksize_h);
  }
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

int enqueue_forward(ievm_handle* h, const void* x, int n, void* logits, cudaStream_t s, int in_mode = kInNative) {
  if (in_mode == kInU8Resize) {
    if (h->rs_in_h == h->in_h && h->rs_in_w == h->in_w) in_mode = kInU8;          // already the right size
    else {
      if (int rc = launch_resize(h, static_cast<const uint8_t*>(x), n, s)) return rc;
      x = h->rs_out;
      in_mode = kInU8;
    }
  }
  const bool u8_input = in_mode == kInU8;
  const bool i8 = h->dtype == IEVM_DTYPE_I8;
  const bool prof = h->profile != 0;
  if (prof) {
    while (h->prof_events.size() < h->layers.size() + 2) {
      cudaEvent_t e;
      CUDA_TRY(cudaEventCreate(&e));
      h->prof_events.push_back(e);
    }
    h->prof_ms.resize(h->layers.size() + 1, 0.0);
    h->prof_calls.resize(h->layers.size() + 1, 0);
    CUDA_TRY(cudaEventRecord(h->prof_events[0], s));
  }
  size_t first_layer = 0;
  if (u8_input && !front_end_is_v2(h))
    return fail(IEVM_ERR_UNSUPPORTED, "8-bit image input needs the fused front end (224-wide input, <= 64 stem channels, "
                                      "keep_tensors = 0, conv_impl = 0)");
  if (u8_input && h->lut_dev == nullptr) return fail(IEVM_ERR_BAD_ARG, "call ievm_set_input_lut before ievm_forward_u8");
#ifdef IEVM_EXP_SKIP
  // A/B build only (scripts/skip_costs.py): leave out the launches whose layer bit is set, to measure what each launch
  // costs INSIDE the graph step (results are wrong, timing is data independent)
  const unsigned long long skip_mask = getenv("IEVM_SKIP_MASK") ? strtoull(getenv("IEVM_SKIP_MASK"), nullptr, 0) : 0ull;
#define IEVM_SKIPPED(li) ((skip_mask >> (li)) & 1ull)
#else
#define IEVM_SKIPPED(li) false
#endif
  if (front_end_is_v2(h)) {
    // profile slots: the fused kernel is attributed to the stem's slot (quantize and maxpool read 0)
    if (prof) CUDA_TRY(cudaEventRecord(h->prof_events[1], s));
    if (!IEVM_SKIPPED(0))
    if (int rc = launch_frontend2(h, x, n, s, nullptr, u8_input)) return rc;
    if (prof) CUDA_TRY(cudaEventRecord(h->prof_events[2], s));
    first_layer = 2;
  } else if (front_end_is_chunked(h)) {
    // profile slots: the whole interleaved front end is attributed to the stem's slot
    if (prof) CUDA_TRY(cudaEventRecord(h->prof_events[1], s));
    const LayerPlan& Ls = h->layers[0];
    const LayerPlan& Lp = h->layers[1];
    const size_t in_img = static_cast<size_t>(h->in_c) * h->in_h * h->in_w;
    const size_t pooled_img = h->tensors[Lp.d.out_tensor].bytes_per_image();
    for (int c0 = 0; c0 < n; c0 += h->front_chunk) {
      const int nc = std::min(h->front_chunk, n - c0);
      if (int rc = launch_quantize(h, static_cast<const float*>(x) + c0 * in_img, nc,
                                   static_cast<uint8_t*>(tensor_ptr(h, 0)), s)) return rc;
      if (int rc = launch_stem(h, Ls, tensor_ptr(h, 0), tensor_ptr(h, Ls.d.out_tensor), nc, s)) return rc;
      if (int rc = launch_maxpool(h, Lp, tensor_ptr(h, Ls.d.out_tensor),
                                  static_cast<uint8_t*>(tensor_ptr(h, Lp.d.out_tensor)) + c0 * pooled_img, nc, s)) return rc;
    }
    if (prof) CUDA_TRY(cudaEventRecord(h->prof_events[2], s));
    first_layer = 2;
  } else {
    if (i8)
      if (int rc = launch_quantize(h, static_cast<const float*>(x), n, static_cast<uint8_t*>(tensor_ptr(h, 0)), s)) return rc;
    if (prof) CUDA_TRY(cudaEventRecord(h->prof_events[1], s));
  }
  for (size_t li = first_layer; li < h->layers.size(); ++li) {
    const LayerPlan& L = h->layers[li];
    const ievm_layer_desc& d = L.d;
    if (prof && li > 0) CUDA_TRY(cudaEventRecord(h->prof_events[li + 1], s));
    if (IEVM_SKIPPED(li)) continue;
    if (d.op == IEVM_OP_CONV && L.is_stem) {
      if (int rc = launch_stem(h, L, i8 ? tensor_ptr(h, 0) : x, tensor_ptr(h, d.out_tensor), n, s)) return rc;
    } else if (d.op == IEVM_OP_CONV) {
      const int mate = L.dual_partner >= 0 ? L.dual_partner : L.dual_of;      // conv_dual.cuh: the 3x3 / 1x1 pair of a block
      if (dual_active(h) && mate >= 0) {
        // one launch for the pair, at the position of whichever comes first (both read only the block input)
        if (mate > static_cast<int>(li))
          if (int rc = launch_conv_dual(h, L.dual_partner >= 0 ? L : h->layers[mate], n, s, nullptr, nullptr)) return rc;
      } else if (int rc = launch_conv(h, L, n, s, nullptr)) return rc;
    } else if (d.op == IEVM_OP_MAXPOOL) {
      if (int rc = launch_maxpool(h, L, tensor_ptr(h, d.in_tensor), tensor_ptr(h, d.out_tensor), n, s)) return rc;
    } else if (d.op == IEVM_OP_ADD_RELU) {
      const TensorInfo& tin = h->tensors[d.in_tensor];
      const long long nvec = static_cast<long long>(n) * tin.h * tin.w * tin.pitch / 8;
      add_relu_f16_kernel<<<static_cast<unsigned>((nvec + 255) / 256), 256, 0, s>>>(
          static_cast<const uint4*>(tensor_ptr(h, d.in_tensor)), static_cast<const uint4*>(tensor_ptr(h, d.res_tensor)),
          static_cast<uint4*>(tensor_ptr(h, d.out_tensor)), nvec);
      CUDA_TRY(cudaGetLastError());
    } else {   // head
      const TensorInfo& tin = h->tensors[d.in_tensor];
      if (i8) {
        HeadParams hp;
        hp.hw = tin.h * tin.w; hp.c = tin.c; hp.cpad = tin.pitch; hp.classes = d.cout; hp.in_zp = d.in_zp;
        hp.w = static_cast<const int8_t*>(L.w_packed); hp.bdiv = L.ep0; hp.mult = L.ep1;
        hp.fc_zp = d.out_zp; hp.fc_scale = d.out_scale;
        const int wbytes = hp.classes * hp.cpad;
        hp.w_smem = wbytes <= kHeadWeightSmemMax ? 1 : 0;
        CUDA_TRY(launch_kernel(head_i8_kernel, n, kHeadThreads, hp.w_smem ? wbytes : 0, s, h->opt_pdl != 0,
                               static_cast<const uint8_t*>(tensor_ptr(h, d.in_tensor)), static_cast<float*>(logits),
                               static_cast<uint8_t*>(nullptr), hp));
      } else {
        HeadF16Params hp;
        hp.hw = tin.h * tin.w; hp.c = tin.c; hp.cpad = tin.pitch; hp.classes = d.cout;
        hp.w = static_cast<const __half*>(L.w_packed); hp.bias = L.ep0;
        hp.pooled = h->obs_pooled;           // non-null only while calibrating (ievm_observe)
        const int wbytes = 2 * hp.classes * hp.cpad;
        hp.w_smem = wbytes <= kHeadWeightSmemMax ? 1 : 0;
        CUDA_TRY(launch_kernel(head_f16_kernel, n, kHeadThreads, hp.w_smem ? wbytes : 0, s, h->opt_pdl != 0,
                               static_cast<const __half*>(tensor_ptr(h, d.in_tensor)), static_cast<__half*>(logits), hp));
      }
      CUDA_TRY(cudaGetLastError());
    }
  }
  h->last_n = n;
  h->last_x = x;
  h->last_logits = logits;
  if (prof) {
    CUDA_TRY(cudaEventRecord(h->prof_events[h->layers.size() + 1], s));
    CUDA_TRY(cudaStreamSynchronize(s));
    for (size_t i = 0; i <= h->layers.size(); ++i) {
      float ms = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&ms, h->prof_events[i], h->prof_events[i + 1]));
      h->prof_ms[i] += ms;
      h->prof_calls[i] += 1;
    }
  }
  return IEVM_OK;
}

constexpr size_t kMaxGraphs = 16;

// Stream ordering between consecutive uses of the handle's workspace (see ievm_handle::order_event).  Skipped while the
// caller is capturing `s` into a graph of their own (an event recorded outside the capture cannot be waited on inside it).
int order_begin(ievm_handle* h, cudaStream_t s, bool* capturing) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  *capturing = cudaStreamIsCapturing(s, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone;
  if (*capturing) return IEVM_OK;
  if (h->order_valid && h->last_stream != s) CUDA_TRY(cudaStreamWaitEvent(s, h->order_event, 0));
  return IEVM_OK;
}
int order_end(ievm_handle* h, cudaStream_t s, bool capturing) {
  if (capturing) return IEVM_OK;
  CUDA_TRY(cudaEventRecord(h->order_event, s));
  h->last_stream = s;
  h->order_valid = true;
  return IEVM_OK;
}

int forward_common(ievm_handle* h, int want_dtype, const void* x, int n, void* logits, void* stream, int in_mode = kInNative) {
  if (!h || !x || !logits) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (h->dtype != want_dtype) return fail(IEVM_ERR_BAD_ARG, "engine dtype does not match this entry point");
  if (n < 0 || n > h->max_batch) return fail(IEVM_ERR_BAD_ARG, "batch %d outside [0, %d]", n, h->max_batch);
  if (n == 0) return IEVM_OK;
  DeviceGuard guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  bool capturing = false;
  if (int rc = order_begin(h, s, &capturing)) return rc;
  if (!h->use_graph || h->profile || capturing) {
    if (int rc = enqueue_forward(h, x, n, logits, s, in_mode)) return rc;
    return order_end(h, s, capturing);
  }
  const auto key = std::make_tuple(n * 4 + in_mode, x, logits);
  auto it = h->graphs.find(key);
  if (it == h->graphs.end()) {
    if (h->graphs.size() >= kMaxGraphs) {          // evict the least recently used graph
      auto victim = h->graphs.begin();
      for (auto g = h->graphs.begin(); g != h->graphs.end(); ++g)
        if (g->second.second < victim->second.second) victim = g;
      cudaGraphExecDestroy(victim->second.first);
      h->graphs.erase(victim);
    }
    cudaStream_t cs = h->own_stream;
    cudaGraph_t graph = nullptr;
    CUDA_TRY(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    const int rc = enqueue_forward(h, x, n, logits, cs, in_mode);
    const cudaError_t ce = cudaStreamEndCapture(cs, &graph);
    if (rc || ce != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      if (rc) return rc;
      return fail(IEVM_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(ce));
    }
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) return fail(IEVM_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
    it = h->graphs.emplace(key, std::make_pair(exec, 0ull)).first;
  }
  it->second.second = ++h->graph_clock;
  CUDA_TRY(cudaGraphLaunch(it->second.first, s));
  h->last_n = n;
  h->last_x = x;
  h->last_logits = logits;
  return order_end(h, s, capturing);
}

int check_stuck(ievm_handle* h, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return IEVM_OK;
  const unsigned code = h->stuck_host ? *reinterpret_cast<volatile unsigned int*>(h->stuck_host) : 0;
  return fail(IEVM_ERR_CUDA, "%s: %s (pipeline stuck code 0x%x: 0x1xx producer/empty, 0x2xx mma/tmem-empty, "
              "0x3xx mma/full, 0x4xx epilogue/tmem-full)", what, cudaGetErrorString(e), code);
}

// Diagnostic: one im2col TMA tile, dumped raw (swizzled) from shared memory.
__global__ void probe_im2col_kernel(const __grid_constant__ CUtensorMap tmap, int c0, int w0, int h0, int n0,
                                    int tap_x, int tap_y, int bytes, uint8_t* out, unsigned int* stuck) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + bytes);
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) smem[i] = 0xEE;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  fence_proxy_async_smem();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, static_cast<uint32_t>(bytes));
    tma_load_im2col_4d(smem, &tmap, bar, c0, w0, h0, n0, static_cast<uint16_t>(tap_x), static_cast<uint16_t>(tap_y));
  }
  wait_or_die(bar, 0, 0x900u, stuck);
  __syncthreads();
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) out[i] = smem[i];
}

// Diagnostic: one tiled 4D TMA box (halo patch), dumped raw from shared memory.
__global__ void probe_patch_kernel(const __grid_constant__ CUtensorMap tmap, int c0, int w0, int h0, int n0, int bytes,
                                   uint8_t* out, unsigned int* stuck) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + ((bytes + 15) & ~15));
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) smem[i] = 0xEE;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  fence_proxy_async_smem();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, static_cast<uint32_t>(bytes));
    tma_load_4d(smem, &tmap, bar, c0, w0, h0, n0);
  }
  wait_or_die(bar, 0, 0x901u, stuck);
  __syncthreads();
  for (int i = threadIdx.x; i < bytes; i += blockDim.x) out[i] = smem[i];
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char* ievm_last_error(void) { return g_last_error.c_str(); }

const char* ievm_build_info(void) { return "ievm-b200 abi=1 arch=sm_100a kernels=tcgen05.mma(kind::i8,kind::f16)+TMA(im2col)"; }

int ievm_create(const ievm_net_desc* nd, int device, int max_batch, ievm_handle** out) {
  if (!nd || !out || !nd->layers || nd->num_layers <= 0 || max_batch <= 0)
    return fail(IEVM_ERR_BAD_ARG, "ievm_create: bad arguments");
  if (nd->dtype != IEVM_DTYPE_I8 && nd->dtype != IEVM_DTYPE_F16) return fail(IEVM_ERR_BAD_ARG, "unknown dtype");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(IEVM_ERR_CUDA, "no CUDA device: this engine has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(IEVM_ERR_BAD_ARG, "device %d out of range", device);
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(IEVM_ERR_UNSUPPORTED, "device is sm_%d%d; this build is sm_100a only", prop.major, prop.minor);
  if (int rc = load_driver_entry_points()) return rc;

  ievm_handle* h = new ievm_handle();
  h->device = device;
  h->dtype = nd->dtype;
  h->elem = nd->dtype == IEVM_DTYPE_I8 ? 1 : 2;
  h->max_batch = max_batch;
  h->num_sms = prop.multiProcessorCount;
  h->smem_optin = static_cast<int>(prop.sharedMemPerBlockOptin);
  h->in_c = nd->in_c; h->in_h = nd->in_h; h->in_w = nd->in_w; h->classes = nd->num_classes;
  h->in_scale = nd->in_scale; h->in_zp = nd->in_zp;
  if (const char* e = getenv("IEVM_HALO")) h->opt_halo = atoi(e);
  if (const char* e = getenv("IEVM_HALO_STATIC")) h->opt_halo_static = atoi(e);
  if (const char* e = getenv("IEVM_TWO_CTA")) h->opt_two_cta = atoi(e);
  if (const char* e = getenv("IEVM_FIXED_BN")) h->opt_fixed_bn = atoi(e);
  if (const char* e = getenv("IEVM_PDL")) h->opt_pdl = atoi(e);
  if (const char* e = getenv("IEVM_DUAL")) h->opt_dual = atoi(e);
  if (const char* e = getenv("IEVM_WIDE")) h->opt_wide = atoi(e);
  if (const char* e = getenv("IEVM_S2")) h->opt_s2 = atoi(e);
  if (const char* e = getenv("IEVM_TINY")) h->opt_tiny = atoi(e);
  if (const char* e = getenv("IEVM_CLUSTER")) h->opt_cluster = atoi(e);
  if (const char* e = getenv("IEVM_HOST_CHUNK")) h->host_chunk = atoi(e);
  if (const char* e = getenv("IEVM_FUSED_FRONT")) h->opt_fused_front = atoi(e);
  if (const char* e = getenv("IEVM_FRONT_CHUNK")) h->front_chunk = atoi(e);
  if (const char* e = getenv("IEVM_FRONT_TPU")) h->front_tpu = atoi(e);
  int rc = plan_shapes(h, nd);
  for (size_t i = 0; rc == IEVM_OK && i < h->layers.size(); ++i) {
    LayerPlan& L = h->layers[i];
    if (L.d.op == IEVM_OP_CONV) rc = upload_conv_operands(h, L);
    else if (L.d.op == IEVM_OP_HEAD) rc = upload_head_operands(h, L);
    // host pointers in the copied descriptor must not be used after create returns
    L.d.weight = nullptr; L.d.bias = nullptr; L.d.w_scale = nullptr;
  }
  if (rc == IEVM_OK && getenv("IEVM_VERBOSE")) {
    for (size_t i = 0; i < h->layers.size(); ++i) {
      const LayerPlan& L = h->layers[i];
      if (L.d.op != IEVM_OP_CONV || L.is_stem) continue;
      // dual: the form of the launch this conv rides in (both convs of a pair print it); subs: halo sub-tiles per image
      const LayerPlan& P = L.dual_of >= 0 ? h->layers[L.dual_of] : L;
      const char* dual = P.dual_partner < 0 ? "none" : P.dual_s2 ? "s2" : P.dual_wide ? "wide" : "plain";
      fprintf(stderr, "[ievm] layer %2zu %dx%d s%d %4d->%4d @%dx%d mode=%s kc=%d kchunks=%d bn=%d n_tiles=%d cluster=%d stages=%d kb_group=%d band=%dx%d rows residentB=%d fast_round=%d smem=%zu two_cta=%d dual=%s zcorr=%d subs=%d\n",
              i, L.d.ksize, L.d.ksize, L.d.stride, L.d.cin, L.d.cout, L.ho, L.wo, L.mode == kModeHalo ? "halo" : "im2col",
              L.kc_bytes, L.kchunks, L.bn, L.n_tiles, L.cluster, L.stages, L.kb_group, L.band_subs, L.sub_rows, L.resident_b, L.fast_round, L.smem_bytes,
              L.two_cta, dual, L.zcorr != nullptr ? 1 : 0, L.subs_per_img);
    }
  }
  if (rc == IEVM_OK) rc = assign_buffers(h);
  if (rc == IEVM_OK) rc = encode_maps(h);
  if (rc == IEVM_OK) {
    size_t max_smem = 0;
    for (const LayerPlan& L : h->layers) max_smem = std::max(max_smem, std::max(L.smem_bytes, std::max(L.dual_smem_bytes, L.s2_smem_bytes)));
    if (max_smem > static_cast<size_t>(prop.sharedMemPerBlockOptin)) rc = fail(IEVM_ERR_UNSUPPORTED, "smem plan exceeds device limit");
    if (rc == IEVM_OK && max_smem > 0) {
      cudaError_t e = cudaSuccess;
      // function attributes are process-wide: always raise the limit to the device maximum so that several
      // engines with different plans can coexist
      const int ms = static_cast<int>(prop.sharedMemPerBlockOptin);
#define IEVM_ATTR(DT, RES, MODE, CL, SH) \
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<DT, RES, MODE, CL, SH>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms)
      IEVM_ATTR(kDtypeI8, false, kModeIm2col, 1, 0); IEVM_ATTR(kDtypeI8, true, kModeIm2col, 1, 0);
      IEVM_ATTR(kDtypeI8, false, kModeIm2col, 2, 0); IEVM_ATTR(kDtypeI8, true, kModeIm2col, 2, 0);
      IEVM_ATTR(kDtypeI8, false, kModeHalo, 1, 0);   IEVM_ATTR(kDtypeI8, true, kModeHalo, 1, 0);
      IEVM_ATTR(kDtypeI8, false, kModeHalo, 1, 1);   IEVM_ATTR(kDtypeI8, true, kModeHalo, 1, 1);
      IEVM_ATTR(kDtypeI8, false, kModeHalo, 1, 2);   IEVM_ATTR(kDtypeI8, true, kModeHalo, 1, 2);
#define IEVM_ATTR_ZC(RES, MODE, CL) \
  if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<kDtypeI8, RES, MODE, CL, 0, kEpiWarps, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms)
      IEVM_ATTR_ZC(false, kModeIm2col, 1); IEVM_ATTR_ZC(true, kModeIm2col, 1);
      IEVM_ATTR_ZC(false, kModeIm2col, 2); IEVM_ATTR_ZC(true, kModeIm2col, 2);
      IEVM_ATTR_ZC(false, kModeHalo, 1);   IEVM_ATTR_ZC(true, kModeHalo, 1);
#undef IEVM_ATTR_ZC
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<kDtypeI8, false, kModeHalo, 1, 1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<kDtypeI8, true, kModeHalo, 1, 1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms);
      IEVM_ATTR(kDtypeF16, false, kModeIm2col, 1, 0); IEVM_ATTR(kDtypeF16, true, kModeIm2col, 1, 0);
      IEVM_ATTR(kDtypeF16, false, kModeIm2col, 2, 0); IEVM_ATTR(kDtypeF16, true, kModeIm2col, 2, 0);
      IEVM_ATTR(kDtypeF16, false, kModeHalo, 1, 0);   IEVM_ATTR(kDtypeF16, true, kModeHalo, 1, 0);
      IEVM_ATTR(kDtypeF16, false, kModeHalo, 1, 3);   IEVM_ATTR(kDtypeF16, true, kModeHalo, 1, 3);
#undef IEVM_ATTR
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_s2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ms);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_dual_kernel<kDtypeI8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_dual_kernel<kDtypeI8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_dual_kernel<kDtypeF16, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms);
      if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_dual_kernel<kDtypeF16, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, ms);
      if (e != cudaSuccess) rc = fail(IEVM_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      // how many 2-CTA clusters of the heaviest configuration can be co-resident (GPC packing may strand SMs)
      for (LayerPlan& L : h->layers) {
        if (rc != IEVM_OK || L.cluster <= 1) continue;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(h->num_sms / L.cluster * L.cluster);
        cfg.blockDim = dim3(kConvThreads);
        cfg.dynamicSmemBytes = L.smem_bytes;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = L.cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        int nc = 0;
        const cudaError_t qe = h->dtype == IEVM_DTYPE_I8
            ? cudaOccupancyMaxActiveClusters(&nc, conv_tc_kernel<kDtypeI8, false, kModeIm2col, 2, 0>, &cfg)
            : cudaOccupancyMaxActiveClusters(&nc, conv_tc_kernel<kDtypeF16, false, kModeIm2col, 2, 0>, &cfg);
        L.max_clusters = (qe == cudaSuccess && nc > 0) ? std::min(nc, h->num_sms / L.cluster) : h->num_sms / L.cluster;
        if (qe != cudaSuccess) cudaGetLastError();
        if (L.dual_partner >= 0) {
          cfg.dynamicSmemBytes = L.dual_smem_bytes;
          nc = 0;
          const cudaError_t de = h->dtype == IEVM_DTYPE_I8 ? cudaOccupancyMaxActiveClusters(&nc, conv_dual_kernel<kDtypeI8, 2>, &cfg)
                                                           : cudaOccupancyMaxActiveClusters(&nc, conv_dual_kernel<kDtypeF16, 2>, &cfg);
          L.dual_max_clusters = (de == cudaSuccess && nc > 0) ? std::min(nc, h->num_sms / L.cluster) : h->num_sms / L.cluster;
          if (de != cudaSuccess) cudaGetLastError();
        }
      }
    }
  }
  if (rc == IEVM_OK && h->front2_ok) {
    if ((h->dtype == IEVM_DTYPE_I8
             ? cudaFuncSetAttribute(frontend2_kernel<kDtypeI8, 0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F2Cfg<kDtypeI8>::kSmemBytes)
             : cudaFuncSetAttribute(frontend2_kernel<kDtypeF16, 0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F2Cfg<kDtypeF16>::kSmemBytes)) != cudaSuccess)
      rc = fail(IEVM_ERR_CUDA, "cudaFuncSetAttribute(frontend2_kernel, debug instantiation) failed");
  }
  if (rc == IEVM_OK && h->front2_ok) {
    const cudaError_t e = h->dtype == IEVM_DTYPE_I8
        ? cudaFuncSetAttribute(frontend2_kernel<kDtypeI8, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F2Cfg<kDtypeI8>::kSmemBytes)
        : cudaFuncSetAttribute(frontend2_kernel<kDtypeF16, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F2Cfg<kDtypeF16>::kSmemBytes);
    if (e != cudaSuccess) rc = fail(IEVM_ERR_CUDA, "cudaFuncSetAttribute(frontend2_kernel): %s", cudaGetErrorString(e));
    if (rc == IEVM_OK && h->dtype == IEVM_DTYPE_I8 &&
        (cudaFuncSetAttribute(frontend2_kernel<kDtypeI8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)F2Cfg<kDtypeI8, 1>::kSmemBytes) != cudaSuccess ||
         cudaFuncSetAttribute(frontend2_kernel<kDtypeI8, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)F2Cfg<kDtypeI8, 1>::kSmemBytes) != cudaSuccess ||
         cudaFuncSetAttribute(frontend2_kernel<kDtypeI8, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)F2Cfg<kDtypeI8>::kSmemBytes) != cudaSuccess))
      rc = fail(IEVM_ERR_CUDA, "cudaFuncSetAttribute(frontend2_kernel, u8 input / fast rounding) failed");
  }
  if (rc == IEVM_OK) {
    for (const LayerPlan& L : h->layers)
      if (L.stem_smem > 0) {
        if (L.stem_smem > static_cast<size_t>(prop.sharedMemPerBlockOptin)) rc = fail(IEVM_ERR_UNSUPPORTED, "stem smem plan exceeds device limit");
        else if (cudaFuncSetAttribute(stem_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop.sharedMemPerBlockOptin) != cudaSuccess)
          rc = fail(IEVM_ERR_CUDA, "cudaFuncSetAttribute(stem_tc_kernel) failed");
      }
  }
  if (rc == IEVM_OK) {
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&h->stuck_host), sizeof(unsigned int), cudaHostAllocMapped);
    if (e == cudaSuccess) {
      *h->stuck_host = 0;
      e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&h->stuck_dev), h->stuck_host, 0);
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->order_event, cudaEventDisableTiming);
    for (auto& sl : h->slots) {
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl.copied, cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming);
    }
    if (const char* w = getenv("IEVM_WAIT_LIMIT_MS")) {
      const unsigned long long ns = static_cast<unsigned long long>(atoll(w)) * 1000000ull;
      if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_wait_limit_ns, &ns, sizeof(ns));
    }
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) rc = fail(IEVM_ERR_CUDA, "runtime setup: %s", cudaGetErrorString(e));
  }
  if (rc != IEVM_OK) {
    const std::string keep = g_last_error;
    ievm_destroy(h);
    g_last_error = keep;
    return rc;
  }
  *out = h;
  return IEVM_OK;
}

void ievm_destroy(ievm_handle* h) {
  if (!h) return;
  DeviceGuard guard(h->device);
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  for (void* p : h->buffers) cudaFree(p);
  for (void* p : h->owned) cudaFree(p);
  for (void* q : {static_cast<void*>(h->rs_bounds_w), static_cast<void*>(h->rs_bounds_h), static_cast<void*>(h->rs_kk_w),
                  static_cast<void*>(h->rs_kk_h), static_cast<void*>(h->rs_tmp), static_cast<void*>(h->rs_out)})
    if (q) cudaFree(q);
  if (h->stage_in) cudaFree(h->stage_in);
  if (h->stage_out) cudaFree(h->stage_out);
  if (h->pin_in) cudaFreeHost(h->pin_in);
  if (h->pin_out) cudaFreeHost(h->pin_out);
  if (h->stuck_host) cudaFreeHost(h->stuck_host);
  if (h->order_event) cudaEventDestroy(h->order_event);
  for (auto& sl : h->slots) {
    if (sl.dev_in) cudaFree(sl.dev_in);
    if (sl.dev_out) cudaFree(sl.dev_out);
    if (sl.copied) cudaEventDestroy(sl.copied);
    if (sl.done) cudaEventDestroy(sl.done);
  }
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  for (cudaEvent_t e : h->copy_events) cudaEventDestroy(e);
  delete h;
}

int ievm_forward_i8(ievm_handle* h, const float* x, int n, float* logits, void* stream) {
  return forward_common(h, IEVM_DTYPE_I8, x, n, logits, stream);
}

int ievm_forward_f16(ievm_handle* h, const void* x, int n, void* logits, void* stream) {
  return forward_common(h, IEVM_DTYPE_F16, x, n, logits, stream);
}

static int forward_host_common(ievm_handle* h, int dtype, const void* x_host, int n, void* logits_host, int in_mode = kInNative) {
  if (!h || !x_host || !logits_host) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (n <= 0 || n > h->max_batch) return fail(IEVM_ERR_BAD_ARG, "batch %d outside [1, %d]", n, h->max_batch);
  DeviceGuard guard(h->device);
  const size_t in_elem = in_mode != kInNative ? 1 : (dtype == IEVM_DTYPE_I8 ? 4 : 2);
  const size_t out_elem = dtype == IEVM_DTYPE_I8 ? 4 : 2;
  const size_t per_img = in_mode == kInU8Resize ? static_cast<size_t>(3) * h->rs_in_h * h->rs_in_w
                                                : static_cast<size_t>(h->in_c) * h->in_h * h->in_w * in_elem;
  if (in_mode == kInU8Resize && !h->rs_out) return fail(IEVM_ERR_BAD_ARG, "call ievm_set_resize before ievm_forward_u8_resize_host");
  {
    const size_t native = static_cast<size_t>(h->in_c) * h->in_h * h->in_w * (dtype == IEVM_DTYPE_I8 ? 4 : 2);
    const size_t need = std::max(native, per_img) * h->max_batch;
    if (h->stage_in_bytes < need) {
      CUDA_TRY(cudaStreamSynchronize(h->own_stream));
      if (h->stage_in) cudaFree(h->stage_in);
      h->stage_in = nullptr;
      h->stage_in_bytes = 0;
      for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);      // graphs captured on the old staging buffer
      h->graphs.clear();
      CUDA_TRY(cudaMalloc(&h->stage_in, need));
      h->stage_in_bytes = need;
    }
    if (!h->stage_out) CUDA_TRY(cudaMalloc(&h->stage_out, out_elem * h->classes * h->max_batch));
  }
  // Chunked pipeline: the H2D copy of chunk i+1 (copy stream) overlaps the forward of chunk i (compute
  // stream); PCIe, not the GPU, bounds this entry point, so the chunk size only has to be large enough
  // to keep the kernels efficient.
  cudaStream_t s = h->own_stream;
  const int chunk = (h->host_chunk > 0 && n > h->host_chunk) ? h->host_chunk : n;
  const int nchunks = (n + chunk - 1) / chunk;
  while (static_cast<int>(h->copy_events.size()) < nchunks) {
    cudaEvent_t e;
    CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->copy_events.push_back(e);
  }
  for (int c = 0; c < nchunks; ++c) {
    const int c0 = c * chunk, nc = std::min(chunk, n - c0);
    CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t*>(h->stage_in) + c0 * per_img,
                             static_cast<const uint8_t*>(x_host) + c0 * per_img, per_img * nc, cudaMemcpyHostToDevice,
                             nchunks > 1 ? h->copy_stream : s));
    if (nchunks > 1) {
      CUDA_TRY(cudaEventRecord(h->copy_events[c], h->copy_stream));
      CUDA_TRY(cudaStreamWaitEvent(s, h->copy_events[c], 0));
    }
    if (int rc = forward_common(h, dtype, static_cast<uint8_t*>(h->stage_in) + c0 * per_img, nc,
                                static_cast<uint8_t*>(h->stage_out) + c0 * out_elem * h->classes, s, in_mode)) return rc;
  }
  CUDA_TRY(cudaMemcpyAsync(logits_host, h->stage_out, out_elem * h->classes * n, cudaMemcpyDeviceToHost, s));
  return check_stuck(h, cudaStreamSynchronize(s), "forward (host buffers)");
}

int ievm_forward_i8_host(ievm_handle* h, const float* x_host, int n, float* logits_host) {
  return forward_host_common(h, IEVM_DTYPE_I8, x_host, n, logits_host);
}
int ievm_forward_f16_host(ievm_handle* h, const void* x_host, int n, void* logits_host) {
  return forward_host_common(h, IEVM_DTYPE_F16, x_host, n, logits_host);
}

// ---- pipelined host entry points: enqueue and return; the H2D copy of call i+1 overlaps the forward of call i ----
static int submit_host_common(ievm_handle* h, int dtype, const void* x_host, int n, void* logits_host, int in_mode,
                              int64_t* ticket) {
  if (!h || !x_host || !logits_host || !ticket) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (h->dtype != dtype) return fail(IEVM_ERR_BAD_ARG, "engine dtype does not match this entry point");
  if (n <= 0 || n > h->max_batch) return fail(IEVM_ERR_BAD_ARG, "batch %d outside [1, %d]", n, h->max_batch);
  if (in_mode == kInU8Resize && !h->rs_out) return fail(IEVM_ERR_BAD_ARG, "call ievm_set_resize first");
  DeviceGuard guard(h->device);
  const size_t in_elem = in_mode != kInNative ? 1 : (dtype == IEVM_DTYPE_I8 ? 4 : 2);
  const size_t out_elem = dtype == IEVM_DTYPE_I8 ? 4 : 2;
  const size_t per_img = in_mode == kInU8Resize ? static_cast<size_t>(3) * h->rs_in_h * h->rs_in_w
                                                : static_cast<size_t>(h->in_c) * h->in_h * h->in_w * in_elem;
  ievm_handle::HostSlot& sl = h->slots[h->next_ticket & 1];
  if (sl.ticket >= 0) {              // the slot's previous call must have left the device (normally long done)
    if (int rc = check_stuck(h, cudaEventSynchronize(sl.done), "submit: previous call of this slot")) return rc;
    sl.ticket = -1;
  }
  const size_t need = per_img * h->max_batch;
  if (sl.in_bytes < need) {
    if (sl.dev_in) {
      for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);    // graphs captured on the old staging buffer
      h->graphs.clear();
      CUDA_TRY(cudaFree(sl.dev_in));
      sl.dev_in = nullptr;
      sl.in_bytes = 0;
    }
    CUDA_TRY(cudaMalloc(&sl.dev_in, need + 256));
    sl.in_bytes = need;
  }
  if (!sl.dev_out) CUDA_TRY(cudaMalloc(&sl.dev_out, out_elem * h->classes * h->max_batch));
  cudaStream_t s = h->own_stream;
  CUDA_TRY(cudaMemcpyAsync(sl.dev_in, x_host, per_img * n, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(cudaEventRecord(sl.copied, h->copy_stream));
  CUDA_TRY(cudaStreamWaitEvent(s, sl.copied, 0));
  if (int rc = forward_common(h, dtype, sl.dev_in, n, sl.dev_out, s, in_mode)) return rc;
  CUDA_TRY(cudaMemcpyAsync(logits_host, sl.dev_out, out_elem * h->classes * n, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaEventRecord(sl.done, s));
  sl.ticket = h->next_ticket;
  *ticket = h->next_ticket++;
  return IEVM_OK;
}

int ievm_submit_i8_host(ievm_handle* h, const float* x_host, int n, float* logits_host, int64_t* ticket) {
  return submit_host_common(h, IEVM_DTYPE_I8, x_host, n, logits_host, kInNative, ticket);
}
int ievm_submit_f16_host(ievm_handle* h, const void* x_host, int n, void* logits_host, int64_t* ticket) {
  return submit_host_common(h, IEVM_DTYPE_F16, x_host, n, logits_host, kInNative, ticket);
}
int ievm_submit_u8_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host, int64_t* ticket) {
  return submit_host_common(h, IEVM_DTYPE_I8, x_nhwc_host, n, logits_host, kInU8, ticket);
}
int ievm_submit_u8_resize_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host, int64_t* ticket) {
  return submit_host_common(h, IEVM_DTYPE_I8, x_nhwc_host, n, logits_host, kInU8Resize, ticket);
}

int ievm_wait(ievm_handle* h, int64_t ticket) {
  if (!h) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (ticket < 0 || ticket >= h->next_ticket) return fail(IEVM_ERR_BAD_ARG, "ievm_wait: unknown ticket %lld", (long long)ticket);
  ievm_handle::HostSlot& sl = h->slots[ticket & 1];
  if (sl.ticket != ticket) return IEVM_OK;          // already waited for (or overtaken by a later submit, which waited)
  DeviceGuard guard(h->device);
  const int rc = check_stuck(h, cudaEventSynchronize(sl.done), "ievm_wait");
  sl.ticket = -1;
  return rc;
}

int ievm_set_wait_limit_ms(int device, int64_t ms) {
  if (ms < 0) return fail(IEVM_ERR_BAD_ARG, "ievm_set_wait_limit_ms: negative limit");
  DeviceGuard guard(device);
  const unsigned long long ns = static_cast<unsigned long long>(ms) * 1000000ull;
  CUDA_TRY(cudaMemcpyToSymbol(g_wait_limit_ns, &ns, sizeof(ns)));
  return IEVM_OK;
}

int ievm_probe_mma_peak(int device, int dtype, int iters, double* tera_ops) {
  if (!tera_ops || iters <= 0 || (dtype != IEVM_DTYPE_I8 && dtype != IEVM_DTYPE_F16))
    return fail(IEVM_ERR_BAD_ARG, "ievm_probe_mma_peak: bad arguments");
  DeviceGuard guard(device);
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(IEVM_ERR_UNSUPPORTED, "device is sm_%d%d; this build is sm_100a only", prop.major, prop.minor);
  const int smem = 1024 + 256 * 128 + 64;
  unsigned int* fail_flag = nullptr;
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&fail_flag), sizeof(unsigned int)));
  CUDA_TRY(cudaMemset(fail_flag, 0, sizeof(unsigned int)));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  cudaError_t e = cudaSuccess;
  for (int rep = 0; rep < 2 && e == cudaSuccess; ++rep) {       // the first launch warms up
    if (rep == 1) cudaEventRecord(e0);
    if (dtype == IEVM_DTYPE_I8) {
      e = cudaFuncSetAttribute(probe_mma_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      if (e == cudaSuccess) probe_mma_kernel<0><<<prop.multiProcessorCount, 128, smem>>>(iters, fail_flag);
    } else {
      e = cudaFuncSetAttribute(probe_mma_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      if (e == cudaSuccess) probe_mma_kernel<1><<<prop.multiProcessorCount, 128, smem>>>(iters, fail_flag);
    }
    if (e == cudaSuccess) e = cudaGetLastError();
  }
  cudaEventRecord(e1);
  if (e == cudaSuccess) e = cudaEventSynchronize(e1);
  float ms = 0.f;
  if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
  unsigned int failed = 0;
  if (e == cudaSuccess) e = cudaMemcpy(&failed, fail_flag, sizeof(failed), cudaMemcpyDeviceToHost);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(fail_flag);
  if (e != cudaSuccess) return fail(IEVM_ERR_CUDA, "ievm_probe_mma_peak: %s", cudaGetErrorString(e));
  if (failed || ms <= 0.f) return fail(IEVM_ERR_CUDA, "ievm_probe_mma_peak: the instruction stream did not complete");
  const double k_per_mma = dtype == IEVM_DTYPE_I8 ? 32.0 : 16.0;
  const double ops = 2.0 * 128.0 * 256.0 * k_per_mma * 16.0 * iters * prop.multiProcessorCount;
  *tera_ops = ops / (ms * 1e-3) / 1e12;
  return IEVM_OK;
}

int ievm_set_input_lut(ievm_handle* h, const uint8_t* lut768) {
  if (!h || !lut768) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (h->dtype != IEVM_DTYPE_I8) return fail(IEVM_ERR_BAD_ARG, "the 8-bit image input path belongs to the INT8 engine");
  DeviceGuard guard(h->device);
  if (!h->lut_dev) {
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, 768));
    h->owned.push_back(p);
    h->lut_dev = static_cast<uint8_t*>(p);
  }
  CUDA_TRY(cudaMemcpy(h->lut_dev, lut768, 768, cudaMemcpyHostToDevice));
  return IEVM_OK;
}

int ievm_forward_u8(ievm_handle* h, const uint8_t* x_nhwc, int n, float* logits, void* stream) {
  return forward_common(h, IEVM_DTYPE_I8, x_nhwc, n, logits, stream, kInU8);
}

int ievm_forward_u8_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host) {
  return forward_host_common(h, IEVM_DTYPE_I8, x_nhwc_host, n, logits_host, kInU8);
}

int ievm_set_resize(ievm_handle* h, int src_h, int src_w, const int32_t* bounds_w, const int32_t* kk_w, int ksize_w,
                    const int32_t* bounds_h, const int32_t* kk_h, int ksize_h) {
  if (!h || src_h <= 0 || src_w <= 0 || !bounds_w || !kk_w || !bounds_h || !kk_h || ksize_w <= 0 || ksize_h <= 0)
    return fail(IEVM_ERR_BAD_ARG, "ievm_set_resize: bad arguments");
  if (h->dtype != IEVM_DTYPE_I8) return fail(IEVM_ERR_BAD_ARG, "the 8-bit image input path belongs to the INT8 engine");
  DeviceGuard guard(h->device);
  CUDA_TRY(cudaDeviceSynchronize());
  for (void* q : {static_cast<void*>(h->rs_bounds_w), static_cast<void*>(h->rs_bounds_h), static_cast<void*>(h->rs_kk_w),
                  static_cast<void*>(h->rs_kk_h), static_cast<void*>(h->rs_tmp), static_cast<void*>(h->rs_out)})
    if (q) cudaFree(q);
  h->rs_bounds_w = h->rs_bounds_h = nullptr;
  h->rs_kk_w = h->rs_kk_h = nullptr;
  h->rs_tmp = h->rs_out = nullptr;
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
  h->graphs.clear();
  h->rs_in_h = src_h; h->rs_in_w = src_w; h->rs_ksize_w = ksize_w; h->rs_ksize_h = ksize_h;
  auto up = [&](const int32_t* src, size_t count, void** dst) -> cudaError_t {
    cudaError_t e = cudaMalloc(dst, count * sizeof(int32_t));
    return e != cudaSuccess ? e : cudaMemcpy(*dst, src, count * sizeof(int32_t), cudaMemcpyHostToDevice);
  };
  CUDA_TRY(up(bounds_w, static_cast<size_t>(h->in_w) * 2, reinterpret_cast<void**>(&h->rs_bounds_w)));
  CUDA_TRY(up(kk_w, static_cast<size_t>(h->in_w) * ksize_w, reinterpret_cast<void**>(&h->rs_kk_w)));
  CUDA_TRY(up(bounds_h, static_cast<size_t>(h->in_h) * 2, reinterpret_cast<void**>(&h->rs_bounds_h)));
  CUDA_TRY(up(kk_h, static_cast<size_t>(h->in_h) * ksize_h, reinterpret_cast<void**>(&h->rs_kk_h)));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&h->rs_tmp), static_cast<size_t>(h->max_batch) * src_h * h->in_w * 3 + 16));
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&h->rs_out), static_cast<size_t>(h->max_batch) * h->in_h * h->in_w * 3 + 16));
  return IEVM_OK;
}

int ievm_forward_u8_resize(ievm_handle* h, const uint8_t* x_nhwc, int n, float* logits, void* stream) {
  return forward_common(h, IEVM_DTYPE_I8, x_nhwc, n, logits, stream, kInU8Resize);
}

int ievm_forward_u8_resize_host(ievm_handle* h, const uint8_t* x_nhwc_host, int n, float* logits_host) {
  return forward_host_common(h, IEVM_DTYPE_I8, x_nhwc_host, n, logits_host, kInU8Resize);
}

int ievm_debug_resize(ievm_handle* h, const uint8_t* x_dev, int n, uint8_t* out_host, uint64_t out_bytes) {
  if (!h || !x_dev || !out_host || n <= 0 || n > h->max_batch) return fail(IEVM_ERR_BAD_ARG, "debug_resize: bad arguments");
  const size_t bytes = static_cast<size_t>(n) * h->in_h * h->in_w * 3;
  if (out_bytes < bytes) return fail(IEVM_ERR_BAD_ARG, "debug_resize: host buffer too small");
  DeviceGuard guard(h->device);
  CUDA_TRY(cudaDeviceSynchronize());      // parity hook: whatever stream wrote the input is done
  if (int rc = launch_resize(h, x_dev, n, h->own_stream)) return rc;
  CUDA_TRY(cudaStreamSynchronize(h->own_stream));
  const uint8_t* src = (h->rs_in_h == h->in_h && h->rs_in_w == h->in_w) ? x_dev : h->rs_out;
  CUDA_TRY(cudaMemcpy(out_host, src, bytes, cudaMemcpyDeviceToHost));
  return IEVM_OK;
}

int ievm_set_option(ievm_handle* h, const char* name, int value) {
  if (!h || !name) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (!strcmp(name, "conv_impl")) {
    if (value != 0 && value != 1) return fail(IEVM_ERR_BAD_ARG, "conv_impl must be 0 or 1");
    h->conv_impl = value;
    for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
    h->graphs.clear();
    return IEVM_OK;
  }
  if (!strcmp(name, "profile")) {
    h->profile = value ? 1 : 0;
    std::fill(h->prof_ms.begin(), h->prof_ms.end(), 0.0);
    std::fill(h->prof_calls.begin(), h->prof_calls.end(), 0);
    return IEVM_OK;
  }
  if (!strcmp(name, "use_graph")) {
    h->use_graph = value ? 1 : 0;
    return IEVM_OK;
  }
  if (!strcmp(name, "dual")) {        // 0: every 1x1 downsample conv is a launch of its own (conv_dual.cuh off)
    h->opt_dual = value ? 1 : 0;
    for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);
    h->graphs.clear();
    return IEVM_OK;
  }
  if (!strcmp(name, "keep_tensors")) {
    if ((value ? 1 : 0) == h->keep_tensors) return IEVM_OK;
    h->keep_tensors = value ? 1 : 0;
    DeviceGuard guard(h->device);
    CUDA_TRY(cudaDeviceSynchronize());
    if (int rc = assign_buffers(h)) return rc;
    return encode_maps(h);
  }
  if (!strcmp(name, "observe")) {
    // calibration mode (observe.cuh): 0 = off, 1 = (min, max) per batch, 2 = additionally torch.histc over the running
    // range (HistogramObserver).  (Re)starts the log and the running ranges; the head also writes its avgpool output.
    if (h->dtype != IEVM_DTYPE_F16) return fail(IEVM_ERR_UNSUPPORTED, "observers run on the FP16 engine (the float forward of PTQ calibration)");
    if (value < 0 || value > 2) return fail(IEVM_ERR_BAD_ARG, "observe must be 0, 1 or 2");
    const int points = static_cast<int>(h->tensors.size()) + 2;
    if (points > kObsMaxPoints) return fail(IEVM_ERR_UNSUPPORTED, "more than %d observation points", kObsMaxPoints);
    DeviceGuard guard(h->device);
    CUDA_TRY(cudaDeviceSynchronize());
    for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.first);   // the pooled-output pointer is baked into captured launches
    h->graphs.clear();
    h->obs_records = 0;
    h->obs_mode = value;
    if (!value) {
      h->obs_pooled = nullptr;
      return IEVM_OK;
    }
    auto alloc = [&](size_t bytes, void** out) -> int {
      CUDA_TRY(cudaMalloc(out, std::max<size_t>(bytes, 16)));
      h->owned.push_back(*out);
      return IEVM_OK;
    };
    if (!h->obs_log) {
      if (int rc = alloc(static_cast<size_t>(kObsMaxRecords) * points * 2 * sizeof(uint32_t), reinterpret_cast<void**>(&h->obs_log))) return rc;
      if (int rc = alloc(static_cast<size_t>(kObsMaxPoints) * 2 * sizeof(uint32_t), reinterpret_cast<void**>(&h->obs_run))) return rc;
      for (int i = 0; i < kObsMaxPoints; ++i) h->obs_group[i] = i;
    }
    if (value == 2 && !h->obs_hist)
      if (int rc = alloc(static_cast<size_t>(kObsHistRecords) * points * kObsBins * sizeof(uint32_t), reinterpret_cast<void**>(&h->obs_hist))) return rc;
    if (!h->obs_pooled_alloc) {
      int head_cin = 0;
      for (const LayerPlan& L : h->layers)
        if (L.d.op == IEVM_OP_HEAD) head_cin = L.d.cin;
      if (int rc = alloc(static_cast<size_t>(h->max_batch) * head_cin * sizeof(__half), reinterpret_cast<void**>(&h->obs_pooled_alloc))) return rc;
    }
    h->obs_pooled = h->obs_pooled_alloc;
    observe_init_kernel<<<1, 256>>>(h->obs_run, kObsMaxPoints);
    CUDA_TRY(cudaGetLastError());
    if (h->obs_hist) CUDA_TRY(cudaMemset(h->obs_hist, 0, static_cast<size_t>(kObsHistRecords) * points * kObsBins * sizeof(uint32_t)));
    CUDA_TRY(cudaDeviceSynchronize());
    return IEVM_OK;
  }
  return fail(IEVM_ERR_BAD_ARG, "unknown option '%s'", name);
}

int ievm_observer_points(const ievm_handle* h) { return h ? static_cast<int>(h->tensors.size()) + 2 : 0; }

int ievm_observer_capacity(const ievm_handle* h) {
  if (!h || !h->obs_mode) return 0;
  return h->obs_mode == 2 ? kObsHistRecords : kObsMaxRecords;
}

int ievm_observer_set_groups(ievm_handle* h, const int32_t* group_of_point, int points) {
  if (!h || !group_of_point) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (!h->obs_log) return fail(IEVM_ERR_BAD_ARG, "ievm_observer_set_groups: set option observe first");
  if (points != static_cast<int>(h->tensors.size()) + 2) return fail(IEVM_ERR_BAD_ARG, "expected %zu points", h->tensors.size() + 2);
  if (h->obs_records != 0) return fail(IEVM_ERR_BAD_ARG, "ievm_observer_set_groups: the log is not empty");
  for (int i = 0; i < points; ++i) {
    if (group_of_point[i] < 0 || group_of_point[i] >= kObsMaxPoints) return fail(IEVM_ERR_BAD_ARG, "group %d out of range", group_of_point[i]);
    h->obs_group[i] = group_of_point[i];
  }
  return IEVM_OK;
}

int ievm_observe(ievm_handle* h, const float* x_f32, void* stream) {
  if (!h) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (!h->obs_mode || !h->obs_log || !h->obs_pooled) return fail(IEVM_ERR_BAD_ARG, "ievm_observe: set option observe first");
  if (!h->keep_tensors) return fail(IEVM_ERR_BAD_ARG, "ievm_observe: needs keep_tensors=1 (every tensor in its own buffer)");
  if (h->last_n <= 0 || !h->last_x || !h->last_logits) return fail(IEVM_ERR_BAD_ARG, "ievm_observe: no forward to observe");
  const int cap = h->obs_mode == 2 ? kObsHistRecords : kObsMaxRecords;
  if (h->obs_records >= cap) return fail(IEVM_ERR_OOM, "ievm_observe: observer log full (%d records): read and clear it", cap);
  const void* x0 = x_f32 ? static_cast<const void*>(x_f32) : h->last_x;
  if (reinterpret_cast<uintptr_t>(x0) % 16 != 0 || reinterpret_cast<uintptr_t>(h->last_logits) % 16 != 0)
    return fail(IEVM_ERR_BAD_ARG, "ievm_observe: input / logits buffers must be 16-byte aligned");
  DeviceGuard guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int T = static_cast<int>(h->tensors.size());
  const int points = T + 2;
  const int n = h->last_n;
  int head_cin = 0;
  for (const LayerPlan& L : h->layers)
    if (L.d.op == IEVM_OP_HEAD) head_cin = L.d.cin;
  // one table for all points; every point gets blocks in proportion to its size (a thread streams ~4 vectors)
  ObsTable tab;
  memset(&tab, 0, sizeof(tab));
  int nblocks = 0;
  auto add = [&](const void* data, long long count, int pitch, int c_real, bool f32) {
    ObsPoint& P = tab.pt[tab.n];
    P.data = data;
    P.count = data ? count : 0;
    P.pitch = pitch;
    P.c_real = c_real;
    P.is_f32 = f32 ? 1 : 0;
    P.group = h->obs_group[tab.n];
    P.first_block = nblocks;
    const long long nvec = P.count / (f32 ? 4 : 8);
    nblocks += static_cast<int>(std::min<long long>(std::max<long long>((nvec + 1023) / 1024, 1), 4LL * h->num_sms));
    ++tab.n;
  };
  add(x0, static_cast<long long>(n) * h->in_c * h->in_h * h->in_w, 1, 1, x_f32 != nullptr);
  for (int id = 1; id < T; ++id) {
    const TensorInfo& t = h->tensors[id];
    const bool ok = t.buffer >= 0 && t.elem == 2;
    add(ok ? tensor_ptr(h, id) : nullptr, static_cast<long long>(n) * t.h * t.w * t.pitch, t.pitch, t.c, false);   // null: "nothing observed"
  }
  add(h->obs_pooled, static_cast<long long>(n) * head_cin, 1, 1, false);
  add(h->last_logits, static_cast<long long>(n) * h->classes, 1, 1, false);
  tab.total_blocks = nblocks;
  bool capturing = false;
  if (int rc = order_begin(h, s, &capturing)) return rc;
  uint32_t* rec = h->obs_log + static_cast<size_t>(h->obs_records) * points * 2;
  observe_init_kernel<<<(2 * points + 255) / 256, 256, 0, s>>>(rec, points);
  observe_minmax_multi_kernel<<<nblocks, 256, 0, s>>>(tab, rec, h->obs_run);
  if (h->obs_mode == 2)
    observe_hist_multi_kernel<<<nblocks, 256, 0, s>>>(tab, h->obs_run, h->obs_hist + static_cast<size_t>(h->obs_records) * points * kObsBins);
  CUDA_TRY(cudaGetLastError());
  ++h->obs_records;
  return order_end(h, s, capturing);
}

int ievm_observer_read(ievm_handle* h, float* minmax_host, int max_records) {
  if (!h || !minmax_host || max_records < 0) return fail(IEVM_ERR_BAD_ARG, "ievm_observer_read: bad arguments");
  const int nrec = std::min(h->obs_records, max_records);
  if (nrec == 0) return 0;
  DeviceGuard guard(h->device);
  if (int rc = check_stuck(h, cudaDeviceSynchronize(), "observer_read sync")) return rc;
  const size_t words = static_cast<size_t>(nrec) * (h->tensors.size() + 2) * 2;
  std::vector<uint32_t> enc(words);
  CUDA_TRY(cudaMemcpy(enc.data(), h->obs_log, words * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < words; ++i) minmax_host[i] = obs_decode(enc[i]);
  return nrec;
}

int ievm_observer_read_hist(ievm_handle* h, uint32_t* hist_host, float* range_host, int max_records) {
  if (!h || !hist_host || max_records < 0) return fail(IEVM_ERR_BAD_ARG, "ievm_observer_read_hist: bad arguments");
  if (h->obs_mode != 2 || !h->obs_hist) return fail(IEVM_ERR_BAD_ARG, "ievm_observer_read_hist: set option observe=2 first");
  const int nrec = std::min(h->obs_records, max_records);
  DeviceGuard guard(h->device);
  if (int rc = check_stuck(h, cudaDeviceSynchronize(), "observer_read_hist sync")) return rc;
  if (range_host) {       // running (min, max) per observer group, as of the last record
    uint32_t enc[2 * kObsMaxPoints];
    CUDA_TRY(cudaMemcpy(enc, h->obs_run, sizeof(enc), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 2 * kObsMaxPoints; ++i) range_host[i] = obs_decode(enc[i]);
  }
  if (nrec == 0) return 0;
  const size_t words = static_cast<size_t>(nrec) * (h->tensors.size() + 2) * kObsBins;
  CUDA_TRY(cudaMemcpy(hist_host, h->obs_hist, words * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  return nrec;
}

int ievm_observer_clear(ievm_handle* h) {
  if (!h) return fail(IEVM_ERR_BAD_ARG, "null argument");
  if (!h->obs_mode) return fail(IEVM_ERR_BAD_ARG, "ievm_observer_clear: set option observe first");
  DeviceGuard guard(h->device);
  CUDA_TRY(cudaDeviceSynchronize());
  if (h->obs_hist && h->obs_records > 0)
    CUDA_TRY(cudaMemset(h->obs_hist, 0, static_cast<size_t>(h->obs_records) * (h->tensors.size() + 2) * kObsBins * sizeof(uint32_t)));
  h->obs_records = 0;
  return IEVM_OK;
}

int ievm_num_tensors(const ievm_handle* h) { return h ? static_cast<int>(h->tensors.size()) : 0; }

int ievm_tensor_shape(const ievm_handle* h, int id, int32_t out6[6]) {
  if (!h || id < 0 || id >= static_cast<int>(h->tensors.size()) || !out6) return fail(IEVM_ERR_BAD_ARG, "bad tensor id");
  const TensorInfo& t = h->tensors[id];
  out6[0] = h->last_n; out6[1] = t.h; out6[2] = t.w; out6[3] = t.c; out6[4] = t.pitch; out6[5] = t.elem;
  return IEVM_OK;
}

int ievm_launches_per_forward(const ievm_handle* h) {
  if (!h) return 0;
  const int n = h->last_n > 0 ? h->last_n : h->max_batch;
  int duals = 0;
  if (dual_active(h))
    for (const LayerPlan& L : h->layers) duals += L.dual_of >= 0 ? 1 : 0;
  if (front_end_is_v2(h)) return static_cast<int>(h->layers.size()) - 1 - duals;
  if (front_end_is_chunked(h))
    return 3 * ((n + h->front_chunk - 1) / h->front_chunk) + static_cast<int>(h->layers.size()) - 2 - duals;
  return static_cast<int>(h->layers.size()) + (h->dtype == IEVM_DTYPE_I8 ? 1 : 0) - duals;
}

int ievm_layer_launch(const ievm_handle* h, int layer) {
  if (!h || layer < 0 || layer >= static_cast<int>(h->layers.size())) return -1;
  if (front_end_is_v2(h) && layer == 1) return 0;
  const LayerPlan& L = h->layers[layer];
  const int mate = L.dual_partner >= 0 ? L.dual_partner : L.dual_of;
  return (dual_active(h) && mate >= 0) ? std::min(mate, layer) : layer;
}

int ievm_profile_read(const ievm_handle* h, int max_slots, float* ms_sum, int32_t* calls) {
  if (!h || !ms_sum || !calls) return fail(IEVM_ERR_BAD_ARG, "null argument");
  const int slots = static_cast<int>(h->prof_ms.size());
  for (int i = 0; i < max_slots; ++i) {
    ms_sum[i] = i < slots ? static_cast<float>(h->prof_ms[i]) : 0.f;
    calls[i] = i < slots ? h->prof_calls[i] : 0;
  }
  return slots;
}

int ievm_debug_read_tensor(ievm_handle* h, int id, void* host_out, uint64_t host_bytes) {
  if (!h || id < 0 || id >= static_cast<int>(h->tensors.size()) || !host_out) return fail(IEVM_ERR_BAD_ARG, "bad tensor id");
  const TensorInfo& t = h->tensors[id];
  if (t.buffer < 0) return fail(IEVM_ERR_BAD_ARG, "tensor %d has no engine-owned buffer", id);
  const size_t row = static_cast<size_t>(t.w) * t.pitch * t.elem;
  const size_t bytes = row * t.h * h->last_n;
  if (host_bytes < bytes) return fail(IEVM_ERR_BAD_ARG, "host buffer too small: need %zu bytes", bytes);
  DeviceGuard guard(h->device);
  if (int rc = check_stuck(h, cudaDeviceSynchronize(), "debug_read_tensor sync")) return rc;
  if (t.hp > 0) {   // strip the border: one 2-D copy per image
    const size_t src_row = static_cast<size_t>(t.wp) * t.pitch * t.elem;
    for (int i = 0; i < h->last_n; ++i) {
      const uint8_t* src = static_cast<const uint8_t*>(tensor_ptr(h, id)) + i * t.bytes_per_image() +
                           t.pad_t * src_row + static_cast<size_t>(t.pad_l) * t.pitch * t.elem;
      CUDA_TRY(cudaMemcpy2D(static_cast<uint8_t*>(host_out) + i * row * t.h, row, src, src_row, row, t.h,
                            cudaMemcpyDeviceToHost));
    }
    return IEVM_OK;
  }
  CUDA_TRY(cudaMemcpy(host_out, tensor_ptr(h, id), bytes, cudaMemcpyDeviceToHost));
  return IEVM_OK;
}

int ievm_debug_conv_acc(ievm_handle* h, int layer, int n, int32_t* host_out, uint64_t host_bytes) {
  if (!h || layer < 0 || layer >= static_cast<int>(h->layers.size()) || !host_out) return fail(IEVM_ERR_BAD_ARG, "bad layer");
  const LayerPlan& L = h->layers[layer];
  if (L.d.op != IEVM_OP_CONV || (L.is_stem && h->dtype != IEVM_DTYPE_I8))
    return fail(IEVM_ERR_BAD_ARG, "layer %d is not a tensor-core conv", layer);
  if (!h->keep_tensors) return fail(IEVM_ERR_BAD_ARG, "set keep_tensors=1 before the forward whose accumulators you want");
  const size_t bytes = static_cast<size_t>(n) * L.ho * L.wo * L.cout_pad * sizeof(int32_t);
  if (host_bytes < bytes) return fail(IEVM_ERR_BAD_ARG, "host buffer too small: need %zu bytes", bytes);
  DeviceGuard guard(h->device);
  int32_t* dacc = nullptr;
  CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&dacc), bytes));
  cudaDeviceSynchronize();                  // parity hook: the forward that produced this layer's input is done
  // a layer that the forward runs as half of a dual launch is re-run the same way, so the accumulators are that kernel's
  int rc = L.is_stem ? launch_stem_tc(h, L, static_cast<const uint8_t*>(tensor_ptr(h, 0)),
                                      static_cast<uint8_t*>(tensor_ptr(h, L.d.out_tensor)), n, h->own_stream, dacc)
           : (dual_active(h) && L.dual_partner >= 0) ? launch_conv_dual(h, L, n, h->own_stream, dacc, nullptr)
           : (dual_active(h) && L.dual_of >= 0)      ? launch_conv_dual(h, h->layers[L.dual_of], n, h->own_stream, nullptr, dacc)
                                                     : launch_conv(h, L, n, h->own_stream, dacc);
  if (rc == IEVM_OK) rc = check_stuck(h, cudaStreamSynchronize(h->own_stream), "debug_conv_acc");
  if (rc == IEVM_OK && cudaMemcpy(host_out, dacc, bytes, cudaMemcpyDeviceToHost) != cudaSuccess)
    rc = fail(IEVM_ERR_CUDA, "accumulator copy failed");
  cudaFree(dacc);
  return rc;
}

int ievm_debug_frontend(ievm_handle* h, const void* x_dev, int n, void* pooled_host, uint64_t pooled_bytes,
                        int32_t* acc_host, uint64_t acc_bytes) {
  if (!h || !x_dev || !pooled_host || n <= 0 || n > h->max_batch) return fail(IEVM_ERR_BAD_ARG, "debug_frontend: bad arguments");
  if (!h->front2_ok) return fail(IEVM_ERR_UNSUPPORTED, "this network's front end does not fit the fused v2 kernel");
  const LayerPlan& Ls = h->layers[0];
  const LayerPlan& Lp = h->layers[1];
  const size_t pooled = static_cast<size_t>(n) * Lp.ho * Lp.wo * Ls.cout_pad * h->elem;
  const size_t acc = static_cast<size_t>(n) * Ls.ho * Ls.wo * Ls.cout_pad * sizeof(int32_t);
  if (pooled_bytes < pooled || (acc_host && acc_bytes < acc)) return fail(IEVM_ERR_BAD_ARG, "debug_frontend: host buffer too small");
  DeviceGuard guard(h->device);
  int32_t* dacc = nullptr;
  if (acc_host) CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&dacc), acc));
  cudaDeviceSynchronize();                  // parity hook: earlier work on other streams is done
  int rc = launch_frontend2(h, x_dev, n, h->own_stream, dacc);
  if (rc == IEVM_OK) rc = check_stuck(h, cudaStreamSynchronize(h->own_stream), "debug_frontend");
  if (rc == IEVM_OK && cudaMemcpy(pooled_host, tensor_ptr(h, Lp.d.out_tensor), pooled, cudaMemcpyDeviceToHost) != cudaSuccess)
    rc = fail(IEVM_ERR_CUDA, "pooled tensor copy failed");
  if (rc == IEVM_OK && acc_host && cudaMemcpy(acc_host, dacc, acc, cudaMemcpyDeviceToHost) != cudaSuccess)
    rc = fail(IEVM_ERR_CUDA, "accumulator copy failed");
  if (dacc) cudaFree(dacc);
  h->last_n = n;
  return rc;
}

int ievm_probe_im2col(const void* in_dev, int n, int h, int w, int c_pitch, int ksize, int stride, int pad,
                      int kc_bytes, int m0, int tap_x, int tap_y, int c0, void* out_dev) {
  if (!in_dev || !out_dev || (kc_bytes != 64 && kc_bytes != 128)) return fail(IEVM_ERR_BAD_ARG, "probe: bad arguments");
  if (int rc = load_driver_entry_points()) return rc;
  CUtensorMap tmap;
  cuuint64_t dims[4] = {(cuuint64_t)c_pitch, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c_pitch, (cuuint64_t)w * c_pitch, (cuuint64_t)h * w * c_pitch};
  int lower[2] = {-pad, -pad};
  int upper[2] = {pad - (ksize - 1), pad - (ksize - 1)};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  const CUresult r = g_encode_im2col(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(in_dev), dims, strides,
                                     lower, upper, (cuuint32_t)kc_bytes, kTileM, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                     kc_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "probe: cuTensorMapEncodeIm2col CUresult %d", (int)r);
  const int ho = (h + 2 * pad - ksize) / stride + 1, wo = (w + 2 * pad - ksize) / stride + 1;
  const int img = m0 / (ho * wo), rem = m0 % (ho * wo);
  const int oy = rem / wo, ox = rem % wo;
  unsigned int* stuck_host = nullptr;
  unsigned int* stuck_dev = nullptr;
  CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&stuck_host), sizeof(unsigned int), cudaHostAllocMapped));
  *stuck_host = 0;
  CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&stuck_dev), stuck_host, 0));
  const int bytes = kTileM * kc_bytes;
  probe_im2col_kernel<<<1, 128, bytes + 1024 + 64>>>(tmap, c0, ox * stride - pad, oy * stride - pad, img, tap_x, tap_y,
                                                     bytes, static_cast<uint8_t*>(out_dev), stuck_dev);
  const cudaError_t e = cudaDeviceSynchronize();
  const unsigned code = *stuck_host;
  cudaFreeHost(stuck_host);
  if (e != cudaSuccess) return fail(IEVM_ERR_CUDA, "probe_im2col: %s (stuck code 0x%x)", cudaGetErrorString(e), code);
  return IEVM_OK;
}

int ievm_probe_patch(const void* in_dev, int n, int h, int w, int c_pitch, int rb, int img, int w0, int h0, int box_w,
                     int box_h, void* out_dev) {
  if (!in_dev || !out_dev || (rb != 64 && rb != 128)) return fail(IEVM_ERR_BAD_ARG, "probe_patch: bad arguments");
  if (int rc = load_driver_entry_points()) return rc;
  CUtensorMap tmap;
  cuuint64_t dims[4] = {(cuuint64_t)c_pitch, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c_pitch, (cuuint64_t)w * c_pitch, (cuuint64_t)h * w * c_pitch};
  cuuint32_t box[4] = {(cuuint32_t)rb, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = g_encode_tiled(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void*>(in_dev), dims, strides, box,
                                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                    rb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                                    CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(IEVM_ERR_CUDA, "probe_patch: cuTensorMapEncodeTiled CUresult %d", (int)r);
  unsigned int* stuck_host = nullptr;
  unsigned int* stuck_dev = nullptr;
  CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&stuck_host), sizeof(unsigned int), cudaHostAllocMapped));
  *stuck_host = 0;
  CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&stuck_dev), stuck_host, 0));
  const int bytes = box_w * box_h * rb;
  CUDA_TRY(cudaFuncSetAttribute(probe_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes + 2048));
  probe_patch_kernel<<<1, 128, bytes + 2048>>>(tmap, 0, w0, h0, img, bytes, static_cast<uint8_t*>(out_dev), stuck_dev);
  const cudaError_t e = cudaDeviceSynchronize();
  const unsigned code = *stuck_host;
  cudaFreeHost(stuck_host);
  if (e != cudaSuccess) return fail(IEVM_ERR_CUDA, "probe_patch: %s (stuck code 0x%x)", cudaGetErrorString(e), code);
  return IEVM_OK;
}

#ifdef IEVM_EXP_TIMING
// A/B instrumentation only (never in the default build): per-layer, per-CTA role timers of conv_tc_kernel.
int ievm_exp_timing_read(unsigned long long* host, int clear) {
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpyFromSymbol(host, g_exp_timing, sizeof(g_exp_timing)));
  if (clear) {
    void* sym = nullptr;
    CUDA_TRY(cudaGetSymbolAddress(&sym, g_exp_timing));
    CUDA_TRY(cudaMemset(sym, 0, sizeof(g_exp_timing)));
  }
  return kExpSlots * kExpCtas * kExpWords;
}
#endif

int ievm_count_correct(const void* logits, int dtype, const int64_t* labels, int n, int classes, uint64_t* counters2,
                       void* stream) {
  if (!logits || !labels || !counters2 || n <= 0 || classes <= 0) return fail(IEVM_ERR_BAD_ARG, "ievm_count_correct: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned blocks = static_cast<unsigned>((n + 127) / 128);
  if (dtype == IEVM_DTYPE_F16)
    count_correct_kernel<__half><<<blocks, 128, 0, st>>>(static_cast<const __half*>(logits), reinterpret_cast<const long long*>(labels),
                                                         n, classes, reinterpret_cast<unsigned long long*>(counters2));
  else
    count_correct_kernel<float><<<blocks, 128, 0, st>>>(static_cast<const float*>(logits), reinterpret_cast<const long long*>(labels),
                                                        n, classes, reinterpret_cast<unsigned long long*>(counters2));
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

int ievm_kd_loss(const float* s, const float* t, const int64_t* y, int n, int classes, float temperature, float* out3,
                 void* stream) {
  if (!s || !t || !y || !out3 || n <= 0 || classes <= 0) return fail(IEVM_ERR_BAD_ARG, "ievm_kd_loss: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemsetAsync(out3, 0, 3 * sizeof(float), st));
  kd_loss_kernel<<<(n + 127) / 128, 128, 0, st>>>(s, t, reinterpret_cast<const long long*>(y), n, classes,
                                                  temperature, out3);
  kd_finalize_kernel<<<1, 32, 0, st>>>(out3, 1.0f / static_cast<float>(n));
  CUDA_TRY(cudaGetLastError());
  return IEVM_OK;
}

}  // extern "C"
