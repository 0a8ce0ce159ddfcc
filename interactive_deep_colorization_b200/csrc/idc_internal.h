// Internal declarations shared by the translation units of libidc_b200.so.
// Layout vocabulary follows the reference network (model.py): blocks model1..model10,
// activations conv1_2 ... conv10_2, hints, bins.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/idc_b200.h"

namespace idc {

constexpr int kMaxTaps = 34;  // up-layer: 4 deconv + 9 shortcut taps; Caffe hyper-column: 4x4 deconv + 2x9 conv taps
constexpr int kMaxSrc = 6;
constexpr int kMaxCls = 4;    // output parity classes of a stride-2 transposed conv

enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_LEAKY02 = 2 };

// tcgen05 engine: activations are stored as FP16 hi/lo planes of (value * 2^kActScaleLog2).
// Measured on B200 (round 1): the tensor core treats FP16 *subnormal* operands as zero, so an
// unscaled lo plane loses the low half of every activation below 0.125 (ab error 1.2e-2 instead
// of 1e-4).  Scaling by 64 keeps lo normal down to |a| = 0.002; FP16 range then covers |a| < 1023.
constexpr int kActScaleLog2 = 6;
constexpr float kActScale = 64.0f;
constexpr float kActInvScale = 1.0f / 64.0f;

// One filter tap of a gather-GEMM convolution.  For logical output pixel (y, x) the tap reads
// source pixel (y*s + ty, x*s + tx) of source `src`; out-of-range pixels read zero
// (= the reference's zero padding).  (ky, kx) is the kernel index used for weight packing.
struct Tap {
  int src;  // 0 = main source, 1 = shortcut source
  int ky, kx;
  int ty, tx;
};

// Activation buffer.  SIMT engine: p0 = float [N,H,W,C].  tcgen05 engine: p0/p1 = __half
// hi/lo planes, each [N,H,W,C]; value = hi + lo.
struct ActBuf {
  std::string name;
  int H = 0, W = 0, C = 0;
  void* p0 = nullptr;
  void* p1 = nullptr;
};

// Per-output-channel epilogue vectors (device, fp32[cout_pad]).
//   v = act(acc + bias) * scale + shift (+ gadd[n][c])
// tcgen05 engine: weights are pre-scaled per output channel by a power of two 2^e (so the FP16 lo
// term stays normal); bias is stored as bias*2^e and scale as scale*2^-e, which is exact and leaves
// the formula unchanged because ReLU / LeakyReLU are positively homogeneous.
struct Epilogue {
  float* bias = nullptr;
  float* scale = nullptr;  // BN gamma / sqrt(var + eps)   (1 when no BN)
  float* shift = nullptr;  // BN beta - mean * scale        (0 when no BN)
  int act = ACT_NONE;
  bool has_bn = false;
  bool gadd = false;  // add global-hints vector [N, cout] (row a15)
};

struct SrcDesc {
  int buf = -1;  // index into Ctx::bufs
  int s = 1;     // logical->source pixel stride (2 = read the ::2 decimation / the skip tensor)
  int cin = 0;
};

enum OpKind { OP_CONV = 0, OP_UP = 1, OP_CLASS = 2, OP_HYPER = 3 };

struct ConvOp {
  std::string name;
  int kind = OP_CONV;
  std::string wkey[kMaxSrc];  // state_dict keys, one per source (main conv / deconv, shortcut conv, ...)
  bool src_deconv[kMaxSrc] = {false, false, false, false, false, false};  // source s is a ConvTranspose2d (IOHW weights)
  int src_k[kMaxSrc] = {3, 3, 3, 3, 3, 3};   // kernel size of source s's filter (3, 4 for the transposed convs, 1)
  std::string bnkey;
  int nsrc = 1;
  SrcDesc src[kMaxSrc];
  int ncls = 1;
  int ntaps = 0;                 // taps per class
  Tap taps[kMaxCls][kMaxTaps];
  int Hl = 0, Wl = 0;            // logical output grid (per class)
  int out_buf = -1;
  int os = 1;                    // output pixel = (y*os + cls/2, x*os + cls%2)
  int cout = 0, cout_pad = 0;
  int K = 0;                     // sum over taps of cin(src)
  Epilogue epi;
  bool fuse_out_head = false;    // tcgen05 engine: model_out (128->2, tanh*110) in the epilogue
  bool out_f32 = false;          // store FP32 [M][cout_pad] instead of an activation (class logits)
  float* out_f32_ptr = nullptr;  // where (ctx->logits or ctx->logits313)
  // packed weights
  float* w_simt = nullptr;       // [ncls][K][cout_pad] fp32
  __half* w_hi = nullptr;        // [ncls*cout_pad][K] fp16 (x wscale)
  __half* w_lo = nullptr;
  // tcgen05 launch plan (filled by umma_plan_op)
  int bn_tile = 0, hbox = 0, wbox = 0;
  void* umma_plan = nullptr;
  double flops_per_image = 0;
};

// conv1_1 weights as a kernel parameter (constant bank): [36][64] with k = tap*4 + cin, then bias
struct Conv11Weights {
  float w[36 * 64];
  float b[64];
};

// Plan-time options (idc_set_option).  -1 = automatic.  They replace the IDC_* environment switches of
// round 1: a C ABI that is embedded in someone else's process must not read process-global state.
struct Options {
  int halo = 1;           // halo-tile A operand: 0 off, 1 = 128-column stride-1 3x3 layers that fill the machine, 3 = every eligible op
  int pairs = 1;          // cta_group::2: 0 never, 1 = launches that give every SM pair >= 2 tiles, 2 = always
  int mt = -1;            // M-tiles per CTA tile on the <= 128-column layers (1 / 2)
  int chunk_kb = -1;      // k-blocks summed in TMEM before the FP32 round-to-nearest add
  int split_k = -1;       // K slices per tile on launches that cannot fill the machine
  int host_pipe = 1;      // idc_forward_host: chunked copy/compute overlap for batches >= 8
  int pdl = 1;            // programmatic dependent launch between the kernels of a forward
  int split_pairs = 1;    // cta_group::2 on the split-K (small batch) path
  int split_bn128 = 1;    // 128-column tiles on the split-K path (halves the partial-tile traffic of the reduction)
  int conv1_1_umma = 1;   // model1.0 on the tensor cores (one padded k-block); 0 = the FP32 CUDA-core kernel
  int side_dist = 1;      // batch <= 4: run the dist head (class + softmax) on a side stream next to levels 9-10
  int tanh_scale = 110;   // regression head: tanh * 110 (model.py:175); the Caffe deploy nets use 100 (SURVEY q4)
};

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> dims;
};

struct Ctx {
  int dev = 0;
  int max_n = 0, H = 0, W = 0;
  unsigned flags = 0;
  Options opt;
  bool simt = false, fast = false, dist = false, glob = false;
  std::map<std::string, HostTensor> raw;
  std::vector<ActBuf> bufs;
  std::map<std::string, int> buf_index;
  std::vector<ConvOp> ops;
  // weight arena
  char* arena = nullptr;
  size_t arena_bytes = 0;
  bool weights_ready = false;
  // conv1_1 (4->64) + regression head + misc small weights (device fp32)
  float* w11 = nullptr;   // [36][64]  k = tap*4 + cin
  float* b11 = nullptr;   // [64]
  Conv11Weights h_w11;    // host copy passed by value to conv1_1_kernel
  uint8_t* w11_umma = nullptr;   // conv1_1_umma_kernel: swizzled hi/lo weight tile + bias' / scale' (device, derived)
  float* wout = nullptr;  // [2][128]
  float* bout = nullptr;  // [2]
  // global hints MLP (device fp32)
  float* gw[4] = {nullptr, nullptr, nullptr, nullptr};      // [cout][cin]
  float* gb[4] = {nullptr, nullptr, nullptr, nullptr};
  float* gscale[4] = {nullptr, nullptr, nullptr, nullptr};
  float* gshift[4] = {nullptr, nullptr, nullptr, nullptr};
  float* gvec = nullptr;   // [max_n][512]
  float* gtmp = nullptr;   // [2][max_n][512]
  // workspace
  float* logits = nullptr;     // [max_n*(H/4)*(W/4)][cout_pad(529)]
  float* logits313 = nullptr;  // Caffe-spec head: [max_n*(H/4)*(W/4)][320]
  bool caffe313 = false;
  float* pts313 = nullptr;     // [313][2] ab bin centres (device)
  // split-K workspace of the tcgen05 engine (sized by umma_plan_op, allocated after planning)
  float* splitk_ws = nullptr; size_t splitk_ws_floats = 0;
  int* splitk_counters = nullptr; int splitk_max_tiles = 0;
  long long* dbgbuf = nullptr;   // experiments: per-CTA cycle counters of the last tcgen05 launch
  bool dbg_graph_timing = false; // experiments: events around the click graph launch (idc_debug_graph_timing)
  cudaEvent_t dbg_ev[2] = {nullptr, nullptr};
  float dbg_graph_ms = 0.f;
  int* d_err = nullptr;        // watchdog flag (mapped pinned host memory: survives a device trap)
  int* h_err = nullptr;
  // staging for idc_forward_host
  float* h_in = nullptr;  float* d_in = nullptr;   size_t in_floats = 0;
  float* h_out = nullptr; float* d_out = nullptr;  size_t out_floats = 0;
  uint8_t* h_rgb = nullptr; uint8_t* d_rgb = nullptr;
  char* h_small = nullptr; char* d_small = nullptr;   // compact [ab | rgb | quantised ab] block of the batch <= 4 graph path
  double* h_abq = nullptr; double* d_abq = nullptr;   // quantised ab (row a11) of the large-batch path
  cudaStream_t own_stream = nullptr;
  // idc_forward_host pipeline (large batches): H2D of image chunk k+1 overlaps conv1_1 of chunk k, D2H of ab
  // chunk k overlaps the last op of chunk k+1
  cudaStream_t s_in = nullptr, s_out = nullptr;
  // dist head off the critical path: class + softmax run on a side stream next to decoder levels 9-10
  cudaStream_t s_side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaStream_t s_click = nullptr;            // announced click: pmf + suggestions next to the full-map softmax
  cudaEvent_t ev_click[2] = {nullptr, nullptr};
  int image_n = 0;                           // idc_set_image: this many L planes are resident at the head of d_in
  cudaEvent_t ev_in[8] = {}, ev_out[8] = {};
  // CUDA graph cache for the batch-1 latency path
  cudaGraphExec_t graph_exec = nullptr;
  const void* graph_ptrs[8] = {nullptr};
  float graph_maskcent = 0.f;
  int launch_count = 0;
  int graph_launches = 0;
  bool chain = false;           // the previous operation on the forward's stream was a kernel of this forward (PDL)
  bool gadd_active = false;     // a global-hints vector was supplied to this forward
  int last_n = 0;
  double* d_reccs = nullptr;    // idc_ab_reccs scratch (results of every restart, then the 529x2 gamut points)
  bool dist_resident = false;   // keep the dist of the last forward_host on the device (idc_fetch_dist)
  int dist_valid_n = 0;
  // idc_set_click: the clicked pixel's pmf + K colour suggestions ride on a side branch of the click graph
  bool click_mode = false;
  int* h_click = nullptr; int* d_click = nullptr;   // {img, y4, x4, K, seq} in mapped host memory, read when the graph runs
  char* d_clickout = nullptr; char* h_clickout = nullptr;   // [8-int header | 544 floats pmf | n_init x (3K+2) doubles]
  bool click_served = false;    // h_clickout holds the answer for the click in its header
  // per-op profiling
  bool profiling = false;
  std::vector<std::vector<cudaEvent_t>> prof_runs;   // one event list per profiled forward
  std::vector<cudaEvent_t> prof_pool;
  std::string err;
};

// ---- engine entry points (idc_simt.cu / idc_umma.cu / idc_heads.cu) ----
cudaError_t simt_run_op(Ctx* c, ConvOp& op, int n, cudaStream_t st);
int umma_plan_op(Ctx* c, ConvOp& op);              // builds tensor maps; returns IDC_* code
void umma_free_op(ConvOp& op);
cudaError_t umma_run_op(Ctx* c, ConvOp& op, int n, float* out_ab_fused, float out_mult, cudaStream_t st, int img0 = 0,
                        int max_ctas = 0);   // max_ctas > 0: cap the persistent grid (side-branch launches)
bool umma_op_uses_split_k(const ConvOp& op);

cudaError_t launch_conv1_1(Ctx* c, int n, const float* L, const float* ab, const float* mask,
                           float maskcent, cudaStream_t st, int img0 = 0);   // L/ab/mask: full arrays; images img0..img0+n
cudaError_t launch_conv1_1_umma(Ctx* c, int n, const float* L, const float* ab, const float* mask, float maskcent,
                                cudaStream_t st, int img0 = 0);              // the same layer on the tensor cores
cudaError_t conv1_1_umma_pack(Ctx* c);                                       // weight tile for it, from the arena (device)
cudaError_t launch_out_head(Ctx* c, int n, float* out_ab, cudaStream_t st);   // SIMT / KEEP_CONV10 path
cudaError_t launch_softmax529(Ctx* c, int n, float* out_dist, cudaStream_t st);
cudaError_t launch_lab2rgb(Ctx* c, int n, int h, int w, const float* L, float l_offset, const float* ab,
                           uint8_t* rgb, cudaStream_t st, double* abq = nullptr);   // c may be null (stand-alone call)
cudaError_t launch_decode313(Ctx* c, int n, float T, float* out_ab, cudaStream_t st);
cudaError_t launch_dist313_pixel(Ctx* c, int img, int y, int x, float S, float* out313_dev, cudaStream_t st);
cudaError_t launch_ab_reccs(const float* pmf, size_t bin_stride, const float* pts_dev, int K, int max_iter,
                            int n_init, double* out_dev, cudaStream_t st, const int* dyn = nullptr);
cudaError_t launch_click_pmf(Ctx* c, const int* click_dev, int n_img, int* out_hdr, float* out_pmf, cudaStream_t st);
cudaError_t launch_global_stats(int h, int w, const uint8_t* rgb, const float* pts, float* out316, cudaStream_t st);
cudaError_t launch_rgb2lab(int n, int h, int w, const uint8_t* rgb, double* lab, cudaStream_t st);
cudaError_t launch_zoom_lab2rgb(const double* ab, int hin, int win, const double* Lfull, int H, int W, uint8_t* rgb,
                                cudaStream_t st);
cudaError_t launch_resize_linear_u8(const uint8_t* src, int hs, int ws, uint8_t* dst, int hd, int wd, cudaStream_t st);
cudaError_t launch_cubic_lab2rgb(const double* ab, int hin, int win, const double* L, int H, int W, uint8_t* rgb,
                                 cudaStream_t st);
cudaError_t launch_global_mlp(Ctx* c, int n, const float* glob, cudaStream_t st);
cudaError_t launch_act_to_nchw(Ctx* c, const ActBuf& b, int n, float* out, cudaStream_t st);
cudaError_t launch_nchw_to_act(Ctx* c, const ActBuf& b, int n, const float* in, cudaStream_t st);

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Programmatic dependent launch bookkeeping: a kernel may carry the programmatic-stream-serialization attribute
// only when the operation enqueued right before it on the same stream is another kernel of this forward (every
// kernel of the library executes griddepcontrol.wait, so completion stays transitive along the chain).
inline bool pdl_take(Ctx* c) {
  const bool r = c && c->opt.pdl && !c->simt && c->chain;
  if (c) c->chain = true;
  return r;
}
inline void pdl_break(Ctx* c) { if (c) c->chain = false; }

#ifdef __CUDACC__
__device__ __forceinline__ void pdl_prologue_done() {   // small kernels: let the successor start, then wait for the predecessor
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(Ctx* c, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                            Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_take(c) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#endif

}  // namespace idc
