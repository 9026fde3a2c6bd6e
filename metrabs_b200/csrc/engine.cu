// libmetrabs_b200.so - engine: handle, weight arena (BN folding + repack), op plan, forward executor, C ABI.
// See include/metrabs_b200.h for the contract and the reference file:line each entry point replaces.
#include "../../include/metrabs_b200.h"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "conv_simt.cuh"
#include "decode.cuh"
#include "tc_gemm.cuh"
#include "tc_fmb.cuh"
#include "tc_expdw.cuh"
#include "tc_tf32.cuh"
#include "dw_tma.cuh"
#include "multiperson.cuh"

using namespace mtb;

namespace {

std::string g_error;

enum OpType { OP_STEM = 0, OP_CONV = 1, OP_DW = 2, OP_POOL = 3, OP_MAXPOOL = 4 };
// kernel classes for the CUDA-event profiler (mtb_profile_begin / mtb_profile_end)
enum KClass { KC_STEM = 0, KC_IGEMM_SIMT = 1, KC_DWCONV = 2, KC_POOL = 3, KC_SE_FC = 4, KC_TC_GEMM = 5, KC_FMB = 6,
              KC_HEAD_FUSED = 7, KC_HEAD_CONV_SIMT = 8, KC_SOFTARGMAX = 9, KC_RECON = 10, KC_OTHER = 11, KC_SE_SCALE = 12, KC_TC32 = 13,
              KC_EXPDW = 14, KC_COUNT = 15 };
const char* kKClassNames[KC_COUNT] = {"stem_conv_kernel", "conv_igemm_kernel", "dwconv_kernel", "pool_mean_kernel",
                                      "se_fc(conv_igemm_kernel)", "tc_conv_kernel", "fmb_kernel",
                                      "tc_head_softargmax_kernel", "head_conv(conv_igemm_kernel)",
                                      "softargmax_bhwn_kernel", "recon_pass1+2_kernel", "other", "se_scale_kernel", "tc32_conv_kernel",
                                      "expdw_kernel"};
enum { BUF_FEATURES = -2, BUF_NONE = -1, BUF_SMALL0 = 4 };  // 0..3 big activation buffers, 4..6 small [B,C]
constexpr int kNumBig = 4, kNumSmall = 3;
constexpr int kPoolSlices = 8;  // the fused depthwise+pool kernel leaves up to 8 partial slices [slice][B][C]

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

struct Op {
  OpType type;
  std::string name;     // reference key prefix of the layer
  std::string wkey;     // conv weight key
  std::string bnkey;    // BN key prefix ("" = none)
  std::string biaskey;  // conv bias key ("" = none)
  int in_buf = 0, out_buf = 0, res_buf = BUF_NONE, scale_buf = BUF_NONE;
  int Hin = 1, Win = 1, Cin = 0, Hout = 1, Wout = 1, Cout = 0;
  int R = 1, S = 1, stride = 1, dil = 1, pad_t = 0, pad_l = 0, act = ACT_NONE;
  bool depthwise = false;
  bool small_io = false;  // squeeze-excitation FCs on [B,1,1,C] fp32 tensors
  float pre_scale[3] = {2.f, 2.f, 2.f}, pre_shift[3] = {-1.f, -1.f, -1.f};  // stem input affine (PreprocLayer: x*2-1)
  bool fused_pool = false;  // bf16 modes: this depthwise op also produces the SE pooled means (next op is skipped)
  bool res_first = false;  // residual added BEFORE the activation (ResNet); EfficientNet adds it after
  int pool_src = -1;       // fc1: index of the OP_POOL op that produces its input (fused pooling leaves partial slices)
  int ksplit = 1;          // split-K (squeeze-excitation fc1): raw sums, bias/act deferred to the consumer
  int a_bias_from = -1;    // op index whose bias (+ a_act) is applied to THIS op's input on load
  int a_act = ACT_NONE;
  bool pad_ok = false;    // weight tensor may be smaller than [Cout,Cin]: channels zero-padded to a multiple of 4
  float bn_eps = 1e-3f;
  float* d_w = nullptr;     // fp32 [R*S*Cin][Cout]  (dw: [R*S][C])
  float* d_bias = nullptr;  // fp32 [Cout]
  TcWeights tc;             // bf16 K-major copy + TMA descriptor state for the tcgen05 path
  Tc32Weights tc32;         // fp32 K-major copy + TMA descriptor state for the 3xTF32 tcgen05 path (MTB_PRECISION_TF32X3)
  FmbWeights fmb;           // bf16 mode: this 3x3 expand conv and the NEXT op (1x1 projection) run as one fmb_kernel launch
  ExpdwWeights expdw;       // bf16 mode: this 1x1 expand conv and the NEXT op (depthwise 3x3 + SE squeeze) run as one expdw_kernel launch
  mutable DwTmaCache dw_cache;  // input tensor map of the TMA-staged depthwise kernel
  double flops = 0;         // 2*MACs per crop
  int stage = 0;            // EfficientNet stage (1-based; 0 = stem / last conv / other backbones)
};

}  // namespace

struct mtb_handle {
  mtb_config cfg;
  std::map<std::string, HostTensor> raw;
  std::vector<Op> ops;
  Op head;
  bool finalized = false;
  mutable std::string err;
  std::vector<void*> dev_allocs;
  // geometry
  int feat_side = 0, feat_c = 0;
  size_t big_elems_per_crop = 0;   // capacity of one big buffer, elements per crop
  int small_c = 0;                 // capacity of one small buffer, floats per crop
  int64_t launches = 0;
  double flops_per_crop = 0;
  // host-path staging
  void* stage = nullptr;
  size_t stage_bytes = 0, stage_ws_bytes = 0;
  int stage_batch = 0;
  // pipelined host path (mtb_forward_host_submit / _wait): two input/output slots, one shared workspace, a copy stream
  struct HostSlot {
    void* buf = nullptr;       // [crops | intrinsics | joints] device staging of this slot
    size_t bytes = 0;
    cudaEvent_t h2d_done = nullptr, done = nullptr;
    bool used = false;         // `done` has been recorded at least once
  };
  HostSlot slots[2];
  // MTB_GRAPH=1: captured forwards keyed by (buffers, batch, stream)
  struct GraphEntry {
    const void *crops = nullptr, *k = nullptr, *out = nullptr, *ws = nullptr;
    int batch = 0;
    cudaStream_t st = nullptr;
    cudaGraphExec_t exec = nullptr;
    int64_t launches = 0;
    bool failed = false;
  };
  std::vector<GraphEntry> graphs;
  void* pipe_ws = nullptr;
  size_t pipe_ws_bytes = 0;
  cudaStream_t copy_stream = nullptr;
  cudaStream_t graph_stream = nullptr;  // MTB_GRAPH=1 with the legacy default stream: captured forwards run here
  cudaEvent_t graph_in = nullptr, graph_out = nullptr;
  // profiler
  unsigned prof_mask = 0;
  std::vector<cudaEvent_t> prof_events;  // pairs
  std::vector<int> prof_cls;
  std::vector<int> prof_op;      // backbone op index of each timed launch (-1: head / decode / reconstruction)
  int prof_cur_op = -1;
  std::vector<double> prof_flops, prof_bytes;
  size_t prof_used = 0;
  std::vector<double> prof_op_ms;
  // NCCL (dlopen'ed)
  void* nccl_lib = nullptr;
  void* nccl_comm = nullptr;
  int nccl_world = 0;
};

namespace {

int fail(const mtb_handle* h, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  g_error = buf;
  return code;
}

#define CUDA_TRY(h, expr)                                                                               \
  do {                                                                                                  \
    cudaError_t e__ = (expr);                                                                           \
    if (e__ != cudaSuccess)                                                                             \
      return fail(h, MTB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
inline bool is_bf16(const mtb_handle* h) { return h->cfg.precision == MTB_PRECISION_BF16_TC || h->cfg.precision == MTB_PRECISION_BF16_SIMT; }
inline size_t elem_size(const mtb_handle* h) { return is_bf16(h) ? 2 : 4; }

// ------------------------------------------------------------------------------------------- plan building
struct Planner {
  mtb_handle* h;
  int H, W, C;       // current activation
  int cur = BUF_NONE;
  size_t max_elems = 0;
  int max_small = 0;

  int pick(std::initializer_list<int> busy) {
    for (int i = 0; i < kNumBig; ++i)
      if (std::find(busy.begin(), busy.end(), i) == busy.end()) return i;
    return 0;
  }
  void track(int h_, int w_, int c_) { max_elems = std::max(max_elems, (size_t)h_ * w_ * c_); }

  // Keras-named conv (TF-only backbones): explicit weight / bias / BN keys
  Op& conv_k(const std::string& name, const std::string& wkey, const std::string& biaskey, const std::string& bnkey, int cout,
             int k, int stride, int pad_beg, int pad_total, int act, int in_buf, int out_buf, bool depthwise = false,
             int dil = 1, float eps = 1e-3f) {
    Op& op = conv(name, cout, k, stride, pad_beg, pad_total, act, in_buf, out_buf, depthwise, dil);
    op.wkey = wkey; op.biaskey = biaskey; op.bnkey = bnkey; op.bn_eps = eps;
    return op;
  }

  // squeeze-excitation on the tensor in `buf` (H x W x C): pool + fc1 + fc2 -> scale in BUF_SMALL0+2
  void squeeze_excite(const std::string& name, const std::string& fc1, const std::string& fc2, int csq_real, int buf,
                      int act1, int act2) {
    const int cexp = C;
    const int csq = (csq_real + 3) / 4 * 4;  // hidden channels zero-padded to a multiple of 4 (128-bit accesses)
    Op op;
    op.type = OP_POOL; op.name = name + ".avgpool";
    op.Hin = H; op.Win = W; op.Cin = op.Cout = cexp;
    op.in_buf = buf; op.out_buf = BUF_SMALL0;
    h->ops.push_back(op);
    const int pool_index = (int)h->ops.size() - 1;
    Op f1;
    f1.type = OP_CONV; f1.name = name + ".fc1"; f1.wkey = fc1 + ".weight"; f1.biaskey = fc1 + ".bias";
    f1.Cin = cexp; f1.Cout = csq; f1.act = act1; f1.small_io = true; f1.pad_ok = true;
    f1.in_buf = BUF_SMALL0; f1.out_buf = BUF_SMALL0 + 1;
    f1.pool_src = pool_index;
    f1.flops = 2.0 * cexp * csq_real;
    // K = cexp is long and M = batch is short: split K over CTAs; the ksplit partial slices [ksplit][B][csq] must fit
    // the small buffer (capacity >= cexp floats per crop)
    f1.ksplit = std::max(1, std::min({32, cexp / 64, cexp / csq}));
    h->ops.push_back(f1);
    const int f1_index = (int)h->ops.size() - 1;
    Op f2;
    f2.type = OP_CONV; f2.name = name + ".fc2"; f2.wkey = fc2 + ".weight"; f2.biaskey = fc2 + ".bias";
    f2.Cin = csq; f2.Cout = cexp; f2.act = act2; f2.small_io = true; f2.pad_ok = true;
    f2.in_buf = BUF_SMALL0 + 1; f2.out_buf = BUF_SMALL0 + 2;
    f2.flops = 2.0 * cexp * csq_real;
    (void)f1_index;  // (fc2 summing the slices on its A load was measured slower than the tiny reduce kernel)
    h->ops.push_back(f2);
    max_small = std::max(max_small, cexp);
  }

  // conv with explicit begin pad; output size = floor((in + pad_total - eff_k)/stride) + 1
  Op& conv(const std::string& name, int cout, int k, int stride, int pad_beg, int pad_total, int act, int in_buf,
           int out_buf, bool depthwise = false, int dil = 1) {
    Op op;
    op.type = depthwise ? OP_DW : OP_CONV;
    op.name = name;
    op.wkey = name + ".0.weight";
    op.bnkey = name + ".1";
    op.Hin = H; op.Win = W; op.Cin = C; op.Cout = cout;
    op.R = op.S = k; op.stride = stride; op.dil = dil; op.pad_t = op.pad_l = pad_beg; op.act = act;
    int eff = k + (k - 1) * (dil - 1);
    op.Hout = (H + pad_total - eff) / stride + 1;
    op.Wout = (W + pad_total - eff) / stride + 1;
    op.depthwise = depthwise;
    op.in_buf = in_buf; op.out_buf = out_buf;
    op.flops = 2.0 * op.Hout * op.Wout * cout * k * k * (depthwise ? 1 : C);
    H = op.Hout; W = op.Wout; C = cout;
    track(H, W, C);
    h->ops.push_back(op);
    return h->ops.back();
  }
};

void plan_effnet(mtb_handle* h) {
  // EfficientNet.features (backbones/efficientnet.py:286-324) with PreprocLayer (:1181-1186) folded in the stem
  const mtb_config& c = h->cfg;
  Planner P{h, c.proc_side, c.proc_side, 3};
  const std::string pre = "backbone.1";
  {
    Op op;
    op.type = OP_STEM;
    op.name = pre + ".0";
    op.wkey = op.name + ".0.weight";
    op.bnkey = op.name + ".1";
    op.Hin = op.Win = c.proc_side; op.Cin = 3; op.Cout = c.stages[0].cin;
    op.R = op.S = 3; op.stride = 2; op.pad_t = op.pad_l = 1; op.act = ACT_SILU;
    op.Hout = op.Wout = (c.proc_side + 2 - 3) / 2 + 1;
    op.in_buf = BUF_NONE; op.out_buf = 0;
    op.flops = 2.0 * op.Hout * op.Wout * op.Cout * 27;
    P.H = op.Hout; P.W = op.Wout; P.C = op.Cout; P.cur = 0;
    P.track(P.H, P.W, P.C);
    h->ops.push_back(op);
  }
  for (int si = 0; si < c.n_stages; ++si) {
    const mtb_stage& st = c.stages[si];
    const size_t stage_first_op = h->ops.size();
    for (int bi = 0; bi < st.layers; ++bi) {
      const bool first = bi == 0;
      const int cin = first ? st.cin : st.cout;
      const int stride = first ? st.stride : 1;
      const int shift = (first && st.bottomright) ? 1 : 0;
      const bool residual = stride == 1 && cin == st.cout;
      const int cexp = cin * st.expand;
      const int k = st.kernel;
      const int pad_beg = (k - 1) / 2 - shift, pad_total = k - 1;  // fixed_padding_layer (:1127-1161)
      char key[64];
      snprintf(key, sizeof(key), "%s.%d.%d.block", pre.c_str(), si + 1, bi);
      const std::string kb = key;
      const int x_in = P.cur;
      if (st.block == 0) {  // FusedMBConv (:176-234)
        if (st.expand != 1) {
          int t1 = P.pick({x_in});
          P.conv(kb + ".0", cexp, k, stride, pad_beg, pad_total, ACT_SILU, x_in, t1);
          int t2 = P.pick({x_in, t1});
          Op& pr = P.conv(kb + ".1", st.cout, 1, 1, 0, 0, ACT_NONE, t1, t2);
          if (residual) pr.res_buf = x_in;
          P.cur = t2;
        } else {
          int t1 = P.pick({x_in});
          Op& cv = P.conv(kb + ".0", st.cout, k, stride, pad_beg, pad_total, ACT_SILU, x_in, t1);
          if (residual) cv.res_buf = x_in;
          P.cur = t1;
        }
      } else {  // MBConv (:110-173)
        int i = 0;
        int t1 = x_in;
        if (st.expand != 1) {
          t1 = P.pick({x_in});
          P.conv(kb + "." + std::to_string(i), cexp, 1, 1, 0, 0, ACT_SILU, x_in, t1);
          ++i;
        }
        int t2 = P.pick({x_in, t1});
        P.conv(kb + "." + std::to_string(i), cexp, k, stride, pad_beg, pad_total, ACT_SILU, t1, t2, true);
        ++i;
        // squeeze-excitation: avgpool -> fc1 + SiLU -> fc2 + sigmoid -> scale (folded into the projection's A load)
        const std::string se = kb + "." + std::to_string(i);
        P.squeeze_excite(se, se + ".fc1", se + ".fc2", std::max(1, cin / 4), t2, ACT_SILU, ACT_SIGMOID);
        ++i;
        int t3 = P.pick({x_in, t2});
        Op& pr = P.conv(kb + "." + std::to_string(i), st.cout, 1, 1, 0, 0, ACT_NONE, t2, t3);
        pr.scale_buf = BUF_SMALL0 + 2;
        if (residual) pr.res_buf = x_in;
        P.cur = t3;
      }
    }
    for (size_t k = stage_first_op; k < h->ops.size(); ++k) h->ops[k].stage = si + 1;
  }
  {
    char key[64];
    snprintf(key, sizeof(key), "%s.%d", pre.c_str(), c.n_stages + 1);
    Op& last = P.conv(key, c.last_channel, 1, 1, 0, 0, ACT_SILU, P.cur, BUF_FEATURES);  // :319-324
    (void)last;
  }
  h->feat_side = P.H;
  h->feat_c = P.C;
  h->big_elems_per_crop = P.max_elems;
  h->small_c = std::max(P.max_small, 4);
}

// ResNet-50 V1 at output stride `stride_test` (metrabs_tf/backbones/resnet.py:75-236 stem/pool, :239-319 bottleneck,
// :601-666 stride/dilation plan; BN eps 1e-5 :71; every conv has a bias :270).  Key schema: Keras layer names,
// "backbone.<layer>.{weight,bias}" / "backbone.<layer>.{weight,bias,running_mean,running_var}" in torch layout.
int plan_resnet50(mtb_handle* h) {
  const mtb_config& c = h->cfg;
  if (c.stride_test != 8 && c.stride_test != 16 && c.stride_test != 32)
    return fail(h, MTB_ERR_UNSUPPORTED, "ResNet-50: stride_test must be 8, 16 or 32 (got %d)", c.stride_test);
  // get_strides_and_dilations(stride_test) (:601-618)
  int strides[3] = {2, 2, 2}, dil_in[3] = {1, 1, 1}, dil_out[3] = {1, 1, 1};
  bool brs[3] = {false, false, false};
  int i_last = 0;
  for (int s_ = c.stride_test; s_ > 8; s_ >>= 1) ++i_last;  // log2(stride) - 3
  if (c.centered_stride) brs[i_last] = true;
  for (int i = i_last + 1; i < 3; ++i) {
    strides[i] = 1;
    dil_in[i] = 1 << (i - (i_last + 1));
    dil_out[i] = dil_in[i] * 2;
  }
  Planner P{h, c.proc_side, c.proc_side, 3};
  const std::string pre = "backbone.";
  const float eps = 1e-5f;
  {
    Op op;
    op.type = OP_STEM;
    op.name = pre + "conv1_conv";
    op.wkey = op.name + ".weight"; op.biaskey = op.name + ".bias"; op.bnkey = pre + "conv1_bn"; op.bn_eps = eps;
    op.Hin = op.Win = c.proc_side; op.Cin = 3; op.Cout = 64;
    op.R = op.S = 7; op.stride = 2; op.pad_t = op.pad_l = 3; op.act = ACT_RELU;
    op.Hout = op.Wout = (c.proc_side + 6 - 7) / 2 + 1;
    const float mean[3] = {103.939f, 116.779f, 123.68f};  // caffe_preproc (builder.py:106-108): 255*x - mean, no channel swap
    for (int i = 0; i < 3; ++i) { op.pre_scale[i] = 255.f; op.pre_shift[i] = -mean[i]; }
    op.in_buf = BUF_NONE; op.out_buf = 0;
    op.flops = 2.0 * op.Hout * op.Wout * 64 * 147;
    P.H = op.Hout; P.W = op.Wout; P.C = 64; P.cur = 0;
    P.track(P.H, P.W, P.C);
    h->ops.push_back(op);
    Op mp;  // ZeroPadding2D((1,1)) + MaxPooling2D(3, 2) (:187-193): the zero pad value takes part in the max
    mp.type = OP_MAXPOOL; mp.name = pre + "pool1_pool";
    mp.Hin = P.H; mp.Win = P.W; mp.Cin = mp.Cout = 64; mp.R = mp.S = 3; mp.stride = 2; mp.pad_t = mp.pad_l = 1;
    mp.Hout = (P.H + 2 - 3) / 2 + 1; mp.Wout = (P.W + 2 - 3) / 2 + 1;
    mp.in_buf = 0; mp.out_buf = 1;
    P.H = mp.Hout; P.W = mp.Wout; P.cur = 1;
    h->ops.push_back(mp);
  }
  const int counts[4] = {3, 4, 6, 3}, filters[4] = {64, 128, 256, 512};
  for (int st = 0; st < 4; ++st) {
    for (int bi = 0; bi < counts[st]; ++bi) {
      const bool first = bi == 0;
      // V1: stride on the first 1x1 and on the shortcut of block1; the 3x3 uses dil_out of its stack in EVERY block
      const int stride = (st > 0 && first) ? strides[st - 1] : 1;
      const int shift = (st > 0 && first && brs[st - 1]) ? 1 : 0;
      const int dil = st == 0 ? dil_in[0] : dil_out[st - 1];
      const int f = filters[st];
      char nm[64];
      snprintf(nm, sizeof(nm), "conv%d_block%d", st + 2, bi + 1);
      const std::string b = pre + nm;
      const int x_in = P.cur;
      const int Hin = P.H, Win = P.W, Cin = P.C;
      int sc = x_in;
      if (first) {  // conv shortcut: strided 1x1 sampled at pixels shift::stride (Conv2DDenseSame semantics)
        sc = P.pick({x_in});
        P.conv_k(b + "_0_conv", b + "_0_conv.weight", b + "_0_conv.bias", b + "_0_bn", 4 * f, 1, stride, -shift, 0, ACT_NONE,
                 x_in, sc, false, 1, eps);
        Op& o = h->ops.back();
        o.Hout = Hin / stride; o.Wout = Win / stride;
        o.flops = 2.0 * o.Hout * o.Wout * o.Cout * Cin;
        P.H = Hin; P.W = Win; P.C = Cin;  // the main branch restarts from the block input
      }
      int t1 = P.pick({x_in, sc});
      P.conv_k(b + "_1_conv", b + "_1_conv.weight", b + "_1_conv.bias", b + "_1_bn", f, 1, stride, -shift, 0, ACT_RELU, x_in, t1,
               false, 1, eps);
      {
        Op& o = h->ops.back();
        o.Hout = Hin / stride; o.Wout = Win / stride;
        o.flops = 2.0 * o.Hout * o.Wout * o.Cout * Cin;
        P.H = o.Hout; P.W = o.Wout;
      }
      int t2 = P.pick({x_in, sc, t1});
      P.conv_k(b + "_2_conv", b + "_2_conv.weight", b + "_2_conv.bias", b + "_2_bn", f, 3, 1, dil, 2 * dil, ACT_RELU, t1, t2,
               false, dil, eps);
      int t3 = P.pick({sc, t2});
      const bool last = st == 3 && bi == counts[3] - 1;
      Op& o3 = P.conv_k(b + "_3_conv", b + "_3_conv.weight", b + "_3_conv.bias", b + "_3_bn", 4 * f, 1, 1, 0, 0, ACT_RELU, t2,
                        last ? BUF_FEATURES : t3, false, 1, eps);
      o3.res_buf = sc;
      o3.res_first = true;  // relu(shortcut + x)
      P.cur = t3;
    }
  }
  h->feat_side = P.H;
  h->feat_c = P.C;
  h->big_elems_per_crop = P.max_elems;
  h->small_c = 4;
  return MTB_OK;
}

// MobileNetV3-Small (metrabs_tf/backbones/mobilenet_v3.py:348-384 table, :490-553 block, :465-487 SE, :258-296 stem and
// Conv_1 / Conv_2, :556-575 correct_pad; preprocessing 255*x then Rescaling(1/127.5, -1) = 2x-1, builder.py:116-117).
int plan_mobilenetv3_small(mtb_handle* h) {
  const mtb_config& c = h->cfg;
  Planner P{h, c.proc_side, c.proc_side, 3};
  const std::string pre = "backbone.";
  {
    Op op;
    op.type = OP_STEM;
    op.name = pre + "Conv";
    op.wkey = op.name + ".weight"; op.bnkey = op.name + ".BatchNorm";
    op.Hin = op.Win = c.proc_side; op.Cin = 3; op.Cout = 16;
    op.R = op.S = 3; op.stride = 2; op.act = ACT_HSWISH;
    op.Hout = op.Wout = (c.proc_side + 1) / 2;
    // TF 'same' with stride 2: pad_total = max((out-1)*2 + 3 - in, 0), begin = pad_total / 2  (even input: (0,1))
    const int pad_total = std::max((op.Hout - 1) * 2 + 3 - c.proc_side, 0);
    op.pad_t = op.pad_l = pad_total / 2;
    op.in_buf = BUF_NONE; op.out_buf = 0;
    op.flops = 2.0 * op.Hout * op.Wout * 16 * 27;
    P.H = op.Hout; P.W = op.Wout; P.C = 16; P.cur = 0;
    P.track(P.H, P.W, P.C);
    h->ops.push_back(op);
  }
  struct Row { int exp_ch, filters, k, stride; bool se; int act; bool br; };
  const Row rows[11] = {{16, 16, 3, 2, true, ACT_RELU, false},     {72, 24, 3, 2, false, ACT_RELU, false},
                        {88, 24, 3, 1, false, ACT_RELU, false},    {96, 40, 5, 2, true, ACT_HSWISH, false},
                        {240, 40, 5, 1, true, ACT_HSWISH, false},  {240, 40, 5, 1, true, ACT_HSWISH, false},
                        {120, 48, 5, 1, true, ACT_HSWISH, false},  {144, 48, 5, 1, true, ACT_HSWISH, false},
                        {288, 96, 5, 2, true, ACT_HSWISH, true},   {576, 96, 5, 1, true, ACT_HSWISH, false},
                        {576, 96, 5, 1, true, ACT_HSWISH, false}};
  auto depth8 = [](double v) {  // _depth (:449-456)
    int nv = std::max(8, (int)(v + 4) / 8 * 8);
    if (nv < 0.9 * v) nv += 8;
    return nv;
  };
  for (int bi = 0; bi < 11; ++bi) {
    const Row& r = rows[bi];
    const std::string b = pre + (bi == 0 ? std::string("expanded_conv") : "expanded_conv_" + std::to_string(bi));
    const int x_in = P.cur, cin = P.C;
    int t1 = x_in;
    if (bi != 0) {
      t1 = P.pick({x_in});
      P.conv_k(b + ".expand", b + ".expand.weight", "", b + ".expand.BatchNorm", r.exp_ch, 1, 1, 0, 0, r.act, x_in, t1);
    }
    int t2 = P.pick({x_in, t1});
    const int shift = (r.br && c.centered_stride) ? 1 : 0;
    const int pad_total = r.k - 1, pad_beg = (r.k - 1) / 2 - (r.stride == 2 ? shift : 0);
    P.conv_k(b + ".depthwise", b + ".depthwise.weight", "", b + ".depthwise.BatchNorm", r.exp_ch, r.k, r.stride, pad_beg, pad_total,
             r.act, t1, t2, true);
    if (r.se)
      P.squeeze_excite(b + ".squeeze_excite", b + ".squeeze_excite.Conv", b + ".squeeze_excite.Conv_1", depth8(r.exp_ch * 0.25), t2,
                       ACT_RELU, ACT_HSIGMOID);
    int t3 = P.pick({x_in, t2});
    Op& pr = P.conv_k(b + ".project", b + ".project.weight", "", b + ".project.BatchNorm", r.filters, 1, 1, 0, 0, ACT_NONE, t2, t3);
    if (r.se) pr.scale_buf = BUF_SMALL0 + 2;
    if (r.stride == 1 && cin == r.filters) pr.res_buf = x_in;
    P.cur = t3;
  }
  {
    int t1 = P.pick({P.cur});
    P.conv_k(pre + "Conv_1", pre + "Conv_1.weight", "", pre + "Conv_1.BatchNorm", depth8(P.C * 6), 1, 1, 0, 0, ACT_HSWISH, P.cur, t1);
    P.conv_k(pre + "Conv_2", pre + "Conv_2.weight", pre + "Conv_2.bias", "", 1024, 1, 1, 0, 0, ACT_HSWISH, t1, BUF_FEATURES);
  }
  h->feat_side = P.H;
  h->feat_c = P.C;
  h->big_elems_per_crop = P.max_elems;
  h->small_c = std::max(P.max_small, 4);
  return MTB_OK;
}

int plan(mtb_handle* h) {
  const mtb_config& c = h->cfg;
  h->ops.clear();
  switch (c.arch) {
    case MTB_ARCH_EFFNET: plan_effnet(h); break;
    case MTB_ARCH_RESNET50: { int rc = plan_resnet50(h); if (rc) return rc; break; }
    case MTB_ARCH_MOBILENETV3_SMALL: { int rc = plan_mobilenetv3_small(h); if (rc) return rc; break; }
    case MTB_ARCH_HEAD_ONLY:
      h->feat_side = c.proc_side / c.stride_test;
      h->feat_c = c.feature_channels;
      h->big_elems_per_crop = 0;
      h->small_c = 4;
      break;
    default: return fail(h, MTB_ERR_UNSUPPORTED, "arch %d is not built yet", c.arch);
  }
  h->flops_per_crop = 0;
  for (auto& op : h->ops) h->flops_per_crop += op.flops;
  // head: MetrabsHeads.conv_final, 1x1 conv with bias (models/metrabs.py:73)
  Op& hd = h->head;
  hd = Op();
  hd.type = OP_CONV;
  hd.name = "heatmap_heads.conv_final";
  hd.wkey = hd.name + ".weight";
  hd.biaskey = hd.name + ".bias";
  hd.Hin = hd.Win = hd.Hout = hd.Wout = h->feat_side;
  hd.Cin = h->feat_c;
  hd.Cout = (c.n_joints * (1 + c.depth) + 3) / 4 * 4;  // channels padded to a multiple of 4 with zero weights (J=122: 1098 -> 1100)
  hd.act = ACT_NONE;
  hd.flops = 2.0 * hd.Hout * hd.Wout * hd.Cin * hd.Cout;
  return MTB_OK;
}

// ------------------------------------------------------------------------------------------------ weights
const HostTensor* find(const mtb_handle* h, const std::string& k) {
  auto it = h->raw.find(k);
  return it == h->raw.end() ? nullptr : &it->second;
}

int upload(mtb_handle* h, const void* host, size_t bytes, void** dev) {
  CUDA_TRY(h, cudaMalloc(dev, bytes));
  h->dev_allocs.push_back(*dev);
  CUDA_TRY(h, cudaMemcpy(*dev, host, bytes, cudaMemcpyHostToDevice));
  return MTB_OK;
}

int prepare_op_weights(mtb_handle* h, Op& op) {
  if (op.type == OP_POOL || op.type == OP_MAXPOOL) return MTB_OK;
  const HostTensor* w = find(h, op.wkey);
  if (!w) return fail(h, MTB_ERR_MISSING_WEIGHT, "missing weight '%s'", op.wkey.c_str());
  const int cin_g = op.depthwise ? 1 : op.Cin;
  const int64_t expect[4] = {op.Cout, cin_g, op.R, op.S};
  bool shape_ok = w->shape.size() == 4 && std::equal(expect, expect + 4, w->shape.begin());
  if (!shape_ok && op.pad_ok && w->shape.size() == 4 && w->shape[2] == op.R && w->shape[3] == op.S &&
      w->shape[0] <= op.Cout && w->shape[0] > op.Cout - 4 && w->shape[1] <= cin_g && w->shape[1] > cin_g - 4)
    shape_ok = true;
  if (!shape_ok)
    return fail(h, MTB_ERR_INVALID_ARG, "weight '%s' has the wrong shape (want [%d,%d,%d,%d])", op.wkey.c_str(),
                op.Cout, cin_g, op.R, op.S);
  const int n_real = (int)w->shape[0], c_real = (int)w->shape[1];
  std::vector<double> scale(op.Cout, 1.0), shift(op.Cout, 0.0);
  if (!op.biaskey.empty()) {
    const HostTensor* b = find(h, op.biaskey);
    if (!b) return fail(h, MTB_ERR_MISSING_WEIGHT, "missing weight '%s'", op.biaskey.c_str());
    if ((int)b->data.size() != n_real) return fail(h, MTB_ERR_INVALID_ARG, "bias '%s' has the wrong size", op.biaskey.c_str());
    for (int n = 0; n < n_real; ++n) shift[n] = b->data[n];
  }
  if (!op.bnkey.empty()) {
    const HostTensor *g = find(h, op.bnkey + ".weight"), *b = find(h, op.bnkey + ".bias"),
                     *m = find(h, op.bnkey + ".running_mean"), *v = find(h, op.bnkey + ".running_var");
    if (!g || !b || !m || !v) return fail(h, MTB_ERR_MISSING_WEIGHT, "missing batch-norm tensors '%s.*'", op.bnkey.c_str());
    for (const HostTensor* t : {g, b, m, v})
      if ((int)t->data.size() != n_real)
        return fail(h, MTB_ERR_INVALID_ARG, "batch-norm tensors '%s.*' must have %d elements (got %zu)", op.bnkey.c_str(), n_real,
                    t->data.size());
    for (int n = 0; n < n_real; ++n) {
      double s = (double)g->data[n] / std::sqrt((double)v->data[n] + (double)op.bn_eps);
      scale[n] = s;
      shift[n] = (shift[n] - (double)m->data[n]) * s + (double)b->data[n];
    }
  }
  const int K = op.R * op.S * cin_g;
  std::vector<float> wk((size_t)K * op.Cout, 0.f), bias(op.Cout, 0.f);
  for (int n = 0; n < n_real; ++n) {
    bias[n] = (float)shift[n];
    for (int c = 0; c < c_real; ++c)
      for (int r = 0; r < op.R; ++r)
        for (int s = 0; s < op.S; ++s) {
          double v = (double)w->data[(((size_t)n * c_real + c) * op.R + r) * op.S + s] * scale[n];
          wk[((size_t)(r * op.S + s) * cin_g + c) * op.Cout + n] = (float)v;
        }
  }
  const bool tc_like = tc_eligible(op.type == OP_CONV, op.depthwise, op.small_io, op.R, op.stride, op.Cin, op.Cout);
  if (is_bf16(h) && tc_like)  // both bf16 modes see the same bf16-rounded GEMM weights
    for (float& v : wk) v = __bfloat162float(host_bf16(v));
  int rc = upload(h, wk.data(), wk.size() * 4, (void**)&op.d_w);
  if (rc) return rc;
  rc = upload(h, bias.data(), bias.size() * 4, (void**)&op.d_bias);
  if (rc) return rc;
  if (h->cfg.precision == MTB_PRECISION_BF16_TC && tc_like && !tc_disabled()) {
    const char* e = tc_prepare_weights(op.tc, wk.data(), bias.data(), K, op.Cout, op.R, op.S, op.Cin, h->dev_allocs);
    if (e) return fail(h, MTB_ERR_CUDA, "tcgen05 weight prep for '%s': %s", op.name.c_str(), e);
  }
  if (h->cfg.precision == MTB_PRECISION_TF32X3 && !tc_disabled() &&
      tc32_eligible(op.type == OP_CONV, op.depthwise, op.small_io, op.R, op.stride, op.Cin, op.Cout)) {
    const char* e = tc32_prepare_weights(op.tc32, wk.data(), bias.data(), K, op.Cout, op.R, op.S, op.Cin, h->dev_allocs);
    if (e) return fail(h, MTB_ERR_CUDA, "3xTF32 weight prep for '%s': %s", op.name.c_str(), e);
  }
  return MTB_OK;
}

// --------------------------------------------------------------------------------------------- workspace
struct Workspace {
  char* base;
  int b0 = 0;  // first crop the ops address (0: every op runs on the whole batch; kept for batch-slice experiments)
  size_t big_stride, small_stride;
  size_t off_small, off_features, off_logits, off_c2d, off_c3d, off_n2d, off_partial, total;
};

Workspace layout(const mtb_handle* h, int B, void* base) {
  Workspace w;
  w.base = (char*)base;
  const size_t es = elem_size(h);
  w.big_stride = align_up(h->big_elems_per_crop * (size_t)B * es, 1024);
  w.small_stride = align_up((size_t)h->small_c * B * 4 * kPoolSlices, 1024);
  size_t o = w.big_stride * kNumBig;
  w.off_small = o; o += w.small_stride * kNumSmall;
  const size_t P = (size_t)h->feat_side * h->feat_side;
  w.off_features = o; o += align_up(P * h->feat_c * B * es, 1024);
  const int N = (h->cfg.n_joints * (1 + h->cfg.depth) + 3) / 4 * 4;
  w.off_logits = o; o += align_up(std::max<size_t>(P, 4) * N * B * 4, 1024);  // also the fused head's state scratch
  w.off_c2d = o; o += align_up((size_t)B * h->cfg.n_joints * 2 * 4, 1024);
  w.off_c3d = o; o += align_up((size_t)B * h->cfg.n_joints * 3 * 4, 1024);
  w.off_n2d = o; o += align_up((size_t)B * h->cfg.n_joints * 2 * 4, 1024);
  w.off_partial = o; o += align_up((size_t)B * 2 * 8, 1024);
  w.total = o;
  return w;
}

void* buf_ptr(const Workspace& w, int id, void* features) {
  if (id == BUF_FEATURES) return features;
  if (id < 0) return nullptr;
  if (id < kNumBig) return w.base + w.big_stride * id;
  return w.base + w.off_small + w.small_stride * (id - BUF_SMALL0);
}

// activation tensor [B,hh,ww,cc] in buffer `id`, from crop w.b0 on (small [B,C] buffers are never sliced)
void* act_ptr(const mtb_handle* h, const Workspace& w, int id, void* features, int hh, int ww, int cc) {
  char* base = (char*)buf_ptr(w, id, features);
  if (!base || id >= kNumBig) return base;
  return base + (size_t)w.b0 * hh * ww * cc * elem_size(h);
}

// ---------------------------------------------------------------------------------------------- profiler
struct ProfScope {
  mtb_handle* h;
  cudaStream_t st;
  bool on;
  // per_op = false keeps the launch out of the per-op table (the in-place SE scale pass is a class of its own; counting it
  // under the projection GEMM's op index made that GEMM look twice as slow as it is)
  ProfScope(mtb_handle* h_, int cls, double flops, double bytes, cudaStream_t st_, bool per_op = true) : h(h_), st(st_) {
    on = (h->prof_mask >> cls) & 1u;
    if (!on) return;
    if (h->prof_used + 2 > h->prof_events.size()) {
      for (int i = 0; i < 2; ++i) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->prof_events.push_back(e);
      }
    }
    h->prof_cls.push_back(cls);
    h->prof_op.push_back(per_op ? h->prof_cur_op : -1);
    h->prof_flops.push_back(flops);
    h->prof_bytes.push_back(bytes);
    cudaEventRecord(h->prof_events[h->prof_used], st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(h->prof_events[h->prof_used + 1], st);
    h->prof_used += 2;
  }
};

// shapes covered by the strip depthwise kernels (dwconv3x3_pool_bf16_kernel / dwconv3x3_pool_f32_kernel)
bool dw_strip_eligible(const Op& op) {
  return op.type == OP_DW && op.R == 3 && op.S == 3 && op.dil == 1 && op.Cout % 8 == 0 && (op.stride == 1 || op.stride == 2) &&
         (op.act == ACT_SILU || op.act == ACT_RELU || op.act == ACT_HSWISH);
}

// number of partial pooling slices the fused depthwise kernel writes (= its gridDim.y)
constexpr int kDwOW = 4;  // outputs per thread along W in dwconv3x3_pool_bf16_kernel (measured: 4 -> 3.65 ms, 2 -> 4.25 ms per 128 crops)
// stride-1 3x3 depthwise ops run the TMA-staged kernel (dw_tma.cuh); MTB_DW_TMA=0 falls back to the strip kernel (A/B runs)
// MTB_DW_F32_TMA=1: the 3xTF32 mode runs the fp32 variant of the TMA-staged depthwise kernel instead of the fp32 strip kernel.
// OFF: measured 11.08 vs 9.92 ms per 256 crops (V2-L; joints 6.9e-6 vs 7.4e-6 from the oracle) - with 32 channels per item and the
// exact expf / divide SiLU of the parity mode the kernel is more issue-bound than the strip kernel is latency-bound.
bool dw_f32_tma_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MTB_DW_F32_TMA");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}
bool dw_tma_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MTB_DW_TMA");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}
// tma_ok: the handle runs a mode the TMA-staged kernel covers (bf16 tensor-core mode; 3xTF32 mode: its fp32 variant, C % 4 == 0)
DwTmaPlan dw_tma_plan_for(const Op& op, bool tma_ok = true) {
  DwTmaPlan none;
  if (!tma_ok) return none;
  if (!dw_tma_enabled() || !dw_strip_eligible(op) || op.stride != 1 || op.Hin != op.Hout || op.Win != op.Wout) return none;
  DwTmaPlan pl = dw_tma_plan(op.Hout, op.Wout);
  if (!pl.ok || pl.n_rb > kPoolSlices) return none;
  return pl;
}
bool dw_tma_mode(const mtb_handle* h, const Op& op) {
  return h->cfg.precision == MTB_PRECISION_BF16_TC || (h->cfg.precision == MTB_PRECISION_TF32X3 && op.Cout % 4 == 0 && dw_f32_tma_enabled());
}
int dw_pool_slices(const Op& dw, bool tma_ok = true) {
  const DwTmaPlan pl = dw_tma_plan_for(dw, tma_ok);
  if (pl.ok) return pl.n_rb;
  const int strips = dw.Hout * ((dw.Wout + kDwOW - 1) / kDwOW);
  return std::min((strips + 7) / 8, kPoolSlices);
}

// (a, d) = 1x1 expand + depthwise pair that expdw_kernel computes exactly as the two launches do (bf16 tensor-core mode;
// the depthwise op runs dw3x3s1_tma_kernel with ONE pooled slice there, the layout the fused kernel writes)
bool expdw_pair_ok(const mtb_handle* h, const Op& a, const Op& d) {
  if (h->cfg.precision != MTB_PRECISION_BF16_TC || !a.tc.ready) return false;
  if (a.type != OP_CONV || a.small_io || a.R != 1 || a.S != 1 || a.stride != 1 || a.act != ACT_SILU) return false;
  if (a.res_buf != BUF_NONE || a.scale_buf != BUF_NONE || a.Hin != a.Hout || a.Win != a.Wout) return false;
  if (d.type != OP_DW || d.act != ACT_SILU || !d.fused_pool || d.in_buf != a.out_buf || d.out_buf == a.in_buf || d.Cout != a.Cout) return false;
  if (d.stride != 1 || d.pad_t != 1 || d.pad_l != 1 || d.Hout != a.Hout || d.Wout != a.Wout) return false;
  const DwTmaPlan dp = dw_tma_plan_for(d);
  return dp.ok && dp.n_rb == 1 && expdw_plan(a.Hout, a.Wout, a.Cin, a.Cout).ok;
}

int op_class(const Op& op) {
  switch (op.type) {
    case OP_STEM: return KC_STEM;
    case OP_DW: return KC_DWCONV;
    case OP_POOL: return KC_POOL;
    case OP_MAXPOOL: return KC_OTHER;
    default: break;
  }
  if (op.small_io) return KC_SE_FC;
  if (op.fmb.ready && fmb_enabled()) return KC_FMB;
  if (op.expdw.ready && expdw_enabled()) return KC_EXPDW;
  if (op.tc.ready) return KC_TC_GEMM;  // one class per kernel: every tensor-core conv/GEMM launch is tc_conv_kernel
  if (op.tc32.ready) return KC_TC32;
  return KC_IGEMM_SIMT;
}

double op_weight_bytes(const Op& op) {
  if (op.type == OP_POOL || op.type == OP_MAXPOOL) return 0.0;
  return (double)op.R * op.S * (op.depthwise ? 1 : op.Cin) * op.Cout * (op.tc.ready ? 2.0 : 4.0);
}

double op_bytes(const mtb_handle* h, const Op& op, int B) {
  const double es = op.small_io ? 4.0 : (double)elem_size(h);
  double in = (double)B * op.Hin * op.Win * op.Cin * (op.type == OP_STEM ? 4.0 : es);
  double out = (double)B * op.Hout * op.Wout * op.Cout * es;
  if (op.type == OP_POOL) out = (double)B * op.Cout * 4.0;
  double res = op.res_buf != BUF_NONE ? out : 0.0;
  double w = (op.type == OP_POOL || op.type == OP_MAXPOOL) ? 0.0 : (double)op.R * op.S * (op.depthwise ? 1 : op.Cin) * op.Cout * (op.tc.ready ? 2.0 : 4.0);
  return in + out + res + w;
}

// ---------------------------------------------------------------------------------------------- executor
bool stem_fast_enabled() {  // MTB_STEM_FAST=0: the generic stem kernel (A/B runs, bit-equality test)
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MTB_STEM_FAST");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

bool pdl_se_enabled() {  // MTB_PDL_SE=1: programmatic dependent launch for the squeeze-excitation chain only
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MTB_PDL_SE");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

template <typename T>
int run_op_t(mtb_handle* h, const Op& op, const float* crops, int B, const Workspace& ws, void* features,
             cudaStream_t st) {
  PdlScope pdl_scope(pdl_se_enabled() && op.small_io);
  if (op.type == OP_CONV && op.tc.ready && op.scale_buf != BUF_NONE && !tc_can_fuse_se(op.R, op.stride, op.Cin, op.act)) {
    // squeeze-excitation scale applied in place ahead of a tensor-core conv that cannot fuse it (1x1 stride-1 projections
    // apply it to the A tiles in shared memory inside tc_conv_kernel)
    void* x = act_ptr(h, ws, op.in_buf, features, op.Hin, op.Win, op.Cin);
    const double bytes = 2.0 * B * op.Hin * op.Win * op.Cin * elem_size(h);
    ProfScope ps(h, KC_SE_SCALE, 0.0, bytes, st, false);
    PdlScope pdl_scale(pdl_se_enabled());
    const char* e = tc_se_scale_launch(x, (const float*)buf_ptr(ws, op.scale_buf, features), B, op.Hin * op.Win, op.Cin, st);
    if (e) return fail(h, MTB_ERR_CUDA, "se scale %s: %s", op.name.c_str(), e);
    h->launches++;
  }
  ProfScope prof(h, op_class(op), op.flops * B, op_bytes(h, op, B), st);
  switch (op.type) {
    case OP_STEM: {
      StemParams p;
      p.in = crops + (size_t)ws.b0 * op.Cin * op.Hin * op.Win;
      p.out = act_ptr(h, ws, op.out_buf, features, op.Hout, op.Wout, op.Cout); p.w = op.d_w; p.bias = op.d_bias;
      for (int i = 0; i < 3; ++i) { p.pre_scale[i] = op.pre_scale[i]; p.pre_shift[i] = op.pre_shift[i]; }
      p.pre_scale[3] = 1.f; p.pre_shift[3] = 0.f;
      p.B = B; p.Hin = op.Hin; p.Win = op.Win; p.Cin = op.Cin; p.Hout = op.Hout; p.Wout = op.Wout; p.Cout = op.Cout;
      p.R = op.R; p.S = op.S; p.stride = op.stride; p.pad_t = op.pad_t; p.pad_l = op.pad_l; p.act = op.act;
      size_t smem = ((size_t)op.R * op.S * op.Cin + 1) * op.Cout * 4;
      const size_t pixels = (size_t)B * op.Hout * op.Wout;
      const bool effnet_stem = op.R == 3 && op.S == 3 && op.Cin == 3 && op.stride == 2 && stem_fast_enabled();
      if (effnet_stem && op.Cout == 32) launch_k(stem3x3s2_kernel<T, 32>, dim3(grid_for(pixels, 128)), dim3(128), (size_t)28 * 32 * 4, st, p);
      else if (effnet_stem && op.Cout == 24) launch_k(stem3x3s2_kernel<T, 24>, dim3(grid_for(pixels, 128)), dim3(128), (size_t)28 * 24 * 4, st, p);
      else if (op.Cout % 32 == 0) launch_k(stem_conv_wide_kernel<T, 32>, dim3(grid_for(pixels * (op.Cout / 32), 128)), dim3(128), smem, st, p);
      else if (op.Cout % 24 == 0) launch_k(stem_conv_wide_kernel<T, 24>, dim3(grid_for(pixels * (op.Cout / 24), 128)), dim3(128), smem, st, p);
      else if (op.Cout % 16 == 0) launch_k(stem_conv_wide_kernel<T, 16>, dim3(grid_for(pixels * (op.Cout / 16), 128)), dim3(128), smem, st, p);
      else launch_k(stem_conv_kernel<T>, dim3(grid_for(pixels * (op.Cout / 4), 256)), dim3(256), smem, st, p);
      h->launches++;
      break;
    }
    case OP_CONV:
    case OP_DW:
    case OP_MAXPOOL: {
      ConvParams p;
      p.in = act_ptr(h, ws, op.in_buf, features, op.Hin, op.Win, op.Cin);
      p.out = act_ptr(h, ws, op.out_buf, features, op.Hout, op.Wout, op.Cout);
      p.res = act_ptr(h, ws, op.res_buf, features, op.Hout, op.Wout, op.Cout);
      p.a_scale = (const float*)buf_ptr(ws, op.scale_buf, features);
      p.w = op.d_w; p.bias = op.d_bias;
      p.B = B; p.Hin = op.Hin; p.Win = op.Win; p.Cin = op.Cin; p.Hout = op.Hout; p.Wout = op.Wout; p.Cout = op.Cout;
      p.R = op.R; p.S = op.S; p.stride = op.stride; p.dil = op.dil; p.pad_t = op.pad_t; p.pad_l = op.pad_l; p.act = op.act;
      p.res_first = op.res_first ? 1 : 0;
      if (op.type == OP_DW) {
        if (h->cfg.precision == MTB_PRECISION_BF16_TC && dw_strip_eligible(op)) {
          float* pooled = op.fused_pool ? (float*)buf_ptr(ws, BUF_SMALL0, features) : nullptr;
          const DwTmaPlan tma_plan = dw_tma_plan_for(op);
          if (tma_plan.ok) {
            const char* e = dw_tma_launch(op.dw_cache, tma_plan, p.in, p.out, op.d_w, op.d_bias, pooled, B, op.Hout, op.Wout, op.Cout,
                                          op.pad_t, op.pad_l, op.act, st);
            if (e) return fail(h, MTB_ERR_CUDA, "depthwise (TMA) launch %s: %s", op.name.c_str(), e);
            h->launches++;
            break;
          }
          dim3 grid((op.Cout / 8 + 31) / 32, dw_pool_slices(op), B), block(32, 8);
          if (op.act == ACT_SILU) {
            if (op.stride == 1) launch_k(dwconv3x3_pool_bf16_kernel<1, ACT_SILU, kDwOW>, dim3(grid), dim3(block), 0, st, p, pooled);
            else launch_k(dwconv3x3_pool_bf16_kernel<2, ACT_SILU, kDwOW>, dim3(grid), dim3(block), 0, st, p, pooled);
          } else if (op.act == ACT_RELU) {
            if (op.stride == 1) launch_k(dwconv3x3_pool_bf16_kernel<1, ACT_RELU, kDwOW>, dim3(grid), dim3(block), 0, st, p, pooled);
            else launch_k(dwconv3x3_pool_bf16_kernel<2, ACT_RELU, kDwOW>, dim3(grid), dim3(block), 0, st, p, pooled);
          } else {
            if (op.stride == 1) launch_k(dwconv3x3_pool_bf16_kernel<1, ACT_HSWISH, kDwOW>, dim3(grid), dim3(block), 0, st, p, pooled);
            else launch_k(dwconv3x3_pool_bf16_kernel<2, ACT_HSWISH, kDwOW>, dim3(grid), dim3(block), 0, st, p, pooled);
          }
        } else if (h->cfg.precision == MTB_PRECISION_TF32X3 && dw_strip_eligible(op) && op.Cout % 4 == 0) {
          float* pooled = op.fused_pool ? (float*)buf_ptr(ws, BUF_SMALL0, features) : nullptr;
          const DwTmaPlan tma_plan = dw_tma_plan_for(op, dw_tma_mode(h, op));
          if (tma_plan.ok) {  // the TMA-staged kernel, fp32 variant (exact activation)
            const char* e = dw_tma_launch(op.dw_cache, tma_plan, p.in, p.out, op.d_w, op.d_bias, pooled, B, op.Hout, op.Wout, op.Cout,
                                          op.pad_t, op.pad_l, op.act, st, true);
            if (e) return fail(h, MTB_ERR_CUDA, "depthwise (TMA, fp32) launch %s: %s", op.name.c_str(), e);
            h->launches++;
            break;
          }
          // fp32 strip kernel: 4 channels x 4 pixels per thread, SE squeeze fused (partial slices summed by fc1)
          dim3 grid((op.Cout / 4 + 31) / 32, dw_pool_slices(op, false), B), block(32, 8);
#define MTB_DWF32(ST, AC) launch_k(dwconv3x3_pool_f32_kernel<ST, AC, kDwOW>, dim3(grid), dim3(block), 0, st, p, pooled)
          if (op.act == ACT_SILU) { if (op.stride == 1) MTB_DWF32(1, ACT_SILU); else MTB_DWF32(2, ACT_SILU); }
          else if (op.act == ACT_RELU) { if (op.stride == 1) MTB_DWF32(1, ACT_RELU); else MTB_DWF32(2, ACT_RELU); }
          else { if (op.stride == 1) MTB_DWF32(1, ACT_HSWISH); else MTB_DWF32(2, ACT_HSWISH); }
#undef MTB_DWF32
        } else {
          size_t total = (size_t)B * op.Hout * op.Wout * (op.Cout / 4);
          launch_k(dwconv_kernel<T>, dim3(grid_for(total, 256)), dim3(256), 0, st, p);
        }
      } else if (op.type == OP_MAXPOOL) {
        size_t total = (size_t)B * op.Hout * op.Wout * (op.Cout / 4);
        launch_k(maxpool_kernel<T>, dim3(grid_for(total, 256)), dim3(256), 0, st, p);
      } else if (op.small_io) {
        if (op.pool_src > 0 && h->ops[op.pool_src].fused_pool) {  // input = partial pooling slices of the depthwise kernel
          p.a_splits = dw_pool_slices(h->ops[op.pool_src - 1], dw_tma_mode(h, h->ops[op.pool_src - 1]));
          p.a_split_stride = (size_t)B * op.Cin;
        }
        float* final_out = (float*)p.out;
        if (op.ksplit > 1) {  // split-K partial slices go to the (still unused) scale buffer, then one tiny reduce kernel
          p.ksplit = op.ksplit;
          p.out = buf_ptr(ws, BUF_SMALL0 + 2, features);
        }
        cudaError_t e = launch_conv_igemm<float, float>(p, st);
        if (e == cudaSuccess && op.ksplit > 1) {
          const int n = B * op.Cout;
          launch_k(se_reduce_kernel, dim3((n + 255) / 256), dim3(256), 0, st, (const float*)p.out, (const float*)op.d_bias, final_out, n,
                   op.Cout, op.ksplit, op.act);
          h->launches++;
          e = cudaGetLastError();
        }
        if (e != cudaSuccess) return fail(h, MTB_ERR_CUDA, "launch %s: %s", op.name.c_str(), cudaGetErrorString(e));
      } else if (op.tc.ready) {
        const char* e = tc_conv_launch(op.tc, p, op.res_first, st);
        if (e) return fail(h, MTB_ERR_CUDA, "tcgen05 launch %s: %s", op.name.c_str(), e);
      } else if (op.tc32.ready) {
        const char* e = tc32_conv_launch(op.tc32, p, op.res_first, st);  // SE scale (p.a_scale) applied by the splitter warps
        if (e) return fail(h, MTB_ERR_CUDA, "3xTF32 launch %s: %s", op.name.c_str(), e);
      } else {
        cudaError_t e = launch_conv_igemm<T, T>(p, st);
        if (e != cudaSuccess) return fail(h, MTB_ERR_CUDA, "launch %s: %s", op.name.c_str(), cudaGetErrorString(e));
      }
      h->launches++;
      break;
    }
    case OP_POOL: {
      dim3 grid((op.Cin + 127) / 128, B), block(32, 8);
      launch_k(pool_mean_kernel<T>, dim3(grid), dim3(block), 0, st, (const T*)act_ptr(h, ws, op.in_buf, features, op.Hin, op.Win, op.Cin),
                                                   (float*)buf_ptr(ws, op.out_buf, features), op.Hin * op.Win, op.Cin);
      h->launches++;
      break;
    }
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(h, MTB_ERR_CUDA, "launch %s: %s", op.name.c_str(), cudaGetErrorString(e));
  return MTB_OK;
}

int run_op(mtb_handle* h, const Op& op, const float* crops, int B, const Workspace& ws, void* features, cudaStream_t st) {
  if (op.type == OP_POOL && op.fused_pool) return MTB_OK;  // produced by the preceding depthwise kernel
  if (is_bf16(h)) return run_op_t<__nv_bfloat16>(h, op, crops, B, ws, features, st);
  return run_op_t<float>(h, op, crops, B, ws, features, st);
}

// Crop chunking (running a stage chunk by chunk so that its intermediates stay in the 126 MB L2) was built and measured
// in round 1: 29.5 ms vs 22.7 ms per 256 crops - these kernels are latency / issue bound at 32-128 crops, not bandwidth
// bound, so smaller launches lose more than L2 residency wins.  The executor therefore runs every op on the whole batch.
// one fmb_kernel launch for the FusedMBConv block (a = 3x3 expand, b = 1x1 projection [+ residual = a's input])
int run_fused_block(mtb_handle* h, const Op& a, const Op& b, int B, const Workspace& ws, void* features, cudaStream_t st) {
  const void* in = act_ptr(h, ws, a.in_buf, features, a.Hin, a.Win, a.Cin);
  void* out = act_ptr(h, ws, b.out_buf, features, b.Hout, b.Wout, b.Cout);
  const double bytes = 2.0 * B * a.Hin * a.Win * (a.Cin + b.Cout) + 2.0 * (9.0 * a.Cin * a.Cout + (double)b.Cin * b.Cout);
  ProfScope prof(h, KC_FMB, (a.flops + b.flops) * B, bytes, st);
  const char* e = fmb_launch(a.fmb, in, out, B, a.Hin, a.Win, a.pad_t, a.pad_l, b.res_buf != BUF_NONE, st);
  if (e) return fail(h, MTB_ERR_CUDA, "fused FusedMBConv launch %s: %s", a.name.c_str(), e);
  h->launches++;
  return MTB_OK;
}

// one expdw_kernel launch for the MBConv front half (a = 1x1 expand + SiLU, d = depthwise 3x3 + SiLU + SE squeeze into the
// pooled buffer that fc1 reads, exactly as d's own launch leaves it)
int run_expdw(mtb_handle* h, const Op& a, const Op& d, int B, const Workspace& ws, void* features, cudaStream_t st) {
  const void* in = act_ptr(h, ws, a.in_buf, features, a.Hin, a.Win, a.Cin);
  void* out = act_ptr(h, ws, d.out_buf, features, d.Hout, d.Wout, d.Cout);
  float* pooled = (float*)buf_ptr(ws, BUF_SMALL0, features);
  // algorithmic bytes: input + depthwise output + expand weights (bf16) + depthwise weights and both biases (fp32) + means
  const double bytes = 2.0 * B * a.Hin * a.Win * (a.Cin + d.Cout) + 2.0 * a.Cin * a.Cout + 4.0 * 11.0 * a.Cout + 4.0 * B * d.Cout;
  ProfScope prof(h, KC_EXPDW, (a.flops + d.flops) * B, bytes, st);
  const char* e = expdw_launch(a.expdw, in, out, pooled, B, st);
  if (e) return fail(h, MTB_ERR_CUDA, "fused expand + depthwise launch %s: %s", a.name.c_str(), e);
  h->launches++;
  return MTB_OK;
}

// ops [first, last): fusable pairs that lie inside the range run fused
int run_ops_range(mtb_handle* h, size_t first, size_t last, const float* crops, int B, const Workspace& ws, void* features,
                  cudaStream_t st) {
  for (size_t k = first; k < last; ++k) {
    h->prof_cur_op = (int)k;
    int rc;
    if (h->ops[k].fmb.ready && fmb_enabled() && k + 1 < last) {
      rc = run_fused_block(h, h->ops[k], h->ops[k + 1], B, ws, features, st);
      ++k;
    } else if (h->ops[k].expdw.ready && expdw_enabled() && k + 1 < last) {
      rc = run_expdw(h, h->ops[k], h->ops[k + 1], B, ws, features, st);
      ++k;  // the depthwise op; its OP_POOL successor is skipped as after the depthwise launch (fused_pool)
    } else {
      rc = run_op(h, h->ops[k], crops, B, ws, features, st);
    }
    if (rc) return rc;
  }
  h->prof_cur_op = -1;
  return MTB_OK;
}

int run_backbone(mtb_handle* h, const float* crops, int B, Workspace& ws, void* features, cudaStream_t st) {
  return run_ops_range(h, 0, h->ops.size(), crops, B, ws, features, st);
}

int check_common(mtb_handle* h, int B, size_t ws_bytes, const void* workspace) {
  if (!h) return fail(nullptr, MTB_ERR_INVALID_ARG, "null handle");
  if (!h->finalized) return fail(h, MTB_ERR_NOT_FINALIZED, "mtb_finalize_weights has not been called");
  if (B <= 0) return fail(h, MTB_ERR_INVALID_ARG, "batch must be positive (got %d)", B);
  if (!workspace || ws_bytes < layout(h, B, nullptr).total)
    return fail(h, MTB_ERR_WORKSPACE, "workspace too small: need %zu bytes for batch %d, got %zu",
                layout(h, B, nullptr).total, B, ws_bytes);
  return MTB_OK;
}

DecodeScale make_scale(const mtb_config& c) {
  // heatmap_to_image / heatmap_to_metric (models/util.py:6-33), inference => stride_test
  DecodeScale s;
  int last = c.proc_side - 1;
  int last_rc = last - (last % c.stride_test);
  float add = 0.f;
  if (c.centered_stride) add += (float)(c.stride_test / 2);
  if (c.legacy_centered_stride_bug) add += (float)(c.stride_test / 2);
  s.img_mul = (float)last_rc;
  s.img_add = add;
  s.met_mul = (float)last_rc * c.box_size_mm / (float)c.proc_side;
  s.met_add = add * c.box_size_mm / (float)c.proc_side;
  s.z_mul = c.box_size_mm;
  s.apply = 1;
  return s;
}

template <typename T>
int launch_softargmax_bhwn(const void* logits, float* out2d, float* out3d, int B, int J, int D, int H, int W,
                           int ld, DecodeScale sc, cudaStream_t st) {
  const int N = J * (1 + D);
  size_t smem = ((size_t)N + 4 * 128) * sizeof(float4);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(softargmax_bhwn_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  launch_k(softargmax_bhwn_kernel<T>, dim3(B), dim3(512), smem, st, (const T*)logits, out2d, out3d, J, D, H, W, ld, sc);
  return (int)cudaGetLastError();
}

int head_decode_impl(mtb_handle* h, const void* features, int B, float* c2d, float* c3d, const Workspace& ws,
                     cudaStream_t st) {
  const mtb_config& c = h->cfg;
  const Op& op = h->head;
  const double P = (double)h->feat_side * h->feat_side;
  const double feat_bytes = (double)B * P * op.Cin * elem_size(h);
  const double out_bytes = (double)B * c.n_joints * 5 * 4;
  if (op.tc.ready) {
    // fused: 1x1-conv GEMM on tcgen05 with the soft-argmax reduction in the epilogue; logits never reach HBM
    ProfScope prof(h, KC_HEAD_FUSED, op.flops * B, feat_bytes + (double)op.Cin * op.Cout * 2 + out_bytes, st);
    const char* e = tc_head_launch(op.tc, features, B, h->feat_side, h->feat_side, c.n_joints, c.depth, make_scale(c),
                                   c2d, c3d, ws.base + ws.off_logits, st);
    if (e) return fail(h, MTB_ERR_CUDA, "fused head: %s", e);
    h->launches += 2;
    return MTB_OK;
  }
  ConvParams p;
  p.in = features; p.out = ws.base + ws.off_logits; p.res = nullptr; p.a_scale = nullptr;
  p.w = op.d_w; p.bias = op.d_bias;
  p.B = B; p.Hin = p.Hout = op.Hin; p.Win = p.Wout = op.Win; p.Cin = op.Cin; p.Cout = op.Cout;
  p.R = p.S = 1; p.stride = 1; p.dil = 1; p.pad_t = p.pad_l = 0; p.act = ACT_NONE;
  const double logit_bytes = (double)B * P * op.Cout * 4;
  cudaError_t e;
  if (op.tc32.ready) {  // 3xTF32 GEMM -> fp32 NHWC logits
    ProfScope prof(h, KC_TC32, op.flops * B, feat_bytes + (double)op.Cin * op.Cout * 4 + logit_bytes, st);
    const char* te = tc32_conv_launch(op.tc32, p, false, st);
    if (te) return fail(h, MTB_ERR_CUDA, "3xTF32 head conv: %s", te);
    e = cudaSuccess;
  } else {
    ProfScope prof(h, KC_HEAD_CONV_SIMT, op.flops * B, feat_bytes + (double)op.Cin * op.Cout * 4 + logit_bytes, st);
    e = is_bf16(h) ? launch_conv_igemm<__nv_bfloat16, float>(p, st)
                                             : launch_conv_igemm<float, float>(p, st);
  }
  if (e != cudaSuccess) return fail(h, MTB_ERR_CUDA, "head conv: %s", cudaGetErrorString(e));
  ProfScope prof(h, KC_SOFTARGMAX, 0.0, logit_bytes + out_bytes, st);
  int rc = launch_softargmax_bhwn<float>(p.out, c2d, c3d, B, c.n_joints, c.depth, op.Hin, op.Win, op.Cout, make_scale(c), st);
  if (rc) return fail(h, MTB_ERR_CUDA, "softargmax: %s", cudaGetErrorString((cudaError_t)rc));
  h->launches += 2;
  return MTB_OK;
}

int recon_impl(mtb_handle* h, const float* c2d, const float* c3d, const float* K, int B, float* out, float* n2d,
               double* partial, cudaStream_t st) {
  const mtb_config& c = h->cfg;
  ReconParams p;
  p.c2d = c2d; p.c3d = c3d; p.K = K; p.out = out; p.partial = partial; p.n2d = n2d;
  p.B = B; p.J = c.n_joints;
  float offset = c.centered_stride ? 0.f : -(float)c.stride_train / 2.f;  // is_within_fov (ptu3d.py:113-121)
  p.fov_lower = (float)c.stride_train * 0.75f + offset;
  p.fov_upper = (float)c.proc_side - (float)c.stride_train * 0.75f + offset;
  p.use_mix = c.mix_3d_inside_fov >= 0.f;
  p.mix = c.mix_3d_inside_fov;
  ProfScope prof(h, KC_RECON, 0.0, (double)B * c.n_joints * 8 * 4 + (double)B * 36, st);
  launch_k(recon_pass1_kernel, dim3(B), dim3(128), 0, st, p);
  launch_k(recon_pass2_kernel, dim3(B), dim3(128), 0, st, p);
  h->launches += 2;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(h, MTB_ERR_CUDA, "reconstruct: %s", cudaGetErrorString(e));
  return MTB_OK;
}

__global__ void to_float_kernel(const __nv_bfloat16* in, float* out, size_t n) {
  pdl_trigger();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __bfloat162float(in[i]);
}

__global__ void from_float_kernel(const float* in, __nv_bfloat16* out, size_t n) {
  pdl_trigger();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16_rn(in[i]);
}

// [b,J,2] + [b,J,3] -> [b,J,5] (what travels in the all-gather) and back
__global__ void pack_decoded_kernel(const float* __restrict__ c2d, const float* __restrict__ c3d, float* __restrict__ packed, int n) {
  pdl_trigger();
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    packed[(size_t)i * 5 + 0] = c2d[(size_t)i * 2 + 0];
    packed[(size_t)i * 5 + 1] = c2d[(size_t)i * 2 + 1];
    packed[(size_t)i * 5 + 2] = c3d[(size_t)i * 3 + 0];
    packed[(size_t)i * 5 + 3] = c3d[(size_t)i * 3 + 1];
    packed[(size_t)i * 5 + 4] = c3d[(size_t)i * 3 + 2];
  }
}
__global__ void unpack_decoded_kernel(const float* __restrict__ packed, float* __restrict__ c2d, float* __restrict__ c3d, int n) {
  pdl_trigger();
  pdl_wait();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    c2d[(size_t)i * 2 + 0] = packed[(size_t)i * 5 + 0];
    c2d[(size_t)i * 2 + 1] = packed[(size_t)i * 5 + 1];
    c3d[(size_t)i * 3 + 0] = packed[(size_t)i * 5 + 2];
    c3d[(size_t)i * 3 + 1] = packed[(size_t)i * 5 + 3];
    c3d[(size_t)i * 3 + 2] = packed[(size_t)i * 5 + 4];
  }
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

}  // namespace

// =================================================================================================== C ABI
extern "C" {

const char* mtb_version(void) { return "metrabs_b200 0.1 (sm_100a)"; }

const char* mtb_last_error(const mtb_handle* h) { return h ? h->err.c_str() : g_error.c_str(); }

int mtb_create(const mtb_config* cfg, mtb_handle** out) {
  if (!cfg || !out) return fail(nullptr, MTB_ERR_INVALID_ARG, "null argument");
  if (cfg->abi_version != MTB_ABI_VERSION)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "ABI version mismatch: header %d, caller %d", MTB_ABI_VERSION, cfg->abi_version);
  if (cfg->weak_perspective)
    return fail(nullptr, MTB_ERR_UNSUPPORTED, "weak_perspective reconstruction is not functional in the reference (ptu.py:30,42)");
  if (cfg->n_joints <= 0 || cfg->depth < 1 || cfg->proc_side <= 0 || cfg->stride_test <= 0 || cfg->stride_train <= 0)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid geometry (n_joints=%d depth=%d proc_side=%d stride=%d)", cfg->n_joints,
                cfg->depth, cfg->proc_side, cfg->stride_test);
  if (cfg->arch == MTB_ARCH_EFFNET && (cfg->n_stages <= 0 || cfg->n_stages > MTB_MAX_STAGES))
    return fail(nullptr, MTB_ERR_INVALID_ARG, "n_stages out of range");
  if (cfg->precision < MTB_PRECISION_FP32 || cfg->precision > MTB_PRECISION_TF32X3)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "unknown precision %d", cfg->precision);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, MTB_ERR_CUDA, "no CUDA device: this library has no CPU fallback");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, MTB_ERR_INVALID_ARG, "device %d out of range", cfg->device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10)
    return fail(nullptr, MTB_ERR_CUDA, "device %d is not sm_100 (compute capability %d.%d)", cfg->device, prop.major, prop.minor);
  mtb_handle* h = new mtb_handle();
  h->cfg = *cfg;
  int rc = plan(h);
  if (rc) {
    g_error = h->err;
    delete h;
    return rc;
  }
  *out = h;
  return MTB_OK;
}

int mtb_destroy(mtb_handle* h) {
  if (!h) return MTB_OK;
  const bool trace = getenv("MTB_TRACE_DESTROY") != nullptr;
  if (trace) fprintf(stderr, "mtb_destroy: handle %p device %d allocs %zu events %zu stage %p\n", (void*)h, h->cfg.device,
                     h->dev_allocs.size(), h->prof_events.size(), h->stage);
  {
    DeviceGuard g(h->cfg.device);
    for (void* p : h->dev_allocs) cudaFree(p);
    if (trace) fprintf(stderr, "mtb_destroy: weights freed\n");
    if (h->stage) {
      cudaError_t e = cudaFree(h->stage);
      if (trace) fprintf(stderr, "mtb_destroy: stage freed (%s)\n", cudaGetErrorString(e));
    }
    for (auto& sl : h->slots) {
      if (sl.buf) cudaFree(sl.buf);
      if (sl.h2d_done) cudaEventDestroy(sl.h2d_done);
      if (sl.done) cudaEventDestroy(sl.done);
    }
    for (auto& e : h->graphs)
      if (e.exec) cudaGraphExecDestroy(e.exec);
    if (h->pipe_ws) cudaFree(h->pipe_ws);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->graph_stream) cudaStreamDestroy(h->graph_stream);
    if (h->graph_in) cudaEventDestroy(h->graph_in);
    if (h->graph_out) cudaEventDestroy(h->graph_out);
    cudaGetLastError();
    for (size_t i = 0; i < h->prof_events.size(); ++i) {
      cudaError_t e = cudaEventDestroy(h->prof_events[i]);
      if (trace && (i < 2 || e != cudaSuccess)) fprintf(stderr, "mtb_destroy: event %zu destroyed (%s)\n", i, cudaGetErrorString(e));
      if (e != cudaSuccess) {  // e.g. cudaErrorContextIsDestroyed during process teardown: the driver owns them now
        cudaGetLastError();
        break;
      }
    }
    if (trace) fprintf(stderr, "mtb_destroy: events destroyed\n");
    if (h->nccl_comm && h->nccl_lib) {
      typedef int (*destroy_t)(void*);
      destroy_t f = (destroy_t)dlsym(h->nccl_lib, "ncclCommDestroy");
      if (f) f(h->nccl_comm);
    }
  }
  delete h;
  if (trace) fprintf(stderr, "mtb_destroy: done\n");
  return MTB_OK;
}

int mtb_load_weight(mtb_handle* h, const char* name, const void* data, int dtype, const int64_t* shape, int ndim) {
  if (!h || !name || !data || (ndim > 0 && !shape)) return fail(h, MTB_ERR_INVALID_ARG, "null argument");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) {
    t.shape.push_back(shape[i]);
    n *= (size_t)shape[i];
  }
  t.data.resize(n);
  switch (dtype) {
    case MTB_DTYPE_F32: memcpy(t.data.data(), data, n * 4); break;
    case MTB_DTYPE_BF16: {
      const uint16_t* s = (const uint16_t*)data;
      for (size_t i = 0; i < n; ++i) {
        uint32_t u = (uint32_t)s[i] << 16;
        memcpy(&t.data[i], &u, 4);
      }
      break;
    }
    case MTB_DTYPE_F16: {
      const __half* s = (const __half*)data;
      for (size_t i = 0; i < n; ++i) t.data[i] = __half2float(s[i]);
      break;
    }
    case MTB_DTYPE_I64: {
      const int64_t* s = (const int64_t*)data;
      for (size_t i = 0; i < n; ++i) t.data[i] = (float)s[i];
      break;
    }
    default: return fail(h, MTB_ERR_INVALID_ARG, "unknown dtype %d for '%s'", dtype, name);
  }
  h->raw[name] = std::move(t);
  h->finalized = false;
  return MTB_OK;
}

int mtb_finalize_weights(mtb_handle* h) {
  if (!h) return fail(nullptr, MTB_ERR_INVALID_ARG, "null handle");
  DeviceGuard g(h->cfg.device);
  for (auto& e : h->graphs)  // captured forwards hold the old weight pointers
    if (e.exec) cudaGraphExecDestroy(e.exec);
  h->graphs.clear();
  for (void* p : h->dev_allocs) cudaFree(p);
  h->dev_allocs.clear();
  for (auto& op : h->ops) op.fused_pool = false;
  for (size_t i = 0; i + 1 < h->ops.size(); ++i) {
    const bool fuse = (h->cfg.precision == MTB_PRECISION_BF16_TC || h->cfg.precision == MTB_PRECISION_TF32X3) &&
                      dw_strip_eligible(h->ops[i]) && h->ops[i + 1].type == OP_POOL;
    if (fuse) h->ops[i].fused_pool = h->ops[i + 1].fused_pool = true;
  }
  for (auto& op : h->ops) {
    int rc = prepare_op_weights(h, op);
    if (rc) return rc;
  }
  // FusedMBConv blocks (3x3 expand + SiLU -> 1x1 projection + residual, stride 1): one fused kernel per block (tc_fmb.cuh)
  for (size_t i = 0; i + 1 < h->ops.size(); ++i) {
    Op& a = h->ops[i];
    const Op& b = h->ops[i + 1];
    a.fmb.ready = false;
    if (h->cfg.precision != MTB_PRECISION_BF16_TC || !a.tc.ready || !b.tc.ready) continue;
    if (a.type != OP_CONV || b.type != OP_CONV || a.small_io || b.small_io) continue;
    if (a.R != 3 || a.S != 3 || a.stride != 1 || a.dil != 1 || a.act != ACT_SILU || a.res_buf != BUF_NONE || a.scale_buf != BUF_NONE) continue;
    if (b.R != 1 || b.stride != 1 || b.act != ACT_NONE || b.scale_buf != BUF_NONE || b.res_first || b.in_buf != a.out_buf) continue;
    if (b.res_buf != BUF_NONE && b.res_buf != a.in_buf) continue;
    if (a.Hin != a.Hout || a.Win != a.Wout || b.out_buf == a.in_buf) continue;
    const char* e = fmb_prepare(a.fmb, a.tc, b.tc, h->dev_allocs);
    if (e) return fail(h, MTB_ERR_CUDA, "fused FusedMBConv weight prep for '%s': %s", a.name.c_str(), e);
  }
  // MBConv front halves (1x1 expand + SiLU -> depthwise 3x3 stride 1 + SiLU + SE squeeze) on 16x16 / 8x8 maps: one fused
  // kernel per block (tc_expdw.cuh); every other shape keeps the two launches
  for (size_t i = 0; i + 1 < h->ops.size(); ++i) {
    Op& a = h->ops[i];
    const Op& d = h->ops[i + 1];
    a.expdw.ready = false;
    if (!expdw_pair_ok(h, a, d)) continue;
    const char* e = expdw_prepare(a.expdw, a.tc, d.d_w, d.d_bias, a.Hout, a.Wout);
    if (e) return fail(h, MTB_ERR_CUDA, "fused expand + depthwise prep for '%s': %s", a.name.c_str(), e);
  }
  {
    Op& hd = h->head;
    const HostTensor* w = find(h, hd.wkey);
    if (!w) return fail(h, MTB_ERR_MISSING_WEIGHT, "missing weight '%s'", hd.wkey.c_str());
    const int n_real = h->cfg.n_joints * (1 + h->cfg.depth);
    if (w->shape.size() != 4 || w->shape[0] != n_real || w->shape[1] != hd.Cin)
      return fail(h, MTB_ERR_INVALID_ARG, "'%s' must be [%d,%d,1,1]", hd.wkey.c_str(), n_real, hd.Cin);
    const HostTensor* hb = find(h, hd.biaskey);
    if (!hb || (int)hb->data.size() != n_real) return fail(h, MTB_ERR_MISSING_WEIGHT, "missing weight '%s'", hd.biaskey.c_str());
    if (n_real != hd.Cout) {  // zero-pad the output channels
      HostTensor wp = *w, bp = *hb;
      wp.data.resize((size_t)hd.Cout * hd.Cin, 0.f);
      wp.shape[0] = hd.Cout;
      bp.data.resize(hd.Cout, 0.f);
      bp.shape[0] = hd.Cout;
      h->raw[hd.wkey] = wp;
      h->raw[hd.biaskey] = bp;
      w = find(h, hd.wkey);
    }
    int rc = prepare_op_weights(h, hd);
    if (rc) return rc;
    if (h->cfg.precision == MTB_PRECISION_BF16_TC) {
      int bnp, cpt, npt;
      if (tc_head_plan(h->feat_side * h->feat_side, &bnp, &cpt, &npt)) {
        // the ORIGINAL (unpadded) [n_real][C] weight: the fused kernel masks rows itself
        std::vector<float> w0((size_t)n_real * hd.Cin), b0(n_real);
        for (int n = 0; n < n_real; ++n) {
          b0[n] = find(h, hd.biaskey)->data[n];
          for (int cc = 0; cc < hd.Cin; ++cc) w0[(size_t)n * hd.Cin + cc] = w->data[(size_t)n * hd.Cin + cc];
        }
        const char* e = tc_prepare_head(hd.tc, w0.data(), b0.data(), hd.Cin, n_real, h->dev_allocs);
        if (e) return fail(h, MTB_ERR_CUDA, "tcgen05 head weight prep: %s", e);
      }
    }
  }
  h->raw.clear();
  h->finalized = true;
  return MTB_OK;
}

size_t mtb_workspace_bytes(const mtb_handle* h, int batch) {
  if (!h || batch <= 0) return 0;
  return layout(h, batch, nullptr).total;
}

int mtb_feature_shape(const mtb_handle* h, int* hw_side, int* channels) {
  if (!h) return fail(nullptr, MTB_ERR_INVALID_ARG, "null handle");
  if (hw_side) *hw_side = h->feat_side;
  if (channels) *channels = h->feat_c;
  return MTB_OK;
}

int mtb_backbone_forward(mtb_handle* h, const float* crops, int batch, void* features, void* workspace,
                         size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch, workspace_bytes, workspace);
  if (rc) return rc;
  if (!crops || !features) return fail(h, MTB_ERR_INVALID_ARG, "null crops/features");
  if (h->ops.empty()) return fail(h, MTB_ERR_UNSUPPORTED, "this handle has no backbone (head-only)");
  DeviceGuard g(h->cfg.device);
  h->launches = 0;
  Workspace ws = layout(h, batch, workspace);
  return run_backbone(h, crops, batch, ws, features, (cudaStream_t)stream);
}

int mtb_head_decode(mtb_handle* h, const void* features, int batch, float* coords2d, float* coords3d_rel,
                    void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch, workspace_bytes, workspace);
  if (rc) return rc;
  if (!features || !coords2d || !coords3d_rel) return fail(h, MTB_ERR_INVALID_ARG, "null argument");
  DeviceGuard g(h->cfg.device);
  h->launches = 0;
  Workspace ws = layout(h, batch, workspace);
  return head_decode_impl(h, features, batch, coords2d, coords3d_rel, ws, (cudaStream_t)stream);
}

int mtb_softargmax(const void* logits, int dtype, int layout_, int batch, int n_joints, int depth, int height,
                   int width, float* out2d, float* out3d, void* stream) {
  if (!logits || batch <= 0 || n_joints <= 0 || depth < 0 || height <= 0 || width <= 0)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid soft-argmax arguments");
  if (dtype != MTB_DTYPE_F32 && dtype != MTB_DTYPE_BF16 && dtype != MTB_DTYPE_F16)
    return fail(nullptr, MTB_ERR_UNSUPPORTED, "soft-argmax dtype must be f32, bf16 or f16");
  if (dtype == MTB_DTYPE_F16 && layout_ != MTB_LAYOUT_BDJHW)
    return fail(nullptr, MTB_ERR_UNSUPPORTED, "f16 logits are supported in the reference layout (BDJHW) only");
  cudaStream_t st = (cudaStream_t)stream;
  if (layout_ == MTB_LAYOUT_BDJHW) {
    const bool two_d = depth == 0;
    float* out = two_d ? out2d : out3d;
    if (!out) return fail(nullptr, MTB_ERR_INVALID_ARG, "null output");
    const int D = two_d ? 1 : depth;
    const int vw = dtype == MTB_DTYPE_F32 ? 4 : 8;  // elements per 16-byte vector
    const bool vec = (width % vw == 0) && (((uintptr_t)logits) % 16 == 0);
    const int rows = batch * n_joints;
    const int hw = height * width;
    const bool pow2 = (hw & (hw - 1)) == 0 && (width & (width - 1)) == 0;
    int hw_shift = 0, w_shift = 0;
    while ((1 << hw_shift) < hw) ++hw_shift;
    while ((1 << w_shift) < width) ++w_shift;
#define MTB_SA_LAUNCH(TT, VV, PP)                                                                                        \
  launch_k(softargmax_bdjhw_kernel<TT, VV, PP>, dim3(rows), dim3(256), 0, st, (const TT*)logits, out, n_joints, D, height, \
           width, (int)two_d, hw_shift, w_shift)
    if (dtype == MTB_DTYPE_F32) {
      if (vec && pow2) MTB_SA_LAUNCH(float, 4, true);
      else if (vec) MTB_SA_LAUNCH(float, 4, false);
      else MTB_SA_LAUNCH(float, 1, false);
    } else if (dtype == MTB_DTYPE_BF16) {
      if (vec && pow2) MTB_SA_LAUNCH(__nv_bfloat16, 8, true);
      else if (vec) MTB_SA_LAUNCH(__nv_bfloat16, 8, false);
      else MTB_SA_LAUNCH(__nv_bfloat16, 1, false);
    } else {  // fp16: what the reference's head emits under its autocast (multiperson_model.py:241, models/metrabs.py:80)
      if (vec && pow2) MTB_SA_LAUNCH(__half, 8, true);
      else if (vec) MTB_SA_LAUNCH(__half, 8, false);
      else MTB_SA_LAUNCH(__half, 1, false);
    }
#undef MTB_SA_LAUNCH
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, MTB_ERR_CUDA, "softargmax launch: %s", cudaGetErrorString(e));
    return MTB_OK;
  }
  if (layout_ == MTB_LAYOUT_BHWN) {
    DecodeScale sc{};
    sc.apply = 0;
    int rc = dtype == MTB_DTYPE_F32
                 ? launch_softargmax_bhwn<float>(logits, out2d, out3d, batch, n_joints, depth, height, width, n_joints * (1 + depth), sc, st)
                 : launch_softargmax_bhwn<__nv_bfloat16>(logits, out2d, out3d, batch, n_joints, depth, height, width, n_joints * (1 + depth), sc, st);
    if (rc) return fail(nullptr, MTB_ERR_CUDA, "softargmax launch: %s", cudaGetErrorString((cudaError_t)rc));
    return MTB_OK;
  }
  return fail(nullptr, MTB_ERR_INVALID_ARG, "unknown layout %d", layout_);
}

size_t mtb_reconstruct_scratch_bytes(int batch) {
  return batch <= 0 ? 0 : align_up((size_t)batch * 2 * 8, 256) + (size_t)batch * 4096 * 2 * 4;
}

int mtb_reconstruct_absolute(mtb_handle* h, const float* coords2d, const float* coords3d_rel, const float* intrinsics,
                             int batch, float* coords3d_abs, void* scratch, void* stream) {
  if (!h) return fail(nullptr, MTB_ERR_INVALID_ARG, "null handle");
  if (!coords2d || !coords3d_rel || !intrinsics || !coords3d_abs || !scratch || batch <= 0)
    return fail(h, MTB_ERR_INVALID_ARG, "null/invalid argument");
  if (h->cfg.n_joints > 4096) return fail(h, MTB_ERR_UNSUPPORTED, "more than 4096 joints");
  DeviceGuard g(h->cfg.device);
  h->launches = 0;
  double* partial = (double*)scratch;
  float* n2d = (float*)((char*)scratch + align_up((size_t)batch * 2 * 8, 256));
  return recon_impl(h, coords2d, coords3d_rel, intrinsics, batch, coords3d_abs, n2d, partial, (cudaStream_t)stream);
}

// the forward proper: every launch of one step on `st` (no allocation, no synchronisation: capturable)
static int forward_body(mtb_handle* h, const float* crops, const float* intrinsics, int batch, float* coords3d_abs, void* workspace,
                        cudaStream_t st) {
  h->launches = 0;
  Workspace ws = layout(h, batch, workspace);
  void* features = ws.base + ws.off_features;
  int rc = run_backbone(h, crops, batch, ws, features, st);
  if (rc) return rc;
  float* c2d = (float*)(ws.base + ws.off_c2d);
  float* c3d = (float*)(ws.base + ws.off_c3d);
  rc = head_decode_impl(h, features, batch, c2d, c3d, ws, st);
  if (rc) return rc;
  return recon_impl(h, c2d, c3d, intrinsics, batch, coords3d_abs, (float*)(ws.base + ws.off_n2d),
                    (double*)(ws.base + ws.off_partial), st);
}

// mtb_forward captures its own launches into a CUDA graph the second time it sees the same (buffers, batch, stream) and
// replays that graph from then on: the ~465 launches of a step cost less as one graph launch than as stream submissions
// (measured, round 2: 12.28 k vs 11.83 k crops/s end to end through mtb_forward_host_submit/_wait, EfficientNetV2-L@256, 256
// crops).  MTB_GRAPH=0 disables it.  A profiling window bypasses it (events cannot be timed inside a graph), a caller that
// is itself capturing the stream just records our launches, any capture failure falls back to plain launches for that key.
static void drop_graphs_on(mtb_handle* h, const void* ws) {
  for (size_t i = 0; i < h->graphs.size();) {
    if (ws == nullptr || h->graphs[i].ws == ws) {
      if (h->graphs[i].exec) cudaGraphExecDestroy(h->graphs[i].exec);
      h->graphs.erase(h->graphs.begin() + (long)i);
    } else {
      ++i;
    }
  }
}

static bool graph_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MTB_GRAPH");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

int mtb_forward(mtb_handle* h, const float* crops, const float* intrinsics, int batch, float* coords3d_abs,
                void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch, workspace_bytes, workspace);
  if (rc) return rc;
  if (!crops || !intrinsics || !coords3d_abs) return fail(h, MTB_ERR_INVALID_ARG, "null argument");
  if (h->ops.empty()) return fail(h, MTB_ERR_UNSUPPORTED, "this handle has no backbone (head-only)");
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  if (graph_enabled() && h->prof_mask == 0) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cs);
    if (cs == cudaStreamCaptureStatusNone) {  // (a caller capturing this stream itself just records our launches)
      // the legacy default stream cannot be captured: fork to an internal stream and join back with events
      const bool side = st == nullptr || st == cudaStreamLegacy || st == cudaStreamPerThread;
      cudaStream_t gs = st;
      if (side) {
        if (!h->graph_stream) {
          CUDA_TRY(h, cudaStreamCreateWithFlags(&h->graph_stream, cudaStreamNonBlocking));
          CUDA_TRY(h, cudaEventCreateWithFlags(&h->graph_in, cudaEventDisableTiming));
          CUDA_TRY(h, cudaEventCreateWithFlags(&h->graph_out, cudaEventDisableTiming));
        }
        gs = h->graph_stream;
      }
      auto launch = [&](cudaGraphExec_t ex) -> cudaError_t {
        cudaError_t e = cudaSuccess;
        if (side) {
          if ((e = cudaEventRecord(h->graph_in, st)) != cudaSuccess) return e;
          if ((e = cudaStreamWaitEvent(gs, h->graph_in, 0)) != cudaSuccess) return e;
        }
        if ((e = cudaGraphLaunch(ex, gs)) != cudaSuccess) return e;
        if (side) {
          if ((e = cudaEventRecord(h->graph_out, gs)) != cudaSuccess) return e;
          if ((e = cudaStreamWaitEvent(st, h->graph_out, 0)) != cudaSuccess) return e;
        }
        return e;
      };
      mtb_handle::GraphEntry* ent = nullptr;
      for (auto& e : h->graphs)
        if (e.crops == crops && e.k == intrinsics && e.out == coords3d_abs && e.ws == workspace && e.batch == batch && e.st == st) ent = &e;
      if (ent && ent->exec) {
        CUDA_TRY(h, launch(ent->exec));
        h->launches = ent->launches;
        return MTB_OK;
      }
      if (ent && !ent->failed) {  // second sighting of this key: capture
        if (side) cudaStreamSynchronize(st);  // (once per key) everything the capture stream must see has completed
        if (cudaStreamBeginCapture(gs, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
          rc = forward_body(h, crops, intrinsics, batch, coords3d_abs, workspace, gs);
          cudaGraph_t gr = nullptr;
          cudaError_t ce = cudaStreamEndCapture(gs, &gr);
          cudaGraphExec_t ex = nullptr;
          if (rc == MTB_OK && ce == cudaSuccess && gr && cudaGraphInstantiate(&ex, gr, 0) == cudaSuccess) {
            cudaGraphDestroy(gr);
            ent->exec = ex;
            ent->launches = h->launches;
            CUDA_TRY(h, launch(ent->exec));
            return MTB_OK;
          }
          if (gr) cudaGraphDestroy(gr);
        }
        cudaGetLastError();  // a refused capture leaves a sticky error behind: clear it before the plain launches
        ent->failed = true;  // plain launches for this key from now on
      } else if (!ent) {
        if (h->graphs.size() >= 8) drop_graphs_on(h, nullptr);  // a caller cycling through many buffers: bounded state
        mtb_handle::GraphEntry e;
        e.crops = crops; e.k = intrinsics; e.out = coords3d_abs; e.ws = workspace; e.batch = batch; e.st = st;
        h->graphs.push_back(e);
      }
    }
  }
  return forward_body(h, crops, intrinsics, batch, coords3d_abs, workspace, st);
}

int mtb_forward_host(mtb_handle* h, const float* host_crops, const float* host_intrinsics, int batch,
                     float* host_coords3d_abs, void* stream) {
  if (!h) return fail(nullptr, MTB_ERR_INVALID_ARG, "null handle");
  if (!h->finalized) return fail(h, MTB_ERR_NOT_FINALIZED, "mtb_finalize_weights has not been called");
  if (!host_crops || !host_intrinsics || !host_coords3d_abs || batch <= 0) return fail(h, MTB_ERR_INVALID_ARG, "null/invalid argument");
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t S = h->cfg.proc_side;
  const size_t crops_b = align_up((size_t)batch * 3 * S * S * 4, 1024), k_b = align_up((size_t)batch * 9 * 4, 1024),
               out_b = align_up((size_t)batch * h->cfg.n_joints * 3 * 4, 1024);
  const size_t ws_b = layout(h, batch, nullptr).total;
  const size_t need = crops_b + k_b + out_b + ws_b;
  if (need > h->stage_bytes) {  // grows only when a larger batch than ever before arrives
    CUDA_TRY(h, cudaStreamSynchronize(st));
    if (h->stage) drop_graphs_on(h, (char*)h->stage + (h->stage_bytes - h->stage_ws_bytes));
    if (h->stage) cudaFree(h->stage);
    h->stage = nullptr;
    h->stage_bytes = 0;
    CUDA_TRY(h, cudaMalloc(&h->stage, need));
    h->stage_bytes = need;
    h->stage_ws_bytes = ws_b;
  }
  char* base = (char*)h->stage;
  float* d_crops = (float*)base;
  float* d_k = (float*)(base + crops_b);
  float* d_out = (float*)(base + crops_b + k_b);
  void* d_ws = base + crops_b + k_b + out_b;
  CUDA_TRY(h, cudaMemcpyAsync(d_crops, host_crops, (size_t)batch * 3 * S * S * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(h, cudaMemcpyAsync(d_k, host_intrinsics, (size_t)batch * 9 * 4, cudaMemcpyHostToDevice, st));
  int rc = mtb_forward(h, d_crops, d_k, batch, d_out, d_ws, ws_b, stream);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(host_coords3d_abs, d_out, (size_t)batch * h->cfg.n_joints * 3 * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaStreamSynchronize(st));
  return MTB_OK;
}

int mtb_forward_host_submit(mtb_handle* h, const float* host_crops, const float* host_intrinsics, int batch,
                            float* host_coords3d_abs, int slot, void* stream) {
  if (!h) return fail(nullptr, MTB_ERR_INVALID_ARG, "null handle");
  if (!h->finalized) return fail(h, MTB_ERR_NOT_FINALIZED, "mtb_finalize_weights has not been called");
  if (!host_crops || !host_intrinsics || !host_coords3d_abs || batch <= 0 || slot < 0 || slot > 1)
    return fail(h, MTB_ERR_INVALID_ARG, "null/invalid argument");
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t S = h->cfg.proc_side;
  const size_t crops_b = align_up((size_t)batch * 3 * S * S * 4, 1024), k_b = align_up((size_t)batch * 9 * 4, 1024),
               out_b = align_up((size_t)batch * h->cfg.n_joints * 3 * 4, 1024);
  const size_t ws_b = layout(h, batch, nullptr).total;
  mtb_handle::HostSlot& sl = h->slots[slot];
  if (!h->copy_stream) CUDA_TRY(h, cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  if (!sl.h2d_done) {
    CUDA_TRY(h, cudaEventCreateWithFlags(&sl.h2d_done, cudaEventDisableTiming));
    CUDA_TRY(h, cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
  }
  if (crops_b + k_b + out_b > sl.bytes || ws_b > h->pipe_ws_bytes) {  // grows only when a larger batch than ever before arrives
    CUDA_TRY(h, cudaDeviceSynchronize());
    if (crops_b + k_b + out_b > sl.bytes) {
      if (sl.buf) cudaFree(sl.buf);
      sl.buf = nullptr; sl.bytes = 0;
      CUDA_TRY(h, cudaMalloc(&sl.buf, crops_b + k_b + out_b));
      sl.bytes = crops_b + k_b + out_b;
    }
    if (ws_b > h->pipe_ws_bytes) {
      drop_graphs_on(h, h->pipe_ws);  // captured forwards that write into the old pipeline workspace
      if (h->pipe_ws) cudaFree(h->pipe_ws);
      h->pipe_ws = nullptr; h->pipe_ws_bytes = 0;
      CUDA_TRY(h, cudaMalloc(&h->pipe_ws, ws_b));
      h->pipe_ws_bytes = ws_b;
    }
  }
  char* base = (char*)sl.buf;
  float* d_crops = (float*)base;
  float* d_k = (float*)(base + crops_b);
  float* d_out = (float*)(base + crops_b + k_b);
  // copy stream: this slot's staging is free once its previous forward + read-back have completed
  if (sl.used) CUDA_TRY(h, cudaStreamWaitEvent(h->copy_stream, sl.done, 0));
  CUDA_TRY(h, cudaMemcpyAsync(d_crops, host_crops, (size_t)batch * 3 * S * S * 4, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(h, cudaMemcpyAsync(d_k, host_intrinsics, (size_t)batch * 9 * 4, cudaMemcpyHostToDevice, h->copy_stream));
  CUDA_TRY(h, cudaEventRecord(sl.h2d_done, h->copy_stream));
  // compute stream: forward of this step behind its own copy (and behind the previous step's forward: one workspace)
  CUDA_TRY(h, cudaStreamWaitEvent(st, sl.h2d_done, 0));
  int rc = mtb_forward(h, d_crops, d_k, batch, d_out, h->pipe_ws, h->pipe_ws_bytes, stream);
  if (rc) return rc;
  CUDA_TRY(h, cudaMemcpyAsync(host_coords3d_abs, d_out, (size_t)batch * h->cfg.n_joints * 3 * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(h, cudaEventRecord(sl.done, st));
  sl.used = true;
  return MTB_OK;
}

int mtb_forward_host_wait(mtb_handle* h, int slot) {
  if (!h || slot < 0 || slot > 1) return fail(h, MTB_ERR_INVALID_ARG, "null handle / invalid slot");
  DeviceGuard g(h->cfg.device);
  if (!h->slots[slot].used) return MTB_OK;
  CUDA_TRY(h, cudaEventSynchronize(h->slots[slot].done));
  return MTB_OK;
}

// ------------------------------------------------------------------------------------------------- NCCL
typedef struct { char internal[128]; } nccl_uid;
static void* open_nccl() {
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    void* l = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (l) return l;
  }
  return nullptr;
}

int mtb_comm_unique_id(void* id128) {
  if (!id128) return fail(nullptr, MTB_ERR_INVALID_ARG, "null id");
  void* lib = open_nccl();
  if (!lib) return fail(nullptr, MTB_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
  typedef int (*fn_t)(nccl_uid*);
  fn_t f = (fn_t)dlsym(lib, "ncclGetUniqueId");
  if (!f) return fail(nullptr, MTB_ERR_NCCL, "ncclGetUniqueId not found");
  int rc = f((nccl_uid*)id128);
  if (rc) return fail(nullptr, MTB_ERR_NCCL, "ncclGetUniqueId failed (%d)", rc);
  return MTB_OK;
}

int mtb_comm_init(mtb_handle* h, const void* id128, int rank, int world_size) {
  if (!h || !id128 || rank < 0 || rank >= world_size) return fail(h, MTB_ERR_INVALID_ARG, "invalid communicator arguments");
  DeviceGuard g(h->cfg.device);
  if (!h->nccl_lib) h->nccl_lib = open_nccl();
  if (!h->nccl_lib) return fail(h, MTB_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
  typedef int (*fn_t)(void**, int, nccl_uid, int);
  fn_t f = (fn_t)dlsym(h->nccl_lib, "ncclCommInitRank");
  if (!f) return fail(h, MTB_ERR_NCCL, "ncclCommInitRank not found");
  nccl_uid id;
  memcpy(&id, id128, sizeof(id));
  int rc = f(&h->nccl_comm, world_size, id, rank);
  if (rc) return fail(h, MTB_ERR_NCCL, "ncclCommInitRank failed (%d)", rc);
  h->nccl_world = world_size;
  return MTB_OK;
}

int mtb_allgather_joints(mtb_handle* h, const float* local, int floats_per_rank, float* all, void* stream) {
  if (!h || !local || !all || floats_per_rank <= 0) return fail(h, MTB_ERR_INVALID_ARG, "invalid all-gather arguments");
  if (!h->nccl_comm) return fail(h, MTB_ERR_NCCL, "mtb_comm_init has not been called");
  DeviceGuard g(h->cfg.device);
  typedef int (*fn_t)(const void*, void*, size_t, int, void*, cudaStream_t);
  static fn_t f = nullptr;
  if (!f) f = (fn_t)dlsym(h->nccl_lib, "ncclAllGather");
  if (!f) return fail(h, MTB_ERR_NCCL, "ncclAllGather not found");
  int rc = f(local, all, (size_t)floats_per_rank, /*ncclFloat32*/ 7, h->nccl_comm, (cudaStream_t)stream);
  if (rc) return fail(h, MTB_ERR_NCCL, "ncclAllGather failed (%d)", rc);
  return MTB_OK;
}

// ------------------------------------------------------------------------------------ multiperson (SURVEY 8f)
int mtb_image_pyramid(const uint8_t* images, int n_images, int height, int width, float* level1, float* level2, void* stream) {
  if (!images || !level1 || !level2 || n_images <= 0 || height < 4 || width < 4)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid pyramid arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int planes = n_images * 3;
  const size_t t1 = (size_t)planes * (height / 2) * (width / 2), t2 = (size_t)planes * (height / 4) * (width / 4);
  launch_k(pyramid_level1_kernel, dim3(grid_for(t1, 256)), dim3(256), 0, st, images, level1, planes, height, width);
  launch_k(pyramid_down_kernel, dim3(grid_for(t2, 256)), dim3(256), 0, st, (const float*)level1, level2, planes, height / 2, width / 2);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, MTB_ERR_CUDA, "pyramid launch: %s", cudaGetErrorString(e));
  return MTB_OK;
}

int mtb_crop_setup(const mtb_crop_setup_args* a, void* stream) {
  if (!a || !a->boxes || !a->intrinsics || !a->camspace_up || !a->aug_rotflipmat || !a->aug_scales || !a->new_intrinsics ||
      !a->rotations || !a->inv_projections || !a->pyramid_levels || (a->n_dist > 0 && !a->distortion))
    return fail(nullptr, MTB_ERR_INVALID_ARG, "null crop-setup argument");
  if (a->n_boxes <= 0 || a->num_aug <= 0 || a->num_aug > MP_MAX_AUG || a->box_stride < 4 || a->n_dist < 0 || a->n_dist > MP_NDIST ||
      a->resolution <= 0)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid crop-setup sizes (n_boxes=%d num_aug=%d n_dist=%d)", a->n_boxes, a->num_aug, a->n_dist);
  if (a->antialias_factor != 1 && a->antialias_factor != 2 && a->antialias_factor != 4)
    return fail(nullptr, MTB_ERR_UNSUPPORTED, "antialias_factor must be 1, 2 or 4 (got %d)", a->antialias_factor);
  CropSetupParams p;
  p.boxes = a->boxes; p.box_stride = a->box_stride; p.K = a->intrinsics; p.dist = a->distortion; p.ncoef = a->n_dist;
  p.up = a->camspace_up; p.rotflip = a->aug_rotflipmat; p.aug_scales = a->aug_scales;
  p.n_box = a->n_boxes; p.num_aug = a->num_aug; p.res = a->resolution; p.antialias = a->antialias_factor;
  p.new_K = a->new_intrinsics; p.R = a->rotations; p.invproj = a->inv_projections; p.level = a->pyramid_levels;
  launch_k(crop_setup_kernel, dim3((a->n_boxes + 127) / 128), dim3(128), 0, (cudaStream_t)stream, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, MTB_ERR_CUDA, "crop setup launch: %s", cudaGetErrorString(e));
  return MTB_OK;
}

int mtb_warp_crops(const mtb_warp_args* a, void* stream) {
  if (!a || !a->images || !a->level1 || !a->level2 || !a->intrinsics || !a->image_ids || !a->inv_projections ||
      !a->pyramid_levels || !a->gamma_exponents || !a->crops || (a->n_dist > 0 && !a->distortion))
    return fail(nullptr, MTB_ERR_INVALID_ARG, "null warp argument");
  if (a->n_boxes <= 0 || a->num_aug <= 0 || a->num_aug > MP_MAX_AUG || a->n_dist < 0 || a->n_dist > MP_NDIST || a->resolution <= 0 ||
      a->height < 4 || a->width < 4 || a->n_images <= 0)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid warp sizes");
  if (a->antialias_factor != 1 && a->antialias_factor != 2 && a->antialias_factor != 4)
    return fail(nullptr, MTB_ERR_UNSUPPORTED, "antialias_factor must be 1, 2 or 4 (got %d)", a->antialias_factor);
  if ((long long)a->n_boxes * a->num_aug > 65535) return fail(nullptr, MTB_ERR_UNSUPPORTED, "more than 65535 crops per call");
  WarpParams p;
  p.img = a->images; p.l1 = a->level1; p.l2 = a->level2; p.N = a->n_images; p.H = a->height; p.W = a->width;
  p.K = a->intrinsics; p.dist = a->distortion; p.ncoef = a->n_dist; p.image_ids = a->image_ids; p.invproj = a->inv_projections;
  p.level = a->pyramid_levels; p.gamma_exp = a->gamma_exponents; p.n_box = a->n_boxes; p.num_aug = a->num_aug;
  p.res = a->resolution; p.antialias = a->antialias_factor; p.crops = a->crops;
  const int npix = a->resolution * a->resolution;
  launch_k(warp_crops_kernel, dim3((npix + 255) / 256, a->n_boxes * a->num_aug), dim3(256), 0, (cudaStream_t)stream, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, MTB_ERR_CUDA, "warp launch: %s", cudaGetErrorString(e));
  return MTB_OK;
}

int mtb_tta_merge(const mtb_tta_args* a, void* stream) {
  if (!a || !a->poses || !a->rotations || !a->aug_should_flip || !a->mirror_mapping || !a->intrinsics || !a->extrinsics_inv ||
      !a->poses3d || !a->poses2d || (a->n_dist > 0 && !a->distortion))
    return fail(nullptr, MTB_ERR_INVALID_ARG, "null TTA-merge argument");
  if (a->n_boxes <= 0 || a->num_aug <= 0 || a->n_joints <= 0 || a->n_dist < 0 || a->n_dist > MP_NDIST)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid TTA-merge sizes");
  TtaParams p;
  p.poses = a->poses; p.R = a->rotations; p.flip = a->aug_should_flip; p.mirror = a->mirror_mapping; p.jt = a->joint_transform;
  p.skel = a->skeleton; p.K = a->intrinsics; p.dist = a->distortion; p.ncoef = a->n_dist; p.ext_inv = a->extrinsics_inv;
  p.n_box = a->n_boxes; p.num_aug = a->num_aug; p.J = a->n_joints;
  p.J2 = a->joint_transform ? a->n_joints_transformed : a->n_joints;
  p.Js = a->skeleton ? a->n_skeleton : p.J2;
  p.average = a->average_aug ? 1 : 0;
  p.poses3d = a->poses3d; p.poses2d = a->poses2d;
  if (p.J2 <= 0 || p.Js <= 0) return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid joint counts");
  launch_k(tta_merge_kernel, dim3(a->n_boxes), dim3(128), 0, (cudaStream_t)stream, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, MTB_ERR_CUDA, "TTA merge launch: %s", cudaGetErrorString(e));
  return MTB_OK;
}

int mtb_filter_poses(const mtb_filter_args* a, void* stream) {
  if (!a || !a->poses3d || !a->poses2d || !a->boxes || !a->image_start || !a->plausible || !a->keep || !a->scratch ||
      (a->n_bones > 0 && (!a->bones || !a->mean_bones)))
    return fail(nullptr, MTB_ERR_INVALID_ARG, "null pose-filter argument");
  if (a->n_images <= 0 || a->n_boxes <= 0 || a->num_aug < 2 || a->num_aug > MP_MAX_AUG || a->n_joints < 4 || a->box_stride < 5)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid pose-filter sizes (num_aug must be 2..16, boxes need a score column)");
  FilterParams p;
  p.poses3d = a->poses3d; p.poses2d = a->poses2d; p.boxes = a->boxes; p.box_stride = a->box_stride; p.bones = a->bones;
  p.mean_bones = a->mean_bones; p.n_bones = a->n_bones; p.image_start = a->image_start; p.num_aug = a->num_aug; p.J = a->n_joints;
  p.plausible = a->plausible; p.keep = a->keep; p.scratch = a->scratch;
  launch_k(pose_filter_kernel, dim3(a->n_images), dim3(128), 0, (cudaStream_t)stream, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, MTB_ERR_CUDA, "pose filter launch: %s", cudaGetErrorString(e));
  return MTB_OK;
}

// Data-parallel forward (SURVEY.md 8e): local crops -> backbone -> head decode, ONE all-gather of [coords2d | coords3d_rel]
// (5 floats per joint), absolute reconstruction of the FULL batch on every rank - reconstruct_ref_fullpersp normalises with
// batch-global RMS scalars (ptu3d.py:71-74), so only a full-batch solve reproduces the unsharded result exactly.
size_t mtb_sharded_scratch_bytes(const mtb_handle* h, int batch_local) {
  if (!h || batch_local <= 0 || h->nccl_world <= 0) return 0;
  const size_t J = (size_t)h->cfg.n_joints, bl = (size_t)batch_local, bt = bl * (size_t)h->nccl_world;
  return align_up(bl * J * 5 * 4, 256) + align_up(bt * J * 5 * 4, 256) + align_up(bt * J * 2 * 4, 256) + align_up(bt * J * 3 * 4, 256) +
         align_up(bt * J * 2 * 4, 256) + align_up(bt * 2 * 8, 256);
}

int mtb_forward_sharded(mtb_handle* h, const float* crops_local, int batch_local, const float* intrinsics_all, float* coords3d_abs_all,
                        void* scratch, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch_local, workspace_bytes, workspace);
  if (rc) return rc;
  if (!crops_local || !intrinsics_all || !coords3d_abs_all || !scratch) return fail(h, MTB_ERR_INVALID_ARG, "null argument");
  if (!h->nccl_comm) return fail(h, MTB_ERR_NCCL, "mtb_comm_init has not been called");
  if (h->ops.empty()) return fail(h, MTB_ERR_UNSUPPORTED, "this handle has no backbone (head-only)");
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t J = (size_t)h->cfg.n_joints, bl = (size_t)batch_local, bt = bl * (size_t)h->nccl_world;
  char* sp = (char*)scratch;
  float* packed_local = (float*)sp; sp += align_up(bl * J * 5 * 4, 256);
  float* packed_all = (float*)sp;   sp += align_up(bt * J * 5 * 4, 256);
  float* c2d_all = (float*)sp;      sp += align_up(bt * J * 2 * 4, 256);
  float* c3d_all = (float*)sp;      sp += align_up(bt * J * 3 * 4, 256);
  float* n2d = (float*)sp;          sp += align_up(bt * J * 2 * 4, 256);
  double* partial = (double*)sp;
  h->launches = 0;
  Workspace ws = layout(h, batch_local, workspace);
  void* features = ws.base + ws.off_features;
  rc = run_backbone(h, crops_local, batch_local, ws, features, st);
  if (rc) return rc;
  float* c2d = (float*)(ws.base + ws.off_c2d);
  float* c3d = (float*)(ws.base + ws.off_c3d);
  rc = head_decode_impl(h, features, batch_local, c2d, c3d, ws, st);
  if (rc) return rc;
  const int64_t before = h->launches;
  launch_k(pack_decoded_kernel, dim3(grid_for(bl * J, 256)), dim3(256), 0, st, (const float*)c2d, (const float*)c3d, packed_local,
           (int)(bl * J));
  rc = mtb_allgather_joints(h, packed_local, (int)(bl * J * 5), packed_all, stream);
  if (rc) return rc;
  launch_k(unpack_decoded_kernel, dim3(grid_for(bt * J, 256)), dim3(256), 0, st, (const float*)packed_all, c2d_all, c3d_all, (int)(bt * J));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(h, MTB_ERR_CUDA, "pack/unpack launch: %s", cudaGetErrorString(e));
  rc = recon_impl(h, c2d_all, c3d_all, intrinsics_all, (int)bt, coords3d_abs_all, n2d, partial, st);
  h->launches = before + 3 + 2;  // pack, all-gather, unpack, reconstruction passes
  return rc;
}

// ---------------------------------------------------------------------------------------- introspection
int mtb_num_ops(const mtb_handle* h) { return h ? (int)h->ops.size() : 0; }

const char* mtb_op_name(const mtb_handle* h, int op) {
  if (!h || op < 0 || op >= (int)h->ops.size()) return "";
  return h->ops[op].name.c_str();
}

int mtb_op_output_shape(const mtb_handle* h, int op, int* height, int* width, int* channels) {
  if (!h || op < 0 || op >= (int)h->ops.size()) return fail(h, MTB_ERR_INVALID_ARG, "op index out of range");
  const Op& o = h->ops[op];
  if (height) *height = (o.type == OP_POOL || o.small_io) ? 1 : o.Hout;
  if (width) *width = (o.type == OP_POOL || o.small_io) ? 1 : o.Wout;
  if (channels) *channels = o.Cout;
  return MTB_OK;
}

int mtb_debug_run_ops(mtb_handle* h, const float* crops, int batch, int n_ops, float* out, size_t out_floats,
                      void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch, workspace_bytes, workspace);
  if (rc) return rc;
  if (n_ops <= 0 || n_ops > (int)h->ops.size() || !out || !crops) return fail(h, MTB_ERR_INVALID_ARG, "invalid debug arguments");
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws = layout(h, batch, workspace);
  void* features = ws.base + ws.off_features;
  rc = run_ops_range(h, 0, (size_t)n_ops, crops, batch, ws, features, st);
  if (rc) return rc;
  const Op& o = h->ops[n_ops - 1];
  const bool small = o.type == OP_POOL || o.small_io;
  size_t n = (size_t)batch * (small ? 1 : (size_t)o.Hout * o.Wout) * o.Cout;
  if (n > out_floats) return fail(h, MTB_ERR_INVALID_ARG, "debug output buffer too small (%zu > %zu)", n, out_floats);
  void* src = buf_ptr(ws, o.out_buf, features);
  if (small || !is_bf16(h)) {
    CUDA_TRY(h, cudaMemcpyAsync(out, src, n * 4, cudaMemcpyDeviceToDevice, st));
  } else {
    launch_k(to_float_kernel, dim3(grid_for(n, 256)), dim3(256), 0, st, (const __nv_bfloat16*)src, out, n);
  }
  return MTB_OK;
}

int mtb_profile_begin(mtb_handle* h, unsigned class_mask) {
  if (!h) return fail(nullptr, MTB_ERR_INVALID_ARG, "null handle");
  h->prof_mask = class_mask;
  h->prof_used = 0;
  h->prof_cls.clear();
  h->prof_op.clear();
  h->prof_flops.clear();
  h->prof_bytes.clear();
  return MTB_OK;
}

int mtb_profile_end(mtb_handle* h, double* ms, double* flops, double* bytes, int64_t* launches) {
  if (!h || !ms || !flops || !bytes || !launches) return fail(h, MTB_ERR_INVALID_ARG, "null argument");
  DeviceGuard g(h->cfg.device);
  for (int i = 0; i < KC_COUNT; ++i) { ms[i] = 0; flops[i] = 0; bytes[i] = 0; launches[i] = 0; }
  h->prof_op_ms.assign(h->ops.size(), 0.0);
  for (size_t i = 0; i < h->prof_cls.size(); ++i) {
    CUDA_TRY(h, cudaEventSynchronize(h->prof_events[2 * i + 1]));
    float t = 0.f;
    CUDA_TRY(h, cudaEventElapsedTime(&t, h->prof_events[2 * i], h->prof_events[2 * i + 1]));
    int cls = h->prof_cls[i];
    ms[cls] += t;
    if (h->prof_op[i] >= 0 && h->prof_op[i] < (int)h->prof_op_ms.size()) h->prof_op_ms[h->prof_op[i]] += t;
    flops[cls] += h->prof_flops[i];
    bytes[cls] += h->prof_bytes[i];
    launches[cls] += (cls == KC_RECON) ? 2 : 1;
  }
  h->prof_mask = 0;
  h->prof_used = 0;
  h->prof_cls.clear();
  h->prof_op.clear();
  h->prof_flops.clear();
  h->prof_bytes.clear();
  return MTB_OK;
}

/* per-op device time (ms) accumulated by the last mtb_profile_begin/end window, plus each op's algorithmic FLOPs and
 * bytes PER CROP and its kernel class */
int mtb_profile_op_times(const mtb_handle* h, double* ms, double* flops_per_crop, double* bytes_per_crop, int* cls, int n) {
  if (!h || !ms || n < (int)h->ops.size()) return fail(h, MTB_ERR_INVALID_ARG, "invalid arguments");
  for (size_t i = 0; i < h->ops.size(); ++i) {
    ms[i] = i < h->prof_op_ms.size() ? h->prof_op_ms[i] : 0.0;
    if (flops_per_crop) flops_per_crop[i] = h->ops[i].flops;
    if (bytes_per_crop) bytes_per_crop[i] = op_bytes(h, h->ops[i], 1) - op_weight_bytes(h->ops[i]);  // activations only
    if (cls) cls[i] = op_class(h->ops[i]);
  }
  return MTB_OK;
}

double mtb_op_weight_bytes(const mtb_handle* h, int op) {
  if (!h || op < 0 || op >= (int)h->ops.size()) return 0.0;
  return op_weight_bytes(h->ops[op]);
}

int mtb_num_kernel_classes(void) { return KC_COUNT; }
const char* mtb_kernel_class_name(int cls) { return (cls >= 0 && cls < KC_COUNT) ? kKClassNames[cls] : ""; }

int mtb_op_input_shape(const mtb_handle* h, int op, int* height, int* width, int* channels, int* has_residual, int* has_scale) {
  if (!h || op < 0 || op >= (int)h->ops.size()) return fail(h, MTB_ERR_INVALID_ARG, "op index out of range");
  const Op& o = h->ops[op];
  if (height) *height = o.Hin;
  if (width) *width = o.Win;
  if (channels) *channels = o.Cin;
  if (has_residual) *has_residual = o.res_buf != BUF_NONE;
  if (has_scale) *has_scale = o.scale_buf != BUF_NONE;
  return MTB_OK;
}

int mtb_debug_run_op(mtb_handle* h, int op_index, const float* in, const float* res, const float* scale, int batch,
                     float* out, size_t out_floats, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch, workspace_bytes, workspace);
  if (rc) return rc;
  if (op_index < 0 || op_index >= (int)h->ops.size() || !in || !out) return fail(h, MTB_ERR_INVALID_ARG, "invalid debug arguments");
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws = layout(h, batch, workspace);
  Op o = h->ops[op_index];  // copy with overridden buffers
  const bool small = o.type == OP_POOL || o.small_io;
  const size_t n_in = (size_t)batch * o.Hin * o.Win * o.Cin;
  const size_t n_out = (size_t)batch * (o.type == OP_POOL ? 1 : (size_t)o.Hout * o.Wout) * o.Cout;
  if (n_out > out_floats) return fail(h, MTB_ERR_INVALID_ARG, "debug output buffer too small");
  if ((o.res_buf != BUF_NONE) != (res != nullptr) || (o.scale_buf != BUF_NONE) != (scale != nullptr))
    return fail(h, MTB_ERR_INVALID_ARG, "op %d: residual/scale inputs do not match the op (see mtb_op_input_shape)", op_index);
  auto put = [&](const float* src, int buf, size_t n, bool as_f32) {
    void* dst = buf_ptr(ws, buf, nullptr);
    if (as_f32 || !is_bf16(h)) cudaMemcpyAsync(dst, src, n * 4, cudaMemcpyDeviceToDevice, st);
    else launch_k(from_float_kernel, dim3(grid_for(n, 256)), dim3(256), 0, st, src, (__nv_bfloat16*)dst, n);
  };
  const float* crops = nullptr;
  if (o.type == OP_STEM) {
    crops = in;
  } else if (o.small_io) {
    o.in_buf = BUF_SMALL0;
    put(in, o.in_buf, n_in, true);
  } else {
    o.in_buf = 0;
    put(in, 0, n_in, false);
  }
  if (res) { o.res_buf = 1; put(res, 1, n_out, false); }
  if (scale) { o.scale_buf = BUF_SMALL0 + 2; put(scale, o.scale_buf, (size_t)batch * o.Cin, true); }
  o.out_buf = (o.type == OP_POOL || o.small_io) ? BUF_SMALL0 + 1 : 2;
  o.tc.cached_in = nullptr;  // the copy must not reuse a tensor map encoded for other buffers
  o.tc.map_sets.clear();
  o.tc32.map_sets.clear();
  o.dw_cache = DwTmaCache();
  o.fused_pool = false;      // in isolation a depthwise op does not pool and a pool op runs its own kernel
  rc = run_op(h, o, crops, batch, ws, nullptr, st);
  if (rc) return rc;
  void* src = buf_ptr(ws, o.out_buf, nullptr);
  if (small || !is_bf16(h)) CUDA_TRY(h, cudaMemcpyAsync(out, src, n_out * 4, cudaMemcpyDeviceToDevice, st));
  else launch_k(to_float_kernel, dim3(grid_for(n_out, 256)), dim3(256), 0, st, (const __nv_bfloat16*)src, out, n_out);
  return MTB_OK;
}

int mtb_op_is_fused_block(const mtb_handle* h, int op_index) {
  return (h && op_index >= 0 && op_index + 1 < (int)h->ops.size() && h->ops[op_index].fmb.ready && fmb_enabled()) ? 1 : 0;
}

int mtb_debug_run_fused_block(mtb_handle* h, int op_index, const float* in, int batch, float* out, size_t out_floats, void* workspace,
                              size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch, workspace_bytes, workspace);
  if (rc) return rc;
  if (op_index < 0 || op_index + 1 >= (int)h->ops.size() || !in || !out) return fail(h, MTB_ERR_INVALID_ARG, "invalid debug arguments");
  if (!h->ops[op_index].fmb.ready) return fail(h, MTB_ERR_UNSUPPORTED, "op %d does not start a fused FusedMBConv block", op_index);
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws = layout(h, batch, workspace);
  Op a = h->ops[op_index], b = h->ops[op_index + 1];
  const size_t n_in = (size_t)batch * a.Hin * a.Win * a.Cin, n_out = (size_t)batch * b.Hout * b.Wout * b.Cout;
  if (n_out > out_floats) return fail(h, MTB_ERR_INVALID_ARG, "debug output buffer too small");
  launch_k(from_float_kernel, dim3(grid_for(n_in, 256)), dim3(256), 0, st, in, (__nv_bfloat16*)buf_ptr(ws, 0, nullptr), n_in);
  a.in_buf = 0; a.out_buf = 1; b.in_buf = 1; b.out_buf = 2;
  if (b.res_buf != BUF_NONE) b.res_buf = 0;
  a.fmb.cached_out = nullptr;  // the copy must not reuse a tensor map encoded for other buffers
  rc = run_fused_block(h, a, b, batch, ws, nullptr, st);
  if (rc) return rc;
  launch_k(to_float_kernel, dim3(grid_for(n_out, 256)), dim3(256), 0, st, (const __nv_bfloat16*)buf_ptr(ws, 2, nullptr), out, n_out);
  return MTB_OK;
}

int64_t mtb_last_launch_count(const mtb_handle* h) { return h ? h->launches : 0; }
double mtb_backbone_flops_per_crop(const mtb_handle* h) { return h ? h->flops_per_crop : 0.0; }

int mtb_debug_fmb_plan(int cin, int cexp, int cout, int pair, int* nstages, int* npatch, int* stage_bytes, int* smem_bytes) {
  if (!nstages || !npatch || !stage_bytes || !smem_bytes) return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid arguments");
  *nstages = *npatch = *stage_bytes = *smem_bytes = 0;
  if (!fmb_shape_ok(cin, cexp, cout) || (pair && (cexp % FMB_NC != 0 || cin != cout))) return MTB_OK;
  const FmbPlan pl = fmb_plan(cin, cexp, cout, pair != 0);
  if (!pl.ok) return MTB_OK;
  *nstages = pl.nstages; *npatch = pl.npatch; *stage_bytes = pl.stage_bytes; *smem_bytes = pl.smem_bytes;
  return MTB_OK;
}

int mtb_debug_fmb_pack(const uint16_t* w1, const uint16_t* w2, int cin, int cexp, int cout, int pair, uint16_t* img1, uint16_t* img2) {
  if (!w1 || !w2 || !img1 || !img2 || !fmb_shape_ok(cin, cexp, cout)) return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid arguments");
  fmb_pack_images(w1, w2, cin, cexp, cout, pair ? 2 : 1, img1, img2);
  return MTB_OK;
}

int mtb_op_is_expdw(const mtb_handle* h, int op_index) {
  return (h && op_index >= 0 && op_index + 1 < (int)h->ops.size() && h->ops[op_index].expdw.ready && expdw_enabled()) ? 1 : 0;
}

int mtb_debug_run_expdw(mtb_handle* h, int op_index, const float* in, int batch, float* out, size_t out_floats, float* pooled,
                        size_t pooled_floats, int fused, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(h, batch, workspace_bytes, workspace);
  if (rc) return rc;
  if (op_index < 0 || op_index + 1 >= (int)h->ops.size() || !in || !out || !pooled) return fail(h, MTB_ERR_INVALID_ARG, "invalid debug arguments");
  if (!h->ops[op_index].expdw.ready) return fail(h, MTB_ERR_UNSUPPORTED, "op %d does not start a fused expand + depthwise pair", op_index);
  DeviceGuard g(h->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws = layout(h, batch, workspace);
  Op a = h->ops[op_index], d = h->ops[op_index + 1];  // copies with overridden buffers and fresh tensor-map caches
  const size_t n_in = (size_t)batch * a.Hin * a.Win * a.Cin, n_out = (size_t)batch * d.Hout * d.Wout * d.Cout;
  const size_t n_pool = (size_t)batch * d.Cout;
  if (n_out > out_floats || n_pool > pooled_floats) return fail(h, MTB_ERR_INVALID_ARG, "debug output buffer too small");
  launch_k(from_float_kernel, dim3(grid_for(n_in, 256)), dim3(256), 0, st, in, (__nv_bfloat16*)buf_ptr(ws, 0, nullptr), n_in);
  a.in_buf = 0; a.out_buf = 1; d.in_buf = 1; d.out_buf = 2;
  a.expdw.cached_in = nullptr;
  a.tc.cached_in = nullptr;
  a.tc.map_sets.clear();
  d.dw_cache = DwTmaCache();
  if (fused) {
    rc = run_expdw(h, a, d, batch, ws, nullptr, st);
  } else {  // the two launches, the depthwise one pooling as in a forward
    rc = run_op(h, a, nullptr, batch, ws, nullptr, st);
    if (!rc) rc = run_op(h, d, nullptr, batch, ws, nullptr, st);
  }
  if (rc) return rc;
  launch_k(to_float_kernel, dim3(grid_for(n_out, 256)), dim3(256), 0, st, (const __nv_bfloat16*)buf_ptr(ws, 2, nullptr), out, n_out);
  CUDA_TRY(h, cudaMemcpyAsync(pooled, buf_ptr(ws, BUF_SMALL0, nullptr), n_pool * 4, cudaMemcpyDeviceToDevice, st));
  return MTB_OK;
}

int mtb_debug_expdw_plan(int height, int width, int cin, int cexp, int* pixels_per_tile, int* crops_per_tile, int* nstages,
                         int* smem_bytes) {
  if (!pixels_per_tile || !crops_per_tile || !nstages || !smem_bytes) return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid arguments");
  const ExpdwPlan pl = expdw_plan(height, width, cin, cexp);
  *pixels_per_tile = pl.ok ? pl.pixels : 0;
  *crops_per_tile = pl.ok ? pl.crops : 0;
  *nstages = pl.ok ? pl.nstages : 0;
  *smem_bytes = pl.ok ? pl.smem_bytes : 0;
  return MTB_OK;
}

int mtb_debug_dw_plan(int height, int width, int* crops_per_item, int* rows_per_item, int* row_bands, int* stage_bytes) {
  if (height <= 0 || width <= 0 || !crops_per_item || !rows_per_item || !row_bands || !stage_bytes)
    return fail(nullptr, MTB_ERR_INVALID_ARG, "invalid arguments");
  const DwTmaPlan pl = dw_tma_plan(height, width);
  if (!pl.ok) { *crops_per_item = *rows_per_item = *row_bands = *stage_bytes = 0; return MTB_OK; }
  *crops_per_item = pl.G;
  *rows_per_item = pl.BH;
  *row_bands = pl.n_rb;
  *stage_bytes = 128 * (width + 2) * (pl.BH + 2) * pl.G;
  return MTB_OK;
}

}  // extern "C"
