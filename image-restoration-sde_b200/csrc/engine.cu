// irsde_b200 engine: context, weight store/repack, ConditionalUNet launch plan, sampler chain
// (CUDA-graph replay of one captured step) and the C ABI declared in include/irsde_b200.h.
//
// Data layout in HBM: activations are NHWC (channels-last) so that the skip concatenations of the
// UNet (DenoisingUNet_arch.py:118,121,127) are channel-offset views into one pre-allocated buffer
// (producers write at their channel offset: no torch.cat copies) and so that a 64-channel slab of a
// pixel row is one 128-byte line (the TMA / UMMA swizzle atom of the tensor-core engine).
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>

#include "../../include/irsde_b200.h"
#include "common.cuh"
#include "nafnet.cuh"

using namespace irsde;

namespace irsde {
bool g_pdl = false;  // IRSDE_PDL=1 enables programmatic dependent launch (read in tc_init)
}

namespace {
thread_local std::string g_last_error;

struct RawTensor {
  std::vector<int64_t> shape;
  float* dev = nullptr;
  long long numel = 0;
};

struct RunCfg {  // per-invocation pointers read by the op closures at launch time
  const float* x = nullptr;
  const float* mu = nullptr;
  float* out = nullptr;
  const float* ss = nullptr;  // time-modulation table
  const int* t_ptr = nullptr;
  int ss_img_stride = 0;
  const float* cam = nullptr;  // lens network: camera table [rows][cam_S] (irsde_set_lens)
  int cam_img_stride = 0;
};

struct Plan;
typedef std::function<void(Plan*, cudaStream_t)> Op;
enum { CAT_TC = 0, CAT_SIMT, CAT_LN, CAT_ATTN, CAT_MISC, CAT_UPDATE, CAT_COUNT };
struct OpRec {
  int cat;
  double flops;  // executed multiply-add flops (2*MAC) of this op, 0 for memory-bound ops
  Op fn;
  std::string label;   // for IRSDE_PROFILE_DUMP
  double bytes = 0.0;  // algorithmic HBM bytes (inputs + outputs + weights once)
  // NHWC view this op writes (irsde_trace_forward reads it back right after the op ran); null for fp32-NCHW outputs
  const void* out_p = nullptr;
  int out_pitch = 0, out_C = 0, out_H = 0, out_W = 0;
};

struct Plan {
  int B, H, W, Hp, Wp;
  std::vector<void*> allocs;
  std::vector<OpRec> ops;
  std::vector<OpRec> ops_dec;  // latent UNet: decode half (ops = encode half)
  int lat_h = 0, lat_w = 0;     // latent spatial size
  std::vector<TcConvDesc*> tc_descs;
  RunCfg cur;
  // chain state
  float *x_state = nullptr, *mu_buf = nullptr, *eps_buf = nullptr;
  StepState* d_step = nullptr;
  int* d_zero = nullptr;
  float *fwd_times = nullptr, *fwd_temb = nullptr, *fwd_table = nullptr;        // module-forward table (B rows)
  float *chain_times = nullptr, *chain_temb = nullptr, *chain_table = nullptr;  // chain table rows 0..cap-1
  int chain_cap = 0;
  cudaGraphExec_t graph[IRSDE_NUM_MODES] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  long long step_launches[IRSDE_NUM_MODES] = {0, 0, 0, 0, 0};
  // camera table pointer / image stride a step graph was captured with (lens network): a change re-captures
  const float* graph_cam[IRSDE_NUM_MODES] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  int graph_cam_stride[IRSDE_NUM_MODES] = {0, 0, 0, 0, 0};
  long long bytes = 0;               // device memory owned by this plan (plan cache accounting)
  unsigned long long last_use = 0;   // LRU stamp
};
}  // namespace

struct NafCfg {
  bool on = false;
  int img_channel = 0, width = 0, middle = 0, n_enc = 0, n_dec = 0;
  int enc[8] = {0}, dec[8] = {0};
  bool latent = false;
  bool lens = false;  // latent-bokeh variant: time_mlp.0/.2 keys, camera-modulated FFN gate, plain ending(x)
};

// Refusion latent autoencoder UNet (codes/config/latent-dehazing/models/modules/UNet_arch.py:17-97)
struct LatCfg {
  bool on = false;
  int in_ch = 0, out_ch = 0, ch = 0, depth = 0, embed = 0;
  int mult[9] = {1, 0, 0, 0, 0, 0, 0, 0, 0};  // [1] + ch_mult
};

struct irsde_ctx {
  irsde_config cfg;
  NafCfg naf;
  LatCfg lat;
  mutable std::string err;
  std::map<std::string, RawTensor> raw;
  bool finalized = false;
  std::map<std::string, float*> w_simt;  // [KH*KW][Cin][Cout] fp32
  std::map<std::string, bf16*> w_tc;     // [phase][tap][Cout][Cin] bf16
  std::map<std::string, float*> w_tc3;   // fp32x3: [phase][tap][2 (hi,lo)][Cout_pad][Cin] fp32 (tf32-rounded parts)
  bool use_tc3 = false;                  // fp32x3 mode: fp32 storage, convs through 3 x tcgen05.mma.kind::tf32
  std::map<std::string, int> ss_off;
  float *wall = nullptr, *ball = nullptr;
  int S = 0;
  // schedule
  bool have_sched = false;
  int T = 0;
  float dt = 0, max_sigma = 0;
  std::vector<float> thetas, sigmas, cumsum, sbars;
  float* coef_dev[IRSDE_NUM_MODES] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  std::map<std::tuple<int, int, int>, Plan*> plans;  // LRU-bounded cache, see build_plan()
  unsigned long long use_clock = 0;
  long long plan_bytes = 0;
  long long launches = 0;
  unsigned long long image_base = 0;  // uid of the first image of the next batch (Philox key; irsde_set_image_base)
  void* nccl_comm = nullptr;             // ncclComm_t (irsde_comm_init)
  int comm_rank = 0, comm_nranks = 1;
  unsigned long long* d_uids = nullptr;  // explicit per-image uids (irsde_set_image_uids), capacity MAX_UIDS
  int n_uids = 0;                        // 0: uid = image_base + b
  long long dev_bytes = 0;
  std::vector<void*> allocs;
  bool tc_ok = false;
  bool prof = false;
  struct ProfEv { int cat; double flops; cudaEvent_t e0, e1; const OpRec* op; };
  std::vector<ProfEv> prof_events;
  bool use_tc = false;  // bf16 mode: route eligible convs through the tcgen05 engine
  std::vector<int> udim;  // UNet channels per level: nf * [1, ch_mult...] (DenoisingUNet_arch.py:51-56)
  // lens network (irsde_create_nafnet_lens): every block's cam_mlp.1 concatenated [cam_S][2w], and the per-image camera
  // table cam_table[lens_n][cam_S] = (cam_scale, cam_shift) of every block, computed by irsde_set_lens.  Captured step graphs
  // read cam_table, so it is only re-written after draining the device and only re-allocated when it must grow.
  std::map<std::string, int> cam_off;
  int cam_S = 0;
  float *cam_wall = nullptr, *cam_ball = nullptr;
  float *cam_table = nullptr, *cam_gate = nullptr, *lens_dev = nullptr;
  int lens_cap = 0, lens_n = 0;
  std::vector<float> lens_host;  // [lens_n][3] as last set
};

namespace {

#define CUDA_TRY(ctx, expr)                                                                      \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      char _b[512];                                                                              \
      snprintf(_b, sizeof(_b), "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      (ctx)->err = _b;                                                                           \
      g_last_error = _b;                                                                         \
      return IRSDE_ERR_CUDA;                                                                     \
    }                                                                                            \
  } while (0)

int fail(const irsde_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  g_last_error = msg;
  return code;
}

void* dev_alloc(irsde_ctx* ctx, size_t bytes, std::vector<void*>* owner) {
  void* p = nullptr;
  if (bytes == 0) bytes = 16;
  if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
  ctx->dev_bytes += (long long)bytes;
  owner->push_back(p);
  return p;
}

// ---- weight repack kernels ---------------------------------------------------------------------
__global__ void pack_simt_kernel(const float* __restrict__ w, float* __restrict__ o, int Cout, int Cin, int KH, int KW) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)Cout * Cin * KH * KW;
  if (idx >= total) return;
  int co = idx % Cout;
  int c = (idx / Cout) % Cin;
  int tap = idx / ((long long)Cout * Cin);
  int r = tap / KW, s = tap % KW;
  o[idx] = w[(((long long)co * Cin + c) * KH + r) * KW + s];
}
// [tap][Cout][Cin] bf16
__global__ void pack_tc_kernel(const float* __restrict__ w, bf16* __restrict__ o, int Cout, int Cin, int KH, int KW) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)Cout * Cin * KH * KW;
  if (idx >= total) return;
  int c = idx % Cin;
  int co = (idx / Cin) % Cout;
  int tap = idx / ((long long)Cout * Cin);
  int r = tap / KW, s = tap % KW;
  o[idx] = __float2bfloat16_rn(w[(((long long)co * Cin + c) * KH + r) * KW + s]);
}
// nearest-x2 upsample followed by 3x3/pad1 == four 2x2 phase convolutions on the low-res input with
// pre-summed weights: [phase=(py,px)][tap=(a,b)][Cout][Cin]
__global__ void pack_tc_up_kernel(const float* __restrict__ w, bf16* __restrict__ o, int Cout, int Cin) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)16 * Cout * Cin;
  if (idx >= total) return;
  int c = idx % Cin;
  int co = (idx / Cin) % Cout;
  int tap = (idx / ((long long)Cout * Cin)) % 4;
  int phase = idx / ((long long)4 * Cout * Cin);
  int py = phase >> 1, px = phase & 1, a = tap >> 1, b = tap & 1;
  // rows of the 3x3 kernel that fall on low-res offset a for phase py
  int r0, r1, s0, s1;
  if (py == 0) { if (a == 0) { r0 = 0; r1 = 0; } else { r0 = 1; r1 = 2; } }
  else         { if (a == 0) { r0 = 0; r1 = 1; } else { r0 = 2; r1 = 2; } }
  if (px == 0) { if (b == 0) { s0 = 0; s1 = 0; } else { s0 = 1; s1 = 2; } }
  else         { if (b == 0) { s0 = 0; s1 = 1; } else { s0 = 2; s1 = 2; } }
  float acc = 0.f;
  for (int r = r0; r <= r1; ++r)
    for (int s = s0; s <= s1; ++s) acc += w[(((long long)co * Cin + c) * 3 + r) * 3 + s];
  o[idx] = __float2bfloat16_rn(acc);
}

// 7x7 stem as 7 row-taps with K=64 = 8 pixels x 8 channels (see conv_tc.cu): [r][Cout][s*8+c]
__global__ void pack_tc_stem_kernel(const float* __restrict__ w, bf16* __restrict__ o, int Cout, int Cin) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)7 * Cout * 64;
  if (idx >= total) return;
  int j = idx % 64;
  int co = (idx / 64) % Cout;
  int r = idx / ((long long)64 * Cout);
  int s = j >> 3, c = j & 7;
  float v = (s < 7 && c < Cin) ? w[(((long long)co * Cin + c) * 7 + r) * 7 + s] : 0.f;
  o[idx] = __float2bfloat16_rn(v);
}
// [tap][Cout_pad][Cin] with zero rows for co >= Cout (head conv, Cout=3)
__global__ void pack_tc_padded_kernel(const float* __restrict__ w, bf16* __restrict__ o, int Cout, int Cout_pad, int Cin,
                                      int KH, int KW) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)Cout_pad * Cin * KH * KW;
  if (idx >= total) return;
  int c = idx % Cin;
  int co = (idx / Cin) % Cout_pad;
  int tap = idx / ((long long)Cout_pad * Cin);
  int r = tap / KW, s = tap % KW;
  o[idx] = __float2bfloat16_rn(co < Cout ? w[(((long long)co * Cin + c) * KH + r) * KW + s] : 0.f);
}

// fp32x3 weights: [tap][2 (hi, lo)][Cout_pad][Cin] fp32, hi = rn_tf32(w), lo = rn_tf32(w - hi) (zero rows for co >= Cout)
__device__ __forceinline__ float rn_tf32_w(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
__global__ void pack_tc3_kernel(const float* __restrict__ w, float* __restrict__ o, int Cout, int Cout_pad, int Cin, int KH, int KW) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)Cout_pad * Cin * KH * KW;
  if (idx >= total) return;
  int c = idx % Cin;
  int co = (idx / Cin) % Cout_pad;
  int tap = idx / ((long long)Cout_pad * Cin);
  int r = tap / KW, s = tap % KW;
  float v = co < Cout ? w[(((long long)co * Cin + c) * KH + r) * KW + s] : 0.f;
  float hi = rn_tf32_w(v);
  long long base = ((long long)tap * 2 * Cout_pad + co) * Cin + c;
  o[base] = hi;
  o[base + (long long)Cout_pad * Cin] = rn_tf32_w(v - hi);
}
// nearest-x2 + 3x3 as four 2x2 phase convolutions (see pack_tc_up_kernel): [phase][tap][2][Cout_pad][Cin]
__global__ void pack_tc3_up_kernel(const float* __restrict__ w, float* __restrict__ o, int Cout, int Cout_pad, int Cin) {
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)16 * Cout_pad * Cin;
  if (idx >= total) return;
  int c = idx % Cin;
  int co = (idx / Cin) % Cout_pad;
  int tap = (idx / ((long long)Cout_pad * Cin)) % 4;
  int phase = idx / ((long long)4 * Cout_pad * Cin);
  int py = phase >> 1, px = phase & 1, a = tap >> 1, b = tap & 1;
  int r0, r1, s0, s1;
  if (py == 0) { if (a == 0) { r0 = 0; r1 = 0; } else { r0 = 1; r1 = 2; } }
  else         { if (a == 0) { r0 = 0; r1 = 1; } else { r0 = 2; r1 = 2; } }
  if (px == 0) { if (b == 0) { s0 = 0; s1 = 0; } else { s0 = 1; s1 = 2; } }
  else         { if (b == 0) { s0 = 0; s1 = 1; } else { s0 = 2; s1 = 2; } }
  float acc = 0.f;
  if (co < Cout)
    for (int r = r0; r <= r1; ++r)
      for (int q = s0; q <= s1; ++q) acc += w[(((long long)co * Cin + c) * 3 + r) * 3 + q];
  float hi = rn_tf32_w(acc);
  long long base = (((long long)(phase * 4 + tap) * 2) * Cout_pad + co) * Cin + c;
  o[base] = hi;
  o[base + (long long)Cout_pad * Cin] = rn_tf32_w(acc - hi);
}

// ---- architecture description --------------------------------------------------------------------
struct ResBlockInfo {
  std::string pre;
  int cin, cout;
};
// D[i] = channels of level i: nf * [1, ch_mult...][i] (nf * 2^i for the plain depth constructor)
std::vector<ResBlockInfo> resblocks(const irsde_config& c, const std::vector<int>& D) {
  std::vector<ResBlockInfo> v;
  char b[64];
  for (int i = 0; i < c.depth; ++i) {
    int di = D[i];
    snprintf(b, sizeof b, "downs.%d.0.", i); v.push_back({b, di, di});
    snprintf(b, sizeof b, "downs.%d.1.", i); v.push_back({b, di, di});
  }
  int mid = D[c.depth];
  v.push_back({"mid_block1.", mid, mid});
  v.push_back({"mid_block2.", mid, mid});
  for (int j = 0; j < c.depth; ++j) {
    int i = c.depth - 1 - j, di = D[i], dout = D[i + 1];
    snprintf(b, sizeof b, "ups.%d.0.", j); v.push_back({b, dout + di, dout});
    snprintf(b, sizeof b, "ups.%d.1.", j); v.push_back({b, dout + di, dout});
  }
  v.push_back({"final_res_block.", 2 * c.nf, c.nf});
  return v;
}

struct ParamSpec {
  std::string name;
  std::vector<int64_t> shape;
};

// NAFBlocks of ConditionalNAFNet in a fixed order (prefix, channels)   DenoisingNAFNet_arch.py:111-141
struct NafBlockInfo {
  std::string pre;
  int c;
};
std::vector<NafBlockInfo> naf_blocks(const NafCfg& n) {
  std::vector<NafBlockInfo> v;
  char b[64];
  int chan = n.width;
  for (int i = 0; i < n.n_enc; ++i) {
    for (int j = 0; j < n.enc[i]; ++j) { snprintf(b, sizeof b, "encoders.%d.%d.", i, j); v.push_back({b, chan}); }
    chan *= 2;
  }
  for (int j = 0; j < n.middle; ++j) { snprintf(b, sizeof b, "middle_blks.%d.", j); v.push_back({b, chan}); }
  for (int i = 0; i < n.n_dec; ++i) {
    chan /= 2;
    for (int j = 0; j < n.dec[i]; ++j) { snprintf(b, sizeof b, "decoders.%d.%d.", i, j); v.push_back({b, chan}); }
  }
  return v;
}
std::vector<ParamSpec> naf_param_specs(const NafCfg& n) {
  std::vector<ParamSpec> v;
  int64_t w = n.width, td = 4 * w, ic = n.img_channel;
  // lens variant (latent-bokeh/.../DenoisingNAFNet_arch.py:102-113): time_mlp without the embedding module (.0/.2), cam_mlp
  const char* tm = n.lens ? "time_mlp.0." : "time_mlp.1.";
  const char* tm2 = n.lens ? "time_mlp.2." : "time_mlp.3.";
  v.push_back({std::string(tm) + "weight", {2 * td, w}});
  v.push_back({std::string(tm) + "bias", {2 * td}});
  v.push_back({std::string(tm2) + "weight", {td, td}});
  v.push_back({std::string(tm2) + "bias", {td}});
  if (n.lens) {
    v.push_back({"cam_mlp.0.weight", {2 * td, 3 * w}});
    v.push_back({"cam_mlp.0.bias", {2 * td}});
    v.push_back({"cam_mlp.2.weight", {td, td}});
    v.push_back({"cam_mlp.2.bias", {td}});
  }
  v.push_back({"intro.weight", {w, 2 * ic, 3, 3}});
  v.push_back({"intro.bias", {w}});
  v.push_back({"ending.weight", {ic, w, 3, 3}});
  v.push_back({"ending.bias", {ic}});
  for (auto& blk : naf_blocks(n)) {
    int64_t c = blk.c;
    const std::string& p = blk.pre;
    v.push_back({p + "beta", {1, c, 1, 1}});
    v.push_back({p + "gamma", {1, c, 1, 1}});
    const std::string mp = p + (n.lens ? "time_mlp.1." : "mlp.1.");
    v.push_back({mp + "weight", {4 * c, td / 2}});
    v.push_back({mp + "bias", {4 * c}});
    if (n.lens) {  // latent-bokeh/.../DenoisingNAFNet_arch.py:22-24
      v.push_back({p + "cam_mlp.1.weight", {2 * c, td / 2}});
      v.push_back({p + "cam_mlp.1.bias", {2 * c}});
    }
    v.push_back({p + "conv1.weight", {2 * c, c, 1, 1}});
    v.push_back({p + "conv1.bias", {2 * c}});
    v.push_back({p + "conv2.weight", {2 * c, 1, 3, 3}});
    v.push_back({p + "conv2.bias", {2 * c}});
    v.push_back({p + "conv3.weight", {c, c, 1, 1}});
    v.push_back({p + "conv3.bias", {c}});
    v.push_back({p + "sca.1.weight", {c, c, 1, 1}});
    v.push_back({p + "sca.1.bias", {c}});
    v.push_back({p + "conv4.weight", {2 * c, c, 1, 1}});
    v.push_back({p + "conv4.bias", {2 * c}});
    v.push_back({p + "conv5.weight", {c, c, 1, 1}});
    v.push_back({p + "conv5.bias", {c}});
    v.push_back({p + "norm1.g", {1, c, 1, 1}});
    v.push_back({p + "norm2.g", {1, c, 1, 1}});
  }
  char b[64];
  int64_t chan = w << n.n_enc;
  for (int i = 0; i < n.n_dec; ++i) {
    snprintf(b, sizeof b, "ups.%d.0.weight", i);
    v.push_back({b, {chan * 2, chan, 1, 1}});
    chan /= 2;
  }
  chan = w;
  for (int i = 0; i < n.n_enc; ++i) {
    snprintf(b, sizeof b, "downs.%d.", i);
    v.push_back({std::string(b) + "weight", {chan * 2, chan, 2, 2}});
    v.push_back({std::string(b) + "bias", {chan * 2}});
    chan *= 2;
  }
  return v;
}
std::vector<ParamSpec> param_specs(const irsde_config& c, const std::vector<int>& D) {
  std::vector<ParamSpec> v;
  int64_t nf = c.nf, td = 4 * nf;
  int64_t cin0 = c.variant == IRSDE_NET_CONDITIONAL ? 2 * c.in_nc : c.in_nc;
  v.push_back({"init_conv.weight", {nf, cin0, 7, 7}});
  v.push_back({"time_mlp.1.weight", {td, nf}});
  v.push_back({"time_mlp.1.bias", {td}});
  v.push_back({"time_mlp.3.weight", {td, td}});
  v.push_back({"time_mlp.3.bias", {td}});
  for (auto& rb : resblocks(c, D)) {
    v.push_back({rb.pre + "mlp.1.weight", {2 * rb.cout, td}});
    v.push_back({rb.pre + "mlp.1.bias", {2 * rb.cout}});
    v.push_back({rb.pre + "block1.proj.weight", {rb.cout, rb.cin, 3, 3}});
    v.push_back({rb.pre + "block2.proj.weight", {rb.cout, rb.cout, 3, 3}});
    if (rb.cin != rb.cout) v.push_back({rb.pre + "res_conv.weight", {rb.cout, rb.cin, 1, 1}});
  }
  auto attn = [&](const std::string& pre, int64_t C, bool full) {
    v.push_back({pre + "fn.fn.to_qkv.weight", {384, C, 1, 1}});
    if (full) {
      v.push_back({pre + "fn.fn.to_out.weight", {C, 128, 1, 1}});
      v.push_back({pre + "fn.fn.to_out.bias", {C}});
    } else {
      v.push_back({pre + "fn.fn.to_out.0.weight", {C, 128, 1, 1}});
      v.push_back({pre + "fn.fn.to_out.0.bias", {C}});
      v.push_back({pre + "fn.fn.to_out.1.g", {1, C, 1, 1}});
    }
    v.push_back({pre + "fn.norm.g", {1, C, 1, 1}});
  };
  char b[64];
  for (int i = 0; i < c.depth; ++i) {
    int64_t di = D[i], dout = D[i + 1];
    snprintf(b, sizeof b, "downs.%d.2.", i);
    attn(b, di, false);
    snprintf(b, sizeof b, "downs.%d.3.", i);
    if (i != c.depth - 1) {
      v.push_back({std::string(b) + "weight", {dout, di, 4, 4}});
      v.push_back({std::string(b) + "bias", {dout}});
    } else {
      v.push_back({std::string(b) + "weight", {dout, di, 3, 3}});
    }
  }
  attn("mid_attn.", D[c.depth], c.variant == IRSDE_NET_DENOISING);
  for (int j = 0; j < c.depth; ++j) {
    int i = c.depth - 1 - j;
    int64_t di = D[i], dout = D[i + 1];
    snprintf(b, sizeof b, "ups.%d.2.", j);
    attn(b, dout, false);
    if (i != 0) {
      snprintf(b, sizeof b, "ups.%d.3.1.", j);
      v.push_back({std::string(b) + "weight", {di, dout, 3, 3}});
      v.push_back({std::string(b) + "bias", {di}});
    } else {
      snprintf(b, sizeof b, "ups.%d.3.", j);
      v.push_back({std::string(b) + "weight", {di, dout, 3, 3}});
    }
  }
  v.push_back({"final_conv.weight", {c.out_nc, nf, 3, 3}});
  v.push_back({"final_conv.bias", {c.out_nc}});
  return v;
}

std::vector<ParamSpec> lat_param_specs(const LatCfg& L) {
  std::vector<ParamSpec> v;
  char b[64];
  v.push_back({"init_conv.weight", {L.ch, L.in_ch, 3, 3}});
  auto rb = [&](const std::string& pre, int64_t ci, int64_t co) {
    v.push_back({pre + "block1.proj.weight", {co, ci, 3, 3}});
    v.push_back({pre + "block2.proj.weight", {co, co, 3, 3}});
    if (ci != co) v.push_back({pre + "res_conv.weight", {co, ci, 1, 1}});
  };
  auto la = [&](const std::string& pre, int64_t C) {
    v.push_back({pre + "fn.fn.to_qkv.weight", {384, C, 1, 1}});
    v.push_back({pre + "fn.fn.to_out.0.weight", {C, 128, 1, 1}});
    v.push_back({pre + "fn.fn.to_out.0.bias", {C}});
    v.push_back({pre + "fn.fn.to_out.1.g", {1, C, 1, 1}});
    v.push_back({pre + "fn.norm.g", {1, C, 1, 1}});
  };
  for (int i = 0; i < L.depth; ++i) {
    int64_t di = (int64_t)L.ch * L.mult[i], dout = (int64_t)L.ch * L.mult[i + 1];
    snprintf(b, sizeof b, "encoder.%d.", i);
    std::string pre = b;
    rb(pre + "0.", di, di);
    rb(pre + "1.", di, di);
    if (i == L.depth - 1) la(pre + "2.", di);
    if (i != L.depth - 1) {
      v.push_back({pre + "3.weight", {dout, di, 4, 4}});
      v.push_back({pre + "3.bias", {dout}});
    } else {
      v.push_back({pre + "3.weight", {dout, di, 3, 3}});
    }
  }
  for (int j = 0; j < L.depth; ++j) {
    int i = L.depth - 1 - j;
    int64_t di = (int64_t)L.ch * L.mult[i], dout = (int64_t)L.ch * L.mult[i + 1];
    snprintf(b, sizeof b, "decoder.%d.", j);
    std::string pre = b;
    rb(pre + "0.", dout + di, dout);
    rb(pre + "1.", dout + di, dout);
    if (i == L.depth - 1) la(pre + "2.", dout);
    if (i != 0) {
      v.push_back({pre + "3.1.weight", {di, dout, 3, 3}});
      v.push_back({pre + "3.1.bias", {di}});
    } else {
      v.push_back({pre + "3.weight", {di, dout, 3, 3}});
    }
  }
  int64_t mid = (int64_t)L.ch * L.mult[L.depth];
  v.push_back({"latent_conv.weight", {L.embed, mid, 1, 1}});
  v.push_back({"post_latent_conv.weight", {mid, L.embed, 1, 1}});
  v.push_back({"final_conv.weight", {L.out_ch, L.ch, 3, 3}});
  v.push_back({"final_conv.bias", {L.out_ch}});
  return v;
}

// ---- plan builder ----------------------------------------------------------------------------------
template <typename T>
struct Builder {
  irsde_ctx* ctx;
  Plan* plan;
  bool ok = true;
  std::string err;
  std::multimap<size_t, void*> free_tmp;
  std::map<void*, size_t> tmp_size;
  const float* pending_mult = nullptr;  // per-output-channel multiplier for the NEXT conv() (NAFBlock beta / gamma)
  int nchw_H = 0, nchw_W = 0;           // crop size of fp32 NCHW outputs (0 = the image size)
  bool stem_padded = false;  // X0 lives in the zero-bordered [B][Hp+6][Wp+8][8] layout of the tcgen05 stem

  T* alloc(long long elems) {
    void* p = dev_alloc(ctx, (size_t)elems * sizeof(T), &plan->allocs);
    if (!p) { ok = false; err = "cudaMalloc failed in plan builder"; }
    return (T*)p;
  }
  T* tmp(long long elems) {
    size_t bytes = (size_t)elems * sizeof(T);
    auto it = free_tmp.lower_bound(bytes);
    if (it != free_tmp.end() && it->first <= bytes * 2 + 4096) {
      void* p = it->second;
      free_tmp.erase(it);
      return (T*)p;
    }
    void* p = alloc(elems);
    tmp_size[p] = bytes;
    return (T*)p;
  }
  void release(void* p) { free_tmp.insert({tmp_size[p], p}); }

  float* fw(const std::string& n) {  // fp32 raw parameter (bias / gain vectors)
    auto it = ctx->raw.find(n);
    if (it == ctx->raw.end()) { ok = false; err = "missing tensor " + n; return nullptr; }
    return it->second.dev;
  }

  struct V { T* p; int pitch; int C; };  // channel-offset NHWC view
  static V view(T* base, int pitch, int off, int C) { return V{base + off, pitch, C}; }
  void mark_out(V out, int H, int W) {  // the op just pushed writes this view (irsde_trace_forward)
    OpRec& r = plan->ops.back();
    r.out_p = out.p; r.out_pitch = out.pitch; r.out_C = out.C; r.out_H = H; r.out_W = W;
  }

  // generic conv op. ss_block = ResBlock prefix whose (scale,shift) modulate the output ("" = none)
  void conv(const std::string& wname, V in, int Hin, int Win, int K, int stride, int pad, int up, const char* bias,
            const std::string& ss_block, int silu, const V* res, V out, int Cout, float** out_nchw_slot = nullptr,
            int tc_flags = 0, const bf16* w_override = nullptr) {
    size_t first = plan->ops.size();
    conv_impl(wname, in, Hin, Win, K, stride, pad, up, bias, ss_block, silu, res, out, Cout, out_nchw_slot, tc_flags, w_override);
    if (plan->ops.size() > first) {
      OpRec& r = plan->ops.back();
      char b[160];
      int Ho = (Hin * up + 2 * pad - K) / stride + 1, Wo = (Win * up + 2 * pad - K) / stride + 1;
      snprintf(b, sizeof b, "%s %dx%d k%d s%d up%d Cin%d Cout%d", wname.c_str(), Hin, Win, K, stride, up, in.C, Cout);
      r.label = b;
      if (!out_nchw_slot) { r.out_p = out.p; r.out_pitch = out.pitch; r.out_C = Cout; r.out_H = Ho; r.out_W = Wo; }
      double esz = sizeof(T);
      r.bytes = (double)plan->B * Hin * Win * in.C * esz + (double)plan->B * Ho * Wo * Cout * (out_nchw_slot ? 4.0 : esz) +
                (double)K * K * in.C * Cout * esz + (res ? (double)plan->B * Ho * Wo * Cout * esz : 0.0);
    }
  }
  void conv_impl(const std::string& wname, V in, int Hin, int Win, int K, int stride, int pad, int up, const char* bias,
                 const std::string& ss_block, int silu, const V* res, V out, int Cout, float** out_nchw_slot, int tc_flags,
                 const bf16* w_override) {
    ConvGeom g;
    g.B = plan->B; g.Hin = Hin; g.Win = Win; g.Cin = in.C; g.up = up; g.KH = K; g.KW = K; g.stride = stride; g.pad = pad;
    g.Hout = (Hin * up + 2 * pad - K) / stride + 1;
    g.Wout = (Win * up + 2 * pad - K) / stride + 1;
    g.Cout = Cout;
    double simt_flops = 2.0 * plan->B * g.Hout * g.Wout * (double)Cout * in.C * K * K;
    // the tensor-core engine runs nearest-x2 + 3x3 as four 2x2 phase convolutions: 4 taps per output pixel
    double tc_flops = (K == 3 && up == 2) ? simt_flops * 4.0 / 9.0 : simt_flops;
    Epilogue ep;
    memset(&ep, 0, sizeof ep);
    ep.bias = bias ? fw(bias) : nullptr;
    ep.mult_vec = pending_mult;
    pending_mult = nullptr;
    ep.silu = silu;
    ep.ss_S = ctx->S;
    bool use_ss = !ss_block.empty();
    ep.ss_off = use_ss ? ctx->ss_off[ss_block] : 0;
    if (res) { ep.res = res->p; ep.res_pitch = res->pitch; }
    irsde_ctx* c = ctx;
    bool nchw = out_nchw_slot != nullptr;
    if constexpr (std::is_same<T, bf16>::value) {
      bool shape_ok = (K == 3 && stride == 1 && pad == 1) || (K == 1 && stride == 1 && pad == 0 && up == 1) ||
                      (K == 4 && stride == 2 && pad == 1 && up == 1 && Hin % 2 == 0 && Win % 2 == 0) ||
                      (K == 2 && stride == 2 && pad == 0 && up == 1 && Hin % 2 == 0 && Win % 2 == 0);
      bool stem_tc = ctx->use_tc && stem_padded && K == 7 && Cout % 8 == 0 && out.pitch % 8 == 0;
      if (stem_tc) {
        const bf16* wt = ctx->w_tc[wname];
        if (!wt) { ok = false; err = "unpacked tc weight " + wname; return; }
        TcTap taps[16];
        for (int r = 0; r < 7; ++r) taps[r] = TcTap{r, 0, 0};
        std::string terr;
        TcConvDesc* d = tc_conv_create(in.p, 8, plan->B, Hin, Win, 64, -1, wt, Cout, 7, taps, 1, ep, out.p, out.pitch, g.Hout,
                                       g.Wout, &terr);
        if (!d) { ok = false; err = "tc_conv_create(stem): " + terr; return; }
        plan->tc_descs.push_back(d);
        double fl = 2.0 * plan->B * g.Hout * g.Wout * (double)Cout * 448;
        plan->ops.push_back(OpRec{CAT_TC, fl, [=](Plan*, cudaStream_t st) {
          tc_conv_launch(d, st);
          c->launches++;
        }});
        return;
      }
      if (ctx->use_tc && shape_ok && in.C % 8 == 0 && in.pitch % 8 == 0 &&
          (nchw ? (K == 3 && up == 1) : (Cout % 8 == 0 && out.pitch % 8 == 0))) {
        const bf16* wt = w_override ? w_override : ctx->w_tc[wname];
        if (!wt) { ok = false; err = "unpacked tc weight " + wname; return; }
        TcTap taps[16];
        int ntaps = 0, nph = 1, planes = 1, Ha = Hin, Wa = Win, a_pitch = in.pitch;
        const bf16* a_ptr = in.p;
        if (K == 3 && up == 1) {
          for (int r = 0; r < 3; ++r) for (int q = 0; q < 3; ++q) taps[ntaps++] = TcTap{r - 1, q - 1, 0};
        } else if (K == 3 && up == 2) {
          nph = 4;
          for (int a = 0; a < 2; ++a) for (int q = 0; q < 2; ++q) taps[ntaps++] = TcTap{a - 1, q - 1, 0};
        } else if (K == 1) {
          taps[ntaps++] = TcTap{0, 0, 0};
        } else {  // stride 2 over space-to-depth planes: 4x4 pad 1 (UNet Downsample) or 2x2 pad 0 (NAFNet downs)
          static const int PY[4] = {1, 0, 1, 0}, DH[4] = {-1, 0, 0, 1};
          if (K == 4) {
            for (int r = 0; r < 4; ++r) for (int q = 0; q < 4; ++q) taps[ntaps++] = TcTap{DH[r], DH[q], PY[r] * 2 + PY[q]};
          } else {
            for (int r = 0; r < 2; ++r) for (int q = 0; q < 2; ++q) taps[ntaps++] = TcTap{0, 0, r * 2 + q};
          }
          planes = 4; Ha = Hin / 2; Wa = Win / 2; a_pitch = in.C;
          bf16* s2d = tmp((long long)plan->B * Hin * Win * in.C);
          int Bc = plan->B, Cc = in.C;
          plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
            launch_space_to_depth<bf16>(in.p, in.pitch, s2d, Bc, Hin, Win, Cc, st);
            c->launches++;
          }});
          a_ptr = s2d;
          release(s2d);  // safe: stream order; the next tmp user runs after this conv
        }
        std::string terr;
        TcConvDesc* d = tc_conv_create(a_ptr, a_pitch, plan->B, Ha, Wa, in.C, planes, wt, Cout, ntaps, taps, nph, ep, out.p,
                                       out.pitch, g.Hout, g.Wout, &terr, tc_flags);
        if (!d) { ok = false; err = "tc_conv_create(" + wname + "): " + terr; return; }
        plan->tc_descs.push_back(d);
        int cH = nchw_H ? nchw_H : plan->H, cW = nchw_W ? nchw_W : plan->W;
        plan->ops.push_back(OpRec{CAT_TC, tc_flops, [=](Plan* p, cudaStream_t st) {
          if (use_ss) tc_conv_set_runtime(d, p->cur.ss, p->cur.t_ptr, p->cur.ss_img_stride);
          if (nchw) tc_conv_set_out_nchw(d, p->cur.out, cH, cW);
          tc_conv_launch(d, st);
          c->launches++;
        }});
        return;
      }
    }
    if constexpr (std::is_same<T, float>::value) {
      bool shape_ok = (K == 3 && stride == 1 && pad == 1) || (K == 1 && stride == 1 && pad == 0 && up == 1) ||
                      (K == 4 && stride == 2 && pad == 1 && up == 1 && Hin % 2 == 0 && Win % 2 == 0) ||
                      (K == 2 && stride == 2 && pad == 0 && up == 1 && Hin % 2 == 0 && Win % 2 == 0);
      if (ctx->use_tc3 && shape_ok && !tc_flags && !w_override && in.C % 4 == 0 && in.pitch % 4 == 0 &&
          (((uintptr_t)in.p) & 15) == 0 && (nchw ? (K == 3 && up == 1) : (Cout % 4 == 0 && out.pitch % 4 == 0))) {
        const float* wt = ctx->w_tc3[wname];
        if (!wt) { ok = false; err = "unpacked fp32x3 weight " + wname; return; }
        TcTap taps[16];
        int ntaps = 0, nph = 1, planes = 1, Ha = Hin, Wa = Win;
        const float* a_src = in.p;
        int a_pitch = in.pitch;
        if (K == 3 && up == 1) {
          for (int r = 0; r < 3; ++r) for (int q = 0; q < 3; ++q) taps[ntaps++] = TcTap{r - 1, q - 1, 0};
        } else if (K == 3 && up == 2) {
          nph = 4;
          for (int a = 0; a < 2; ++a) for (int q = 0; q < 2; ++q) taps[ntaps++] = TcTap{a - 1, q - 1, 0};
        } else if (K == 1) {
          taps[ntaps++] = TcTap{0, 0, 0};
        } else {
          static const int PY[4] = {1, 0, 1, 0}, DH[4] = {-1, 0, 0, 1};
          if (K == 4) {
            for (int r = 0; r < 4; ++r) for (int q = 0; q < 4; ++q) taps[ntaps++] = TcTap{DH[r], DH[q], PY[r] * 2 + PY[q]};
          } else {
            for (int r = 0; r < 2; ++r) for (int q = 0; q < 2; ++q) taps[ntaps++] = TcTap{0, 0, r * 2 + q};
          }
          planes = 4; Ha = Hin / 2; Wa = Win / 2;
          float* s2d = tmp((long long)plan->B * Hin * Win * in.C);
          int Bc = plan->B, Cc = in.C;
          plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
            launch_space_to_depth<float>(in.p, in.pitch, s2d, Bc, Hin, Win, Cc, st);
            c->launches++;
          }});
          a_src = s2d; a_pitch = in.C;
          release(s2d);
        }
        // operand split (hi, lo) of the conv input: [2][planes][B][Ha][Wa][C]
        const long long npix_a = (long long)planes * plan->B * Ha * Wa;
        float* split = tmp(2 * npix_a * in.C);
        {
          int Cc = in.C;
          plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
            launch_split_tf32(a_src, a_pitch, split, npix_a, Cc, st);
            c->launches++;
          }});
          plan->ops.back().label = wname + " tf32 hi/lo split of the input";
          plan->ops.back().bytes = 3.0 * npix_a * in.C * 4.0;
        }
        std::string terr;
        TcConvDesc* d = tc_conv_create_f32x3(split, plan->B, Ha, Wa, in.C, planes, wt, Cout, ntaps, taps, nph, ep, out.p, out.pitch,
                                             g.Hout, g.Wout, &terr);
        release(split);
        if (!d) { ok = false; err = "tc_conv_create_f32x3(" + wname + "): " + terr; return; }
        plan->tc_descs.push_back(d);
        int cH = nchw_H ? nchw_H : plan->H, cW = nchw_W ? nchw_W : plan->W;
        plan->ops.push_back(OpRec{CAT_TC, tc_flops, [=](Plan* p, cudaStream_t st) {
          if (use_ss) tc_conv_set_runtime(d, p->cur.ss, p->cur.t_ptr, p->cur.ss_img_stride);
          if (nchw) tc_conv_set_out_nchw(d, p->cur.out, cH, cW);
          tc_conv_launch(d, st);
          c->launches++;
        }});
        return;
      }
    }
    if (tc_flags || w_override) { ok = false; err = "fused attention conv needs the tensor-core engine: " + wname; return; }
    const float* w = ctx->w_simt[wname];
    if (!w) { ok = false; err = "unpacked weight " + wname; return; }
    int H = nchw_H ? nchw_H : plan->H, Wd = nchw_W ? nchw_W : plan->W;
    plan->ops.push_back(OpRec{CAT_SIMT, simt_flops, [=](Plan* p, cudaStream_t st) {
      Epilogue e = ep;
      if (use_ss) { e.ss = p->cur.ss; e.t_ptr = p->cur.t_ptr; e.ss_img_stride = p->cur.ss_img_stride; }
      launch_conv_simt<T>(g, in.p, in.pitch, w, e, out.p, out.pitch, nchw ? p->cur.out : nullptr, H, Wd, st);
      c->launches++;
    }});
  }

  void resblock(const std::string& pre, V in, int Cout, V out, int H, int W, bool time_mod = true) {
    long long npix = (long long)plan->B * H * W;
    T* h1 = tmp(npix * Cout);
    V vh1{h1, Cout, Cout};
    conv(pre + "block1.proj.weight", in, H, W, 3, 1, 1, 1, nullptr, time_mod ? pre : std::string(), 1, nullptr, vh1, Cout);
    V res = in;
    T* r = nullptr;
    if (in.C != Cout) {
      r = tmp(npix * Cout);
      res = V{r, Cout, Cout};
      conv(pre + "res_conv.weight", in, H, W, 1, 1, 0, 1, nullptr, "", 0, nullptr, res, Cout);
    }
    conv(pre + "block2.proj.weight", vh1, H, W, 3, 1, 1, 1, nullptr, "", 1, &res, out, Cout);
    release(h1);
    if (r) release(r);
  }

  // Residual(PreNorm(LinearAttention)) or Residual(PreNorm(Attention)); pre = "...2." / "mid_attn."
  void attention(const std::string& pre, V in, V out, int H, int W, bool full, float* la_partial, float* la_ctx) {
    int C = in.C, B = plan->B, N = H * W;
    long long npix = (long long)B * N;
    T* xn = tmp(npix * C);
    float* g1 = fw(pre + "fn.norm.g");
    irsde_ctx* c = ctx;
    plan->ops.push_back(OpRec{CAT_LN, 0.0, [=](Plan*, cudaStream_t st) {
      launch_layernorm<T>(in.p, in.pitch, g1, nullptr, 0, xn, C, npix, C, st);
      c->launches++;
    }});
    plan->ops.back().label = pre + "norm";
    plan->ops.back().bytes = 2.0 * npix * C * sizeof(T);
    mark_out(V{xn, C, C}, H, W);
    T* qkv = tmp(npix * 384);
    if constexpr (std::is_same<T, bf16>::value) {
      if (!full && ctx->use_tc && tc_fused_attention_available() && C % 8 == 0) {
        // Fused LinearAttention: (1) the to_qkv GEMM epilogue applies softmax_d(q)*32^-.5 per head, (2) k,v -> ctx,
        // (3) ctx is folded into the to_out weights per image, (4) ONE per-image-weight 1x1 GEMM on q gives to_out's
        // output (module_util.py:163-178 with the two einsums + to_out conv re-associated), (5) LayerNorm + residual.
        conv(pre + "fn.fn.to_qkv.weight", V{xn, C, C}, H, W, 1, 1, 0, 1, nullptr, "", 0, nullptr, V{qkv, 384, 384}, 384, nullptr,
             TC_FLAG_QSOFTMAX);
        release(xn);
        plan->ops.push_back(OpRec{CAT_ATTN, 0.0, [=](Plan*, cudaStream_t st) {
          launch_linattn_ctx<T>(qkv, 384, la_partial, la_ctx, B, N, st);
          c->launches += 2;
        }});
        plan->ops.back().label = pre + "linattn kv->ctx (2 kernels)";
        plan->ops.back().bytes = (double)npix * 256 * sizeof(T);
        bf16* Mb = tmp((long long)B * C * 128);
        float* wout = fw(pre + "fn.fn.to_out.0.weight");
        // (combine + fold in ONE kernel was tried in round 2: 8-64 blocks of latency-bound work instead of 32 + 256..4096
        //  measured 0.62 vs 0.55 ms of attention time per step, same box ABAB - kept as two launches)
        plan->ops.push_back(OpRec{CAT_ATTN, 0.0, [=](Plan*, cudaStream_t st) {
          launch_la_fold(la_ctx, wout, Mb, B, C, st);
          c->launches++;
        }});
        plan->ops.back().label = pre + "fold ctx into to_out";
        T* y = tmp(npix * C);
        std::string bn = pre + "fn.fn.to_out.0.bias";
        conv(pre + "fn.fn.to_out.0.weight", V{qkv, 384, 128}, H, W, 1, 1, 0, 1, bn.c_str(), "", 0, nullptr, V{y, C, C}, C, nullptr,
             TC_FLAG_W_PER_IMAGE, Mb);
        float* g2 = fw(pre + "fn.fn.to_out.1.g");
        plan->ops.push_back(OpRec{CAT_LN, 0.0, [=](Plan*, cudaStream_t st) {
          launch_layernorm<T>(y, C, g2, in.p, in.pitch, out.p, out.pitch, npix, C, st);
          c->launches++;
        }});
        plan->ops.back().label = pre + "to_out.norm+res";
        plan->ops.back().bytes = 3.0 * npix * C * sizeof(T);
        mark_out(out, H, W);
        release(y);
        release(Mb);
        release(qkv);
        return;
      }
    }
    conv(pre + "fn.fn.to_qkv.weight", V{xn, C, C}, H, W, 1, 1, 0, 1, nullptr, "", 0, nullptr, V{qkv, 384, 384}, 384);
    release(xn);
    T* hid = tmp(npix * 128);
    if (full) {
      plan->ops.push_back(OpRec{CAT_ATTN, 0.0, [=](Plan*, cudaStream_t st) {
        launch_fullattn<T>(qkv, 384, hid, 128, B, N, st);
        c->launches++;
      }});
      plan->ops.back().label = pre + "full attention";
      mark_out(V{hid, 128, 128}, H, W);
      std::string bn = pre + "fn.fn.to_out.bias";
      conv(pre + "fn.fn.to_out.weight", V{hid, 128, 128}, H, W, 1, 1, 0, 1, bn.c_str(), "", 0, &in, out, C);
    } else {
      plan->ops.push_back(OpRec{CAT_ATTN, 0.0, [=](Plan*, cudaStream_t st) {
        launch_linattn<T>(qkv, 384, la_partial, la_ctx, hid, 128, B, N, st);
        c->launches += 3;
      }});
      plan->ops.back().label = pre + "linattn(3 kernels)";
      plan->ops.back().bytes = (double)npix * (384 + 128) * sizeof(T);
      T* y = tmp(npix * C);
      std::string bn = pre + "fn.fn.to_out.0.bias";
      conv(pre + "fn.fn.to_out.0.weight", V{hid, 128, 128}, H, W, 1, 1, 0, 1, bn.c_str(), "", 0, nullptr, V{y, C, C}, C);
      float* g2 = fw(pre + "fn.fn.to_out.1.g");
      plan->ops.push_back(OpRec{CAT_LN, 0.0, [=](Plan*, cudaStream_t st) {
        launch_layernorm<T>(y, C, g2, in.p, in.pitch, out.p, out.pitch, npix, C, st);
        c->launches++;
      }});
      plan->ops.back().label = pre + "to_out.norm+res";
      plan->ops.back().bytes = 3.0 * npix * C * sizeof(T);
      mark_out(out, H, W);
      release(y);
    }
    release(qkv);
    release(hid);
  }

  // ---- latent autoencoder UNet.encode / UNet.decode (UNet_arch.py:59-91) --------------------------------------
  // plan->ops = encode (image -> z, skips stay in the decoder's concat buffers), plan->ops_dec = decode (z -> image).
  void build_latent() {
    const LatCfg& L = ctx->lat;
    const int B = plan->B, depth = L.depth;
    const int s = 1 << depth;
    plan->Hp = plan->H + (s - plan->H % s) % s;
    plan->Wp = plan->W + (s - plan->W % s) % s;
    std::vector<int> hs(depth), ws(depth);
    hs[0] = plan->Hp; ws[0] = plan->Wp;
    for (int i = 1; i < depth; ++i) { hs[i] = hs[i - 1] / 2; ws[i] = ws[i - 1] / 2; }
    plan->lat_h = hs[depth - 1]; plan->lat_w = ws[depth - 1];
    float* la_partial = (float*)dev_alloc(ctx, linattn_partial_floats(B, hs[depth - 1] * ws[depth - 1]) * sizeof(float), &plan->allocs);
    float* la_ctx = (float*)dev_alloc(ctx, (size_t)B * 4096 * sizeof(float), &plan->allocs);
    if (!la_partial || !la_ctx) { ok = false; err = "cudaMalloc failed"; return; }
    const int C0 = L.in_ch, pitch0 = (C0 + 7) / 8 * 8;
    const long long np0 = (long long)B * hs[0] * ws[0];
    T* X0 = alloc(np0 * pitch0);
    T* H0 = alloc(np0 * L.ch);  // h[0] = init_conv output, added back before final_conv
    int in_ch = L.in_ch, Hh = plan->H, Ww = plan->W, Hp = plan->Hp, Wp = plan->Wp;
    irsde_ctx* cx = ctx;
    plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan* p, cudaStream_t st) {
      launch_prep_input<T>(p->cur.x, nullptr, X0, B, in_ch, Hh, Ww, Hp, Wp, pitch0, 0, st);  // reflect pad, no condition
      cx->launches++;
    }});
    conv("init_conv.weight", V{X0, pitch0, C0}, hs[0], ws[0], 3, 1, 1, 1, nullptr, "", 0, nullptr, V{H0, L.ch, L.ch}, L.ch);
    V cur{H0, L.ch, L.ch};
    std::vector<T*> U1(depth), U2(depth);
    char nb[64];
    for (int i = 0; i < depth; ++i) {
      const int di = L.ch * L.mult[i], dout = L.ch * L.mult[i + 1], H = hs[i], W = ws[i];
      const long long npix = (long long)B * H * W;
      U1[i] = alloc(npix * (dout + di));
      U2[i] = alloc(npix * (dout + di));
      snprintf(nb, sizeof nb, "encoder.%d.", i);
      std::string pre = nb;
      V s2 = view(U2[i], dout + di, dout, di), s1 = view(U1[i], dout + di, dout, di);
      resblock(pre + "0.", cur, di, s2, H, W, false);
      if (i == depth - 1) {
        T* ta = tmp(npix * di);
        resblock(pre + "1.", s2, di, V{ta, di, di}, H, W, false);
        attention(pre + "2.", V{ta, di, di}, s1, H, W, false, la_partial, la_ctx);
        release(ta);
        T* xm = alloc(npix * dout);
        conv(pre + "3.weight", s1, H, W, 3, 1, 1, 1, nullptr, "", 0, nullptr, V{xm, dout, dout}, dout);
        cur = V{xm, dout, dout};
      } else {
        resblock(pre + "1.", s2, di, s1, H, W, false);  // Identity attention: the skip is b2's output
        T* xn = alloc((long long)B * hs[i + 1] * ws[i + 1] * dout);
        std::string bn = pre + "3.bias";
        conv(pre + "3.weight", s1, H, W, 4, 2, 1, 1, bn.c_str(), "", 0, nullptr, V{xn, dout, dout}, dout);
        cur = V{xn, dout, dout};
      }
    }
    {  // z = latent_conv(x): fp32 NCHW [B, embed, lat_h, lat_w] straight from the epilogue
      float* dummy = nullptr;
      nchw_H = plan->lat_h; nchw_W = plan->lat_w;
      conv("latent_conv.weight", cur, plan->lat_h, plan->lat_w, 1, 1, 0, 1, nullptr, "", 0, nullptr, V{nullptr, 0, 0}, L.embed, &dummy);
      nchw_H = nchw_W = 0;
    }
    // ----- decode half
    std::vector<OpRec> enc_ops;
    enc_ops.swap(plan->ops);
    const int mid = L.ch * L.mult[depth];
    const long long npl = (long long)B * plan->lat_h * plan->lat_w;
    const int zp = (L.embed + 7) / 8 * 8;
    T* Z = alloc(npl * zp);
    int embed = L.embed, lh = plan->lat_h, lw = plan->lat_w;
    plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan* p, cudaStream_t st) {
      launch_nchw_to_nhwc<T>(p->cur.x, Z, B, embed, lh, lw, zp, st);
      cx->launches++;
    }});
    {
      const int i = depth - 1, di = L.ch * L.mult[i];
      conv("post_latent_conv.weight", V{Z, zp, L.embed}, lh, lw, 1, 1, 0, 1, nullptr, "", 0, nullptr, view(U1[i], mid + di, 0, mid), mid);
    }
    for (int j = 0; j < depth; ++j) {
      const int i = depth - 1 - j, di = L.ch * L.mult[i], dout = L.ch * L.mult[i + 1], H = hs[i], W = ws[i];
      const long long npix = (long long)B * H * W;
      snprintf(nb, sizeof nb, "decoder.%d.", j);
      std::string pre = nb;
      resblock(pre + "0.", V{U1[i], dout + di, dout + di}, dout, view(U2[i], dout + di, 0, dout), H, W, false);
      T* tb = tmp(npix * dout);
      resblock(pre + "1.", V{U2[i], dout + di, dout + di}, dout, V{tb, dout, dout}, H, W, false);
      V xo{tb, dout, dout};
      T* tc = nullptr;
      if (i == depth - 1) {
        tc = tmp(npix * dout);
        attention(pre + "2.", V{tb, dout, dout}, V{tc, dout, dout}, H, W, false, la_partial, la_ctx);
        xo = V{tc, dout, dout};
      }
      if (i != 0) {
        const int dprev_total = L.ch * L.mult[i] + L.ch * L.mult[i - 1];  // concat width of level i-1: dout_{i-1} + di_{i-1}
        std::string bn = pre + "3.1.bias";
        conv(pre + "3.1.weight", xo, H, W, 3, 1, 1, 2, bn.c_str(), "", 0, nullptr, view(U1[i - 1], dprev_total, 0, di), di);
      } else {
        T* xf = tmp(np0 * L.ch);
        conv(pre + "3.weight", xo, H, W, 3, 1, 1, 1, nullptr, "", 0, nullptr, V{xf, L.ch, L.ch}, L.ch);
        T* xs = tmp(np0 * L.ch);
        int chn = L.ch;
        plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
          launch_add<T>(xf, chn, H0, chn, xs, chn, np0, chn, st);   // x + h[0]
          cx->launches++;
        }});
        float* dummy = nullptr;
        conv("final_conv.weight", V{xs, L.ch, L.ch}, hs[0], ws[0], 3, 1, 1, 1, "final_conv.bias", "", 0, nullptr, V{nullptr, 0, 0},
             L.out_ch, &dummy);
        release(xf);
        release(xs);
      }
      release(tb);
      if (tc) release(tc);
    }
    plan->ops_dec.swap(plan->ops);
    plan->ops.swap(enc_ops);
  }

  // ---- ConditionalNAFNet (DenoisingNAFNet_arch.py:87-188) -------------------------------------------------
  float* naf_partial = nullptr;
  float* naf_sca = nullptr;

  void ln_mod(const std::string& gname, const std::string& blk, int off_scale, int off_shift, V in, V out, int H, int W) {
    int C = in.C, B = plan->B;
    long long npix = (long long)B * H * W;
    float* g = fw(gname);
    int base = ctx->ss_off[blk], S = ctx->S, ppi = H * W;
    irsde_ctx* c = ctx;
    plan->ops.push_back(OpRec{CAT_LN, 0.0, [=](Plan* p, cudaStream_t st) {
      LnMod m;
      m.ss = p->cur.ss; m.t_ptr = p->cur.t_ptr; m.S = S; m.off_scale = base + off_scale; m.off_shift = base + off_shift;
      m.img_stride = p->cur.ss_img_stride; m.pix_per_img = ppi;
      launch_layernorm<T>(in.p, in.pitch, g, nullptr, 0, out.p, out.pitch, npix, C, st, &m);
      c->launches++;
    }});
    plan->ops.back().label = gname + " (LN+mod)";
    plan->ops.back().bytes = 2.0 * npix * C * sizeof(T);
  }

  void nafblock(const std::string& pre, V x, V out, int H, int W) {
    const int c = x.C, B = plan->B, N = H * W;
    const long long npix = (long long)B * N;
    irsde_ctx* cx = ctx;
    T* t1 = tmp(npix * c);
    ln_mod(pre + "norm1.g", pre, c, 0, x, V{t1, c, c}, H, W);            // x * (scale_att + 1) + shift_att
    T* t2 = tmp(npix * 2 * c);
    std::string b1 = pre + "conv1.bias";
    conv(pre + "conv1.weight", V{t1, c, c}, H, W, 1, 1, 0, 1, b1.c_str(), "", 0, nullptr, V{t2, 2 * c, 2 * c}, 2 * c);
    release(t1);
    T* g = tmp(npix * c);
    {
      float* w2 = fw(pre + "conv2.weight"); float* bb2 = fw(pre + "conv2.bias");
      float* ws = fw(pre + "sca.1.weight"); float* bs = fw(pre + "sca.1.bias");
      float* partial = naf_partial; float* sca = naf_sca;
      const int nch = dwgate_chunks(H, W);
      plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
        launch_dwgate<T>(t2, 2 * c, w2, bb2, g, c, partial, B, H, W, c, st);
        int nl = 0;
        launch_sca_scale<T>(partial, ws, bs, sca, g, c, B, c, nch, N, &nl, st);
        cx->launches += 1 + nl;
      }});
      plan->ops.back().label = pre + "dw3x3+gate+sca";
      plan->ops.back().bytes = (double)npix * (2 * c + c + 2 * c) * sizeof(T);
    }
    release(t2);
    T* y = tmp(npix * c);
    std::string b3 = pre + "conv3.bias";
    pending_mult = fw(pre + "beta");
    conv(pre + "conv3.weight", V{g, c, c}, H, W, 1, 1, 0, 1, b3.c_str(), "", 0, &x, V{y, c, c}, c);     // y = inp + conv3(.)*beta
    release(g);
    t1 = tmp(npix * c);
    ln_mod(pre + "norm2.g", pre, 3 * c, 2 * c, V{y, c, c}, V{t1, c, c}, H, W);                          // * (scale_ffn+1) + shift_ffn
    t2 = tmp(npix * 2 * c);
    std::string b4 = pre + "conv4.bias";
    conv(pre + "conv4.weight", V{t1, c, c}, H, W, 1, 1, 0, 1, b4.c_str(), "", 0, nullptr, V{t2, 2 * c, 2 * c}, 2 * c);
    release(t1);
    g = tmp(npix * c);
    if (ctx->naf.lens) {  // x = SimpleGate(x) * (cam_scale + 1) + cam_shift   (latent-bokeh/.../DenoisingNAFNet_arch.py:82-83)
      const int coff = ctx->cam_off[pre], cS = ctx->cam_S;
      plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan* p, cudaStream_t st) {
        CamMod m{p->cur.cam, cS, coff, p->cur.cam_img_stride, N};
        launch_simple_gate<T>(t2, 2 * c, g, c, npix, c, st, m, B);
        cx->launches++;
      }});
      plan->ops.back().label = pre + "simple_gate+cam";
    } else {
      plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
        launch_simple_gate<T>(t2, 2 * c, g, c, npix, c, st);
        cx->launches++;
      }});
      plan->ops.back().label = pre + "simple_gate";
    }
    release(t2);
    std::string b5 = pre + "conv5.bias";
    pending_mult = fw(pre + "gamma");
    V vy{y, c, c};
    conv(pre + "conv5.weight", V{g, c, c}, H, W, 1, 1, 0, 1, b5.c_str(), "", 0, &vy, out, c);           // out = y + conv5(.)*gamma
    release(g);
    release(y);
  }

  void build_naf() {
    const NafCfg& n = ctx->naf;
    const int B = plan->B, w = n.width, ic = n.img_channel;
    const int s = 1 << n.n_enc;
    plan->Hp = plan->H + (s - plan->H % s) % s;
    plan->Wp = plan->W + (s - plan->W % s) % s;
    std::vector<int> hs(n.n_enc + 1), ws(n.n_enc + 1);
    hs[0] = plan->Hp; ws[0] = plan->Wp;
    for (int i = 1; i <= n.n_enc; ++i) { hs[i] = hs[i - 1] / 2; ws[i] = ws[i - 1] / 2; }
    size_t pmax = 0, cmax = 0;
    for (int i = 0; i <= n.n_enc; ++i) {
      size_t cc = (size_t)w << i;
      pmax = std::max(pmax, (size_t)B * dwgate_chunks(hs[i], ws[i]) * cc);
      cmax = std::max(cmax, cc);
    }
    naf_partial = (float*)dev_alloc(ctx, pmax * sizeof(float), &plan->allocs);
    naf_sca = (float*)dev_alloc(ctx, (size_t)B * cmax * sizeof(float), &plan->allocs);
    if (!naf_partial || !naf_sca) { ok = false; err = "cudaMalloc failed"; return; }
    const int C0 = 2 * ic, pitch0 = (C0 + 7) / 8 * 8;
    const long long np0 = (long long)B * hs[0] * ws[0];
    T* X0 = alloc(np0 * pitch0);
    int Hh = plan->H, Ww = plan->W, Hp = plan->Hp, Wp = plan->Wp;
    irsde_ctx* cx = ctx;
    plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan* p, cudaStream_t st) {
      launch_prep_input<T>(p->cur.x, p->cur.mu, X0, B, ic, Hh, Ww, Hp, Wp, pitch0, 1, st, 0, 0, 0, 0, 1);  // zero pad
      cx->launches++;
    }});
    T* xin = alloc(np0 * w);
    conv("intro.weight", V{X0, pitch0, C0}, hs[0], ws[0], 3, 1, 1, 1, "intro.bias", "", 0, nullptr, V{xin, w, w}, w);
    V cur{xin, w, w};
    std::vector<V> encs;
    char nb[64];
    for (int i = 0; i < n.n_enc; ++i) {
      const int c = w << i;
      const long long npix = (long long)B * hs[i] * ws[i];
      for (int j = 0; j < n.enc[i]; ++j) {
        T* o = alloc(npix * c);
        snprintf(nb, sizeof nb, "encoders.%d.%d.", i, j);
        nafblock(nb, cur, V{o, c, c}, hs[i], ws[i]);
        cur = V{o, c, c};
      }
      encs.push_back(cur);
      T* d = alloc((long long)B * hs[i + 1] * ws[i + 1] * 2 * c);
      snprintf(nb, sizeof nb, "downs.%d.", i);
      std::string wn = std::string(nb) + "weight", bn = std::string(nb) + "bias";
      conv(wn, cur, hs[i], ws[i], 2, 2, 0, 1, bn.c_str(), "", 0, nullptr, V{d, 2 * c, 2 * c}, 2 * c);
      cur = V{d, 2 * c, 2 * c};
    }
    {
      const int c = w << n.n_enc;
      const long long npix = (long long)B * hs[n.n_enc] * ws[n.n_enc];
      for (int j = 0; j < n.middle; ++j) {
        T* o = alloc(npix * c);
        snprintf(nb, sizeof nb, "middle_blks.%d.", j);
        nafblock(nb, cur, V{o, c, c}, hs[n.n_enc], ws[n.n_enc]);
        cur = V{o, c, c};
      }
    }
    for (int i = 0; i < n.n_dec; ++i) {
      const int l = n.n_enc - 1 - i;           // level after upsampling
      const int chan = w << (l + 1), q = chan / 2;
      const int hl = hs[l + 1], wl = ws[l + 1];
      const long long np_lo = (long long)B * hl * wl, np_hi = (long long)B * hs[l] * ws[l];
      T* u = tmp(np_lo * 2 * chan);
      snprintf(nb, sizeof nb, "ups.%d.0.weight", i);
      conv(nb, cur, hl, wl, 1, 1, 0, 1, nullptr, "", 0, nullptr, V{u, 2 * chan, 2 * chan}, 2 * chan);
      T* v = alloc(np_hi * q);
      V skip = encs[l];
      plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
        launch_pixel_shuffle_add<T>(u, 2 * chan, skip.p, skip.pitch, v, q, B, hl, wl, q, st);
        cx->launches++;
      }});
      plan->ops.back().label = std::string(nb) + " pixel_shuffle+skip";
      release(u);
      cur = V{v, q, q};
      for (int j = 0; j < n.dec[i]; ++j) {
        T* o = alloc(np_hi * q);
        snprintf(nb, sizeof nb, "decoders.%d.%d.", i, j);
        nafblock(nb, cur, V{o, q, q}, hs[l], ws[l]);
        cur = V{o, q, q};
      }
    }
    if (n.latent) {  // latent variant: ending(x + encs[0]) with encs[0] = intro output
      T* e = alloc(np0 * w);
      V a = cur;
      plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan*, cudaStream_t st) {
        launch_add<T>(a.p, a.pitch, xin, w, e, w, np0, w, st);
        cx->launches++;
      }});
      cur = V{e, w, w};
    }
    float* dummy = nullptr;
    conv("ending.weight", cur, hs[0], ws[0], 3, 1, 1, 1, "ending.bias", "", 0, nullptr, V{nullptr, 0, 0}, ic, &dummy);
  }

  void build() {
    const irsde_config& c = ctx->cfg;
    int B = plan->B, nf = c.nf, depth = c.depth;
    const std::vector<int>& D = ctx->udim;
    int s = 1 << depth;
    plan->Hp = plan->H + (s - plan->H % s) % s;
    plan->Wp = plan->W + (s - plan->W % s) % s;
    std::vector<int> hs(depth), ws(depth);
    hs[0] = plan->Hp; ws[0] = plan->Wp;
    for (int i = 1; i < depth; ++i) { hs[i] = hs[i - 1] / 2; ws[i] = ws[i - 1] / 2; }
    bool cond = c.variant == IRSDE_NET_CONDITIONAL;
    int C0 = cond ? 2 * c.in_nc : c.in_nc;
    int pitch0 = (C0 + 7) / 8 * 8;
    long long np0 = (long long)B * hs[0] * ws[0];
    // linear-attention scratch sized for the largest level
    float* la_partial = (float*)dev_alloc(ctx, linattn_partial_floats(B, hs[0] * ws[0]) * sizeof(float), &plan->allocs);
    float* la_ctx = (float*)dev_alloc(ctx, (size_t)B * 4096 * sizeof(float), &plan->allocs);
    if (!la_partial || !la_ctx) { ok = false; err = "cudaMalloc failed"; return; }

    int in_nc = c.in_nc, Hh = plan->H, Ww = plan->W, Hp = plan->Hp, Wp = plan->Wp;
    stem_padded = std::is_same<T, bf16>::value && ctx->use_tc && pitch0 == 8 && nf % 8 == 0;
    long long x0_elems = stem_padded ? (long long)B * (Hp + 6) * (Wp + 8) * 8 + 64 : np0 * pitch0;
    T* X0 = alloc(x0_elems);
    if (X0 && stem_padded) cudaMemset(X0, 0, (size_t)x0_elems * sizeof(T));  // borders stay zero forever
    T* F = alloc(np0 * 2 * nf);
    irsde_ctx* cx = ctx;
    bool sp = stem_padded;
    plan->ops.push_back(OpRec{CAT_MISC, 0.0, [=](Plan* p, cudaStream_t st) {
      if (sp) launch_prep_input<T>(p->cur.x, p->cur.mu, X0, B, in_nc, Hh, Ww, Hp, Wp, pitch0, cond ? 1 : 0, st, 3, 3, Wp + 8, Hp + 6);
      else launch_prep_input<T>(p->cur.x, p->cur.mu, X0, B, in_nc, Hh, Ww, Hp, Wp, pitch0, cond ? 1 : 0, st);
      cx->launches++;
    }});
    conv("init_conv.weight", V{X0, pitch0, C0}, hs[0], ws[0], 7, 1, 3, 1, nullptr, "", 0, nullptr, view(F, 2 * nf, nf, nf), nf);
    V cur = view(F, 2 * nf, nf, nf);
    std::vector<T*> U1(depth), U2(depth);
    char nb[64];
    for (int i = 0; i < depth; ++i) {
      int di = D[i], dout = D[i + 1], H = hs[i], W = ws[i];
      long long npix = (long long)B * H * W;
      U1[i] = alloc(npix * (dout + di));
      U2[i] = alloc(npix * (dout + di));
      snprintf(nb, sizeof nb, "downs.%d.", i);
      std::string pre = nb;
      V s2 = view(U2[i], dout + di, dout, di), s1 = view(U1[i], dout + di, dout, di);
      resblock(pre + "0.", cur, di, s2, H, W);
      T* ta = tmp(npix * di);
      resblock(pre + "1.", s2, di, V{ta, di, di}, H, W);
      attention(pre + "2.", V{ta, di, di}, s1, H, W, false, la_partial, la_ctx);
      release(ta);
      if (i != depth - 1) {
        T* xn = alloc((long long)B * hs[i + 1] * ws[i + 1] * dout);
        std::string bn = pre + "3.bias";
        conv(pre + "3.weight", s1, H, W, 4, 2, 1, 1, bn.c_str(), "", 0, nullptr, V{xn, dout, dout}, dout);
        cur = V{xn, dout, dout};
      } else {
        T* xn = alloc(npix * dout);
        conv(pre + "3.weight", s1, H, W, 3, 1, 1, 1, nullptr, "", 0, nullptr, V{xn, dout, dout}, dout);
        cur = V{xn, dout, dout};
      }
    }
    {
      int i = depth - 1, di = D[i], mid = D[depth], H = hs[i], W = ws[i];
      long long npix = (long long)B * H * W;
      T* m1 = tmp(npix * mid);
      T* m2 = tmp(npix * mid);
      resblock("mid_block1.", cur, mid, V{m1, mid, mid}, H, W);
      attention("mid_attn.", V{m1, mid, mid}, V{m2, mid, mid}, H, W, c.variant == IRSDE_NET_DENOISING, la_partial, la_ctx);
      resblock("mid_block2.", V{m2, mid, mid}, mid, view(U1[i], mid + di, 0, mid), H, W);
      release(m1);
      release(m2);
    }
    for (int j = 0; j < depth; ++j) {
      int i = depth - 1 - j, di = D[i], dout = D[i + 1], H = hs[i], W = ws[i];
      long long npix = (long long)B * H * W;
      snprintf(nb, sizeof nb, "ups.%d.", j);
      std::string pre = nb;
      resblock(pre + "0.", V{U1[i], dout + di, dout + di}, dout, view(U2[i], dout + di, 0, dout), H, W);
      T* tb = tmp(npix * dout);
      resblock(pre + "1.", V{U2[i], dout + di, dout + di}, dout, V{tb, dout, dout}, H, W);
      T* tc = tmp(npix * dout);
      attention(pre + "2.", V{tb, dout, dout}, V{tc, dout, dout}, H, W, false, la_partial, la_ctx);
      release(tb);
      if (i != 0) {
        int dprev = D[i];  // == dout of level i-1
        std::string bn = pre + "3.1.bias";
        conv(pre + "3.1.weight", V{tc, dout, dout}, H, W, 3, 1, 1, 2, bn.c_str(), "", 0, nullptr,
             view(U1[i - 1], dprev + D[i - 1], 0, dprev), di);
      } else {
        conv(pre + "3.weight", V{tc, dout, dout}, H, W, 3, 1, 1, 1, nullptr, "", 0, nullptr, view(F, 2 * nf, 0, nf), di);
      }
      release(tc);
    }
    T* G = tmp(np0 * nf);
    resblock("final_res_block.", V{F, 2 * nf, 2 * nf}, nf, V{G, nf, nf}, hs[0], ws[0]);
    float* dummy = nullptr;
    conv("final_conv.weight", V{G, nf, nf}, hs[0], ws[0], 3, 1, 1, 1, "final_conv.bias", "", 0, nullptr, V{nullptr, 0, 0},
         c.out_nc, &dummy);
  }
};

void free_plan(irsde_ctx* ctx, Plan* p) {
  for (int m = 0; m < IRSDE_NUM_MODES; ++m)
    if (p->graph[m]) cudaGraphExecDestroy(p->graph[m]);
  for (auto* d : p->tc_descs) tc_conv_destroy(d);
  for (void* q : p->allocs) cudaFree(q);  // cudaFree waits for in-flight work that may still use the buffer
  ctx->dev_bytes -= p->bytes;
  ctx->plan_bytes -= p->bytes;
  delete p;
}

// The plan cache is bounded: every (B,H,W) plan owns its activation workspace, TMA descriptors and step graphs, so a
// loop over a dataset of variable-size images (test.py runs batch 1 at native size) would otherwise grow without limit.
// Least-recently-used plans are dropped while the cache holds more than IRSDE_PLAN_CACHE_MB (default 24576) or
// IRSDE_PLAN_CACHE_MAX (default 8) entries; `keep` is never evicted.
void evict_plans(irsde_ctx* ctx, Plan* keep, bool all) {
  static long long budget = -1, maxn = -1;
  if (budget < 0) {
    const char* e = getenv("IRSDE_PLAN_CACHE_MB");
    budget = (e && atoll(e) > 0 ? atoll(e) : 24576LL) << 20;
    e = getenv("IRSDE_PLAN_CACHE_MAX");
    maxn = e && atoll(e) > 0 ? atoll(e) : 8;
  }
  for (;;) {
    const bool over = all || ctx->plan_bytes > budget || (long long)ctx->plans.size() > maxn;
    if (!over) return;
    auto victim = ctx->plans.end();
    for (auto it = ctx->plans.begin(); it != ctx->plans.end(); ++it)
      if (it->second != keep && (victim == ctx->plans.end() || it->second->last_use < victim->second->last_use)) victim = it;
    if (victim == ctx->plans.end()) return;
    free_plan(ctx, victim->second);
    ctx->plans.erase(victim);
  }
}

int build_plan(irsde_ctx* ctx, int B, int H, int W, Plan** out) {
  auto key = std::make_tuple(B, H, W);
  auto it = ctx->plans.find(key);
  if (it != ctx->plans.end()) { it->second->last_use = ++ctx->use_clock; *out = it->second; return IRSDE_OK; }
  if (B <= 0 || H <= 0 || W <= 0) return fail(ctx, IRSDE_ERR_INVALID, "bad image shape");
  const long long bytes_before = ctx->dev_bytes;
  int s = 1 << ctx->cfg.depth;
  // reflect pad needs pad < size (F.pad 'reflect' raises otherwise, DenoisingUNet_arch.py:82)
  if (!ctx->naf.on && ((s - H % s) % s >= H || (s - W % s) % s >= W))
    return fail(ctx, IRSDE_ERR_INVALID, "image too small for reflect padding");
  Plan* p = new Plan();
  p->B = B; p->H = H; p->W = W;
  std::string err;
  bool ok;
  if (ctx->cfg.precision != IRSDE_PREC_BF16) {
    Builder<float> b{ctx, p};
    if (ctx->lat.on) b.build_latent(); else if (ctx->naf.on) b.build_naf(); else b.build();
    ok = b.ok; err = b.err;
  } else {
    Builder<bf16> b{ctx, p};
    if (ctx->lat.on) b.build_latent(); else if (ctx->naf.on) b.build_naf(); else b.build();
    ok = b.ok; err = b.err;
  }
  long long n = (long long)B * ctx->cfg.in_nc * H * W;
  long long no = (long long)B * ctx->cfg.out_nc * H * W;
  p->x_state = (float*)dev_alloc(ctx, n * 4, &p->allocs);
  p->mu_buf = (float*)dev_alloc(ctx, n * 4, &p->allocs);
  p->eps_buf = (float*)dev_alloc(ctx, no * 4, &p->allocs);
  p->d_step = (StepState*)dev_alloc(ctx, sizeof(StepState), &p->allocs);
  p->d_zero = (int*)dev_alloc(ctx, sizeof(int), &p->allocs);
  int td = ctx->cfg.nf * 4;
  p->fwd_times = (float*)dev_alloc(ctx, (size_t)B * 4, &p->allocs);
  p->fwd_temb = (float*)dev_alloc(ctx, (size_t)B * td * 4, &p->allocs);
  p->fwd_table = (float*)dev_alloc(ctx, (size_t)B * ctx->S * 4, &p->allocs);
  if (!ok || !p->x_state || !p->mu_buf || !p->eps_buf || !p->d_step || !p->d_zero || !p->fwd_table) {
    for (auto* d : p->tc_descs) tc_conv_destroy(d);
    for (void* q : p->allocs) cudaFree(q);
    ctx->dev_bytes = bytes_before;
    delete p;
    return fail(ctx, IRSDE_ERR_CUDA, err.empty() ? "plan allocation failed" : err);
  }
  cudaMemset(p->d_zero, 0, sizeof(int));
  p->bytes = ctx->dev_bytes - bytes_before;
  p->last_use = ++ctx->use_clock;
  ctx->plan_bytes += p->bytes;
  ctx->plans[key] = p;
  evict_plans(ctx, p, false);
  *out = p;
  return IRSDE_OK;
}

void run_ops(irsde_ctx* ctx, Plan* p, std::vector<OpRec>& ops, cudaStream_t st) {
  if (!ctx->prof) {
    for (auto& op : ops) op.fn(p, st);
    return;
  }
  for (auto& op : ops) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, st);
    op.fn(p, st);
    cudaEventRecord(e1, st);
    ctx->prof_events.push_back({op.cat, op.flops, e0, e1, &op});
  }
}
void run_forward(irsde_ctx* ctx, Plan* p, cudaStream_t st) { run_ops(ctx, p, p->ops, st); }

// default per-timestep scalars in fp32, same op order as the reference's 0-dim tensor math
void fill_default_coeffs(irsde_ctx* c, int mode, std::vector<float>& tab) {
  int T = c->T;
  tab.assign((size_t)(T + 1) * IRSDE_NUM_COEF, 0.f);
  float dt = c->dt, sqdt = (float)sqrt((double)dt);
  for (int t = 1; t <= T; ++t) {
    float* r = &tab[(size_t)t * IRSDE_NUM_COEF];
    float th = c->thetas[t], sg = c->sigmas[t], cs = c->cumsum[t], cs1 = c->cumsum[t - 1], sb = c->sbars[t];
    float sg2 = sg * sg;
    switch (mode) {
      case IRSDE_MODE_SDE: r[0] = th; r[1] = sg2; r[2] = sb; r[3] = dt; r[4] = sg; r[5] = sqdt; break;
      case IRSDE_MODE_ODE: r[0] = th; r[1] = 0.5f * sg2; r[2] = sb; r[3] = dt; break;
      case IRSDE_MODE_POSTERIOR: {
        float A0 = expf(cs * dt);
        float A = expf(-th * dt), Bv = expf(-cs * dt), Cv = expf(-cs1 * dt);
        float term1 = A * (1.f - Cv * Cv) / (1.f - Bv * Bv);
        float term2 = Cv * (1.f - A * A) / (1.f - Bv * Bv);
        float A2 = expf(-2.f * th * dt), B2 = expf(-2.f * cs * dt), C2 = expf(-2.f * cs1 * dt);
        float var = (1.f - A2) * (1.f - C2) / (1.f - B2);
        float mn = 1e-20f * dt;
        float lv = logf(var < mn ? mn : var);
        float sd = expf(0.5f * lv) * c->max_sigma;
        r[0] = A0; r[1] = sb; r[2] = term1; r[3] = term2; r[4] = sd;
        break;
      }
      case IRSDE_MODE_DSDE_SDE: {
        float A = expf(-2.f * cs * dt);
        r[0] = -0.5f * sg2 * (1.f + A); r[1] = sb; r[2] = dt; r[3] = sg; r[4] = sqdt;
        break;
      }
      default: {
        float A = expf(-2.f * cs * dt);
        r[0] = -0.5f * sg2 * A; r[1] = sb; r[2] = dt;
        break;
      }
    }
  }
}

int upload_coeffs(irsde_ctx* ctx, int mode, const float* tab, int T) {
  size_t bytes = (size_t)(T + 1) * IRSDE_NUM_COEF * sizeof(float);
  if (ctx->coef_dev[mode]) {
    // keep pointer stable across re-uploads of the same T (captured graphs reference it)
  } else {
    ctx->coef_dev[mode] = (float*)dev_alloc(ctx, (size_t)(4096 + 1) * IRSDE_NUM_COEF * sizeof(float), &ctx->allocs);
    if (!ctx->coef_dev[mode]) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc coef failed");
  }
  if (T > 4096) return fail(ctx, IRSDE_ERR_UNSUPPORTED, "T > 4096 not supported");
  CUDA_TRY(ctx, cudaDeviceSynchronize());  // chains in flight on non-blocking streams still read the old table
  CUDA_TRY(ctx, cudaMemcpy(ctx->coef_dev[mode], tab, bytes, cudaMemcpyHostToDevice));
  return IRSDE_OK;
}

// times[rows] -> table[rows][S] for either network family
void time_rows(irsde_ctx* ctx, const float* times, int rows, float* temb_ws, float* table, cudaStream_t st) {
  if (ctx->naf.on) {
    const std::string a = ctx->naf.lens ? "time_mlp.0." : "time_mlp.1.", b = ctx->naf.lens ? "time_mlp.2." : "time_mlp.3.";
    launch_naf_time_gate(times, rows, ctx->naf.width, ctx->raw[a + "weight"].dev, ctx->raw[a + "bias"].dev,
                         ctx->raw[b + "weight"].dev, ctx->raw[b + "bias"].dev, temb_ws, st);
    launch_time_rows(temb_ws, rows, 2 * ctx->naf.width, ctx->wall, ctx->ball, ctx->S, table, st);
  } else {
    launch_time_table(times, rows, ctx->cfg.nf, ctx->raw["time_mlp.1.weight"].dev, ctx->raw["time_mlp.1.bias"].dev,
                      ctx->raw["time_mlp.3.weight"].dev, ctx->raw["time_mlp.3.bias"].dev, ctx->wall, ctx->ball, ctx->S, temb_ws,
                      table, st);
  }
  ctx->launches += 2;
}

int ensure_chain_table(irsde_ctx* ctx, Plan* p, int T, cudaStream_t st) {
  int rows = T + 1;
  if (rows > p->chain_cap) {
    int cap = rows < 128 ? 128 : rows;
    int td = ctx->cfg.nf * 4;
    p->chain_times = (float*)dev_alloc(ctx, (size_t)cap * 4, &p->allocs);
    p->chain_temb = (float*)dev_alloc(ctx, (size_t)cap * td * 4, &p->allocs);
    p->chain_table = (float*)dev_alloc(ctx, (size_t)cap * ctx->S * 4, &p->allocs);
    if (!p->chain_times || !p->chain_temb || !p->chain_table) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc chain table failed");
    { const long long add = ((long long)cap * 4 + (long long)cap * td * 4 + (long long)cap * ctx->S * 4); p->bytes += add; ctx->plan_bytes += add; }
    std::vector<float> tv(cap);
    for (int i = 0; i < cap; ++i) tv[i] = (float)i;
    CUDA_TRY(ctx, cudaMemcpy(p->chain_times, tv.data(), (size_t)cap * 4, cudaMemcpyHostToDevice));
    p->chain_cap = cap;
    for (int m = 0; m < IRSDE_NUM_MODES; ++m)
      if (p->graph[m]) { cudaGraphExecDestroy(p->graph[m]); p->graph[m] = nullptr; }
  }
  time_rows(ctx, p->chain_times, rows, p->chain_temb, p->chain_table, st);
  return IRSDE_OK;
}

// lens network: lens_host [lens_n][3] -> cam_table [lens_n][cam_S].  cam_mlp is the time MLP kernel with k = 3 scalars per
// row; every block's cam_mlp.1 is one concatenated rows pass (cam_wall), as the time table's mlp.1 are.  Independent of t.
int compute_cam(irsde_ctx* ctx, cudaStream_t st) {
  const int n = ctx->lens_n, w = ctx->naf.width;
  CUDA_TRY(ctx, cudaMemcpy(ctx->lens_dev, ctx->lens_host.data(), (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice));
  launch_naf_time_gate_k(ctx->lens_dev, n, 3, w, ctx->raw["cam_mlp.0.weight"].dev, ctx->raw["cam_mlp.0.bias"].dev,
                       ctx->raw["cam_mlp.2.weight"].dev, ctx->raw["cam_mlp.2.bias"].dev, ctx->cam_gate, st);
  launch_time_rows(ctx->cam_gate, n, 2 * w, ctx->cam_wall, ctx->cam_ball, ctx->cam_S, ctx->cam_table, st);
  ctx->launches += 2;
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

// run-time state of a lens network for a batch of B: the camera rows must be set, one shared or one per image
int lens_ready(irsde_ctx* ctx, int B, Plan* p) {
  p->cur.cam = nullptr;
  p->cur.cam_img_stride = 0;
  if (!ctx->naf.lens) return IRSDE_OK;
  if (ctx->lens_n == 0) return fail(ctx, IRSDE_ERR_STATE, "lens network: irsde_set_lens must be called first");
  if (ctx->lens_n != 1 && ctx->lens_n != B) return fail(ctx, IRSDE_ERR_INVALID, "lens count must be 1 or the batch size");
  p->cur.cam = ctx->cam_table;
  p->cur.cam_img_stride = ctx->lens_n > 1 ? 1 : 0;
  return IRSDE_OK;
}

}  // namespace

// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

const char* irsde_version(void) { return "irsde_b200 0.1 sm_100a"; }

const char* irsde_last_error(const irsde_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

int irsde_create(const irsde_config* cfg, irsde_ctx** out) {
  if (!cfg || !out) return fail(nullptr, IRSDE_ERR_INVALID, "null argument");
  if (cfg->nf < 4 || cfg->nf % 2 || cfg->depth < 1 || cfg->depth > 6 || cfg->in_nc < 1 || cfg->out_nc < 1)
    return fail(nullptr, IRSDE_ERR_INVALID, "bad network configuration");
  if (cfg->variant != IRSDE_NET_CONDITIONAL && cfg->variant != IRSDE_NET_DENOISING)
    return fail(nullptr, IRSDE_ERR_INVALID, "bad variant");
  if (cfg->precision != IRSDE_PREC_FP32 && cfg->precision != IRSDE_PREC_BF16 && cfg->precision != IRSDE_PREC_FP32X3)
    return fail(nullptr, IRSDE_ERR_INVALID, "bad precision");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) return fail(nullptr, IRSDE_ERR_CUDA, "no CUDA device available (this library has no CPU path)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, IRSDE_ERR_INVALID, "bad device ordinal");
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, cfg->device);
  if (prop.major != 10) return fail(nullptr, IRSDE_ERR_UNSUPPORTED, "irsde_b200 is built for sm_100a (B200) only");
  irsde_ctx* c = new irsde_ctx();
  c->cfg = *cfg;
  if (cudaSetDevice(cfg->device) != cudaSuccess) { delete c; return fail(nullptr, IRSDE_ERR_CUDA, "cudaSetDevice failed"); }
  std::string terr;
  c->tc_ok = tc_init(&terr);
  if (cfg->precision != IRSDE_PREC_FP32 && !c->tc_ok) {
    delete c;
    return fail(nullptr, IRSDE_ERR_CUDA, "tensor-core engine init failed: " + terr);
  }
  c->use_tc = cfg->precision == IRSDE_PREC_BF16 && !(cfg->flags & IRSDE_FLAG_FORCE_SIMT);
  c->use_tc3 = cfg->precision == IRSDE_PREC_FP32X3 && !(cfg->flags & IRSDE_FLAG_FORCE_SIMT);
  for (int i = 0; i <= cfg->depth; ++i) c->udim.push_back(cfg->nf * (1 << i));
  *out = c;
  return IRSDE_OK;
}

int irsde_create_ch_mult(const irsde_config* cfg, const int32_t* ch_mult, int32_t n_levels, irsde_ctx** out) {
  if (!cfg || !ch_mult || !out || n_levels < 1 || n_levels > 6) return fail(nullptr, IRSDE_ERR_INVALID, "bad ch_mult");
  for (int i = 0; i < n_levels; ++i)
    if (ch_mult[i] < 1 || (long long)ch_mult[i] * cfg->nf > 65536) return fail(nullptr, IRSDE_ERR_INVALID, "bad ch_mult entry");
  irsde_config c2 = *cfg;
  c2.depth = n_levels;
  int rc = irsde_create(&c2, out);
  if (rc) return rc;
  (*out)->udim.assign(1, cfg->nf);
  for (int i = 0; i < n_levels; ++i) (*out)->udim.push_back(cfg->nf * ch_mult[i]);
  return IRSDE_OK;
}

int irsde_create_latent_unet(const irsde_latent_unet_config* lcfg, irsde_ctx** out) {
  if (!lcfg || !out) return fail(nullptr, IRSDE_ERR_INVALID, "null argument");
  if (lcfg->ch < 1 || lcfg->in_ch < 1 || lcfg->out_ch < 1 || lcfg->n_levels < 1 || lcfg->n_levels > 8 || lcfg->embed_dim < 1)
    return fail(nullptr, IRSDE_ERR_INVALID, "bad latent UNet configuration");
  irsde_config cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.in_nc = lcfg->in_ch; cfg.out_nc = lcfg->out_ch; cfg.nf = 8; cfg.depth = lcfg->n_levels;
  cfg.variant = IRSDE_NET_CONDITIONAL; cfg.precision = lcfg->precision; cfg.device = lcfg->device; cfg.flags = lcfg->flags;
  int rc = irsde_create(&cfg, out);
  if (rc) return rc;
  irsde_ctx* c = *out;
  c->lat.on = true;
  c->lat.in_ch = lcfg->in_ch; c->lat.out_ch = lcfg->out_ch; c->lat.ch = lcfg->ch; c->lat.depth = lcfg->n_levels;
  c->lat.embed = lcfg->embed_dim;
  c->lat.mult[0] = 1;
  for (int i = 0; i < lcfg->n_levels; ++i) c->lat.mult[i + 1] = lcfg->ch_mult[i];
  return IRSDE_OK;
}

static int latent_run(irsde_ctx* ctx, bool decode, const float* in, float* out, int32_t B, int32_t H, int32_t W, void* stream) {
  if (!ctx || !in || !out) return fail(ctx, IRSDE_ERR_INVALID, "null argument");
  if (!ctx->lat.on) return fail(ctx, IRSDE_ERR_STATE, "not a latent UNet context");
  if (!ctx->finalized) return fail(ctx, IRSDE_ERR_STATE, "weights not finalized");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Plan* p;
  auto key = std::make_tuple(B, H, W);
  bool existed = ctx->plans.find(key) != ctx->plans.end();
  if (decode && !existed) return fail(ctx, IRSDE_ERR_STATE, "decode needs a preceding encode of the same shape (skip features)");
  int rc = build_plan(ctx, B, H, W, &p);
  if (rc) return rc;
  p->cur.x = in; p->cur.mu = nullptr; p->cur.out = out;
  p->cur.ss = nullptr; p->cur.t_ptr = p->d_zero; p->cur.ss_img_stride = 0;
  run_ops(ctx, p, decode ? p->ops_dec : p->ops, st);
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

int irsde_latent_encode(irsde_ctx* ctx, const float* x, float* z, int32_t B, int32_t H, int32_t W, void* stream) {
  return latent_run(ctx, false, x, z, B, H, W, stream);
}
int irsde_latent_decode(irsde_ctx* ctx, const float* z, float* out, int32_t B, int32_t H, int32_t W, void* stream) {
  return latent_run(ctx, true, z, out, B, H, W, stream);
}
int irsde_latent_shape(irsde_ctx* ctx, int32_t H, int32_t W, int32_t* lat_h, int32_t* lat_w) {
  if (!ctx || !ctx->lat.on || !lat_h || !lat_w) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  const int s = 1 << ctx->lat.depth;
  const int Hp = H + (s - H % s) % s, Wp = W + (s - W % s) % s;
  *lat_h = Hp >> (ctx->lat.depth - 1);
  *lat_w = Wp >> (ctx->lat.depth - 1);
  return IRSDE_OK;
}

int irsde_create_nafnet(const irsde_nafnet_config* ncfg, irsde_ctx** out) {
  if (!ncfg || !out) return fail(nullptr, IRSDE_ERR_INVALID, "null argument");
  if (ncfg->width < 4 || ncfg->width % 2 || ncfg->img_channel < 1 || ncfg->n_levels < 0 || ncfg->n_levels > 8 ||
      ncfg->middle_blk_num < 0)
    return fail(nullptr, IRSDE_ERR_INVALID, "bad NAFNet configuration");
  irsde_config cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.in_nc = cfg.out_nc = ncfg->img_channel;
  cfg.nf = ncfg->width;
  cfg.depth = ncfg->n_levels > 0 ? ncfg->n_levels : 1;
  cfg.variant = IRSDE_NET_CONDITIONAL;
  cfg.precision = ncfg->precision;
  cfg.device = ncfg->device;
  cfg.flags = ncfg->flags;
  int rc = irsde_create(&cfg, out);
  if (rc) return rc;
  irsde_ctx* c = *out;
  c->cfg.depth = ncfg->n_levels;
  c->naf.on = true;
  c->naf.img_channel = ncfg->img_channel;
  c->naf.width = ncfg->width;
  c->naf.middle = ncfg->middle_blk_num;
  c->naf.n_enc = c->naf.n_dec = ncfg->n_levels;
  for (int i = 0; i < ncfg->n_levels; ++i) { c->naf.enc[i] = ncfg->enc_blk_nums[i]; c->naf.dec[i] = ncfg->dec_blk_nums[i]; }
  c->naf.latent = ncfg->latent != 0;
  return IRSDE_OK;
}

int irsde_create_nafnet_lens(const irsde_nafnet_config* ncfg, irsde_ctx** out) {
  if (ncfg && ncfg->latent) return fail(nullptr, IRSDE_ERR_INVALID, "the lens network ends in a plain ending(x): latent must be 0");
  int rc = irsde_create_nafnet(ncfg, out);
  if (rc) return rc;
  irsde_ctx* c = *out;
  c->naf.lens = true;
  int S = 0;
  for (auto& b : naf_blocks(c->naf)) { c->cam_off[b.pre] = S; S += 2 * b.c; }
  c->cam_S = S;
  return IRSDE_OK;
}

int irsde_set_lens(irsde_ctx* ctx, const float* lens, int32_t n, void* stream) {
  if (!ctx || !lens) return fail(ctx, IRSDE_ERR_INVALID, "null argument");
  if (!ctx->naf.on || !ctx->naf.lens) return fail(ctx, IRSDE_ERR_INVALID, "irsde_set_lens: not a lens network context");
  if (n < 1) return fail(ctx, IRSDE_ERR_INVALID, "irsde_set_lens: n must be >= 1");
  cudaSetDevice(ctx->cfg.device);
  std::vector<float> v(lens, lens + (size_t)n * 3);
  if (n == ctx->lens_n && v == ctx->lens_host) return IRSDE_OK;  // the table already holds these rows
  // captured step graphs and chains in flight on any stream read the table: drain before it is re-written or re-allocated
  CUDA_TRY(ctx, cudaDeviceSynchronize());
  if (n > ctx->lens_cap) {
    for (float* q : {ctx->cam_table, ctx->cam_gate, ctx->lens_dev}) {
      if (!q) continue;
      auto it = std::find(ctx->allocs.begin(), ctx->allocs.end(), (void*)q);
      if (it != ctx->allocs.end()) ctx->allocs.erase(it);
      cudaFree(q);
    }
    const int cap = n < 16 ? 16 : n;
    ctx->dev_bytes -= (long long)ctx->lens_cap * (ctx->cam_S + 2 * ctx->naf.width + 3) * 4;
    ctx->cam_table = (float*)dev_alloc(ctx, (size_t)cap * ctx->cam_S * 4, &ctx->allocs);
    ctx->cam_gate = (float*)dev_alloc(ctx, (size_t)cap * 2 * ctx->naf.width * 4, &ctx->allocs);
    ctx->lens_dev = (float*)dev_alloc(ctx, (size_t)cap * 3 * 4, &ctx->allocs);
    ctx->lens_cap = cap;
    if (!ctx->cam_table || !ctx->cam_gate || !ctx->lens_dev) {
      ctx->lens_cap = 0; ctx->lens_n = 0; ctx->lens_host.clear();
      return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc camera table failed");
    }
  }
  ctx->lens_host.swap(v);
  ctx->lens_n = n;
  return ctx->finalized ? compute_cam(ctx, (cudaStream_t)stream) : IRSDE_OK;  // else irsde_finalize_weights computes it
}

// ---- NCCL behind the C ABI (SURVEY 8 b): dlopen()ed on first use so that single-GPU users keep a library without
// an NCCL dependency.  Only the two collectives of the path: one weight broadcast, one gather of x0. ----------------
struct NcclId { char internal[128]; };  // ncclUniqueId (NCCL_UNIQUE_ID_BYTES = 128), passed by value like the original
namespace {
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
}  // namespace
namespace {
NcclApi g_nccl;
const int kNcclFloat = 7;  // ncclFloat32
bool nccl_load(std::string* err) {
  if (g_nccl.lib) return true;
  const char* names[] = {getenv("IRSDE_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names)
    if (n && n[0] && (h = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
  if (!h) { *err = "libnccl.so.2 not found (set IRSDE_NCCL_LIB)"; return false; }
  NcclApi a;
  a.lib = h;
  a.GetUniqueId = (int (*)(void*))dlsym(h, "ncclGetUniqueId");
  a.CommInitRank = (int (*)(void**, int, NcclId, int))dlsym(h, "ncclCommInitRank");
  a.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
  a.Broadcast = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclBroadcast");
  a.GroupStart = (int (*)())dlsym(h, "ncclGroupStart");
  a.GroupEnd = (int (*)())dlsym(h, "ncclGroupEnd");
  a.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
  if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.Broadcast || !a.GroupStart || !a.GroupEnd) { *err = "incomplete NCCL library"; return false; }
  g_nccl = a;
  return true;
}
int nccl_fail(irsde_ctx* ctx, const char* what, int rc) {
  return fail(ctx, IRSDE_ERR_CUDA, std::string(what) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "NCCL error"));
}
}  // namespace

int irsde_comm_unique_id(void* id128) {
  std::string err;
  if (!id128) return fail(nullptr, IRSDE_ERR_INVALID, "null id buffer");
  if (!nccl_load(&err)) return fail(nullptr, IRSDE_ERR_UNSUPPORTED, err);
  int rc = g_nccl.GetUniqueId(id128);
  return rc ? nccl_fail(nullptr, "ncclGetUniqueId", rc) : IRSDE_OK;
}

int irsde_comm_init(irsde_ctx* ctx, const void* id128, int32_t rank, int32_t nranks) {
  if (!ctx || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  if (ctx->nccl_comm) return fail(ctx, IRSDE_ERR_STATE, "communicator already initialised");
  std::string err;
  if (!nccl_load(&err)) return fail(ctx, IRSDE_ERR_UNSUPPORTED, err);
  cudaSetDevice(ctx->cfg.device);
  NcclId id;
  memcpy(id.internal, id128, sizeof id.internal);
  int rc = g_nccl.CommInitRank(&ctx->nccl_comm, nranks, id, rank);
  if (rc) { ctx->nccl_comm = nullptr; return nccl_fail(ctx, "ncclCommInitRank", rc); }
  ctx->comm_rank = rank; ctx->comm_nranks = nranks;
  return IRSDE_OK;
}

int irsde_broadcast_weights(irsde_ctx* ctx, int32_t src, void* stream) {
  if (!ctx || !ctx->nccl_comm) return fail(ctx, IRSDE_ERR_STATE, "irsde_comm_init first");
  if (src < 0 || src >= ctx->comm_nranks) return fail(ctx, IRSDE_ERR_INVALID, "bad source rank");
  if (ctx->raw.empty()) return fail(ctx, IRSDE_ERR_STATE, "load a state dict of the architecture on every rank first");
  cudaSetDevice(ctx->cfg.device);
  // every rank has loaded a state dict of the same names/shapes (std::map: same iteration order on every rank); the raw
  // fp32 tensors are overwritten in place inside ONE NCCL group (a single fused launch), then repacked for the kernels
  CUDA_TRY(ctx, cudaDeviceSynchronize());  // chains in flight still read the packed weights
  int rc = g_nccl.GroupStart();
  if (rc) return nccl_fail(ctx, "ncclGroupStart", rc);
  for (auto& kv : ctx->raw) {
    rc = g_nccl.Broadcast(kv.second.dev, kv.second.dev, (size_t)kv.second.numel, kNcclFloat, src, ctx->nccl_comm, (cudaStream_t)stream);
    if (rc) { g_nccl.GroupEnd(); return nccl_fail(ctx, "ncclBroadcast", rc); }
  }
  rc = g_nccl.GroupEnd();
  if (rc) return nccl_fail(ctx, "ncclGroupEnd", rc);
  CUDA_TRY(ctx, cudaStreamSynchronize((cudaStream_t)stream));
  ctx->finalized = false;
  return irsde_finalize_weights(ctx);
}

int irsde_gather(irsde_ctx* ctx, const float* x_local, float* x_all, const int64_t* counts, void* stream) {
  if (!ctx || !ctx->nccl_comm) return fail(ctx, IRSDE_ERR_STATE, "irsde_comm_init first");
  if (!x_all || !counts) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  cudaSetDevice(ctx->cfg.device);
  // rank r's slice (counts[r] floats; the contiguous batch partition may be ragged) lands at the running offset in
  // x_all on EVERY rank: one broadcast per root inside a single group = an all-gather with per-rank counts
  int rc = g_nccl.GroupStart();
  if (rc) return nccl_fail(ctx, "ncclGroupStart", rc);
  int64_t off = 0;
  for (int r = 0; r < ctx->comm_nranks; ++r) {
    if (counts[r] < 0 || (r == ctx->comm_rank && counts[r] > 0 && !x_local)) { g_nccl.GroupEnd(); return fail(ctx, IRSDE_ERR_INVALID, "bad counts"); }
    if (counts[r] > 0) {
      rc = g_nccl.Broadcast(r == ctx->comm_rank ? (const void*)x_local : (const void*)(x_all + off), x_all + off, (size_t)counts[r],
                            kNcclFloat, r, ctx->nccl_comm, (cudaStream_t)stream);
      if (rc) { g_nccl.GroupEnd(); return nccl_fail(ctx, "ncclBroadcast", rc); }
    }
    off += counts[r];
  }
  rc = g_nccl.GroupEnd();
  return rc ? nccl_fail(ctx, "ncclGroupEnd", rc) : IRSDE_OK;
}

void irsde_destroy(irsde_ctx* ctx) {
  if (!ctx) return;
  if (ctx->nccl_comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->nccl_comm);
  cudaSetDevice(ctx->cfg.device);
  cudaDeviceSynchronize();
  for (auto& kv : ctx->plans) free_plan(ctx, kv.second);
  ctx->plans.clear();
  for (void* q : ctx->allocs) cudaFree(q);
  delete ctx;
}

int irsde_load_tensor(irsde_ctx* ctx, const char* name, const void* data, int32_t ndim, const int64_t* shape) {
  if (!ctx || !name || !data || ndim < 0 || ndim > 4) return fail(ctx, IRSDE_ERR_INVALID, "bad argument to irsde_load_tensor");
  cudaSetDevice(ctx->cfg.device);
  // Weights are pointer-stable buffers that captured step graphs read: a re-upload (load_state_dict, broadcast) must not
  // overtake chains still in flight on the caller's (possibly non-blocking) streams.  The first tensor of an upload
  // round drains the device; the copies below are synchronous, so later launches see the new values.
  if (ctx->finalized || ctx->raw.empty()) CUDA_TRY(ctx, cudaDeviceSynchronize());
  long long n = 1;
  std::vector<int64_t> sh(shape, shape + ndim);
  for (auto d : sh) n *= d;
  RawTensor& t = ctx->raw[name];
  if (t.dev && t.numel != n) return fail(ctx, IRSDE_ERR_INVALID, std::string("shape change for ") + name);
  if (!t.dev) {
    t.dev = (float*)dev_alloc(ctx, (size_t)n * 4, &ctx->allocs);
    if (!t.dev) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
  }
  t.shape = sh;
  t.numel = n;
  CUDA_TRY(ctx, cudaMemcpy(t.dev, data, (size_t)n * 4, cudaMemcpyDefault));
  ctx->finalized = false;
  return IRSDE_OK;
}

int irsde_finalize_weights(irsde_ctx* ctx) {
  if (!ctx) return fail(nullptr, IRSDE_ERR_INVALID, "null ctx");
  cudaSetDevice(ctx->cfg.device);
  auto specs = ctx->lat.on ? lat_param_specs(ctx->lat) : (ctx->naf.on ? naf_param_specs(ctx->naf) : param_specs(ctx->cfg, ctx->udim));
  for (auto& s : specs) {
    auto it = ctx->raw.find(s.name);
    if (it == ctx->raw.end()) return fail(ctx, IRSDE_ERR_STATE, "missing state-dict entry " + s.name);
    if (it->second.shape != s.shape) return fail(ctx, IRSDE_ERR_INVALID, "shape mismatch for " + s.name);
  }
  if (ctx->raw.size() != specs.size()) return fail(ctx, IRSDE_ERR_INVALID, "unexpected extra state-dict entries");
  // conv weights -> engine layouts (buffers are allocated once; reload keeps pointers stable)
  for (auto& s : specs) {
    if (s.shape.size() != 4) continue;  // vectors / Linear matrices stay fp32 as loaded
    if (s.name.size() > 2 && s.name.substr(s.name.size() - 2) == ".g") continue;
    if (ctx->naf.on && (s.shape[0] == 1 || s.name.find("conv2.weight") != std::string::npos ||
                        s.name.find("sca.1.weight") != std::string::npos))
      continue;  // beta/gamma vectors, depthwise and SCA weights are consumed raw
    int Cout = (int)s.shape[0], Cin = (int)s.shape[1], KH = (int)s.shape[2], KW = (int)s.shape[3];
    long long n = (long long)Cout * Cin * KH * KW;
    float*& ws = ctx->w_simt[s.name];
    if (!ws) ws = (float*)dev_alloc(ctx, (size_t)n * 4, &ctx->allocs);
    if (!ws) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
    pack_simt_kernel<<<(unsigned)((n + 255) / 256), 256>>>(ctx->raw[s.name].dev, ws, Cout, Cin, KH, KW);
    if (ctx->cfg.precision == IRSDE_PREC_FP32X3 && !(KH == 7)) {
      bool is_up = s.name.find(".3.1.weight") != std::string::npos && KH == 3;
      int Cout_pad = (Cout + 7) / 8 * 8;
      long long nt = (long long)(is_up ? 16 : KH * KW) * 2 * Cout_pad * Cin;
      float*& wt = ctx->w_tc3[s.name];
      if (!wt) wt = (float*)dev_alloc(ctx, (size_t)nt * 4, &ctx->allocs);
      if (!wt) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
      long long nthreads = nt / 2;
      if (is_up)
        pack_tc3_up_kernel<<<(unsigned)((nthreads + 255) / 256), 256>>>(ctx->raw[s.name].dev, wt, Cout, Cout_pad, Cin);
      else
        pack_tc3_kernel<<<(unsigned)((nthreads + 255) / 256), 256>>>(ctx->raw[s.name].dev, wt, Cout, Cout_pad, Cin, KH, KW);
    }
    if (ctx->cfg.precision == IRSDE_PREC_BF16) {
      bool is_up = s.name.find(".3.1.weight") != std::string::npos;
      bool is_stem = s.name == "init_conv.weight" && KH == 7;
      int Cout_pad = (Cout + 7) / 8 * 8;
      long long nt = is_up ? (long long)16 * Cout * Cin : (is_stem ? (long long)7 * Cout * 64 : (long long)Cout_pad * Cin * KH * KW);
      bf16*& wt = ctx->w_tc[s.name];
      if (!wt) wt = (bf16*)dev_alloc(ctx, (size_t)nt * 2, &ctx->allocs);
      if (!wt) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
      if (is_up)
        pack_tc_up_kernel<<<(unsigned)((nt + 255) / 256), 256>>>(ctx->raw[s.name].dev, wt, Cout, Cin);
      else if (is_stem && Cin <= 8)
        pack_tc_stem_kernel<<<(unsigned)((nt + 255) / 256), 256>>>(ctx->raw[s.name].dev, wt, Cout, Cin);
      else if (Cout_pad != Cout)
        pack_tc_padded_kernel<<<(unsigned)((nt + 255) / 256), 256>>>(ctx->raw[s.name].dev, wt, Cout, Cout_pad, Cin, KH, KW);
      else
        pack_tc_kernel<<<(unsigned)((n + 255) / 256), 256>>>(ctx->raw[s.name].dev, wt, Cout, Cin, KH, KW);
    }
  }
  // time-modulation: concatenate every block's mlp.1 into one [S][td_in] matrix
  // (UNet ResBlock: Linear(4nf -> 2*Cout); NAFBlock: Linear(2w -> 4c))
  struct TB { std::string pre; int rows; };
  std::vector<TB> tbs;
  std::string mlp_name = "mlp.1.";  // the block's time Linear (lens variant: time_mlp.1)
  int td = 0;
  if (ctx->lat.on) {
    td = 1;  // no time conditioning in the autoencoder
  } else if (ctx->naf.on) {
    td = 2 * ctx->naf.width;
    for (auto& b : naf_blocks(ctx->naf)) tbs.push_back({b.pre, 4 * b.c});
    if (ctx->naf.lens) mlp_name = "time_mlp.1.";
  } else {
    td = ctx->cfg.nf * 4;
    for (auto& rb : resblocks(ctx->cfg, ctx->udim)) tbs.push_back({rb.pre, 2 * rb.cout});
  }
  int S = 0;
  for (auto& t : tbs) { ctx->ss_off[t.pre] = S; S += t.rows; }
  if (!ctx->wall) {
    ctx->wall = (float*)dev_alloc(ctx, (size_t)S * td * 4, &ctx->allocs);
    ctx->ball = (float*)dev_alloc(ctx, (size_t)S * 4, &ctx->allocs);
    if (!ctx->wall || !ctx->ball) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
  }
  ctx->S = S;
  for (auto& t : tbs) {
    int off = ctx->ss_off[t.pre];
    CUDA_TRY(ctx, cudaMemcpy(ctx->wall + (size_t)off * td, ctx->raw[t.pre + mlp_name + "weight"].dev, (size_t)t.rows * td * 4,
                             cudaMemcpyDeviceToDevice));
    CUDA_TRY(ctx, cudaMemcpy(ctx->ball + off, ctx->raw[t.pre + mlp_name + "bias"].dev, (size_t)t.rows * 4, cudaMemcpyDeviceToDevice));
  }
  if (ctx->naf.lens) {  // camera modulation: every block's cam_mlp.1 (Linear(2w -> 2c)) into one [cam_S][2w] matrix
    if (!ctx->cam_wall) {
      ctx->cam_wall = (float*)dev_alloc(ctx, (size_t)ctx->cam_S * td * 4, &ctx->allocs);
      ctx->cam_ball = (float*)dev_alloc(ctx, (size_t)ctx->cam_S * 4, &ctx->allocs);
      if (!ctx->cam_wall || !ctx->cam_ball) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
    }
    for (auto& b : naf_blocks(ctx->naf)) {
      const int off = ctx->cam_off[b.pre], rows = 2 * b.c;
      CUDA_TRY(ctx, cudaMemcpy(ctx->cam_wall + (size_t)off * td, ctx->raw[b.pre + "cam_mlp.1.weight"].dev, (size_t)rows * td * 4,
                               cudaMemcpyDeviceToDevice));
      CUDA_TRY(ctx, cudaMemcpy(ctx->cam_ball + off, ctx->raw[b.pre + "cam_mlp.1.bias"].dev, (size_t)rows * 4, cudaMemcpyDeviceToDevice));
    }
    if (ctx->lens_n) {  // the table was computed from the previous weights (or not yet): recompute it
      int rc = compute_cam(ctx, 0);
      if (rc) return rc;
    }
  }
  CUDA_TRY(ctx, cudaDeviceSynchronize());
  ctx->finalized = true;
  return IRSDE_OK;
}

int irsde_set_schedule(irsde_ctx* ctx, const float* thetas, const float* sigmas, const float* thetas_cumsum,
                       const float* sigma_bars, float dt, float max_sigma, int32_t T) {
  if (!ctx || !thetas || !sigmas || !thetas_cumsum || !sigma_bars || T < 1) return fail(ctx, IRSDE_ERR_INVALID, "bad schedule");
  cudaSetDevice(ctx->cfg.device);
  ctx->T = T; ctx->dt = dt; ctx->max_sigma = max_sigma;
  ctx->thetas.assign(thetas, thetas + T + 1);
  ctx->sigmas.assign(sigmas, sigmas + T + 1);
  ctx->cumsum.assign(thetas_cumsum, thetas_cumsum + T + 1);
  ctx->sbars.assign(sigma_bars, sigma_bars + T + 1);
  std::vector<float> tab;
  for (int m = 0; m < IRSDE_NUM_MODES; ++m) {
    fill_default_coeffs(ctx, m, tab);
    int rc = upload_coeffs(ctx, m, tab.data(), T);
    if (rc) return rc;
  }
  ctx->have_sched = true;
  return IRSDE_OK;
}

int irsde_set_coeffs(irsde_ctx* ctx, int32_t mode, const float* table, int32_t T) {
  if (!ctx || !table || mode < 0 || mode >= IRSDE_NUM_MODES) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  if (!ctx->have_sched || T != ctx->T) return fail(ctx, IRSDE_ERR_STATE, "irsde_set_schedule must be called first with the same T");
  cudaSetDevice(ctx->cfg.device);
  return upload_coeffs(ctx, mode, table, T);
}

int irsde_noise_fn(irsde_ctx* ctx, const float* x, const float* mu, const float* times, int32_t n_times, float* out,
                   int32_t B, int32_t H, int32_t W, void* stream) {
  if (!ctx || !x || !times || !out) return fail(ctx, IRSDE_ERR_INVALID, "null argument");
  if (!ctx->finalized) return fail(ctx, IRSDE_ERR_STATE, "weights not finalized");
  if (ctx->cfg.variant == IRSDE_NET_CONDITIONAL && !mu) return fail(ctx, IRSDE_ERR_INVALID, "mu required for the conditional network");
  if (n_times != 1 && n_times != B) return fail(ctx, IRSDE_ERR_INVALID, "n_times must be 1 or B");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Plan* p;
  int rc = build_plan(ctx, B, H, W, &p);
  if (rc) return rc;
  rc = lens_ready(ctx, B, p);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(p->fwd_times, times, (size_t)n_times * 4, cudaMemcpyHostToDevice, st));
  time_rows(ctx, p->fwd_times, n_times, p->fwd_temb, p->fwd_table, st);
  p->cur.x = x; p->cur.mu = mu; p->cur.out = out;
  p->cur.ss = p->fwd_table; p->cur.t_ptr = p->d_zero; p->cur.ss_img_stride = (n_times > 1) ? 1 : 0;
  run_forward(ctx, p, st);
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

int irsde_step(irsde_ctx* ctx, int32_t mode, const float* x, const float* mu, const float* noise, const float* z,
               int32_t t, float* out, int64_t n, void* stream) {
  if (!ctx || !x || !noise || !out || mode < 0 || mode >= IRSDE_NUM_MODES) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  if (!ctx->have_sched) return fail(ctx, IRSDE_ERR_STATE, "schedule not set");
  if (t < 1 || t > ctx->T) return fail(ctx, IRSDE_ERR_INVALID, "t out of range [1,T]");
  bool need_z = mode == IRSDE_MODE_SDE || mode == IRSDE_MODE_POSTERIOR || mode == IRSDE_MODE_DSDE_SDE;
  if (need_z && !z) return fail(ctx, IRSDE_ERR_INVALID, "z required for stochastic modes");
  if (mode <= IRSDE_MODE_POSTERIOR && !mu) return fail(ctx, IRSDE_ERR_INVALID, "mu required for IRSDE modes");
  cudaSetDevice(ctx->cfg.device);
  launch_sde_update(mode, x, mu, noise, z, 0, ctx->coef_dev[mode], nullptr, t, out, n, 0, 0, 0, (cudaStream_t)stream);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

int irsde_reverse(irsde_ctx* ctx, int32_t mode, const float* xT, const float* mu, const float* z, float* x0, int32_t B,
                  int32_t H, int32_t W, int32_t T, uint64_t seed, int32_t use_graph, void* stream) {
  if (!ctx || !xT || !x0 || mode < 0 || mode >= IRSDE_NUM_MODES) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  if (!ctx->finalized) return fail(ctx, IRSDE_ERR_STATE, "weights not finalized");
  if (!ctx->have_sched) return fail(ctx, IRSDE_ERR_STATE, "schedule not set");
  if (T < 0) T = ctx->T;
  if (T > ctx->T) return fail(ctx, IRSDE_ERR_INVALID, "T exceeds the schedule length");
  bool irs = mode <= IRSDE_MODE_POSTERIOR;
  if (irs != (ctx->cfg.variant == IRSDE_NET_CONDITIONAL))
    return fail(ctx, IRSDE_ERR_INVALID, "sampler mode does not match the network variant");
  if (irs && !mu) return fail(ctx, IRSDE_ERR_INVALID, "mu required");
  if (ctx->cfg.in_nc != ctx->cfg.out_nc) return fail(ctx, IRSDE_ERR_INVALID, "chain needs in_nc == out_nc");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Plan* p;
  int rc = build_plan(ctx, B, H, W, &p);
  if (rc) return rc;
  rc = lens_ready(ctx, B, p);
  if (rc) return rc;
  long long n = (long long)B * ctx->cfg.in_nc * H * W;
  CUDA_TRY(ctx, cudaMemcpyAsync(p->x_state, xT, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  if (mu) CUDA_TRY(ctx, cudaMemcpyAsync(p->mu_buf, mu, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  if (T == 0) {
    CUDA_TRY(ctx, cudaMemcpyAsync(x0, p->x_state, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    return IRSDE_OK;
  }
  rc = ensure_chain_table(ctx, p, ctx->T, st);
  if (rc) return rc;
  if (ctx->n_uids && ctx->n_uids != B) return fail(ctx, IRSDE_ERR_INVALID, "irsde_set_image_uids count does not match the batch");
  launch_set_step(p->d_step, T, 0, z, seed, ctx->image_base, ctx->n_uids ? ctx->d_uids : nullptr, st);
  ctx->launches++;
  p->cur.x = p->x_state; p->cur.mu = p->mu_buf; p->cur.out = p->eps_buf;
  p->cur.ss = p->chain_table; p->cur.t_ptr = &p->d_step->t; p->cur.ss_img_stride = 0;
  const float* mu_arg = irs ? p->mu_buf : nullptr;
  auto one_step = [&](cudaStream_t s) {
    run_forward(ctx, p, s);
    launch_sde_update(mode, p->x_state, mu_arg, p->eps_buf, nullptr, n, ctx->coef_dev[mode], p->d_step, 0, p->x_state, n, 0,
                      n / B, 0, s);
    launch_advance_step(p->d_step, s);
    ctx->launches += 2;
  };
  if (use_graph && !ctx->prof) {
    if (p->graph[mode] && (p->graph_cam[mode] != p->cur.cam || p->graph_cam_stride[mode] != p->cur.cam_img_stride)) {
      cudaGraphExecDestroy(p->graph[mode]);  // captured with another camera table / lens count
      p->graph[mode] = nullptr;
    }
    if (!p->graph[mode]) {
      cudaStream_t cs;
      CUDA_TRY(ctx, cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      long long before = ctx->launches;
      cudaGraph_t g;
      cudaError_t e = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
      if (e == cudaSuccess) {
        one_step(cs);
        e = cudaStreamEndCapture(cs, &g);
      }
      p->step_launches[mode] = ctx->launches - before;  // kernels in one captured step
      ctx->launches = before;                            // capture does not execute
      if (e != cudaSuccess) {
        cudaStreamDestroy(cs);
        return fail(ctx, IRSDE_ERR_CUDA, std::string("graph capture failed: ") + cudaGetErrorString(e));
      }
      e = cudaGraphInstantiate(&p->graph[mode], g, 0);
      cudaGraphDestroy(g);
      cudaStreamDestroy(cs);
      if (e != cudaSuccess) return fail(ctx, IRSDE_ERR_CUDA, std::string("graph instantiate failed: ") + cudaGetErrorString(e));
      p->graph_cam[mode] = p->cur.cam;
      p->graph_cam_stride[mode] = p->cur.cam_img_stride;
    }
    for (int i = 0; i < T; ++i) CUDA_TRY(ctx, cudaGraphLaunch(p->graph[mode], st));
    ctx->launches += (long long)T * p->step_launches[mode];
  } else {
    for (int i = 0; i < T; ++i) one_step(st);
  }
  CUDA_TRY(ctx, cudaMemcpyAsync(x0, p->x_state, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

int irsde_noise_state(irsde_ctx* ctx, const float* mu, float* out, int64_t n, uint64_t seed, void* stream) {
  if (!ctx || !mu || !out) return fail(ctx, IRSDE_ERR_INVALID, "null argument");
  if (!ctx->have_sched) return fail(ctx, IRSDE_ERR_STATE, "schedule not set");
  cudaSetDevice(ctx->cfg.device);
  launch_noise_state(mu, out, n, ctx->max_sigma, seed, n, ctx->image_base, nullptr, (cudaStream_t)stream);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

int irsde_noise_state_images(irsde_ctx* ctx, const float* mu, float* out, int32_t B, int64_t image_elems, uint64_t seed,
                             void* stream) {
  if (!ctx || !mu || !out || B < 1 || image_elems < 1) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  if (!ctx->have_sched) return fail(ctx, IRSDE_ERR_STATE, "schedule not set");
  cudaSetDevice(ctx->cfg.device);
  if (ctx->n_uids && ctx->n_uids != B) return fail(ctx, IRSDE_ERR_INVALID, "irsde_set_image_uids count does not match the batch");
  launch_noise_state(mu, out, (long long)B * image_elems, ctx->max_sigma, seed, image_elems, ctx->image_base,
                     ctx->n_uids ? ctx->d_uids : nullptr, (cudaStream_t)stream);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

int irsde_random_states(const float* x0, const float* mu, const float* noise, const float* w, const float* sigma_bar, float* out,
                        int32_t B, int64_t image_elems, void* stream) {
  if (!x0 || !mu || !noise || !w || !sigma_bar || !out || B < 1 || image_elems < 1)
    return fail(nullptr, IRSDE_ERR_INVALID, "bad argument to irsde_random_states");
  launch_random_states(x0, mu, noise, w, sigma_bar, out, B, image_elems, (cudaStream_t)stream);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, IRSDE_ERR_CUDA, std::string("random_states: ") + cudaGetErrorString(e));
  return IRSDE_OK;
}

int irsde_set_image_base(irsde_ctx* ctx, uint64_t first_image_uid) {
  if (!ctx) return fail(ctx, IRSDE_ERR_INVALID, "null ctx");
  ctx->image_base = first_image_uid;
  ctx->n_uids = 0;
  return IRSDE_OK;
}

int irsde_set_image_uids(irsde_ctx* ctx, const uint64_t* uids, int32_t n, void* stream) {
  const int MAX_UIDS = 4096;
  if (!ctx || !uids || n < 1 || n > MAX_UIDS) return fail(ctx, IRSDE_ERR_INVALID, "uids: need 1..4096 host values");
  cudaSetDevice(ctx->cfg.device);
  if (!ctx->d_uids) {
    ctx->d_uids = (unsigned long long*)dev_alloc(ctx, sizeof(unsigned long long) * MAX_UIDS, &ctx->allocs);
    if (!ctx->d_uids) return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
  }
  // pageable host source: the copy is staged before the call returns, so the caller may reuse `uids` at once
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->d_uids, uids, sizeof(uint64_t) * n, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  ctx->n_uids = n;
  return IRSDE_OK;
}

int irsde_profile_begin(irsde_ctx* ctx) {
  if (!ctx) return fail(nullptr, IRSDE_ERR_INVALID, "null ctx");
  for (auto& e : ctx->prof_events) { cudaEventDestroy(e.e0); cudaEventDestroy(e.e1); }
  ctx->prof_events.clear();
  ctx->prof = true;
  return IRSDE_OK;
}

int irsde_profile_end(irsde_ctx* ctx, double* ms, double* flops, int64_t* launches, int32_t ncat) {
  return irsde_profile_end_bytes(ctx, ms, flops, launches, nullptr, ncat);
}

int irsde_profile_end_bytes(irsde_ctx* ctx, double* ms, double* flops, int64_t* launches, double* bytes, int32_t ncat) {
  if (!ctx || !ms || !flops || !launches || ncat < CAT_COUNT) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  cudaSetDevice(ctx->cfg.device);
  ctx->prof = false;
  CUDA_TRY(ctx, cudaDeviceSynchronize());
  for (int i = 0; i < ncat; ++i) { ms[i] = 0; flops[i] = 0; launches[i] = 0; if (bytes) bytes[i] = 0; }
  const char* dump = getenv("IRSDE_PROFILE_DUMP");
  for (auto& e : ctx->prof_events) {
    float t = 0.f;
    cudaEventElapsedTime(&t, e.e0, e.e1);
    if (dump && dump[0] == '1' && e.op)
      fprintf(stderr, "PROF\t%d\t%.4f\t%.1f\t%.1f\t%s\n", e.cat, t, e.op->flops > 0 ? e.op->flops / (t * 1e-3) / 1e12 : 0.0,
              e.op->bytes > 0 ? e.op->bytes / (t * 1e-3) / 1e9 : 0.0, e.op->label.c_str());
    ms[e.cat] += t;
    if (bytes && e.op) bytes[e.cat] += e.op->bytes;
    flops[e.cat] += e.flops;
    launches[e.cat] += 1;
    cudaEventDestroy(e.e0);
    cudaEventDestroy(e.e1);
  }
  ctx->prof_events.clear();
  return IRSDE_OK;
}

int irsde_trim(irsde_ctx* ctx) {
  if (!ctx) return fail(nullptr, IRSDE_ERR_INVALID, "null ctx");
  cudaSetDevice(ctx->cfg.device);
  evict_plans(ctx, nullptr, true);
  return IRSDE_OK;
}

int32_t irsde_plan_num_ops(irsde_ctx* ctx, int32_t B, int32_t H, int32_t W) {
  if (!ctx) return fail(nullptr, IRSDE_ERR_INVALID, "null ctx");
  if (!ctx->finalized) return fail(ctx, IRSDE_ERR_STATE, "weights not finalized");
  cudaSetDevice(ctx->cfg.device);
  Plan* p;
  int rc = build_plan(ctx, B, H, W, &p);
  return rc ? rc : (int32_t)p->ops.size();
}

int irsde_plan_op_info(irsde_ctx* ctx, int32_t B, int32_t H, int32_t W, int32_t op, char* label, int32_t label_cap,
                       int32_t* dims) {
  if (!ctx || !label || label_cap < 1 || !dims) return fail(ctx, IRSDE_ERR_INVALID, "bad argument");
  if (!ctx->finalized) return fail(ctx, IRSDE_ERR_STATE, "weights not finalized");
  cudaSetDevice(ctx->cfg.device);
  Plan* p;
  int rc = build_plan(ctx, B, H, W, &p);
  if (rc) return rc;
  if (op < 0 || op >= (int)p->ops.size()) return fail(ctx, IRSDE_ERR_INVALID, "op index out of range");
  const OpRec& r = p->ops[op];
  snprintf(label, (size_t)label_cap, "%s", r.label.c_str());
  dims[0] = r.out_p ? r.out_C : 0; dims[1] = r.out_H; dims[2] = r.out_W; dims[3] = r.cat;
  return IRSDE_OK;
}

int irsde_trace_forward(irsde_ctx* ctx, const float* x, const float* mu, const float* times, int32_t n_times, int32_t B,
                        int32_t H, int32_t W, int32_t op, float* dump, void* stream) {
  if (!ctx || !x || !times || !dump) return fail(ctx, IRSDE_ERR_INVALID, "null argument");
  if (!ctx->finalized) return fail(ctx, IRSDE_ERR_STATE, "weights not finalized");
  if (ctx->cfg.variant == IRSDE_NET_CONDITIONAL && !ctx->lat.on && !mu) return fail(ctx, IRSDE_ERR_INVALID, "mu required");
  if (n_times != 1 && n_times != B) return fail(ctx, IRSDE_ERR_INVALID, "n_times must be 1 or B");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  Plan* p;
  int rc = build_plan(ctx, B, H, W, &p);
  if (rc) return rc;
  if (op < 0 || op >= (int)p->ops.size()) return fail(ctx, IRSDE_ERR_INVALID, "op index out of range");
  const OpRec& r = p->ops[op];
  if (!r.out_p) return fail(ctx, IRSDE_ERR_UNSUPPORTED, "this op has no NHWC output view to read back");
  rc = lens_ready(ctx, B, p);
  if (rc) return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(p->fwd_times, times, (size_t)n_times * 4, cudaMemcpyHostToDevice, st));
  time_rows(ctx, p->fwd_times, n_times, p->fwd_temb, p->fwd_table, st);
  p->cur.x = x; p->cur.mu = mu; p->cur.out = p->eps_buf;
  p->cur.ss = p->fwd_table; p->cur.t_ptr = p->d_zero; p->cur.ss_img_stride = (n_times > 1) ? 1 : 0;
  for (int i = 0; i <= op; ++i) p->ops[i].fn(p, st);
  if (ctx->cfg.precision != IRSDE_PREC_BF16)
    launch_nhwc_to_nchw<float>((const float*)r.out_p, r.out_pitch, dump, B, r.out_C, r.out_H, r.out_W, st);
  else
    launch_nhwc_to_nchw<bf16>((const bf16*)r.out_p, r.out_pitch, dump, B, r.out_C, r.out_H, r.out_W, st);
  CUDA_TRY(ctx, cudaGetLastError());
  return IRSDE_OK;
}

int64_t irsde_launch_count(const irsde_ctx* ctx) { return ctx ? ctx->launches : 0; }
int64_t irsde_device_bytes(const irsde_ctx* ctx) { return ctx ? ctx->dev_bytes : 0; }

int irsde_conv2d(irsde_ctx* ctx, int32_t engine, const float* x, const float* w, const float* bias, float* y, int32_t B,
                 int32_t Cin, int32_t H, int32_t W, int32_t Cout, int32_t KH, int32_t KW, int32_t stride, int32_t pad,
                 int32_t upsample, int32_t silu, void* stream) {
  return irsde_conv2d_ex(ctx, engine, x, w, bias, nullptr, y, B, Cin, H, W, Cout, KH, KW, stride, pad, upsample, silu, 0, stream);
}

int irsde_conv2d_ex(irsde_ctx* ctx, int32_t engine, const float* x, const float* w, const float* bias, const float* residual,
                    float* y, int32_t B, int32_t Cin, int32_t H, int32_t W, int32_t Cout, int32_t KH, int32_t KW, int32_t stride,
                    int32_t pad, int32_t upsample, int32_t silu, int32_t flags, void* stream) {
  if (!ctx || !x || !w || !y) return fail(ctx, IRSDE_ERR_INVALID, "null argument");
  const bool f_qsm = (flags & IRSDE_CONV_QSOFTMAX) != 0, f_wimg = (flags & IRSDE_CONV_W_PER_IMAGE) != 0;
  if ((f_qsm || f_wimg) && engine != 1) return fail(ctx, IRSDE_ERR_UNSUPPORTED, "q-softmax / per-image weights are bf16 tensor-core epilogues");
  if (residual && engine == 0) return fail(ctx, IRSDE_ERR_UNSUPPORTED, "residual is an epilogue of the tensor-core engines");
  if ((f_qsm || f_wimg) && !(KH == 1 && KW == 1 && stride == 1 && pad == 0 && !upsample && Cout % 8 == 0))
    return fail(ctx, IRSDE_ERR_INVALID, "q-softmax / per-image weights need a 1x1 conv with Cout % 8 == 0");
  if (f_qsm && Cout < 128) return fail(ctx, IRSDE_ERR_INVALID, "q-softmax needs Cout >= 128 (4 heads x 32)");
  cudaSetDevice(ctx->cfg.device);
  cudaStream_t st = (cudaStream_t)stream;
  int up = upsample ? 2 : 1;
  if (engine == 1) {
    // tcgen05 engine: same taps/weight packing as the plan builder
    std::string terr;
    if (!tc_init(&terr)) return fail(ctx, IRSDE_ERR_CUDA, "tc_init: " + terr);
    bool k3 = KH == 3 && KW == 3 && stride == 1 && pad == 1, k1 = KH == 1 && KW == 1 && stride == 1 && pad == 0 && up == 1,
         k4 = KH == 4 && KW == 4 && stride == 2 && pad == 1 && up == 1 && H % 2 == 0 && W % 2 == 0,
         k7 = KH == 7 && KW == 7 && stride == 1 && pad == 3 && up == 1 && Cin <= 8 && Cout % 8 == 0;
    bool nchw = Cout % 8 != 0;  // head-style output: fp32 NCHW straight from the epilogue
    if (!(k3 || k1 || k4 || k7) || (!k7 && Cin % 8) || (nchw && !(k3 && up == 1)))
      return fail(ctx, IRSDE_ERR_UNSUPPORTED, "shape not supported by the tensor-core engine");
    int Ho = (H * up + 2 * pad - KH) / stride + 1, Wo = (W * up + 2 * pad - KW) / stride + 1;
    int Cout_pad = (Cout + 7) / 8 * 8;
    std::vector<void*> tmp;
    long long nin = k7 ? (long long)B * (H + 6) * (W + 8) * 8 + 64 : (long long)B * H * W * Cin;
    long long nw = (long long)Cout * Cin * KH * KW, nout = (long long)B * Ho * Wo * Cout_pad;
    long long nwt = (k3 && up == 2) ? (long long)16 * Cout * Cin : (k7 ? (long long)7 * Cout * 64 : (long long)Cout_pad * Cin * KH * KW);
    if (f_wimg) nwt *= B;  // w is [B][Cout][Cin]
    (void)nw;
    bf16* resb = nullptr;
    if (residual) {
      if (nchw) return fail(ctx, IRSDE_ERR_UNSUPPORTED, "residual needs Cout % 8 == 0");
      resb = (bf16*)dev_alloc(ctx, nout * 2, &tmp);
      if (!resb) { for (void* q : tmp) cudaFree(q); return fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed"); }
      launch_nchw_to_nhwc<bf16>(residual, resb, B, Cout, Ho, Wo, Cout, st);
    }
    bf16* xin = (bf16*)dev_alloc(ctx, nin * 2, &tmp);
    bf16* xs2d = (bf16*)dev_alloc(ctx, nin * 2, &tmp);
    bf16* wp = (bf16*)dev_alloc(ctx, nwt * 2, &tmp);
    bf16* yo = (bf16*)dev_alloc(ctx, nout * 2, &tmp);
    int rc = IRSDE_OK;
    TcConvDesc* d = nullptr;
    if (!xin || !xs2d || !wp || !yo) rc = fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
    if (!rc) {
      if (k7) {
        cudaMemsetAsync(xin, 0, nin * 2, st);
        launch_prep_input<bf16>(x, nullptr, xin, B, Cin, H, W, H, W, 8, 0, st, 3, 3, W + 8, H + 6);
        pack_tc_stem_kernel<<<(unsigned)((nwt + 255) / 256), 256, 0, st>>>(w, wp, Cout, Cin);
      } else {
        launch_nchw_to_nhwc<bf16>(x, xin, B, Cin, H, W, Cin, st);
        if (k3 && up == 2) pack_tc_up_kernel<<<(unsigned)((nwt + 255) / 256), 256, 0, st>>>(w, wp, Cout, Cin);
        else if (f_wimg) pack_tc_kernel<<<(unsigned)((nwt + 255) / 256), 256, 0, st>>>(w, wp, B * Cout, Cin, 1, 1);
        else pack_tc_padded_kernel<<<(unsigned)((nwt + 255) / 256), 256, 0, st>>>(w, wp, Cout, Cout_pad, Cin, KH, KW);
      }
      TcTap taps[16];
      int ntaps = 0, nph = 1, planes = 1, Ha = H, Wa = W, Ca = Cin, a_pitch = Cin;
      const bf16* a_ptr = xin;
      if (k7) { for (int r = 0; r < 7; ++r) taps[ntaps++] = TcTap{r, 0, 0}; planes = -1; Ca = 64; a_pitch = 8; }
      else if (k3 && up == 1) { for (int r = 0; r < 3; ++r) for (int q = 0; q < 3; ++q) taps[ntaps++] = TcTap{r - 1, q - 1, 0}; }
      else if (k3) { nph = 4; for (int a = 0; a < 2; ++a) for (int q = 0; q < 2; ++q) taps[ntaps++] = TcTap{a - 1, q - 1, 0}; }
      else if (k1) { taps[ntaps++] = TcTap{0, 0, 0}; }
      else {
        static const int PY[4] = {1, 0, 1, 0}, DH[4] = {-1, 0, 0, 1};
        for (int r = 0; r < 4; ++r) for (int q = 0; q < 4; ++q) taps[ntaps++] = TcTap{DH[r], DH[q], PY[r] * 2 + PY[q]};
        planes = 4; Ha = H / 2; Wa = W / 2;
        launch_space_to_depth<bf16>(xin, Cin, xs2d, B, H, W, Cin, st);
        a_ptr = xs2d;
      }
      Epilogue ep;
      memset(&ep, 0, sizeof ep);
      ep.bias = bias;
      ep.silu = silu;
      if (resb) { ep.res = resb; ep.res_pitch = Cout; }
      d = tc_conv_create(a_ptr, a_pitch, B, Ha, Wa, Ca, planes, wp, Cout, ntaps, taps, nph, ep, nchw ? nullptr : yo, Cout, Ho, Wo, &terr,
                         (f_qsm ? TC_FLAG_QSOFTMAX : 0) | (f_wimg ? TC_FLAG_W_PER_IMAGE : 0));
      if (!d) rc = fail(ctx, IRSDE_ERR_INVALID, "tc_conv_create: " + terr);
    }
    if (!rc) {
      if (nchw) tc_conv_set_out_nchw(d, y, Ho, Wo);
      tc_conv_launch(d, st);
      if (!nchw) launch_nhwc_to_nchw<bf16>(yo, Cout, y, B, Cout, Ho, Wo, st);
      ctx->launches += 4;
      cudaError_t e = cudaStreamSynchronize(st);
      if (e == cudaSuccess) e = cudaGetLastError();
      if (e != cudaSuccess) rc = fail(ctx, IRSDE_ERR_CUDA, std::string("tensor-core conv2d failed: ") + cudaGetErrorString(e));
    }
    if (d) tc_conv_destroy(d);
    for (void* q : tmp) cudaFree(q);
    return rc;
  }
  if (engine == 2) {
    // fp32x3 engine: fp32 NHWC, hi/lo split, 3 x tcgen05.mma.kind::tf32 (conv_tc.cu MODE 3)
    std::string terr;
    if (!tc_init(&terr)) return fail(ctx, IRSDE_ERR_CUDA, "tc_init: " + terr);
    bool k3 = KH == 3 && KW == 3 && stride == 1 && pad == 1, k1 = KH == 1 && KW == 1 && stride == 1 && pad == 0 && up == 1,
         k4 = KH == 4 && KW == 4 && stride == 2 && pad == 1 && up == 1 && H % 2 == 0 && W % 2 == 0;
    bool nchw = Cout % 4 != 0;
    if (!(k3 || k1 || k4) || Cin % 4 || (nchw && !(k3 && up == 1)) || residual && nchw)
      return fail(ctx, IRSDE_ERR_UNSUPPORTED, "shape not supported by the fp32x3 engine");
    int Ho = (H * up + 2 * pad - KH) / stride + 1, Wo = (W * up + 2 * pad - KW) / stride + 1;
    int Cout_pad = (Cout + 7) / 8 * 8;
    std::vector<void*> tmp;
    long long nin = (long long)B * H * W * Cin, nout = (long long)B * Ho * Wo * Cout;
    long long nwt = (long long)((k3 && up == 2) ? 16 : KH * KW) * 2 * Cout_pad * Cin;
    float* xin = (float*)dev_alloc(ctx, nin * 4, &tmp);
    float* xs2d = (float*)dev_alloc(ctx, nin * 4, &tmp);
    float* xsp = (float*)dev_alloc(ctx, 2 * nin * 4, &tmp);
    float* wp = (float*)dev_alloc(ctx, nwt * 4, &tmp);
    float* yo = (float*)dev_alloc(ctx, (nout + 16) * 4, &tmp);
    float* resb = residual ? (float*)dev_alloc(ctx, nout * 4, &tmp) : nullptr;
    int rc = IRSDE_OK;
    TcConvDesc* d = nullptr;
    if (!xin || !xs2d || !xsp || !wp || !yo || (residual && !resb)) rc = fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
    if (!rc) {
      launch_nchw_to_nhwc<float>(x, xin, B, Cin, H, W, Cin, st);
      if (resb) launch_nchw_to_nhwc<float>(residual, resb, B, Cout, Ho, Wo, Cout, st);
      if (k3 && up == 2) pack_tc3_up_kernel<<<(unsigned)((nwt / 2 + 255) / 256), 256, 0, st>>>(w, wp, Cout, Cout_pad, Cin);
      else pack_tc3_kernel<<<(unsigned)((nwt / 2 + 255) / 256), 256, 0, st>>>(w, wp, Cout, Cout_pad, Cin, KH, KW);
      TcTap taps[16];
      int ntaps = 0, nph = 1, planes = 1, Ha = H, Wa = W;
      const float* a_src = xin;
      if (k3 && up == 1) { for (int r = 0; r < 3; ++r) for (int q = 0; q < 3; ++q) taps[ntaps++] = TcTap{r - 1, q - 1, 0}; }
      else if (k3) { nph = 4; for (int a = 0; a < 2; ++a) for (int q = 0; q < 2; ++q) taps[ntaps++] = TcTap{a - 1, q - 1, 0}; }
      else if (k1) { taps[ntaps++] = TcTap{0, 0, 0}; }
      else {
        static const int PY[4] = {1, 0, 1, 0}, DH[4] = {-1, 0, 0, 1};
        for (int r = 0; r < 4; ++r) for (int q = 0; q < 4; ++q) taps[ntaps++] = TcTap{DH[r], DH[q], PY[r] * 2 + PY[q]};
        planes = 4; Ha = H / 2; Wa = W / 2;
        launch_space_to_depth<float>(xin, Cin, xs2d, B, H, W, Cin, st);
        a_src = xs2d;
      }
      launch_split_tf32(a_src, Cin, xsp, (long long)planes * B * Ha * Wa, Cin, st);
      Epilogue ep;
      memset(&ep, 0, sizeof ep);
      ep.bias = bias;
      ep.silu = silu;
      if (resb) { ep.res = resb; ep.res_pitch = Cout; }
      d = tc_conv_create_f32x3(xsp, B, Ha, Wa, Cin, planes, wp, Cout, ntaps, taps, nph, ep, nchw ? nullptr : yo, Cout, Ho, Wo, &terr);
      if (!d) rc = fail(ctx, IRSDE_ERR_INVALID, "tc_conv_create_f32x3: " + terr);
    }
    if (!rc) {
      if (nchw) tc_conv_set_out_nchw(d, y, Ho, Wo);
      tc_conv_launch(d, st);
      if (!nchw) launch_nhwc_to_nchw<float>(yo, Cout, y, B, Cout, Ho, Wo, st);
      ctx->launches += 5;
      cudaError_t e = cudaStreamSynchronize(st);
      if (e == cudaSuccess) e = cudaGetLastError();
      if (e != cudaSuccess) rc = fail(ctx, IRSDE_ERR_CUDA, std::string("fp32x3 conv2d failed: ") + cudaGetErrorString(e));
    }
    if (d) tc_conv_destroy(d);
    for (void* q : tmp) cudaFree(q);
    return rc;
  }
  if (engine != 0) return fail(ctx, IRSDE_ERR_INVALID, "unknown engine");
  ConvGeom g;
  g.B = B; g.Hin = H; g.Win = W; g.Cin = Cin; g.up = up; g.KH = KH; g.KW = KW; g.stride = stride; g.pad = pad;
  g.Hout = (H * up + 2 * pad - KH) / stride + 1;
  g.Wout = (W * up + 2 * pad - KW) / stride + 1;
  g.Cout = Cout;
  std::vector<void*> tmp;
  long long nin = (long long)B * H * W * Cin, nw = (long long)Cout * Cin * KH * KW, nout = (long long)B * g.Hout * g.Wout * Cout;
  float* xin = (float*)dev_alloc(ctx, nin * 4, &tmp);
  float* wp = (float*)dev_alloc(ctx, nw * 4, &tmp);
  float* yo = (float*)dev_alloc(ctx, nout * 4, &tmp);
  int rc = IRSDE_OK;
  if (!xin || !wp || !yo) rc = fail(ctx, IRSDE_ERR_CUDA, "cudaMalloc failed");
  if (!rc) {
    launch_nchw_to_nhwc<float>(x, xin, B, Cin, H, W, Cin, st);
    pack_simt_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, st>>>(w, wp, Cout, Cin, KH, KW);
    Epilogue ep;
    memset(&ep, 0, sizeof ep);
    ep.bias = bias;
    ep.silu = silu;
    launch_conv_simt<float>(g, xin, Cin, wp, ep, yo, Cout, nullptr, 0, 0, st);
    launch_nhwc_to_nchw<float>(yo, Cout, y, B, Cout, g.Hout, g.Wout, st);
    ctx->launches += 4;
    if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) rc = fail(ctx, IRSDE_ERR_CUDA, "conv2d failed");
  }
  for (void* q : tmp) { cudaFree(q); }
  return rc;
}

// ---- image conversion / metrics (stateless) ----------------------------------------------------------------
static int img_args_ok(const void* a, const void* b, int B, int C, int H, int W) {
  if (!a || !b || B < 1 || H < 1 || W < 1 || (C != 1 && C != 3)) return fail(nullptr, IRSDE_ERR_INVALID, "bad image argument");
  return IRSDE_OK;
}
static int img_launch_status(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(nullptr, IRSDE_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  return IRSDE_OK;
}
int irsde_tensor2img_u8(const float* chw, uint8_t* hwc, int32_t B, int32_t C, int32_t H, int32_t W, double lo, double hi,
                        void* stream) {
  if (int rc = img_args_ok(chw, hwc, B, C, H, W)) return rc;
  if (!(hi > lo)) return fail(nullptr, IRSDE_ERR_INVALID, "min_max must be increasing");
  launch_tensor2img(chw, hwc, B, C, H, W, lo, hi, (cudaStream_t)stream);
  return img_launch_status("tensor2img");
}
int irsde_img2tensor_u8(const uint8_t* hwc, float* chw, int32_t B, int32_t C, int32_t H, int32_t W, void* stream) {
  if (int rc = img_args_ok(hwc, chw, B, C, H, W)) return rc;
  launch_img2tensor(hwc, chw, B, C, H, W, (cudaStream_t)stream);
  return img_launch_status("img2tensor");
}
int irsde_sqerr_u8(const uint8_t* a, const uint8_t* b, int32_t B, int32_t H, int32_t W, int32_t C, int32_t crop, uint64_t* sums,
                   void* stream) {
  if (int rc = img_args_ok(a, b, B, C, H, W)) return rc;
  if (!sums || crop < 0 || H - 2 * crop < 1 || W - 2 * crop < 1) return fail(nullptr, IRSDE_ERR_INVALID, "bad crop / output");
  launch_sqerr_u8(a, b, B, H, W, C, crop, (unsigned long long*)sums, (cudaStream_t)stream);
  return img_launch_status("sqerr_u8");
}
int64_t irsde_ssim_workspace(int32_t B, int32_t H, int32_t W, int32_t C, int32_t crop) {
  if (B < 1 || crop < 0 || H - 2 * crop < 11 || W - 2 * crop < 11) return 0;
  return (int64_t)B * ssim_partial_count(H, W, C, crop);
}
int irsde_ssim_u8(const uint8_t* a, const uint8_t* b, int32_t B, int32_t H, int32_t W, int32_t C, int32_t crop, double* workspace,
                  double* ssim, void* stream) {
  if (int rc = img_args_ok(a, b, B, C, H, W)) return rc;
  if (!workspace || !ssim || crop < 0 || H - 2 * crop < 11 || W - 2 * crop < 11)
    return fail(nullptr, IRSDE_ERR_INVALID, "SSIM needs at least 11x11 pixels after cropping");
  launch_ssim_u8(a, b, B, H, W, C, crop, workspace, ssim, (cudaStream_t)stream);
  return img_launch_status("ssim_u8");
}

}  // extern "C"
