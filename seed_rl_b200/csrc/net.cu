// (a5) Policy network graph: dmlab/networks.py:63-171 ImpalaDeep (and the IMPALA-paper
// shallow net) as a fixed schedule of this library's kernels -- forward unroll
// (_torso folded over T*B by batch_apply, utils.py:714-732; LSTM over T with
// done-resets; heads) and the matching backward (what tf.GradientTape computes at
// agents/vtrace/learner.py:261-264).
//
// Parameters: one flat fp32 arena, tensors in tf.Module.trainable_variables order
// (_baseline, _conv_to_linear, _core, _policy_logits, _stacks...), Keras layouts,
// every tensor start aligned to 64 floats (256 B), then the scalar entropy_cost_param
// (learner.py:225-234).
#include <vector>

#include "kernels.h"

namespace seedrl {

constexpr int kHidden = 256;   // LSTMCell(256), Dense(256)

struct ConvLayer {
  int cin, cout;
  int w, b;        // param indices
};
struct Stack {
  int hin, win, cin, c, hout, wout;
  ConvLayer conv, r00, r01, r10, r11;
};

}  // namespace seedrl

struct seedrl_net {
  seedrl_net_config cfg;
  seedrl::ParamTable pt;                   // network tensors, then entropy_cost_param
  size_t logical_params;
  int p_base_w, p_base_b, p_dense_w, p_dense_b, p_core_w, p_core_u, p_core_b, p_pol_w, p_pol_b;
  std::vector<seedrl::Stack> stacks;       // deep
  seedrl::StridedConv sh[2];               // shallow: conv 8x8/4 -> 16, conv 4x4/2 -> 32
  int flat;                                // conv features fed to Dense(256)
  int lstm_mode = 2;                       // 2 = tiled persistent kernels (lstm_tiled.cu), 0 = per-step launches
  int conv_mode = 0;                       // 0 = fp32 SIMT, 1 = tcgen05 bf16, 2 = tcgen05 bf16x3 (fp32-faithful)
  int core_in;                             // 256 + 1 + A
};

namespace seedrl {

static ConvLayer add_conv(seedrl_net* n, const std::string& prefix, int k, int cin, int cout) {
  ConvLayer l;
  l.cin = cin; l.cout = cout;
  l.w = n->pt.add(prefix + "/kernel", {k, k, cin, cout});
  l.b = n->pt.add(prefix + "/bias", {cout});
  return l;
}

// ---- workspace plan -----------------------------------------------------------
struct StackBufs {
  size_t a0, p, idx, c0, o0, c1, o1;
  // conv_mode 3 (plane tensors, conv_planes.cu): raw / ReLU'd pooled activation, ReLU'd c0 / c1,
  // raw / ReLU'd o0, raw o1 (the last stack's o1 stays fp32 NHWC for the Dense layer)
  size_t praw, prelu, c0r, o0raw, o0relu, c1r, o1p;
};

// packed-weight slot: (hi + lo) x 9 x 32 x 32 bf16; deferred weight-gradient partials of all
// 15 convs: 148 CTAs x 97 680 floats (57.8 MB) rounded up
constexpr size_t kPackSlotBytes = 2 * 9 * 32 * 32 * 2;
constexpr size_t kPartialAllBytes = (size_t)64 << 20;

struct Plan {
  int N;                       // T1 * B frames
  std::vector<StackBufs> st;
  size_t sh_a1, sh_a2;         // shallow conv outputs (post-relu)
  size_t sh_col0, sh_col1;     // shallow net, tensor-core modes: im2col matrices (kept for the backward)
  LstmBufs lstm;
  // backward scratch
  size_t gA, gB, gC, gFull, wt, partial, wq, tcerr, counter, gemm_ws, wq_all, partial_all;
  size_t gP1, gP2, gP3, gFP;   // conv_mode 3: plane-tensor gradients (pooled resolution x3, full resolution)
  size_t obs4, w0pad, dw0pad;  // 3-channel frames: zero-padded frames / first-conv weights / their gradient
  size_t total;
};

static Plan make_plan(const seedrl_net* n, int T1, int B) {
  Plan p;
  Bump b;
  const size_t N = (size_t)T1 * B;
  p.N = (int)N;
  size_t pooled_max = 0, full_max = 0, pooled_planes_max = 0, full_planes_max = 0;
  const bool planes = n->conv_mode == 3 && n->cfg.net == SEEDRL_NET_DEEP;
  if (n->cfg.net == SEEDRL_NET_DEEP) {
    for (size_t si = 0; si < n->stacks.size(); ++si) {
      const Stack& s = n->stacks[si];
      StackBufs sb = StackBufs();
      const size_t full = N * s.hin * s.win * s.c, pooled = N * s.hout * s.wout * s.c;
      sb.a0 = b.take(full * 4);
      sb.idx = b.take(pooled);
      if (!planes) {
        sb.p = b.take(pooled * 4);
        sb.c0 = b.take(pooled * 4);
        sb.o0 = b.take(pooled * 4);
        sb.c1 = b.take(pooled * 4);
        sb.o1 = b.take(pooled * 4);
      } else {
        const size_t pb = planes_bytes((int)N, s.hout, s.wout, s.c);
        sb.praw = b.take(pb); sb.prelu = b.take(pb); sb.c0r = b.take(pb);
        sb.o0raw = b.take(pb); sb.o0relu = b.take(pb); sb.c1r = b.take(pb);
        if (si + 1 < n->stacks.size()) sb.o1p = b.take(pb); else sb.o1 = b.take(pooled * 4);
        if (pb > pooled_planes_max) pooled_planes_max = pb;
        if (si > 0) {
          const size_t fb = planes_bytes((int)N, s.hin, s.win, s.c);
          if (fb > full_planes_max) full_planes_max = fb;
        }
      }
      p.st.push_back(sb);
      if (pooled > pooled_max) pooled_max = pooled;
      if (full > full_max) full_max = full;
    }
    p.sh_a1 = p.sh_a2 = 0;
  } else {
    const StridedConv& c0 = n->sh[0];
    const StridedConv& c1 = n->sh[1];
    const size_t a1 = N * c0.hout * c0.wout * 16, a2 = N * c1.hout * c1.wout * 32;
    p.sh_a1 = b.take(a1 * 4);
    p.sh_a2 = b.take(a2 * 4);
    p.sh_col0 = p.sh_col1 = 0;
    if (n->conv_mode >= 1) {
      p.sh_col0 = b.take(N * c0.hout * c0.wout * (size_t)(64 * n->cfg.obs_c) * 4);
      p.sh_col1 = b.take(N * c1.hout * c1.wout * (size_t)(16 * 16) * 4);
    }
    pooled_max = a1 > a2 ? a1 : a2;
    full_max = 0;
  }
  p.lstm = lstm_bufs(&b, N, B, kHidden, n->core_in);
  p.obs4 = p.w0pad = p.dw0pad = 0;
  if (n->cfg.net == SEEDRL_NET_DEEP && n->cfg.obs_c == 3) {
    p.obs4 = b.take(N * n->cfg.obs_h * n->cfg.obs_w * 4);
    p.w0pad = b.take(9 * 4 * 16 * 4);
    p.dw0pad = b.take(9 * 4 * 16 * 4);
  }
  p.gA = b.take(pooled_max * 4);
  p.gB = p.gC = p.gP1 = p.gP2 = p.gP3 = p.gFP = 0;
  if (!planes) {
    p.gB = b.take(pooled_max * 4);
    p.gC = b.take(pooled_max * 4);
  } else {
    p.gP1 = b.take(pooled_planes_max);
    p.gP2 = b.take(pooled_planes_max);
    p.gP3 = b.take(pooled_planes_max);
    p.gFP = b.take(full_planes_max);
  }
  p.gFull = b.take(full_max * 4);
  p.wt = b.take(64 * 1024 * 4);
  p.wq = b.take(2 * 64 * 1024 * 2);
  p.gemm_ws = b.take(gemm_tc_workspace_bytes());
  p.wq_all = b.take((size_t)kMaxPackJobs * kPackSlotBytes);
  p.partial_all = b.take(kPartialAllBytes);
  p.tcerr = b.take(256);
  p.counter = b.take(256);
  p.partial = b.take(conv3x3_wgrad_partial_bytes());
  p.total = b.off;
  return p;
}

#define SEEDRL_TRY(expr) SEEDRL_TRY_RC(expr)

// 3-channel frames (DMLab's 72x96x3, dmlab/env.py:44-54): the first convolution's kernels are built
// for 4 input channels, so a forward/backward call works on a zero-padded copy of the frames and of
// the first conv's weights ([3,3,3,16] -> [3,3,4,16]); its weight gradient is computed in the padded
// shape and copied back without the 4th channel.  These thread-local overrides redirect the one
// parameter for the duration of a call.
static thread_local int t_w0_index = -1;
static thread_local const float* t_w0_pad = nullptr;
static thread_local float* t_dw0_pad = nullptr;
static inline const float* P(const seedrl_net* n, const float* arena, int idx) {
  if (idx == t_w0_index && t_w0_pad) return t_w0_pad;
  return n->pt.at(arena, idx);
}
static inline float* G(const seedrl_net* n, float* arena, int idx) {
  if (idx == t_w0_index && t_dw0_pad) return t_dw0_pad;
  return n->pt.at(arena, idx);
}

__global__ void pad_frames3_kernel(size_t npix, const uint8_t* __restrict__ src, uchar4* __restrict__ dst) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  dst[i] = make_uchar4(src[3 * i], src[3 * i + 1], src[3 * i + 2], 0);
}
// w[tap][3][co] <-> wp[tap][4][co]
__global__ void pad_w0_kernel(int cout, const float* __restrict__ w, float* __restrict__ wp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 9 * 4 * cout) return;
  const int co = i % cout, ci = (i / cout) % 4, tap = i / (4 * cout);
  wp[i] = ci < 3 ? w[(tap * 3 + ci) * cout + co] : 0.f;
}
__global__ void unpad_dw0_kernel(int cout, const float* __restrict__ dwp, float* __restrict__ dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 9 * 3 * cout) return;
  const int co = i % cout, ci = (i / cout) % 3, tap = i / (3 * cout);
  dw[i] = dwp[(tap * 4 + ci) * cout + co];
}
// The dense contractions of the schedule run on the tensor cores in every tensor-core conv mode.
static GemmRunner gemm_runner(const seedrl_net* n, void* ws, const Plan& pl) {
  return GemmRunner{n->conv_mode >= 1, n->conv_mode >= 2, W<float>(ws, pl.gemm_ws), W<int>(ws, pl.tcerr)};
}
static LstmCore net_lstm_core(const seedrl_net* n, void* ws, const Plan& pl, int T1, int B) {
  return lstm_core(kHidden, n->core_in, T1, B, n->lstm_mode == 2, pl.lstm, ws, W<unsigned int>(ws, pl.counter));
}

// Per-call context of the tensor-core path (thread-local: forward/backward of different nets
// may run on different host threads): where the pre-packed weights of this call live and the
// deferred weight-gradient reductions.
struct StepCtx {
  PackTable packed;
  WgradBatch wb;
};
static thread_local StepCtx* t_ctx = nullptr;
static thread_local void* t_head_ready = nullptr;   // cudaEvent_t recorded by seedrl_net_backward_overlap
// test hook: 1 = keep the dense (pool backward + full-resolution weight gradient) first-layer path
static int g_first_dense = 0;

// Packs the weights of every conv of the deep torso with one launch: forward forms, or the
// flipped/transposed forms of the data-gradient convolutions (all but the first layer).
static int pack_all_weights(const seedrl_net* n, const float* prm, void* ws, const Plan& pl, int flip,
                            StepCtx* ctx, cudaStream_t st) {
  ctx->packed.n = 0;
  if (n->conv_mode < 1 || n->cfg.net != SEEDRL_NET_DEEP) return SEEDRL_OK;
  char* base = W<char>(ws, pl.wq_all);
  for (size_t s = 0; s < n->stacks.size(); ++s) {
    const Stack& k = n->stacks[s];
    const ConvLayer* ls[5] = {&k.conv, &k.r00, &k.r01, &k.r10, &k.r11};
    for (int i = 0; i < 5; ++i) {
      const ConvLayer& l = *ls[i];
      if (flip && s == 0 && i == 0) continue;          // no data gradient into the frames
      const int cin = flip ? l.cout : l.cin, cout = flip ? l.cin : l.cout;
      if (ctx->packed.n >= kMaxPackJobs) return SEEDRL_OK;
      PackJob j;
      j.w = P(n, prm, l.w);
      j.wq = base + (size_t)ctx->packed.n * kPackSlotBytes;
      j.ck = cin < 16 ? 16 : cin; j.cout = cout; j.cin_src = cin; j.flip = flip;
      j.legacy = (s == 0 && i == 0) ? 1 : 0;           // the uint8 first conv runs the staged kernel
      ctx->packed.jobs[ctx->packed.n++] = j;
    }
  }
  return conv3x3_tc_pack_weights_batch(ctx->packed, n->conv_mode == 3 ? 2 : (n->conv_mode >= 2 ? 1 : 0), st);
}
static const void* find_packed(const float* w, int flip) {
  if (!t_ctx) return nullptr;
  for (int i = 0; i < t_ctx->packed.n; ++i)
    if (t_ctx->packed.jobs[i].w == w && t_ctx->packed.jobs[i].flip == flip) return t_ctx->packed.jobs[i].wq;
  return nullptr;
}

// One 3x3 'same' convolution of the schedule.  flip != 0: data-gradient (weights flipped and
// transposed; cin/cout are those of the *gradient* convolution).  Dispatches to the tcgen05
// kernel when the net runs in tensor-core mode and the shape is supported, else fp32 SIMT.
static int run_conv(const seedrl_net* n, void* ws, const Plan& pl, int cin, int cout, int in_mode,
                    int N, int H, int Wd, const void* in, const float* w, const float* bias,
                    const float* mask, const float* res, float* out, int flip, cudaStream_t st) {
  if (n->conv_mode >= 1 && conv3x3_tc_supported(cin, cout, in_mode)) {
    const int split = n->conv_mode >= 2;
    const void* wq = find_packed(w, flip);
    if (!wq) {
      void* scratch = W<void>(ws, pl.wq);
      SEEDRL_TRY(conv3x3_tc_pack_weights(cin, cout, flip, split, w, scratch, st));
      wq = scratch;
    }
    return conv3x3_tc_forward(cin, cout, in_mode, split, N, H, Wd, in, wq, bias, mask, res, out, 0,
                              W<int>(ws, pl.tcerr), st);
  }
  if (flip) {
    float* wt = W<float>(ws, pl.wt);
    SEEDRL_TRY(conv3x3_flip_weights(cout, cin, w, wt, st));   // source layout is [tap][cout][cin]
    return conv3x3_forward(cin, cout, in_mode, N, H, Wd, in, wt, bias, mask, res, out, st);
  }
  return conv3x3_forward(cin, cout, in_mode, N, H, Wd, in, w, bias, mask, res, out, st);
}

// Scope of one forward/backward call on 3-channel frames: builds the padded frames and first-conv
// weights in the workspace and installs the parameter overrides; no-op for 4-channel frames.
struct PadScope {
  int rc = SEEDRL_OK;
  bool active = false;
  const uint8_t* obs;
  PadScope(const seedrl_net* n, const float* prm, const Plan& pl, const uint8_t* observation, void* ws,
           cudaStream_t st) : obs(observation) {
    if (n->cfg.net != SEEDRL_NET_DEEP || n->cfg.obs_c != 3) return;
    active = true;
    const size_t npix = (size_t)pl.N * n->cfg.obs_h * n->cfg.obs_w;
    pad_frames3_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(npix, observation, W<uchar4>(ws, pl.obs4));
    count_launch(PC_MISC, st);
    const int wi = n->stacks[0].conv.w;
    pad_w0_kernel<<<ceil_div(9 * 4 * 16, 128), 128, 0, st>>>(16, n->pt.at(prm, wi), W<float>(ws, pl.w0pad));
    count_launch(PC_MISC, st);
    if (cudaGetLastError() != cudaSuccess) rc = set_error(SEEDRL_ERR_INTERNAL, "3-channel padding launch failed");
    obs = W<uint8_t>(ws, pl.obs4);
    t_w0_index = wi; t_w0_pad = W<float>(ws, pl.w0pad); t_dw0_pad = W<float>(ws, pl.dw0pad);
  }
  ~PadScope() { t_w0_index = -1; t_w0_pad = nullptr; t_dw0_pad = nullptr; }
};

}  // namespace seedrl

using namespace seedrl;

extern "C" int seedrl_net_create(const seedrl_net_config* cfg, seedrl_net** out) {
  SEEDRL_CHECK_ARG(cfg && out, "null pointer");
  SEEDRL_CHECK_ARG(cfg->net == SEEDRL_NET_DEEP || cfg->net == SEEDRL_NET_SHALLOW, "unknown net");
  SEEDRL_CHECK_ARG(cfg->num_actions >= 1 && cfg->obs_h > 0 && cfg->obs_w > 0, "bad shape");
  seedrl_net* n = new seedrl_net();
  n->cfg = *cfg;
  const int A = cfg->num_actions;
  n->core_in = kHidden + 1 + A;
  // tf.Module order: _baseline, _conv_to_linear, _core, _policy_logits, _stacks
  n->p_base_w = n->pt.add("baseline/kernel", {kHidden, 1});
  n->p_base_b = n->pt.add("baseline/bias", {1});
  int flat = 0;
  if (cfg->net == SEEDRL_NET_DEEP) {
    if (cfg->obs_c != 4 && cfg->obs_c != 3) {
      delete n;
      return set_error(SEEDRL_ERR_INVALID_ARGUMENT,
                       "seedrl_net_create: the deep net takes 3- or 4-channel uint8 frames");
    }
    int h = cfg->obs_h, w = cfg->obs_w;
    const int chans[3] = {16, 32, 32};
    for (int s = 0; s < 3; ++s) { h = (h + 1) / 2; w = (w + 1) / 2; }
    flat = h * w * chans[2];
  } else {
    n->sh[0] = strided_conv(8, 4, cfg->obs_c, 16, cfg->obs_h, cfg->obs_w);
    n->sh[1] = strided_conv(4, 2, 16, 32, n->sh[0].hout, n->sh[0].wout);
    flat = n->sh[1].hout * n->sh[1].wout * 32;
  }
  n->flat = flat;
  n->p_dense_w = n->pt.add("conv_to_linear/kernel", {flat, kHidden});
  n->p_dense_b = n->pt.add("conv_to_linear/bias", {kHidden});
  n->p_core_w = n->pt.add("core/kernel", {n->core_in, 4 * kHidden});
  n->p_core_u = n->pt.add("core/recurrent_kernel", {kHidden, 4 * kHidden});
  n->p_core_b = n->pt.add("core/bias", {4 * kHidden});
  n->p_pol_w = n->pt.add("policy_logits/kernel", {kHidden, A});
  n->p_pol_b = n->pt.add("policy_logits/bias", {A});
  if (cfg->net == SEEDRL_NET_DEEP) {
    int h = cfg->obs_h, w = cfg->obs_w, c = cfg->obs_c;
    const int chans[3] = {16, 32, 32};
    for (int s = 0; s < 3; ++s) {
      Stack st;
      const std::string pre = "stack" + std::to_string(s);
      st.hin = h; st.win = w; st.cin = (s == 0 && c == 3) ? 4 : c; st.c = chans[s];
      st.hout = (h + 1) / 2; st.wout = (w + 1) / 2;
      st.conv = add_conv(n, pre + "/conv", 3, c, st.c);      // the parameter keeps the frame's channel count
      st.conv.cin = st.cin;                                  // ... the kernels see the padded one
      // tf.Module order inside _Stack: _conv, _res_convs0[0..1], _res_convs1[0..1]
      st.r00 = add_conv(n, pre + "/res_0/conv2d_0", 3, st.c, st.c);
      st.r10 = add_conv(n, pre + "/res_1/conv2d_0", 3, st.c, st.c);
      st.r01 = add_conv(n, pre + "/res_0/conv2d_1", 3, st.c, st.c);
      st.r11 = add_conv(n, pre + "/res_1/conv2d_1", 3, st.c, st.c);
      n->stacks.push_back(st);
      h = st.hout; w = st.wout; c = st.c;
    }
  } else {
    for (int i = 0; i < 2; ++i) {
      const ConvLayer l = add_conv(n, "conv" + std::to_string(i), n->sh[i].k, n->sh[i].cin, n->sh[i].cout);
      n->sh[i].w = l.w; n->sh[i].b = l.b;
    }
  }
  n->logical_params = 0;
  for (const ParamInfo& p : n->pt.params) n->logical_params += p.size;
  n->pt.add("entropy_cost_param", {});
  *out = n;
  return SEEDRL_OK;
}

extern "C" void seedrl_net_destroy(seedrl_net* net) { delete net; }
extern "C" int seedrl_net_num_param_tensors(const seedrl_net* net) {
  return net ? (int)net->pt.params.size() - 1 : 0;
}
extern "C" size_t seedrl_net_num_params(const seedrl_net* net) { return net ? net->logical_params : 0; }
extern "C" size_t seedrl_net_arena_floats(const seedrl_net* net) { return net ? net->pt.arena_floats : 0; }
extern "C" int seedrl_net_set_lstm_mode(seedrl_net* net, int mode) {
  SEEDRL_CHECK_ARG(net && (mode == 0 || mode == 2),
                   "mode must be 0 (per-step launches) or 2 (persistent, CTA = batch tile x 16 units)");
  net->lstm_mode = mode;
  return SEEDRL_OK;
}
extern "C" int seedrl_net_set_conv_mode(seedrl_net* net, int mode) {
  SEEDRL_CHECK_ARG(net && mode >= 0 && mode <= 3,
                   "mode must be 0 (fp32 SIMT), 1 (tcgen05 bf16), 2 (tcgen05 bf16x3) or 3 (bf16x3 plane tensors)");
  SEEDRL_CHECK_ARG(mode != 3 || net->cfg.net == SEEDRL_NET_DEEP, "mode 3 is built for the deep net");
  net->conv_mode = mode;
  return SEEDRL_OK;
}

extern "C" int seedrl_net_param_info(const seedrl_net* net, int index, char* name_buf,
                                     size_t name_buf_len, int64_t* dims, size_t* offset) {
  return net ? net->pt.info(index, name_buf, name_buf_len, dims, offset) : -1;
}

extern "C" size_t seedrl_net_workspace_bytes(const seedrl_net* net, int T1, int B) {
  if (!net || T1 <= 0 || B <= 0) return 0;
  return make_plan(net, T1, B).total;
}

// ---- forward --------------------------------------------------------------------
static int torso_forward_deep(const seedrl_net* n, const float* prm, const Plan& pl,
                              const uint8_t* obs, void* ws, cudaStream_t st) {
  const int N = pl.N;
  const void* in = obs;
  int in_mode = IN_U8;
  for (size_t s = 0; s < n->stacks.size(); ++s) {
    const Stack& k = n->stacks[s];
    const StackBufs& b = pl.st[s];
    float* a0 = W<float>(ws, b.a0); float* p = W<float>(ws, b.p);
    float* c0 = W<float>(ws, b.c0); float* o0 = W<float>(ws, b.o0);
    float* c1 = W<float>(ws, b.c1); float* o1 = W<float>(ws, b.o1);
    // _Stack.__call__, dmlab/networks.py:46-60
    SEEDRL_TRY(run_conv(n, ws, pl, k.cin, k.c, in_mode, N, k.hin, k.win, in, P(n, prm, k.conv.w),
                        P(n, prm, k.conv.b), nullptr, nullptr, a0, 0, st));
    SEEDRL_TRY(maxpool3s2_forward(N, k.hin, k.win, k.c, a0, p, W<uint8_t>(ws, b.idx), st));
    SEEDRL_TRY(run_conv(n, ws, pl, k.c, k.c, IN_RELU, N, k.hout, k.wout, p, P(n, prm, k.r00.w),
                        P(n, prm, k.r00.b), nullptr, nullptr, c0, 0, st));
    SEEDRL_TRY(run_conv(n, ws, pl, k.c, k.c, IN_RELU, N, k.hout, k.wout, c0, P(n, prm, k.r01.w),
                        P(n, prm, k.r01.b), nullptr, p, o0, 0, st));
    SEEDRL_TRY(run_conv(n, ws, pl, k.c, k.c, IN_RELU, N, k.hout, k.wout, o0, P(n, prm, k.r10.w),
                        P(n, prm, k.r10.b), nullptr, nullptr, c1, 0, st));
    SEEDRL_TRY(run_conv(n, ws, pl, k.c, k.c, IN_RELU, N, k.hout, k.wout, c1, P(n, prm, k.r11.w),
                        P(n, prm, k.r11.b), nullptr, o0, o1, 0, st));
    in = o1;
    in_mode = IN_F32;
  }
  return SEEDRL_OK;
}

// conv_mode 3: the same _Stack schedule on plane tensors (conv_planes.cu).  The first conv reads the
// uint8 frames with the staged tcgen05 kernel (bf16x3) and writes fp32 NHWC for the max-pool; from
// there on every conv input is a TMA tile of an HBM-resident operand.
static int planes_conv(const seedrl_net* n, void* ws, const Plan& pl, int cin, int cout, int N, int H, int Wd,
                       const void* in, const float* w, int flip, const float* bias, const void* mask,
                       const void* res, void* out_raw, void* out_relu, float* out_nhwc, cudaStream_t st) {
  const void* wq = find_packed(w, flip);
  if (!wq) {
    void* scratch = W<void>(ws, pl.wq);
    SEEDRL_TRY(conv3x3_tc_pack_weights(cin, cout, flip, 2, w, scratch, st));
    wq = scratch;
  }
  PlaneConv c;
  c.N = N; c.H = H; c.W = Wd; c.in = in; c.wq = wq; c.bias = bias; c.mask = mask; c.res = res;
  c.out_raw = out_raw; c.out_relu = out_relu; c.out_nhwc = out_nhwc; c.err = W<int>(ws, pl.tcerr);
  return convp_forward(cin, cout, c, st);
}

static int torso_forward_planes(const seedrl_net* n, const float* prm, const Plan& pl,
                                const uint8_t* obs, void* ws, cudaStream_t st) {
  const int N = pl.N;
  const void* prev = nullptr;
  const size_t ns = n->stacks.size();
  for (size_t s = 0; s < ns; ++s) {
    const Stack& k = n->stacks[s];
    const StackBufs& b = pl.st[s];
    float* a0 = W<float>(ws, b.a0);
    void* praw = W<void>(ws, b.praw); void* prelu = W<void>(ws, b.prelu);
    void* c0r = W<void>(ws, b.c0r); void* o0raw = W<void>(ws, b.o0raw);
    void* o0relu = W<void>(ws, b.o0relu); void* c1r = W<void>(ws, b.c1r);
    const bool last = s + 1 == ns;
    if (s == 0 && conv0pool_supported(k.cin, k.c, k.hin, k.win) && !g_first_dense) {
      // first conv + bias + max-pool in one kernel: the full-resolution activation never reaches HBM
      SEEDRL_TRY(conv0pool_forward(N, k.hin, k.win, obs, P(n, prm, k.conv.w), P(n, prm, k.conv.b), praw, prelu,
                                   W<uint8_t>(ws, b.idx), W<int>(ws, pl.tcerr), st));
    } else {
      if (s == 0)
        SEEDRL_TRY(run_conv(n, ws, pl, k.cin, k.c, IN_U8, N, k.hin, k.win, obs, P(n, prm, k.conv.w),
                            P(n, prm, k.conv.b), nullptr, nullptr, a0, 0, st));
      else
        SEEDRL_TRY(planes_conv(n, ws, pl, k.cin, k.c, N, k.hin, k.win, prev, P(n, prm, k.conv.w), 0,
                               P(n, prm, k.conv.b), nullptr, nullptr, nullptr, nullptr, a0, st));
      SEEDRL_TRY(poolp_forward(N, k.hin, k.win, k.c, a0, praw, prelu, W<uint8_t>(ws, b.idx), st));
    }
    const int H = k.hout, Wd = k.wout, C = k.c;
    // res block 0: c0 = conv00(relu(p)); o0 = conv01(relu(c0)) + p        (networks.py:52-58)
    SEEDRL_TRY(planes_conv(n, ws, pl, C, C, N, H, Wd, prelu, P(n, prm, k.r00.w), 0, P(n, prm, k.r00.b), nullptr,
                           nullptr, nullptr, c0r, nullptr, st));
    SEEDRL_TRY(planes_conv(n, ws, pl, C, C, N, H, Wd, c0r, P(n, prm, k.r01.w), 0, P(n, prm, k.r01.b), nullptr,
                           praw, o0raw, o0relu, nullptr, st));
    // res block 1: c1 = conv10(relu(o0)); o1 = conv11(relu(c1)) + o0
    SEEDRL_TRY(planes_conv(n, ws, pl, C, C, N, H, Wd, o0relu, P(n, prm, k.r10.w), 0, P(n, prm, k.r10.b), nullptr,
                           nullptr, nullptr, c1r, nullptr, st));
    SEEDRL_TRY(planes_conv(n, ws, pl, C, C, N, H, Wd, c1r, P(n, prm, k.r11.w), 0, P(n, prm, k.r11.b), nullptr,
                           o0raw, last ? nullptr : W<void>(ws, b.o1p), nullptr,
                           last ? W<float>(ws, b.o1) : nullptr, st));
    prev = W<void>(ws, b.o1p);
  }
  return SEEDRL_OK;
}

// Shallow net: layer 0 = conv 8x8/4 on the uint8 frames, layer 1 = conv 4x4/2 on a1.
static int torso_forward_shallow(const seedrl_net* n, const float* prm, const Plan& pl,
                                 const uint8_t* obs, void* ws, cudaStream_t st) {
  const int N = pl.N;
  const StridedConv& c0 = n->sh[0];
  const StridedConv& c1 = n->sh[1];
  float* a1 = W<float>(ws, pl.sh_a1);
  float* a2 = W<float>(ws, pl.sh_a2);
  if (n->conv_mode >= 1 && n->cfg.obs_c % 4 == 0) {
    // tensor-core modes: GEMMs over the im2col matrices, bias + ReLU in the epilogue (as the R2D2 body)
    const GemmRunner g = gemm_runner(n, ws, pl);
    SEEDRL_TRY(strided_conv_forward(g, N, c0, true, obs, P(n, prm, c0.w), P(n, prm, c0.b), W<float>(ws, pl.sh_col0),
                                    a1, st));
    return strided_conv_forward(g, N, c1, false, a1, P(n, prm, c1.w), P(n, prm, c1.b), W<float>(ws, pl.sh_col1), a2,
                                st);
  }
  SEEDRL_TRY(convgen_forward(N, c0.hin, c0.win, c0.cin, 16, 8, 4, 1, obs, P(n, prm, c0.w), P(n, prm, c0.b), 1, a1,
                             st));
  SEEDRL_TRY(convgen_forward(N, c1.hin, c1.win, 16, 32, 4, 2, 0, a1, P(n, prm, c1.w), P(n, prm, c1.b), 1, a2, st));
  return SEEDRL_OK;
}

extern "C" int seedrl_net_forward(const seedrl_net* n, const float* prm, int T1, int B,
                                  const int64_t* prev_actions, const float* reward,
                                  const uint8_t* done, const uint8_t* observation,
                                  const float* h0, const float* c0, float* policy_logits,
                                  float* baseline, float* h_out, float* c_out, void* ws,
                                  size_t ws_bytes, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(n && prm && prev_actions && reward && done && observation && h0 && c0 &&
                       policy_logits && baseline && ws, "null pointer");
  SEEDRL_CHECK_ARG(T1 >= 1 && B >= 1, "T1, B must be >= 1");
  const Plan pl = make_plan(n, T1, B);
  SEEDRL_CHECK_ARG(ws_bytes >= pl.total, "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = pl.N, A = n->cfg.num_actions, CI = n->core_in;
  // bounded-wait error flag of the tcgen05 / persistent kernels: cleared here, set by any kernel of
  // this forward or the matching backward, read back by seedrl_net_check_error
  SEEDRL_CUDA(cudaMemsetAsync(W<int>(ws, pl.tcerr), 0, sizeof(int), st));
  const float* flat_src;
  int flat_relu;
  if (n->cfg.net == SEEDRL_NET_DEEP) {
    StepCtx ctx;
    ctx.wb = WgradBatch{nullptr, 0, 0, 0, {}};
    PadScope pad(n, prm, pl, observation, ws, st);
    SEEDRL_TRY(pad.rc);
    observation = pad.obs;
    SEEDRL_TRY(pack_all_weights(n, prm, ws, pl, 0, &ctx, st));
    t_ctx = &ctx;
    const int rc_t = n->conv_mode == 3 ? torso_forward_planes(n, prm, pl, observation, ws, st)
                                       : torso_forward_deep(n, prm, pl, observation, ws, st);
    t_ctx = nullptr;
    SEEDRL_TRY(rc_t);
    flat_src = W<float>(ws, pl.st.back().o1);
    flat_relu = 1;                         // tf.nn.relu before Flatten, networks.py:105
  } else {
    SEEDRL_TRY(torso_forward_shallow(n, prm, pl, observation, ws, st));
    flat_src = W<float>(ws, pl.sh_a2);
    flat_relu = 0;                         // already relu'd
  }
  const GemmRunner g = gemm_runner(n, ws, pl);
  const LstmCore core = net_lstm_core(n, ws, pl, T1, B);
  float* xc = core.xc;
  float* hs = core.hs;
  float* cs = core.cs;
  // Dense(256) + relu written straight into the first 256 columns of the core input
  GemmEpi e = epi_none();
  e.bias = P(n, prm, n->p_dense_b); e.relu = 1; e.a_relu = flat_relu;
  SEEDRL_TRY(g.gemm(false, false, N, kHidden, n->flat, flat_src, n->flat, P(n, prm, n->p_dense_w), kHidden, xc, CI,
                    e, st));
  SEEDRL_TRY(core_input_tail(N, kHidden, A, reward, prev_actions, xc, st));
  SEEDRL_TRY(lstm_core_forward(g, core, P(n, prm, n->p_core_w), P(n, prm, n->p_core_u), P(n, prm, n->p_core_b), done,
                               h0, c0, st));
  // heads, networks.py:116-118
  e = epi_none();
  e.bias = P(n, prm, n->p_pol_b);
  SEEDRL_TRY(g.gemm(false, false, N, A, kHidden, hs, kHidden, P(n, prm, n->p_pol_w), A, policy_logits, A, e, st));
  e.bias = P(n, prm, n->p_base_b);
  SEEDRL_TRY(g.gemm(false, false, N, 1, kHidden, hs, kHidden, P(n, prm, n->p_base_w), 1, baseline, 1, e, st));
  if (h_out)
    SEEDRL_CUDA(cudaMemcpyAsync(h_out, hs + (size_t)(T1 - 1) * B * kHidden, (size_t)B * kHidden * 4,
                                cudaMemcpyDeviceToDevice, st));
  if (c_out)
    SEEDRL_CUDA(cudaMemcpyAsync(c_out, cs + (size_t)(T1 - 1) * B * kHidden, (size_t)B * kHidden * 4,
                                cudaMemcpyDeviceToDevice, st));
  return SEEDRL_OK;
}

// Reads back the device-side error flag of the last forward/backward that used this workspace
// (set when a bounded mbarrier / grid-barrier wait of a tcgen05 or persistent kernel expired, i.e.
// the results are garbage).  Synchronises `stream`.
extern "C" int seedrl_net_check_error(const seedrl_net* n, int T1, int B, void* ws, size_t ws_bytes,
                                      seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(n && ws && T1 >= 1 && B >= 1, "bad arguments");
  const Plan pl = make_plan(n, T1, B);
  SEEDRL_CHECK_ARG(ws_bytes >= pl.total, "workspace too small");
  return read_error_flag(W<int>(ws, pl.tcerr), (cudaStream_t)stream);
}

// ---- backward -------------------------------------------------------------------
static int conv_bwd(const seedrl_net* n, const float* prm, float* grd, const ConvLayer& l, int N,
                    int H, int Wd, const void* x, int x_mode, const float* dy, const float* dmask,
                    const float* dres, float* dx, void* ws, const Plan& pl, cudaStream_t st) {
  // weight + bias gradient
  if (n->conv_mode >= 1 && conv3x3_wgrad_tc_supported(l.cin, l.cout, x_mode)) {
    SEEDRL_TRY(conv3x3_wgrad_tc(l.cin, l.cout, x_mode, n->conv_mode >= 2, N, H, Wd, x, dy,
                                G(n, grd, l.w), G(n, grd, l.b), W<float>(ws, pl.partial),
                                conv3x3_wgrad_partial_bytes(), W<int>(ws, pl.tcerr),
                                t_ctx ? &t_ctx->wb : nullptr, st));
  } else {
    SEEDRL_TRY(conv3x3_wgrad(l.cin, l.cout, x_mode, N, H, Wd, x, dy, G(n, grd, l.w), G(n, grd, l.b),
                             W<float>(ws, pl.partial), conv3x3_wgrad_partial_bytes(), st));
  }
  if (dx) {  // data gradient = conv with flipped, transposed weights
    g_conv_cat = PC_CONV_DGRAD;
    const int rc = run_conv(n, ws, pl, l.cout, l.cin, IN_F32, N, H, Wd, dy, P(n, prm, l.w), nullptr,
                            dmask, dres, dx, 1, st);
    g_conv_cat = PC_CONV_FWD;
    SEEDRL_TRY(rc);
  }
  return SEEDRL_OK;
}

static int torso_backward_deep(const seedrl_net* n, const float* prm, float* grd, const Plan& pl,
                               const uint8_t* obs, void* ws, cudaStream_t st) {
  // On entry gA holds d loss / d o1 of the last stack.
  const int N = pl.N;
  float* gA = W<float>(ws, pl.gA); float* gB = W<float>(ws, pl.gB);
  float* gC = W<float>(ws, pl.gC); float* gF = W<float>(ws, pl.gFull);
  for (int s = (int)n->stacks.size() - 1; s >= 0; --s) {
    const Stack& k = n->stacks[s];
    const StackBufs& b = pl.st[s];
    const float* p = W<float>(ws, b.p);  const float* c0 = W<float>(ws, b.c0);
    const float* o0 = W<float>(ws, b.o0); const float* c1 = W<float>(ws, b.c1);
    const int H = k.hout, Wd = k.wout;
    // block 1: o1 = conv11(relu(c1)) + o0 ; c1 = conv10(relu(o0))
    SEEDRL_TRY(conv_bwd(n, prm, grd, k.r11, N, H, Wd, c1, IN_RELU, gA, c1, nullptr, gB, ws, pl, st));
    SEEDRL_TRY(conv_bwd(n, prm, grd, k.r10, N, H, Wd, o0, IN_RELU, gB, o0, gA, gC, ws, pl, st));
    // block 0: o0 = conv01(relu(c0)) + p ; c0 = conv00(relu(p))
    SEEDRL_TRY(conv_bwd(n, prm, grd, k.r01, N, H, Wd, c0, IN_RELU, gC, c0, nullptr, gB, ws, pl, st));
    SEEDRL_TRY(conv_bwd(n, prm, grd, k.r00, N, H, Wd, p, IN_RELU, gB, p, gC, gA, ws, pl, st));
    // max-pool, then the stack's first conv
    SEEDRL_TRY(maxpool3s2_backward(N, k.hin, k.win, k.c, gA, W<uint8_t>(ws, b.idx), gF, st));
    const void* x = s == 0 ? (const void*)obs : (const void*)W<float>(ws, pl.st[s - 1].o1);
    SEEDRL_TRY(conv_bwd(n, prm, grd, k.conv, N, k.hin, k.win, x, s == 0 ? IN_U8 : IN_F32, gF, nullptr,
                        nullptr, s == 0 ? nullptr : gA, ws, pl, st));
  }
  return SEEDRL_OK;
}

// conv_mode 3 backward: every gradient between the Dense layer and the first conv is a plane tensor.
static int planes_conv_bwd(const seedrl_net* n, const float* prm, float* grd, const ConvLayer& l, int N, int H,
                           int Wd, const void* x, const void* dy, const void* dmask, const void* dres,
                           void* dx, void* ws, const Plan& pl, cudaStream_t st) {
  SEEDRL_TRY(wgradp(l.cin, l.cout, N, H, Wd, x, dy, G(n, grd, l.w), G(n, grd, l.b), W<int>(ws, pl.tcerr),
                    t_ctx ? &t_ctx->wb : nullptr, st));
  if (dx) {
    g_conv_cat = PC_CONV_DGRAD;
    const int rc = planes_conv(n, ws, pl, l.cout, l.cin, N, H, Wd, dy, P(n, prm, l.w), 1, nullptr, dmask, dres,
                               dx, nullptr, nullptr, st);
    g_conv_cat = PC_CONV_FWD;
    SEEDRL_TRY(rc);
  }
  return SEEDRL_OK;
}

static int torso_backward_planes(const seedrl_net* n, const float* prm, float* grd, const Plan& pl,
                                 const uint8_t* obs, void* ws, cudaStream_t st) {
  // On entry gA (fp32 NHWC) holds d loss / d o1 of the last stack.
  const int N = pl.N;
  void* g1 = W<void>(ws, pl.gP1); void* g2 = W<void>(ws, pl.gP2); void* g3 = W<void>(ws, pl.gP3);
  void* gfp = W<void>(ws, pl.gFP); float* gF = W<float>(ws, pl.gFull);
  {
    const Stack& k = n->stacks.back();
    SEEDRL_TRY(to_planes(N, k.hout, k.wout, k.c, 0, W<float>(ws, pl.gA), g1, st));
  }
  for (int s = (int)n->stacks.size() - 1; s >= 0; --s) {
    const Stack& k = n->stacks[s];
    const StackBufs& b = pl.st[s];
    const int H = k.hout, Wd = k.wout;
    const void* prelu = W<void>(ws, b.prelu); const void* c0r = W<void>(ws, b.c0r);
    const void* o0relu = W<void>(ws, b.o0relu); const void* c1r = W<void>(ws, b.c1r);
    // block 1: o1 = conv11(relu(c1)) + o0 ; c1 = conv10(relu(o0))
    SEEDRL_TRY(planes_conv_bwd(n, prm, grd, k.r11, N, H, Wd, c1r, g1, c1r, nullptr, g2, ws, pl, st));
    SEEDRL_TRY(planes_conv_bwd(n, prm, grd, k.r10, N, H, Wd, o0relu, g2, o0relu, g1, g3, ws, pl, st));
    // block 0: o0 = conv01(relu(c0)) + p ; c0 = conv00(relu(p))
    SEEDRL_TRY(planes_conv_bwd(n, prm, grd, k.r01, N, H, Wd, c0r, g3, c0r, nullptr, g2, ws, pl, st));
    SEEDRL_TRY(planes_conv_bwd(n, prm, grd, k.r00, N, H, Wd, prelu, g2, prelu, g3, g1, ws, pl, st));
    // max-pool, then the stack's first conv
    if (s == 0 && t_ctx && first_wgrad_pooled_supported(k.cin, k.c, k.hin, k.win) && !g_first_dense) {
      // no gradient flows into the frames: the weight gradient is taken straight from the pooled
      // gradient and the pool's arg-max taps (conv_first.cu), the full-resolution tensor never exists
      SEEDRL_TRY(first_wgrad_pooled(N, k.hin, k.win, obs, g1, W<uint8_t>(ws, b.idx), G(n, grd, k.conv.w),
                                    G(n, grd, k.conv.b), &t_ctx->wb, st));
    } else if (s == 0) {
      SEEDRL_TRY(poolp_backward(N, k.hin, k.win, k.c, g1, W<uint8_t>(ws, b.idx), nullptr, gF, st));
      SEEDRL_TRY(conv_bwd(n, prm, grd, k.conv, N, k.hin, k.win, obs, IN_U8, gF, nullptr, nullptr, nullptr, ws, pl,
                          st));
    } else {
      SEEDRL_TRY(poolp_backward(N, k.hin, k.win, k.c, g1, W<uint8_t>(ws, b.idx), gfp, nullptr, st));
      SEEDRL_TRY(planes_conv_bwd(n, prm, grd, k.conv, N, k.hin, k.win, W<void>(ws, pl.st[s - 1].o1p), gfp, nullptr,
                                 nullptr, g1, ws, pl, st));
    }
  }
  return SEEDRL_OK;
}

static int torso_backward_shallow(const seedrl_net* n, const float* prm, float* grd, const Plan& pl,
                                  const uint8_t* obs, void* ws, cudaStream_t st) {
  // On entry gA holds d loss / d a2 (already masked by a2 > 0).
  const int N = pl.N;
  const StridedConv& c0 = n->sh[0];
  const StridedConv& c1 = n->sh[1];
  float* gA = W<float>(ws, pl.gA); float* gB = W<float>(ws, pl.gB);
  const float* a1 = W<float>(ws, pl.sh_a1);
  if (n->conv_mode >= 1 && n->cfg.obs_c % 4 == 0) {
    const GemmRunner g = gemm_runner(n, ws, pl);
    SEEDRL_TRY(strided_conv_backward(g, N, c1, false, a1, W<float>(ws, pl.sh_col1), P(n, prm, c1.w), gA,
                                     G(n, grd, c1.w), G(n, grd, c1.b), gB, st));
    return strided_conv_backward(g, N, c0, true, obs, W<float>(ws, pl.sh_col0), P(n, prm, c0.w), gB, G(n, grd, c0.w),
                                 G(n, grd, c0.b), nullptr, st);
  }
  SEEDRL_TRY(convgen_wgrad(N, c1.hin, c1.win, 16, 32, 4, 2, 0, a1, gA, G(n, grd, c1.w), G(n, grd, c1.b),
                           W<float>(ws, pl.partial), conv3x3_wgrad_partial_bytes(), st));
  SEEDRL_TRY(convgen_dgrad(N, c1.hin, c1.win, 16, 32, 4, 2, gA, P(n, prm, c1.w), a1, gB, st));
  SEEDRL_TRY(convgen_wgrad(N, c0.hin, c0.win, c0.cin, 16, 8, 4, 1, obs, gB, G(n, grd, c0.w), G(n, grd, c0.b),
                           W<float>(ws, pl.partial), conv3x3_wgrad_partial_bytes(), st));
  return SEEDRL_OK;
}

extern "C" int seedrl_net_backward(const seedrl_net* n, const float* prm, int T1, int B,
                                   const int64_t* prev_actions, const float* reward,
                                   const uint8_t* done, const uint8_t* observation,
                                   const float* dlogits, const float* dbaseline, float* grd,
                                   void* ws, size_t ws_bytes, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(n && prm && done && observation && dlogits && dbaseline && grd && ws,
                   "null pointer");
  (void)prev_actions; (void)reward;
  const Plan pl = make_plan(n, T1, B);
  SEEDRL_CHECK_ARG(ws_bytes >= pl.total, "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = pl.N, A = n->cfg.num_actions;
  const GemmRunner g = gemm_runner(n, ws, pl);
  const LstmCore core = net_lstm_core(n, ws, pl, T1, B);
  float* hs = core.hs;
  float* dhs = core.dhs;
  float* dd = core.dd;
  // padding floats and the entropy_cost_param slot must not carry garbage into Adam / all-reduce
  SEEDRL_CUDA(cudaMemsetAsync(grd, 0, n->pt.arena_floats * sizeof(float), st));

  // heads
  GemmEpi e = epi_none();
  SEEDRL_TRY(g.gemm(true, false, kHidden, A, N, hs, kHidden, dlogits, A, G(n, grd, n->p_pol_w), A, e, st));
  SEEDRL_TRY(g.colsum(N, A, dlogits, A, G(n, grd, n->p_pol_b), st));
  SEEDRL_TRY(g.gemm(true, false, kHidden, 1, N, hs, kHidden, dbaseline, 1, G(n, grd, n->p_base_w), 1, e, st));
  SEEDRL_TRY(g.colsum(N, 1, dbaseline, 1, G(n, grd, n->p_base_b), st));
  SEEDRL_TRY(g.gemm(false, true, N, kHidden, A, dlogits, A, P(n, prm, n->p_pol_w), A, dhs, kHidden, e, st));
  GemmEpi eacc = epi_none();
  eacc.accumulate = 1;
  SEEDRL_TRY(g.gemm(false, true, N, kHidden, 1, dbaseline, 1, P(n, prm, n->p_base_w), 1, dhs, kHidden, eacc, st));
  SEEDRL_TRY(lstm_core_backward(g, core, P(n, prm, n->p_core_w), P(n, prm, n->p_core_u), done, G(n, grd, n->p_core_w),
                                G(n, grd, n->p_core_u), G(n, grd, n->p_core_b), st));
  // Dense(256)
  const float* flat_src = n->cfg.net == SEEDRL_NET_DEEP ? W<float>(ws, pl.st.back().o1)
                                                        : W<float>(ws, pl.sh_a2);
  GemmEpi ea = epi_none();
  ea.a_relu = n->cfg.net == SEEDRL_NET_DEEP ? 1 : 0;
  SEEDRL_TRY(g.gemm(true, false, n->flat, kHidden, N, flat_src, n->flat, dd, kHidden, G(n, grd, n->p_dense_w), kHidden,
                    ea, st));
  SEEDRL_TRY(g.colsum(N, kHidden, dd, kHidden, G(n, grd, n->p_dense_b), st));
  // every gradient of the arena's first bucket (heads, Dense, LSTM: floats [0, seedrl_net_grad_split))
  // is final here -- the conv torso's backward below only writes the second bucket
  if (t_head_ready) SEEDRL_CUDA(cudaEventRecord((cudaEvent_t)t_head_ready, st));
  GemmEpi ef = epi_none();
  ef.mask = flat_src; ef.ldm = n->flat;
  SEEDRL_TRY(g.gemm(false, true, N, n->flat, kHidden, dd, kHidden, P(n, prm, n->p_dense_w), kHidden,
                    W<float>(ws, pl.gA), n->flat, ef, st));
  if (n->cfg.net == SEEDRL_NET_DEEP) {
    StepCtx ctx;
    ctx.wb = WgradBatch{W<float>(ws, pl.partial_all), kPartialAllBytes / sizeof(float), 0, 0, {}};
    PadScope pad(n, prm, pl, observation, ws, st);
    SEEDRL_TRY(pad.rc);
    observation = pad.obs;
    SEEDRL_TRY(pack_all_weights(n, prm, ws, pl, 1, &ctx, st));
    t_ctx = &ctx;
    int rc_t = n->conv_mode == 3 ? torso_backward_planes(n, prm, grd, pl, observation, ws, st)
                                 : torso_backward_deep(n, prm, grd, pl, observation, ws, st);
    t_ctx = nullptr;
    if (rc_t == SEEDRL_OK) rc_t = wgrad_reduce_batch(&ctx.wb, st);
    if (rc_t == SEEDRL_OK && pad.active) {        // padded [3,3,4,16] gradient -> the [3,3,3,16] parameter slot
      unpad_dw0_kernel<<<ceil_div(9 * 3 * 16, 128), 128, 0, st>>>(16, W<float>(ws, pl.dw0pad),
                                                                   n->pt.at(grd, n->stacks[0].conv.w));
      count_launch(PC_MISC, st);
    }
    return rc_t;
  }
  return torso_backward_shallow(n, prm, grd, pl, observation, ws, st);
}

// Data-parallel overlap (SURVEY 8e: the one exchange step): same as seedrl_net_backward, and
// `head_ready_event` (a cudaEvent_t) is recorded on `stream` as soon as the gradients of the first
// arena bucket -- floats [0, seedrl_net_grad_split(net)): baseline, conv_to_linear, core,
// policy_logits = 94 % of ImpalaDeep's parameters -- are final, i.e. before the convolution torso's
// backward (about half of the backward's time): the caller all-reduces that bucket on a side
// stream while the torso runs, then the remaining bucket.
extern "C" int seedrl_net_backward_overlap(const seedrl_net* n, const float* prm, int T1, int B,
                                           const int64_t* prev_actions, const float* reward, const uint8_t* done,
                                           const uint8_t* observation, const float* dlogits, const float* dbaseline,
                                           float* grd, void* ws, size_t ws_bytes, void* head_ready_event,
                                           seedrl_stream_t stream) {
  t_head_ready = head_ready_event;
  const int rc = seedrl_net_backward(n, prm, T1, B, prev_actions, reward, done, observation, dlogits, dbaseline, grd,
                                     ws, ws_bytes, stream);
  t_head_ready = nullptr;
  return rc;
}
extern "C" size_t seedrl_net_grad_split(const seedrl_net* n) {
  if (!n) return 0;
  const int first_conv = n->cfg.net == SEEDRL_NET_DEEP ? n->stacks[0].conv.w : n->sh[0].w;
  return n->pt.params[first_conv].offset;
}

// ---- single-kernel test hooks (exported so the GPU parity tests can localise a
// failure to one kernel; not used by the product path) ------------------------------
extern "C" int seedrl_debug_conv3x3(int cin, int cout, int in_mode, int N, int H, int W,
                                    const void* in, const float* w, const float* bias,
                                    const float* mask, const float* res, float* out,
                                    seedrl_stream_t stream) {
  return conv3x3_forward(cin, cout, in_mode, N, H, W, in, w, bias, mask, res, out,
                         (cudaStream_t)stream);
}
extern "C" int seedrl_debug_conv3x3_flip(int cin, int cout, const float* w, float* wt,
                                         seedrl_stream_t stream) {
  return conv3x3_flip_weights(cin, cout, w, wt, (cudaStream_t)stream);
}
extern "C" size_t seedrl_debug_wgrad_partial_bytes(void) { return conv3x3_wgrad_partial_bytes(); }
extern "C" int seedrl_debug_conv3x3_wgrad(int cin, int cout, int in_mode, int N, int H, int W,
                                          const void* x, const float* dy, float* dw, float* db,
                                          float* partial, size_t partial_bytes,
                                          seedrl_stream_t stream) {
  return conv3x3_wgrad(cin, cout, in_mode, N, H, W, x, dy, dw, db, partial, partial_bytes,
                       (cudaStream_t)stream);
}
extern "C" int seedrl_debug_maxpool(int backward, int N, int H, int W, int C, const float* x_or_dy,
                                    float* y_or_dx, uint8_t* idx, seedrl_stream_t stream) {
  if (backward) return maxpool3s2_backward(N, H, W, C, x_or_dy, idx, y_or_dx, (cudaStream_t)stream);
  return maxpool3s2_forward(N, H, W, C, x_or_dy, y_or_dx, idx, (cudaStream_t)stream);
}
// tcgen05 GEMM test hook (same contract as seedrl_debug_sgemm; split != 0: bf16x3 operands;
// ws: >= ws_bytes of scratch for split-K partials, may be null).
extern "C" int seedrl_debug_gemm_tc(int ta, int tb, int split, int M, int N, int K, const float* A, int lda,
                                    const float* B, int ldb, float* C, int ldc, const float* bias,
                                    const float* mask, int ldm, int relu, int accumulate, int a_relu,
                                    float* ws, size_t ws_bytes, int* error_flag, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(M >= 1 && N >= 1 && K >= 1 && A && B && C, "bad arguments");
  GemmEpi e{bias, mask, ldm, relu, accumulate, a_relu};
  return gemm_tc(ta != 0, tb != 0, split, M, N, K, A, lda, B, ldb, C, ldc, e, ws, ws_bytes, error_flag,
                 (cudaStream_t)stream);
}

extern "C" int seedrl_debug_sgemm(int ta, int tb, int M, int N, int K, const float* A, int lda,
                                  const float* B, int ldb, float* C, int ldc, const float* bias,
                                  const float* mask, int ldm, int relu, int accumulate, int a_relu,
                                  seedrl_stream_t stream) {
  GemmEpi e{bias, mask, ldm, relu, accumulate, a_relu};
  return sgemm(ta != 0, tb != 0, M, N, K, A, lda, B, ldb, C, ldc, e, (cudaStream_t)stream);
}

// 0: the im2col convolutions (shallow net, R2D2 body) materialise their matrices instead of gathering
// them inside the GEMM (A/B parity tests; results are bit-identical).
extern "C" int seedrl_debug_set_gemm_gather(int on) {
  gemm_tc_set_gather(on);
  return SEEDRL_OK;
}

// Column-sum test hook (bias gradients): out[n] = sum_m X[m*ld + n]; `ws` enables the row-slab path.
extern "C" int seedrl_debug_colsum(int M, int N, const float* X, int ld, float* out, float* ws, size_t ws_bytes,
                                   seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(M >= 1 && N >= 1 && X && out && ld >= N, "bad arguments");
  return colsum(M, N, X, ld, out, (cudaStream_t)stream, ws, ws_bytes);
}

// tcgen05 conv test hook: packs fp32 HWIO weights (optionally flipped/transposed for the
// data-gradient) into `wq_scratch` (>= 2*9*max(cin,16)*cout*2 bytes) and runs the tensor-core conv.
// `variant` bit0/bit1 swap LBO/SBO of the A/B descriptors (bring-up aid); *error_flag is
// set to 1 by the kernel if its bounded mbarrier wait expires.
// Host evaluation of the tall-image position -> pixel maps the conv kernels use (multiply-high
// division): which = 0 padded-input position, 1 output position.  No GPU involved.
extern "C" int seedrl_debug_conv_pixels(int N, int H, int W, int which, int start, int count, int* out) {
  SEEDRL_CHECK_ARG(N >= 1 && H >= 1 && W >= 1 && start >= 0 && count >= 0 && out, "bad arguments");
  const ConvGeom g = make_geom(N, H, W);
  for (int i = 0; i < count; ++i) out[i] = which ? out_pixel(g, start + i) : in_pixel(g, start + i);
  return SEEDRL_OK;
}

// Bench knob: K positions per pipeline stage of the tensor-core weight-gradient kernel
// (the largest of 512/256/128 not above `kc` whose stages fit shared memory is used; default 512).
extern "C" int seedrl_debug_set_wgrad_chunk(int kc) {
  SEEDRL_CHECK_ARG(kc == 128 || kc == 256 || kc == 512, "chunk must be 128, 256 or 512");
  conv3x3_wgrad_tc_set_chunk(kc);
  return SEEDRL_OK;
}

extern "C" int seedrl_debug_conv3x3_wgrad_tc(int cin, int cout, int in_mode, int split, int N, int H, int W,
                                             const void* x, const float* dy, float* dw, float* db,
                                             float* partial, size_t partial_bytes, int* error_flag,
                                             seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(conv3x3_wgrad_tc_supported(cin, cout, in_mode), "unsupported (cin,cout,mode)");
  return conv3x3_wgrad_tc(cin, cout, in_mode, split, N, H, W, x, dy, dw, db, partial, partial_bytes,
                          error_flag, nullptr, (cudaStream_t)stream);
}
// Bench knob: output positions per tile of the tensor-core forward / data-gradient kernel
// (the largest of 512/256/128 not above `mt` that keeps >= 2 CTAs per SM is used; default 512).
extern "C" int seedrl_debug_conv0pool(int N, int H, int W, const uint8_t* frames, const float* w, const float* bias,
                                      void* praw, void* prelu, uint8_t* idx, int* err, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(frames && w && bias && praw && prelu && idx && err, "null pointer");
  SEEDRL_CHECK_ARG(conv0pool_supported(4, 16, H, W), "unsupported frame size");
  return conv0pool_forward(N, H, W, frames, w, bias, praw, prelu, idx, err, (cudaStream_t)stream);
}
extern "C" int seedrl_debug_set_first_layer_dense(int on) {
  g_first_dense = on ? 1 : 0;
  return SEEDRL_OK;
}
extern "C" int seedrl_debug_set_gemm_bk(int bk) {
  gemm_tc_set_bk(bk);
  return SEEDRL_OK;
}
extern "C" int seedrl_debug_set_conv_tile(int mt) {
  SEEDRL_CHECK_ARG(mt == 128 || mt == 256 || mt == 512, "tile must be 128, 256 or 512");
  conv3x3_tc_set_tile(mt);
  return SEEDRL_OK;
}

extern "C" int seedrl_debug_conv3x3_tc(int cin, int cout, int in_mode, int split, int N, int H, int W,
                                       const void* in, const float* w, const float* bias,
                                       const float* mask, const float* res, float* out, int flip,
                                       int variant, void* wq_scratch, int* error_flag,
                                       seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(conv3x3_tc_supported(cin, cout, in_mode), "unsupported (cin,cout,mode)");
  SEEDRL_TRY(conv3x3_tc_pack_weights(cin, cout, flip, split, w, wq_scratch, (cudaStream_t)stream));
  return conv3x3_tc_forward(cin, cout, in_mode, split, N, H, W, in, wq_scratch, bias, mask, res, out,
                            variant, error_flag, (cudaStream_t)stream);
}

// ---- plane-tensor path test hooks (conv_planes.cu) ---------------------------------------------
extern "C" size_t seedrl_debug_planes_bytes(int N, int H, int W, int C) {
  if (N < 1 || H < 1 || W < 1 || C < 8 || C % 8) return 0;
  return planes_bytes(N, H, W, C);
}
extern "C" int seedrl_debug_to_planes(int N, int H, int W, int C, int relu, const float* x, void* out,
                                      seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(N >= 1 && H >= 1 && W >= 1 && C >= 8 && C % 8 == 0 && x && out, "bad arguments");
  return to_planes(N, H, W, C, relu, x, out, (cudaStream_t)stream);
}
extern "C" int seedrl_debug_from_planes(int N, int H, int W, int C, const void* in, float* y,
                                        seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(N >= 1 && H >= 1 && W >= 1 && C >= 8 && C % 8 == 0 && in && y, "bad arguments");
  return from_planes(N, H, W, C, in, y, (cudaStream_t)stream);
}
// 3x3 'same' conv on plane tensors.  w: fp32 HWIO of the FORWARD layer; flip != 0 runs the data
// gradient (cin/cout are those of the gradient convolution).  wq_scratch >= 2*9*cin*cout*2 bytes.
extern "C" int seedrl_debug_convp(int cin, int cout, int N, int H, int W, const void* in, const float* w,
                                  const float* bias, const void* mask, const void* res, int flip,
                                  void* out_raw, void* out_relu, float* out_nhwc, void* wq_scratch,
                                  int* error_flag, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(convp_supported(cin, cout) && in && w && wq_scratch, "unsupported (cin,cout) or null pointer");
  SEEDRL_TRY(conv3x3_tc_pack_weights(cin, cout, flip, 2, w, wq_scratch, (cudaStream_t)stream));
  PlaneConv c;
  c.N = N; c.H = H; c.W = W; c.in = in; c.wq = wq_scratch; c.bias = bias; c.mask = mask; c.res = res;
  c.out_raw = out_raw; c.out_relu = out_relu; c.out_nhwc = out_nhwc; c.err = error_flag;
  return convp_forward(cin, cout, c, (cudaStream_t)stream);
}
extern "C" int seedrl_debug_wgradp(int cin, int cout, int N, int H, int W, const void* x, const void* dy,
                                   float* dw, float* db, float* partial, size_t partial_bytes,
                                   int* error_flag, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(x && dy && dw && db && partial, "null pointer");
  WgradBatch wb{partial, partial_bytes / sizeof(float), 0, 0, {}};
  SEEDRL_TRY(wgradp(cin, cout, N, H, W, x, dy, dw, db, error_flag, &wb, (cudaStream_t)stream));
  return wgrad_reduce_batch(&wb, (cudaStream_t)stream);
}
// max-pool 3x3/2 'SAME' on the plane path.  forward: x fp32 NHWC -> out_raw / out_relu plane tensors
// + idx; backward: dy plane tensor (pooled) + idx -> dx plane tensor (out_raw) or fp32 NHWC (out_nhwc).
extern "C" int seedrl_debug_poolp(int backward, int N, int H, int W, int C, const void* in, void* out_raw,
                                  void* out_relu, float* out_nhwc, uint8_t* idx, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(N >= 1 && H >= 1 && W >= 1 && C >= 8 && C % 8 == 0 && in && idx, "bad arguments");
  if (backward) return poolp_backward(N, H, W, C, in, idx, out_raw, out_nhwc, (cudaStream_t)stream);
  SEEDRL_CHECK_ARG(out_raw && out_relu, "null pointer");
  return poolp_forward(N, H, W, C, reinterpret_cast<const float*>(in), out_raw, out_relu, idx,
                       (cudaStream_t)stream);
}
