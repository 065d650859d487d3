// (a11) R2D2 agent network: atari/networks.py:221-340 DuelingLSTMDQNNet as a fixed schedule of
// this library's kernels -- forward unroll (_torso folded over T*B by batch_apply; LSTMCell(512)
// over T with done-resets, _unroll_cell :176-218; dueling _head :275-288) and the matching
// backward (what tf.GradientTape computes at agents/r2d2/learner.py:596-609).
//
// The three 'valid' strided convolutions (8x8/4 -> 32, 4x4/2 -> 64, 3x3/1 -> 64) run as
// im2col + tensor-core GEMM (net_common.cu strided_conv_*; gemm_tc_kernel, bf16x3 = fp32-faithful;
// fp32 SIMT sgemm in mode 0):
//   forward   col = im2col(x);  y = relu(col W + b)           (W is Keras HWIO = [k*k*cin, cout])
//   weights   dW = col^T dy (deterministic split-K), db = column sums of dy
//   data      dcol = dy W^T (written over col), dx = col2im(dcol) * (x > 0)   (gather form, no atomics)
// The im2col matrices of the training unroll are kept for the backward (HBM is plentiful: 4.5 GB at
// T=101, B=64).  Frames arrive already stacked ([T,B,H,W,C] uint8, C = stack_size; the bit-packed
// frame stacking is r2d2_kernels.cu::stack_frames) and are scaled by 1/255 inside im2col.
//
// Parameters: one flat fp32 arena in tf.Module.trainable_variables order (attribute-name order:
// _advantage, _body, _core, _value), Keras layouts, tensor starts aligned to 64 floats.
#include "kernels.h"

#define SEEDRL_TRY(expr) SEEDRL_TRY_RC(expr)

namespace seedrl {

constexpr int kRH = 512;                 // LSTMCell(512), Dense(512) (networks.py:240-252)

}  // namespace seedrl

struct seedrl_r2d2_net {
  int A, H, W, C;
  int mode;                               // 0 = fp32 SIMT GEMMs, 2 = tcgen05 bf16x3
  int lstm_mode = 2;                      // 2 = tiled persistent LSTM (lstm_tiled.cu), 0 = per-step launches
  seedrl::ParamTable pt;
  size_t logical_params;
  seedrl::StridedConv conv[3];
  int flat, core_in;
  int p_ah_w, p_ah_b, p_a_w, p_dense_w, p_dense_b, p_core_w, p_core_u, p_core_b, p_vh_w, p_vh_b, p_v_w, p_v_b;
};

namespace seedrl {

struct RPlan {
  size_t N;
  size_t col[3], act[3];                  // im2col matrices, post-ReLU conv outputs (NHWC)
  LstmBufs lstm;
  size_t vh, ah, v, adv, dv, dadv, dvh, dah, g[3];
  size_t gemm_ws, tcerr, counter;
  size_t total;
};

static RPlan r_plan(const seedrl_r2d2_net* n, int T, int B) {
  RPlan p;
  Bump b;
  const size_t N = (size_t)T * B;
  p.N = N;
  for (int i = 0; i < 3; ++i) {
    const StridedConv& c = n->conv[i];
    p.col[i] = b.take(N * c.hout * c.wout * (size_t)(c.k * c.k * c.cin) * 4);
    p.act[i] = b.take(N * c.hout * c.wout * (size_t)c.cout * 4);
    p.g[i] = b.take(N * c.hout * c.wout * (size_t)c.cout * 4);
  }
  p.lstm = lstm_bufs(&b, N, B, kRH, n->core_in);
  p.vh = b.take(N * kRH * 4);
  p.ah = b.take(N * kRH * 4);
  p.v = b.take(N * 4);
  p.adv = b.take(N * (size_t)n->A * 4);
  p.dv = b.take(N * 4);
  p.dadv = b.take(N * (size_t)n->A * 4);
  p.dvh = b.take(N * kRH * 4);
  p.dah = b.take(N * kRH * 4);
  p.gemm_ws = b.take(gemm_tc_workspace_bytes());
  p.tcerr = b.take(256);
  p.counter = b.take(256);
  p.total = b.off;
  return p;
}

// The dense contractions of the schedule run on the tensor cores in mode 2.
static GemmRunner gemm_runner(const seedrl_r2d2_net* n, void* ws, const RPlan& pl) {
  return GemmRunner{n->mode >= 1, n->mode >= 2, W<float>(ws, pl.gemm_ws), W<int>(ws, pl.tcerr)};
}
static LstmCore r_lstm_core(const seedrl_r2d2_net* n, void* ws, const RPlan& pl, int T, int B) {
  return lstm_core(kRH, n->core_in, T, B, n->lstm_mode == 2, pl.lstm, ws, W<unsigned int>(ws, pl.counter));
}

// _torso tail (networks.py:262-273): core_in[n] = concat(dense_out[n] (512, already ReLU'd),
// reward[n] (NOT clipped, unlike ImpalaDeep), one_hot(prev_action[n], A)).
__global__ void r2d2_core_tail_kernel(int Nrows, int D, int A, const float* __restrict__ reward,
                                      const int64_t* __restrict__ prev_action, float* __restrict__ core_in) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int Wd = 1 + A;
  if (i >= Nrows * Wd) return;
  const int n = i / Wd, j = i - n * Wd;
  core_in[(size_t)n * (D + Wd) + D + j] = j == 0 ? reward[n] : (prev_action[n] == (int64_t)(j - 1) ? 1.f : 0.f);
}

// _head (networks.py:275-288): q = value + advantage - mean(advantage); action = argmax_a q (first
// maximum, tf.argmax).  Thread per row.
__global__ void dueling_fwd_kernel(int Nrows, int A, const float* __restrict__ v, const float* __restrict__ adv,
                                   float* __restrict__ q, int32_t* __restrict__ action) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= Nrows) return;
  const float* a = adv + (size_t)n * A;
  float s = 0.f;
  for (int j = 0; j < A; ++j) s += a[j];
  const float mean = s / (float)A, val = v[n];
  float best = -INFINITY;
  int arg = 0;
  for (int j = 0; j < A; ++j) {
    const float x = val + (a[j] - mean);
    q[(size_t)n * A + j] = x;
    if (x > best) { best = x; arg = j; }
  }
  if (action) action[n] = arg;
}
// dvalue = sum_a dq ; dadvantage = dq - mean_a dq
__global__ void dueling_bwd_kernel(int Nrows, int A, const float* __restrict__ dq, float* __restrict__ dv,
                                   float* __restrict__ dadv) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= Nrows) return;
  const float* d = dq + (size_t)n * A;
  float s = 0.f;
  for (int j = 0; j < A; ++j) s += d[j];
  dv[n] = s;
  const float mean = s / (float)A;
  for (int j = 0; j < A; ++j) dadv[(size_t)n * A + j] = d[j] - mean;
}

}  // namespace seedrl

using namespace seedrl;

extern "C" int seedrl_r2d2_net_create(int num_actions, int obs_h, int obs_w, int channels, seedrl_r2d2_net** out) {
  SEEDRL_CHECK_ARG(out, "null pointer");
  SEEDRL_CHECK_ARG(num_actions >= 1 && channels >= 1, "bad shape");
  SEEDRL_CHECK_ARG(obs_h >= 36 && obs_w >= 36, "frames too small for the 8x8/4, 4x4/2, 3x3/1 body");
  seedrl_r2d2_net* n = new seedrl_r2d2_net();
  n->A = num_actions; n->H = obs_h; n->W = obs_w; n->C = channels;
  n->mode = 2;
  const int spec[3][3] = {{32, 8, 4}, {64, 4, 2}, {64, 3, 1}};     // (filters, kernel, stride) :233-238
  int h = obs_h, w = obs_w, c = channels;
  for (int i = 0; i < 3; ++i) {
    StridedConv& k = n->conv[i];
    k = strided_conv(spec[i][1], spec[i][2], c, spec[i][0], h, w);
    h = k.hout; w = k.wout; c = k.cout;
  }
  n->flat = h * w * c;
  n->core_in = kRH + 1 + num_actions;
  // tf.Module attribute order: _advantage, _body, _core, _value
  ParamTable& pt = n->pt;
  n->p_ah_w = pt.add("advantage/hidden/kernel", {kRH, 512});
  n->p_ah_b = pt.add("advantage/hidden/bias", {512});
  n->p_a_w = pt.add("advantage/head/kernel", {512, num_actions});
  for (int i = 0; i < 3; ++i) {
    StridedConv& k = n->conv[i];
    const std::string pre = "body/conv" + std::to_string(i);
    k.w = pt.add(pre + "/kernel", {k.k, k.k, k.cin, k.cout});
    k.b = pt.add(pre + "/bias", {k.cout});
  }
  n->p_dense_w = pt.add("body/dense/kernel", {n->flat, 512});
  n->p_dense_b = pt.add("body/dense/bias", {512});
  n->p_core_w = pt.add("core/kernel", {n->core_in, 4 * kRH});
  n->p_core_u = pt.add("core/recurrent_kernel", {kRH, 4 * kRH});
  n->p_core_b = pt.add("core/bias", {4 * kRH});
  n->p_vh_w = pt.add("value/hidden/kernel", {kRH, 512});
  n->p_vh_b = pt.add("value/hidden/bias", {512});
  n->p_v_w = pt.add("value/head/kernel", {512, 1});
  n->p_v_b = pt.add("value/head/bias", {1});
  n->logical_params = 0;
  for (const ParamInfo& p : pt.params) n->logical_params += p.size;
  *out = n;
  return SEEDRL_OK;
}

extern "C" void seedrl_r2d2_net_destroy(seedrl_r2d2_net* net) { delete net; }
extern "C" int seedrl_r2d2_net_num_param_tensors(const seedrl_r2d2_net* net) {
  return net ? (int)net->pt.params.size() : 0;
}
extern "C" size_t seedrl_r2d2_net_num_params(const seedrl_r2d2_net* net) { return net ? net->logical_params : 0; }
extern "C" size_t seedrl_r2d2_net_arena_floats(const seedrl_r2d2_net* net) { return net ? net->pt.arena_floats : 0; }
extern "C" int seedrl_r2d2_net_set_mode(seedrl_r2d2_net* net, int mode) {
  SEEDRL_CHECK_ARG(net && (mode == 0 || mode == 2), "mode must be 0 (fp32 SIMT) or 2 (tcgen05 bf16x3)");
  net->mode = mode;
  return SEEDRL_OK;
}
extern "C" int seedrl_r2d2_net_set_lstm_mode(seedrl_r2d2_net* net, int mode) {
  SEEDRL_CHECK_ARG(net && (mode == 0 || mode == 2), "mode must be 0 (per-step launches) or 2 (tiled persistent)");
  net->lstm_mode = mode;
  return SEEDRL_OK;
}
extern "C" int seedrl_r2d2_net_param_info(const seedrl_r2d2_net* net, int index, char* name_buf, size_t name_cap,
                                          int64_t* dims4, int* rank, size_t* offset_floats) {
  SEEDRL_CHECK_ARG(net && index >= 0 && index < (int)net->pt.params.size(), "bad index");
  const int r = net->pt.info(index, name_buf, name_cap, dims4, offset_floats);
  if (rank) *rank = r;
  return SEEDRL_OK;
}
extern "C" size_t seedrl_r2d2_net_workspace_bytes(const seedrl_r2d2_net* net, int T, int B) {
  if (!net || T < 1 || B < 1) return 0;
  return r_plan(net, T, B).total;
}

extern "C" int seedrl_r2d2_net_forward(const seedrl_r2d2_net* n, const float* prm, int T, int B,
                                       const int64_t* prev_actions, const float* reward, const uint8_t* done,
                                       const uint8_t* frames, const float* h0, const float* c0, float* q_values,
                                       int32_t* action, float* h_out, float* c_out, void* ws, size_t ws_bytes,
                                       seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(n && prm && prev_actions && reward && done && frames && h0 && c0 && q_values && ws,
                   "null pointer");
  SEEDRL_CHECK_ARG(T >= 1 && B >= 1, "T, B must be >= 1");
  const RPlan pl = r_plan(n, T, B);
  SEEDRL_CHECK_ARG(ws_bytes >= pl.total, "workspace too small");
  SEEDRL_CHECK_ARG(pl.N * (size_t)n->conv[0].hout * n->conv[0].wout < (size_t)8000000,
                   "unroll batch too large (GEMM row count)");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = (int)pl.N, A = n->A, CI = n->core_in;
  const ParamTable& pt = n->pt;
  const GemmRunner g = gemm_runner(n, ws, pl);
  SEEDRL_CUDA(cudaMemsetAsync(g.err, 0, sizeof(int), st));
  // ---- body: three strided convolutions (bias + ReLU in the GEMM epilogue) ----------------------
  const void* x = frames;
  for (int i = 0; i < 3; ++i) {
    const StridedConv& c = n->conv[i];
    float* act = W<float>(ws, pl.act[i]);
    SEEDRL_TRY(strided_conv_forward(g, N, c, i == 0, x, pt.at(prm, c.w), pt.at(prm, c.b), W<float>(ws, pl.col[i]),
                                    act, st));
    x = act;
  }
  const LstmCore core = r_lstm_core(n, ws, pl, T, B);
  float* xc = core.xc; float* hs = core.hs; float* cs = core.cs;
  // Flatten (NHWC order) + Dense(512) + ReLU written into the first 512 columns of the core input
  GemmEpi e = epi_none();
  e.bias = pt.at(prm, n->p_dense_b); e.relu = 1;
  SEEDRL_TRY(g.gemm(false, false, N, kRH, n->flat, W<float>(ws, pl.act[2]), n->flat, pt.at(prm, n->p_dense_w), kRH,
                    xc, CI, e, st));
  r2d2_core_tail_kernel<<<ceil_div(N * (1 + A), 256), 256, 0, st>>>(N, kRH, A, reward, prev_actions, xc);
  count_launch(PC_MISC, st);
  SEEDRL_CHECK_LAUNCH();
  SEEDRL_TRY(lstm_core_forward(g, core, pt.at(prm, n->p_core_w), pt.at(prm, n->p_core_u), pt.at(prm, n->p_core_b),
                               done, h0, c0, st));
  // dueling heads
  float* vh = W<float>(ws, pl.vh); float* ah = W<float>(ws, pl.ah);
  float* v = W<float>(ws, pl.v); float* adv = W<float>(ws, pl.adv);
  e = epi_none();
  e.bias = pt.at(prm, n->p_vh_b); e.relu = 1;
  SEEDRL_TRY(g.gemm(false, false, N, 512, kRH, hs, kRH, pt.at(prm, n->p_vh_w), 512, vh, 512, e, st));
  e.bias = pt.at(prm, n->p_ah_b);
  SEEDRL_TRY(g.gemm(false, false, N, 512, kRH, hs, kRH, pt.at(prm, n->p_ah_w), 512, ah, 512, e, st));
  e = epi_none();
  e.bias = pt.at(prm, n->p_v_b);
  SEEDRL_TRY(g.gemm(false, false, N, 1, 512, vh, 512, pt.at(prm, n->p_v_w), 1, v, 1, e, st));
  e = epi_none();
  SEEDRL_TRY(g.gemm(false, false, N, A, 512, ah, 512, pt.at(prm, n->p_a_w), A, adv, A, e, st));
  dueling_fwd_kernel<<<ceil_div(N, 128), 128, 0, st>>>(N, A, v, adv, q_values, action);
  count_launch(PC_MISC, st);
  SEEDRL_CHECK_LAUNCH();
  if (h_out)
    SEEDRL_CUDA(cudaMemcpyAsync(h_out, hs + (size_t)(T - 1) * B * kRH, (size_t)B * kRH * 4, cudaMemcpyDeviceToDevice,
                                st));
  if (c_out)
    SEEDRL_CUDA(cudaMemcpyAsync(c_out, cs + (size_t)(T - 1) * B * kRH, (size_t)B * kRH * 4, cudaMemcpyDeviceToDevice,
                                st));
  return SEEDRL_OK;
}

// Backward of the unroll whose forward last used `ws` (same T, B, frames).  grads = flat arena (overwritten).
extern "C" int seedrl_r2d2_net_backward(const seedrl_r2d2_net* n, const float* prm, int T, int B,
                                        const uint8_t* frames, const uint8_t* done, const float* dq, float* grd,
                                        void* ws, size_t ws_bytes, seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(n && prm && frames && done && dq && grd && ws, "null pointer");
  const RPlan pl = r_plan(n, T, B);
  SEEDRL_CHECK_ARG(ws_bytes >= pl.total, "workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int N = (int)pl.N, A = n->A;
  const ParamTable& pt = n->pt;
  const GemmRunner g = gemm_runner(n, ws, pl);
  const LstmCore core = r_lstm_core(n, ws, pl, T, B);
  float* hs = core.hs; float* dhs = core.dhs; float* dd = core.dd;
  float* vh = W<float>(ws, pl.vh); float* ah = W<float>(ws, pl.ah);
  float* dv = W<float>(ws, pl.dv); float* dadv = W<float>(ws, pl.dadv);
  float* dvh = W<float>(ws, pl.dvh); float* dah = W<float>(ws, pl.dah);
  SEEDRL_CUDA(cudaMemsetAsync(grd, 0, pt.arena_floats * sizeof(float), st));
  const GemmEpi e0 = epi_none();
  GemmEpi eacc = epi_none();
  eacc.accumulate = 1;
  // dueling combination
  dueling_bwd_kernel<<<ceil_div(N, 128), 128, 0, st>>>(N, A, dq, dv, dadv);
  count_launch(PC_MISC, st);
  SEEDRL_CHECK_LAUNCH();
  // advantage stream
  SEEDRL_TRY(g.gemm(true, false, 512, A, N, ah, 512, dadv, A, pt.at(grd, n->p_a_w), A, e0, st));
  GemmEpi em = epi_none();
  em.mask = ah; em.ldm = 512;
  SEEDRL_TRY(g.gemm(false, true, N, 512, A, dadv, A, pt.at(prm, n->p_a_w), A, dah, 512, em, st));
  SEEDRL_TRY(g.gemm(true, false, kRH, 512, N, hs, kRH, dah, 512, pt.at(grd, n->p_ah_w), 512, e0, st));
  SEEDRL_TRY(g.colsum(N, 512, dah, 512, pt.at(grd, n->p_ah_b), st));
  // value stream
  SEEDRL_TRY(g.gemm(true, false, 512, 1, N, vh, 512, dv, 1, pt.at(grd, n->p_v_w), 1, e0, st));
  SEEDRL_TRY(g.colsum(N, 1, dv, 1, pt.at(grd, n->p_v_b), st));
  em.mask = vh;
  SEEDRL_TRY(g.gemm(false, true, N, 512, 1, dv, 1, pt.at(prm, n->p_v_w), 1, dvh, 512, em, st));
  SEEDRL_TRY(g.gemm(true, false, kRH, 512, N, hs, kRH, dvh, 512, pt.at(grd, n->p_vh_w), 512, e0, st));
  SEEDRL_TRY(g.colsum(N, 512, dvh, 512, pt.at(grd, n->p_vh_b), st));
  // d core output
  SEEDRL_TRY(g.gemm(false, true, N, kRH, 512, dah, 512, pt.at(prm, n->p_ah_w), 512, dhs, kRH, e0, st));
  SEEDRL_TRY(g.gemm(false, true, N, kRH, 512, dvh, 512, pt.at(prm, n->p_vh_w), 512, dhs, kRH, eacc, st));
  SEEDRL_TRY(lstm_core_backward(g, core, pt.at(prm, n->p_core_w), pt.at(prm, n->p_core_u), done,
                                pt.at(grd, n->p_core_w), pt.at(grd, n->p_core_u), pt.at(grd, n->p_core_b), st));
  const float* flat = W<float>(ws, pl.act[2]);
  SEEDRL_TRY(g.gemm(true, false, n->flat, kRH, N, flat, n->flat, dd, kRH, pt.at(grd, n->p_dense_w), kRH, e0, st));
  SEEDRL_TRY(g.colsum(N, kRH, dd, kRH, pt.at(grd, n->p_dense_b), st));
  em.mask = flat; em.ldm = n->flat;
  SEEDRL_TRY(g.gemm(false, true, N, n->flat, kRH, dd, kRH, pt.at(prm, n->p_dense_w), kRH, W<float>(ws, pl.g[2]),
                    n->flat, em, st));
  // convolutions, last to first; no gradient flows into the frames
  for (int i = 2; i >= 0; --i) {
    const StridedConv& c = n->conv[i];
    const void* xin = i == 0 ? (const void*)frames : (const void*)W<float>(ws, pl.act[i - 1]);
    SEEDRL_TRY(strided_conv_backward(g, N, c, i == 0, xin, W<float>(ws, pl.col[i]), pt.at(prm, c.w),
                                     W<float>(ws, pl.g[i]), pt.at(grd, c.w), pt.at(grd, c.b),
                                     i > 0 ? W<float>(ws, pl.g[i - 1]) : nullptr, st));
  }
  return SEEDRL_OK;
}

extern "C" int seedrl_r2d2_net_check_error(const seedrl_r2d2_net* n, int T, int B, void* ws, size_t ws_bytes,
                                           seedrl_stream_t stream) {
  SEEDRL_CHECK_ARG(n && ws && T >= 1 && B >= 1, "bad arguments");
  const RPlan pl = r_plan(n, T, B);
  SEEDRL_CHECK_ARG(ws_bytes >= pl.total, "workspace too small");
  return read_error_flag(W<int>(ws, pl.tcerr), (cudaStream_t)stream);
}
