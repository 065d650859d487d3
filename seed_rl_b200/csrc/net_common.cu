// Host-side pieces both network schedules are built from (net.cu: ImpalaDeep and the shallow IMPALA
// net; r2d2_net.cu: DuelingLSTMDQNNet): the parameter table, the workspace bump allocator, the GEMM
// dispatch, the strided 'valid' convolution layer and the LSTM core.
#include <string.h>

#include "kernels.h"

namespace seedrl {

constexpr size_t kAlignFloats = 64;

int ParamTable::add(const std::string& name, std::initializer_list<int64_t> dims) {
  ParamInfo p;
  p.name = name;
  p.rank = (int)dims.size();
  size_t sz = 1;
  int i = 0;
  for (int64_t d : dims) { p.dims[i++] = d; sz *= (size_t)d; }
  for (; i < 4; ++i) p.dims[i] = 1;
  p.size = sz;
  p.offset = arena_floats;
  arena_floats += (sz + kAlignFloats - 1) / kAlignFloats * kAlignFloats;
  params.push_back(p);
  return (int)params.size() - 1;
}

int ParamTable::info(int index, char* name_buf, size_t name_buf_len, int64_t* dims, size_t* offset) const {
  if (index < 0 || index >= (int)params.size()) return -1;
  const ParamInfo& p = params[index];
  if (name_buf && name_buf_len) {
    strncpy(name_buf, p.name.c_str(), name_buf_len - 1);
    name_buf[name_buf_len - 1] = 0;
  }
  if (dims) for (int i = 0; i < 4; ++i) dims[i] = p.dims[i];
  if (offset) *offset = p.offset;
  return p.rank;
}

size_t Bump::take(size_t bytes) {
  const size_t o = off;
  off += (bytes + 255) / 256 * 256;
  return o;
}

int GemmRunner::gemm(bool ta, bool tb, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                     float* C, int ldc, const GemmEpi& e, cudaStream_t st) const {
  if (tc && gemm_tc_supported(M, N, K))
    return gemm_tc(ta, tb, split, M, N, K, A, lda, B, ldb, C, ldc, e, ws, gemm_tc_workspace_bytes(), err, st);
  return sgemm(ta, tb, M, N, K, A, lda, B, ldb, C, ldc, e, st);
}

int GemmRunner::gemm_gather(bool ta, int M, int N, int K, const ConvGather& cg, const float* B, int ldb, float* C,
                            int ldc, const GemmEpi& e, cudaStream_t st) const {
  return gemm_tc(ta, false, split, M, N, K, nullptr, 0, B, ldb, C, ldc, e, ws, gemm_tc_workspace_bytes(), err, st,
                 &cg);
}

int GemmRunner::colsum(int M, int N, const float* X, int ld, float* out, cudaStream_t st) const {
  return seedrl::colsum(M, N, X, ld, out, st, ws, gemm_tc_workspace_bytes());
}

int read_error_flag(const int* flag, cudaStream_t st) {
  int h = 0;
  SEEDRL_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  SEEDRL_CUDA(cudaStreamSynchronize(st));
  if (h != 0)
    return set_error(SEEDRL_ERR_INTERNAL,
                     "a tensor-core / persistent kernel timed out on a barrier: results of this step are invalid");
  return SEEDRL_OK;
}

// ---- strided 'valid' convolution ---------------------------------------------------------------
StridedConv strided_conv(int k, int s, int cin, int cout, int hin, int win) {
  StridedConv c;
  c.k = k; c.s = s; c.cin = cin; c.cout = cout;
  c.hin = hin; c.win = win; c.hout = (hin - k) / s + 1; c.wout = (win - k) / s + 1;
  c.w = c.b = -1;
  return c;
}

// im2col: col[(n*Ho + ho)*Wo + wo][(kh*K + kw)*C + c] = x[n][ho*S + kh][wo*S + kw][c]  (* 1/255 for
// uint8 frames).  Thread = VEC consecutive channels of one col element (VEC = 4 when C % 4 == 0).
template <bool U8, int VEC>
__global__ void __launch_bounds__(256)
im2col_kernel(long long total, int H, int W, int C, int K, int S, int Ho, int Wo, const void* __restrict__ x_,
              float* __restrict__ col) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int CV = C / VEC;
  const int KK = K * K * CV;
  const long long row = i / KK;
  const int e = (int)(i - row * KK);
  const int cv = e % CV, kk = e / CV, kw = kk % K, kh = kk / K;
  const int wo = (int)(row % Wo);
  const long long r2 = row / Wo;
  const int ho = (int)(r2 % Ho);
  const long long n = r2 / Ho;
  const size_t src = (((size_t)n * H + (ho * S + kh)) * W + (wo * S + kw)) * C + (size_t)cv * VEC;
  float* dst = col + (size_t)row * (K * K * C) + (size_t)kk * C + cv * VEC;
  if (VEC == 4) {
    float4 v;
    if (U8) {
      const uchar4 u = __ldg(reinterpret_cast<const uchar4*>(reinterpret_cast<const uint8_t*>(x_) + src));
      const float k = 1.0f / 255.0f;
      v = make_float4(u.x * k, u.y * k, u.z * k, u.w * k);
    } else {
      v = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(x_) + src));
    }
    *reinterpret_cast<float4*>(dst) = v;
  } else {
    if (U8) *dst = (float)__ldg(reinterpret_cast<const uint8_t*>(x_) + src) * (1.0f / 255.0f);
    else *dst = __ldg(reinterpret_cast<const float*>(x_) + src);
  }
}

static int im2col(int N, const StridedConv& c, bool u8, const void* x, float* col, cudaStream_t st) {
  const int vec = (c.cin % 4 == 0) ? 4 : 1;
  const long long total = (long long)N * c.hout * c.wout * c.k * c.k * (c.cin / vec);
  const unsigned grid = (unsigned)((total + 255) / 256);
#define SEEDRL_I2C(U8_, V_) \
  im2col_kernel<U8_, V_><<<grid, 256, 0, st>>>(total, c.hin, c.win, c.cin, c.k, c.s, c.hout, c.wout, x, col)
  if (u8) { if (vec == 4) SEEDRL_I2C(true, 4); else SEEDRL_I2C(true, 1); }
  else    { if (vec == 4) SEEDRL_I2C(false, 4); else SEEDRL_I2C(false, 1); }
#undef SEEDRL_I2C
  count_launch(PC_CONV_FWD, st);
  SEEDRL_CHECK_LAUNCH();
  return SEEDRL_OK;
}

// col2im (gather form): dx[n][h][w][c] = sum over (kh, kw) with (h - kh) % S == 0, (w - kw) % S == 0,
// ho = (h - kh) / S < Ho, wo < Wo of dcol[(n, ho, wo)][(kh, kw, c)], masked by x > 0 (x = the ReLU'd
// activation this gradient flows into).  Thread = 4 channels of one input pixel.
__global__ void __launch_bounds__(256)
col2im_kernel(long long total, int H, int W, int C, int K, int S, int Ho, int Wo, const float* __restrict__ dcol,
              const float* __restrict__ xmask, float* __restrict__ dx) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int C4 = C >> 2;
  const int c4 = (int)(i % C4);
  long long r = i / C4;
  const int w = (int)(r % W); r /= W;
  const int h = (int)(r % H);
  const long long n = r / H;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const int KC = K * K * C;
  for (int kh = h % S; kh < K; kh += S) {
    const int ho = (h - kh) / S;
    if (h - kh < 0) break;
    if (ho >= Ho) continue;
    for (int kw = w % S; kw < K; kw += S) {
      const int wo = (w - kw) / S;
      if (w - kw < 0) break;
      if (wo >= Wo) continue;
      const float4 d = __ldg(reinterpret_cast<const float4*>(
          dcol + (((size_t)n * Ho + ho) * Wo + wo) * KC + (size_t)(kh * K + kw) * C + c4 * 4));
      acc.x += d.x; acc.y += d.y; acc.z += d.z; acc.w += d.w;
    }
  }
  const float4 m = __ldg(reinterpret_cast<const float4*>(xmask) + i);
  acc.x = m.x > 0.f ? acc.x : 0.f; acc.y = m.y > 0.f ? acc.y : 0.f;
  acc.z = m.z > 0.f ? acc.z : 0.f; acc.w = m.w > 0.f ? acc.w : 0.f;
  reinterpret_cast<float4*>(dx)[i] = acc;
}

static int col2im(int N, const StridedConv& c, const float* dcol, const float* xmask, float* dx, cudaStream_t st) {
  const long long total = (long long)N * c.hin * c.win * (c.cin / 4);
  col2im_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(total, c.hin, c.win, c.cin, c.k, c.s, c.hout,
                                                                 c.wout, dcol, xmask, dx);
  count_launch(PC_CONV_DGRAD, st);
  SEEDRL_CHECK_LAUNCH();
  return SEEDRL_OK;
}

// Tensor-core modes read the im2col matrix straight from the NHWC input while the GEMM stages its A
// blocks (kernels.h ConvGather): nothing is materialised for the forward or the weight gradient.
// False: SIMT mode, gathering switched off, a GEMM shape (forward M x cout x K or weight gradient
// K x cout x M) below a tcgen05 tile, or a geometry without aligned 8-element groups.  (The IMPALA
// shallow net's K is 256 or 64 * C >= 256, so for it the weight-gradient check reduces to M >= 32,
// which the forward's M >= 64 already implies.)
static bool gathered(const GemmRunner& g, int N, const StridedConv& c, bool u8, const void* x, ConvGather* cg) {
  const int K = c.k * c.k * c.cin, M = N * c.hout * c.wout;
  return g.tc && gemm_tc_gather_enabled() && gemm_tc_supported(M, c.cout, K) && gemm_tc_supported(K, c.cout, M) &&
         conv_gather_setup(x, u8 ? 1 : 0, N, c.hin, c.win, c.cin, c.k, c.s, cg);
}

int strided_conv_forward(const GemmRunner& g, int N, const StridedConv& c, bool u8, const void* x, const float* w,
                         const float* bias, float* col, float* y, cudaStream_t st) {
  const int K = c.k * c.k * c.cin, M = N * c.hout * c.wout;
  GemmEpi e = epi_none();
  e.bias = bias; e.relu = 1;
  ConvGather cg;
  if (gathered(g, N, c, u8, x, &cg)) return g.gemm_gather(false, M, c.cout, K, cg, w, c.cout, y, c.cout, e, st);
  SEEDRL_TRY_RC(im2col(N, c, u8, x, col, st));
  return g.gemm(false, false, M, c.cout, K, col, K, w, c.cout, y, c.cout, e, st);
}

int strided_conv_backward(const GemmRunner& g, int N, const StridedConv& c, bool u8, const void* x, float* col,
                          const float* w, const float* dy, float* dw, float* db, float* dx, cudaStream_t st) {
  const int K = c.k * c.k * c.cin, M = N * c.hout * c.wout;
  const GemmEpi e0 = epi_none();
  ConvGather cg;
  if (gathered(g, N, c, u8, x, &cg))
    SEEDRL_TRY_RC(g.gemm_gather(true, K, c.cout, M, cg, dy, c.cout, dw, c.cout, e0, st));
  else
    SEEDRL_TRY_RC(g.gemm(true, false, K, c.cout, M, col, K, dy, c.cout, dw, c.cout, e0, st));
  SEEDRL_TRY_RC(g.colsum(M, c.cout, dy, c.cout, db, st));
  if (!dx) return SEEDRL_OK;
  SEEDRL_TRY_RC(g.gemm(false, true, M, K, c.cout, dy, c.cout, w, c.cout, col, K, e0, st));
  return col2im(N, c, col, reinterpret_cast<const float*>(x), dx, st);
}

// ---- LSTM core ----------------------------------------------------------------------------------
LstmBufs lstm_bufs(Bump* b, size_t N, int B, int H, int CI) {
  LstmBufs o;
  o.xc = b->take(N * CI * 4);
  o.z = b->take(N * 4 * H * 4);
  o.hp = b->take(N * H * 4);
  o.cs = b->take(N * H * 4);
  o.hs = b->take(N * H * 4);
  o.c0buf = b->take((size_t)B * H * 4);
  o.dhs = b->take(N * H * 4);
  o.dz = b->take(N * 4 * H * 4);
  o.dhrec = b->take((size_t)B * H * 4);
  o.dc0 = b->take((size_t)B * H * 4);
  o.dc1 = b->take((size_t)B * H * 4);
  o.dd = b->take(N * H * 4);
  return o;
}

LstmCore lstm_core(int H, int CI, int T1, int B, bool tiled, const LstmBufs& o, void* ws, unsigned int* counter) {
  LstmCore c;
  c.H = H; c.CI = CI; c.T1 = T1; c.B = B; c.tiled = tiled;
  c.xc = W<float>(ws, o.xc); c.z = W<float>(ws, o.z); c.hp = W<float>(ws, o.hp);
  c.cs = W<float>(ws, o.cs); c.hs = W<float>(ws, o.hs); c.c0buf = W<float>(ws, o.c0buf);
  c.dhs = W<float>(ws, o.dhs); c.dz = W<float>(ws, o.dz); c.dhrec = W<float>(ws, o.dhrec);
  c.dc0 = W<float>(ws, o.dc0); c.dc1 = W<float>(ws, o.dc1); c.dd = W<float>(ws, o.dd);
  c.counter = counter;
  return c;
}

int lstm_core_forward(const GemmRunner& g, const LstmCore& c, const float* W, const float* U, const float* b,
                      const uint8_t* done, const float* h0, const float* c0, cudaStream_t st) {
  const int H = c.H, B = c.B, T1 = c.T1, N = T1 * B;
  // input projection for all T at once: z = xc W + b
  GemmEpi e = epi_none();
  e.bias = b;
  SEEDRL_TRY_RC(g.gemm(false, false, N, 4 * H, c.CI, c.xc, c.CI, W, 4 * H, c.z, 4 * H, e, st));
  SEEDRL_CUDA(cudaMemcpyAsync(c.c0buf, c0, (size_t)B * H * 4, cudaMemcpyDeviceToDevice, st));
  if (c.tiled)   // one kernel for the whole recurrence, CTA = (batch tile, 16 units)
    return lstm_forward_tiled(H, T1, B, U, done, c.z, h0, c.c0buf, c.hs, c.cs, c.hp, c.counter, g.err, st);
  SEEDRL_TRY_RC(lstm_mask_state(B, H, done, h0, c.hp, st));
  GemmEpi eacc = epi_none();
  eacc.accumulate = 1;
  for (int t = 0; t < T1; ++t) {
    float* zt = c.z + (size_t)t * B * 4 * H;
    SEEDRL_TRY_RC(g.gemm(false, false, B, 4 * H, H, c.hp + (size_t)t * B * H, H, U, 4 * H, zt, 4 * H, eacc, st));
    const bool last = (t + 1 == T1);
    SEEDRL_TRY_RC(lstm_pointwise_fwd(B, H, zt, t == 0 ? c.c0buf : c.cs + (size_t)(t - 1) * B * H,
                                     done + (size_t)t * B, last ? nullptr : done + (size_t)(t + 1) * B,
                                     c.cs + (size_t)t * B * H, c.hs + (size_t)t * B * H,
                                     last ? nullptr : c.hp + (size_t)(t + 1) * B * H, st));
  }
  return SEEDRL_OK;
}

int lstm_core_backward(const GemmRunner& g, const LstmCore& c, const float* W, const float* U,
                       const uint8_t* done, float* dW, float* dU, float* db, cudaStream_t st) {
  const int H = c.H, B = c.B, T1 = c.T1, N = T1 * B, CI = c.CI;
  const GemmEpi e0 = epi_none();
  if (c.tiled) {
    SEEDRL_TRY_RC(lstm_backward_tiled(H, T1, B, U, done, c.z, c.cs, c.c0buf, c.dhs, c.dz, c.counter, g.err, st));
  } else {
    float* dcb[2] = {c.dc0, c.dc1};
    for (int t = T1 - 1; t >= 0; --t) {
      const bool last = (t + 1 == T1);
      const size_t o = (size_t)t * B * H;
      SEEDRL_TRY_RC(lstm_pointwise_bwd(B, H, c.z + (size_t)t * B * 4 * H, c.cs + o,
                                       t == 0 ? c.c0buf : c.cs + o - (size_t)B * H, done + (size_t)t * B,
                                       last ? nullptr : done + (size_t)(t + 1) * B, c.dhs + o,
                                       last ? nullptr : c.dhrec, last ? nullptr : dcb[(t + 1) & 1],
                                       c.dz + (size_t)t * B * 4 * H, dcb[t & 1], st));
      if (t > 0)
        SEEDRL_TRY_RC(g.gemm(false, true, B, H, 4 * H, c.dz + (size_t)t * B * 4 * H, 4 * H, U, 4 * H, c.dhrec, H,
                             e0, st));
    }
  }
  SEEDRL_TRY_RC(g.gemm(true, false, H, 4 * H, N, c.hp, H, c.dz, 4 * H, dU, 4 * H, e0, st));
  SEEDRL_TRY_RC(g.gemm(true, false, CI, 4 * H, N, c.xc, CI, c.dz, 4 * H, dW, 4 * H, e0, st));
  SEEDRL_TRY_RC(g.colsum(N, 4 * H, c.dz, 4 * H, db, st));
  GemmEpi em = epi_none();
  em.mask = c.xc; em.ldm = CI;
  return g.gemm(false, true, N, H, 4 * H, c.dz, 4 * H, W, 4 * H, c.dd, H, em, st);
}

}  // namespace seedrl
