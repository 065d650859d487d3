// Internal host-side launchers shared between translation units.
#pragma once
#include <initializer_list>
#include <vector>

#include "common.cuh"

namespace seedrl {

enum { IN_F32 = 0, IN_RELU = 1, IN_U8 = 2 };

// "Tall image" geometry shared by the SIMT and tensor-core 3x3 convolutions (see
// conv_kernels.cu): N images stacked into one zero-padded tall image, positions flattened.
struct ConvGeom {
  int N, H, W;       // images, spatial size (stride 1, 'same': out == in size)
  int PW;            // W + 2
  int RH;            // H + 1 (rows per image in the tall layout)
  long long Q;       // N * RH * PW flattened output positions
  // division by PW / RH as multiply-high + shift (positions are < 2^31, checked on the host):
  // l = ceil(log2 d), m = ceil(2^(31+l) / d) < 2^32, n / d == umulhi(n, m) >> (l - 1).
  // [error n*e/2^(31+l) < 2^-l <= 1/d with 0 <= e < 1, so the floor is exact]
  unsigned int pw_mul, rh_mul;
  int pw_sh, rh_sh;
};

__host__ __device__ inline void fast_div_setup(unsigned int d, unsigned int* mul, int* sh) {
  int l = 1;                                   // d >= 2
  while ((1u << l) < d) ++l;
  *mul = (unsigned int)(((1ULL << (31 + l)) + d - 1) / d);
  *sh = l - 1;
}
__host__ __device__ __forceinline__ unsigned int fast_div(unsigned int n, unsigned int mul, int sh) {
#ifdef __CUDA_ARCH__
  return __umulhi(n, mul) >> sh;
#else
  return (unsigned int)(((unsigned long long)n * mul) >> 32) >> sh;
#endif
}

__host__ __device__ inline ConvGeom make_geom(int N, int H, int W) {
  ConvGeom g;
  g.N = N; g.H = H; g.W = W; g.PW = W + 2; g.RH = H + 1;
  g.Q = (long long)N * g.RH * g.PW;
  fast_div_setup((unsigned int)g.PW, &g.pw_mul, &g.pw_sh);   // PW >= 3, RH >= 2
  fast_div_setup((unsigned int)g.RH, &g.rh_mul, &g.rh_sh);
  return g;
}

// padded-input position -> pixel index (n*H + h)*W + w, or -1 for padding.
// (positions fit in 31 bits: checked on the host)
__host__ __device__ __forceinline__ int in_pixel(const ConvGeom& g, int gp) {
  const int Rp = (int)fast_div((unsigned int)gp, g.pw_mul, g.pw_sh);
  const int c = gp - Rp * g.PW;
  const int n = (int)fast_div((unsigned int)Rp, g.rh_mul, g.rh_sh);
  const int rr = Rp - n * g.RH;
  if (rr == 0 || c == 0 || c > g.W || n >= g.N) return -1;
  return (n * g.H + (rr - 1)) * g.W + (c - 1);
}
// output position -> pixel index or -1.
__host__ __device__ __forceinline__ int out_pixel(const ConvGeom& g, int p) {
  const int Ro = (int)fast_div((unsigned int)p, g.pw_mul, g.pw_sh);
  const int c = p - Ro * g.PW;
  const int n = (int)fast_div((unsigned int)Ro, g.rh_mul, g.rh_sh);
  const int h = Ro - n * g.RH;
  if (h >= g.H || c >= g.W || n >= g.N) return -1;
  return (n * g.H + h) * g.W + c;
}

// Job tables: one launch packs every layer's weights / reduces every layer's weight-gradient
// partials (passed to the kernels by value as __grid_constant__ parameters).
constexpr int kMaxPackJobs = 32, kMaxReduceJobs = 16;
struct PackJob { const float* w; void* wq; int ck, cout, cin_src, flip, legacy; };
struct PackTable { PackJob jobs[kMaxPackJobs]; int n; };
struct ReduceJob { const float* partial; float* dw; float* db; int nparts, nw, nb; };
struct ReduceTable { ReduceJob jobs[kMaxReduceJobs]; };
struct WgradBatch { float* buf; size_t cap_floats, used; int n; ReduceJob jobs[kMaxReduceJobs]; };

// conv_tc_kernels.cu (tcgen05 tensor-core path)
bool conv3x3_tc_supported(int cin, int cout, int in_mode);
int conv3x3_tc_pack_weights(int cin, int cout, int flip, int split, const float* w, void* wq,
                            cudaStream_t st);
bool conv3x3_wgrad_tc_supported(int cin, int cout, int in_mode);
void conv3x3_wgrad_tc_set_chunk(int kc);   // upper bound: 512 (default), 256 or 128
int conv3x3_wgrad_tc(int cin, int cout, int in_mode, int split, int N, int H, int W, const void* x,
                     const float* dy, float* dw, float* db, float* partial, size_t partial_bytes,
                     int* err, WgradBatch* batch, cudaStream_t st);
int wgrad_reduce_batch(WgradBatch* b, cudaStream_t st);
int conv3x3_tc_pack_weights_batch(const PackTable& t, int split, cudaStream_t st);
void conv3x3_tc_set_tile(int mt);           // upper bound: 512 (default), 256 or 128
int conv3x3_tc_forward(int cin, int cout, int in_mode, int split, int N, int H, int W, const void* in,
                       const void* wq, const float* bias, const float* mask, const float* res,
                       float* out, int variant, int* err, cudaStream_t st);

// conv_planes.cu ("planes" path: activations stored in HBM as bf16 hi/lo channel-group planes of
// the padded tall image = the UMMA operand format; TMA-fed, warp-specialised kernels)
constexpr int kPlanesTryNext = -12347;
#define SEEDRL_TRY_RC(expr)             \
  do {                                  \
    const int rc__ = (expr);            \
    if (rc__ != SEEDRL_OK) return rc__; \
  } while (0)
long long planes_positions(int N, int H, int W);          // storage positions per plane (Lp)
size_t planes_bytes(int N, int H, int W, int C);          // 2 * C/8 planes x Lp x 16 B
struct PlaneConv {
  int N, H, W;
  const void* in;        // plane tensor, CIN channels
  const void* wq;        // packed weights (hi | lo), conv3x3_tc_pack_weights layout, split = 1
  const float* bias;     // [COUT] or null
  const void* mask;      // plane tensor (COUT ch) of the ReLU'd forward activation: out = 0 where it is 0
  const void* res;       // plane tensor (COUT ch) added to the result, or null
  void* out_raw;         // plane tensor, or null
  void* out_relu;        // plane tensor holding relu(result), or null
  float* out_nhwc;       // fp32 [N,H,W,COUT], or null
  int* err;
};
bool convp_supported(int cin, int cout);
int convp_forward(int cin, int cout, const PlaneConv& c, cudaStream_t st);
int wgradp(int cin, int cout, int N, int H, int W, const void* x, const void* dy, float* dw, float* db,
           int* err, WgradBatch* batch, cudaStream_t st);
int to_planes(int N, int H, int W, int C, int relu, const float* x, void* out, cudaStream_t st);
int from_planes(int N, int H, int W, int C, const void* in, float* y, cudaStream_t st);
int poolp_forward(int N, int H, int W, int C, const float* x, void* out_raw, void* out_relu, uint8_t* idx,
                  cudaStream_t st);
int poolp_backward(int N, int H, int W, int C, const void* dy, const uint8_t* idx, void* dx_planes,
                   float* dx_nhwc, cudaStream_t st);

// conv_first.cu (first layer of the deep net: weight gradient straight from the pooled gradient)
bool first_wgrad_pooled_supported(int cin, int cout, int H, int W);
int first_wgrad_pooled(int N, int H, int W, const uint8_t* frames, const void* g_planes, const uint8_t* idx,
                       float* dw, float* db, WgradBatch* batch, cudaStream_t st);
bool conv0pool_supported(int cin, int cout, int H, int W);
int conv0pool_forward(int N, int H, int W, const uint8_t* frames, const float* w, const float* bias, void* praw,
                      void* prelu, uint8_t* idx, int* err, cudaStream_t st);

// conv_kernels.cu
int conv3x3_forward(int cin, int cout, int in_mode, int N, int H, int W, const void* in,
                    const float* w, const float* bias, const float* mask, const float* res,
                    float* out, cudaStream_t st);
int conv3x3_flip_weights(int cin, int cout, const float* w, float* wt, cudaStream_t st);
size_t conv3x3_wgrad_partial_bytes();
int wgrad_reduce(int nparts, int nw, int nb, const float* partial, float* dw, float* db,
                 cudaStream_t st);
int conv3x3_wgrad(int cin, int cout, int in_mode, int N, int H, int W, const void* x,
                  const float* dy, float* dw, float* db, float* partial, size_t partial_bytes,
                  cudaStream_t st);
int maxpool3s2_forward(int N, int H, int W, int C, const float* x, float* y, uint8_t* idx,
                       cudaStream_t st);
int maxpool3s2_backward(int N, int H, int W, int C, const float* dy, const uint8_t* idx, float* dx,
                        cudaStream_t st);

// convgen_kernels.cu (arbitrary kernel/stride 'valid' conv: shallow net)
int convgen_forward(int N, int H, int W, int cin, int cout, int k, int stride, int in_u8,
                    const void* in, const float* w, const float* bias, int relu, float* out,
                    cudaStream_t st);
int convgen_dgrad(int N, int H, int W, int cin, int cout, int k, int stride, const float* dy,
                  const float* w, const float* mask, float* dx, cudaStream_t st);
int convgen_wgrad(int N, int H, int W, int cin, int cout, int k, int stride, int in_u8,
                  const void* x, const float* dy, float* dw, float* db, float* partial,
                  size_t partial_bytes, cudaStream_t st);

// gemm_kernels.cu
struct GemmEpi {
  const float* bias;
  const float* mask;
  int ldm;
  int relu;
  int accumulate;
  int a_relu;
};
inline GemmEpi epi_none() { return GemmEpi{nullptr, nullptr, 0, 0, 0, 0}; }
int sgemm(bool ta, bool tb, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
          float* C, int ldc, const GemmEpi& e, cudaStream_t st);
// out[n] = sum_m X[m*ld + n].  `ws` (optional scratch, e.g. the split-K workspace -- stream-ordered reuse)
// enables the row-slab path for tall matrices.
int colsum(int M, int N, const float* X, int ld, float* out, cudaStream_t st, float* ws = nullptr,
           size_t ws_bytes = 0);
// gemm_tc_kernels.cu (tcgen05): same contract as sgemm; split = bf16x3 operands; `ws` holds
// split-K partials (gemm_tc_workspace_bytes()); *err is set if a bounded mbarrier wait expires.
bool gemm_tc_supported(int M, int N, int K);
void gemm_tc_set_bk(int bk);                 // K elements per staged block: 64 or 32 (tuning knob)
size_t gemm_tc_workspace_bytes();
// op(A) = the im2col matrix of an NHWC tensor x[N][H][W][C] for a K x K / stride S 'valid' convolution
// (rows = output positions (n, ho, wo), columns = (kh, kw, c)), gathered while the GEMM stages its A
// blocks and never materialised: 8 consecutive columns of a row are 8 consecutive elements of x.
struct ConvGather {
  const void* x;
  int u8;                    // uint8 frames, scaled by 1/255 (atari/networks.py:283, dmlab/networks.py:93)
  int H, W, C, S, Ho, Wo;
  int KC;                    // K * C: one kernel row, contiguous in x
  unsigned int wo_mul, ho_mul, kc_mul;   // fast_div by Wo / Ho / KC
  int wo_sh, ho_sh, kc_sh;
};
// False when the geometry does not give aligned 8-element groups (the caller materialises the matrix).
bool conv_gather_setup(const void* x, int u8, int N, int H, int W, int C, int K, int S, ConvGather* g);
void gemm_tc_set_gather(int on);             // 0: callers keep the explicit im2col (A/B tests)
bool gemm_tc_gather_enabled();
// cg != nullptr: op(A) is the gathered im2col matrix (A / lda ignored; tb must be false).  ta = false:
// C[positions, N] = col * B (the convolution);  ta = true: C[K*K*C, N] = col^T * B (its weight gradient).
int gemm_tc(bool ta, bool tb, int split, int M, int N, int K, const float* A, int lda, const float* B,
            int ldb, float* C, int ldc, const GemmEpi& e, float* ws, size_t ws_bytes, int* err,
            cudaStream_t st, const ConvGather* cg = nullptr);
int core_input_tail(int Nrows, int D, int A, const float* reward, const int64_t* prev_action,
                    float* core_in, cudaStream_t st);
int lstm_mask_state(int B, int Hd, const uint8_t* done, const float* h_src, float* h_dst,
                    cudaStream_t st);
int lstm_pointwise_fwd(int B, int Hd, float* z, const float* c_prev_src, const uint8_t* done_t,
                       const uint8_t* done_next, float* c_out, float* h_out, float* hprev_next,
                       cudaStream_t st);
int lstm_pointwise_bwd(int B, int Hd, const float* gates, const float* c_t, const float* c_prev_src,
                       const uint8_t* done_t, const uint8_t* done_next, const float* dh_out,
                       const float* dh_rec, const float* dc_next, float* dz, float* dc_prev_out,
                       cudaStream_t st);
int fill(size_t n, float* p, float v, cudaStream_t st);

// lstm_tiled.cu (H = 256: ImpalaDeep core; H = 512: DuelingLSTMDQNNet core): CTA = (batch tile, 16
// hidden units), one barrier counter per batch tile
int lstm_forward_tiled(int H, int T1, int B, const float* U, const uint8_t* done, float* z, const float* h0,
                       const float* c0, float* hs, float* cs, float* hp, unsigned int* counter, int* err,
                       cudaStream_t st);
int lstm_backward_tiled(int H, int T1, int B, const float* U, const uint8_t* done, const float* gates,
                        const float* cs, const float* c0, const float* dhs, float* dz, unsigned int* counter,
                        int* err, cudaStream_t st);

// ---- net_common.cu: host-side pieces of the two network schedules (net.cu, r2d2_net.cu) ----------

// Parameter table of one flat fp32 arena: tensors in creation order, every start aligned to 64 floats
// (256 B).
struct ParamInfo {
  std::string name;
  int rank;
  int64_t dims[4];   // trailing dims beyond the rank are 1
  size_t offset;     // floats
  size_t size;       // floats
};
struct ParamTable {
  std::vector<ParamInfo> params;
  size_t arena_floats = 0;
  int add(const std::string& name, std::initializer_list<int64_t> dims);   // returns the tensor's index
  // Copies the name (NUL-terminated, truncated to name_buf_len), dims[0..3] and offset of tensor
  // `index`, each when its pointer is non-null; returns the rank, or -1 for an index out of range.
  int info(int index, char* name_buf, size_t name_buf_len, int64_t* dims, size_t* offset) const;
  template <typename T>
  T* at(T* arena, int idx) const { return arena + params[idx].offset; }
};

// Workspace plan: consecutive 256-byte aligned offsets, and the typed pointer at one of them.
struct Bump {
  size_t off = 0;
  size_t take(size_t bytes);
};
template <typename T>
inline T* W(void* ws, size_t off) {
  return reinterpret_cast<T*>(reinterpret_cast<char*>(ws) + off);
}

// The dense contractions of a schedule: tcgen05 when `tc` is set and the shape is worth a 128-row
// tile (gemm_tc_supported), else the fp32 SIMT kernel.  `ws` holds the split-K partials
// (gemm_tc_workspace_bytes()); *err is set when a bounded barrier wait expires.
struct GemmRunner {
  bool tc;
  int split;        // bf16x3 operands
  float* ws;
  int* err;
  int gemm(bool ta, bool tb, int M, int N, int K, const float* A, int lda, const float* B, int ldb, float* C,
           int ldc, const GemmEpi& e, cudaStream_t st) const;
  // op(A) = the gathered im2col matrix `cg` (tcgen05 only, see gemm_tc)
  int gemm_gather(bool ta, int M, int N, int K, const ConvGather& cg, const float* B, int ldb, float* C, int ldc,
                  const GemmEpi& e, cudaStream_t st) const;
  // bias gradient: out[n] = sum_m X[m*ld + n], with `ws` as the row-slab scratch
  int colsum(int M, int N, const float* X, int ld, float* out, cudaStream_t st) const;
};

// Reads back the error flag the tcgen05 / persistent kernels of the last forward/backward set when a
// bounded barrier wait expired (their results are then garbage).  Synchronises `st`.
int read_error_flag(const int* flag, cudaStream_t st);

// A 'valid' k x k / stride s convolution of NHWC tensors as a GEMM over its im2col matrix (rows =
// output positions (n, ho, wo), columns = (kh, kw, c)); Keras HWIO weights = [k*k*cin, cout].
struct StridedConv { int k, s, cin, cout, hin, win, hout, wout, w, b; };   // w, b: parameter indices
StridedConv strided_conv(int k, int s, int cin, int cout, int hin, int win);
// y = relu(im2col(x) W + b).  The im2col matrix is gathered inside the GEMM where the geometry allows
// it, else materialised in `col` and kept there for the backward.  u8: x holds uint8 frames, scaled
// by 1/255.
int strided_conv_forward(const GemmRunner& g, int N, const StridedConv& c, bool u8, const void* x, const float* w,
                         const float* bias, float* col, float* y, cudaStream_t st);
// dW = im2col(x)^T dy (gathered from x, or from the matrix the forward kept in `col`), db = column sums
// of dy; with dx (x = the ReLU'd fp32 activation): dcol = dy W^T written over `col`, dx = col2im(dcol)
// masked by x > 0.
int strided_conv_backward(const GemmRunner& g, int N, const StridedConv& c, bool u8, const void* x, float* col,
                          const float* w, const float* dy, float* dw, float* db, float* dx, cudaStream_t st);

// Keras LSTMCell(H) over T1 steps with done-resets, on N = T1 * B rows: the input projection of all
// steps as one GEMM, then the recurrence as the tiled kernels (lstm_tiled.cu) or, as their reference,
// a GEMM + a pointwise kernel per step.  Workspace offsets of its buffers:
//   xc [N, CI] core input (filled by the net), z / dz [N, 4H] gates, hp [N, H] masked h(t-1),
//   cs / hs / dhs / dd [N, H], c0buf / dhrec / dc0 / dc1 [B, H].
struct LstmBufs { size_t xc, z, hp, cs, hs, c0buf, dhs, dz, dhrec, dc0, dc1, dd; };
LstmBufs lstm_bufs(Bump* b, size_t N, int B, int H, int CI);
struct LstmCore {
  int H, CI, T1, B;
  bool tiled;
  float *xc, *z, *hp, *cs, *hs, *c0buf, *dhs, *dz, *dhrec, *dc0, *dc1, *dd;
  unsigned int* counter;   // barrier counters of the tiled kernels
};
LstmCore lstm_core(int H, int CI, int T1, int B, bool tiled, const LstmBufs& o, void* ws, unsigned int* counter);
// z = xc W + b; c0buf = c0; the recurrence -> z (activated gates), hs, cs, hp.
int lstm_core_forward(const GemmRunner& g, const LstmCore& c, const float* W, const float* U, const float* b,
                      const uint8_t* done, const float* h0, const float* c0, cudaStream_t st);
// BPTT of dhs -> dz; dU = hp^T dz, dW = xc^T dz, db = column sums of dz; dd = (dz W[:H]^T) masked by
// xc[:, :H] > 0 (the gradient of the ReLU'd Dense output at the head of the core input).
int lstm_core_backward(const GemmRunner& g, const LstmCore& c, const float* W, const float* U,
                       const uint8_t* done, float* dW, float* dU, float* db, cudaStream_t st);

}  // namespace seedrl
