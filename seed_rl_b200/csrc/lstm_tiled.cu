// Persistent LSTM recurrence, second form ("tiled"): Keras LSTMCell(H) unrolled over time with
// done-resets (dmlab/networks.py:157-169, atari/networks.py:176-218) -- forward and BPTT -- as ONE
// launch each, CTA = (batch tile, unit group).
//
// A CTA that owns a few hidden units for ALL batch rows (CTA = 2..4 units, 128 CTAs at H = 256) has to
// re-read the whole h[t] (64 KB) / dZ[t+1] (256 KB) through L2 each step and synchronise all CTAs with
// one grid barrier per step: measured at 8.4 us (forward) / 18 us (backward) per step at H = 256,
// B = 64.  Here a CTA owns NU = 16 hidden units x RB batch rows:
//   * it needs only ITS batch rows of h[t] / dZ[t+1] (8x less L2 traffic at B = 64),
//   * it depends only on the CTAs of the SAME batch tile, so the per-step barrier is one counter per
//     batch tile (H/16 arrivals) instead of one grid-wide counter -- batch tiles run independently,
//   * the recurrent matrix slice (forward: U[:, 4 x 16 gate columns]; backward: the 16 rows of U,
//     stored k-major) stays in shared memory for all T steps, the cell state / its gradient stay on
//     chip,
//   * the product is register-tiled: thread = (column pair | unit, K-slice) holds 8 batch rows'
//     accumulators, operands come from shared memory as broadcast 16-byte loads (3 loads per 16 / 8
//     FMAs), K-slices are reduced through shared memory in fixed order (deterministic).
// Barriers are monotonic counters with a bounded spin (sets *err, never hangs).  CTAs of a batch
// tile are contiguous in blockIdx so that a grid larger than the machine still makes progress tile
// by tile; grids that fit are launched cooperatively (co-residency guaranteed).
#include "kernels.h"

namespace seedrl {

constexpr int kTlThreads = 256;
constexpr int kTlNU = 16;            // hidden units per CTA
constexpr int kTlNC = 4 * kTlNU;     // gate columns per CTA (forward)
constexpr int kTlMaxRB = 32;         // batch rows per CTA

struct Lstm2Args {
  int T1, B, RB, nbt, nug;
  const float* U;          // [H, 4H]
  const uint8_t* done;     // [T1, B]
  float* z;                // fwd: in x W + b, out activated gates; bwd: activated gates (in)
  const float* h0; const float* c0;
  float* hs; float* cs; float* hp;
  const float* dhs;        // bwd
  float* dz;               // bwd out
  unsigned int* counter;   // [nbt], zeroed by the host
  int* err;
};

__device__ __forceinline__ void tile_barrier_arrive(unsigned int* counter) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
  }
}
__device__ __forceinline__ void tile_barrier_wait(unsigned int* counter, unsigned int target, int* err) {
  if (threadIdx.x == 0) {
    int spins = 0;
    while (*reinterpret_cast<volatile unsigned int*>(counter) < target) {
      if (++spins > (1 << 24)) { if (err) atomicExch(err, 2); break; }
    }
    __threadfence();
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(kTlThreads, 1) lstm2_fwd_kernel(const Lstm2Args a) {
  extern __shared__ __align__(16) float sm2[];
  const int RB = a.RB;                         // multiple of 8
  float* s_U = sm2;                            // [H][64]   column c = gate*16 + ul
  float* s_hT = s_U + H * kTlNC;               // [H][RB]   h of this batch tile, k-major
  float* s_part = s_hT + H * RB;               // [8 k-slices][RB][64]
  float* s_c = s_part + 8 * RB * kTlNC;        // [RB][16]
  const int tid = threadIdx.x;
  const int bt = blockIdx.x / a.nug, ug = blockIdx.x - bt * a.nug;
  const int b0 = bt * RB, u0 = ug * kTlNU;
  const int nb = min(RB, a.B - b0);            // valid rows of this tile (> 0 by construction)
  unsigned int* ctr = a.counter + bt;
  for (int i = tid; i < H * kTlNC; i += kTlThreads) {
    const int k = i >> 6, c = i & 63;
    s_U[i] = __ldg(a.U + (size_t)k * 4 * H + (c >> 4) * H + u0 + (c & 15));
  }
  for (int i = tid; i < RB * kTlNU; i += kTlThreads) {
    const int b = i >> 4, ul = i & 15;
    s_c[i] = b < nb ? __ldg(a.c0 + (size_t)(b0 + b) * H + u0 + ul) : 0.f;
  }
  __syncthreads();
  const int cp = tid & 31, ks = tid >> 5;      // column pair, K-slice (H/8 long)
  constexpr int KS = H / 8;

  for (int t = 0; t < a.T1; ++t) {
    const uint8_t* done_t = a.done + (size_t)t * a.B;
    const uint8_t* done_n = (t + 1 < a.T1) ? a.done + (size_t)(t + 1) * a.B : nullptr;
    if (t > 0) tile_barrier_wait(ctr, (unsigned int)t * a.nug, a.err);
    // ---- this tile's recurrent input rows -> s_hT (k-major): thread = (row b fastest, float4 of k) ----
    for (int i = tid; i < RB * (H / 4); i += kTlThreads) {
      const int b = i % RB, k4 = i / RB;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b < nb) {
        if (t == 0) {
          if (!done_t[b0 + b]) v = __ldg(reinterpret_cast<const float4*>(a.h0 + (size_t)(b0 + b) * H) + k4);
          if (ug == 0) reinterpret_cast<float4*>(a.hp + (size_t)(b0 + b) * H)[k4] = v;     // hp[0], kept for dU
        } else {
          v = __ldcg(reinterpret_cast<const float4*>(a.hp + ((size_t)t * a.B + b0 + b) * H) + k4);
        }
      }
      s_hT[(k4 * 4 + 0) * RB + b] = v.x; s_hT[(k4 * 4 + 1) * RB + b] = v.y;
      s_hT[(k4 * 4 + 2) * RB + b] = v.z; s_hT[(k4 * 4 + 3) * RB + b] = v.w;
    }
    __syncthreads();
    // ---- partial z[b, 2 cols] over this thread's K-slice, 8 batch rows at a time ----------------
    for (int sb = 0; sb < RB; sb += 8) {
      float acc0[8], acc1[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { acc0[j] = 0.f; acc1[j] = 0.f; }
      const float* up = s_U + (size_t)(ks * KS) * kTlNC + cp * 2;
      const float* hp_ = s_hT + (size_t)(ks * KS) * RB + sb;
#pragma unroll 4
      for (int k = 0; k < KS; ++k) {
        const float2 u = *reinterpret_cast<const float2*>(up + k * kTlNC);
        const float4 ha = *reinterpret_cast<const float4*>(hp_ + k * RB);
        const float4 hb = *reinterpret_cast<const float4*>(hp_ + k * RB + 4);
        acc0[0] = fmaf(ha.x, u.x, acc0[0]); acc1[0] = fmaf(ha.x, u.y, acc1[0]);
        acc0[1] = fmaf(ha.y, u.x, acc0[1]); acc1[1] = fmaf(ha.y, u.y, acc1[1]);
        acc0[2] = fmaf(ha.z, u.x, acc0[2]); acc1[2] = fmaf(ha.z, u.y, acc1[2]);
        acc0[3] = fmaf(ha.w, u.x, acc0[3]); acc1[3] = fmaf(ha.w, u.y, acc1[3]);
        acc0[4] = fmaf(hb.x, u.x, acc0[4]); acc1[4] = fmaf(hb.x, u.y, acc1[4]);
        acc0[5] = fmaf(hb.y, u.x, acc0[5]); acc1[5] = fmaf(hb.y, u.y, acc1[5]);
        acc0[6] = fmaf(hb.z, u.x, acc0[6]); acc1[6] = fmaf(hb.z, u.y, acc1[6]);
        acc0[7] = fmaf(hb.w, u.x, acc0[7]); acc1[7] = fmaf(hb.w, u.y, acc1[7]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float2*>(s_part + ((size_t)ks * RB + sb + j) * kTlNC + cp * 2) = make_float2(acc0[j], acc1[j]);
    }
    __syncthreads();
    // ---- reduce the 8 K-slices (fixed order) + pointwise: thread = (b, unit) ---------------------
    for (int i = tid; i < nb * kTlNU; i += kTlThreads) {
      const int b = i >> 4, ul = i & 15;
      const int gb = b0 + b, u = u0 + ul;
      float* zrow = a.z + ((size_t)t * a.B + gb) * 4 * H;
      float zz[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) s += s_part[((size_t)q * RB + b) * kTlNC + g * 16 + ul];
        zz[g] = s + __ldg(zrow + g * H + u);
      }
      const float gi = sigmoidf_(zz[0]), gf = sigmoidf_(zz[1]), gg = tanhf(zz[2]), go = sigmoidf_(zz[3]);
      const float cp_ = done_t[gb] ? 0.f : s_c[i];
      const float c = gf * cp_ + gi * gg;
      const float h = go * tanhf(c);
      s_c[i] = c;
      zrow[u] = gi; zrow[H + u] = gf; zrow[2 * H + u] = gg; zrow[3 * H + u] = go;
      a.cs[((size_t)t * a.B + gb) * H + u] = c;
      a.hs[((size_t)t * a.B + gb) * H + u] = h;
      if (done_n) a.hp[((size_t)(t + 1) * a.B + gb) * H + u] = done_n[gb] ? 0.f : h;
    }
    if (t + 1 < a.T1) tile_barrier_arrive(ctr);
  }
}

// ------------------------------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(kTlThreads, 1) lstm2_bwd_kernel(const Lstm2Args a) {
  extern __shared__ __align__(16) float sm2[];
  constexpr int KC = 4 * H < 1024 ? 4 * H : 1024;    // dZ columns per chunk
  const int RB = a.RB;
  float* s_UT = sm2;                           // [4H][16]  U[u0+ul, k] stored k-major
  float* s_dzT = s_UT + 4 * H * kTlNU;         // [KC][RB]  chunk of dZ[t+1], k-major
  float* s_part = s_dzT + KC * RB;             // [16 k-slices][RB][16]
  float* s_dc = s_part + 16 * RB * kTlNU;      // [RB][16]  dc flowing to the previous step
  const int tid = threadIdx.x;
  const int bt = blockIdx.x / a.nug, ug = blockIdx.x - bt * a.nug;
  const int b0 = bt * RB, u0 = ug * kTlNU;
  const int nb = min(RB, a.B - b0);
  unsigned int* ctr = a.counter + bt;
  for (int i = tid; i < 4 * H * kTlNU; i += kTlThreads) {
    const int ul = i / (4 * H), k = i - ul * (4 * H);            // coalesced read of U's rows
    s_UT[k * kTlNU + ul] = __ldg(a.U + (size_t)(u0 + ul) * 4 * H + k);
  }
  for (int i = tid; i < RB * kTlNU; i += kTlThreads) s_dc[i] = 0.f;
  __syncthreads();
  const int ul_t = tid & 15, ks = tid >> 4;    // unit, K-slice (KC/16 long)
  constexpr int KS = KC / 16;

  unsigned int arrivals = 0;
  for (int t = a.T1 - 1; t >= 0; --t) {
    const bool last = (t + 1 == a.T1);
    const uint8_t* done_t = a.done + (size_t)t * a.B;
    const uint8_t* done_n = last ? nullptr : a.done + (size_t)(t + 1) * a.B;
    // ---- dh_rec[b, 16 units] = dZ[t+1][b, :] . U[u, :]^T, in chunks of KC columns ----------------
    if (!last) {
      tile_barrier_wait(ctr, arrivals * a.nug, a.err);
      for (int k0 = 0; k0 < 4 * H; k0 += KC) {
        const float* dzn = a.dz + ((size_t)(t + 1) * a.B + b0) * 4 * H + k0;
        for (int i = tid; i < RB * (KC / 4); i += kTlThreads) {
          const int b = i % RB, k4 = i / RB;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (b < nb) v = __ldcg(reinterpret_cast<const float4*>(dzn + (size_t)b * 4 * H) + k4);
          s_dzT[(k4 * 4 + 0) * RB + b] = v.x; s_dzT[(k4 * 4 + 1) * RB + b] = v.y;
          s_dzT[(k4 * 4 + 2) * RB + b] = v.z; s_dzT[(k4 * 4 + 3) * RB + b] = v.w;
        }
        __syncthreads();
        for (int sb = 0; sb < RB; sb += 8) {
          float acc[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] = 0.f;
          const float* up = s_UT + (size_t)(k0 + ks * KS) * kTlNU + ul_t;
          const float* dp = s_dzT + (size_t)(ks * KS) * RB + sb;
#pragma unroll 4
          for (int k = 0; k < KS; ++k) {
            const float u = up[k * kTlNU];
            const float4 da = *reinterpret_cast<const float4*>(dp + k * RB);
            const float4 db = *reinterpret_cast<const float4*>(dp + k * RB + 4);
            acc[0] = fmaf(da.x, u, acc[0]); acc[1] = fmaf(da.y, u, acc[1]);
            acc[2] = fmaf(da.z, u, acc[2]); acc[3] = fmaf(da.w, u, acc[3]);
            acc[4] = fmaf(db.x, u, acc[4]); acc[5] = fmaf(db.y, u, acc[5]);
            acc[6] = fmaf(db.z, u, acc[6]); acc[7] = fmaf(db.w, u, acc[7]);
          }
          float* pp = s_part + ((size_t)ks * RB + sb) * kTlNU + ul_t;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (k0 == 0) pp[j * kTlNU] = acc[j]; else pp[j * kTlNU] += acc[j];
          }
        }
        __syncthreads();                       // the chunk buffer is refilled / the partials are read
      }
    }
    // ---- reduce the 16 K-slices (fixed order) + pointwise backward: thread = (b, unit) ------------
    for (int i = tid; i < nb * kTlNU; i += kTlThreads) {
      const int b = i >> 4, ul = i & 15;
      const int gb = b0 + b, u = u0 + ul;
      const float* gr = a.z + ((size_t)t * a.B + gb) * 4 * H;
      const float gi = __ldg(gr + u), gf = __ldg(gr + H + u), gg = __ldg(gr + 2 * H + u), go = __ldg(gr + 3 * H + u);
      const bool cut = done_n && done_n[gb];
      float dh = __ldg(a.dhs + ((size_t)t * a.B + gb) * H + u);
      if (!last && !cut) {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 16; ++q) s += s_part[((size_t)q * RB + b) * kTlNU + ul];
        dh += s;
      }
      const float tc = tanhf(__ldg(a.cs + ((size_t)t * a.B + gb) * H + u));
      float dc = dh * go * (1.f - tc * tc);
      if (!last && !cut) dc += s_dc[i];
      const float cprev = done_t[gb] ? 0.f
                          : (t == 0 ? __ldg(a.c0 + (size_t)gb * H + u)
                                    : __ldg(a.cs + ((size_t)(t - 1) * a.B + gb) * H + u));
      float* dzr = a.dz + ((size_t)t * a.B + gb) * 4 * H;
      dzr[u] = dc * gg * gi * (1.f - gi);
      dzr[H + u] = dc * cprev * gf * (1.f - gf);
      dzr[2 * H + u] = dc * gi * (1.f - gg * gg);
      dzr[3 * H + u] = dh * tc * go * (1.f - go);
      s_dc[i] = dc * gf;
    }
    if (t > 0) { tile_barrier_arrive(ctr); ++arrivals; }
  }
}

// ------------------------------------------------------------------------------------------------
static int tile_rows(int B, int nug) {
  // up to 8 batch tiles, but no more than keep the whole grid (tiles x unit groups) co-resident: every
  // further tile only starts when an earlier one has finished all T steps (H = 512: 32 unit groups =>
  // 4 tiles of 16 rows at B = 64 instead of two waves of 8-row tiles).  Rows per tile: a multiple of 8,
  // at most kTlMaxRB.
  int tiles = kNumSMs / nug;
  if (tiles > 8) tiles = 8;
  if (tiles < 1) tiles = 1;
  int rb = ((B + tiles - 1) / tiles + 7) / 8 * 8;
  if (rb < 8) rb = 8;
  if (rb > kTlMaxRB) rb = kTlMaxRB;
  return rb;
}
static size_t fwd_smem(int H, int RB) {
  return ((size_t)H * kTlNC + (size_t)H * RB + (size_t)8 * RB * kTlNC + (size_t)RB * kTlNU) * sizeof(float);
}
static size_t bwd_smem(int H, int RB) {
  const int KC = 4 * H < 1024 ? 4 * H : 1024;
  return ((size_t)4 * H * kTlNU + (size_t)KC * RB + (size_t)16 * RB * kTlNU + (size_t)RB * kTlNU) * sizeof(float);
}

template <int H>
static int launch_lstm2(bool bwd, Lstm2Args a, cudaStream_t st) {
  int RB = tile_rows(a.B, H / kTlNU);
  while (RB > 8 && (bwd ? bwd_smem(H, RB) : fwd_smem(H, RB)) > 220 * 1024) RB -= 8;
  const size_t smem = bwd ? bwd_smem(H, RB) : fwd_smem(H, RB);
  if (smem > 220 * 1024) return set_error(SEEDRL_ERR_INVALID_ARGUMENT, "lstm (tiled): does not fit shared memory");
  a.RB = RB;
  a.nbt = (a.B + RB - 1) / RB;
  a.nug = H / kTlNU;
  if (a.nbt > 64) return set_error(SEEDRL_ERR_INVALID_ARGUMENT, "lstm (tiled): batch too large");
  const void* fn = bwd ? (const void*)lstm2_bwd_kernel<H> : (const void*)lstm2_fwd_kernel<H>;
  static bool attr[2] = {false, false};
  if (!attr[bwd ? 1 : 0]) {
    SEEDRL_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    attr[bwd ? 1 : 0] = true;
  }
  SEEDRL_CUDA(cudaMemsetAsync(a.counter, 0, 64 * sizeof(unsigned int), st));
  const int grid = a.nbt * a.nug;
  void* args[] = {&a};
  if (grid <= kNumSMs) {
    SEEDRL_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kTlThreads), args, smem, st));
  } else {
    // more CTAs than SMs: batch tiles are contiguous in blockIdx, resident tiles finish and make
    // room for the next ones (a tile's CTAs only wait for each other)
    SEEDRL_CUDA(cudaLaunchKernel(fn, dim3(grid), dim3(kTlThreads), args, smem, st));
  }
  count_launch(PC_LSTM_PW, st);
  return SEEDRL_OK;
}

int lstm_forward_tiled(int H, int T1, int B, const float* U, const uint8_t* done, float* z, const float* h0,
                       const float* c0, float* hs, float* cs, float* hp, unsigned int* counter, int* err,
                       cudaStream_t st) {
  Lstm2Args a;
  a.T1 = T1; a.B = B; a.U = U; a.done = done; a.z = z; a.h0 = h0; a.c0 = c0; a.hs = hs; a.cs = cs; a.hp = hp;
  a.dhs = nullptr; a.dz = nullptr; a.counter = counter; a.err = err;
  if (H == 256) return launch_lstm2<256>(false, a, st);
  if (H == 512) return launch_lstm2<512>(false, a, st);
  return set_error(SEEDRL_ERR_INVALID_ARGUMENT, "lstm: hidden size must be 256 or 512");
}

int lstm_backward_tiled(int H, int T1, int B, const float* U, const uint8_t* done, const float* gates,
                        const float* cs, const float* c0, const float* dhs, float* dz, unsigned int* counter,
                        int* err, cudaStream_t st) {
  Lstm2Args a;
  a.T1 = T1; a.B = B; a.U = U; a.done = done; a.z = const_cast<float*>(gates); a.h0 = nullptr; a.c0 = c0;
  a.hs = nullptr; a.cs = const_cast<float*>(cs); a.hp = nullptr; a.dhs = dhs; a.dz = dz; a.counter = counter; a.err = err;
  if (H == 256) return launch_lstm2<256>(true, a, st);
  if (H == 512) return launch_lstm2<512>(true, a, st);
  return set_error(SEEDRL_ERR_INVALID_ARGUMENT, "lstm: hidden size must be 256 or 512");
}

}  // namespace seedrl
