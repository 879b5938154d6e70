// CTA-tile MLP engine (fp32 FFMA path): forward and backward of the reference's MLPNet
// (model.py:20-43: Dense(H,act) -> Dense(H,act) -> Dense(out)) on a tile of TILE_R rows.
// The hidden activation ACT (common.cuh: act_fwd / act_grad_from_out) is a template parameter beside H.
//
// Shared-memory activation tiles are stored [feature][row] with row pitch RP (68 floats) so that
//   * the "row GEMM" (out[r][n] = sum_k in[k][r] W[k][n]) reads its A operand as warp-broadcast
//     float4s and its B operand (a weight slab staged by cp.async) as conflict-free float4s;
//   * the "dW GEMM" (dW[k][n] += sum_r X[k][r] Y[n][r]) reads both operands as float4s along rows.
// The hidden width H (64, 128 or 256) is a template parameter; NT = 256 threads and TILE_R = 64 rows for every width.
// Thread mapping of the row GEMM: warp w owns rows 8w..8w+7, lane l owns columns l + 32 j (j < H/32).
// Weights are re-packed once per set_weights so that those columns are read as vectors of G = min(4, H/32) floats at a
// 4G-byte lane stride (a 32-byte lane stride made every weight read a 2-way bank conflict and the loop shared-memory
// bound in round 1); packed_col<H> below is that map.  At H = 256:
//   Wp[k][4 l + j] = W[k][l + 32 j] (j < 4),  Wp[k][128 + 4 l + j - 4] = W[k][l + 32 j] (j >= 4).
// Where a step gives thread tid feature tid, at H < NT the P = NT/H threads tid = f + H p of feature f split the rows
// into P equal slices; their partial sums are combined in the order p = 0, 1, .. when the accumulators are flushed.
#pragma once
#include "common.cuh"

namespace mpg {

// packed column (within a row of W1p / W2p / W2Tp) of natural column c = l + 32 j: vector j / G of lane l, element j % G
template <int H>
__host__ __device__ __forceinline__ constexpr int packed_col(int c) {
  constexpr int G = H / 32 < 4 ? H / 32 : 4;
  return ((c >> 5) / G) * (32 * G) + G * (c & 31) + (c >> 5) % G;
}

struct NetDev {
  const float* W1p;   // [in_dim][H] packed columns
  const float* b1;    // [H]
  const float* W2p;   // [H][H] packed columns
  const float* b2;    // [H]
  const float* W2Tp;  // [H(n)][H(k)] = W2^T, packed columns
  const float* W3;    // [H][out_dim] natural
  const float* b3;    // [out_dim]
  const float* W1;    // [in_dim][H] natural (for the input gradient)
  int in_dim, out_dim;
};

// flat gradient layout (Keras order W1|b1|W2|b2|W3|b3)
struct GradLayout {
  int oW1, ob1, oW2, ob2, oW3, ob3, total;
  __host__ __device__ GradLayout(int in_dim, int out_dim, int H) {
    oW1 = 0; ob1 = oW1 + in_dim * H; oW2 = ob1 + H; ob2 = oW2 + H * H; oW3 = ob2 + H; ob3 = oW3 + H * out_dim;
    total = ob3 + out_dim;
  }
};

// shared memory carve-up (floats)
template <int H>
struct Smem {
  // the slab doubles as scratch of the input-gradient partials, [4][MAX_IN][RP]: at H < 256 that is the larger of the two
  static constexpr int SLAB = 2 * KS * H > 4 * MAX_IN * RP ? 2 * KS * H : 4 * MAX_IN * RP;
  float* bufA;   // [H][RP]
  float* bufB;   // [H][RP]
  float* slab;   // [2][KS*H]  (also scratch for the input-gradient partials)
  float* xin;    // [MAX_IN][RP]  processed obs rows, then action rows (Q input = concat)
  float* gx;     // [MAX_IN][RP]  gradient w.r.t. xin
  float* d3;     // [4][RP]       output-layer deltas
  float* y3;     // [4][RP]       output-layer pre-activations / outputs
  __device__ explicit Smem(float* base) {
    bufA = base; bufB = bufA + H * RP; slab = bufB + H * RP; xin = slab + SLAB; gx = xin + MAX_IN * RP;
    d3 = gx + MAX_IN * RP; y3 = d3 + 4 * RP;
  }
  static constexpr int FLOATS = 2 * H * RP + SLAB + 2 * MAX_IN * RP + 8 * RP;
};
static_assert(Smem<256>::SLAB == 2 * KS * 256, "the H = 256 carve-up is unchanged");

// ---------------------------------------------------------------------------------------------
// row GEMM: acc[i][j] = sum_k in_s[k][8w+i] * W[k][l+32j]; weight slabs double-buffered via cp.async.
// Contains __syncthreads(): on entry-side (before first read of in_s) and after the last read.
// ---------------------------------------------------------------------------------------------
template <int H>
__device__ __forceinline__ void rowgemm(const float* __restrict__ in_s, int K, const float* __restrict__ Wp_g,
                                        float* __restrict__ slab, float (&acc)[8][H / 32]) {
  constexpr int NJ = H / 32, G = NJ < 4 ? NJ : 4;
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < NJ; ++j) acc[i][j] = 0.f;
  const int nslab = (K + KS - 1) / KS;
  auto issue = [&](int s) {
    const int k0 = s * KS, kn = min(KS, K - k0);
    float* dst = slab + (s & 1) * KS * H;
    const float* src = Wp_g + (size_t)k0 * H;
    for (int c = tid; c < kn * (H / 4); c += NT) cp_async16(dst + c * 4, src + c * 4);
    cp_async_commit();
  };
  issue(0);
  for (int s = 0; s < nslab; ++s) {
    if (s + 1 < nslab) { issue(s + 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    __syncthreads();
    const float* sb = slab + (s & 1) * KS * H;
    const int k0 = s * KS, kn = min(KS, K - k0);
    const float* ap = in_s + (size_t)k0 * RP + w * 8;
#pragma unroll 4
    for (int kk = 0; kk < kn; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(ap + kk * RP);
      const float4 a1 = *reinterpret_cast<const float4*>(ap + kk * RP + 4);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float b[NJ];
#pragma unroll
      for (int v = 0; v < NJ / G; ++v) {   // vector v holds columns l + 32 (G v + e), e < G
        const float* bp = sb + kk * H + packed_col<H>(l + 32 * G * v);
        if constexpr (G == 4) {
          const float4 t = *reinterpret_cast<const float4*>(bp);
          b[4 * v] = t.x; b[4 * v + 1] = t.y; b[4 * v + 2] = t.z; b[4 * v + 3] = t.w;
        } else {
          const float2 t = *reinterpret_cast<const float2*>(bp);
          b[2 * v] = t.x; b[2 * v + 1] = t.y;
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
}

// epilogue: out[c][rows] = act(acc + bias[c])
template <int H, int ACT>
__device__ __forceinline__ void store_bias_act(const float (&acc)[8][H / 32], const float* __restrict__ bias,
                                               float* __restrict__ out_s) {
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
#pragma unroll
  for (int j = 0; j < H / 32; ++j) {
    const int c = l + 32 * j;
    const float bv = __ldg(bias + c);
    float4 v0, v1;
    v0.x = act_fwd<ACT>(acc[0][j] + bv); v0.y = act_fwd<ACT>(acc[1][j] + bv);
    v0.z = act_fwd<ACT>(acc[2][j] + bv); v0.w = act_fwd<ACT>(acc[3][j] + bv);
    v1.x = act_fwd<ACT>(acc[4][j] + bv); v1.y = act_fwd<ACT>(acc[5][j] + bv);
    v1.z = act_fwd<ACT>(acc[6][j] + bv); v1.w = act_fwd<ACT>(acc[7][j] + bv);
    *reinterpret_cast<float4*>(out_s + c * RP + w * 8) = v0;
    *reinterpret_cast<float4*>(out_s + c * RP + w * 8 + 4) = v1;
  }
}

// epilogue: act_s[c][rows] <- acc * act'(act_s[c][rows])   (in place: activation -> delta)
template <int H, int ACT>
__device__ __forceinline__ void store_times_actgrad(const float (&acc)[8][H / 32], float* __restrict__ act_s) {
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
#pragma unroll
  for (int j = 0; j < H / 32; ++j) {
    const int c = l + 32 * j;
    float4* p0 = reinterpret_cast<float4*>(act_s + c * RP + w * 8);
    float4 h0 = p0[0], h1 = p0[1];
    h0.x = acc[0][j] * act_grad_from_out<ACT>(h0.x); h0.y = acc[1][j] * act_grad_from_out<ACT>(h0.y);
    h0.z = acc[2][j] * act_grad_from_out<ACT>(h0.z); h0.w = acc[3][j] * act_grad_from_out<ACT>(h0.w);
    h1.x = acc[4][j] * act_grad_from_out<ACT>(h1.x); h1.y = acc[5][j] * act_grad_from_out<ACT>(h1.y);
    h1.z = acc[6][j] * act_grad_from_out<ACT>(h1.z); h1.w = acc[7][j] * act_grad_from_out<ACT>(h1.w);
    p0[0] = h0; p0[1] = h1;
  }
}

// ---------------------------------------------------------------------------------------------
// forward: xin[0..in_dim) -> h1 (bufA) -> h2 (bufB) -> y3[j][r] = h2 W3 + b3 for j < n_out
// (n_out = number of output columns actually consumed: act_dim for the policy mean, 1 for Q)
// ---------------------------------------------------------------------------------------------
template <int H, int ACT>
__device__ __forceinline__ void mlp_forward_tile(const NetDev& net, Smem<H>& sm, int n_out) {
  float acc[8][H / 32];
  rowgemm<H>(sm.xin, net.in_dim, net.W1p, sm.slab, acc);
  store_bias_act<H, ACT>(acc, net.b1, sm.bufA);
  rowgemm<H>(sm.bufA, H, net.W2p, sm.slab, acc);   // first internal barrier publishes bufA
  store_bias_act<H, ACT>(acc, net.b2, sm.bufB);
  __syncthreads();
  // output layer: thread (r, q) sums features k = q, q+4, ... for every consumed column, then the
  // four partial sums are combined in a fixed order through shared memory (deterministic)
  const int tid = threadIdx.x, r = tid & 63, q = tid >> 6;
  float part[MAX_A] = {0.f, 0.f};
  for (int k = q; k < H; k += 4) {
    const float h = sm.bufB[k * RP + r];
#pragma unroll
    for (int j = 0; j < MAX_A; ++j)
      if (j < n_out) part[j] = fmaf(h, __ldg(net.W3 + k * net.out_dim + j), part[j]);
  }
  float* scratch = sm.slab;  // [4][MAX_A][RP]
#pragma unroll
  for (int j = 0; j < MAX_A; ++j)
    if (j < n_out) scratch[(q * MAX_A + j) * RP + r] = part[j];
  __syncthreads();
  if (tid < 64 * n_out) {
    const int j = tid >> 6;
    float v = __ldg(net.b3 + j);
    for (int qq = 0; qq < 4; ++qq) v += scratch[(qq * MAX_A + j) * RP + r];
    sm.y3[j * RP + r] = v;
  }
  __syncthreads();
}

// persistent per-thread gradient accumulators: thread tid owns feature tid % H, rows slice tid / H (see the top)
template <int H>
struct GradAcc {
  float dW1[MAX_IN];  // dW1[i][tid % H]
  float db1, db2;
  float dW3[MAX_A];   // dW3[tid % H][j]
  float db3;          // db3[tid] for tid < n_out
  __device__ void zero() {
    db3 = 0.f;
#pragma unroll
    for (int i = 0; i < MAX_IN; ++i) dW1[i] = 0.f;
    db1 = db2 = 0.f;
#pragma unroll
    for (int j = 0; j < MAX_A; ++j) dW3[j] = 0.f;
  }
};

// dW2[k][n] += sum_r X[k][r] Y[n][r] into this CTA's private global partial (natural (k,n) layout).
// H/64 chunks of 64 columns n (warp w: n = 64 chunk + 8 w + j, j < 8); lane l owns the rows k = l + 32 i, i < H/32.
template <int H>
__device__ __forceinline__ void dw2_accumulate(const float* __restrict__ X, const float* __restrict__ Y,
                                               float* __restrict__ dW2g) {
  constexpr int NI = H / 32;
  const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
  for (int chunk = 0; chunk < H / 64; ++chunk) {
    float acc[NI][8];
#pragma unroll
    for (int i = 0; i < NI; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    const float* yb = Y + (chunk * 64 + w * 8) * RP;
#pragma unroll 2
    for (int r4 = 0; r4 < TILE_R; r4 += 4) {
      float4 x[NI];
#pragma unroll
      for (int i = 0; i < NI; ++i) x[i] = *reinterpret_cast<const float4*>(X + (l + 32 * i) * RP + r4);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 y = *reinterpret_cast<const float4*>(yb + j * RP + r4);
#pragma unroll
        for (int i = 0; i < NI; ++i) {
          acc[i][j] = fmaf(x[i].x, y.x, acc[i][j]);
          acc[i][j] = fmaf(x[i].y, y.y, acc[i][j]);
          acc[i][j] = fmaf(x[i].z, y.z, acc[i][j]);
          acc[i][j] = fmaf(x[i].w, y.w, acc[i][j]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      float4* g = reinterpret_cast<float4*>(dW2g + (size_t)(l + 32 * i) * H + chunk * 64 + w * 8);
      float4 g0 = g[0], g1 = g[1];
      g0.x += acc[i][0]; g0.y += acc[i][1]; g0.z += acc[i][2]; g0.w += acc[i][3];
      g1.x += acc[i][4]; g1.y += acc[i][5]; g1.z += acc[i][6]; g1.w += acc[i][7];
      g[0] = g0; g[1] = g1;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// backward. On entry: xin = layer input, bufA = h1, bufB = h2 (from mlp_forward_tile) and
// d3[j][r] = dL/d y3[j][r] for j < n_out (rows >= valid must hold 0). On exit (want_gin):
// gx[i][r] = dL/d xin[i][r].  With want_dw the parameter gradients are accumulated into `ga`
// (registers) and dW2g (global partial).
// ---------------------------------------------------------------------------------------------
template <int H, int ACT>
__device__ __forceinline__ void mlp_backward_tile(const NetDev& net, Smem<H>& sm, int n_out, bool want_dw, bool want_gin,
                                                  GradAcc<H>& ga, float* __restrict__ dW2g) {
  const int tid = threadIdx.x;
  // feature f of this thread and its slice [r0, r0 + RS) of the tile rows (P = 1: all rows)
  constexpr int P = NT / H, RS = TILE_R / P;
  const int f = P == 1 ? tid : tid % H, r0 = P == 1 ? 0 : (tid / H) * RS;
  // (1) thread (f, slice) walks its feature row: dW3 += h2 d3, delta2 = (d3 W3^T) act'(h2) in place, db2
  {
    float w3[MAX_A];
#pragma unroll
    for (int j = 0; j < MAX_A; ++j) w3[j] = (j < n_out) ? __ldg(net.W3 + f * net.out_dim + j) : 0.f;
    float* hrow = sm.bufB + f * RP;
    float s_db2 = 0.f, s_dw3[MAX_A] = {0.f, 0.f};
    for (int r4 = r0; r4 < r0 + RS; r4 += 4) {
      float4 h = *reinterpret_cast<float4*>(hrow + r4);
      float hv[4] = {h.x, h.y, h.z, h.w}, dv[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float g = 0.f;
#pragma unroll
        for (int j = 0; j < MAX_A; ++j)
          if (j < n_out) {
            const float d = sm.d3[j * RP + r4 + e];
            g = fmaf(d, w3[j], g);
            s_dw3[j] = fmaf(hv[e], d, s_dw3[j]);
          }
        dv[e] = g * act_grad_from_out<ACT>(hv[e]);
        s_db2 += dv[e];
      }
      *reinterpret_cast<float4*>(hrow + r4) = make_float4(dv[0], dv[1], dv[2], dv[3]);
    }
    if (want_dw) {
      ga.db2 += s_db2;
#pragma unroll
      for (int j = 0; j < MAX_A; ++j) ga.dW3[j] += s_dw3[j];
    }
  }
  if (want_dw && tid < n_out) {
    float s_db3 = 0.f;
    for (int r = 0; r < TILE_R; ++r) s_db3 += sm.d3[tid * RP + r];
    ga.db3 += s_db3;
  }
  __syncthreads();
  // (2) dW2 += h1^T delta2
  if (want_dw) dw2_accumulate<H>(sm.bufA, sm.bufB, dW2g);
  // (3) delta1 = (delta2 W2^T) act'(h1), in place over h1
  {
    float acc[8][H / 32];
    rowgemm<H>(sm.bufB, H, net.W2Tp, sm.slab, acc);
    store_times_actgrad<H, ACT>(acc, sm.bufA);
  }
  __syncthreads();
  // (4) dW1 += xin^T delta1, db1 (thread (f, slice) as in (1))
  if (want_dw) {
    const float* drow = sm.bufA + f * RP;
    float s_db1 = 0.f;
    for (int r4 = r0; r4 < r0 + RS; r4 += 4) {
      const float4 d = *reinterpret_cast<const float4*>(drow + r4);
      s_db1 += (d.x + d.y) + (d.z + d.w);
#pragma unroll
      for (int i = 0; i < MAX_IN; ++i)
        if (i < net.in_dim) {
          const float4 x = *reinterpret_cast<const float4*>(sm.xin + i * RP + r4);
          ga.dW1[i] = fmaf(x.x, d.x, fmaf(x.y, d.y, fmaf(x.z, d.z, fmaf(x.w, d.w, ga.dW1[i]))));
        }
    }
    ga.db1 += s_db1;
  }
  // (5) gx[i][r] = sum_n delta1[n][r] W1[i][n]: thread (r, q) covers n in [q H/4, (q+1) H/4), partials
  //     combined in fixed order
  if (want_gin) {
    const int r = tid & 63, q = tid >> 6;
    float part[MAX_IN];
#pragma unroll
    for (int i = 0; i < MAX_IN; ++i) part[i] = 0.f;
    for (int n = q * (H / 4); n < (q + 1) * (H / 4); ++n) {
      const float d = sm.bufA[n * RP + r];
#pragma unroll
      for (int i = 0; i < MAX_IN; ++i)
        if (i < net.in_dim) part[i] = fmaf(d, __ldg(net.W1 + i * H + n), part[i]);
    }
    float* scratch = sm.slab;  // [4][MAX_IN][RP] = 5440 floats <= Smem<H>::SLAB
#pragma unroll
    for (int i = 0; i < MAX_IN; ++i)
      if (i < net.in_dim) scratch[(q * MAX_IN + i) * RP + r] = part[i];
    __syncthreads();
    for (int idx = tid; idx < net.in_dim * 64; idx += NT) {
      const int i = idx >> 6, rr = idx & 63;
      sm.gx[i * RP + rr] = (scratch[(0 * MAX_IN + i) * RP + rr] + scratch[(1 * MAX_IN + i) * RP + rr])
                           + (scratch[(2 * MAX_IN + i) * RP + rr] + scratch[(3 * MAX_IN + i) * RP + rr]);
    }
  }
  __syncthreads();
}

// write the register-resident accumulators of this CTA into its private partial buffer.  At H < NT the row slices of a
// feature are added in the order slice 0, 1, .. (one barrier between slices): bit-reproducible, no atomics.
// Every thread of the CTA must call it.
template <int H>
__device__ __forceinline__ void flush_grad_acc(const NetDev& net, const GradAcc<H>& ga, float* __restrict__ partial) {
  const GradLayout L(net.in_dim, net.out_dim, H);
  constexpr int P = NT / H;
  const int tid = threadIdx.x, f = P == 1 ? tid : tid % H, slice = P == 1 ? 0 : tid / H;
  for (int p = 0; p < P; ++p) {
    if (p > 0) __syncthreads();   // the previous slice's sums are in place
    if (slice != p) continue;
    auto put = [&](int idx, float v) { partial[idx] = p == 0 ? v : partial[idx] + v; };
#pragma unroll
    for (int i = 0; i < MAX_IN; ++i)
      if (i < net.in_dim) put(L.oW1 + i * H + f, ga.dW1[i]);
    put(L.ob1 + f, ga.db1);
    put(L.ob2 + f, ga.db2);
#pragma unroll
    for (int j = 0; j < MAX_A; ++j)
      if (j < net.out_dim) put(L.oW3 + f * net.out_dim + j, ga.dW3[j]);
  }
  if (tid < MAX_A && tid < net.out_dim) partial[L.ob3 + tid] = ga.db3;
  // columns j >= MAX_A (the unused log-std half of the policy head, policy.py:198) keep their zeros
}

}  // namespace mpg
