// Target-location encoder (CLoSD / "DiP with target conditioning": reference model/mdm.py:197-199,399-480,
// utils/misc.py:5-16).  Runs once per sampling loop (or DiP chunk), never inside the step graph: the embedding depends on
// the sample, not on the timestep, so b200mdm_set_target computes it here and b200mdm_set_cond* folds it into the
// per-sample conditioning rows (condproj / memproj) that the step already reads.
//
// n = len(all_goal_joint_names) + 2 rows ('traj', 'heading'); target [B, n, 3] fp32, valid [B, n] in {0, 1}.
//   single : mlp([target | valid].view(B, 4n)): Linear(4n, d), then layers x (SiLU, Linear(d, d))
//   split  : row j: [target[b,j] | valid[b,j]] -> Linear(4, d/n), then layers x (SiLU, Linear(d/n, d/n)); concatenated
//   multi  : valid rows only: e_j = L2_j(SiLU(L1_j(target[b,j]))), L1_j: 3 -> d, L2_j: d -> d; invalid rows are 0;
//            out = sum_j (w_j / sum(w)) e_j
// Every product is one launch of `tgt_linear_kernel`, a grouped fp32 CUDA-core GEMM: group g has its own W / bias /
// column offsets and (for multi) its own list of samples, and a block computes a 128-sample x 32-column tile, so each
// weight matrix is read from memory once per 128 samples rather than once per sample.  fp32 throughout (~0.6 GFLOP at
// B = 128 once per loop: tensor cores would buy nothing, and fp32 keeps the embedding ~1e-6 from the reference).
#pragma once
#include <cuda_runtime.h>

namespace b200 {

constexpr int TGT_BM = 128, TGT_BN = 32, TGT_BK = 16, TGT_THREADS = 256;

struct TgtLinear {
  const float* x; long long x_gs; int ldx;   // input row of sample b in group g: x + g*x_gs + b*ldx
  const float* w; long long w_gs;            // W_g [N, K] row-major at w + g*w_gs
  const float* bias; long long b_gs;         // [N] at bias + g*b_gs
  float* y; long long y_gs; int ldy;         // output row of sample b in group g: y + g*y_gs + b*ldy
  const int* rows; const int* counts;        // group g computes samples rows[g*rows_gs + r], r < counts[g];
  int rows_gs;                               //   rows == nullptr: samples 0..R-1
  int R, N, K, silu_in;                      // silu_in: SiLU(x) = x / (1 + exp(-x)) applied to the input as it is read
};

// grid = (ceil(N / 32), ceil(R / 128), groups), block = 256: thread (ty = t / 8, tx = t % 8) owns rows 4ty..4ty+3 and
// columns 4tx..4tx+3 of the tile.  The k-sum runs in order, in fp32 fma.
__global__ void __launch_bounds__(TGT_THREADS) tgt_linear_kernel(TgtLinear p) {
  __shared__ float xs[TGT_BK][TGT_BM + 4];
  __shared__ float ws[TGT_BK][TGT_BN + 4];
  __shared__ int srow[TGT_BM];
  const int g = blockIdx.z, n0 = blockIdx.x * TGT_BN, r0 = blockIdx.y * TGT_BM;
  const int count = p.rows ? p.counts[g] : p.R;
  if (r0 >= count) return;
  const int t = threadIdx.x, tx = t % 8, ty = t / 8;
  const float* x = p.x + g * p.x_gs;
  const float* w = p.w + g * p.w_gs;
  for (int r = t; r < TGT_BM; r += TGT_THREADS)
    srow[r] = (r0 + r < count) ? (p.rows ? p.rows[g * p.rows_gs + r0 + r] : r0 + r) : -1;
  __syncthreads();
  float acc[4][4] = {};
  for (int k0 = 0; k0 < p.K; k0 += TGT_BK) {
    for (int i = t; i < TGT_BK * TGT_BM; i += TGT_THREADS) {
      const int k = i % TGT_BK, r = i / TGT_BK, b = srow[r];
      float v = 0.f;
      if (b >= 0 && k0 + k < p.K) {
        v = x[static_cast<long long>(b) * p.ldx + k0 + k];
        if (p.silu_in) v = v / (1.f + expf(-v));
      }
      xs[k][r] = v;
    }
    for (int i = t; i < TGT_BK * TGT_BN; i += TGT_THREADS) {
      const int k = i % TGT_BK, n = i / TGT_BK;
      ws[k][n] = (n0 + n < p.N && k0 + k < p.K) ? w[static_cast<long long>(n0 + n) * p.K + k0 + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TGT_BK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&xs[k][4 * ty]);
      const float4 c = *reinterpret_cast<const float4*>(&ws[k][4 * tx]);
      const float av[4] = {a.x, a.y, a.z, a.w}, cv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], cv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const float* bias = p.bias + g * p.b_gs;
  float* y = p.y + g * p.y_gs;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = srow[4 * ty + i];
    if (b < 0) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + 4 * tx + j;
      if (n < p.N) y[static_cast<long long>(b) * p.ldy + n] = acc[i][j] + bias[n];
    }
  }
}

// x0[b, 4j + c] = c < 3 ? target[b, j, c] : valid[b, j]: the [target | validity] rows of the single / split encoders
// (mdm.py:417,445; the targets of invalid rows are fed in as they are).  valid: int [B, n].
__global__ void tgt_input_kernel(const float* __restrict__ target, const int* __restrict__ valid, float* __restrict__ x0,
                                 int B, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * n * 4) return;
  const int b = i / (4 * n), j = (i / 4) % n, c = i % 4;
  x0[i] = c < 3 ? target[(static_cast<long long>(b) * n + j) * 3 + c] : static_cast<float>(valid[b * n + j]);
}

// multi: out[b, c] = sum_j wn[j] * (valid[b, j] ? e[j, b, c] : 0)   (WeightedSum over all n rows, utils/misc.py:12-15)
__global__ void tgt_weighted_sum_kernel(const float* __restrict__ e, const float* __restrict__ wn, const int* __restrict__ valid,
                                        float* __restrict__ out, int B, int n, int d) {
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j < n; ++j) {
      const float v = valid[b * n + j] ? e[(static_cast<long long>(j) * B + b) * d + c] : 0.f;
      acc = fmaf(wn[j], v, acc);
    }
    out[static_cast<long long>(b) * d + c] = acc;
  }
}

// WeightedSum's normalisation w / w.sum() (utils/misc.py:12), computed once at finalize.  One thread.
__global__ void tgt_normalise_kernel(const float* __restrict__ w, float* __restrict__ wn, int n) {
  float s = 0.f;
  for (int j = 0; j < n; ++j) s += w[j];
  for (int j = 0; j < n; ++j) wn[j] = w[j] / s;
}

}  // namespace b200
