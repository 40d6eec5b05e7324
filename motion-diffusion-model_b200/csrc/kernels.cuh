// Small HBM/L2-bound kernels around the GEMMs: input packing (transpose + fp16 hi/lo split), per-step
// conditioning token, LayerNorm rows, CFG blend of the hidden rows, weight repacking, table set-up.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include "epilogues.cuh"

namespace b200 {

// ---------------------------------------------------------------------------------------------------------
// x [B, JF, T] fp32 (reference layout, T contiguous)  ->  xin16 [B*S, ld] fp16 rows (b, s = 1 + t_off + t):
//   columns [0,Kp) = hi, [Kp,2Kp) = lo, [2Kp,3Kp) = hi    (A' of the 3-pass split GEMM  A_hi*W_hi + A_lo*W_hi + A_hi*W_lo)
// Row s = 0 (conditioning token slot) and the pad columns stay zero from allocation time.
__global__ void pack_input_kernel(const float* __restrict__ x, __half* __restrict__ xin, int B, int JF, int T, int S,
                                  int Kp, int ld, int row_off) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int j0 = blockIdx.y * 32, t0 = blockIdx.x * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int j = j0 + i, t = t0 + tx;
    tile[i][tx] = (j < JF && t < T) ? x[(static_cast<size_t>(b) * JF + j) * T + t] : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int t = t0 + i, j = j0 + tx;
    if (t < T && j < JF) {
      const float v = tile[tx][i];
      const __half hi = __float2half_rn(v);
      const __half lo = __float2half_rn(v - __half2float(hi));
      __half* dst = xin + (static_cast<size_t>(b) * S + row_off + t) * ld + j;
      dst[0] = hi;
      dst[Kp] = lo;
      dst[2 * Kp] = hi;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Conditioning-token rows of the sequence (reference model/mdm.py:195,218-220,251-252):
//   h[b', s=0, :] = (condproj[b', :] + temb_table[t(b'), :]) + pe[0, :]
//   t(b') = tvec[b' % B] when tvec != nullptr (model called with explicit timesteps), else timestep_map[state->cur]
// Runs right after the embedding GEMM (which leaves placeholder values in these rows).
// The residual stream is an fp16 [hi | lo] pair per element (row = 2d halves, hi + lo carries ~22 bits).
__global__ void tok0_rows_kernel(__half* __restrict__ hres, const float* __restrict__ condproj,
                                 const float* __restrict__ temb_table, const float* __restrict__ pe,
                                 const int* __restrict__ tvec, const int* __restrict__ tmap,
                                 const StepState* __restrict__ state, int B, int S, int d, int temb_rows) {
  pdl_launch_dependents();
  pdl_wait();
  const int bp = blockIdx.x;
  int t = (tvec != nullptr) ? tvec[bp % B] : tmap[state->cur];
  t = min(max(t, 0), temb_rows - 1);
  const size_t row = static_cast<size_t>(bp) * S;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const float v = (condproj[static_cast<size_t>(bp) * d + c] + temb_table[static_cast<size_t>(t) * d + c]) + pe[c];
    const __half hi = __float2half_rn(v);
    hres[row * 2 * d + c] = hi;
    hres[row * 2 * d + d + c] = __float2half_rn(v - __half2float(hi));
  }
}

// pe_bias[s, c] = pe[s, c] + bias[c]  (per (B,T) workspace table for the embedding epilogue)
__global__ void pe_bias_kernel(float* __restrict__ out, const float* __restrict__ pe, const float* __restrict__ bias,
                               int S, int d) {
  const int s = blockIdx.x;
  for (int c = threadIdx.x; c < d; c += blockDim.x) out[static_cast<size_t>(s) * d + c] = bias[c] + pe[static_cast<size_t>(s) * d + c];
}

__global__ void step_advance_kernel(StepState* state) {
  pdl_launch_dependents();
  pdl_wait();
  state->done += 1;
  state->cur -= 1;
}
__global__ void step_set_kernel(StepState* state, int done, int cur, const float* noise, long long noise_step_stride,
                                unsigned long long seed, long long sample_base) {
  state->done = done;
  state->cur = cur;
  state->start = cur;
  state->noise = noise;
  state->noise_step_stride = noise_step_stride;
  state->seed = seed;
  state->sample_base = sample_base;
}

// ---------------------------------------------------------------------------------------------------------
// The engine's own noise stream (B200MDM_FLAG_PHILOX_NOISE / b200mdm_philox_normal): replaces the reference's
// th.randn_like(x) per step (diffusion/gaussian_diffusion.py:525, :770) when the caller asks for a stream that does not
// depend on how the batch is split over GPUs or on how many steps are drawn at once.
//   Philox4x32-10 (Salmon et al., SC'11), key = (seed_lo, seed_hi),
//   counter = (q, step_id, g_lo, g_hi ^ 0x4d444d42)   q = element index / 4 inside the sample, g = global sample index
//   the 4 output words w0..w3 -> u_k = ((w_k >> 8) + 0.5) * 2^-24 in (0, 1);
//   elements 4q..4q+3 = r0 cos(2 pi u1), r0 sin(2 pi u1), r1 cos(2 pi u3), r1 sin(2 pi u3),  r0 = sqrt(-2 ln u0), r1 = sqrt(-2 ln u2)
// step_id = schedule index of the step that consumes the eps (state->cur when `state` != nullptr); x_T uses 0xffffffff.
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}
__global__ void philox_normal_kernel(float* __restrict__ out, int B, long long n, unsigned long long seed,
                                     long long sample_base, uint32_t step_id, const StepState* __restrict__ state) {
  pdl_launch_dependents();
  pdl_wait();
  if (state != nullptr) {
    seed = state->seed;
    sample_base = state->sample_base;
    step_id = static_cast<uint32_t>(state->cur);
  }
  const long long qn = (n + 3) / 4, total = qn * B;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / qn, q = i - b * qn;
    const unsigned long long g = static_cast<unsigned long long>(sample_base + b);
    uint32_t c[4] = {static_cast<uint32_t>(q), step_id, static_cast<uint32_t>(g), static_cast<uint32_t>(g >> 32) ^ 0x4d444d42u};
    philox4x32_10(c, static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
    float z[4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float u0 = (static_cast<float>(c[2 * h] >> 8) + 0.5f) * 5.9604644775390625e-08f;
      const float u1 = (static_cast<float>(c[2 * h + 1] >> 8) + 0.5f) * 5.9604644775390625e-08f;
      const float r = sqrtf(-2.0f * logf(u0));
      float sn, cs;
      sincospif(2.0f * u1, &sn, &cs);
      z[2 * h] = r * cs;
      z[2 * h + 1] = r * sn;
    }
    float* dst = out + b * n + 4 * q;
    if (4 * q + 3 < n && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
      *reinterpret_cast<float4*>(dst) = make_float4(z[0], z[1], z[2], z[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (4 * q + j < n) dst[j] = z[j];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// CFG blend on the hidden rows + fp16 hi/lo split for the 3-pass output GEMM.
//   v = h_u + scale[b] * (h_c - h_u)   (same expression as utils/sampler_util.py:34, applied before the linear
//   OutputProcess: W(h_u + s(h_c-h_u)) + b == out_u + s(out_c - out_u) exactly in real arithmetic)
//   halves == 1: v = h.       g16 row layout: [hi | lo | hi], ld = 3*d.
__global__ void blend_split_kernel(const __half* __restrict__ hres, __half* __restrict__ g16,
                                   const float* __restrict__ scale, int B, int S, int T, int s_off, int d, int halves) {
  pdl_launch_dependents();
  pdl_wait();
  // one warp per FRAME row: the rows s < s_off of a sequence (condition token / DiP prefix) never reach x, so g16
  // holds B*T rows only (12544 = 98 tiles of 128 at B=64, T=196 -- 294 output tiles, two full waves of 148 CTAs)
  const int orow = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (orow >= B * T) return;
  const int b = orow / T;
  const int row = b * S + s_off + (orow - b * T);
  const __half* hc = hres + static_cast<size_t>(row) * 2 * d;                         // [hi | lo] rows
  const __half* hu = hres + (static_cast<size_t>(B) * S + row) * 2 * d;
  const float sc = (halves == 2) ? scale[b] : 0.f;
  __half* dst = g16 + static_cast<size_t>(orow) * 3 * d;
  for (int c = lane * 2; c < d; c += 64) {
    const float2 ah = __half22float2(*reinterpret_cast<const __half2*>(hc + c));
    const float2 al = __half22float2(*reinterpret_cast<const __half2*>(hc + d + c));
    float2 a = make_float2(ah.x + al.x, ah.y + al.y);
    if (halves == 2) {
      const float2 uh = __half22float2(*reinterpret_cast<const __half2*>(hu + c));
      const float2 ul = __half22float2(*reinterpret_cast<const __half2*>(hu + d + c));
      const float2 u = make_float2(uh.x + ul.x, uh.y + ul.y);
      a.x = __fadd_rn(u.x, __fmul_rn(sc, __fsub_rn(a.x, u.x)));
      a.y = __fadd_rn(u.y, __fmul_rn(sc, __fsub_rn(a.y, u.y)));
    }
    const __half2 hi = __floats2half2_rn(a.x, a.y);
    const float2 hif = __half22float2(hi);
    const __half2 lo = __floats2half2_rn(a.x - hif.x, a.y - hif.y);
    *reinterpret_cast<__half2*>(dst + c) = hi;
    *reinterpret_cast<__half2*>(dst + d + c) = lo;
    *reinterpret_cast<__half2*>(dst + 2 * d + c) = hi;
  }
}

// ---------------------------------------------------------------------------------------------------------
// Weight repacking (one-time, at load).
__global__ void f32_to_f16_kernel(const float* __restrict__ src, __half* __restrict__ dst, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    dst[i] = __float2half_rn(src[i]);
}
// W [N, K] fp32 -> [W16 | W16] fp16 [N, 2K]: partner of activations stored as [hi | lo] along K (the trans_dec engine keeps
// its fp16 activations to ~22 mantissa bits this way; the product A_hi W + A_lo W accumulates in fp32 on the tensor core).
__global__ void f32_to_f16_dup_kernel(const float* __restrict__ src, __half* __restrict__ dst, int N, int K) {
  const size_t n = static_cast<size_t>(N) * K;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t r = i / K, k = i % K;
    const __half h = __float2half_rn(src[i]);
    dst[r * 2 * K + k] = h;
    dst[r * 2 * K + K + k] = h;
  }
}
// W [N, K] fp32 -> W' [Npad, 3*Kp] fp16 = [hi | hi | lo] (zero padding), partner of the [hi | lo | hi] activations.
__global__ void split_weight_kernel(const float* __restrict__ w, __half* __restrict__ out, int N, int K, int Kp) {
  const int n = blockIdx.x;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const float v = w[static_cast<size_t>(n) * K + k];
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn(v - __half2float(hi));
    __half* dst = out + static_cast<size_t>(n) * 3 * Kp + k;
    dst[0] = hi;
    dst[Kp] = hi;
    dst[2 * Kp] = lo;
  }
}

// y[r, c] = act( sum_k x[r, k] * w[c, k] + b[c] ), fp32, one warp per output element (tiny set-up GEMVs:
// timestep-embedding MLP for every model timestep, text projection once per loop)
template <int ACT>  // 0 none, 1 SiLU
__global__ void small_linear_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                    const float* __restrict__ b, float* __restrict__ y, int R, int C, int K,
                                    int x_ld) {
  const size_t widx = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (widx >= static_cast<size_t>(R) * C) return;
  const int r = static_cast<int>(widx / C), c = static_cast<int>(widx % C);
  const float* xr = x + static_cast<size_t>(r) * x_ld;
  const float* wr = w + static_cast<size_t>(c) * K;
  float acc = 0.f;
  for (int k = lane; k < K; k += 32) acc = fmaf(xr[k], wr[k], acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    acc += (b != nullptr) ? b[c] : 0.f;
    if (ACT == 1) acc = acc / (1.f + expf(-acc));
    y[static_cast<size_t>(r) * C + c] = acc;
  }
}

// condproj rows for the packed batch: first B rows conditional, next B rows unconditional.
//   text  : cond = (W clip + b) already in proj[B, d];  uncond = bias          (mask_cond zeros => bias only)
//   action: cond = action_embedding[a[b]];              uncond = 0             (model/mdm.py:225-227)
//   none  : 0
// tgt (optional, [B, d]): the target-location embedding of b200mdm_set_target, added to every row of both halves after
// the masking (the reference adds it to time_emb, mdm.py:199; (text + target) + time here instead of text + (time +
// target): only the fp32 association differs).  nullptr: the rows are exactly the above.
__global__ void condproj_fill_kernel(float* __restrict__ condproj, const float* __restrict__ proj,
                                     const float* __restrict__ bias, const float* __restrict__ action_emb,
                                     const int* __restrict__ action, int B, int d, int rows, int first_uncond,
                                     int cond_mode, const float* __restrict__ tgt) {
  const int bp = blockIdx.x;
  if (bp >= rows) return;
  const bool unc = first_uncond ? true : (bp >= B);
  const int b = bp % B;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float v = 0.f;
    if (cond_mode == 1) v = unc ? bias[c] : proj[static_cast<size_t>(b) * d + c];
    else if (cond_mode == 2) v = unc ? 0.f : action_emb[static_cast<size_t>(action[b]) * d + c];
    if (tgt != nullptr) v += tgt[static_cast<size_t>(b) * d + c];
    condproj[static_cast<size_t>(bp) * d + c] = v;
  }
}

// x_t = sqrt_ac * x0 + sqrt_1mac * noise   (q_sample, diffusion/gaussian_diffusion.py:226-244)
__global__ void q_sample_kernel(float* __restrict__ out, const float* __restrict__ x0, const float* __restrict__ noise,
                                float a, float b, size_t n) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float s = (x0 != nullptr) ? x0[i] : 0.f;
    out[i] = __fadd_rn(__fmul_rn(a, s), __fmul_rn(b, noise[i]));
  }
}

}  // namespace b200

// ===================================================================================================================
// trans_dec (DiP) helpers -- reference model/mdm.py:255-270 and torch nn.TransformerDecoderLayer cross-attention
namespace b200 {

// mem16[b', m, :] = [hi | lo] fp16 of ( memproj[b', m, :] + temb_table[t(b'), :] )   (emb = text_emb + time_emb,
// mdm.py:218-220; the time embedding is broadcast over the text tokens).  Rows are 2d wide.  grid = (Mt, Bp)
__global__ void mem_build_kernel(__half* __restrict__ mem16, const float* __restrict__ memproj,
                                 const float* __restrict__ temb_table, const int* __restrict__ tvec,
                                 const int* __restrict__ tmap, const StepState* __restrict__ state, int B, int Mt, int d,
                                 int temb_rows) {
  pdl_launch_dependents();
  pdl_wait();
  const int m = blockIdx.x, bp = blockIdx.y;
  int t = (tvec != nullptr) ? tvec[bp % B] : tmap[state->cur];
  t = min(max(t, 0), temb_rows - 1);
  const size_t row = static_cast<size_t>(bp) * Mt + m;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const float v = memproj[row * d + c] + temb_table[static_cast<size_t>(t) * d + c];
    const __half hi = __float2half_rn(v);
    mem16[row * 2 * d + c] = hi;
    mem16[row * 2 * d + d + c] = __float2half_rn(v - __half2float(hi));
  }
}

// memproj rows of the packed batch: cond half = W enc + b (already in proj [B*Mt, d], row (b, m)), uncond half = b.
// tgt (optional, [B, d]): target-location embedding added to every token row of both halves (see condproj_fill_kernel).
__global__ void memproj_fill_kernel(float* __restrict__ memproj, const float* __restrict__ proj,
                                    const float* __restrict__ bias, int B, int Mt, int d, int rows_bp, int first_uncond,
                                    const float* __restrict__ tgt) {
  const int m = blockIdx.x, bp = blockIdx.y;
  if (bp >= rows_bp) return;
  const bool unc = first_uncond ? true : (bp >= B);
  const int b = bp % B;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float v = unc ? bias[c] : proj[(static_cast<size_t>(b) * Mt + m) * d + c];
    if (tgt != nullptr) v += tgt[static_cast<size_t>(b) * d + c];
    memproj[(static_cast<size_t>(bp) * Mt + m) * d + c] = v;
  }
}

// enc_text [Mt, B, C] (reference layout, model/mdm.py:185) -> [B*Mt, C] rows (b, m) so that one small GEMM projects it
__global__ void permute_mbc_kernel(const float* __restrict__ src, float* __restrict__ dst, int Mt, int B, int C) {
  const int m = blockIdx.x, b = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += blockDim.x)
    dst[(static_cast<size_t>(b) * Mt + m) * C + c] = src[(static_cast<size_t>(m) * B + b) * C + c];
}

// Cross-attention core: softmax(q k^T / sqrt(128) + mask) v with a handful of memory tokens (Mt <= 64).
//   q16 [n_samples*S, d] (head h at columns h*128), kv16 rows (sample, token) of pitch ld_kv holding k | v (v at +d), mask
//   [n_samples, Mt] (1 = ignore), out16 [n_samples*S, 2d]: the hi half only (the output projection reads K = d).
// 60 query rows x 16 tokens x 128 per (sample, head): far too small for a 128-row tcgen05 tile and bound by the ~40 MB
// of q / kv / out traffic, so each warp runs one 16-row m16n8k16 tile straight from registers:
//   * q and k fragments are read from global memory as 64 contiguous bytes per thread -- a dot product does not care
//     about the order of its terms, so thread t of a quad owns columns [32t, 32t+32) of the row for BOTH operands;
//   * softmax on the accumulator fragment (row statistics across the quad with two shuffles), exp2 with the scale
//     folded in; P is fed back as the A operand of the P.V product in two fp16 terms (hi + lo) so that the
//     probabilities carry fp32-like precision like the CUDA-core kernel this replaces;
//   * V is staged transposed in shared memory (pitch padded by 8 halves: conflict-free 32-bit fragment loads).
// A fully masked row yields 0 (the reference's softmax would give NaN there; it never occurs with a CLS token).
// grid = (heads, n_samples), block = 128 (4 warps x 16 rows per pass)
__device__ __forceinline__ void mma_m16n8k16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                             uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t pack_half2_u32(float x, float y) {
  const __half2 h = __floats2half2_rn(x, y);
  return *reinterpret_cast<const uint32_t*>(&h);
}

template <int MAX_NT>   // key tiles of 8 tokens: Mt <= 8 * MAX_NT, MAX_NT even
__global__ void __launch_bounds__(128) cross_attention_kernel(const __half* __restrict__ q16, const __half* __restrict__ kv16,
                                                              const unsigned char* __restrict__ mask,
                                                              __half* __restrict__ out16, int S, int Mt, int d, int ld_kv,
                                                              float scale_log2) {
  pdl_launch_dependents();
  pdl_wait();
  constexpr int KEYS = 8 * MAX_NT, VS = KEYS + 8;
  __shared__ __align__(16) __half sVt[128 * VS];
  __shared__ float sBias[KEYS];
  const int h = blockIdx.x, smp = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const __half* kv = kv16 + static_cast<size_t>(smp) * Mt * ld_kv + h * 128;
  for (int i = threadIdx.x; i < KEYS * 16; i += 128) {
    const int m = i >> 4, ch = i & 15;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (m < Mt) v = *reinterpret_cast<const uint4*>(kv + static_cast<size_t>(m) * ld_kv + d + ch * 8);
    const __half* hv = reinterpret_cast<const __half*>(&v);
#pragma unroll
    for (int j = 0; j < 8; ++j) sVt[(ch * 8 + j) * VS + m] = hv[j];
  }
  if (threadIdx.x < KEYS)
    sBias[threadIdx.x] = (threadIdx.x < Mt && !mask[static_cast<size_t>(smp) * Mt + threadIdx.x]) ? 0.f : -INFINITY;
  __syncthreads();

  for (int m0 = warp * 16; m0 < S; m0 += 64) {
    const int r0 = m0 + g, r1 = r0 + 8;
    const size_t row0 = static_cast<size_t>(smp) * S + min(r0, S - 1), row1 = static_cast<size_t>(smp) * S + min(r1, S - 1);
    uint32_t qa[16], qb[16];
    {
      const uint4* p0 = reinterpret_cast<const uint4*>(q16 + row0 * d + h * 128 + t * 32);
      const uint4* p1 = reinterpret_cast<const uint4*>(q16 + row1 * d + h * 128 + t * 32);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint4 a = p0[i], b = p1[i];
        qa[4 * i] = a.x; qa[4 * i + 1] = a.y; qa[4 * i + 2] = a.z; qa[4 * i + 3] = a.w;
        qb[4 * i] = b.x; qb[4 * i + 1] = b.y; qb[4 * i + 2] = b.z; qb[4 * i + 3] = b.w;
      }
    }
    float sc[MAX_NT][4];
#pragma unroll
    for (int nt = 0; nt < MAX_NT; ++nt) {
      sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
      const int key = min(nt * 8 + g, Mt - 1);                        // padded tokens are masked through sBias
      const uint4* kp = reinterpret_cast<const uint4*>(kv + static_cast<size_t>(key) * ld_kv + t * 32);
      uint32_t kw[16];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint4 a = kp[i];
        kw[4 * i] = a.x; kw[4 * i + 1] = a.y; kw[4 * i + 2] = a.z; kw[4 * i + 3] = a.w;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) mma_m16n8k16(sc[nt], qa[2 * j], qb[2 * j], qa[2 * j + 1], qb[2 * j + 1], kw[2 * j], kw[2 * j + 1]);
    }
    // softmax over the tokens: thread holds tokens nt*8 + 2t, +1 of rows g (c0, c1) and g+8 (c2, c3)
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < MAX_NT; ++nt) {
      const float b0 = sBias[nt * 8 + 2 * t], b1 = sBias[nt * 8 + 2 * t + 1];
      sc[nt][0] = fmaf(sc[nt][0], scale_log2, b0); sc[nt][1] = fmaf(sc[nt][1], scale_log2, b1);
      sc[nt][2] = fmaf(sc[nt][2], scale_log2, b0); sc[nt][3] = fmaf(sc[nt][3], scale_log2, b1);
      mx0 = fmaxf(mx0, fmaxf(sc[nt][0], sc[nt][1]));
      mx1 = fmaxf(mx1, fmaxf(sc[nt][2], sc[nt][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float off0 = (mx0 == -INFINITY) ? 0.f : mx0, off1 = (mx1 == -INFINITY) ? 0.f : mx1;
    float sum0 = 0.f, sum1 = 0.f;
    uint32_t phi[MAX_NT][2], plo[MAX_NT][2];
#pragma unroll
    for (int nt = 0; nt < MAX_NT; ++nt) {
      const float p0 = exp2f(sc[nt][0] - off0), p1 = exp2f(sc[nt][1] - off0);
      const float p2 = exp2f(sc[nt][2] - off1), p3 = exp2f(sc[nt][3] - off1);
      sum0 += p0 + p1; sum1 += p2 + p3;
      const __half2 h01 = __floats2half2_rn(p0, p1), h23 = __floats2half2_rn(p2, p3);
      const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
      phi[nt][0] = *reinterpret_cast<const uint32_t*>(&h01); phi[nt][1] = *reinterpret_cast<const uint32_t*>(&h23);
      plo[nt][0] = pack_half2_u32(p0 - f01.x, p1 - f01.y); plo[nt][1] = pack_half2_u32(p2 - f23.x, p3 - f23.y);
    }
    sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
    sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
    const float inv0 = (mx0 == -INFINITY || !(sum0 > 0.f)) ? 0.f : 1.f / sum0;
    const float inv1 = (mx1 == -INFINITY || !(sum1 > 0.f)) ? 0.f : 1.f / sum1;
    __half* o0 = out16 + (static_cast<size_t>(smp) * S + r0) * 2 * d + h * 128 + 2 * t;
    __half* o1 = out16 + (static_cast<size_t>(smp) * S + r1) * 2 * d + h * 128 + 2 * t;
#pragma unroll
    for (int nd = 0; nd < 16; ++nd) {
      float o[4] = {0.f, 0.f, 0.f, 0.f};
      const __half* vrow = sVt + (nd * 8 + g) * VS + 2 * t;
#pragma unroll
      for (int kk = 0; kk < MAX_NT / 2; ++kk) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(vrow + 16 * kk);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(vrow + 16 * kk + 8);
        mma_m16n8k16(o, phi[2 * kk][0], phi[2 * kk][1], phi[2 * kk + 1][0], phi[2 * kk + 1][1], b0, b1);
        mma_m16n8k16(o, plo[2 * kk][0], plo[2 * kk][1], plo[2 * kk + 1][0], plo[2 * kk + 1][1], b0, b1);
      }
      if (r0 < S) *reinterpret_cast<__half2*>(o0 + nd * 8) = __floats2half2_rn(o[0] * inv0, o[1] * inv0);
      if (r1 < S) *reinterpret_cast<__half2*>(o1 + nd * 8) = __floats2half2_rn(o[2] * inv1, o[3] * inv1);
    }
  }
}

}  // namespace b200
